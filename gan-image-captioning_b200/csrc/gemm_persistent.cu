// Persistent Blackwell tensor-core GEMM (sm_100a only) for the dense contractions of the hot path.
//   * operands fp32 in HBM, fed as TF32 (kind::tf32): TMA (128B swizzle) -> shared-memory ring -> tcgen05.mma
//     128 x BN x 8 issued by one thread, fp32 accumulation in TMEM
//   * persistent: one CTA per SM walks a static schedule of work segments; the accumulator is double-buffered in
//     TMEM (2 x BN columns) so the epilogue of segment i overlaps the main loop of segment i+1
//   * schedule = data-parallel rounds over whole output tiles + a stream-K tail: the tiles that do not fill a
//     round are cut along K into equal shares per CTA and combined with fp32 reductions (red.global.add) into the
//     zero-initialised / beta = 1 output
//   * epilogue: TMEM -> registers -> per-warp smem staging -> TMA store (plain stores of whole 32 x 32 blocks) or
//     128-byte coalesced global accesses (alpha/beta/bias stores, stream-K reductions)
//   * K-major and MN-major operands through the UMMA descriptor "major" bits (no transposes in the backward pass)
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue.
#include "tcgen05_common.cuh"

namespace gic {
namespace tc {

struct EpiArgs {
  float alpha, beta;
  float* C;
  int ldc;
  const float* bias;   // [N] or nullptr
  int vec_red;         // C is 16-byte aligned with ldc % 4 == 0: stream-K shares use red.global.add.v4.f32
  int tma_store;       // tmC is valid: full-width chunks of plain stores leave through cp.async.bulk.tensor
};

template <int BN>
struct PCfg {
  static constexpr int A_BYTES = BM * BK * 4;     // 16 KB
  static constexpr int B_BYTES = BN * BK * 4;
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int STG_WARP = 5120;   // per-warp staging: 32 x 33 floats (padded transpose) or a 1024-aligned 4 KB TMA tile
  static constexpr int STG_BYTES = 4 * STG_WARP;
  static constexpr int BAR_BYTES = 512;
  static constexpr int BIAS_BYTES = 1024;         // the tile's slice of the bias, staged once per tile
  static constexpr int AVAIL = 227 * 1024 - 1024 - STG_BYTES - BAR_BYTES - BIAS_BYTES;
  static constexpr int STAGES = (AVAIL / STAGE) > 8 ? 8 : (AVAIL / STAGE);
  static constexpr int TOTAL = STAGES * STAGE + STG_BYTES + BAR_BYTES + BIAS_BYTES + 1024;
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
};

// Static schedule shared by the three warp roles.  Segment = (tile, k-block range).
struct Sched {
  int tiles, tiles_n, nkb, dp_tiles;
  long long sk_lo, sk_hi;   // this CTA's share of the stream-K iteration space [0, (tiles - dp_tiles) * nkb)
  int dp_next;
  long long sk_it;
  __device__ Sched(int tiles_, int tiles_n_, int nkb_, int dp_tiles_) : tiles(tiles_), tiles_n(tiles_n_), nkb(nkb_),
                                                                        dp_tiles(dp_tiles_) {
    const long long sk_total = (long long)(tiles - dp_tiles) * nkb;
    sk_lo = sk_total * blockIdx.x / gridDim.x;
    sk_hi = sk_total * (blockIdx.x + 1) / gridDim.x;
    dp_next = blockIdx.x;
    sk_it = sk_lo;
  }
  __device__ bool next(int& tile, int& kb_lo, int& kb_hi) {
    if (dp_next < dp_tiles) {
      tile = dp_next; kb_lo = 0; kb_hi = nkb;
      dp_next += gridDim.x;
      return true;
    }
    if (sk_it < sk_hi) {
      const int t = (int)(sk_it / nkb);
      kb_lo = (int)(sk_it - (long long)t * nkb);
      const long long end = min(sk_hi, (long long)(t + 1) * nkb);
      kb_hi = kb_lo + (int)(end - sk_it);
      tile = dp_tiles + t;
      sk_it = end;
      return true;
    }
    return false;
  }
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// DT: 0 = fp32 operands fed as TF32 (k-block = 32 elements), 1 = bf16 operands (k-block = 64 elements); both are 128-byte
// rows in shared memory, so tile sizes, the ring and the K-major descriptors are identical.
template <int BN, bool A_MN, bool B_MN, int DT = 0>
__global__ void __launch_bounds__(NTHREADS, 1)
gemm_p_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
              const __grid_constant__ CUtensorMap tmC, int M, int N, int K, int tiles_n, int tiles, int dp_tiles,
              EpiArgs ea) {
  using S = PCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* stg_all = reinterpret_cast<float*>(smem + S::STAGES * S::STAGE);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::STAGES * S::STAGE + S::STG_BYTES);
  uint64_t* empty = full + S::STAGES;
  uint64_t* tmem_full = empty + S::STAGES;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* bias_s = reinterpret_cast<float*>(smem + S::STAGES * S::STAGE + S::STG_BYTES + S::BAR_BYTES);   // [BN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int BKE = DT ? 64 : 32;            // elements per k-block (128 bytes)
  constexpr int SLAB = DT ? 64 : 32;           // MN elements per 128-byte row of an MN-major slab
  constexpr int SLAB_BYTES = BKE * 128;        // one slab = BKE k-rows of 128 bytes
  const int nkb = (K + BKE - 1) / BKE;
  // one segment per CTA (tiles <= grid, no stream-K): a single accumulator is enough
  const bool single = (dp_tiles == tiles) && (tiles <= (int)gridDim.x);
  constexpr uint32_t COLS1 = (BN <= 32) ? 32 : (BN <= 64) ? 64 : (BN <= 128) ? 128 : 256;
  const uint32_t tmem_cols = single ? COLS1 : S::TMEM_COLS;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int s = 0; s < S::STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      Sched sch(tiles, tiles_n, nkb, dp_tiles);
      int tile, kb_lo, kb_hi;
      uint32_t it = 0;
      while (sch.next(tile, kb_lo, kb_hi)) {
        const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BN;
        for (int kb = kb_lo; kb < kb_hi; ++kb, ++it) {
          const int s = it % S::STAGES;
          const uint32_t ph = (it / S::STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * S::STAGE;
          uint8_t* sb = sa + S::A_BYTES;
          mbar_expect_tx(&full[s], S::STAGE);
          const int k0 = kb * BKE;
          if (A_MN) {
#pragma unroll
            for (int j = 0; j < BM / SLAB; ++j) tma_load_2d(sa + j * SLAB_BYTES, &tmA, &full[s], m0 + SLAB * j, k0);
          } else {
            tma_load_2d(sa, &tmA, &full[s], k0, m0);
          }
          if (B_MN) {
#pragma unroll
            for (int j = 0; j < BN / SLAB; ++j) tma_load_2d(sb + j * SLAB_BYTES, &tmB, &full[s], n0 + SLAB * j, k0);
          } else {
            tma_load_2d(sb, &tmB, &full[s], k0, n0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = DT ? make_idesc_bf16(A_MN ? 1 : 0, B_MN ? 1 : 0, BN) : make_idesc(A_MN ? 1 : 0, B_MN ? 1 : 0, BN);
      Sched sch(tiles, tiles_n, nkb, dp_tiles);
      int tile, kb_lo, kb_hi;
      uint32_t it = 0, seg = 0;
      while (sch.next(tile, kb_lo, kb_hi)) {
        const uint32_t acc = seg & 1, accph = (seg >> 1) & 1;
        mbar_wait(&tmem_empty[acc], accph ^ 1);          // epilogue has drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb_lo; kb < kb_hi; ++kb, ++it) {
          const int s = it % S::STAGES;
          const uint32_t ph = (it / S::STAGES) & 1;
          mbar_wait(&full[s], ph);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + s * S::STAGE);
          const uint32_t sb = sa + S::A_BYTES;
          const int kmax = min(4, (K - kb * BKE + (BKE / 4) - 1) / (BKE / 4));   // K tail: only the MMAs that hold data (TMA zero-fills the rest)
#pragma unroll
          for (int k = 0; k < 4; ++k) {          // 4 MMAs of 32 bytes of K per k-block
            if (k >= kmax) break;
            // MN-major: tf32 uses SWIZZLE_128B_BASE32B (atoms of 4 k-rows, 512 B), bf16 plain SWIZZLE_128B (atoms of
            // 8 k-rows, 1024 B); one MMA consumes 8 resp. 16 k-rows = 1024 resp. 2048 bytes
            const uint64_t da = A_MN ? (DT ? make_desc(sa + k * 2048, SLAB_BYTES, 1024, 2) : make_desc(sa + k * 1024, SLAB_BYTES, 512, 1))
                                     : make_desc(sa + k * 32, 16, 1024, 2);
            const uint64_t db = B_MN ? (DT ? make_desc(sb + k * 2048, SLAB_BYTES, 1024, 2) : make_desc(sb + k * 1024, SLAB_BYTES, 512, 1))
                                     : make_desc(sb + k * 32, 16, 1024, 2);
            if (DT) umma_bf16(d_tmem, da, db, idesc, (kb > kb_lo || k > 0) ? 1u : 0u);
            else umma_tf32(d_tmem, da, db, idesc, (kb > kb_lo || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(&tmem_full[acc]);
        ++seg;
      }
    }
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    float* stg = stg_all + q * (S::STG_WARP / 4);
    Sched sch(tiles, tiles_n, nkb, dp_tiles);
    int tile, kb_lo, kb_hi;
    uint32_t seg = 0;
    while (sch.next(tile, kb_lo, kb_hi)) {
      const uint32_t acc = seg & 1, accph = (seg >> 1) & 1;
      const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BN;
      const bool partial = (kb_hi - kb_lo) < nkb;            // stream-K share: reduce into C
      const bool first = (kb_lo == 0);
      const bool bias_smem = ea.tma_store && ea.beta == 0.f && ea.bias != nullptr;   // kernel-uniform
      if (bias_smem) {
        // the tile's bias slice goes to shared memory while the tile's MMAs still run (a global load per block inside
        // the drain loop was a dependent L2 round trip per 32 columns: 73 us instead of 45 on the EW GEMM of the step)
        asm volatile("bar.sync 1, 128;" ::: "memory");        // the previous tile's readers are done
        for (int j = (int)threadIdx.x - 64; j < BN; j += 128) bias_s[j] = (n0 + j < N) ? ea.bias[n0 + j] : 0.f;
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      mbar_wait(&tmem_full[acc], accph);
      tcgen05_fence_after();
      const uint32_t t_addr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16);
      const int m_base = m0 + q * 32;
      const int rows = min(32, M - m_base);                  // may be <= 0
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        const int W = (BN - c0 >= 32) ? 32 : 16;             // BN % 16 == 0
        uint32_t r[32];
        if (W == 32) {
          tmem_ld32(t_addr + c0, r);
        } else {
          uint32_t r16[16];
          tmem_ld16(t_addr + c0, r16);
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = r16[j];
        }
        if (c0 + 32 >= BN) {                                 // last chunk read: hand the accumulator back
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty[acc]);
        }
        if (n0 + c0 >= N || rows <= 0) continue;             // warp-uniform
        if (ea.tma_store && !partial && ea.beta == 0.f && W == 32) {
          // TMA store: the warp's 32 x 32 block goes to a 128B-swizzled 4 KB staging tile (lane = row, 16-byte chunk
          // c at physical chunk c ^ (row & 7): conflict-free STS.128), then one bulk tensor store (clipped at M, N)
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // staging tile free again
          __syncwarp();
          uint8_t* srow = reinterpret_cast<uint8_t*>(stg) + lane * 128;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            float4 v;
            v.x = ea.alpha * __uint_as_float(r[4 * c + 0]); v.y = ea.alpha * __uint_as_float(r[4 * c + 1]);
            v.z = ea.alpha * __uint_as_float(r[4 * c + 2]); v.w = ea.alpha * __uint_as_float(r[4 * c + 3]);
            if (ea.bias != nullptr) {                        // bias_smem holds on this path (zero beyond N)
              const float4 bb = *reinterpret_cast<const float4*>(bias_s + c0 + 4 * c);
              v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
            }
            *reinterpret_cast<float4*>(srow + ((c ^ (lane & 7)) << 4)) = v;
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(&tmC), "r"(smem_u32(stg)), "r"(n0 + c0), "r"(m_base) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          continue;
        }
        if (ea.tma_store) {                                  // generic path below reuses the staging tile
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < W) stg[lane * 33 + j] = __uint_as_float(r[j]);
        __syncwarp();
        const int n = n0 + c0 + lane;
        const bool n_ok = (lane < W) && (n < N);
        float bv = 0.f;
        if (ea.bias != nullptr && n_ok && first) bv = ea.bias[n];
        float* cptr = ea.C + (size_t)m_base * ea.ldc + n;
        if (partial) {
          if (ea.vec_red) {
            // 16-byte vector reductions: lane = (row lane/8, 4 columns starting at 4*(lane%8)), 4 rows per instruction
            const int cg = (lane & 7) * 4, rsub = lane >> 3;
            const int nn = n0 + c0 + cg;
            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ea.bias != nullptr && first && cg < W && nn + 3 < N) b4 = *reinterpret_cast<const float4*>(ea.bias + nn);
#pragma unroll 4
            for (int r0 = 0; r0 < 32; r0 += 4) {
              const int rr = r0 + rsub;
              if (rr < rows && cg < W && nn + 3 < N) {
                const float* sp = stg + rr * 33 + cg;
                float* gp = ea.C + (size_t)(m_base + rr) * ea.ldc + nn;
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gp), "f"(ea.alpha * sp[0] + b4.x),
                             "f"(ea.alpha * sp[1] + b4.y), "f"(ea.alpha * sp[2] + b4.z), "f"(ea.alpha * sp[3] + b4.w) : "memory");
              } else if (rr < rows && cg < W) {
                for (int e = 0; e < 4; ++e)
                  if (nn + e < N)
                    atomicAdd(ea.C + (size_t)(m_base + rr) * ea.ldc + nn + e,
                              ea.alpha * stg[rr * 33 + cg + e] + ((ea.bias != nullptr && first) ? ea.bias[nn + e] : 0.f));
              }
            }
          } else {
#pragma unroll 8
            for (int rr = 0; rr < 32; ++rr) {
              if (rr < rows && n_ok) atomicAdd(cptr + (size_t)rr * ea.ldc, ea.alpha * stg[rr * 33 + lane] + bv);
            }
          }
        } else if (ea.beta != 0.f) {
          float cv[32];                                    // all 32 row loads in flight, then the stores
#pragma unroll
          for (int i = 0; i < 32; ++i) cv[i] = ((i < rows) && n_ok) ? cptr[(size_t)i * ea.ldc] : 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if ((i < rows) && n_ok) cptr[(size_t)i * ea.ldc] = ea.alpha * stg[i * 33 + lane] + bv + ea.beta * cv[i];
        } else {
#pragma unroll 8
          for (int rr = 0; rr < 32; ++rr) {
            if (rr < rows && n_ok) cptr[(size_t)rr * ea.ldc] = ea.alpha * stg[rr * 33 + lane] + bv;
          }
        }
        __syncwarp();
      }
      ++seg;
    }
    if (ea.tma_store && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols));
  }
}

template <int BN, bool A_MN, bool B_MN, int DT = 0>
static int launch_p(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tcm, int M, int N, int K, int tiles_n, int tiles,
                    int dp_tiles, int grid, const EpiArgs& ea, cudaStream_t s) {
  using S = PCfg<BN>;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(gemm_p_kernel<BN, A_MN, B_MN, DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    attr = true;
  }
  gemm_p_kernel<BN, A_MN, B_MN, DT><<<grid, NTHREADS, S::TOTAL, s>>>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, ea);
  return check_launch("gemm_p_kernel");
}

// Tile width: minimise (segments per CTA) x (cycles per k-block) with the k-block cost = max(MMA floor 2*BN cycles,
// shared-memory feed (16 KB + 128*BN B) at ~48 B/cycle/SM when every SM pulls from L2) plus a per-tile epilogue.
static int choose_bn(int M, int N, int K, bool b_mn, bool allow_sk) {
  static const int kBN[6] = {64, 128, 144, 192, 240, 256};
  const int G = num_sms();
  const int nkb = cdiv(K, BK);
  double best = -1.0;
  int BN = 128;
  for (int i = 0; i < 6; ++i) {
    const int bn = kBN[i];
    if (b_mn && (bn % 32)) continue;                   // MN-major B is loaded as 32-wide slabs
    const long long tiles = (long long)cdiv(N, bn) * cdiv(M, BM);
    const double t_kb = fmax(2.0 * bn, (16384.0 + 128.0 * bn) / 48.0);
    const double t_epi = 13.0 * bn;
    double iters;                                       // k-block iterations on the busiest CTA
    double epis;
    if (allow_sk && tiles * 2 <= G) { iters = fmax(1.0, (double)tiles * nkb / G); epis = 2.0 * 3.0; }   // reductions ~3x a store
    else { iters = (double)cdiv(tiles, G) * nkb; epis = (double)cdiv(tiles, G); }
    const double cost = iters * t_kb + epis * t_epi;
    if (best < 0 || cost < best) { best = cost; BN = bn; }
  }
  return BN;
}

}  // namespace tc

// Persistent GEMM entry: C = alpha*op(A)*op(B) + beta*C + bias.  handled = false (nothing launched) when the operands do
// not meet TMA's constraints or the shape is left to the other kernels.
int gemm_tc_persistent(bool transA, bool transB, int M, int N, int K, float alpha, const float* A, int lda,
                       const float* B, int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream,
                       bool* handled) {
  using namespace tc;
  *handled = false;
  if (M <= 0 || N <= 0 || K <= 0) return GIC_OK;
  if (!aligned16(A) || !aligned16(B) || (lda % 4) || (ldb % 4)) return GIC_OK;
  if ((long long)M * N < 64 * 64 || K < 32) return GIC_OK;
  const bool rn = tf32_round_in_tma();
  const bool a_mn = transA, b_mn = !transB;
  const bool allow_sk = (beta == 0.f || beta == 1.f);
  int BN = choose_bn(M, N, K, b_mn, allow_sk);
  { const int f = option("GIC_GEMM_BN", 0); if (f == 64 || f == 128 || f == 192 || f == 256 || (!b_mn && (f == 144 || f == 240))) BN = f; }   // tuning
  CUtensorMap ta, tb;
  bool ok;
  if (a_mn) ok = make_map(&ta, A, K, M, lda, 32, BK, rn, true);
  else      ok = make_map(&ta, A, M, K, lda, BK, BM, rn, false);
  if (ok) {
    if (b_mn) ok = make_map(&tb, B, K, N, ldb, 32, BK, rn, true);
    else      ok = make_map(&tb, B, N, K, ldb, BK, BN, rn, false);
  }
  if (!ok) return GIC_OK;
  const int G = num_sms();
  const int tiles_n = cdiv(N, BN), tiles_m = cdiv(M, BM), tiles = tiles_n * tiles_m, nkb = cdiv(K, BK);
  int dp_tiles = tiles;
  if (allow_sk && option("GIC_SK", 1)) {
    // stream-K only when whole tiles cannot occupy half the machine (long-K / small-MN shapes of the backward pass):
    // every CTA gets an equal share of the (tile, k-block) iteration space.  fp32 reductions into L2 cost ~5 ps per
    // element, so a tail of partial tiles after full data-parallel rounds does not pay off.
    if (tiles * 2 <= G && (long long)tiles * nkb >= 4LL * G) dp_tiles = 0;
  }
  // Long-K shapes that need no stream-K (dW_out, dhtop of the generator backward) measure ~20% faster on the
  // one-tile-per-CTA kernel of gemm_tcgen05.cu (profiles/README.md, "GEMM A/B"): leave them to it.
  if (dp_tiles == tiles && nkb >= 128) return GIC_OK;
  const int grid = (dp_tiles < tiles) ? G : min(tiles, G);
  if (dp_tiles < tiles && beta == 0.f) {
    // zero the rows that hold stream-K tiles (a superset: data-parallel tiles in those rows are stored afterwards)
    const int row0 = (dp_tiles / tiles_n) * BM;
    cudaError_t e = cudaMemset2DAsync(C + (size_t)row0 * ldc, (size_t)ldc * sizeof(float), 0, (size_t)N * sizeof(float),
                                      M - row0, stream);
    if (e != cudaSuccess) { set_error("memset2D: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  }
  EpiArgs ea;
  ea.alpha = alpha; ea.beta = beta; ea.C = C; ea.ldc = ldc; ea.bias = bias;
  CUtensorMap tcm;
  ea.vec_red = (aligned16(C) && (ldc % 4) == 0 && (!bias || aligned16(bias))) ? 1 : 0;
  ea.tma_store = 0;
  if (beta == 0.f && aligned16(C) && (ldc % 4) == 0 && (!bias || aligned16(bias)))
    ea.tma_store = make_map(&tcm, C, M, N, ldc, 32, 32, false, false) ? 1 : 0;
  if (!ea.tma_store) tcm = ta;                       // unused placeholder
  int rc = GIC_OK;
#define GIC_P(BN_)                                                                                                  \
  do {                                                                                                              \
    if (!a_mn && !b_mn) rc = launch_p<BN_, false, false>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
    else if (a_mn && !b_mn) rc = launch_p<BN_, true, false>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
    else if constexpr ((BN_ % 32) == 0) {                                                                           \
      if (!a_mn) rc = launch_p<BN_, false, true>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream);  \
      else rc = launch_p<BN_, true, true>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream);         \
    }                                                                                                               \
  } while (0)
  switch (BN) {
    case 64: GIC_P(64); break;
    case 128: GIC_P(128); break;
    case 144: GIC_P(144); break;
    case 192: GIC_P(192); break;
    case 240: GIC_P(240); break;
    default: GIC_P(256); break;
  }
#undef GIC_P
  if (rc == GIC_OK) *handled = true;
  return rc;
}

int gemm_tc_bf16_pair(bool b_mn, int M, int N, int K, float alpha, const void* A, int lda, const void* B, int ldb, float* C,
                      int ldc, const float* bias, cudaStream_t stream, bool* handled);

// bf16 operands (kind::f16), fp32 accumulate and fp32 output: the discriminator's [N*R, F] x [F, F] contractions in
// GIC_GEMM_BF16 mode.  A / B are bf16 with leading dimensions in elements (multiples of 8); layouts as gemm().
int gemm_tc_bf16(bool transA, bool transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B,
                 int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream, bool* handled) {
  using namespace tc;
  *handled = false;
  if (M <= 0 || N <= 0 || K <= 0) return GIC_OK;
  if (!aligned16(A) || !aligned16(B) || (lda % 8) || (ldb % 8)) return GIC_OK;
  const bool a_mn = transA, b_mn = !transB;
  // whole-tile shapes with a K-major A and a plain-store epilogue: CTA pairs (gemm_pair_tcgen05.cu)
  if (!a_mn && beta == 0.f) {
    GIC_TRY(gemm_tc_bf16_pair(b_mn, M, N, K, alpha, A, lda, B, ldb, C, ldc, bias, stream, handled));
    if (*handled) return GIC_OK;
  }
  const bool allow_sk = (beta == 0.f || beta == 1.f);
  const int G = num_sms();
  // tile width: as choose_bn with 64-element k-blocks; MN-major B needs BN % 64 == 0
  int BN = 256;
  {
    static const int kBN[4] = {64, 128, 192, 256};
    double best = -1.0;
    const int nkb = cdiv(K, 64);
    for (int i = 0; i < 4; ++i) {
      const int bn = kBN[i];
      if (b_mn && (bn % 64)) continue;
      const long long tiles = (long long)cdiv(N, bn) * cdiv(M, BM);
      const double t_kb = fmax(1.0 * bn, (16384.0 + 128.0 * bn) / 48.0);
      double iters, epis;
      if (allow_sk && tiles * 2 <= G) { iters = fmax(1.0, (double)tiles * nkb / G); epis = 6.0; }
      else { iters = (double)cdiv(tiles, G) * nkb; epis = (double)cdiv(tiles, G); }
      const double cost = iters * t_kb + epis * 13.0 * bn;
      if (best < 0 || cost < best) { best = cost; BN = bn; }
    }
  }
  CUtensorMap ta, tb;
  bool ok;
  if (a_mn) ok = make_map_bf16(&ta, A, K, M, lda, 64, 64);
  else      ok = make_map_bf16(&ta, A, M, K, lda, 64, BM);
  if (ok) {
    if (b_mn) ok = make_map_bf16(&tb, B, K, N, ldb, 64, 64);
    else      ok = make_map_bf16(&tb, B, N, K, ldb, 64, BN);
  }
  if (!ok) return GIC_OK;
  const int tiles_n = cdiv(N, BN), tiles_m = cdiv(M, BM), tiles = tiles_n * tiles_m, nkb = cdiv(K, 64);
  int dp_tiles = tiles;
  if (allow_sk && tiles * 2 <= G && (long long)tiles * nkb >= 4LL * G) dp_tiles = 0;
  const int grid = (dp_tiles < tiles) ? G : min(tiles, G);
  if (dp_tiles < tiles && beta == 0.f) {
    cudaError_t e = cudaMemset2DAsync(C, (size_t)ldc * sizeof(float), 0, (size_t)N * sizeof(float), M, stream);
    if (e != cudaSuccess) { set_error("memset2D: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  }
  EpiArgs ea;
  ea.alpha = alpha; ea.beta = beta; ea.C = C; ea.ldc = ldc; ea.bias = bias;
  ea.vec_red = (aligned16(C) && (ldc % 4) == 0 && (!bias || aligned16(bias))) ? 1 : 0;
  CUtensorMap tcm;
  ea.tma_store = 0;
  if (beta == 0.f && aligned16(C) && (ldc % 4) == 0 && (!bias || aligned16(bias)))
    ea.tma_store = make_map(&tcm, C, M, N, ldc, 32, 32, false, false) ? 1 : 0;
  if (!ea.tma_store) tcm = ta;
  int rc = GIC_OK;
#define GIC_PB(BN_)                                                                                                  \
  do {                                                                                                              \
    if (!a_mn && !b_mn) rc = launch_p<BN_, false, false, 1>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
    else if (a_mn && !b_mn) rc = launch_p<BN_, true, false, 1>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
    else if (!a_mn) rc = launch_p<BN_, false, true, 1>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
    else rc = launch_p<BN_, true, true, 1>(ta, tb, tcm, M, N, K, tiles_n, tiles, dp_tiles, grid, ea, stream); \
  } while (0)
  switch (BN) {
    case 64: GIC_PB(64); break;
    case 128: GIC_PB(128); break;
    case 192: GIC_PB(192); break;
    default: GIC_PB(256); break;
  }
#undef GIC_PB
  if (rc == GIC_OK) *handled = true;
  return rc;
}

}  // namespace gic
