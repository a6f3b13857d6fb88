// Beam-search caption generation (EXTENSION, parity unpinned by reference: oracle/ref_beam.py beam_search).
//
// Per decode step the vocab projection of every live beam row is reduced on chip to what the search needs: each row's
// log-softmax normaliser and its K largest logits.  The candidate producers write, per (vocabulary slice, row),
//   part_ms  [slices][Mpad]     float2 (m, s): running max of the slice's logits and sum of exp(logit - m)
//   part_cand[slices][Mpad][K]  float2 (logit, column as int bits), descending, ties -> lower column
// and the shared consumers combine the slices:
//   topk_rows_kernel   per row: lse = log-sum-exp, logp / tokens of the row's top K       (gic_vocab_topk)
//   beam_merge_kernel  per image: the image's K best (parent, token) candidates, scores / frozen flags / lengths, the
//                      (parent, token) trace, the parents' (h, c) of every layer gathered into the next state, x = embed[tok]
//   beam_finalize_kernel per image: backtrack, PAD after EOS, sort by score / length^length_penalty
// Producers:
//   vocab_topk_kernel  (tensor-core modes) one CTA per (128-row block, vocabulary slice); TMA ring for h and W_out,
//                      tcgen05.mma kind::tf32 into a double-buffered TMEM accumulator (tile j's epilogue runs under tile
//                      j + 1's MMAs); the epilogue adds the bias and keeps the online (max, sum of exp) and a running top-K
//                      in registers, one row per thread.  Nothing of size V leaves the chip and no CTA waits on another.
//   row_topk_kernel    (exact-fp32 mode, and shapes TMA rejects) the logits from gemm(...) in workspace, one block per row,
//                      the same layout as ONE slice.
#include "tcgen05_common.cuh"

namespace gic {
namespace tc {

constexpr int TK_BN = 128;                       // columns per tile (one TMEM accumulator buffer)
constexpr int TK_G = 2;                          // epilogue warps per TMEM lane quarter: they split a tile's 16-column units
constexpr int TK_EPI = 128 * TK_G;
constexpr int TK_THREADS = 64 + TK_EPI;          // warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, 8 epilogue warps
constexpr int TK_STAGE = BM * BK * 4 + TK_BN * BK * 4;    // 32 KB: 128 rows of h + 128 rows of W_out, 32 fp32 of K
constexpr int TK_STAGES = 5;
constexpr int TK_SMEM = TK_STAGES * TK_STAGE + 256 + 1024;
constexpr uint32_t TK_TMEM_COLS = 2 * TK_BN;
static_assert(TK_G * BM * (16 + 1) * 8 <= TK_STAGES * TK_STAGE, "vocab_topk: merge buffers exceed the ring");

struct TKArgs {
  int M, N, K, tiles_n, tiles_per_slice, Mpad, topk;
  const float* bias;
  float2* part_ms;
  float2* part_cand;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tk_epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(TK_EPI) : "memory"); }

// (v, col) into a descending list of KMAX entries.  Columns arrive in increasing order per thread, so a value equal to one
// already listed goes behind it: ties keep the lower column first.
template <int KMAX>
__device__ __forceinline__ void topk_insert(float (&tv)[KMAX], int (&ti)[KMAX], float v, int col) {
  if (!(v > tv[KMAX - 1])) return;
  bool ins = false;
#pragma unroll
  for (int j = 0; j < KMAX; ++j) {
    const bool sw = ins || (v > tv[j]);
    const float a = tv[j];
    const int b = ti[j];
    tv[j] = sw ? v : a; ti[j] = sw ? col : b;
    v = sw ? a : v; col = sw ? b : col;
    ins = sw;
  }
}
// a ranks before b: higher value, then lower column
__device__ __forceinline__ bool cand_before(float av, int ac, float bv, int bc) { return av > bv || (av == bv && ac < bc); }
// (m, s) pairs of the online log-sum-exp
__device__ __forceinline__ void ms_combine(float& M, float& S, float m, float s) {
  if (m == -INFINITY) return;
  if (m > M) { S = S * ((M > -INFINITY) ? expf(M - m) : 0.f) + s; M = m; }
  else S += s * expf(m - M);
}

template <int KMAX>
__global__ void __launch_bounds__(TK_THREADS, 1)
vocab_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, TKArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + TK_STAGES * TK_STAGE);
  uint64_t* empty = full + TK_STAGES;
  uint64_t* tfull = empty + TK_STAGES;            // [2] accumulator buffer b holds a finished tile
  uint64_t* tempty = tfull + 2;                   // [2] the epilogue has read accumulator buffer b
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int slice = blockIdx.x, mtile = blockIdx.y;
  const int m0 = mtile * BM;
  const int jt0 = slice * a.tiles_per_slice;
  const int nt = min(a.tiles_n - jt0, a.tiles_per_slice);
  const int nkb = (a.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int s = 0; s < TK_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], TK_EPI / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TK_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer: (h rows, W_out rows) k-blocks of every tile of the slice through one ring =====
    if (lane == 0) {
      int it = 0;
      for (int j = 0; j < nt; ++j) {
        const int n0 = (jt0 + j) * TK_BN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % TK_STAGES;
          const uint32_t ph = (it / TK_STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * TK_STAGE;
          mbar_expect_tx(&full[s], TK_STAGE);
          tma_load_2d(sa, &tmA, &full[s], kb * BK, m0);
          tma_load_2d(sa + BM * BK * 4, &tmB, &full[s], kb * BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: tile j accumulates into TMEM buffer j & 1 once the epilogue has drained tile j - 2 =====
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(0, 0, TK_BN);
      int it = 0;
      for (int j = 0; j < nt; ++j) {
        const int buf = j & 1;
        if (j >= 2) mbar_wait(&tempty[buf], ((j >> 1) - 1) & 1);
        tcgen05_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(buf * TK_BN);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % TK_STAGES;
          const uint32_t ph = (it / TK_STAGES) & 1;
          mbar_wait(&full[s], ph);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + s * TK_STAGE);
          const uint32_t sb = sa + BM * BK * 4;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t da = make_desc(sa + k * 32, 16, 1024, 2);
            const uint64_t db = make_desc(sb + k * 32, 16, 1024, 2);
            umma_tf32(d, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(&tfull[buf]);
      }
    }
  } else {
    // ===== epilogue: thread = (row, column group g); group g takes the 16-column units g, g + TK_G, ... of every tile =====
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int g = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int m = m0 + row;
    float tv[KMAX];
    int ti[KMAX];
#pragma unroll
    for (int i = 0; i < KMAX; ++i) { tv[i] = -INFINITY; ti[i] = 0x7fffffff; }
    float m_run = -INFINITY, s_run = 0.f;
    for (int j = 0; j < nt; ++j) {
      const int buf = j & 1;
      mbar_wait(&tfull[buf], (j >> 1) & 1);
      tcgen05_fence_after();
      const int n0 = (jt0 + j) * TK_BN;
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * TK_BN);
      // (one 16-column unit at a time, not unrolled: the insertion network is large and the epilogue would become
      //  instruction-fetch bound fully unrolled)
#pragma unroll 1
      for (int i = 0; i < TK_BN / 16 / TK_G; ++i) {
        uint32_t r[16];
        tmem_ld16(t_addr + 16 * (g + i * TK_G), r);
        if (i == TK_BN / 16 / TK_G - 1) {
          // the accumulator buffer is free for tile j + 2 once every epilogue warp holds its last unit in registers
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[buf]);
        }
        const int nb = n0 + 16 * (g + i * TK_G);
        float z[16];
        float cm = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int n = nb + 4 * k;
          if (n < a.N) {                         // N % 4 == 0: a float4 is entirely inside or outside
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.bias + n));
            z[4 * k + 0] = __uint_as_float(r[4 * k + 0]) + b4.x;
            z[4 * k + 1] = __uint_as_float(r[4 * k + 1]) + b4.y;
            z[4 * k + 2] = __uint_as_float(r[4 * k + 2]) + b4.z;
            z[4 * k + 3] = __uint_as_float(r[4 * k + 3]) + b4.w;
          } else {
            z[4 * k + 0] = z[4 * k + 1] = z[4 * k + 2] = z[4 * k + 3] = -INFINITY;
          }
          cm = fmaxf(cm, fmaxf(fmaxf(z[4 * k + 0], z[4 * k + 1]), fmaxf(z[4 * k + 2], z[4 * k + 3])));
        }
        if (cm > -INFINITY) {
          const float m_new = fmaxf(m_run, cm);
          s_run *= (m_run > -INFINITY) ? __expf(m_run - m_new) : 0.f;
          m_run = m_new;
          float cs = 0.f;
#pragma unroll
          for (int e = 0; e < 16; ++e) cs += __expf(z[e] - m_new);
          s_run += cs;
          if (cm > tv[KMAX - 1]) {
#pragma unroll
            for (int e = 0; e < 16; ++e) topk_insert<KMAX>(tv, ti, z[e], nb + e);
          }
        }
      }
    }
    // ---- the TK_G lists of a row meet in shared memory (the operand ring is dead: every MMA has completed)
    float2* xs = reinterpret_cast<float2*>(smem);                  // [TK_G][BM][KMAX]
    float2* xm = xs + TK_G * BM * KMAX;                            // [TK_G][BM]
#pragma unroll
    for (int i = 0; i < KMAX; ++i) xs[(g * BM + row) * KMAX + i] = make_float2(tv[i], __int_as_float(ti[i]));
    xm[g * BM + row] = make_float2(m_run, s_run);
    tk_epi_bar();
    if (g == 0 && m < a.M) {
      float M = -INFINITY, S = 0.f;
#pragma unroll
      for (int h = 0; h < TK_G; ++h) { const float2 v = xm[h * BM + row]; ms_combine(M, S, v.x, v.y); }
      a.part_ms[(size_t)slice * a.Mpad + m] = make_float2(M, S);
      float2* out = a.part_cand + ((size_t)slice * a.Mpad + m) * a.topk;
      int head[TK_G];
#pragma unroll
      for (int h = 0; h < TK_G; ++h) head[h] = 0;
      for (int k = 0; k < a.topk; ++k) {
        int best = 0;
        float2 bv = xs[(0 * BM + row) * KMAX + head[0]];
#pragma unroll
        for (int h = 1; h < TK_G; ++h) {
          const float2 v = xs[(h * BM + row) * KMAX + head[h]];
          if (cand_before(v.x, __float_as_int(v.y), bv.x, __float_as_int(bv.y))) { bv = v; best = h; }
        }
        out[k] = bv;
#pragma unroll
        for (int h = 0; h < TK_G; ++h) head[h] += (h == best) ? 1 : 0;
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TK_TMEM_COLS));
  }
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------------------
// CUDA-core producer: logits[M, V] already in memory (gemm(...) with the bias), one block per row -> slice 0
// ---------------------------------------------------------------------------------------------------------
constexpr int RT_THREADS = 256;

template <int KMAX>
__global__ void __launch_bounds__(RT_THREADS)
row_topk_kernel(const float* __restrict__ logits, int V, int topk, float2* part_ms, float2* part_cand) {
  using namespace tc;
  __shared__ float2 s_list[RT_THREADS * KMAX];
  __shared__ float2 s_ms[RT_THREADS / 32];
  __shared__ float2 s_win[RT_THREADS / 32];
  __shared__ int s_wt[RT_THREADS / 32];
  const int m = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const float* row = logits + (size_t)m * V;
  float tv[KMAX];
  int ti[KMAX];
#pragma unroll
  for (int i = 0; i < KMAX; ++i) { tv[i] = -INFINITY; ti[i] = 0x7fffffff; }
  float M = -INFINITY, S = 0.f;
  for (int n = tid; n < V; n += RT_THREADS) {
    const float z = row[n];
    if (z == -INFINITY) continue;
    if (z > M) { S = S * expf(M - z) + 1.f; M = z; }
    else S += expf(z - M);
    topk_insert<KMAX>(tv, ti, z, n);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, M, o), os = __shfl_xor_sync(0xffffffffu, S, o);
    ms_combine(M, S, om, os);
  }
  if (lane == 0) s_ms[w] = make_float2(M, S);
#pragma unroll
  for (int i = 0; i < KMAX; ++i) s_list[tid * KMAX + i] = make_float2(tv[i], __int_as_float(ti[i]));
  __syncthreads();
  if (tid == 0) {
    float Mb = -INFINITY, Sb = 0.f;
    for (int i = 0; i < RT_THREADS / 32; ++i) ms_combine(Mb, Sb, s_ms[i].x, s_ms[i].y);
    part_ms[m] = make_float2(Mb, Sb);
  }
  // K rounds: every thread offers the head of its list, the block's best is emitted and its owner advances
  int head = 0;
  float2* out = part_cand + (size_t)m * topk;
  for (int k = 0; k < topk; ++k) {
    float2 v = (head < KMAX) ? s_list[tid * KMAX + head] : make_float2(-INFINITY, __int_as_float(0x7fffffff));
    int owner = tid;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, v.x, o);
      const int oc = __shfl_xor_sync(0xffffffffu, __float_as_int(v.y), o);
      const int ow = __shfl_xor_sync(0xffffffffu, owner, o);
      if (cand_before(ov, oc, v.x, __float_as_int(v.y)) || (ov == v.x && oc == __float_as_int(v.y) && ow < owner)) {
        v = make_float2(ov, __int_as_float(oc)); owner = ow;
      }
    }
    if (lane == 0) { s_win[w] = v; s_wt[w] = owner; }
    __syncthreads();
    float2 b = s_win[0];
    int bo = s_wt[0];
    for (int i = 1; i < RT_THREADS / 32; ++i)
      if (cand_before(s_win[i].x, __float_as_int(s_win[i].y), b.x, __float_as_int(b.y)) ||
          (s_win[i].x == b.x && __float_as_int(s_win[i].y) == __float_as_int(b.y) && s_wt[i] < bo)) { b = s_win[i]; bo = s_wt[i]; }
    if (tid == 0) out[k] = b;
    if (tid == bo) ++head;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------
// consumers
// ---------------------------------------------------------------------------------------------------------
// log-sum-exp of row m over the slices, computed by one warp
__device__ __forceinline__ float row_lse(const float2* part_ms, int slices, int Mpad, int m, int lane) {
  float M = -INFINITY, S = 0.f;
  for (int s = lane; s < slices; s += 32) { const float2 v = part_ms[(size_t)s * Mpad + m]; tc::ms_combine(M, S, v.x, v.y); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, M, o), os = __shfl_xor_sync(0xffffffffu, S, o);
    tc::ms_combine(M, S, om, os);
  }
  return M + logf(S);
}

// A candidate of the beam search: score, parent beam, token.  Ranking: higher score, then lower parent, then lower token.
struct BKey { float v; int p; int c; };
__device__ __forceinline__ bool key_before(const BKey& a, const BKey& b) {
  return a.v > b.v || (a.v == b.v && (a.p < b.p || (a.p == b.p && a.c < b.c)));
}
__device__ __forceinline__ BKey key_shfl(const BKey& k, int o) {
  return BKey{__shfl_xor_sync(0xffffffffu, k.v, o), __shfl_xor_sync(0xffffffffu, k.p, o), __shfl_xor_sync(0xffffffffu, k.c, o)};
}
// The best key of the block that ranks strictly after `prev` (every thread offers its own best); all threads get it.
template <int NT>
__device__ __forceinline__ BKey block_best(BKey k, BKey* s_red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { const BKey x = key_shfl(k, o); if (key_before(x, k)) k = x; }
  if (lane == 0) s_red[w] = k;
  __syncthreads();
  BKey b = s_red[0];
#pragma unroll
  for (int i = 1; i < NT / 32; ++i) if (key_before(s_red[i], b)) b = s_red[i];
  __syncthreads();
  return b;
}
constexpr BKey KEY_NONE = {-INFINITY, 0x7fffffff, 0x7fffffff};

// gic_vocab_topk: one block per row
constexpr int TR_THREADS = 128;
__global__ void __launch_bounds__(TR_THREADS)
topk_rows_kernel(const float2* part_ms, const float2* part_cand, int slices, int Mpad, int topk, int V, float* logp,
                 int64_t* tokens, float* lse_out) {
  __shared__ BKey s_red[TR_THREADS / 32];
  __shared__ float s_lse;
  const int m = blockIdx.x, tid = threadIdx.x;
  if (tid < 32) { const float l = row_lse(part_ms, slices, Mpad, m, tid); if (tid == 0) s_lse = l; }
  __syncthreads();
  const float lse = s_lse;
  const int n = slices * topk;
  BKey prev = {INFINITY, -1, -1};
  for (int k = 0; k < topk; ++k) {
    BKey best = KEY_NONE;
    for (int i = tid; i < n; i += TR_THREADS) {
      const int s = i / topk, j = i - s * topk;
      const float2 c = part_cand[((size_t)s * Mpad + m) * topk + j];
      const BKey x = {c.x, 0, __float_as_int(c.y)};
      if (x.c < V && key_before(prev, x) && key_before(x, best)) best = x;
    }
    best = block_best<TR_THREADS>(best, s_red);
    if (tid == 0) {
      logp[(size_t)m * topk + k] = best.v - lse;
      tokens[(size_t)m * topk + k] = best.c;
      if (k == 0 && lse_out) lse_out[m] = lse;
    }
    prev = best;
  }
}

constexpr int BEAM_MAX_LAYERS = 8;
struct BeamState {
  float* hA[BEAM_MAX_LAYERS]; float* cA[BEAM_MAX_LAYERS];       // state the next step reads (gathered by the merge)
  const float* hB[BEAM_MAX_LAYERS]; const float* cB[BEAM_MAX_LAYERS];   // state the LSTM step just wrote
  float* x;                 // [B K, E] next LSTM input
  float* score;             // [B K] running sums of log-probabilities
  int* fin;                 // [B K] frozen (has emitted EOS)
  int* len;                 // [B K] tokens up to and including EOS, L while none was emitted
  int2* trace;              // [L][B][K] (parent slot, token)
  const float* embed;
  int layers, H, E, K, L, V, B;
  int eos;
};

// One CTA per image: select the image's K best candidates and reorder the beam state (kernel comment at the top).
constexpr int BM_THREADS = 256;
__global__ void __launch_bounds__(BM_THREADS)
beam_merge_kernel(const float2* part_ms, const float2* part_cand, int slices, int Mpad, int t, BeamState st) {
  __shared__ BKey s_red[BM_THREADS / 32];
  __shared__ float s_lse[16], s_sc[16], s_new[16];
  __shared__ int s_fin[16], s_len[16], s_par[16], s_tok[16];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int K = st.K;
  const int r0 = b * K;
  for (int k = w; k < K; k += BM_THREADS / 32) {
    const float l = row_lse(part_ms, slices, Mpad, r0 + k, lane);
    if (lane == 0) { s_lse[k] = l; s_sc[k] = st.score[r0 + k]; s_fin[k] = st.fin[r0 + k]; s_len[k] = st.len[r0 + k]; }
  }
  __syncthreads();
  // candidates: live beam k -> its slices' top K tokens, score + logit - lse; frozen beam k -> (k, PAD) at its own score
  const int per_beam = slices * K;
  const int n = K * per_beam + K;
  BKey prev = {INFINITY, -1, -1};
  for (int r = 0; r < K; ++r) {
    BKey best = KEY_NONE;
    for (int i = tid; i < n; i += BM_THREADS) {
      BKey x;
      if (i < K * per_beam) {
        const int k = i / per_beam, rest = i - k * per_beam;
        if (s_fin[k]) continue;
        const int s = rest / K, j = rest - s * K;
        const float2 c = part_cand[((size_t)s * Mpad + r0 + k) * K + j];
        x.c = __float_as_int(c.y);
        if (x.c >= st.V) continue;
        x.v = s_sc[k] + (c.x - s_lse[k]);
        x.p = k;
      } else {
        const int k = i - K * per_beam;
        if (!s_fin[k]) continue;
        x = BKey{s_sc[k], k, 0};
      }
      if (key_before(prev, x) && key_before(x, best)) best = x;
    }
    best = block_best<BM_THREADS>(best, s_red);
    if (tid == 0) { s_par[r] = best.p; s_tok[r] = best.c; s_new[r] = best.v; }
    prev = best;
  }
  __syncthreads();
  if (tid < K) {
    const int p = s_par[tid], tok = s_tok[tid];
    const int pf = s_fin[p];
    st.score[r0 + tid] = s_new[tid];
    st.fin[r0 + tid] = (pf || tok == st.eos) ? 1 : 0;
    st.len[r0 + tid] = pf ? s_len[p] : (tok == st.eos ? t + 1 : st.L);
    st.trace[((size_t)t * st.B + b) * K + tid] = make_int2(p, tok);
  }
  if (t + 1 >= st.L) return;
  // next state: the parents' (h, c) of every layer, x = embed[token]
  const int H = st.H, E = st.E;
  for (int l = 0; l < st.layers; ++l) {
    for (int i = tid; i < K * H; i += BM_THREADS) {
      const int k = i / H, u = i - k * H;
      const size_t src = (size_t)(r0 + s_par[k]) * H + u, dst = (size_t)(r0 + k) * H + u;
      st.hA[l][dst] = st.hB[l][src];
      st.cA[l][dst] = st.cB[l][src];
    }
  }
  for (int i = tid; i < K * E; i += BM_THREADS) {
    const int k = i / E, u = i - k * E;
    st.x[(size_t)(r0 + k) * E + u] = __ldg(st.embed + (size_t)s_tok[k] * E + u);
  }
}

// step 0: x = features of the image for every beam, beam 0 at score 0 and the others at -inf, nothing frozen
__global__ void beam_init_kernel(const float* features, BeamState st) {
  const int r = blockIdx.x, k = r % st.K, b = r / st.K;
  for (int u = threadIdx.x; u < st.E; u += blockDim.x) st.x[(size_t)r * st.E + u] = features[(size_t)b * st.E + u];
  if (threadIdx.x == 0) { st.score[r] = (k == 0) ? 0.f : -INFINITY; st.fin[r] = 0; st.len[r] = st.L; }
}

// one warp per image: rank by score / length^length_penalty (ties -> lower slot), backtrack the trace
__global__ void beam_finalize_kernel(BeamState st, float length_penalty, int64_t* ids, float* scores, int32_t* lengths) {
  const int b = blockIdx.x, k = threadIdx.x, K = st.K;
  const int r = b * K + k;
  float ns = 0.f;
  if (k < K) ns = (length_penalty == 0.f) ? st.score[r] : st.score[r] / powf((float)st.len[r], length_penalty);
  int rank = 0;
  for (int j = 0; j < K; ++j) {
    const float o = __shfl_sync(0xffffffffu, ns, j);
    if (k < K && (o > ns || (o == ns && j < k))) ++rank;
  }
  if (k >= K) return;
  const int o = b * K + rank;
  scores[o] = st.score[r];
  lengths[o] = st.len[r];
  int slot = k;
  for (int t = st.L - 1; t >= 0; --t) {
    const int2 pt = st.trace[((size_t)t * st.B + b) * K + slot];
    ids[(size_t)o * st.L + t] = pt.y;
    slot = pt.x;
  }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
static size_t a4(size_t x) { return (x + 3) & ~(size_t)3; }

// workspace of the candidate producers (floats): part_ms | part_cand | logits[M, V] (exact-fp32 / unaligned path)
struct TopkWs {
  size_t ms, cand, logits, total;
  int Mpad, smax;
  TopkWs(int M, int V, int K) {
    Mpad = cdiv(M, tc::BM) * tc::BM;
    smax = cdiv(V, tc::TK_BN);
    ms = 0;
    cand = a4((size_t)2 * smax * Mpad);
    logits = cand + a4((size_t)2 * smax * Mpad * K);
    total = logits + a4((size_t)M * V);
  }
};
size_t vocab_topk_ws_floats(int M, int V, int K) { return TopkWs(M, V, K).total; }

template <int KMAX>
static int launch_tk(const CUtensorMap& ta, const CUtensorMap& tb, const tc::TKArgs& a, dim3 grid, cudaStream_t s) {
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(tc::vocab_topk_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TK_SMEM);
    attr = true;
  }
  tc::vocab_topk_kernel<KMAX><<<grid, tc::TK_THREADS, tc::TK_SMEM, s>>>(ta, tb, a);
  return check_launch("vocab_topk_kernel");
}

// Per-slice (m, s) and top-K candidates of the rows of h[M, H] W_out^T + b_out into ws; *slices = how many slices.
int vocab_topk_partials(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K,
                        float* ws, cudaStream_t s, int* slices) {
  using namespace tc;
  const TopkWs w(M, V, K);
  float2* part_ms = reinterpret_cast<float2*>(ws + w.ms);
  float2* part_cand = reinterpret_cast<float2*>(ws + w.cand);
  const bool tensor = (mode == GEMM_TF32 || mode == GEMM_BF16) && option("GIC_FUSED_TOPK", 1) != 0;
  if (tensor && (V % 4) == 0 && (H % 4) == 0 && aligned16(h) && aligned16(W_out) && aligned16(b_out)) {
    const int tiles_m = cdiv(M, BM), tiles_n = cdiv(V, TK_BN);
    int ns = num_sms() / tiles_m;
    ns = ns < 1 ? 1 : (ns > tiles_n ? tiles_n : ns);
    const int tps = cdiv(tiles_n, ns);
    ns = cdiv(tiles_n, tps);
    const bool rn = tf32_round_in_tma();
    CUtensorMap ta, tb;
    if (make_map(&ta, h, M, H, H, BK, BM, rn, false) && make_map(&tb, W_out, V, H, H, BK, TK_BN, rn, false)) {
      TKArgs a;
      a.M = M; a.N = V; a.K = H; a.tiles_n = tiles_n; a.tiles_per_slice = tps; a.Mpad = w.Mpad; a.topk = K;
      a.bias = b_out; a.part_ms = part_ms; a.part_cand = part_cand;
      const dim3 grid(ns, tiles_m);
      *slices = ns;
      if (K <= 4) return launch_tk<4>(ta, tb, a, grid, s);
      if (K <= 8) return launch_tk<8>(ta, tb, a, grid, s);
      return launch_tk<16>(ta, tb, a, grid, s);
    }
  }
  float* logits = ws + w.logits;
  GIC_TRY(gemm(mode, false, true, M, V, H, 1.f, h, H, W_out, H, 0.f, logits, V, b_out, s, PROF_GEMM_DECODE));
  *slices = 1;
  if (K <= 4) row_topk_kernel<4><<<M, RT_THREADS, 0, s>>>(logits, V, K, part_ms, part_cand);
  else if (K <= 8) row_topk_kernel<8><<<M, RT_THREADS, 0, s>>>(logits, V, K, part_ms, part_cand);
  else row_topk_kernel<16><<<M, RT_THREADS, 0, s>>>(logits, V, K, part_ms, part_cand);
  return check_launch("row_topk_kernel");
}

int vocab_topk(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K, float* logp,
               int64_t* tokens, float* lse, float* ws, cudaStream_t s) {
  int slices = 1;
  GIC_TRY(vocab_topk_partials(mode, h, W_out, b_out, M, V, H, K, ws, s, &slices));
  const TopkWs w(M, V, K);
  topk_rows_kernel<<<M, TR_THREADS, 0, s>>>(reinterpret_cast<const float2*>(ws + w.ms), reinterpret_cast<const float2*>(ws + w.cand),
                                            slices, w.Mpad, K, V, logp, tokens, lse);
  return check_launch("topk_rows_kernel");
}

// lstm_cell_fwd / lstm_step_tc live in decode.cu / lstm_tcgen05.cu
int lstm_cell_fwd(const float*, const float*, int, int, float*, float*, float*, float*, int, int, cudaStream_t);
int lstm_step_tc(const float*, int, const float*, const float*, const float*, const float*, const float*, const float*,
                 int, int, float*, float*, float*, float*, int, int, cudaStream_t, bool*);

// decode_beam workspace (floats): x[BK,E] | per layer hA, cA, hB, cB [BK,H] | gates[BK,4H] | score[BK] | fin[BK] | len[BK]
// | trace[L,B,K,2] | candidate-producer workspace
struct BeamWs {
  size_t x, state, gates, score, fin, len, trace, topk, total;
  size_t BKH;
  BeamWs(int B, int K, int L, int V, int E, int H, int layers) {
    const size_t BK = (size_t)B * K;
    BKH = a4(BK * H);
    x = 0;
    state = a4(BK * E);
    gates = state + 4 * BKH * layers;
    score = gates + a4(BK * 4 * H);
    fin = score + a4(BK);
    len = fin + a4(BK);
    trace = len + a4(BK);
    topk = trace + a4((size_t)2 * L * BK);
    total = topk + TopkWs((int)BK, V, K).total;
  }
};
size_t decode_beam_ws_floats(int B, int K, int L, int V, int E, int H, int layers) {
  return BeamWs(B, K, L, V, E, H, layers).total;
}

int decode_beam(int mode, const float* features, const float* W_emb, const float* const* W_ih, const float* const* W_hh,
                const float* const* b_ih, const float* const* b_hh, const float* W_out, const float* b_out, int B, int K,
                int L, int V, int E, int H, int layers, int64_t eos, float length_penalty, int64_t* ids, float* scores,
                int32_t* lengths, int32_t* trace, float* ws, cudaStream_t s) {
  const BeamWs w(B, K, L, V, E, H, layers);
  const int BK = B * K;
  BeamState st;
  for (int l = 0; l < BEAM_MAX_LAYERS; ++l) {
    const bool on = l < layers;
    float* base = ws + w.state + 4 * w.BKH * (on ? l : 0);
    st.hA[l] = base; st.cA[l] = base + w.BKH; st.hB[l] = base + 2 * w.BKH; st.cB[l] = base + 3 * w.BKH;
  }
  st.x = ws + w.x;
  st.score = ws + w.score;
  st.fin = reinterpret_cast<int*>(ws + w.fin);
  st.len = reinterpret_cast<int*>(ws + w.len);
  st.trace = trace ? reinterpret_cast<int2*>(trace) : reinterpret_cast<int2*>(ws + w.trace);
  st.embed = W_emb;
  st.layers = layers; st.H = H; st.E = E; st.K = K; st.L = L; st.V = V; st.B = B; st.eos = (int)eos;
  for (int l = 0; l < layers; ++l) {
    cudaMemsetAsync(st.hA[l], 0, (size_t)BK * H * sizeof(float), s);
    cudaMemsetAsync(st.cA[l], 0, (size_t)BK * H * sizeof(float), s);
  }
  beam_init_kernel<<<BK, 128, 0, s>>>(features, st);
  GIC_TRY(check_launch("beam_init_kernel"));
  const TopkWs tw(BK, V, K);
  float* tws = ws + w.topk;
  float* gates = ws + w.gates;
  for (int t = 0; t < L; ++t) {
    for (int l = 0; l < layers; ++l) {
      const float* xin = (l == 0) ? st.x : st.hB[l - 1];
      const int In = (l == 0) ? E : H;
      bool fused = false;
      if (mode == GEMM_TF32 || mode == GEMM_BF16)
        GIC_TRY(lstm_step_tc(xin, In, st.hA[l], W_ih[l], W_hh[l], b_ih[l], b_hh[l], st.cA[l], BK, H, nullptr,
                             const_cast<float*>(st.cB[l]), const_cast<float*>(st.hB[l]), nullptr, L, t, s, &fused));
      if (!fused) {
        GIC_TRY(gemm(mode, false, true, BK, 4 * H, In, 1.f, xin, In, W_ih[l], In, 0.f, gates, 4 * H, b_ih[l], s));
        GIC_TRY(gemm(mode, false, true, BK, 4 * H, H, 1.f, st.hA[l], H, W_hh[l], H, 1.f, gates, 4 * H, b_hh[l], s));
        GIC_TRY(lstm_cell_fwd(gates, st.cA[l], BK, H, nullptr, const_cast<float*>(st.cB[l]), const_cast<float*>(st.hB[l]),
                              nullptr, L, t, s));
      }
    }
    int slices = 1;
    GIC_TRY(vocab_topk_partials(mode, st.hB[layers - 1], W_out, b_out, BK, V, H, K, tws, s, &slices));
    beam_merge_kernel<<<B, BM_THREADS, 0, s>>>(reinterpret_cast<const float2*>(tws + tw.ms),
                                               reinterpret_cast<const float2*>(tws + tw.cand), slices, tw.Mpad, t, st);
    GIC_TRY(check_launch("beam_merge_kernel"));
  }
  beam_finalize_kernel<<<B, 32, 0, s>>>(st, length_penalty, ids, scores, lengths);
  return check_launch("beam_finalize_kernel");
}

}  // namespace gic
