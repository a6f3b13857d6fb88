// One step of the decoder's backward-through-time recurrence as ONE kernel (sm_100a only):
//     dh_rec      = dG_t W_hh                          ([B, 4H] x [4H, H]; autograd of nn.LSTM, src/generator.py:61)
//     dh          = dh_rec + dh_top[:, t-1, :]
//     dG_{t-1}, dc = LSTM cell backward at step t-1    (lstm_cell_bwd_kernel's equations)
// It replaces, per step, a stream-K GEMM whose 8 partial tiles met through red.global.add in L2 (~12 us for 0.5 GFLOP)
// plus the separate cell kernel (~4 us): 19 serial pairs on the generator's critical path at c2.
//
// Split-K over a thread-block cluster: the 4 CTAs of a cluster share one 128-row x 32-column tile of dh_rec and each
// contracts 1 / 4 of K = 4H (TMA ring -> tcgen05.mma kind::tf32 -> TMEM).  The partial tiles meet over distributed
// shared memory: every CTA stages its partial grouped by destination rank, the cluster synchronises, and CTA r adds the
// 4 partials of columns 8r .. 8r+7 in rank order (deterministic) and applies the cell backward to those 8 hidden units
// -- the cell update is elementwise in (row, unit), so no further exchange is needed.
// Measured (ncu, c2): 13.4 us per step against 12.0 + 4.3 us for the stream-K GEMM + cell kernel.
// Clusters of 8 (64 columns) would need 16 co-resident clusters at c2, and a B200 fits 15 (cudaOccupancyMaxActiveClusters):
// the grid ran in two waves, 2.585 ms per training step against 2.503 with clusters of 4.
#include "tcgen05_common.cuh"

namespace gic {
namespace tc {

// BP_CL = cluster size = K splits = column groups of the tile; tile width BP_BN = 8 * BP_CL hidden units (every rank
// finishes 8)
constexpr int BP_CL = 4;
constexpr int BP_BN = 8 * BP_CL;
constexpr int BP_A_BYTES = BM * BK * 4;       // 16 KB: 128 rows x 32 fp32 of dG
constexpr int BP_B_BYTES = BK * BP_BN * 4;    // 32 k-rows x BP_BN columns of W_hh (MN-major, 32-column slabs)
constexpr int BP_STAGES = 8;
constexpr int BP_STAGE = BP_A_BYTES + BP_B_BYTES;
constexpr int BP_SMEM = BP_STAGES * BP_STAGE + 1024 + 256;

__device__ __forceinline__ void bp_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t bp_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ float4 bp_ld_dsmem_f4(uint32_t local_addr, uint32_t rank) {
  uint32_t ra;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(local_addr), "r"(rank));
  float4 v;
  asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ra) : "memory");
  return v;
}

struct BpttArgs {
  int B, H, L, t;                 // this launch produces dG of step t - 1 from dG of step t
  const float* acts;              // [B, 4H] gate activations of step t - 1
  const float* c_prev;            // [B, H]  c_{t-2} (cell state entering step t - 1)
  const float* c_cur;             // [B, H]  c_{t-1}
  const float* dh_top;            // [B, L, H] gradient from the vocab projection; row (b, t - 1) is added
  float* dc_rec;                  // [B, H]  in: dc flowing into step t - 1; out: dc flowing into step t - 2
  float* dG_out;                  // [B, 4H] gate pre-activation gradients of step t - 1
};

__global__ void __launch_bounds__(NTHREADS, 1)
bptt_step_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, BpttArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + BP_STAGES * BP_STAGE);
  uint64_t* empty = full + BP_STAGES;
  uint64_t* tmem_full = empty + BP_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  uint8_t* part = smem;                       // [dest rank 4][chunk 2][row 128][16 B]: aliases the ring after tmem_full

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ks = bp_cluster_rank();      // K split of this CTA = the column group it finishes
  const int tile = blockIdx.x / BP_CL;
  const int tiles_n = a.H / BP_BN;
  const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BP_BN;
  const int nkb = (4 * a.H) / BK / BP_CL;     // k-blocks of this CTA
  const int kb0 = (int)ks * nkb;
  constexpr uint32_t TMEM_COLS = (BP_BN < 32) ? 32 : BP_BN;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int s = 0; s < BP_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % BP_STAGES;
        const uint32_t ph = (i / BP_STAGES) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * BP_STAGE;
        uint8_t* sb = sa + BP_A_BYTES;
        mbar_expect_tx(&full[s], BP_STAGE);
        const int k0 = (kb0 + i) * BK;
        tma_load_2d(sa, &tmA, &full[s], k0, m0);
#pragma unroll
        for (int j = 0; j < BP_BN / 32; ++j) tma_load_2d(sb + j * 4096, &tmB, &full[s], n0 + 32 * j, k0);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(0, 1, BP_BN);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % BP_STAGES;
        const uint32_t ph = (i / BP_STAGES) & 1;
        mbar_wait(&full[s], ph);
        tcgen05_fence_after();
        const uint32_t sa = smem_u32(smem + s * BP_STAGE);
        const uint32_t sb = sa + BP_A_BYTES;
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)
          umma_tf32(tmem_base, make_desc(sa + k * 32, 16, 1024, 2), make_desc(sb + k * 1024, 4096, 512, 1), idesc,
                    (i > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty[s]);
      }
      umma_commit(tmem_full);
    }
  } else {
    // stage this CTA's partial tile, grouped by the rank that will finish each 8-column group
    mbar_wait(tmem_full, 0);
    tcgen05_fence_after();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll
    for (int h = 0; h < BP_BN / 32; ++h) {
      uint32_t r[32];
      tmem_ld32(lane_addr + 32 * h, r);                // columns 32h .. 32h+31 = ranks 4h .. 4h+3
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        uint8_t* dst = part + (size_t)(4 * h + rr) * (2 * BM * 16) + row * 16;
        *reinterpret_cast<float4*>(dst) = make_float4(__uint_as_float(r[8 * rr + 0]), __uint_as_float(r[8 * rr + 1]),
                                                      __uint_as_float(r[8 * rr + 2]), __uint_as_float(r[8 * rr + 3]));
        *reinterpret_cast<float4*>(dst + BM * 16) = make_float4(__uint_as_float(r[8 * rr + 4]), __uint_as_float(r[8 * rr + 5]),
                                                                __uint_as_float(r[8 * rr + 6]), __uint_as_float(r[8 * rr + 7]));
      }
    }
  }
  __syncwarp();
  bp_cluster_sync();                                   // every CTA's partial is in its shared memory

  if (warp >= 2) {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int b = m0 + row;
    const uint32_t my = smem_u32(part + (size_t)ks * (2 * BM * 16) + row * 16);
    float dh[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) dh[e] = 0.f;
#pragma unroll
    for (int src = 0; src < BP_CL; ++src) {            // fixed order: the sum does not depend on scheduling
      const float4 v0 = bp_ld_dsmem_f4(my, (uint32_t)src);
      const float4 v1 = bp_ld_dsmem_f4(my + BM * 16, (uint32_t)src);
      dh[0] += v0.x; dh[1] += v0.y; dh[2] += v0.z; dh[3] += v0.w;
      dh[4] += v1.x; dh[5] += v1.y; dh[6] += v1.z; dh[7] += v1.w;
    }
    if (b < a.B) {
      const int j = n0 + 8 * (int)ks;
      const int H = a.H;
      auto ld8 = [](const float* p, float (&v)[8]) {
        const float4 x = *reinterpret_cast<const float4*>(p), y = *reinterpret_cast<const float4*>(p + 4);
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
      };
      auto st8 = [](float* p, const float (&v)[8]) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
      };
      float gi[8], gf[8], gg[8], go[8], cp[8], cc[8], dt[8], dcr[8];
      const float* ar = a.acts + (size_t)b * 4 * H + j;
      ld8(ar, gi); ld8(ar + H, gf); ld8(ar + 2 * H, gg); ld8(ar + 3 * H, go);
      ld8(a.c_prev + (size_t)b * H + j, cp);
      ld8(a.c_cur + (size_t)b * H + j, cc);
      ld8(a.dh_top + ((size_t)b * a.L + (a.t - 1)) * H + j, dt);
      ld8(a.dc_rec + (size_t)b * H + j, dcr);
      float di[8], df[8], dgg[8], dout[8], dcn[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d = dh[e] + dt[e];
        const float tcv = tanhf(cc[e]);
        const float dc = d * go[e] * (1.f - tcv * tcv) + dcr[e];
        di[e] = dc * gg[e] * gi[e] * (1.f - gi[e]);
        df[e] = dc * cp[e] * gf[e] * (1.f - gf[e]);
        dgg[e] = dc * gi[e] * (1.f - gg[e] * gg[e]);
        dout[e] = d * tcv * go[e] * (1.f - go[e]);
        dcn[e] = dc * gf[e];
      }
      float* gr = a.dG_out + (size_t)b * 4 * H + j;
      st8(gr, di); st8(gr + H, df); st8(gr + 2 * H, dgg); st8(gr + 3 * H, dout);
      st8(a.dc_rec + (size_t)b * H + j, dcn);
    }
  }
  __syncwarp();
  bp_cluster_sync();                                   // peers have read this CTA's partial: its shared memory may go
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}


// ---------------------------------------------------------------------------------------------------------
// The whole recurrence t = L-1 .. 1 as ONE persistent launch.  Per step a kernel of this family spends ~4 us in its
// main loop and ~9 us on being a kernel (launch, barrier / TMEM set-up, first-load latency, tear-down), and the chain is
// serial.  Here the grid stays resident: the CTA's slice of W_hh is loaded into shared memory once, each step streams
// only the dG_t rows through the TMA ring, and the all-to-all dependency between steps (every CTA reads columns of
// dG_{t-1} that other clusters wrote) is a grid-wide arrival counter in global memory: epilogue threads fence their
// stores, one thread per CTA adds 1, the TMA producer polls for (step * CTAs) and crosses into the async proxy before
// it issues the next loads.  dc stays in the registers of the thread that owns the (row, unit) pair.
// Requires every CTA co-resident (checked with cudaOccupancyMaxActiveClusters before the launch).
// ---------------------------------------------------------------------------------------------------------
constexpr int BPP_CL = 4;
constexpr int BPP_BN = 8 * BPP_CL;                 // 32 columns per cluster tile
constexpr int BPP_WBLK = BK * BPP_BN * 4;          // 4 KB: one k-block of the resident W_hh slice
constexpr int BPP_MAX_KB = 16;                     // k-blocks per CTA (H <= 512)
constexpr int BPP_STAGES = 8;
constexpr int BPP_PART = BPP_CL * 2 * BM * 16;     // 16 KB
constexpr int BPP_SMEM = BPP_MAX_KB * BPP_WBLK + BPP_STAGES * BP_A_BYTES + BPP_PART + 1024 + 256;

struct BpttPArgs {
  int B, H, L;
  const float* acts;              // [L][B][4H]
  const float* cs;                // [L+1][B][H]   cs[t] = cell state entering step t
  const float* dh_top;            // [B][L][H]
  const float* dc_in;             // [B][H] dc flowing into step L-2 (written by the cell kernel of step L-1)
  float* dG;                      // [L][B][4H]    dG[L-1] valid on entry; dG[L-2 .. 0] produced here
  unsigned int* counter;          // zero on entry
};

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__global__ void __launch_bounds__(NTHREADS, 1)
bptt_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, BpttPArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* wres = smem;                                        // [nkb][4 KB] resident slice of W_hh
  uint8_t* ring = wres + BPP_MAX_KB * BPP_WBLK;                // [BPP_STAGES][16 KB] dG tiles
  uint8_t* part = ring + BPP_STAGES * BP_A_BYTES;              // [rank 4][chunk 2][row 128][16 B]
  uint64_t* full = reinterpret_cast<uint64_t*>(part + BPP_PART);
  uint64_t* empty = full + BPP_STAGES;
  uint64_t* tmem_full = empty + BPP_STAGES;
  uint64_t* w_full = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ks = bp_cluster_rank();
  const int tile = blockIdx.x / BPP_CL;
  const int tiles_n = a.H / BPP_BN;
  const int m0 = (tile / tiles_n) * BM, n0 = (tile % tiles_n) * BPP_BN;
  const int nkb = (4 * a.H) / BK / BPP_CL;
  const int kb0 = (int)ks * nkb;
  const int nsteps = a.L - 1;
  constexpr uint32_t TMEM_COLS = 32;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int s = 0; s < BPP_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(w_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // one-time: this CTA's slice of W_hh becomes resident
  if (warp == 0 && lane == 0) {
    mbar_expect_tx(w_full, (uint32_t)nkb * BPP_WBLK);
    for (int i = 0; i < nkb; ++i) tma_load_2d(wres + i * BPP_WBLK, &tmB, w_full, n0, (kb0 + i) * BK);
  }
  if (warp == 1 && lane == 0) mbar_wait(w_full, 0);
  uint32_t it = 0;                                       // ring position (producer and MMA threads count alike)

  // ===== per-step epilogue: all threads take part in the two cluster barriers =====
  const int q = warp & 3;
  const int row = q * 32 + lane;
  const int b = m0 + row;
  const bool epi = warp >= 2;
  const bool live = epi && b < a.B;
  const int H = a.H;
  const int j = n0 + 8 * (int)ks;
  const size_t BH = (size_t)a.B * H;
  float dcr[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) dcr[e] = 0.f;
  auto ld8 = [](const float* p, float (&v)[8]) {
    const float4 x = *reinterpret_cast<const float4*>(p), y = *reinterpret_cast<const float4*>(p + 4);
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
  };
  auto st8 = [](float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  };
  if (live) ld8(a.dc_in + (size_t)b * H + j, dcr);
  for (int st = 0; st < nsteps; ++st) {
    const int t = a.L - 1 - st;                          // consumes dG[t], produces dG[t-1]
    if (warp == 0) {
      // ===== TMA producer =====
      if (lane == 0) {
        if (st > 0) {
          // every CTA has published its part of dG[t] (arrival counter), then cross into the async proxy
          const unsigned int want = (unsigned int)st * gridDim.x;
          const long long t0 = clock64();
          while (ld_acquire_u32(a.counter) < want) {
            if (clock64() - t0 > 4000000000ll) trap_report(6u, ((unsigned long long)ld_acquire_u32(a.counter) << 32) | want);   // a protocol bug traps instead of hanging the GPU
          }
          asm volatile("fence.proxy.async;" ::: "memory");
        }
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % BPP_STAGES;
          const uint32_t ph = (it / BPP_STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          mbar_expect_tx(&full[s], BP_A_BYTES);
          tma_load_2d(ring + s * BP_A_BYTES, &tmA, &full[s], (kb0 + i) * BK, t * a.B + m0);
        }
      }
    } else if (warp == 1) {
      // ===== MMA issuer.  The accumulator is overwritten by the next step's first MMA, which cannot be issued before
      //       this CTA's own arrival on the grid counter (after its epilogue has read TMEM): no tmem_empty barrier =====
      if (lane == 0) {
        constexpr uint32_t idesc = make_idesc(0, 1, BPP_BN);
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % BPP_STAGES;
          const uint32_t ph = (it / BPP_STAGES) & 1;
          mbar_wait(&full[s], ph);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(ring + s * BP_A_BYTES);
          const uint32_t sb = smem_u32(wres + i * BPP_WBLK);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_tf32(tmem_base, make_desc(sa + k * 32, 16, 1024, 2), make_desc(sb + k * 1024, 4096, 512, 1), idesc,
                      (i > 0 || k > 0) ? 1u : 0u);
          umma_commit(&empty[s]);
        }
        umma_commit(tmem_full);
      }
    }
    float gi[8], gf[8], gg[8], go[8], cp[8], cc[8], dt[8];
    if (live) {
      // inputs of the cell backward of step t - 1: independent of the contraction, requested before the wait
      const float* ar = a.acts + (size_t)(t - 1) * BH * 4 + (size_t)b * 4 * H + j;
      ld8(ar, gi); ld8(ar + H, gf); ld8(ar + 2 * H, gg); ld8(ar + 3 * H, go);
      ld8(a.cs + (size_t)(t - 1) * BH + (size_t)b * H + j, cp);
      ld8(a.cs + (size_t)t * BH + (size_t)b * H + j, cc);
      ld8(a.dh_top + ((size_t)b * a.L + (t - 1)) * H + j, dt);
#pragma unroll
      for (int e = 0; e < 8; ++e) cc[e] = tanhf(cc[e]);  // off the critical path: the contraction has not finished yet
    }
    if (epi) {
      mbar_wait(tmem_full, (uint32_t)(st & 1));
      tcgen05_fence_after();
      const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
      uint32_t r[32];
      tmem_ld32(lane_addr, r);
      tcgen05_fence_before();
#pragma unroll
      for (int rr = 0; rr < BPP_CL; ++rr) {
        uint8_t* dst = part + (size_t)rr * (2 * BM * 16) + row * 16;
        *reinterpret_cast<float4*>(dst) = make_float4(__uint_as_float(r[8 * rr + 0]), __uint_as_float(r[8 * rr + 1]),
                                                      __uint_as_float(r[8 * rr + 2]), __uint_as_float(r[8 * rr + 3]));
        *reinterpret_cast<float4*>(dst + BM * 16) = make_float4(__uint_as_float(r[8 * rr + 4]), __uint_as_float(r[8 * rr + 5]),
                                                                __uint_as_float(r[8 * rr + 6]), __uint_as_float(r[8 * rr + 7]));
      }
    }
    __syncwarp();
    bp_cluster_sync();                                   // every CTA's partial is in its shared memory
    if (epi) {
      const uint32_t my = smem_u32(part + (size_t)ks * (2 * BM * 16) + row * 16);
      float dh[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) dh[e] = 0.f;
#pragma unroll
      for (int src = 0; src < BPP_CL; ++src) {           // fixed order: the sum does not depend on scheduling
        const float4 v0 = bp_ld_dsmem_f4(my, (uint32_t)src);
        const float4 v1 = bp_ld_dsmem_f4(my + BM * 16, (uint32_t)src);
        dh[0] += v0.x; dh[1] += v0.y; dh[2] += v0.z; dh[3] += v0.w;
        dh[4] += v1.x; dh[5] += v1.y; dh[6] += v1.z; dh[7] += v1.w;
      }
      if (live) {
        float di[8], df[8], dgg[8], dout[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float d = dh[e] + dt[e];
          const float tcv = cc[e];
          const float dc = d * go[e] * (1.f - tcv * tcv) + dcr[e];
          di[e] = dc * gg[e] * gi[e] * (1.f - gi[e]);
          df[e] = dc * cp[e] * gf[e] * (1.f - gf[e]);
          dgg[e] = dc * gi[e] * (1.f - gg[e] * gg[e]);
          dout[e] = d * tcv * go[e] * (1.f - go[e]);
          dcr[e] = dc * gf[e];
        }
        float* gr = a.dG + (size_t)(t - 1) * BH * 4 + (size_t)b * 4 * H + j;
        st8(gr, di); st8(gr + H, df); st8(gr + 2 * H, dgg); st8(gr + 3 * H, dout);
      }
      __threadfence();                                   // this thread's part of dG[t-1] is visible device-wide
      asm volatile("bar.sync 1, 128;" ::: "memory");     // the four epilogue warps
      // One arrival per CTA.  No second cluster barrier: this CTA's `part` is overwritten only after its producer has
      // passed the next grid-wide wait, which needs the arrival of every peer -- issued after the peer's DSMEM reads.
      if (threadIdx.x == 64) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(a.counter) : "memory");
    }
  }
  __syncwarp();
  bp_cluster_sync();                                     // no CTA leaves while a peer may still read its shared memory
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS));
  }
}

}  // namespace tc

// dG_{t-1} (and dc) from dG_t: recurrent contraction + cell backward of step t - 1 in one launch.  handled = false
// (nothing launched) when the shape does not fit; the caller then runs the GEMM and the cell kernel separately.
int bptt_step_tc(const float* dG_t, const float* W_hh, const float* acts_prev, const float* c_prev, const float* c_cur,
                 const float* dh_top, float* dc_rec, float* dG_out, int B, int H, int L, int t, cudaStream_t stream,
                 bool* handled) {
  using namespace tc;
  *handled = false;
  if (option("GIC_BPTT_FUSED", 1) == 0) return GIC_OK;
  if (B <= 0 || t < 1 || (H % BP_BN) || ((4 * H) % (BK * BP_CL))) return GIC_OK;
  const void* ptrs[] = {dG_t, W_hh, acts_prev, c_prev, c_cur, dh_top, dc_rec, dG_out};
  for (const void* p : ptrs)
    if (!aligned16(p)) return GIC_OK;
  const bool rn = tf32_round_in_tma();
  CUtensorMap ta, tb;
  if (!make_map(&ta, dG_t, B, 4 * H, 4 * H, BK, BM, rn, false)) return GIC_OK;
  if (!make_map(&tb, W_hh, 4 * H, H, H, 32, BK, rn, true)) return GIC_OK;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(bptt_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BP_SMEM);
    attr = true;
  }
  BpttArgs a;
  a.B = B; a.H = H; a.L = L; a.t = t; a.acts = acts_prev; a.c_prev = c_prev; a.c_cur = c_cur; a.dh_top = dh_top;
  a.dc_rec = dc_rec; a.dG_out = dG_out;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cdiv(B, BM) * (H / BP_BN) * BP_CL, 1, 1);
  cfg.blockDim = dim3(NTHREADS, 1, 1);
  cfg.dynamicSmemBytes = BP_SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = BP_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, bptt_step_kernel, ta, tb, a);
  if (e != cudaSuccess) { set_error("bptt_step_kernel launch: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  int rc = check_launch("bptt_step_kernel");
  if (rc == GIC_OK) *handled = true;
  return rc;
}

// The whole recurrence in one persistent launch: dG[L-2 .. 0] from dG[L-1] (see bptt_persistent_kernel).  counter: one
// zero-initialised 32-bit word of caller workspace.  handled = false when the shape does not fit or the grid cannot be
// co-resident; the caller then runs the per-step path.
int bptt_persistent_tc(float* dG, const float* W_hh, const float* acts, const float* cs, const float* dh_top, const float* dc_in,
                       unsigned int* counter, int B, int H, int L, cudaStream_t stream, bool* handled) {
  using namespace tc;
  *handled = false;
  if (option("GIC_BPTT_PERSISTENT", 1) == 0) return GIC_OK;
  if (B <= 0 || L < 2 || (H % BPP_BN) || ((4 * H) % (BK * BPP_CL)) || (4 * H) / BK / BPP_CL > BPP_MAX_KB) return GIC_OK;
  const void* ptrs[] = {dG, W_hh, acts, cs, dh_top, dc_in};
  for (const void* p : ptrs)
    if (!aligned16(p)) return GIC_OK;
  const bool rn = tf32_round_in_tma();
  CUtensorMap ta, tb;
  if (!make_map(&ta, dG, L * B, 4 * H, 4 * H, BK, BM, rn, false)) return GIC_OK;
  if (!make_map(&tb, W_hh, 4 * H, H, H, 32, BK, rn, true)) return GIC_OK;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(bptt_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BPP_SMEM);
    attr = true;
  }
  cudaLaunchConfig_t cfg = {};
  const int clusters = cdiv(B, BM) * (H / BPP_BN);
  cfg.gridDim = dim3(clusters * BPP_CL, 1, 1);
  cfg.blockDim = dim3(NTHREADS, 1, 1);
  cfg.dynamicSmemBytes = BPP_SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = BPP_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  static int max_clusters = -1;
  if (max_clusters < 0) {
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, bptt_persistent_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); nc = 0; }
    max_clusters = nc;
  }
  if (clusters > max_clusters) return GIC_OK;        // the grid-wide barrier needs every CTA resident
  BpttPArgs a;
  a.B = B; a.H = H; a.L = L; a.acts = acts; a.cs = cs; a.dh_top = dh_top; a.dc_in = dc_in; a.dG = dG; a.counter = counter;
  cudaError_t e = cudaLaunchKernelEx(&cfg, bptt_persistent_kernel, ta, tb, a);
  if (e != cudaSuccess) { set_error("bptt_persistent_kernel launch: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  int rc = check_launch("bptt_persistent_kernel");
  if (rc == GIC_OK) *handled = true;
  return rc;
}

}  // namespace gic
