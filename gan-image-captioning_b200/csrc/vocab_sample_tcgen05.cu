// Fused vocab projection + Gumbel-softmax + sample for ONE decode step (sm_100a only):
//   logits = h_t W_out^T + b_out                                     (src/generator.py:64,68)
//   z      = (logits - log(-log(u + eps) + eps)) * T                 (add_gumbel, :84-96; :69)
//   p      = softmax(z)          -> written in place to out[b, t, :] (:69-70, no torch.stack copy)
//   tok    = first index of max p -> ids[b, t]; x_{t+1} = embed[tok] (:73-76)
// The logits never leave the chip: every CTA owns one 128 x BN tile of the [B, V] logits, accumulated by tcgen05.mma
// (kind::tf32) in TMEM from a TMA-fed shared-memory ring, while a second TMA stream prefetches the matching tile of
// the uniform draws u_t into 128-byte-swizzled shared memory underneath the main loop.  The row statistics of the
// softmax span all column tiles, so the tiles of one 128-row block exchange their row statistics through global
// memory (L2) and wait for each other there (the whole grid is co-resident: tiles <= SMs, one CTA per SM):
//   pass 1  TMEM -> registers (lane = row), perturb with the Gumbel noise, running max m and sum s of exp(z - m)
//           (online rescaling, one row per thread: no shuffles needed); e = exp(z - m_running) replaces u in shared memory
//   publish (m, s) per row and tile as one 8-byte store whose s != 0 is the ready flag; poll the other tiles' entries
//   combine M = max m_j, S = sum s_j exp(m_j - M), winner tile = first j with m_j == M
//   pass 2  p = e * exp(m_running - M) / S in shared memory, TMA store to out[b, t, n0:n0+BN]; the winner tile finds the
//           first column with p == max p (the reference's first-max tie rule), writes ids and gathers embed[tok]
// HBM traffic per step: read u (4 B V bytes), write p (4 B V bytes); W_out streams from L2.
// Warp roles (576 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..17 = epilogue: four
// warps per TMEM lane quarter split the tile's columns in 16-column units; they turn u into the Gumbel term while the
// main loop runs (pass 0), so only the exp / normalise passes remain after the last MMA.
//
// FUSED DECODE STEP (single-layer decoder; decode_step_tc below).  The LSTM pre-activation of the NEXT step is
//     gates_{t+1} = embed[tok_t] W_ih^T + h_t W_hh^T + b_ih + b_hh              (src/generator.py:61,75-76)
// and only its first term depends on the token this kernel is about to sample.  So the same launch also carries
//   * "rec" tiles (the CTAs with the LOWEST block indices, on the SMs the projection tiles leave idle): plain 128 x RBN
//     tiles of R = h_t W_hh^T, same A operand and pipeline as the projection tiles, accumulator stored to global memory,
//     one arrival per tile on a per-row-block counter;
//   * a cell tail in the projection tiles: the CTA that ends up holding a row's maximum (= knows tok_t) waits for the
//     row block's rec tiles, adds the token's row of EW = embed W_ih^T + b_ih + b_hh (a [V, 4H] table rebuilt once per
//     decode by the caller), applies the LSTM cell and writes h_{t+1}, c_{t+1}, the saved activations and
//     htop -- one warp per row, rows dealt over all 16 epilogue warps.
// One launch per decode step instead of two, and the recurrent contraction runs UNDER the projection instead of after it.
#include "tcgen05_common.cuh"
#include "philox.cuh"

namespace gic {
long long* vs_stamps_buffer();
namespace tc {

template <int BN>
struct VSCfg {
  static constexpr int A_BYTES = BM * BK * 4;          // 16 KB
  static constexpr int B_BYTES = BN * BK * 4;
  static constexpr int STAGE = A_BYTES + B_BYTES;
  static constexpr int NBOX = BN / 32;                 // 32-column boxes of the u / p tile
  static constexpr int BOX_BYTES = BM * 128;           // 128 rows x 128 bytes
  static constexpr int U_BYTES = NBOX * BOX_BYTES;
  static constexpr int BAR_BYTES = 256 + 1024;          // mbarriers + TMEM slot | bias tile (BN floats)
  static constexpr int AVAIL = 227 * 1024 - 1024 - U_BYTES - BAR_BYTES;
  static constexpr int STAGES = (AVAIL / STAGE) > 6 ? 6 : (AVAIL / STAGE);
  static constexpr int TOTAL = STAGES * STAGE + U_BYTES + BAR_BYTES + 1024;
  static constexpr uint32_t TMEM_COLS = 256;           // a rec tile of the fused decode step is up to 256 columns wide
  static_assert(STAGES >= 2, "vocab_sample: shared memory ring too small");
  static_assert(BN % 32 == 0 && BN <= 256, "vocab_sample: BN must be a multiple of 32, <= 256");
};

struct VSArgs {
  int M, N, K, tiles_n, Mpad;
  const float* bias;          // [N]
  float T;
  const float* T_dev;         // temperature read at run time when non-null (CUDA-graph replay)
  float2* part;               // [tiles_n][Mpad] (m, s) per row and column tile of THIS step; s != 0 doubles as the ready flag
  float2* part_next;          // the other buffer: every CTA clears its own entries for the next step
  int64_t* ids;               // [M, L]
  const int64_t* forced;      // [M, L] or null: token fed to the next step instead of the sampled one
  int L, t;
  const float* embed;         // [V, E]
  int E;
  float* x_next;              // [M, E] or null
  long long* stamps;          // debug (GIC_VS_STAMPS=1): 16 clock64 stamps per CTA, else null
  int use_rng;                // no uniforms supplied: draw u[t, m, n] in the kernel (Philox, same numbers as gic_philox_uniform)
  RngState rng;
  int2* tokpub;               // [Mpad] (token fed back, step tag t + 1) per row: one 8-byte store, polled by the row's assigned tile
  // ---- fused decode step (all zero / null for the plain projection + sample kernel) ----
  int n_rec;                  // CTAs [0, n_rec) are rec tiles; projection tile index = blockIdx.x - n_rec
  int rec_tiles_n, RBN;       // rec column tiles per row block, their width (multiple of 16, <= 256)
  int G4;                     // 4 H
  float* R;                   // [M, 4H] h_t W_hh^T
  unsigned int* rec_done;     // [tiles_m] arrivals of rec tiles (monotonic over the steps of one decode)
  unsigned int rec_expect;    // value rec_done[mtile] has reached when this launch's rec tiles of the row block are done
  int do_cell;                // apply the LSTM cell of step t + 1 for the rows whose token this CTA feeds back
  const float* EW;            // [V, 4H] embed W_ih^T + b_ih + b_hh
  const float* c_prev;        // [M, H] c_t
  float* c_out;               // [M, H] c_{t+1}
  float* h_out;               // [M, H] h_{t+1}
  float* acts;                // [M, 4H] sig(i), sig(f), tanh(g), sig(o) of step t + 1 (saved for the backward)
  float* htop;                // [M, L, H]: row (m, t + 1) written
};

template <int BN>
struct RecCfg {               // operand ring of a rec tile: it has no u / p tile, so the whole carve-out is ring
  static constexpr int STAGE = BM * BK * 4 + 256 * BK * 4;     // A 16 KB + up to 256 rows of W_hh
  static constexpr int STAGES = ((VSCfg<BN>::STAGES * VSCfg<BN>::STAGE + VSCfg<BN>::U_BYTES) / STAGE) > 4
                                    ? 4 : ((VSCfg<BN>::STAGES * VSCfg<BN>::STAGE + VSCfg<BN>::U_BYTES) / STAGE);
  static_assert(STAGES >= 2, "decode step: rec ring too small");
};
constexpr int VS_NBAR = 8;    // mbarrier slots per direction (>= the stages of either ring)

#define VS_STAMP(i) do { if (a.stamps) a.stamps[blockIdx.x * 32 + (i)] = (long long)globaltimer_ns(); } while (0)

__device__ __forceinline__ float2 ld_relaxed_f2(const float2* p) {
  float2 v;
  asm volatile("ld.relaxed.gpu.global.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_f2(float2* p, float2 v) {
  asm volatile("st.relaxed.gpu.global.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

constexpr int VS_G = 4;                              // epilogue warps per TMEM lane quarter (they split the tile's columns)
constexpr int VS_EPI_THREADS = 128 * VS_G;
constexpr int VS_THREADS = 64 + VS_EPI_THREADS;      // warp 0 = TMA producer, warp 1 = MMA issuer, 16 epilogue warps

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(VS_EPI_THREADS) : "memory"); }

// LSTM cell of step t + 1 (fused decode step) and the next-step input x_{t+1} = embed[fed], for the rows a projection
// tile is ASSIGNED: row r of a row block belongs to column tile r mod tiles_n, whatever tile sampled its token.  (Letting
// the tile that holds a row's maximum do the row's cell was the first design; the sampled tokens of a trained -- or
// collapsing -- generator concentrate on a few vocabulary entries, one tile then wins most of the 128 rows and its tail
// serialises: the step slowed from 2.4 to 3.1 ms over 400 training steps.)  The sampling tile publishes (token, step tag) as
// one 8-byte store to tokpub[row]; the assigned tile polls that entry -- the same self-flagging idiom as the row statistics.
// A team of four warps per row, four rows at a time; every lane issues all loads of its four hidden units at once as 16-byte
// loads -- the token's row of EW (biases folded in), c_t, R -- so a row costs ONE round trip to L2 / HBM.  (Thread-per-unit
// with 4-byte loads was measured slower: four times the load instructions.)  Activations use the MUFU forms (ex2 + rcp;
// |error| ~3e-7, far below the TF32 rounding of the pre-activations).
// The FIRST round (one row per team, units 0..511) is inlined into the kernel's epilogue, where its loads are issued BEFORE
// the normalisation pass and the p tile's TMA stores and consumed after them.  The out-of-line function is the remainder:
// further rounds (tiles_n < 32), hidden units beyond 512, x_{t+1} when it did not ride along, and the whole job for the plain
// projection + sample kernel (x_{t+1} only).
struct CellTailArgs {       // by value: a reference to the kernel's parameter block would force a local-memory copy of it
  const float* embed; float* x_next; const float* R; const float* EW; const float* c_prev;
  float* c_out; float* h_out; float* acts; float* htop;
  int E, G4, L, t, do_cell;
  const int2* tokpub; int ntile, tiles_n, M;
};
__device__ __forceinline__ void st_relaxed_i2(int2* p, int2 v) {
  asm volatile("st.relaxed.gpu.global.v2.s32 [%0], {%1, %2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
// the token fed back for global row m at step tag - 1, once its sampling tile has published it (bounded wait)
__device__ __forceinline__ int wait_token(const int2* tokpub, int m, int tag, int lane) {
  int tok = 0;
  if (lane == 0) {
    const unsigned long long t0 = globaltimer_ns();
    for (;;) {
      int2 v;
      asm volatile("ld.relaxed.gpu.global.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(tokpub + m) : "memory");
      if (v.y == tag) { tok = v.x; break; }
      __nanosleep(20);
      if (globaltimer_ns() - t0 > 4000000000ull) tc::trap_report(2u, ((unsigned long long)(unsigned)m << 32) | (unsigned)tag);   // a protocol bug traps instead of hanging the GPU
    }
  }
  return __shfl_sync(0xffffffffu, tok, 0);
}
__device__ __forceinline__ float sigmoid_mufu(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float tanh_mufu(float x) { return 2.f * __fdividef(1.f, 1.f + __expf(-2.f * x)) - 1.f; }

// four hidden units (j .. j+3) of one row: pre-activations = EW row + R row, cell, stores
__device__ __forceinline__ void lstm_cell_store4(const CellTailArgs& a, int H, int mr, int j, const float4 (&ev)[4], const float4 (&rv)[4],
                                                 float4 cp) {
  float ai[4], af[4], ag[4], ao[4], cn[4], hn[4];
  const float pi[4] = {ev[0].x + rv[0].x, ev[0].y + rv[0].y, ev[0].z + rv[0].z, ev[0].w + rv[0].w};
  const float pf[4] = {ev[1].x + rv[1].x, ev[1].y + rv[1].y, ev[1].z + rv[1].z, ev[1].w + rv[1].w};
  const float pg[4] = {ev[2].x + rv[2].x, ev[2].y + rv[2].y, ev[2].z + rv[2].z, ev[2].w + rv[2].w};
  const float po[4] = {ev[3].x + rv[3].x, ev[3].y + rv[3].y, ev[3].z + rv[3].z, ev[3].w + rv[3].w};
  const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    ai[e] = sigmoid_mufu(pi[e]); af[e] = sigmoid_mufu(pf[e]); ag[e] = tanh_mufu(pg[e]); ao[e] = sigmoid_mufu(po[e]);
    cn[e] = af[e] * cpv[e] + ai[e] * ag[e];
    hn[e] = ao[e] * tanh_mufu(cn[e]);
  }
  float* arow = a.acts + (size_t)mr * a.G4 + j;
  *reinterpret_cast<float4*>(arow) = make_float4(ai[0], ai[1], ai[2], ai[3]);
  *reinterpret_cast<float4*>(arow + H) = make_float4(af[0], af[1], af[2], af[3]);
  *reinterpret_cast<float4*>(arow + 2 * H) = make_float4(ag[0], ag[1], ag[2], ag[3]);
  *reinterpret_cast<float4*>(arow + 3 * H) = make_float4(ao[0], ao[1], ao[2], ao[3]);
  *reinterpret_cast<float4*>(a.c_out + (size_t)mr * H + j) = make_float4(cn[0], cn[1], cn[2], cn[3]);
  const float4 h4 = make_float4(hn[0], hn[1], hn[2], hn[3]);
  *reinterpret_cast<float4*>(a.h_out + (size_t)mr * H + j) = h4;
  *reinterpret_cast<float4*>(a.htop + ((size_t)mr * a.L + (a.t + 1)) * H + j) = h4;
}

// Remainder of the cell (see the comment above CellTailArgs).  Team k of four warps takes the assigned rows
// ntile + (k + 4 j) tiles_n, j = 0, 1, ...; lane tl of the team owns the hidden units 4 tl .. 4 tl + 3 (+ 512 per further pass
// over H).  first_done: the epilogue already handled round j = 0 for the units [0, 512) and, if x_first_done, its x.
__device__ __noinline__ void decode_cell_tail(const CellTailArgs a, int etid, int m0, bool first_done, bool x_first_done) {
  const int team = etid >> 7, tl = etid & 127, lane = etid & 31;
  const int H = a.G4 >> 2;
  const bool vec = ((a.E & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.embed) & 15u) == 0) &&
                   ((reinterpret_cast<uintptr_t>(a.x_next) & 15u) == 0);
  for (int round = 0, r = a.ntile + team * a.tiles_n; r < BM && m0 + r < a.M; ++round, r += VS_G * a.tiles_n) {
    const bool cell_round = a.do_cell && !(first_done && round == 0 && H <= 4 * 128);     // uniform over the CTA
    const bool x_todo = a.x_next != nullptr && !(x_first_done && round == 0);
    if (!cell_round && !x_todo) continue;
    const int mr = m0 + r;
    const int tok = wait_token(a.tokpub, mr, a.t + 1, lane);
    if (cell_round) {
      const float* Er = a.EW + (size_t)tok * a.G4;
      const float* Rr = a.R + (size_t)mr * a.G4;
      for (int j = 4 * tl + ((first_done && round == 0) ? 4 * 128 : 0); j < H; j += 4 * 128) {
        float4 ev[4], rv[4];
#pragma unroll
        for (int gt = 0; gt < 4; ++gt) {
          ev[gt] = __ldcg(reinterpret_cast<const float4*>(Er + gt * H + j));
          rv[gt] = __ldcg(reinterpret_cast<const float4*>(Rr + gt * H + j));
        }
        const float4 cp = __ldcg(reinterpret_cast<const float4*>(a.c_prev + (size_t)mr * H + j));
        lstm_cell_store4(a, H, mr, j, ev, rv, cp);
      }
    }
    if (x_todo) {
      const float* er = a.embed + (size_t)tok * a.E;
      float* xr = a.x_next + (size_t)mr * a.E;
      if (vec) { for (int c = tl; c < (a.E >> 2); c += 128) reinterpret_cast<float4*>(xr)[c] = __ldcg(reinterpret_cast<const float4*>(er) + c); }
      else { for (int c = tl; c < a.E; c += 128) xr[c] = __ldg(er + c); }
    }
  }
}

template <int BN>
__global__ void __launch_bounds__(VS_THREADS, 1)
vocab_sample_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmU, const __grid_constant__ CUtensorMap tmP,
                    const __grid_constant__ CUtensorMap tmW, VSArgs a) {
  using S = VSCfg<BN>;
  constexpr int NUNIT = BN / 16;                     // 16-column units, dealt round-robin to the VS_G warps of a quarter
  constexpr int MAXU = (NUNIT + VS_G - 1) / VS_G;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* ubox = smem + S::STAGES * S::STAGE;                    // NBOX boxes of [128 rows][128 B], 128B-swizzled
  uint64_t* full = reinterpret_cast<uint64_t*>(ubox + S::U_BYTES);
  uint64_t* empty = full + VS_NBAR;
  uint64_t* tmem_full = empty + VS_NBAR;
  uint64_t* u_full = tmem_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(u_full + 1);
  // small exchange buffers of the epilogue live in stage 0 of the operand ring, which is dead once tmem_full fires
  float2 (*s_part)[BM] = reinterpret_cast<float2 (*)[BM]>(smem);              // [VS_G][BM] row statistics of pass 1
  float4* s_row = reinterpret_cast<float4*>(smem + VS_G * BM * 8);            // [VS_G][BM] (M, S, first tile, -) per group
  int* s_hit = reinterpret_cast<int*>(smem + VS_G * BM * 8 + VS_G * BM * 16); // first column holding the row maximum
  static_assert(VS_G * BM * 8 + VS_G * BM * 16 + 3 * BM * 4 + 16 <= 16384, "vocab_sample: exchange buffers exceed 16 KB");
  static_assert(16384 + ((BN / 16 + VS_G - 1) / VS_G) * VS_EPI_THREADS * 4 <= S::STAGE, "vocab_sample: per-unit running maxima exceed stage 0");
  // "this row block's rec tiles have arrived": set by the producer thread (idle once its loads are issued), read by the
  // cell tail; lives next to the mbarriers because the operand ring is still in use when it may be set
  uint32_t* s_recflag = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(full) + 192);
  static_assert(S::STAGES <= VS_NBAR && RecCfg<BN>::STAGES <= VS_NBAR, "vocab_sample: mbarrier slots");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = (a.K + BK - 1) / BK;
  const bool is_rec = (int)blockIdx.x < a.n_rec;
  const int vb = (int)blockIdx.x - a.n_rec;                       // projection tile index
  const int mtile = is_rec ? (int)blockIdx.x / a.rec_tiles_n : vb / a.tiles_n;
  const int ntile = is_rec ? (int)blockIdx.x % a.rec_tiles_n : vb % a.tiles_n;
  const int m0 = mtile * BM, n0 = ntile * (is_rec ? a.RBN : BN);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmU) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmP) : "memory");
    if (a.n_rec) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
    for (int s = 0; s < VS_NBAR; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tmem_full, 1);
    mbar_init(u_full, 1);
    *s_recflag = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(S::TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                      // the LSTM step that produced h_t has completed; the set-up above overlapped its tail
  pdl_trigger();

  if (is_rec) {
    // ===== rec tile: R[m0 : m0+128, n0 : n0+RBN] = h_t W_hh^T (K = H), accumulator straight to global memory =====
    using RC = RecCfg<BN>;
    const uint32_t b_bytes = (uint32_t)a.RBN * BK * 4;
    if (warp == 0) {
      if (lane == 0) {
        VS_STAMP(0);
        for (int kb = 0; kb < nkb; ++kb) {
          const int s = kb % RC::STAGES;
          const uint32_t ph = (kb / RC::STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          uint8_t* sa = smem + s * RC::STAGE;
          mbar_expect_tx(&full[s], S::A_BYTES + b_bytes);
          tma_load_2d(sa, &tmA, &full[s], kb * BK, m0);
          tma_load_2d(sa + S::A_BYTES, &tmW, &full[s], kb * BK, n0);      // RBN rows of W_hh
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        const uint32_t idesc = make_idesc(0, 0, a.RBN);
        for (int kb = 0; kb < nkb; ++kb) {
          const int s = kb % RC::STAGES;
          const uint32_t ph = (kb / RC::STAGES) & 1;
          mbar_wait(&full[s], ph);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + s * RC::STAGE);
          const uint32_t sb = sa + S::A_BYTES;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint64_t da = make_desc(sa + k * 32, 16, 1024, 2);
            const uint64_t db = make_desc(sb + k * 32, 16, 1024, 2);
            umma_tf32(tmem_base, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty[s]);
        }
        umma_commit(tmem_full);
        VS_STAMP(3);
      }
    } else {
      const int q = warp & 3, g = (warp - 2) >> 2;
      const int m = m0 + q * 32 + lane;
      mbar_wait(tmem_full, 0);
      tcgen05_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16);
      const int nunit = a.RBN >> 4;
      for (int j = g; j < nunit; j += VS_G) {                     // warp-uniform
        uint32_t r[16];
        tmem_ld16(t_addr + 16 * j, r);
        const int n = n0 + 16 * j;
        if (m < a.M && n < a.G4) {                                // 4H % 16 == 0: a unit is entirely inside or outside
          float4* dst = reinterpret_cast<float4*>(a.R + (size_t)m * a.G4 + n);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            dst[k] = make_float4(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1]), __uint_as_float(r[4 * k + 2]),
                                 __uint_as_float(r[4 * k + 3]));
        }
      }
      __threadfence();                                            // this thread's slice of R before the arrival below
      epi_bar();
      if (threadIdx.x == 64) { atomicAdd(a.rec_done + mtile, 1u); VS_STAMP(12); }   // one arrival per rec tile (release: fence + barrier above)
    }
  } else
  if (warp == 0) {
    // ===== TMA producer: operand ring; the u tile is queued once the ring is primed (the epilogue warps turn it into
    //       Gumbel noise underneath the rest of the main loop) =====
    if (lane == 0) {
      VS_STAMP(0);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % S::STAGES;
        const uint32_t ph = (kb / S::STAGES) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        uint8_t* sa = smem + s * S::STAGE;
        mbar_expect_tx(&full[s], S::STAGE);
        tma_load_2d(sa, &tmA, &full[s], kb * BK, m0);
        tma_load_2d(sa + S::A_BYTES, &tmB, &full[s], kb * BK, n0);
        if (!a.use_rng && kb == min(nkb, S::STAGES) - 1) {   // ring primed: now the u tile (comes from HBM)
          mbar_expect_tx(u_full, S::U_BYTES);
#pragma unroll
          for (int c = 0; c < S::NBOX; ++c) tma_load_2d(ubox + c * S::BOX_BYTES, &tmU, u_full, n0 + 32 * c, m0);
        }
      }
      VS_STAMP(1);
      if (a.do_cell) {
        // the row block's rec tiles (lower block indices: scheduled before this CTA) have stored R and arrived; polled
        // here, off the epilogue's critical path, and handed over through shared memory
        const unsigned long long t0 = globaltimer_ns();
        for (;;) {
          unsigned int v;
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(a.rec_done + mtile) : "memory");
          if (v >= a.rec_expect) break;
          __nanosleep(100);
          if (globaltimer_ns() - t0 > 4000000000ull) trap_report(3u, ((unsigned long long)v << 32) | a.rec_expect);   // a protocol bug traps instead of hanging the GPU
        }
        asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(smem_u32(s_recflag)), "r"(1u) : "memory");
        VS_STAMP(13);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(0, 0, BN);
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % S::STAGES;
        const uint32_t ph = (kb / S::STAGES) & 1;
        mbar_wait(&full[s], ph);
        if (kb == 0) VS_STAMP(2);
        tcgen05_fence_after();
        const uint32_t sa = smem_u32(smem + s * S::STAGE);
        const uint32_t sb = sa + S::A_BYTES;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint64_t da = make_desc(sa + k * 32, 16, 1024, 2);
          const uint64_t db = make_desc(sb + k * 32, 16, 1024, 2);
          umma_tf32(tmem_base, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&empty[s]);
      }
      umma_commit(tmem_full);
      VS_STAMP(3);
    }
  } else {
    // ===== epilogue warps: thread = (row, column group g); unit = 16 columns =====
    const int q = warp & 3;                          // TMEM lane quarter this warp may access
    const int g = (warp - 2) >> 2;                   // column group 0..VS_G-1
    const int row = q * 32 + lane;                   // row inside the tile
    const int m = m0 + row;
    const int etid = threadIdx.x - 64;
    const float T = a.T_dev ? __ldg(a.T_dev) : a.T;
    const float eps = 1e-10f;
    uint8_t* urow = ubox + row * 128;
    const int sw = row & 7;
    // unit j (16 columns) = box j/2, 16-byte chunks 4*(j&1) .. 4*(j&1)+3
#define VS_CHUNK(j, k) (urow + ((j) >> 1) * S::BOX_BYTES + (((4 * ((j) & 1) + (k)) ^ sw) << 4))

    // ---- housekeeping under the main loop: clear this CTA's entries of the other statistics buffer (read again in
    //      the step after next), stage the bias tile in shared memory
    float* s_bias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + 256);
    if (g == VS_G - 1) st_relaxed_f2(a.part_next + (size_t)ntile * a.Mpad + m, make_float2(0.f, 0.f));
    if (etid < BN / 4) {
      const int n = n0 + 4 * etid;
      reinterpret_cast<float4*>(s_bias)[etid] = (n < a.N) ? __ldg(reinterpret_cast<const float4*>(a.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // ---- pass 0 (under the main loop): u -> log2(-log(u + eps) + eps), the Gumbel term subtracted from the logits
    unsigned long long rseed = 0ull, roff = 0ull;
    if (a.use_rng) rng_load(a.rng, rseed, roff); else mbar_wait(u_full, 0);
    if (etid == 0) VS_STAMP(4);
    // (the unit loops of the three passes are deliberately NOT unrolled: fully unrolled this kernel was 107 KB of SASS, every
    //  pass straight-line code that a warp executes once per launch, and ncu showed an instruction-cache hit rate of 66 %
    //  with "no instruction" the second largest stall reason -- the epilogue was fetch-bound, not math-bound)
#pragma unroll 1
    for (int i = 0; i < MAXU; ++i) {
      const int j = g + i * VS_G;
      if (j < NUNIT && n0 + 16 * j < a.N) {
#pragma unroll 1
        for (int k = 0; k < 4; ++k) {
          float4* sp = reinterpret_cast<float4*>(VS_CHUNK(j, k));
          float4 u4;
          if (a.use_rng) {
            // element (t, m, n) of the logical u[L, M, N]; a float4 chunk is one Philox group (N % 4 == 0)
            const int n = n0 + 16 * j + 4 * k;
            const unsigned long long e = ((unsigned long long)a.t * a.M + (unsigned long long)min(m, a.M - 1)) * a.N + min(n, a.N - 4);
            u4 = philox_uniform4(rseed, roff, RNG_TAG_GUMBEL, e >> 2);
          } else {
            u4 = *sp;
          }
          // log2 of the inner term: the ln 2 factor is applied in pass 1 inside the same fused multiply-subtract the
          // separate sampler kernel compiles to (logit - lg2 * ln2), so both paths round identically
          u4.x = __log2f(-logf(u4.x + eps) + eps); u4.y = __log2f(-logf(u4.y + eps) + eps);
          u4.z = __log2f(-logf(u4.z + eps) + eps); u4.w = __log2f(-logf(u4.w + eps) + eps);
          *sp = u4;
        }
      }
    }

    // ---- pass 1: z = (acc + b - noise) * T, online (max, sum); e = exp(z - running max) replaces the noise
    if (etid == 0) VS_STAMP(5);
    epi_bar();                                         // bias tile visible to all epilogue warps
    mbar_wait(tmem_full, 0);
    if (etid == 0) VS_STAMP(6);
    tcgen05_fence_after();
    const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    float m_run = -INFINITY, s_run = 0.f;
    float* s_mrun = reinterpret_cast<float*>(smem + 16384) + etid;    // [MAXU][VS_EPI_THREADS]: running max after each of this thread's units
#pragma unroll 1
    for (int i = 0; i < MAXU; ++i) {
      const int j = g + i * VS_G;
      if (j < NUNIT) {                                 // warp-uniform
        uint32_t r[16];
        tmem_ld16(t_addr + 16 * j, r);
        float z[16];
        float cm = -INFINITY;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int n = n0 + 16 * j + 4 * k;
          if (n < a.N) {                               // N % 4 == 0: a float4 is entirely inside or outside
            const float4 ng = *reinterpret_cast<const float4*>(VS_CHUNK(j, k));
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 16 * j + 4 * k);
            constexpr float LN2 = 0.693147182f;
            z[4 * k + 0] = (__uint_as_float(r[4 * k + 0]) + b4.x - ng.x * LN2) * T;
            z[4 * k + 1] = (__uint_as_float(r[4 * k + 1]) + b4.y - ng.y * LN2) * T;
            z[4 * k + 2] = (__uint_as_float(r[4 * k + 2]) + b4.z - ng.z * LN2) * T;
            z[4 * k + 3] = (__uint_as_float(r[4 * k + 3]) + b4.w - ng.w * LN2) * T;
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
          for (int e = 0; e < 16; ++e) { z[e] = __expf(z[e] - m_new); cs += z[e]; }
          s_run += cs;
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) z[e] = 0.f;
        }
        s_mrun[i * VS_EPI_THREADS] = m_run;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          *reinterpret_cast<float4*>(VS_CHUNK(j, k)) = make_float4(z[4 * k + 0], z[4 * k + 1], z[4 * k + 2], z[4 * k + 3]);
      }
    }
    s_part[g][row] = make_float2(m_run, s_run);
    if (g == 0) s_hit[row] = 0x7fffffff;
    if (etid == 0) VS_STAMP(7);
    epi_bar();

    // ---- the tile's row statistics (column groups combined in group order), published for the other column tiles.
    //      (m, s) is ONE 8-byte relaxed store and s != 0 is its own ready flag (the buffer was cleared two steps ago),
    //      so no counter, fence or second round trip is needed: consumers poll the data itself.
    if (g == 0) {
      float Mt = -INFINITY, St = 0.f;
#pragma unroll
      for (int i = 0; i < VS_G; ++i) {
        const float2 v = s_part[i][row];
        if (v.x > Mt) { St = St * ((Mt > -INFINITY) ? __expf(Mt - v.x) : 0.f) + v.y; Mt = v.x; }
        else if (v.x > -INFINITY) St += v.y * __expf(v.x - Mt);
      }
      if (St == 0.f) St = 1e-37f;                      // keep the flag set for a degenerate (all -inf) row
      st_relaxed_f2(a.part + (size_t)ntile * a.Mpad + m, make_float2(Mt, St));
      if (etid == 0) VS_STAMP(8);
    }

    // ---- combine over the column tiles: M, S, winner tile (first tile holding the row maximum).  The four column
    //      groups of a row each take every fourth tile, polled in batches of 8 (all loads of a batch in flight: the
    //      partials live in L2 and a dependent chain of ~tiles_n round trips would cost more than the main loop);
    //      the four partial results then meet in shared memory and every thread folds them in group order.
    {
      float Mg = -INFINITY, Sg = 0.f;
      int jb = 0x7fffffff;
      const float2* pp = a.part + m;
      const unsigned long long t0 = globaltimer_ns();
      for (int j0 = g; j0 < a.tiles_n; j0 += 8 * VS_G) {
        float2 v[8];
        for (;;) {
          bool ready = true;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int j = j0 + i * VS_G;
            v[i] = (j < a.tiles_n) ? ld_relaxed_f2(pp + (size_t)j * a.Mpad) : make_float2(-INFINITY, 1.f);
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) ready = ready && (__float_as_uint(v[i].y) != 0u);
          if (ready) break;
          __nanosleep(20);
          if (globaltimer_ns() - t0 > 4000000000ull) trap_report(4u, ((unsigned long long)(unsigned)a.t << 32) | (unsigned)j0);   // a protocol bug traps instead of hanging the GPU
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (j0 + i * VS_G >= a.tiles_n) continue;
          if (v[i].x > Mg) {
            Sg = Sg * ((Mg > -INFINITY) ? __expf(Mg - v[i].x) : 0.f) + v[i].y;
            Mg = v[i].x; jb = j0 + i * VS_G;
          } else if (v[i].x > -INFINITY) {
            Sg += v[i].y * __expf(v[i].x - Mg);
          }
        }
      }
      if (etid == 0) VS_STAMP(9);
      s_row[g * BM + row] = make_float4(Mg, Sg, __int_as_float(jb), 0.f);
    }
    epi_bar();
    float M = -INFINITY, Ssum = 0.f;
    int jbest = 0x7fffffff;
#pragma unroll
    for (int i = 0; i < VS_G; ++i) {
      const float4 v = s_row[i * BM + row];
      const int jv = __float_as_int(v.z);
      if (v.x > M) {
        Ssum = Ssum * ((M > -INFINITY) ? __expf(M - v.x) : 0.f) + v.y;
        M = v.x; jbest = jv;
      } else if (v.x > -INFINITY) {
        Ssum += v.y * __expf(v.x - M);
        if (v.x == M && jv < jbest) jbest = jv;
      }
    }
    if (jbest == 0x7fffffff) jbest = 0;
    const float inv = 1.0f / Ssum;
    const bool winner = (jbest == ntile);
    if (etid == 0) VS_STAMP(10);

    // ---- first-max column of the rows this tile won, BEFORE the normalisation pass: the token -- and with it the gather
    //      loads of the cell below -- is known one pass earlier.  e == 1 marks a column that equals the running maximum of
    //      its unit; the first such column of the first unit whose running maximum is the row maximum M is the first maximum.
    if (winner) {
      int hit = 0x7fffffff;
#pragma unroll 1
      for (int i = 0; i < MAXU && hit == 0x7fffffff; ++i) {
        const int j = g + i * VS_G;
        if (j < NUNIT && n0 + 16 * j < a.N && s_mrun[i * VS_EPI_THREADS] == M) {
#pragma unroll 1
          for (int k = 0; k < 4 && hit == 0x7fffffff; ++k) {
            const float4 e = *reinterpret_cast<const float4*>(VS_CHUNK(j, k));
            if (e.x == 1.0f) hit = 16 * j + 4 * k;
            else if (e.y == 1.0f) hit = 16 * j + 4 * k + 1;
            else if (e.z == 1.0f) hit = 16 * j + 4 * k + 2;
            else if (e.w == 1.0f) hit = 16 * j + 4 * k + 3;
          }
        }
      }
      if (hit != 0x7fffffff) atomicMin(&s_hit[row], hit);
    }
    epi_bar();

    // ---- token id; (token, step tag) published for the tile the row is assigned to (decode_cell_tail's comment)
    if (g == 0) {
      int fed = -1;
      const bool m_ok = m < a.M;
      if (winner && m_ok) {
        const int h = s_hit[row];
        int tok = n0 + (h == 0x7fffffff ? 0 : h);
        if (tok >= a.N) tok = a.N - 1;
        a.ids[(size_t)m * a.L + a.t] = tok;
        fed = tok;
      }
      if (a.forced != nullptr) {
        fed = -1;
        if (ntile == 0 && m_ok) {
          const int64_t fz = a.forced[(size_t)m * a.L + a.t];
          fed = (fz >= 0 && fz < a.N) ? (int)fz : 0;
        }
      }
      if (fed >= 0 && a.tokpub != nullptr) st_relaxed_i2(a.tokpub + m, make_int2(fed, a.t + 1));
    }
    if (etid == 0) VS_STAMP(11);

    // ---- fused decode step, first pass of the cell (decode_cell_tail's comment): issue every load of up to four fed-back
    //      rows now -- thread = hidden unit; x_{t+1} rides along, one float4 per thread and row
    CellTailArgs ct;
    ct.embed = a.embed; ct.x_next = a.x_next; ct.R = a.R; ct.EW = a.EW; ct.c_prev = a.c_prev; ct.c_out = a.c_out;
    ct.h_out = a.h_out; ct.acts = a.acts; ct.htop = a.htop; ct.E = a.E; ct.G4 = a.G4; ct.L = a.L; ct.t = a.t; ct.do_cell = a.do_cell;
    ct.tokpub = a.tokpub; ct.ntile = ntile; ct.tiles_n = a.tiles_n; ct.M = a.M;
    const int Hh = a.G4 >> 2;
    const int team = etid >> 7, tl = etid & 127;          // team of four warps per assigned row; lane tl owns units 4 tl .. 4 tl + 3
    const int r1 = ntile + team * a.tiles_n;              // this team's row of round 0
    const bool row_first = r1 < BM && m0 + r1 < a.M;
    const bool cell_first = a.do_cell && row_first;
    const bool has_u = cell_first && 4 * tl < Hh;
    const bool x_first = a.do_cell && a.x_next != nullptr && ((a.E & 3) == 0) && (a.E >> 2) <= 128 &&
                         ((reinterpret_cast<uintptr_t>(a.embed) & 15u) == 0) && ((reinterpret_cast<uintptr_t>(a.x_next) & 15u) == 0);
    const bool has_x = x_first && row_first && tl < (a.E >> 2);
    int mr1 = 0;
    float4 ev[4], rv[4], cp4 = make_float4(0.f, 0.f, 0.f, 0.f), xv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cell_first) {
      mr1 = m0 + r1;
      const int tok1 = wait_token(a.tokpub, mr1, a.t + 1, lane);
      // ld.global.cg (L2 only): the shared-memory carve-out leaves L1 ~29 KB, a row is 20 KB of gathers (EW 8, R 8, c 2, x 2)
      if (has_u) {
        const float* Er = a.EW + (size_t)tok1 * a.G4 + 4 * tl;
#pragma unroll
        for (int gt = 0; gt < 4; ++gt) ev[gt] = __ldcg(reinterpret_cast<const float4*>(Er + gt * Hh));
        cp4 = __ldcg(reinterpret_cast<const float4*>(a.c_prev + (size_t)mr1 * Hh + 4 * tl));
      }
      if (has_x) xv = __ldcg(reinterpret_cast<const float4*>(a.embed + (size_t)tok1 * a.E) + tl);
      if (has_u) {
        // the row block's rec tiles have stored R and arrived (polled by the producer thread, handed over in shared memory)
        const unsigned am = __activemask();
        if (lane == 0) {
          uint32_t f = 0;
          const unsigned long long t0 = globaltimer_ns();
          while (f == 0) {
            asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(f) : "r"(smem_u32(s_recflag)) : "memory");
            if (globaltimer_ns() - t0 > 4000000000ull) trap_report(5u, (unsigned long long)(unsigned)a.t);
          }
        }
        __syncwarp(am);
        const float* Rr = a.R + (size_t)mr1 * a.G4 + 4 * tl;       // written by another SM in this launch: L2, not L1
#pragma unroll
        for (int gt = 0; gt < 4; ++gt) rv[gt] = __ldcg(reinterpret_cast<const float4*>(Rr + gt * Hh));
      }
    }
    if (etid == 0) VS_STAMP(15);

    // ---- pass 2: p = e * exp(m_running - M) / S in shared memory
#pragma unroll 1
    for (int i = 0; i < MAXU; ++i) {
      const int j = g + i * VS_G;
      if (j < NUNIT && n0 + 16 * j < a.N) {
        const float f = __expf(s_mrun[i * VS_EPI_THREADS] - M) * inv;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float4* sp = reinterpret_cast<float4*>(VS_CHUNK(j, k));
          float4 e = *sp;
          e.x *= f; e.y *= f; e.z *= f; e.w *= f;
          *sp = e;
        }
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    epi_bar();

    // ---- TMA stores of the finished tile (one 32 x 32 box per row quarter and column box)
    if (g == 0 && lane == 0) {
#pragma unroll
      for (int c = 0; c < S::NBOX; ++c) {
        if (n0 + 32 * c < a.N)
          asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                       ::"l"(&tmP), "r"(smem_u32(ubox + c * S::BOX_BYTES + q * 4096)), "r"(n0 + 32 * c), "r"(m0 + q * 32)
                       : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (etid == 0) VS_STAMP(16);
    // ---- the cell of the first four rows (one per team), then whatever is left (further rows, units beyond 512, x_{t+1} otherwise)
    if (has_x) reinterpret_cast<float4*>(a.x_next + (size_t)mr1 * a.E)[tl] = xv;
    if (has_u) lstm_cell_store4(ct, Hh, mr1, 4 * tl, ev, rv, cp4);
    if (etid == 0) VS_STAMP(17);
    const bool more_rounds = ntile + VS_G * a.tiles_n < BM;
    if ((a.x_next != nullptr && (!x_first || more_rounds)) || (a.do_cell && (more_rounds || Hh > 4 * 128)))
      decode_cell_tail(ct, etid, m0, a.do_cell != 0, x_first);
    if (etid == 0) VS_STAMP(14);
    if (g == 0 && lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem may be released; the writes land by grid end
    if (etid == 0) VS_STAMP(12);
#undef VS_CHUNK
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(S::TMEM_COLS));
  }
}

template <int BN>
static int launch_vs(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tu, const CUtensorMap& tp,
                     const CUtensorMap& tw, const VSArgs& a, int grid, cudaStream_t s) {
  using S = VSCfg<BN>;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(vocab_sample_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
    attr = true;
  }
  cudaError_t e = launch_pdl(vocab_sample_kernel<BN>, dim3(grid), dim3(VS_THREADS), S::TOTAL, s, ta, tb, tu, tp, tw, a);
  if (e != cudaSuccess) { set_error("vocab_sample_kernel launch: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  // the same kernel, counted under the role it was launched in (tests assert on the names)
  return check_launch((a.n_rec > 0 || a.do_cell) ? "decode_step_kernel" : "vocab_sample_kernel");
}


}  // namespace tc

// debug timeline (GIC_VS_STAMPS=1): a static device buffer of 16 clock64 stamps per CTA, printed by gic_vs_stamps_dump()
static long long* g_stamps = nullptr;
long long* vs_stamps_buffer() {
  if (option("GIC_VS_STAMPS", 0) != 1) return nullptr;
  if (!g_stamps) { cudaMalloc(&g_stamps, 256 * 32 * sizeof(long long)); cudaMemset(g_stamps, 0, 256 * 32 * sizeof(long long)); }
  return g_stamps;
}
extern "C" void gic_vs_stamps_dump(int cta) {
  if (!g_stamps) return;
  long long h[16];
  cudaDeviceSynchronize();
  cudaMemcpy(h, g_stamps + cta * 32, sizeof(h), cudaMemcpyDeviceToHost);
  static const char* nm[13] = {"producer start", "last load issued", "first operands landed", "last mma issued", "u tile landed",
                               "pass0 done", "tmem_full", "pass1 done", "barrier in", "barrier out", "combine done", "pass2 done", "end"};
  for (int i = 0; i < 13; ++i) printf("  cta %3d  %-22s %8lld ns\n", cta, nm[i], h[i] ? h[i] - h[0] : -1);
}
extern "C" void gic_vs_stamps_table(int ncta) {
  if (!g_stamps) return;
  static long long h[256 * 32];
  cudaDeviceSynchronize();
  cudaMemcpy(h, g_stamps, sizeof(h), cudaMemcpyDeviceToHost);
  long long t0 = h[0];
  for (int c = 0; c < ncta; ++c) if (h[c * 32] && h[c * 32] < t0) t0 = h[c * 32];
  printf("cta start first_ops last_mma u_landed pass0 tmem_full pass1 publish polled combine tokens_known rec_seen tail_done end cell_loads_in stores_issued cell_done - (ns since the earliest CTA start; -1 = not stamped)\n");
  for (int c = 0; c < ncta; ++c) {
    const long long* r = h + c * 32;
    auto d = [&](int i) { return r[i] ? r[i] - t0 : -1ll; };
    printf("%3d %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld %6lld\n", c, d(0), d(2), d(3), d(4), d(5),
           d(6), d(7), d(8), d(9), d(10), d(11), d(13), d(14), d(12), d(15), d(16), d(17), d(18), d(19), d(20), d(21));
  }
}

// Scratch of vocab_sample_kernel (floats): part[0] | part[1] | tokpub | 4 spare.  part[t & 1] holds the (m, s) row
// statistics of step t, float2 [tiles_n][Mpad] sized for the narrowest tile; the two buffers alternate between steps.
// tokpub is int2 [Mpad].  [0, zeroed) is cleared before step 0.
struct VSScratch {
  size_t part[2], tokpub, zeroed, total;
  VSScratch(int B, int V) {
    const size_t Mpad = (size_t)cdiv(B, tc::BM) * tc::BM;
    part[0] = 0; part[1] = 2 * Mpad * (size_t)cdiv(V, 128);
    tokpub = 2 * part[1]; zeroed = tokpub + 2 * Mpad; total = zeroed + 4;
  }
};
size_t vocab_sample_scratch_floats(int B, int V) { return VSScratch(B, V).total; }

// Launch of vocab_sample_kernel at column-tile width BN, shared by its two roles (vocab_sample_tc, decode_step_tc): the
// h / W_out / u / out tensor maps, the VSArgs fields both roles set, the scratch carve-up (zeroed at t == 0) and the
// BN dispatch.  `a` arrives with the role's rec / cell fields set; tw is the W_hh map of the rec tiles (null in the plain
// role, which has none: ta is passed in its place).  handled stays false when TMA rejects an operand.
static int launch_vocab_sample(int BN, const float* h, int lda, const float* W_out, const float* b_out, const float* u_t,
                               float T, const float* T_dev, int B, int V, int H, int L, int t, float* out, int64_t* ids,
                               const int64_t* forced, const float* embed, int E, float* x_next, float* scratch,
                               long long* stamps, const CUtensorMap* tw, tc::VSArgs& a, cudaStream_t stream, bool* handled) {
  extern RngState rng_state();
  using namespace tc;
  const int tiles_m = cdiv(B, BM), tiles_n = cdiv(V, BN);
  const bool rn = tf32_round_in_tma();
  CUtensorMap ta, tb, tu, tp;
  bool ok = make_map(&ta, h, B, H, lda, BK, BM, rn, false) && make_map(&tb, W_out, V, H, H, BK, BN, rn, false) &&
            make_map(&tu, u_t ? u_t : out, B, V, V, 32, BM, false, false) &&
            make_map(&tp, out + (size_t)t * V, B, V, L * V, 32, 32, false, false);
  if (!ok) return GIC_OK;
  if (!tw) tw = &ta;
  const VSScratch sc(B, V);
  a.M = B; a.N = V; a.K = H; a.tiles_n = tiles_n; a.Mpad = tiles_m * BM;
  a.bias = b_out; a.T = T; a.T_dev = T_dev;
  a.part = reinterpret_cast<float2*>(scratch + sc.part[t & 1]);
  a.part_next = reinterpret_cast<float2*>(scratch + sc.part[(t + 1) & 1]);
  a.ids = ids; a.forced = forced; a.L = L; a.t = t; a.embed = embed; a.E = E; a.x_next = x_next;
  a.stamps = stamps;
  a.use_rng = (u_t == nullptr) ? 1 : 0;
  a.rng = rng_state();
  a.tokpub = reinterpret_cast<int2*>(scratch + sc.tokpub);
  if (t == 0) {
    cudaError_t e = cudaMemsetAsync(scratch, 0, sc.zeroed * sizeof(float), stream);   // statistics "not ready", token tags 0
    if (e != cudaSuccess) { set_error("vocab_sample memset: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  }
  int rc;
  const int grid = a.n_rec + tiles_m * tiles_n;
  switch (BN) {
    case 128: rc = launch_vs<128>(ta, tb, tu, tp, *tw, a, grid, stream); break;
    case 160: rc = launch_vs<160>(ta, tb, tu, tp, *tw, a, grid, stream); break;
    case 192: rc = launch_vs<192>(ta, tb, tu, tp, *tw, a, grid, stream); break;
    case 224: rc = launch_vs<224>(ta, tb, tu, tp, *tw, a, grid, stream); break;
    default: rc = launch_vs<256>(ta, tb, tu, tp, *tw, a, grid, stream); break;
  }
  if (rc == GIC_OK) *handled = true;
  return rc;
}

// One fused decode step on the tensor cores.  handled = false (nothing launched) when the shape does not fit the
// co-resident grid or TMA's alignment rules; the caller then runs the separate projection + sampler kernels.
int vocab_sample_tc(const float* htop, int lda, const float* W_out, const float* b_out, const float* u_t, float T,
                    const float* T_dev, int B, int V, int H, int L, int t, float* out, int64_t* ids, const int64_t* forced,
                    const float* embed, int E, float* x_next, float* scratch, cudaStream_t stream, bool* handled) {
  using namespace tc;
  *handled = false;
  if (option("GIC_FUSED_SAMPLE", 1) == 0) return GIC_OK;
  if (B <= 0 || V <= 0 || H <= 0) return GIC_OK;
  if ((V % 4) || (H % 4) || (lda % 4) || !aligned16(htop) || !aligned16(W_out) || !aligned16(b_out) || (u_t && !aligned16(u_t)) ||
      !aligned16(out) || (((size_t)L * V) % 4))
    return GIC_OK;
  const int tiles_m = cdiv(B, BM);
  if (tiles_m > 64) return GIC_OK;
  const int G = num_sms();
  static const int kBN[6] = {128, 160, 192, 224, 256, 0};
  int BN = 0;
  for (int i = 0; kBN[i]; ++i)
    if ((long long)tiles_m * cdiv(V, kBN[i]) <= G) { BN = kBN[i]; break; }
  if (!BN) return GIC_OK;
  VSArgs a = {};                // no rec tiles, no cell tail
  a.rec_tiles_n = 1; a.RBN = 16;
  return launch_vocab_sample(BN, htop, lda, W_out, b_out, u_t, T, T_dev, B, V, H, L, t, out, ids, forced, embed, E, x_next,
                             scratch, vs_stamps_buffer(), nullptr, a, stream, handled);
}

// ---------------------------------------------------------------------------------------------------------
// Fused decode step (single layer, Gumbel-softmax mode): projection + sample of step t, the recurrent contraction
// R = h_t W_hh^T of step t + 1 on the SMs the projection leaves idle, and the LSTM cell of step t + 1 in the tail of the
// CTA that sampled the row's token (kernel comment at the top of this file).
//   hs_t1  [B, H]  h after LSTM step t (the projection's and the rec tiles' A operand)
//   EW     [V, 4H] embed W_ih^T + b_ih + b_hh (built by the caller), R [B, 4H] scratch, rec_done: tiles_m counters zeroed by the caller
//          before step 0, `scratch` as vocab_sample_tc (zeroed by this function at t == 0)
//   last != 0: no next step -- the kernel degenerates to the plain projection + sample.
// decode_step_plan says whether the shape fits (co-resident grid: projection tiles + at least ceil(4H / 256) rec tiles per
// row block <= SMs); the caller falls back to lstm_step_tc + vocab_sample_tc otherwise.
// ---------------------------------------------------------------------------------------------------------
struct DecodeStepPlan { int BN, tiles_m, rec_tiles_n, RBN; };

static bool decode_step_plan_impl(int B, int V, int H, DecodeStepPlan* p) {
  using namespace tc;
  if (B <= 0 || V <= 0 || H <= 0 || (V % 4) || (H % 32)) return false;
  const int tiles_m = cdiv(B, BM);
  if (tiles_m > 64) return false;
  const int G = num_sms(), G4 = 4 * H;
  static const int kBN[6] = {128, 160, 192, 224, 256, 0};
  for (int i = 0; kBN[i]; ++i) {
    const int tiles_v = tiles_m * cdiv(V, kBN[i]);
    const int spare = G - tiles_v;
    if (spare < tiles_m * cdiv(G4, 256)) continue;
    int per = spare / tiles_m;                                   // rec tiles per row block
    if (per > G4 / 32) per = G4 / 32;                            // no narrower than 32 columns
    int RBN = ((cdiv(G4, per) + 15) / 16) * 16;
    if (RBN > 256) RBN = 256;
    p->BN = kBN[i]; p->tiles_m = tiles_m; p->RBN = RBN; p->rec_tiles_n = cdiv(G4, RBN);
    return true;
  }
  return false;
}
bool decode_step_plan(int B, int V, int H) {
  if (option("GIC_FUSED_SAMPLE", 1) == 0 || option("GIC_DECODE_STEP", 1) == 0) return false;
  DecodeStepPlan p;
  return decode_step_plan_impl(B, V, H, &p);
}
int decode_step_tc(const float* hs_t1, const float* W_out, const float* b_out, const float* W_hh, const float* EW, float* R, unsigned int* rec_done, const float* u_t, float T,
                   const float* T_dev, int B, int V, int H, int L, int t, int last, float* out, int64_t* ids,
                   const int64_t* forced, const float* embed, int E, float* x_next, const float* c_prev, float* c_out,
                   float* h_out, float* acts, float* htop, float* scratch, cudaStream_t stream, bool* handled) {
  using namespace tc;
  *handled = false;
  DecodeStepPlan pl;
  if (!decode_step_plan_impl(B, V, H, &pl)) return GIC_OK;
  const void* ptrs[] = {hs_t1, W_out, b_out, W_hh, EW, R, out, c_prev, c_out, h_out, acts, htop, u_t ? u_t : out};
  for (const void* p : ptrs)
    if (!aligned16(p)) return GIC_OK;
  if (((size_t)L * V) % 4) return GIC_OK;
  CUtensorMap tw;
  if (!make_map(&tw, W_hh, 4 * H, H, H, BK, pl.RBN, tf32_round_in_tma(), false)) return GIC_OK;
  VSArgs a = {};
  a.n_rec = last ? 0 : pl.tiles_m * pl.rec_tiles_n;
  a.rec_tiles_n = pl.rec_tiles_n; a.RBN = pl.RBN; a.G4 = 4 * H; a.R = R; a.rec_done = rec_done;
  a.rec_expect = (unsigned int)(t + 1) * (unsigned int)pl.rec_tiles_n;
  a.do_cell = last ? 0 : 1;
  a.EW = EW; a.c_prev = c_prev; a.c_out = c_out; a.h_out = h_out; a.acts = acts; a.htop = htop;
  long long* stamps = vs_stamps_buffer();     // debug timeline of ONE step (GIC_VS_STAMPS=1, GIC_VS_STAMPS_T=t; default L - 2)
  if (stamps && t != option("GIC_VS_STAMPS_T", L - 2)) stamps = nullptr;
  return launch_vocab_sample(pl.BN, hs_t1, H, W_out, b_out, u_t, T, T_dev, B, V, H, L, t, out, ids, forced, embed, E, x_next,
                             scratch, stamps, &tw, a, stream, handled);
}

}  // namespace gic
