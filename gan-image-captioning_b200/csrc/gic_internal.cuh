// Internal helpers shared by the sm_100a kernels of libgic_b200.  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/gic_b200.h"

namespace gic {

// status codes: GIC_OK / GIC_ERR_* macros from the public header

void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define GIC_REQUIRE(cond, code, ...)            \
  do {                                          \
    if (!(cond)) {                              \
      gic::set_error(__VA_ARGS__);              \
      return (code);                            \
    }                                           \
  } while (0)

#define GIC_TRY(expr)                           \
  do {                                          \
    int _rc = (expr);                           \
    if (_rc != GIC_OK) return _rc;         \
  } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// float count rounded up to a multiple of 4: every region of a caller-allocated buffer starts 16-byte aligned
static inline size_t a4(size_t x) { return (x + 3) & ~(size_t)3; }

int num_sms();

// ---- per-caller state (include/gic_b200.h "contexts") ------------------------------------------------------------
// What used to be process-global setters lives in a context; every host thread has a current one (a thread-local default
// until gic_ctx_set_current installs another), so two instructors -- or two threads -- in one process cannot corrupt each other.
struct RngStateHost { unsigned long long seed, offset; const unsigned long long* dev; };
struct Ctx {
  const float* t_dev = nullptr;           // gic_set_temperature_device
  const float* prepared = nullptr;        // gic_disc_set_prepared
  RngStateHost rng = {0ull, 0ull, nullptr};   // gic_set_rng
  cudaEvent_t vocab_grads_event = nullptr;    // gic_set_vocab_grads_event
  cudaEvent_t embed_grads_event = nullptr;    // gic_set_embed_grads_event
  // A/B and tuning switches (gic_ctx_set_option).  A name that was never set is looked up in the environment ONCE per
  // context (the first time a launch path asks) and remembered: no getenv on the launch paths after that.
  struct Opt { char name[28]; int value; bool has; };
  static constexpr int MAX_OPTS = 48;
  Opt opts[MAX_OPTS];
  int n_opts = 0;
};
Ctx& ctx();                               // the calling thread's current context
// Diagnostics of the bounded device-side waits: the site that gave up writes four words to this host-mapped buffer before
// it traps (the context is dead afterwards, pinned host memory is not).  [0] site id (0 = none), [1] site-specific,
// [2] blockIdx.x << 32 | threadIdx.x, [3] globaltimer.  gic_trap_info() reads it.
unsigned long long* trap_slot();          // host-mapped; the same pointer is valid on the device (UVA); nullptr if unavailable
int option(const char* name, int dflt);   // the current context's value of a switch (set_option > environment > dflt)
bool option_is_set(const char* name);
void option_set(const char* name, int value);
void option_clear(const char* name);      // forget it: the next lookup consults the environment again

// ---- optional per-kernel-class device timing (bench.py roofline): CUDA events on the launching stream ----
enum ProfKind : int { PROF_GEMM = 0, PROF_SAMPLE = 1, PROF_CONVPOOL = 2, PROF_SOFTMAX_BWD = 3, PROF_ADAM = 4,
                      PROF_HEAD = 5, PROF_GEMM_D = 6, PROF_GEMM_DECODE = 7, PROF_VOCAB_SAMPLE = 8, PROF_KINDS = 9 };
bool prof_enabled();
void prof_open(int kind, double work, cudaStream_t s);    // work = algorithmic flops (GEMM) or bytes
void prof_close(cudaStream_t s);
struct ProfScope {
  cudaStream_t s; bool on;
  ProfScope(int kind, double work, cudaStream_t st) : s(st), on(prof_enabled()) { if (on) prof_open(kind, work, s); }
  ~ProfScope() { if (on) prof_close(s); }
};

// ---- fp32 GEMM (CUDA cores, exact-fp32 path) -------------------------------------------
// C[M,N] = alpha * op(A)[M,K] * op(B)[K,N] + beta * C + bias[N]   (row-major everywhere)
//   transA == 0: A is [M,K] with leading dim lda;  transA == 1: A is [K,M]
//   transB == 0: B is [K,N] with leading dim ldb;  transB == 1: B is [N,K]  (nn.Linear weight)
int gemm_f32(bool transA, bool transB, int M, int N, int K, float alpha, const float* A, int lda,
             const float* B, int ldb, float beta, float* C, int ldc, const float* bias,
             cudaStream_t stream);

// Precision selector for the dense contractions of the hot path.
enum GemmMode : int {
  GEMM_FP32 = 0,     // CUDA-core FFMA, exact fp32 (parity mode)
  GEMM_TF32 = 1,     // tcgen05 kind::tf32, single pass (throughput mode)
  GEMM_BF16 = 3      // as GEMM_TF32, with the discriminator's [N*R,F] x [F,F] contractions on bf16 operands (kind::f16)
};

// bf16-operand GEMM (fp32 accumulate / output); A, B are bf16 with leading dimensions in elements.
int gemm_bf16(bool transA, bool transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B,
              int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream, int prof_kind = PROF_GEMM);
// dst[r, c] = bf16(src[r, c]) for c < cols (pitches in elements)
int f32_to_bf16(const float* src, int rows, int cols, int ld_src, void* dst, int ld_dst, cudaStream_t stream);

// Dispatching GEMM used by the path: routes to tcgen05 when the mode/shape allow, else FFMA.
int gemm(int mode, bool transA, bool transB, int M, int N, int K, float alpha, const float* A,
         int lda, const float* B, int ldb, float beta, float* C, int ldc, const float* bias,
         cudaStream_t stream, int prof_kind = PROF_GEMM);

// Fused vocab projection + Gumbel-softmax + sample of one decode step (vocab_sample_tcgen05.cu).
size_t vocab_sample_scratch_floats(int B, int V);
int vocab_sample_tc(const float* htop, int lda, const float* W_out, const float* b_out, const float* u_t, float T,
                    const float* T_dev, int B, int V, int H, int L, int t, float* out, int64_t* ids, const int64_t* forced,
                    const float* embed, int E, float* x_next, float* scratch, cudaStream_t stream, bool* handled);

// Per-row state of the sampled-caption decode (beam_tcgen05.cu sample_rows_kernel): ids[M,L] (PAD after EOS), the frozen
// flag, lengths, caption log-likelihoods and the next LSTM input x[M,E] = embed[token].
struct SampleDecode {
  int64_t* ids; int* fin; int32_t* len; float* caption_logp; float* x; const float* embed;
  int L, E, eos;
};

// Constrained generation (beam_tcgen05.cu ban_rows_kernel): the ban-bitmap regions of a decode's workspace, in floats from
// the region's start; all of size 0 when c == NULL (unconstrained).  base[words] (the bad ids) | ban[M][words] (per row,
// rebuilt every step) | prefix[M][L] (int, the rows' prefixes; no_repeat_ngram_size >= 1 only), words = ceil(V / 32).
struct BanWs {
  size_t base, ban, prefix, total;
  int words;
  BanWs(int M, int V, int L, const gic_decode_constraints_t* c) {
    words = (V + 31) / 32;
    const bool on = c != nullptr;
    base = 0;
    ban = on ? a4((size_t)words) : 0;
    prefix = ban + (on ? a4((size_t)M * words) : 0);
    total = prefix + ((on && c->no_repeat_ngram_size > 0) ? a4((size_t)M * L) : 0);
  }
};
// base bitmap of c->bad_ids (once per call), then per step the bitmap of rows m < M; fin[M] marks frozen rows (skipped),
// the prefix is ids[m, :t] (ids[M][L], sampling) or the trace[L][B][K] backtrack of beam slot m % K (ids == NULL)
int ban_base(const gic_decode_constraints_t* c, int V, const BanWs& bw, float* region, cudaStream_t s);
int ban_rows(const gic_decode_constraints_t* c, int M, int V, int L, int t, int eos, const int* fin, const int64_t* ids,
             const int32_t* trace, int B, int K, const BanWs& bw, float* region, cudaStream_t s);

// dz (bf16) = T p (demb W_e - dot) and db_out = colsum(dz) in one streaming tcgen05 kernel (dz_fused_tcgen05.cu)
int dz_fused_tc(const float* demb, int K, const float* W_e, const float* p, const float* dot, float T, const float* T_dev,
                int M, int V, void* dz_bf, int Vp, float* db_out, int accumulate, cudaStream_t stream, bool* handled);

// ---- discriminator buffers (disc.cu).  Each struct is the one definition of a buffer's layout: the fields are region
// offsets in floats, `total` is the size the gic_disc_*_floats queries return.
// pitch (elements) of the bf16 copies used by GIC_GEMM_BF16: rows of 128-byte multiples (TMA fetches whole lines)
static inline int bf_pitch(int F) { return ((F + 63) / 64) * 64; }
// saved for backward: emb[N*L*De] | pooled[N*R*F] | hpre[N*R*F] | arg(u8)[N*R*F] | pooled_bf(bf16)[N*R*Fp]
struct DiscSaved {
  size_t emb, pooled, hpre, arg, pooled_bf, total;
  DiscSaved(int N, int L, int De, int R, int F) {
    const size_t rows = (size_t)N * R;
    emb = 0; pooled = a4((size_t)N * L * De); hpre = pooled + a4(rows * F); arg = hpre + a4(rows * F);
    pooled_bf = arg + a4((rows * F + 3) / 4); total = pooled_bf + a4(rows * bf_pitch(F) / 2);
  }
};
// forward workspace, also the layout of the prepared blob: weff[F+1] (collapsed head) | W_h_bf(bf16)[F*Fp]
struct DiscFwdWs {
  size_t weff, W_h_bf, total;
  explicit DiscFwdWs(int F) { weff = 0; W_h_bf = a4((size_t)F + 1); total = W_h_bf + a4((size_t)F * bf_pitch(F) / 2); }
};
// backward workspace: weff[F+1] | dh | dx[rows*F] | s[F] | dbh[F] | demb[N*L*De] | W_h_bf(bf16)[F*Fp] | dxg[rows*F]
//   dh is fp32 [rows,F], or bf16 [rows,Fp] in GIC_GEMM_BF16 mode; dxg = dh W_h (beta = 0), added to dx by the conv / pool backward
struct DiscBwdWs {
  size_t weff, dh, dx, s, dbh, demb, W_h_bf, dxg, total;
  DiscBwdWs(int N, int L, int De, int R, int F) {
    const size_t rows = (size_t)N * R, dh_f32 = a4(rows * F), dh_bf16 = a4(rows * bf_pitch(F) / 2);
    weff = 0; dh = a4((size_t)F + 1); dx = dh + (dh_f32 > dh_bf16 ? dh_f32 : dh_bf16); s = dx + a4(rows * F);
    dbh = s + a4(F); demb = dbh + a4(F); W_h_bf = demb + a4((size_t)N * L * De);
    dxg = W_h_bf + a4((size_t)F * bf_pitch(F) / 2); total = dxg + a4(rows * F);
  }
};

// out[N] (+)= scale * sum_rows A[M,N]
int colsum_f32(const float* A, int M, int N, int lda, float scale, bool accumulate, float* out,
               cudaStream_t stream);

// ---- programmatic dependent launch (serial kernel chains: decode steps, BPTT) ---------------------------
// A kernel that executes pdl_wait() before its first global-memory access may be launched with launch_pdl(): the
// launch is processed while its predecessor in the stream still runs, so launch latency, barrier initialisation, TMEM
// allocation and tensor-map prefetch overlap the predecessor's tail.  pdl_wait() returns once the predecessor grid has
// completed and its writes are visible; pdl_trigger() (after the wait: a kernel two places down the chain must never
// start before the one two places up has finished) lets the successor's launch begin.  Both are no-ops in a kernel
// launched without the attribute.  ONLY kernels containing pdl_wait() may be launched through launch_pdl().
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();          // GIC_PDL=0 turns the attribute off (read per call: tests and A/B runs toggle it)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- device helpers ---------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// Block-wide sum; `red` is >= 32 floats of shared memory.  All threads get the result.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.0f;
  r = warp_sum(r);
  return r;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : -INFINITY;
  r = warp_max(r);
  return r;
}

}  // namespace gic
