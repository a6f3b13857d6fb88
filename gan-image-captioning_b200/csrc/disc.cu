// Discriminator hot path (RelGAN multi-representation CNN): embedding (soft GEMM or hard
// column gather), fused conv + bias + ReLU + max-over-time emitting [N*R, F] directly, highway
// mix, dropout and the collapsed 900->100->1 score head, plus the backward of all of it.
// Replaces Discriminator.forward (src/discriminator.py:34-62) and its autograd backward.
#include <stdlib.h>

#include "gic_internal.cuh"

namespace gic {

constexpr int MAX_GROUPS = 8;

// packed fp32 pair helpers for fma.rn.f32x2 (Blackwell packed FP32 pipe)
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// fp32 -> bf16, round to nearest even (finite inputs)
__device__ __forceinline__ unsigned short f2bf(float x) {
  unsigned int u = __float_as_uint(x);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (unsigned short)(u >> 16);
}

struct ConvGroups {
  const float* w[MAX_GROUPS];   // [n, 1, f, es] contiguous == [n][f*es]
  const float* b[MAX_GROUPS];   // [n]
  float* dw[MAX_GROUPS];
  float* db[MAX_GROUPS];
  int f[MAX_GROUPS];
  int n[MAX_GROUPS];
  int col0[MAX_GROUPS];
  int ngroups;
  int F;                        // sum n
  int kmax;                     // max f*es
};

// ---------------------------------------------------------------------------------------
// hard-token embedding: Linear(one_hot(id)) == column `id` of embeddings.weight[De, V]
// (src/training.py:158 + src/discriminator.py:40).  Bit-identical to the dense product.
// ---------------------------------------------------------------------------------------
__global__ void disc_embed_ids_kernel(const int64_t* __restrict__ ids, int n_tok, int V, int De,
                                      const float* __restrict__ W_e, float* __restrict__ emb) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_tok * De) return;
  const int i = idx / De, r = idx % De;
  int64_t id = ids[i];
  if (id < 0 || id >= V) id = 0;
  emb[idx] = W_e[(size_t)r * V + id];
}

// dW_e[r, id] += demb[i, r]
__global__ void disc_embed_ids_bwd_kernel(const int64_t* __restrict__ ids, int n_tok, int V, int De,
                                          const float* __restrict__ demb, float* __restrict__ dW_e) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_tok * De) return;
  const int i = idx / De, r = idx % De;
  int64_t id = ids[i];
  if (id < 0 || id >= V) id = 0;
  atomicAdd(dW_e + (size_t)r * V + id, demb[idx]);
}

// ---------------------------------------------------------------------------------------
// fused conv(f, es) + bias + ReLU + max over time, all filter groups, all R representations.
// One CTA per caption.  smem: emb[L*De] | wk[kmax][F] | bias[F] | fsz[F].
// Lanes run along the feature column c, so the [N*R, F] output rows are written coalesced and
// the embedding reads are warp broadcasts.  ES1 fast path: float4 over 4 representations.
// out: pooled[(n*R + r)*F + c] = max_t relu(conv), arg = first t attaining it (uint8).
// ---------------------------------------------------------------------------------------
// arg value stored when the pooled activation is not positive: ReLU passes no gradient there, so the backward
// kernels need neither the pooled value nor a time index for that entry.
constexpr int ARG_DEAD = 255;

// one (feature column, 4 representations) work item of the ES1 fast path, filter size FK.  The FK embedding rows under
// the filter are kept in a register window that slides one row per time step (one LDS.128 per step instead of FK); the
// ReLU is hoisted out of the max (max_t relu(x_t) = relu(max_t x_t), same first arg-max whenever the max is positive).
template <int FK>
__device__ __forceinline__ void conv_item_es1(const float* emb_s, const float* wk_s, int F, int c, float bias,
                                              int L, int R, int rb, float4& best, int (&a)[4]) {
  float w[FK];
#pragma unroll
  for (int k = 0; k < FK; ++k) w[k] = wk_s[k * F + c];
  best = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  a[0] = a[1] = a[2] = a[3] = 0;
  const int T = L - FK + 1;
  const float4* e4 = reinterpret_cast<const float4*>(emb_s) + rb;     // row t at e4[t * (R / 4)]
  const int RS = R >> 2;
  float4 win[FK];
#pragma unroll
  for (int k = 0; k < FK - 1; ++k) win[k] = e4[k * RS];
#pragma unroll 4
  for (int t = 0; t < T; ++t) {
    win[FK - 1] = e4[(t + FK - 1) * RS];
    // packed fp32 FMAs (fma.rn.f32x2, sm_100): two representations per instruction, same rounding as fmaf
    unsigned long long a01 = pack2(bias, bias), a23 = a01;
#pragma unroll
    for (int k = 0; k < FK; ++k) {
      const unsigned long long ww = pack2(w[k], w[k]);
      a01 = ffma2(ww, pack2(win[k].x, win[k].y), a01);
      a23 = ffma2(ww, pack2(win[k].z, win[k].w), a23);
    }
    float4 acc;
    unpack2(a01, acc.x, acc.y);
    unpack2(a23, acc.z, acc.w);
    if (acc.x > best.x) { best.x = acc.x; a[0] = t; }
    if (acc.y > best.y) { best.y = acc.y; a[1] = t; }
    if (acc.z > best.z) { best.z = acc.z; a[2] = t; }
    if (acc.w > best.w) { best.w = acc.w; a[3] = t; }
#pragma unroll
    for (int k = 0; k < FK - 1; ++k) win[k] = win[k + 1];
  }
  if (!(best.x > 0.f)) { best.x = 0.f; a[0] = ARG_DEAD; }
  if (!(best.y > 0.f)) { best.y = 0.f; a[1] = ARG_DEAD; }
  if (!(best.z > 0.f)) { best.z = 0.f; a[2] = ARG_DEAD; }
  if (!(best.w > 0.f)) { best.w = 0.f; a[3] = ARG_DEAD; }
}

// grid = (captions, column slices): CTA (n, y) handles feature columns [y*cs, (y+1)*cs) of caption n for all R
// representations, so that N * slices CTAs balance over the SMs even at N = 256.
template <bool ES1>
__global__ void __launch_bounds__(256)
conv_pool_fwd_kernel(const float* __restrict__ emb, int L, int De, int R, int es, ConvGroups g, int cs,
                     float* __restrict__ pooled, uint8_t* __restrict__ arg, unsigned short* __restrict__ pooled_bf,
                     int Fp) {
  extern __shared__ __align__(16) float sm[];
  const int F = g.F, kmax = g.kmax;
  const int c_lo = blockIdx.y * cs, c_hi = min(F, c_lo + cs), CW = c_hi - c_lo;
  float* emb_s = sm;                                // L*De (De % 4 == 0 on the ES1 path)
  float* wk_s = emb_s + ((L * De + 3) & ~3);        // [kmax][cs]   (this slice's columns)
  float* bias_s = wk_s + kmax * cs;                 // [cs]
  int* fk_s = reinterpret_cast<int*>(bias_s + cs);  // [cs]  f*es per column
  const int n = blockIdx.x;
  for (int i = threadIdx.x; i < L * De; i += blockDim.x) emb_s[i] = emb[(size_t)n * L * De + i];
  for (int i = threadIdx.x; i < CW * kmax; i += blockDim.x) {
    const int cl = i / kmax, k = i % kmax, c = c_lo + cl;
    int gi = 0;
    while (gi + 1 < g.ngroups && c >= g.col0[gi + 1]) ++gi;
    const int fk = g.f[gi] * es;
    wk_s[k * cs + cl] = (k < fk) ? g.w[gi][(c - g.col0[gi]) * fk + k] : 0.f;
    if (k == 0) { bias_s[cl] = g.b[gi][c - g.col0[gi]]; fk_s[cl] = fk; }
  }
  __syncthreads();

  if (ES1) {
    const int RB = R / 4;
    for (int item = threadIdx.x; item < CW * RB; item += blockDim.x) {
      const int cl = item % CW, rb = item / CW, c = c_lo + cl;
      const float bias = bias_s[cl];
      float4 best;
      int a[4];
      switch (fk_s[cl]) {   // lanes of a warp share a filter group except at group boundaries
        case 1: conv_item_es1<1>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 2: conv_item_es1<2>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 3: conv_item_es1<3>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 4: conv_item_es1<4>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 5: conv_item_es1<5>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 6: conv_item_es1<6>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        case 7: conv_item_es1<7>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
        default: conv_item_es1<8>(emb_s, wk_s, cs, cl, bias, L, R, rb, best, a); break;
      }
      const size_t row = (size_t)n * R + rb * 4;
      pooled[(row + 0) * F + c] = best.x; arg[(row + 0) * F + c] = (uint8_t)a[0];
      pooled[(row + 1) * F + c] = best.y; arg[(row + 1) * F + c] = (uint8_t)a[1];
      pooled[(row + 2) * F + c] = best.z; arg[(row + 2) * F + c] = (uint8_t)a[2];
      pooled[(row + 3) * F + c] = best.w; arg[(row + 3) * F + c] = (uint8_t)a[3];
      if (pooled_bf) {           // bf16 copy (pitch Fp) for the tensor-core contractions of GIC_GEMM_BF16
        pooled_bf[(row + 0) * Fp + c] = f2bf(best.x); pooled_bf[(row + 1) * Fp + c] = f2bf(best.y);
        pooled_bf[(row + 2) * Fp + c] = f2bf(best.z); pooled_bf[(row + 3) * Fp + c] = f2bf(best.w);
      }
    }
  } else {
    for (int item = threadIdx.x; item < CW * R; item += blockDim.x) {
      const int cl = item % CW, r = item / CW, c = c_lo + cl;
      const int fk = fk_s[cl], f = fk / es;
      const float bias = bias_s[cl];
      float best = -INFINITY;
      int a = 0;
      const int T = L - f + 1;
      for (int t = 0; t < T; ++t) {
        float acc = bias;
        for (int kk = 0; kk < fk; ++kk)
          acc = fmaf(wk_s[kk * cs + cl], emb_s[(t + kk / es) * De + r * es + kk % es], acc);
        if (acc > best) { best = acc; a = t; }
      }
      if (!(best > 0.f)) { best = 0.f; a = ARG_DEAD; }
      pooled[((size_t)n * R + r) * F + c] = best;
      arg[((size_t)n * R + r) * F + c] = (uint8_t)a;
      if (pooled_bf) pooled_bf[((size_t)n * R + r) * Fp + c] = f2bf(best);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Tensor-core variant of conv_pool_fwd_kernel for the tensor-core GEMM modes (ES1 layout, f <= 5).
// The conv over time is a tiny contraction out[c, t, r] = sum_k w[c, k] emb[t + k, r] (k < f): one warp-level
// mma.sync.m16n8k16 (bf16 operands, fp32 accumulate) per 16 channels x 8 representations x 1 time step, and the max /
// first arg-max over t is a per-register compare on the accumulator fragment -- the 250 M conv outputs of a c2 call never
// leave registers.  The CUDA-core kernel spends ~10 instructions per output (ncu), this one ~3.5.
// Precision: both operands are split x = hi + lo with hi, lo in bf16 (round to nearest), and the three significant
// products share the K = 16 slots of ONE instruction:
//     k = 0..4   w_hi[k]    * x_hi[t + k]
//     k = 5..9   w_hi[k-5]  * x_lo[t + k - 5]
//     k = 10..14 w_lo[k-10] * x_hi[t + k - 10]            (k = 15 unused; the dropped lo * lo term is 2^-16 relative)
// so the result carries ~16 mantissa bits per operand: 30 x finer than the TF32 contraction that produced emb in these
// modes.  The pooled value itself is stored with its low 5 mantissa bits cleared (see the arg-max trick in the loop).  (Three TF32 m16n8k8 MMAs per step reach fp32 accuracy but measured SLOWER than the CUDA-core kernel, 131 vs
// 121 us: the legacy tensor path issues one HMMA per ~12 cycles and sub-partition.  A tcgen05/TMEM formulation was
// rejected: TMEM reads back at 64 B/clk/SM, and all outputs would have to come back through it, ~55 us.)
// grid = (captions, slices of channel blocks); a channel block = 16 channels of ONE filter group (groups padded to 16).
// smem: XB[T_max][4 (tg)][68] uint2 = the two B-fragment registers of lane (tg, r) at time t, ready-made
//       | WA[blocks][16][12] uint32 (bf16 pairs, A fragment order) | bias[blocks][16] | meta[blocks] int4
// ---------------------------------------------------------------------------------------
constexpr int CM_XS = 68;     // uint2 row pitch of one (t, tg) row: the 8-byte loads of a half-warp hit 32 distinct banks
constexpr int CM_WS = 12;     // 32-bit row pitch of a weight block: the four A-fragment loads are conflict-free
constexpr int CM_FMAX = 5;    // taps per part: 3 parts x 5 taps fill the 16 K slots

__device__ __forceinline__ void mma_bf16_16x8x16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float bf2f(unsigned short h) { return __uint_as_float((uint32_t)h << 16); }
__device__ __forceinline__ float fmax3(float a, float b, float c) {       // 3-input maximum (sm_100: one FMNMX3)
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
__device__ __forceinline__ unsigned short cvt_bf16(float x) {     // round to nearest even, one instruction
  unsigned short h;
  asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(h) : "f"(x));
  return h;
}
// number of 16-channel blocks over all groups
static inline int conv_mma_blocks(const ConvGroups& g) {
  int nb = 0;
  for (int i = 0; i < g.ngroups; ++i) nb += (g.n[i] + 15) / 16;
  return nb;
}

template <int NBLK>
__device__ __forceinline__ void conv_mma_unit(const uint2* __restrict__ xs, const uint32_t* __restrict__ wa,
                                              const float* __restrict__ bias_s, const int4* __restrict__ meta, int b0,
                                              int T, int gq, int tg, size_t row0, int F, float* __restrict__ pooled,
                                              uint8_t* __restrict__ arg, unsigned short* __restrict__ pooled_bf, int Fp) {
  uint32_t af[NBLK][4];
  float bs[NBLK][2], best[NBLK][4];
  uint32_t tinv = 31u;
#pragma unroll
  for (int i = 0; i < NBLK; ++i) {
    const uint32_t* w = wa + (size_t)(b0 + i) * 16 * CM_WS;
    af[i][0] = w[gq * CM_WS + tg];
    af[i][1] = w[(gq + 8) * CM_WS + tg];
    af[i][2] = w[gq * CM_WS + tg + 4];
    af[i][3] = w[(gq + 8) * CM_WS + tg + 4];
    bs[i][0] = bias_s[(b0 + i) * 16 + gq];
    bs[i][1] = bias_s[(b0 + i) * 16 + gq + 8];
#pragma unroll
    for (int e = 0; e < 4; ++e) best[i][e] = -INFINITY;
  }
  // (max, first arg-max) in ONE maximum: the low 5 mantissa bits of a candidate are replaced by 31 - t, so that among
  // candidates equal in the upper 27 bits the earliest step wins and the winner's step can be read back from the maximum
  // itself.  Compare / select instructions run on the half-rate ALU pipe and were the bound of this kernel (FSETP + FSEL +
  // SEL per output: ncu ALU pipe 68 %, math-pipe throttle); this is one LOP3 per output and one 3-input FMNMX per two.
  // The 2^-19 truncation is below the 2^-16 of the bf16 split; only positive maxima are used (ReLU), where float
  // order = bit order.
  int t = 0;
#pragma unroll 2
  for (; t + 1 < T; t += 2) {
    const uint2 q0 = xs[(size_t)t * 4 * CM_XS], q1 = xs[(size_t)(t + 1) * 4 * CM_XS];
#pragma unroll
    for (int i = 0; i < NBLK; ++i) {
      float c0[4] = {bs[i][0], bs[i][0], bs[i][1], bs[i][1]};
      float c1[4] = {bs[i][0], bs[i][0], bs[i][1], bs[i][1]};
      mma_bf16_16x8x16(c0, af[i], q0.x, q0.y);
      mma_bf16_16x8x16(c1, af[i], q1.x, q1.y);
#pragma unroll
      for (int e = 0; e < 4; ++e)
        best[i][e] = fmax3(best[i][e], __uint_as_float((__float_as_uint(c0[e]) & 0xffffffe0u) | tinv),
                           __uint_as_float((__float_as_uint(c1[e]) & 0xffffffe0u) | (tinv - 1u)));
    }
    tinv -= 2u;
  }
  if (t < T) {
    const uint2 q = xs[(size_t)t * 4 * CM_XS];
#pragma unroll
    for (int i = 0; i < NBLK; ++i) {
      float c[4] = {bs[i][0], bs[i][0], bs[i][1], bs[i][1]};
      mma_bf16_16x8x16(c, af[i], q.x, q.y);
#pragma unroll
      for (int e = 0; e < 4; ++e)
        best[i][e] = fmaxf(best[i][e], __uint_as_float((__float_as_uint(c[e]) & 0xffffffe0u) | tinv));
    }
  }
  // ReLU hoisted out of the max; outputs: channels (gq, gq + 8) x representations (2 tg, 2 tg + 1)
#pragma unroll
  for (int i = 0; i < NBLK; ++i) {
    const int4 m = meta[b0 + i];                   // x = first global column of the block, y = valid channels
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int ch = gq + ((e >> 1) << 3), rr = 2 * tg + (e & 1);
      if (ch < m.y) {
        const uint32_t kb = __float_as_uint(best[i][e]);
        float v = __uint_as_float(kb & 0xffffffe0u);
        int a = 31 - (int)(kb & 31u);
        if (!(v > 0.f)) { v = 0.f; a = ARG_DEAD; }
        const size_t o = (row0 + rr) * F + m.x + ch;
        pooled[o] = v;
        arg[o] = (uint8_t)a;
        if (pooled_bf) pooled_bf[(row0 + rr) * Fp + m.x + ch] = cvt_bf16(v);
      }
    }
  }
}

__global__ void __launch_bounds__(256)
conv_pool_fwd_mma_kernel(const float* __restrict__ emb, int L, int R, ConvGroups g, int bps /*blocks per slice*/,
                         int nblocks, int Tmax, float* __restrict__ pooled, uint8_t* __restrict__ arg,
                         unsigned short* __restrict__ pooled_bf, int Fp) {
  extern __shared__ __align__(16) float sm[];
  const int F = g.F;
  const int n = blockIdx.x;
  const int blk_lo = blockIdx.y * bps, nb = min(bps, nblocks - blk_lo);
  uint2* xb = reinterpret_cast<uint2*>(sm);                                     // [Tmax][4][CM_XS]
  uint32_t* wa = reinterpret_cast<uint32_t*>(sm + (size_t)Tmax * 4 * CM_XS * 2);  // [bps][16][CM_WS]
  float* bias_s = reinterpret_cast<float*>(wa + (size_t)bps * 16 * CM_WS);      // [bps][16]
  int4* meta = reinterpret_cast<int4*>(bias_s + (size_t)bps * 16);              // [bps]: first column, valid channels, f, -
  // stage 1: hl[t][r] = bf16 hi | bf16 lo << 16 of the caption's embedding rows (rows past the end are zero; their
  // weights are zero as well).  hl aliases the tail of the dynamic shared memory (after meta).
  uint32_t* hl = reinterpret_cast<uint32_t*>(meta + bps);                       // [(Tmax + 4)][R]
  const float* en = emb + (size_t)n * L * R;
  for (int i = threadIdx.x; i < (Tmax + 4) * R; i += blockDim.x) {
    const int t = i / R;
    uint32_t v = 0;
    if (t < L) {
      const float x = en[i];
      const unsigned short h = cvt_bf16(x);
      v = (uint32_t)h | ((uint32_t)cvt_bf16(x - bf2f(h)) << 16);
    }
    hl[i] = v;
  }
  __syncthreads();
  // stage 2: B fragments.  Lane (tg, gq) needs K rows 2 tg, 2 tg + 1 (register 0) and 2 tg + 8, 2 tg + 9 (register 1)
  // of column r0 + gq at every time step; with the slot map above (H = hi, L = lo of the embedding row):
  //   tg 0: H[t] H[t+1] | L[t+3] L[t+4]      tg 1: H[t+2] H[t+3] | H[t] H[t+1]
  //   tg 2: H[t+4] L[t] | H[t+2] H[t+3]      tg 3: L[t+1] L[t+2] | H[t+4] 0
  for (int i = threadIdx.x; i < Tmax * R; i += blockDim.x) {
    const int r = i % R, t = i / R;
    const uint32_t* c = hl + (size_t)t * R + r;
    const uint32_t e0 = c[0], e1 = c[R], e2 = c[2 * R], e3 = c[3 * R], e4 = c[4 * R];
    const uint32_t H01 = __byte_perm(e0, e1, 0x5410), H23 = __byte_perm(e2, e3, 0x5410);    // lo halves = hi parts
    const uint32_t L34 = __byte_perm(e3, e4, 0x7632), L12 = __byte_perm(e1, e2, 0x7632);    // hi halves = lo parts
    const uint32_t H4L0 = __byte_perm(e4, e0, 0x7610), H4Z = e4 & 0xffffu;
    uint2* o = xb + (size_t)t * 4 * CM_XS + r;
    o[0 * CM_XS] = make_uint2(H01, L34);
    o[1 * CM_XS] = make_uint2(H23, H01);
    o[2 * CM_XS] = make_uint2(H4L0, H23);
    o[3 * CM_XS] = make_uint2(L12, H4Z);
  }
  // A fragments of this slice's weight blocks: one thread per (block, channel row) splits the row's f <= 5 taps once and
  // writes the 16 K slots [hi(5) | hi(5) | lo(5) | 0] as 8 bf16 pairs (channels past the group's end and taps past f
  // are zero)
  for (int i = threadIdx.x; i < nb * 16; i += blockDim.x) {
    const int bl = i >> 4, row = i & 15;
    int b = blk_lo + bl, gi = 0;
    while (gi + 1 < g.ngroups && b >= (g.n[gi] + 15) / 16) { b -= (g.n[gi] + 15) / 16; ++gi; }
    const int ch = b * 16 + row, f = g.f[gi];
    const bool live = ch < g.n[gi];
    uint32_t hi[CM_FMAX + 1], lo[CM_FMAX + 1];
#pragma unroll
    for (int k = 0; k < CM_FMAX; ++k) {
      const float w = (live && k < f) ? g.w[gi][ch * f + k] : 0.f;
      const unsigned short h = cvt_bf16(w);
      hi[k] = h;
      lo[k] = cvt_bf16(w - bf2f(h));
    }
    hi[CM_FMAX] = lo[CM_FMAX] = 0;
    uint32_t* o = wa + (size_t)(bl * 16 + row) * CM_WS;
    o[0] = hi[0] | (hi[1] << 16); o[1] = hi[2] | (hi[3] << 16); o[2] = hi[4] | (hi[0] << 16); o[3] = hi[1] | (hi[2] << 16);
    o[4] = hi[3] | (hi[4] << 16); o[5] = lo[0] | (lo[1] << 16); o[6] = lo[2] | (lo[3] << 16); o[7] = lo[4];
    bias_s[bl * 16 + row] = live ? g.b[gi][ch] : 0.f;
    if (row == 0) meta[bl] = make_int4(g.col0[gi] + b * 16, min(16, g.n[gi] - b * 16), f, 0);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int gq = lane >> 2, tg = lane & 3;
  // work units: (representation block of 8, pair of channel blocks with the same filter size)
  for (int rb = warp; rb < R / 8; rb += nwarps) {
    const uint2* xs = xb + (size_t)tg * CM_XS + rb * 8 + gq;
    const size_t row0 = (size_t)n * R + rb * 8;
    int b = 0;
    while (b < nb) {
      const int f = meta[b].z;
      const int T = L - f + 1;
      if (b + 1 < nb && meta[b + 1].z == f) {
        conv_mma_unit<2>(xs, wa, bias_s, meta, b, T, gq, tg, row0, F, pooled, arg, pooled_bf, Fp);
        b += 2;
      } else {
        conv_mma_unit<1>(xs, wa, bias_s, meta, b, T, gq, tg, row0, F, pooled, arg, pooled_bf, Fp);
        b += 1;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// backward of conv + ReLU + max-pool, two kernels (both stream dx / pooled / arg once, coalesced):
//
//  (a) conv_pool_bwd_demb_kernel: one warp per (caption n, representation r) row of [N*R, F].  Lanes stride over
//      the feature columns; every lane accumulates into its OWN copy of demb[n, :, r*es .. r*es+es) in shared
//      memory (layout [entry][lane]: bank = lane, so plain read-modify-write, no atomics), then the 32 copies
//      are summed with a rotated conflict-free read.
//  (b) conv_pool_bwd_dw_kernel: thread = feature column, CTA = chunk of rows; conv-weight / bias gradients
//      accumulate in registers over the chunk, one global atomic per weight per CTA.
// ---------------------------------------------------------------------------------------
constexpr int BWD_KMAX = 8;      // f * es <= 8 on the register path

// (a) demb.  One warp per (caption n, representation r) row of [N*R, F].  Each lane owns groups of 4 consecutive
// feature columns (float4 / uchar4 loads, all of a row's loads issued before any use); every lane accumulates into
// its OWN copy of demb[n, :, r*es .. r*es+es) in shared memory (layout [entry][lane]: bank = lane, plain
// read-modify-write, no atomics), then the 32 copies are summed with a rotated conflict-free read.
// VEC requires F % 4 == 0 and every filter group a multiple of 4 columns wide (a float4 never straddles groups).
template <bool ES1, bool VEC>
__global__ void __launch_bounds__(256)
conv_pool_bwd_demb_kernel(const uint8_t* __restrict__ arg, const float* __restrict__ dx, const float* __restrict__ dx2,
                          int rows /*N*R*/, int L, int De, int R, int es, ConvGroups g, float* __restrict__ demb) {
  extern __shared__ __align__(16) float sm[];
  const int F = g.F, kmax = g.kmax;
  const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int LE = L * es;                       // entries of one (n, r) slice of demb
  float* wk_s = sm;                            // [kmax][F]
  int* fk_s = reinterpret_cast<int*>(wk_s + kmax * F);        // [F]
  float* priv = reinterpret_cast<float*>(fk_s + F) + (size_t)warp * LE * 32;   // [LE][32] per warp
  for (int gi = 0; gi < g.ngroups; ++gi) {
    const int fk = g.f[gi] * es;
    for (int i = threadIdx.x; i < g.n[gi] * kmax; i += blockDim.x) {
      const int c = i / kmax, k = i % kmax;
      wk_s[k * F + g.col0[gi] + c] = (k < fk) ? g.w[gi][c * fk + k] : 0.f;
    }
    for (int c = threadIdx.x; c < g.n[gi]; c += blockDim.x) fk_s[g.col0[gi] + c] = fk;
  }
  __syncthreads();
  for (int row = blockIdx.x * nwarps + warp; row < rows; row += gridDim.x * nwarps) {
    const int n = row / R, r = row % R;
    for (int e = 0; e < LE; ++e) priv[e * 32 + lane] = 0.f;
    const size_t base = (size_t)row * F;
    if (VEC) {
      const int F4 = F >> 2;
      const float4* dx4 = reinterpret_cast<const float4*>(dx + base);
      const float4* dy4 = reinterpret_cast<const float4*>(dx2 + base);
      const uint32_t* a4 = reinterpret_cast<const uint32_t*>(arg + base);
      for (int q0 = 0; q0 < F4; q0 += 128) {   // 4 float4 groups per lane in flight
        float4 gv[4], hv[4];
        uint32_t av[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int q = q0 + j * 32 + lane;
          const bool ok = q < F4;
          gv[j] = ok ? dx4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
          hv[j] = ok ? dy4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
          av[j] = ok ? __ldg(a4 + q) : 0xffffffffu;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) { gv[j].x += hv[j].x; gv[j].y += hv[j].y; gv[j].z += hv[j].z; gv[j].w += hv[j].w; }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int q = q0 + j * 32 + lane;
          if (q >= F4) continue;
          const int c = q << 2;
          const int fk = fk_s[c];
          const float gg[4] = {gv[j].x, gv[j].y, gv[j].z, gv[j].w};
          const int aa[4] = {(int)(av[j] & 0xffu), (int)((av[j] >> 8) & 0xffu), (int)((av[j] >> 16) & 0xffu), (int)(av[j] >> 24)};
          bool on[4];
          bool any = false;
#pragma unroll
          for (int e4 = 0; e4 < 4; ++e4) { on[e4] = (aa[e4] != ARG_DEAD) && (gg[e4] != 0.f); any |= on[e4]; }
          if (!any) continue;
          for (int k = 0; k < fk; ++k) {
            const float4 w4 = *reinterpret_cast<const float4*>(&wk_s[k * F + c]);   // conflict-free LDS.128
            const float ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
              if (on[e4]) {
                const int e = ES1 ? (aa[e4] + k) : ((aa[e4] + k / es) * es + k % es);
                priv[e * 32 + lane] = fmaf(ww[e4], gg[e4], priv[e * 32 + lane]);
              }
            }
          }
        }
      }
    } else {
      for (int c0 = 0; c0 < F; c0 += 128) {      // 4 columns per lane in flight
        float gv[4];
        int av[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = c0 + j * 32 + lane;
          const bool ok = c < F;
          gv[j] = ok ? dx[base + c] + dx2[base + c] : 0.f;
          av[j] = ok ? (int)arg[base + c] : ARG_DEAD;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = c0 + j * 32 + lane;
          if (c < F && av[j] != ARG_DEAD && gv[j] != 0.f) {
            const int fk = fk_s[c];
            for (int k = 0; k < fk; ++k) {
              const int e = ES1 ? (av[j] + k) : ((av[j] + k / es) * es + k % es);
              priv[e * 32 + lane] = fmaf(wk_s[k * F + c], gv[j], priv[e * 32 + lane]);
            }
          }
        }
      }
    }
    __syncwarp();
    // sum the 32 lane-private copies: lane handles entries e = lane, lane+32, ...; rotated column order
    for (int e = lane; e < LE; e += 32) {
      float acc = 0.f;
#pragma unroll 8
      for (int i = 0; i < 32; ++i) acc += priv[e * 32 + ((i + lane) & 31)];
      const int t = ES1 ? e : e / es, ee = ES1 ? 0 : e % es;
      demb[((size_t)n * L + t) * De + r * es + ee] = acc;
    }
    __syncwarp();
  }
}

// (b) conv-weight / bias gradients.  Thread = feature column, CTA = chunk of rows processed RC rows at a time: the
// RC rows' embedding slices emb[n, :, r*es..] (L*es floats each) are staged in shared memory first, so the gather
// emb[arg + k] is a shared-memory read instead of L2 traffic; dx / arg loads of all RC rows are issued before use.
// Weight gradients accumulate in registers over the chunk, one global atomic per weight per CTA.
constexpr int DW_RC = 8;
template <bool ES1>
__global__ void __launch_bounds__(256)
conv_pool_bwd_dw_kernel(const float* __restrict__ emb, const uint8_t* __restrict__ arg, const float* __restrict__ dx,
                        const float* __restrict__ dx2, int rows, int L, int De, int R, int es, ConvGroups g,
                        int rows_per_cta) {
  extern __shared__ __align__(16) float sm[];   // [DW_RC][L*es]
  const int F = g.F, LE = L * es;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = c < F;
  int gi = 0;
  while (gi + 1 < g.ngroups && c >= g.col0[gi + 1]) ++gi;
  const int cin = c - g.col0[gi], fk = g.f[gi] * es;
  float dw[BWD_KMAX];
#pragma unroll
  for (int k = 0; k < BWD_KMAX; ++k) dw[k] = 0.f;
  float dbias = 0.f;
  const int r0 = blockIdx.y * rows_per_cta, r1 = min(rows, r0 + rows_per_cta);
  for (int rb = r0; rb < r1; rb += DW_RC) {
    __syncthreads();
    for (int i = threadIdx.x; i < DW_RC * LE; i += blockDim.x) {
      const int j = i / LE, e = i % LE, row = rb + j;
      if (row < r1) {
        const int n = row / R, r = row % R;
        sm[i] = emb[((size_t)n * L + e / es) * De + r * es + e % es];
      }
    }
    float gv[DW_RC];
    int av[DW_RC];
#pragma unroll
    for (int j = 0; j < DW_RC; ++j) {
      const int row = rb + j;
      const bool ok = active && row < r1;
      const size_t i = (size_t)row * F + c;
      gv[j] = ok ? dx[i] + dx2[i] : 0.f;
      av[j] = ok ? (int)arg[i] : ARG_DEAD;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < DW_RC; ++j) {
      if (av[j] != ARG_DEAD && gv[j] != 0.f) {
        const float* e0 = sm + j * LE + av[j] * es;
#pragma unroll
        for (int k = 0; k < BWD_KMAX; ++k)
          if (k < fk) dw[k] = fmaf(gv[j], e0[k], dw[k]);
        dbias += gv[j];
      }
    }
  }
  if (!active) return;
#pragma unroll
  for (int k = 0; k < BWD_KMAX; ++k)
    if (k < fk) atomicAdd(g.dw[gi] + cin * fk + k, dw[k]);
  atomicAdd(g.db[gi] + cin, dbias);
}

// ---------------------------------------------------------------------------------------
// score head.  feature2out (F->100) and out2logits (100->1) have no nonlinearity between them
// (src/discriminator.py:58-60), so logits = yd . w_eff + b_eff with
//   w_eff[j] = sum_k w_o[k] W_f[k, j],  b_eff = sum_k w_o[k] b_f[k] + b_o.
// ---------------------------------------------------------------------------------------
// grid = ceil((F+1)/32) CTAs of 256 threads: lane = column, the 8 warps split the Hd rows (coalesced 128-byte reads of
// W_f rows, 8 x fewer dependent FMAs per thread than one thread per column), fixed-order reduction in shared memory.
__global__ void __launch_bounds__(256)
head_collapse_kernel(const float* __restrict__ W_f, const float* __restrict__ b_f,
                     const float* __restrict__ w_o, const float* __restrict__ b_o, int F,
                     int Hd, float* __restrict__ weff /*[F+1]*/) {
  __shared__ float part[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (j < F) {
#pragma unroll 4
    for (int k = w; k < Hd; k += 8) s = fmaf(w_o[k], W_f[(size_t)k * F + j], s);
  } else if (j == F) {
    for (int k = w; k < Hd; k += 8) s = fmaf(w_o[k], b_f[k], s);
  }
  part[w][lane] = s;
  __syncthreads();
  if (w == 0 && j <= F) {
    float t = (j == F) ? b_o[0] : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += part[i][lane];
    weff[j] = t;
  }
}

// tensor-core modes: exp and reciprocal on the MUFU unit (2 ulp each); the exact-fp32 mode keeps expf and the IEEE division
template <bool FAST>
__device__ __forceinline__ float sigmoid_sel(float x) {
  if (FAST) return __fdividef(1.0f, 1.0f + __expf(-x));
  return sigmoidf_acc(x);
}

constexpr int MAX_HEADS = 4;
struct HeadPtrs {
  const uint8_t* keep[MAX_HEADS];
  float* logits[MAX_HEADS];
  int n;
};

// highway mix + dropout + collapsed head; one warp per row (row = n*R + r).
//   y = sig(h) relu(h) + (1 - sig(h)) x          (src/discriminator.py:55)
__global__ void __launch_bounds__(256)
head_fwd_kernel(const float* __restrict__ hpre, const float* __restrict__ pooled, int rows, int F,
                const float* __restrict__ weff, float drop_scale, HeadPtrs hp) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float acc[MAX_HEADS] = {0.f, 0.f, 0.f, 0.f};
  const size_t base = (size_t)row * F;
  for (int j = lane; j < F; j += 32) {
    const float h = hpre[base + j], x = pooled[base + j];
    const float sg = sigmoidf_acc(h);
    const float y = sg * fmaxf(h, 0.f) + (1.f - sg) * x;
    const float yw = y * weff[j];
#pragma unroll
    for (int m = 0; m < MAX_HEADS; ++m)
      if (m < hp.n) acc[m] += hp.keep[m] ? (hp.keep[m][base + j] ? yw : 0.f) : yw;
  }
#pragma unroll
  for (int m = 0; m < MAX_HEADS; ++m) {
    if (m < hp.n) {
      const float s = warp_sum(acc[m]);
      if (lane == 0) hp.logits[m][row] = s * (hp.keep[m] ? drop_scale : 1.f) + weff[F];
    }
  }
}

// float4 variant of head_fwd_kernel for F % 4 == 0: one warp per row, every lane issues all of its loads of the row
// (up to NQ float4 of hpre and pooled plus the uchar4 mask words) before the first use.
template <int NQ, bool FAST>
__global__ void __launch_bounds__(256)
head_fwd_vec_kernel(const float* __restrict__ hpre, const float* __restrict__ pooled, int rows, int F,
                    const float* __restrict__ weff, float drop_scale, HeadPtrs hp) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int F4 = F >> 2;
  const size_t base = (size_t)row * F;
  const float4* h4 = reinterpret_cast<const float4*>(hpre + base);
  const float4* x4 = reinterpret_cast<const float4*>(pooled + base);
  const float4* w4 = reinterpret_cast<const float4*>(weff);
  float4 hv[NQ], xv[NQ];
  uint32_t kv[MAX_HEADS][NQ];      // raw 4-byte mask words: unpacking at load time would serialise the loads
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    const int q = lane + 32 * i;
    const bool ok = q < F4;
    hv[i] = ok ? h4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    xv[i] = ok ? x4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int m = 0; m < MAX_HEADS; ++m)
      if (m < hp.n && hp.keep[m]) kv[m][i] = ok ? __ldg(reinterpret_cast<const uint32_t*>(hp.keep[m] + base) + q) : 0u;
  }
  float acc[MAX_HEADS] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    const int q = lane + 32 * i;
    if (q < F4) {
      const float4 ww = __ldg(w4 + q);
      const float hh[4] = {hv[i].x, hv[i].y, hv[i].z, hv[i].w};
      const float xx[4] = {xv[i].x, xv[i].y, xv[i].z, xv[i].w};
      const float wv[4] = {ww.x, ww.y, ww.z, ww.w};
      float yw[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float sg = sigmoid_sel<FAST>(hh[e]);
        yw[e] = (sg * fmaxf(hh[e], 0.f) + (1.f - sg) * xx[e]) * wv[e];
      }
#pragma unroll
      for (int m = 0; m < MAX_HEADS; ++m) {
        if (m < hp.n) {
          if (hp.keep[m]) {
            const uint32_t k = kv[m][i];
            acc[m] += ((k & 0xffu) ? yw[0] : 0.f) + ((k & 0xff00u) ? yw[1] : 0.f) + ((k & 0xff0000u) ? yw[2] : 0.f) +
                      ((k & 0xff000000u) ? yw[3] : 0.f);
          } else {
            acc[m] += (yw[0] + yw[1]) + (yw[2] + yw[3]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MAX_HEADS; ++m) {
    if (m < hp.n) {
      const float s = warp_sum(acc[m]);
      if (lane == 0) hp.logits[m][row] = s * (hp.keep[m] ? drop_scale : 1.f) + weff[F];
    }
  }
}

// float4 variant of head_bwd_kernel (F % 4 == 0): thread = 4 consecutive feature columns, CTA = row chunk, 4 rows of
// loads in flight per thread.
// DH_BF16: dh is written as bf16 with row pitch Fp (it is only read by tensor-core contractions in GIC_GEMM_BF16 mode)
template <bool DH_BF16>
__global__ void __launch_bounds__(256)
head_bwd_vec_kernel(const float* __restrict__ dlogit, const uint8_t* __restrict__ keep, float drop_scale,
                    const float* __restrict__ hpre, const float* __restrict__ pooled, int rows, int F,
                    const float* __restrict__ weff, int rows_per_cta, float* __restrict__ dh,
                    float* __restrict__ dx, float* __restrict__ s_acc, float* __restrict__ dbh_acc, int Fp) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;      // float4 column group
  const int F4 = F >> 2;
  if (q >= F4) return;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(rows, r0 + rows_per_cta);
  const float4 w4 = reinterpret_cast<const float4*>(weff)[q];
  const float wj[4] = {w4.x, w4.y, w4.z, w4.w};
  const float sc = keep ? drop_scale : 1.f;
  float s[4] = {0.f, 0.f, 0.f, 0.f}, sb[4] = {0.f, 0.f, 0.f, 0.f};
  for (int rb = r0; rb < r1; rb += 4) {
    float4 hv[4], xv[4];
    uint32_t kv[4];
    float dl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = rb + j;
      const bool ok = r < r1;
      const size_t i = (size_t)r * F4 + q;
      hv[j] = ok ? reinterpret_cast<const float4*>(hpre)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      xv[j] = ok ? reinterpret_cast<const float4*>(pooled)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      kv[j] = (ok && keep) ? __ldg(reinterpret_cast<const uint32_t*>(keep) + i) : 0x01010101u;
      dl[j] = ok ? dlogit[r] * sc : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = rb + j;
      if (r >= r1) break;
      const float hh[4] = {hv[j].x, hv[j].y, hv[j].z, hv[j].w};
      const float xx[4] = {xv[j].x, xv[j].y, xv[j].z, xv[j].w};
      const float kp[4] = {(kv[j] & 0xffu) ? 1.f : 0.f, (kv[j] & 0xff00u) ? 1.f : 0.f, (kv[j] & 0xff0000u) ? 1.f : 0.f,
                           (kv[j] & 0xff000000u) ? 1.f : 0.f};
      float dhv[4], dxv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float sg = sigmoid_sel<DH_BF16>(hh[e]);      // DH_BF16 <=> GIC_GEMM_BF16 mode
        const float rl = fmaxf(hh[e], 0.f);
        const float y = sg * rl + (1.f - sg) * xx[e];
        const float dy = dl[j] * kp[e] * wj[e];
        s[e] = fmaf(dl[j] * kp[e], y, s[e]);
        dhv[e] = dy * (sg * (1.f - sg) * (rl - xx[e]) + (hh[e] > 0.f ? sg : 0.f));
        dxv[e] = dy * (1.f - sg);
        sb[e] += dhv[e];
      }
      const size_t i = (size_t)r * F4 + q;
      if (DH_BF16) {
        uint2 pk;
        pk.x = (unsigned int)cvt_bf16(dhv[0]) | ((unsigned int)cvt_bf16(dhv[1]) << 16);
        pk.y = (unsigned int)cvt_bf16(dhv[2]) | ((unsigned int)cvt_bf16(dhv[3]) << 16);
        *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(dh) + (size_t)r * Fp + 4 * q) = pk;
      } else {
        reinterpret_cast<float4*>(dh)[i] = make_float4(dhv[0], dhv[1], dhv[2], dhv[3]);
      }
      reinterpret_cast<float4*>(dx)[i] = make_float4(dxv[0], dxv[1], dxv[2], dxv[3]);
    }
  }
  // one 16-byte vector reduction per accumulator (the scalar version issued 8 atomics per thread: with 820 CTAs the
  // 1.5 M atomics on 1 800 addresses were a visible tail)
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(s_acc + 4 * q), "f"(s[0]), "f"(s[1]), "f"(s[2]), "f"(s[3]) : "memory");
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dbh_acc + 4 * q), "f"(sb[0]), "f"(sb[1]), "f"(sb[2]), "f"(sb[3]) : "memory");
}

// backward of head + dropout + highway for one head.  Thread = feature column, CTA = row chunk.
// Writes dh (gradient at the highway pre-activation) and the direct part of dx; accumulates
// s[j] = sum_r dlogit_r * yd[r,j] and dbh[j] = sum_r dh[r,j] with one atomic per thread.
__global__ void __launch_bounds__(256)
head_bwd_kernel(const float* __restrict__ dlogit, const uint8_t* __restrict__ keep, float drop_scale,
                const float* __restrict__ hpre, const float* __restrict__ pooled, int rows, int F,
                const float* __restrict__ weff, int rows_per_cta, float* __restrict__ dh,
                float* __restrict__ dx, float* __restrict__ s_acc, float* __restrict__ dbh_acc) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= F) return;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(rows, r0 + rows_per_cta);
  const float wj = weff[j];
  const float sc = keep ? drop_scale : 1.f;
  float s = 0.f, sb = 0.f;
  for (int r = r0; r < r1; ++r) {
    const size_t i = (size_t)r * F + j;
    const float dl = dlogit[r] * sc;
    const float kp = keep ? (keep[i] ? 1.f : 0.f) : 1.f;
    const float h = hpre[i], x = pooled[i];
    const float sg = sigmoidf_acc(h);
    const float rl = fmaxf(h, 0.f);
    const float y = sg * rl + (1.f - sg) * x;
    const float dy = dl * kp * wj;
    s = fmaf(dl * kp, y, s);
    const float dhv = dy * (sg * (1.f - sg) * (rl - x) + (h > 0.f ? sg : 0.f));
    dh[i] = dhv;
    dx[i] = dy * (1.f - sg);
    sb += dhv;
  }
  atomicAdd(s_acc + j, s);
  atomicAdd(dbh_acc + j, sb);
}

// parameter gradients of the collapsed head, expanded back to the reference's tensors:
//   dW_f[k,j] = w_o[k] s[j];  db_f[k] = w_o[k] S;  dw_o[k] = sum_j W_f[k,j] s[j] + b_f[k] S;
//   db_o = S;  db_h[j] = dbh[j]          with S = sum_r dlogit_r.
// grid = Hd CTAs (one per hidden unit k of feature2out).
__global__ void __launch_bounds__(256)
head_param_grads_kernel(const float* __restrict__ dlogit, int rows, const float* __restrict__ s_acc,
                        const float* __restrict__ dbh_acc, const float* __restrict__ W_f,
                        const float* __restrict__ b_f, const float* __restrict__ w_o, int F, int Hd,
                        float beta, float* __restrict__ dW_f, float* __restrict__ db_f,
                        float* __restrict__ dw_o, float* __restrict__ db_o, float* __restrict__ db_h) {
  __shared__ float red[32];
  const int k = blockIdx.x;
  // eight loads in flight per thread (one dependent L2 round trip per element made this 100-CTA kernel 30 us long); the
  // order of the partial sums is fixed, so every CTA gets the same S
  float S = 0.f;
  for (int r0 = threadIdx.x; r0 < rows; r0 += 8 * blockDim.x) {
    float t[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = r0 + u * blockDim.x;
      t[u] = (r < rows) ? __ldg(dlogit + r) : 0.f;
    }
    S += ((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]));
  }
  S = block_sum(S, red);
  const float wo = w_o[k];
  float dot = 0.f;
  for (int j = threadIdx.x; j < F; j += blockDim.x) {
    const float sj = s_acc[j];
    const size_t i = (size_t)k * F + j;
    dW_f[i] = (beta != 0.f ? beta * dW_f[i] : 0.f) + wo * sj;
    dot = fmaf(W_f[i], sj, dot);
    if (k == 0) db_h[j] = (beta != 0.f ? beta * db_h[j] : 0.f) + dbh_acc[j];
  }
  dot = block_sum(dot, red);
  if (threadIdx.x == 0) {
    db_f[k] = (beta != 0.f ? beta * db_f[k] : 0.f) + wo * S;
    dw_o[k] = (beta != 0.f ? beta * dw_o[k] : 0.f) + dot + b_f[k] * S;
    if (k == 0) db_o[0] = (beta != 0.f ? beta * db_o[0] : 0.f) + S;
  }
}

__global__ void scale_kernel(float* __restrict__ p, size_t n, float a) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    p[i] = (a == 0.f) ? 0.f : p[i] * a;
}
int scale_inplace(float* p, size_t n, float a, cudaStream_t s) {
  if (n == 0 || a == 1.f) return GIC_OK;
  if (a == 0.f) {
    cudaError_t e = cudaMemsetAsync(p, 0, n * sizeof(float), s);
    if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
    return GIC_OK;
  }
  scale_kernel<<<min(cdiv((long long)n, 256), 4 * num_sms()), 256, 0, s>>>(p, n, a);
  return check_launch("scale_kernel");
}

// ---------------------------------------------------------------------------------------
// host-side composition
// ---------------------------------------------------------------------------------------
struct DiscDims {
  int N, L, V, De, R, es, F, Hd, ngroups, kmax;
  size_t rows() const { return (size_t)N * R; }
};

int disc_fill_groups(ConvGroups& g, int ngroups, const int* fs, const int* nf, const float* const* cw,
                     const float* const* cb, float* const* dcw, float* const* dcb, int es) {
  GIC_REQUIRE(ngroups >= 1 && ngroups <= MAX_GROUPS, GIC_ERR_SHAPE, "disc: 1..%d filter groups supported", MAX_GROUPS);
  g.ngroups = ngroups; g.F = 0; g.kmax = 0;
  for (int i = 0; i < MAX_GROUPS; ++i) { g.w[i] = g.b[i] = nullptr; g.dw[i] = g.db[i] = nullptr; g.f[i] = g.n[i] = g.col0[i] = 0; }
  for (int i = 0; i < ngroups; ++i) {
    GIC_REQUIRE(fs[i] >= 1 && nf[i] >= 1, GIC_ERR_SHAPE, "disc: bad filter group %d", i);
    GIC_REQUIRE(cw[i] && cb[i], GIC_ERR_NULL, "disc: NULL conv weights for group %d", i);
    g.w[i] = cw[i]; g.b[i] = cb[i];
    g.dw[i] = dcw ? dcw[i] : nullptr; g.db[i] = dcb ? dcb[i] : nullptr;
    g.f[i] = fs[i]; g.n[i] = nf[i]; g.col0[i] = g.F; g.F += nf[i];
    if (fs[i] * es > g.kmax) g.kmax = fs[i] * es;
  }
  return GIC_OK;
}

// Derived weights shared by every discriminator call of one step (collapsed head, bf16 copy of highway.weight):
// layout = the forward workspace (DiscFwdWs).  While a prepared blob is registered the forward /
// backward read it instead of recomputing (one adversarial step makes 2 forward and 3 backward calls on the same
// pre-update weights, SURVEY.md Q1).
void disc_set_prepared(const float* prep) { ctx().prepared = prep; }
#define g_prepared (ctx().prepared)

int disc_prepare(int mode, const float* W_h, const float* W_f, const float* b_f, int Hd, const float* W_o,
                 const float* b_o, int F, float* prep, cudaStream_t s) {
  GIC_REQUIRE(W_h && W_f && b_f && W_o && b_o && prep, GIC_ERR_NULL, "disc_prepare: NULL pointer");
  GIC_REQUIRE(F >= 1 && Hd >= 1, GIC_ERR_SHAPE, "disc_prepare: bad shape");
  const DiscFwdWs w(F);
  head_collapse_kernel<<<cdiv(F + 1, 32), 256, 0, s>>>(W_f, b_f, W_o, b_o, F, Hd, prep + w.weff);
  GIC_TRY(check_launch("head_collapse_kernel"));
  if (mode == GEMM_BF16 && (F % 4 == 0)) {
    unsigned short* W_h_bf = reinterpret_cast<unsigned short*>(prep + w.W_h_bf);
    GIC_TRY(f32_to_bf16(W_h, F, F, F, W_h_bf, bf_pitch(F), s));
  }
  return GIC_OK;
}

int disc_forward(int mode, const float* inp_soft, const int64_t* ids, const DiscDims& d, const ConvGroups& g,
                 const float* W_e, const float* W_h, const float* b_h, const float* W_f, const float* b_f,
                 const float* W_o, const float* b_o, int n_heads, const uint8_t* const* keep, float drop_p,
                 float* const* logits, float* saved, float* ws, cudaStream_t s) {
  const size_t rows = d.rows();
  const DiscSaved sv(d.N, d.L, d.De, d.R, d.F);
  const DiscFwdWs w(d.F);
  float* emb = saved + sv.emb;
  float* pooled = saved + sv.pooled;
  float* hpre = saved + sv.hpre;
  uint8_t* arg = reinterpret_cast<uint8_t*>(saved + sv.arg);
  const bool bf = (mode == GEMM_BF16) && (d.F % 4 == 0);
  const int Fp = bf_pitch(d.F);
  unsigned short* pooled_bf = reinterpret_cast<unsigned short*>(saved + sv.pooled_bf);
  const float* prep = g_prepared;
  const float* derived = prep ? prep : ws;          // the prepared blob has the forward workspace's layout
  const float* weff = derived + w.weff;
  const unsigned short* W_h_bf = reinterpret_cast<const unsigned short*>(derived + w.W_h_bf);
  if (d.N == 0) return GIC_OK;
  // 1. embedding
  if (inp_soft) {
    GIC_TRY(gemm(mode, false, true, d.N * d.L, d.De, d.V, 1.f, inp_soft, d.V, W_e, d.V, 0.f, emb, d.De, nullptr, s));
  } else {
    const int tot = d.N * d.L * d.De;
    disc_embed_ids_kernel<<<cdiv(tot, 256), 256, 0, s>>>(ids, d.N * d.L, d.V, d.De, W_e, emb);
    GIC_TRY(check_launch("disc_embed_ids_kernel"));
  }
  // 2. conv + relu + max-pool
  {
    GIC_REQUIRE(g.kmax <= 16, GIC_ERR_SHAPE, "disc: filter_size*emb_dim_single <= 16 supported");
    GIC_REQUIRE(d.L <= 254, GIC_ERR_SHAPE, "disc: caption length <= 254 supported");
    // column slices: enough CTAs to balance the SMs (>= ~6 per SM), slice width a multiple of 32
    int slices = max(1, min(cdiv(6 * num_sms(), d.N), cdiv(d.F, 32)));
    int cs = ((cdiv(d.F, slices) + 31) / 32) * 32;
    slices = cdiv(d.F, cs);
    const size_t smem = (((size_t)d.L * d.De + 3) & ~(size_t)3) * 4 + ((size_t)g.kmax + 2) * cs * 4;
    GIC_REQUIRE(smem <= 200 * 1024, GIC_ERR_SHAPE, "disc: conv tile needs %zu B of shared memory", smem);
    ProfScope prof(PROF_CONVPOOL, 5.0 * rows * d.F + 4.0 * d.N * d.L * d.De, s);   // write pooled f32 + arg u8, read emb
    const bool es1 = (d.es == 1) && (d.R % 4 == 0) && g.kmax <= 8;
    static bool attr = false;
    if (!attr) {
      cudaFuncSetAttribute(conv_pool_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaFuncSetAttribute(conv_pool_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      attr = true;
    }
    unsigned short* pbf = bf ? pooled_bf : nullptr;
    // tensor-core modes: mma.sync formulation (bf16 hi/lo split along K, one HMMA per step); GIC_CONV_MMA=0 keeps the
    // CUDA-core kernel
    int fmin = g.kmax;
    for (int i = 0; i < g.ngroups; ++i) fmin = min(fmin, g.f[i]);
    bool use_mma = (mode == GEMM_TF32 || mode == GEMM_BF16) && d.es == 1 && d.De == d.R && (d.R % 8 == 0) && g.kmax <= CM_FMAX &&
                   d.L >= g.kmax && d.L - fmin + 1 <= 32;
    if (option("GIC_CONV_MMA", 1) == 0) use_mma = false;
    if (use_mma) {
      const int nblocks = conv_mma_blocks(g);
      const int Tmax = d.L - fmin + 1;
      // slices: enough CTAs to balance the SMs, and at least two so that a CTA's weight fragments leave room for a second
      // resident CTA next to the B-fragment table (measured: c5 shape 3.09 ms with one slice, 2.63 ms with two)
      int sl = max(1, min(max(2, cdiv(4 * num_sms(), d.N)), nblocks));
      { const int o = option("GIC_CONV_MMA_SLICES", 0); if (o > 0) sl = min(o, nblocks); }   // tuning
      const int bps = cdiv(nblocks, sl);
      sl = cdiv(nblocks, bps);
      const size_t msmem = (size_t)Tmax * 4 * CM_XS * 8 + (size_t)bps * 16 * CM_WS * 4 + (size_t)bps * 16 * 4 + (size_t)bps * 16 +
                           (size_t)(Tmax + 4) * d.R * 4;
      if (msmem <= 200 * 1024) {
        static bool mattr = false;
        if (!mattr) { cudaFuncSetAttribute(conv_pool_fwd_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); mattr = true; }
        conv_pool_fwd_mma_kernel<<<dim3(d.N, sl), 256, msmem, s>>>(emb, d.L, d.R, g, bps, nblocks, Tmax, pooled, arg, pbf, Fp);
        GIC_TRY(check_launch("conv_pool_fwd_mma_kernel"));
      } else {
        use_mma = false;
      }
    }
    if (!use_mma) {
      if (es1) conv_pool_fwd_kernel<true><<<dim3(d.N, slices), 256, smem, s>>>(emb, d.L, d.De, d.R, d.es, g, cs, pooled, arg, pbf, Fp);
      else conv_pool_fwd_kernel<false><<<dim3(d.N, slices), 256, smem, s>>>(emb, d.L, d.De, d.R, d.es, g, cs, pooled, arg, pbf, Fp);
      GIC_TRY(check_launch("conv_pool_fwd_kernel"));
    }
  }
  // 3. highway pre-activation
  if (bf) {
    // bf16 operands: pooled_bf written by the conv kernel, W_h converted here (1.6 MB); fp32 accumulate / output
    if (!prep) GIC_TRY(f32_to_bf16(W_h, d.F, d.F, d.F, const_cast<unsigned short*>(W_h_bf), Fp, s));
    GIC_TRY(gemm_bf16(false, true, (int)rows, d.F, d.F, 1.f, pooled_bf, Fp, W_h_bf, Fp, 0.f, hpre, d.F, b_h, s, PROF_GEMM_D));
  } else {
    GIC_TRY(gemm(mode, false, true, (int)rows, d.F, d.F, 1.f, pooled, d.F, W_h, d.F, 0.f, hpre, d.F, b_h, s, PROF_GEMM_D));
  }
  // 4. collapsed head
  if (!prep) {
    head_collapse_kernel<<<cdiv(d.F + 1, 32), 256, 0, s>>>(W_f, b_f, W_o, b_o, d.F, d.Hd, ws + w.weff);
    GIC_TRY(check_launch("head_collapse_kernel"));
  }
  HeadPtrs hp;
  hp.n = n_heads;
  for (int m = 0; m < MAX_HEADS; ++m) {
    hp.keep[m] = (m < n_heads && keep) ? keep[m] : nullptr;
    hp.logits[m] = (m < n_heads) ? logits[m] : nullptr;
  }
  ProfScope prof(PROF_HEAD, (8.0 + n_heads) * rows * d.F, s);      // read hpre, pooled (f32) + one u8 mask per head
  bool vec = (d.F % 4 == 0) && d.F <= 4 * 32 * 8;
  for (int m = 0; m < n_heads; ++m) vec = vec && (!hp.keep[m] || (reinterpret_cast<uintptr_t>(hp.keep[m]) & 3u) == 0);
  if (vec) {
    const int nq = cdiv(d.F / 4, 32);
    const int grid = cdiv((long long)rows, 8);
    const float dsc = 1.f / (1.f - drop_p);
    const bool fast = (mode == GEMM_TF32 || mode == GEMM_BF16);
#define GIC_HF(NQ_) do { if (fast) head_fwd_vec_kernel<NQ_, true><<<grid, 256, 0, s>>>(hpre, pooled, (int)rows, d.F, weff, dsc, hp); \
                         else head_fwd_vec_kernel<NQ_, false><<<grid, 256, 0, s>>>(hpre, pooled, (int)rows, d.F, weff, dsc, hp); } while (0)
    if (nq <= 2) GIC_HF(2); else if (nq <= 4) GIC_HF(4); else GIC_HF(8);
#undef GIC_HF
  } else {
    head_fwd_kernel<<<cdiv((long long)rows, 8), 256, 0, s>>>(hpre, pooled, (int)rows, d.F, weff, 1.f / (1.f - drop_p), hp);
  }
  return check_launch("head_fwd_kernel");
}

int disc_backward(int mode, const float* dlogit, const uint8_t* keep, float drop_p, const float* inp_soft,
                  const int64_t* ids, const DiscDims& d, ConvGroups& g, const float* W_e, const float* W_h,
                  const float* W_f, const float* b_f, const float* W_o, const float* b_o, const float* saved,
                  float* ws, float* dW_e, float* dW_h, float* db_h, float* dW_f, float* db_f, float* dW_o,
                  float* db_o, float* dinp, int want_param, int accumulate, cudaStream_t s) {
  const size_t rows = d.rows();
  if (d.N == 0) return GIC_OK;
  const DiscSaved sv(d.N, d.L, d.De, d.R, d.F);
  const DiscBwdWs w(d.N, d.L, d.De, d.R, d.F);
  const DiscFwdWs pw(d.F);                          // layout of the prepared blob
  const float* emb = saved + sv.emb;
  const float* pooled = saved + sv.pooled;
  const float* hpre = saved + sv.hpre;
  const uint8_t* arg = reinterpret_cast<const uint8_t*>(saved + sv.arg);
  const bool bf = (mode == GEMM_BF16) && (d.F % 4 == 0) && (!keep || (reinterpret_cast<uintptr_t>(keep) & 3u) == 0);
  const int Fp = bf_pitch(d.F);
  const unsigned short* pooled_bf = reinterpret_cast<const unsigned short*>(saved + sv.pooled_bf);
  const float* prep = g_prepared;
  const float* weff = prep ? prep + pw.weff : ws + w.weff;
  float* dh = ws + w.dh;
  float* dx = ws + w.dx;
  float* sacc = ws + w.s;
  float* dbh = ws + w.dbh;
  float* demb = ws + w.demb;
  unsigned short* W_h_bf_ws = reinterpret_cast<unsigned short*>(ws + w.W_h_bf);
  const unsigned short* W_h_bf = prep ? reinterpret_cast<const unsigned short*>(prep + pw.W_h_bf) : W_h_bf_ws;
  float* dxg = ws + w.dxg;
  const float beta = accumulate ? 1.f : 0.f;

  if (!prep) {
    head_collapse_kernel<<<cdiv(d.F + 1, 32), 256, 0, s>>>(W_f, b_f, W_o, b_o, d.F, d.Hd, ws + w.weff);
    GIC_TRY(check_launch("head_collapse_kernel"));
  }
  cudaMemsetAsync(sacc, 0, (w.demb - w.s) * sizeof(float), s);      // s and dbh
  if ((d.F % 4 == 0) && (!keep || (reinterpret_cast<uintptr_t>(keep) & 3u) == 0)) {
    const int colb = cdiv(d.F / 4, 256);
    int per_sm = 3;           // measured (ncu, c2): 3 -> 51 us, 4 -> 55, 6 -> 61, 8 -> 69, 2 -> 52, 1 -> 69
    { const int o = option("GIC_HB_CTAS_PER_SM", 0); if (o > 0) per_sm = o; }   // tuning
    int chunks = max(1, (per_sm * num_sms()) / colb);
    int rpc = cdiv((long long)rows, chunks);
    rpc = (rpc + 3) & ~3;
    chunks = cdiv((long long)rows, rpc);
    if (bf)
      head_bwd_vec_kernel<true><<<dim3(colb, chunks), 256, 0, s>>>(dlogit, keep, 1.f / (1.f - drop_p), hpre, pooled,
                                                                  (int)rows, d.F, weff, rpc, dh, dx, sacc, dbh, Fp);
    else
      head_bwd_vec_kernel<false><<<dim3(colb, chunks), 256, 0, s>>>(dlogit, keep, 1.f / (1.f - drop_p), hpre, pooled,
                                                                   (int)rows, d.F, weff, rpc, dh, dx, sacc, dbh, Fp);
    GIC_TRY(check_launch("head_bwd_vec_kernel"));
  } else {
    const int colb = cdiv(d.F, 256);
    int chunks = max(1, (4 * num_sms()) / colb);
    int rpc = cdiv((long long)rows, chunks);
    chunks = cdiv((long long)rows, rpc);
    head_bwd_kernel<<<dim3(colb, chunks), 256, 0, s>>>(dlogit, keep, 1.f / (1.f - drop_p), hpre, pooled, (int)rows,
                                                      d.F, weff, rpc, dh, dx, sacc, dbh);
    GIC_TRY(check_launch("head_bwd_kernel"));
  }
  if (want_param) {
    head_param_grads_kernel<<<d.Hd, 256, 0, s>>>(dlogit, (int)rows, sacc, dbh, W_f, b_f, W_o, d.F, d.Hd, beta, dW_f,
                                                db_f, dW_o, db_o, db_h);
    GIC_TRY(check_launch("head_param_grads_kernel"));
    // dW_h[F,F] (+)= dh^T [F, rows] * pooled [rows, F]
    if (bf)
      GIC_TRY(gemm_bf16(true, false, d.F, d.F, (int)rows, 1.f, dh, Fp, pooled_bf, Fp, beta, dW_h, d.F, nullptr, s, PROF_GEMM_D));
    else
      GIC_TRY(gemm(mode, true, false, d.F, d.F, (int)rows, 1.f, dh, d.F, pooled, d.F, beta, dW_h, d.F, nullptr, s, PROF_GEMM_D));
  }
  // dxg = dh * W_h        ([rows,F] x [F,F], W_h is [out,in] so this is the non-transposed product).  Written with
  // beta = 0 (TMA-store epilogue); the conv/pool backward kernels read dx + dxg: a beta = 1 epilogue has to pull the C
  // tile through the LSU and measured 97 us vs 45 us (profiles/README.md).
  if (bf) {
    if (!prep) GIC_TRY(f32_to_bf16(W_h, d.F, d.F, d.F, W_h_bf_ws, Fp, s));
    GIC_TRY(gemm_bf16(false, false, (int)rows, d.F, d.F, 1.f, dh, Fp, W_h_bf, Fp, 0.f, dxg, d.F, nullptr, s, PROF_GEMM_D));
  } else {
    GIC_TRY(gemm(mode, false, false, (int)rows, d.F, d.F, 1.f, dh, d.F, W_h, d.F, 0.f, dxg, d.F, nullptr, s, PROF_GEMM_D));
  }
  // conv / pool backward
  {
    GIC_REQUIRE(g.kmax <= BWD_KMAX, GIC_ERR_SHAPE, "disc bwd: filter_size*emb_dim_single <= %d supported", BWD_KMAX);
    if (want_param && !accumulate) {
      for (int i = 0; i < g.ngroups; ++i) {
        cudaMemsetAsync(g.dw[i], 0, (size_t)g.n[i] * g.f[i] * d.es * sizeof(float), s);
        cudaMemsetAsync(g.db[i], 0, (size_t)g.n[i] * sizeof(float), s);
      }
    }
    // (a) demb
    {
      const size_t fixed = ((size_t)g.kmax + 1) * d.F * 4;
      const size_t per_warp = (size_t)d.L * d.es * 32 * 4;
      int nwarps = 8;
      while (nwarps > 1 && fixed + nwarps * per_warp > 100 * 1024) nwarps >>= 1;
      const size_t smem = fixed + nwarps * per_warp;
      GIC_REQUIRE(smem <= 200 * 1024, GIC_ERR_SHAPE, "disc bwd: L*emb_dim_single too large for shared memory");
      const int grid = min(cdiv((long long)rows, nwarps), 4 * num_sms());
      bool vec = (d.F % 4 == 0) && aligned16(dx) && aligned16(dxg) && ((reinterpret_cast<uintptr_t>(arg) & 3u) == 0);
      for (int i = 0; i < g.ngroups; ++i) vec = vec && (g.n[i] % 4 == 0);
      static bool attr = false;
      if (!attr) {
        cudaFuncSetAttribute(conv_pool_bwd_demb_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(conv_pool_bwd_demb_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(conv_pool_bwd_demb_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(conv_pool_bwd_demb_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr = true;
      }
#define GIC_DEMB(ES1_, VEC_) conv_pool_bwd_demb_kernel<ES1_, VEC_><<<grid, nwarps * 32, smem, s>>>(arg, dx, dxg, (int)rows, d.L, d.De, d.R, d.es, g, demb)
      if (d.es == 1) { if (vec) GIC_DEMB(true, true); else GIC_DEMB(true, false); }
      else { if (vec) GIC_DEMB(false, true); else GIC_DEMB(false, false); }
#undef GIC_DEMB
      GIC_TRY(check_launch("conv_pool_bwd_demb_kernel"));
    }
    // (b) conv weight / bias gradients
    if (want_param) {
      const int colb = cdiv(d.F, 256);
      int per_sm = 4;
      { const int o = option("GIC_DW_CTAS_PER_SM", 0); if (o > 0) per_sm = o; }   // tuning
      int chunks = max(1, (per_sm * num_sms()) / colb);
      int rpc = cdiv((long long)rows, chunks);
      rpc = ((rpc + DW_RC - 1) / DW_RC) * DW_RC;
      chunks = cdiv((long long)rows, rpc);
      const size_t smem = (size_t)DW_RC * d.L * d.es * 4;
      GIC_REQUIRE(smem <= 48 * 1024, GIC_ERR_SHAPE, "disc bwd: L*emb_dim_single too large for shared memory");
      if (d.es == 1)
        conv_pool_bwd_dw_kernel<true><<<dim3(colb, chunks), 256, smem, s>>>(emb, arg, dx, dxg, (int)rows, d.L, d.De, d.R, d.es, g, rpc);
      else
        conv_pool_bwd_dw_kernel<false><<<dim3(colb, chunks), 256, smem, s>>>(emb, arg, dx, dxg, (int)rows, d.L, d.De, d.R, d.es, g, rpc);
      GIC_TRY(check_launch("conv_pool_bwd_dw_kernel"));
    }
  }
  // embedding backward
  if (want_param) {
    if (inp_soft) {
      // dW_e[De,V] (+)= demb^T [De, N*L] * inp [N*L, V]
      GIC_TRY(gemm(mode, true, false, d.De, d.V, d.N * d.L, 1.f, demb, d.De, inp_soft, d.V, beta, dW_e, d.V, nullptr, s));
    } else {
      if (!accumulate) cudaMemsetAsync(dW_e, 0, (size_t)d.De * d.V * sizeof(float), s);
      const int tot = d.N * d.L * d.De;
      disc_embed_ids_bwd_kernel<<<cdiv(tot, 256), 256, 0, s>>>(ids, d.N * d.L, d.V, d.De, demb, dW_e);
      GIC_TRY(check_launch("disc_embed_ids_bwd_kernel"));
    }
  }
  if (dinp) {
    // dinp[N*L, V] = demb [N*L, De] * W_e [De, V]
    GIC_TRY(gemm(mode, false, false, d.N * d.L, d.V, d.De, 1.f, demb, d.De, W_e, d.V, 0.f, dinp, d.V, nullptr, s));
  }
  return GIC_OK;
}

// ---------------------------------------------------------------------------------------
// C-ABI facing wrappers (argument validation + descriptor set-up)
// ---------------------------------------------------------------------------------------
static int disc_dims(DiscDims& d, int N, int L, int V, int De, int R, int Hd, const ConvGroups& g) {
  GIC_REQUIRE(N >= 0 && L >= 1 && V >= 1 && De >= 1 && R >= 1 && Hd >= 1, GIC_ERR_SHAPE, "disc: bad shape");
  GIC_REQUIRE(De % R == 0, GIC_ERR_SHAPE, "disc: disc_embed_dim %d not divisible by disc_num_rep %d", De, R);
  d.N = N; d.L = L; d.V = V; d.De = De; d.R = R; d.es = De / R; d.F = g.F; d.Hd = Hd; d.ngroups = g.ngroups;
  d.kmax = g.kmax;
  for (int i = 0; i < g.ngroups; ++i)
    GIC_REQUIRE(L >= g.f[i], GIC_ERR_SHAPE, "disc: caption length %d shorter than filter size %d", L, g.f[i]);
  GIC_REQUIRE(L <= 254, GIC_ERR_SHAPE, "disc: caption length <= 254 supported");
  return GIC_OK;
}

int disc_fwd_entry(int mode, const float* inp_soft, const int64_t* ids, int N, int L, int V, int De, int R,
                   int n_groups, const int* fs, const int* nf, const float* W_e, const float* const* cw,
                   const float* const* cb, const float* W_h, const float* b_h, const float* W_f, const float* b_f,
                   int Hd, const float* W_o, const float* b_o, int n_heads, const uint8_t* const* keep, float drop_p,
                   float* const* logits, float* saved, float* ws, cudaStream_t s) {
  GIC_REQUIRE((inp_soft != nullptr) != (ids != nullptr), GIC_ERR_NULL, "disc_fwd: exactly one of inp_soft / ids");
  GIC_REQUIRE(fs && nf && cw && cb && W_e && W_h && b_h && W_f && b_f && W_o && b_o && logits && saved && ws,
              GIC_ERR_NULL, "disc_fwd: NULL pointer");
  GIC_REQUIRE(n_heads >= 1 && n_heads <= MAX_HEADS, GIC_ERR_SHAPE, "disc_fwd: 1..%d heads", MAX_HEADS);
  GIC_REQUIRE(drop_p >= 0.f && drop_p < 1.f, GIC_ERR_SHAPE, "disc_fwd: dropout p in [0,1)");
  const int es = (R > 0 && De % R == 0) ? De / R : 1;
  ConvGroups g;
  GIC_TRY(disc_fill_groups(g, n_groups, fs, nf, cw, cb, nullptr, nullptr, es));
  DiscDims d;
  GIC_TRY(disc_dims(d, N, L, V, De, R, Hd, g));
  for (int m = 0; m < n_heads; ++m) GIC_REQUIRE(logits[m], GIC_ERR_NULL, "disc_fwd: NULL logits[%d]", m);
  return disc_forward(mode, inp_soft, ids, d, g, W_e, W_h, b_h, W_f, b_f, W_o, b_o, n_heads, keep, drop_p, logits,
                      saved, ws, s);
}

int disc_bwd_entry(int mode, const float* dlogits, const uint8_t* keep, float drop_p, const float* inp_soft,
                   const int64_t* ids, int N, int L, int V, int De, int R, int n_groups, const int* fs, const int* nf,
                   const float* W_e, const float* const* cw, const float* const* cb, const float* W_h,
                   const float* W_f, const float* b_f, int Hd, const float* W_o, const float* b_o, const float* saved,
                   float* ws, float* dW_e, float* const* dcw, float* const* dcb, float* dW_h, float* db_h,
                   float* dW_f, float* db_f, float* dW_o, float* db_o, float* dinp, int want_param, int accumulate,
                   cudaStream_t s) {
  GIC_REQUIRE((inp_soft != nullptr) != (ids != nullptr), GIC_ERR_NULL, "disc_bwd: exactly one of inp_soft / ids");
  GIC_REQUIRE(dlogits && fs && nf && cw && cb && W_e && W_h && W_f && b_f && W_o && b_o && saved && ws, GIC_ERR_NULL,
              "disc_bwd: NULL pointer");
  GIC_REQUIRE(!want_param || (dW_e && dcw && dcb && dW_h && db_h && dW_f && db_f && dW_o && db_o), GIC_ERR_NULL,
              "disc_bwd: NULL gradient buffer");
  GIC_REQUIRE(!(dinp && ids), GIC_ERR_UNSUPPORTED, "disc_bwd: hard-token input has no gradient");
  const int es = (R > 0 && De % R == 0) ? De / R : 1;
  ConvGroups g;
  GIC_TRY(disc_fill_groups(g, n_groups, fs, nf, cw, cb, want_param ? dcw : nullptr, want_param ? dcb : nullptr, es));
  DiscDims d;
  GIC_TRY(disc_dims(d, N, L, V, De, R, Hd, g));
  return disc_backward(mode, dlogits, keep, drop_p, inp_soft, ids, d, g, W_e, W_h, W_f, b_f, W_o, b_o, saved, ws, dW_e,
                       dW_h, db_h, dW_f, db_f, dW_o, db_o, dinp, want_param, accumulate, s);
}

}  // namespace gic
