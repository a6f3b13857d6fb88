// Caption generator hot path: LSTM decode step, Gumbel-softmax sampling, and their backward.
// Replaces Decoder.sample / Decoder.add_gumbel (src/generator.py:55-96) and the autograd
// backward of that graph (SURVEY.md §3.3, §3.4).  Encoder.linear + Encoder.bn
// (src/generator.py:15-16,23-24) is here too because it feeds step 0 of the decode.
#include "gic_internal.cuh"
#include "philox.cuh"

namespace gic {

// Temperature source: the by-value argument, or (CUDA-graph replay: by-value arguments are frozen at capture) a device
// scalar registered with gic_set_temperature_device().
void set_temperature_device(const float* p) { ctx().t_dev = p; }
const float* temperature_device() { return ctx().t_dev; }
#define g_t_dev (ctx().t_dev)
__device__ __forceinline__ float pick_t(float by_value, const float* t_dev) { return t_dev ? __ldg(t_dev) : by_value; }

// ---------------------------------------------------------------------------------------
// shim-side random draws (caller passed no uniforms / no dropout masks): Philox4x32-10, see philox.cuh
// ---------------------------------------------------------------------------------------
void set_rng(unsigned long long seed, unsigned long long offset, const unsigned long long* state_dev) {
  Ctx& c = ctx();
  c.rng.seed = seed; c.rng.offset = offset; c.rng.dev = state_dev;
}
RngState rng_state() { const Ctx& c = ctx(); RngState r; r.seed = c.rng.seed; r.offset = c.rng.offset; r.dev = c.rng.dev; return r; }
#define g_rng (rng_state())

__global__ void philox_uniform_kernel(RngState st, uint32_t tag, unsigned long long base, size_t n, float* __restrict__ out) {
  unsigned long long seed, offset;
  rng_load(st, seed, offset);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  // thread = one Philox group (4 consecutive logical elements); base may start inside a group
  const unsigned long long g0 = base >> 2, g1 = (base + n + 3) >> 2;
  for (unsigned long long gi = g0 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; gi < g1; gi += stride) {
    const float4 u = philox_uniform4(seed, offset, tag, gi);
    const float v[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const unsigned long long i = 4 * gi + e;
      if (i >= base && i < base + n) out[i - base] = v[e];
    }
  }
}
int philox_uniform(uint32_t tag, unsigned long long base, size_t n, float* out, cudaStream_t s) {
  if (n == 0) return GIC_OK;
  GIC_REQUIRE(out, GIC_ERR_NULL, "philox_uniform: NULL output");
  const int grid = (int)min((size_t)num_sms() * 16, (n / 4 + 255) / 256 + 1);
  philox_uniform_kernel<<<grid, 256, 0, s>>>(g_rng, tag, base, n, out);
  return check_launch("philox_uniform_kernel");
}

// keep[i] = (u_i >= p) as uint8, four per thread (n % 4 == 0 and a 4-byte aligned output take the packed store)
__global__ void philox_keep_mask_kernel(RngState st, uint32_t tag, size_t n, float p, uint8_t* __restrict__ out, int packed) {
  unsigned long long seed, offset;
  rng_load(st, seed, offset);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t groups = (n + 3) >> 2;
  for (size_t gi = blockIdx.x * (size_t)blockDim.x + threadIdx.x; gi < groups; gi += stride) {
    const float4 u = philox_uniform4(seed, offset, tag, gi);
    const uint32_t k0 = u.x >= p, k1 = u.y >= p, k2 = u.z >= p, k3 = u.w >= p;
    if (packed) {
      reinterpret_cast<uint32_t*>(out)[gi] = k0 | (k1 << 8) | (k2 << 16) | (k3 << 24);
    } else {
      const uint32_t kk[4] = {k0, k1, k2, k3};
#pragma unroll
      for (int e = 0; e < 4; ++e) if (4 * gi + e < n) out[4 * gi + e] = (uint8_t)kk[e];
    }
  }
}
int philox_keep_mask(uint32_t tag, size_t n, float p, uint8_t* out, cudaStream_t s) {
  if (n == 0) return GIC_OK;
  GIC_REQUIRE(out, GIC_ERR_NULL, "philox_keep_mask: NULL output");
  GIC_REQUIRE(p >= 0.f && p < 1.f, GIC_ERR_SHAPE, "philox_keep_mask: dropout p in [0,1)");
  const int packed = ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) ? 1 : 0;
  const int grid = (int)min((size_t)num_sms() * 16, (n / 4 + 255) / 256 + 1);
  philox_keep_mask_kernel<<<grid, 256, 0, s>>>(g_rng, tag, n, p, out, packed);
  return check_launch("philox_keep_mask_kernel");
}

// ---------------------------------------------------------------------------------------
// batch contract (collate_fn, src/tasks.py:138-158): ragged token lists arrive as ONE flat int32 array + B+1 offsets
// (sum(len) + B + 1 ints over PCIe instead of a padded [B, Lm] int64 tensor) and are packed on the device into
// captions[B, Lm] = <S>=1, tokens, <E>=2, <PAD>=0 ... and lengths[b] = len + 2.  Thread = one (caption, position).
// ---------------------------------------------------------------------------------------
__global__ void pack_captions_kernel(const int32_t* __restrict__ tokens, const int32_t* __restrict__ offsets, int B,
                                     int Lm, int64_t* __restrict__ captions, int32_t* __restrict__ lengths) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * Lm) return;
  const int b = idx / Lm, pos = idx - b * Lm;
  const int o = offsets[b];
  int len = offsets[b + 1] - o;
  if (len > Lm - 2) len = Lm - 2;                    // the host shim rejects this case; stay in bounds regardless
  int64_t v = 0;                                     // <PAD>
  if (pos == 0) v = 1;                               // <S>
  else if (pos <= len) v = tokens[o + pos - 1];
  else if (pos == len + 1) v = 2;                    // <E>
  captions[idx] = v;
  if (pos == 0 && lengths) lengths[b] = len + 2;
}

int pack_captions(const int32_t* tokens, const int32_t* offsets, int B, int Lm, int64_t* captions, int32_t* lengths,
                  cudaStream_t s) {
  GIC_REQUIRE(B >= 0 && Lm >= 2, GIC_ERR_SHAPE, "pack_captions: bad shape B=%d max_caption_len=%d", B, Lm);
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(offsets && captions, GIC_ERR_NULL, "pack_captions: NULL pointer");
  pack_captions_kernel<<<cdiv((long long)B * Lm, 256), 256, 0, s>>>(tokens, offsets, B, Lm, captions, lengths);
  return check_launch("pack_captions_kernel");
}

// ---------------------------------------------------------------------------------------
// row gather: out[i, :] = table[ids[i], :]     (nn.Embedding lookup, src/generator.py:75)
// ---------------------------------------------------------------------------------------
__global__ void gather_rows_kernel(const float* __restrict__ table, const int64_t* __restrict__ ids,
                                   int n, int E, int V, float* __restrict__ out) {
  const int i = blockIdx.x;
  if (i >= n) return;
  int64_t id = ids[i];
  if (id < 0 || id >= V) id = 0;   // out-of-range ids never occur on the path; stay in bounds
  const float* src = table + (size_t)id * E;
  float* dst = out + (size_t)i * E;
  for (int e = threadIdx.x; e < E; e += blockDim.x) dst[e] = src[e];
}

int gather_rows(const float* table, const int64_t* ids, int n, int E, int V, float* out,
                cudaStream_t s) {
  if (n == 0) return GIC_OK;
  gather_rows_kernel<<<n, 128, 0, s>>>(table, ids, n, E, V, out);
  return check_launch("gather_rows_kernel");
}

// ---------------------------------------------------------------------------------------
// LSTM cell, forward.  gates[B,4H] pre-activation (i,f,g,o chunks) -> acts (post-activation,
// saved for backward), c_new, h_new; the top layer also writes h into htop[B,L,H] at step t.
// ---------------------------------------------------------------------------------------
__global__ void lstm_cell_fwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev,
                                     int B, int H, float* __restrict__ acts, float* __restrict__ c_new,
                                     float* __restrict__ h_new, float* __restrict__ htop, int L, int t) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, j = idx % H;
  const float* g = gates + (size_t)b * 4 * H;
  const float i_ = sigmoidf_acc(g[j]);
  const float f_ = sigmoidf_acc(g[H + j]);
  const float g_ = tanhf(g[2 * H + j]);
  const float o_ = sigmoidf_acc(g[3 * H + j]);
  const float c = f_ * c_prev[idx] + i_ * g_;
  const float h = o_ * tanhf(c);
  if (acts) {
    float* a = acts + (size_t)b * 4 * H;
    a[j] = i_; a[H + j] = f_; a[2 * H + j] = g_; a[3 * H + j] = o_;
  }
  c_new[idx] = c;
  h_new[idx] = h;
  if (htop) htop[((size_t)b * L + t) * H + j] = h;
}

// LSTM cell, backward for one (layer, step).  dh_in = gradient arriving at h_t from above
// (vocab projection or the next layer) with row stride dh_stride; dh_rec / dc_rec are the
// recurrent gradients from step t+1 (dc_rec is updated in place to dc_{t-1}).
__global__ void lstm_cell_bwd_kernel(const float* __restrict__ acts, const float* __restrict__ c_prev,
                                     const float* __restrict__ c_cur, const float* __restrict__ dh_in,
                                     long long dh_stride, const float* __restrict__ dh_rec,
                                     float* __restrict__ dc_rec, int B, int H, float* __restrict__ dgates) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * H) return;
  const int b = idx / H, j = idx % H;
  const float* a = acts + (size_t)b * 4 * H;
  const float i_ = a[j], f_ = a[H + j], g_ = a[2 * H + j], o_ = a[3 * H + j];
  float dh = dh_rec ? dh_rec[idx] : 0.f;
  if (dh_in) dh += dh_in[(size_t)b * dh_stride + j];
  const float tc = tanhf(c_cur[idx]);
  const float dc = dh * o_ * (1.f - tc * tc) + dc_rec[idx];
  float* dg = dgates + (size_t)b * 4 * H;
  const float di = dc * g_ * i_ * (1.f - i_), df = dc * c_prev[idx] * f_ * (1.f - f_);
  const float dgg = dc * i_ * (1.f - g_ * g_), dout = dh * tc * o_ * (1.f - o_);
  dg[j] = di; dg[H + j] = df; dg[2 * H + j] = dgg; dg[3 * H + j] = dout;
  dc_rec[idx] = dc * f_;
}

// ---------------------------------------------------------------------------------------
// Fused Gumbel perturbation + temperature + vocab softmax + first-max sample + next-input
// embedding gather.  One CTA per caption row; the perturbed logits are staged in shared
// memory (or, for huge vocabularies, in the output row itself) so u and the logits are read
// from HBM exactly once and the probabilities are written exactly once: 8*V bytes per row.
//   adversarial mode: out = softmax((logits + g(u)) * T)              (src/generator.py:68-70)
//   pretrain mode   : out = logits, choice = argmax softmax(logits)   (src/generator.py:63-66)
// Tie rule: lowest index among equal probabilities (torch.max first-max, :73).
// ---------------------------------------------------------------------------------------
template <bool PRETRAIN>
__global__ void __launch_bounds__(256)
sample_step_kernel(const float* __restrict__ logits, const float* __restrict__ u, float temperature_v,
                   const float* __restrict__ t_dev, int V, int L, int t, float* __restrict__ out /*[B,L,V]*/,
                   int64_t* __restrict__ ids, const int64_t* __restrict__ forced, const float* __restrict__ embed, int E,
                   float* __restrict__ x_next, int stage_in_smem) {
  const float temperature = pick_t(temperature_v, t_dev);
  extern __shared__ float zbuf[];
  __shared__ float red[32];
  __shared__ int red_i[32];
  __shared__ int s_tok;
  const int b = blockIdx.x;
  const float* lrow = logits + (size_t)b * V;
  float* orow = out + ((size_t)b * L + t) * V;
  float* z = stage_in_smem ? zbuf : orow;
  const float eps = 1e-10f;

  // pass 1: z = (logit + gumbel(u)) * T, row max
  float mx = -INFINITY;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    float x = lrow[v];
    if (!PRETRAIN) {
      const float uu = u[(size_t)b * V + v];
      const float g = -logf(-logf(uu + eps) + eps);
      x = (x + g) * temperature;
    }
    z[v] = x;
    mx = fmaxf(mx, x);
  }
  mx = block_max(mx, red);
  // pass 2: sum of exp
  float sum = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float e = expf(z[v] - mx);
    z[v] = e;
    sum += e;
  }
  sum = block_sum(sum, red);
  // pass 3: probabilities, first-max index
  float best = -1.f;
  int best_i = 0x7fffffff;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float p = z[v] / sum;
    if (PRETRAIN) orow[v] = lrow[v]; else orow[v] = p;
    if (p > best) { best = p; best_i = v; }
  }
  // (value, index) arg-max across the block; ties -> lowest index
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) { red[w] = best; red_i[w] = best_i; }
  __syncthreads();
  if (w == 0) {
    best = lane < nw ? red[lane] : -2.f;
    best_i = lane < nw ? red_i[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
      if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
    }
    if (lane == 0) {
      if (best_i < 0 || best_i >= V) best_i = 0;      // all-NaN row: stay in bounds
      ids[(size_t)b * L + t] = best_i;
      int fed = best_i;
      if (forced) {
        const int64_t f = forced[(size_t)b * L + t];
        fed = (f >= 0 && f < V) ? (int)f : 0;
      }
      s_tok = fed;
    }
  }
  __syncthreads();
  if (x_next) {
    const float* src = embed + (size_t)s_tok * E;
    float* dst = x_next + (size_t)b * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) dst[e] = src[e];
  }
}

// Register-resident variant for V % 4 == 0 and V <= 256 * 4 * NV4: every thread issues all of its float4 loads of
// the logits row and the uniform row up front (2 * NV4 outstanding 16-byte loads), keeps its NV4 * 4 perturbed
// logits in registers through the max / sum / normalise passes, and writes the probabilities with float4 stores.
// Same arithmetic (accurate logf / expf, true division) and tie rule as sample_step_kernel.
// FAST (tensor-core mode only, where the logits already carry TF32 rounding): MUFU-based __logf / __expf and a
// reciprocal multiply for the outer log / exp / normalisation.  The inner log(u) stays accurate: for u -> 1 its
// value is tiny and __logf's absolute error would become a relative error of the Gumbel noise.
template <bool FAST> __device__ __forceinline__ float log_f(float x) { return FAST ? __logf(x) : logf(x); }
template <bool FAST> __device__ __forceinline__ float exp_f(float x) { return FAST ? __expf(x) : expf(x); }

template <bool PRETRAIN, int NV4, bool FAST>
__global__ void __launch_bounds__(256)
sample_step_reg_kernel(const float* __restrict__ logits, const float* __restrict__ u, float temperature_v,
                       const float* __restrict__ t_dev, int V, int L, int t, float* __restrict__ out,
                       int64_t* __restrict__ ids, const int64_t* __restrict__ forced, const float* __restrict__ embed,
                       int E, float* __restrict__ x_next) {
  const float temperature = pick_t(temperature_v, t_dev);
  __shared__ float red[32];
  __shared__ int red_i[32];
  __shared__ int s_tok;
  const int b = blockIdx.x;
  const int nv4 = V >> 2;
  const float4* lrow = reinterpret_cast<const float4*>(logits + (size_t)b * V);
  const float4* urow = PRETRAIN ? nullptr : reinterpret_cast<const float4*>(u + (size_t)b * V);
  float4* orow = reinterpret_cast<float4*>(out + ((size_t)b * L + t) * V);
  const float eps = 1e-10f;
  float4 z[NV4];
  float4 uu[NV4];
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    const int v = threadIdx.x + i * 256;
    z[i] = (v < nv4) ? lrow[v] : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (!PRETRAIN) uu[i] = (v < nv4) ? urow[v] : make_float4(0.5f, 0.5f, 0.5f, 0.5f);
  }
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    if (PRETRAIN) {
      if (threadIdx.x + i * 256 < nv4) orow[threadIdx.x + i * 256] = z[i];       // out = raw logits
    } else {
      z[i].x = (z[i].x - log_f<FAST>(-logf(uu[i].x + eps) + eps)) * temperature;
      z[i].y = (z[i].y - log_f<FAST>(-logf(uu[i].y + eps) + eps)) * temperature;
      z[i].z = (z[i].z - log_f<FAST>(-logf(uu[i].z + eps) + eps)) * temperature;
      z[i].w = (z[i].w - log_f<FAST>(-logf(uu[i].w + eps) + eps)) * temperature;
    }
    mx = fmaxf(mx, fmaxf(fmaxf(z[i].x, z[i].y), fmaxf(z[i].z, z[i].w)));
  }
  mx = block_max(mx, red);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    z[i].x = exp_f<FAST>(z[i].x - mx); z[i].y = exp_f<FAST>(z[i].y - mx);
    z[i].z = exp_f<FAST>(z[i].z - mx); z[i].w = exp_f<FAST>(z[i].w - mx);
    sum += (z[i].x + z[i].y) + (z[i].z + z[i].w);
  }
  sum = block_sum(sum, red);
  const float inv = 1.0f / sum;
  float best = -1.f;
  int best_i = 0x7fffffff;
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    const int v = threadIdx.x + i * 256;
    if (v < nv4) {
      float4 p;
      if (FAST) { p.x = z[i].x * inv; p.y = z[i].y * inv; p.z = z[i].z * inv; p.w = z[i].w * inv; }
      else { p.x = z[i].x / sum; p.y = z[i].y / sum; p.z = z[i].z / sum; p.w = z[i].w / sum; }
      if (!PRETRAIN) orow[v] = p;
      if (p.x > best) { best = p.x; best_i = 4 * v; }
      if (p.y > best) { best = p.y; best_i = 4 * v + 1; }
      if (p.z > best) { best = p.z; best_i = 4 * v + 2; }
      if (p.w > best) { best = p.w; best_i = 4 * v + 3; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) { red[w] = best; red_i[w] = best_i; }
  __syncthreads();
  if (w == 0) {
    best = lane < 8 ? red[lane] : -2.f;
    best_i = lane < 8 ? red_i[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
      if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
    }
    if (lane == 0) {
      if (best_i < 0 || best_i >= V) best_i = 0;
      ids[(size_t)b * L + t] = best_i;
      int fed = best_i;
      if (forced) {
        const int64_t f = forced[(size_t)b * L + t];
        fed = (f >= 0 && f < V) ? (int)f : 0;
      }
      s_tok = fed;
    }
  }
  __syncthreads();
  if (x_next) {
    const float* src = embed + (size_t)s_tok * E;
    float* dst = x_next + (size_t)b * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) dst[e] = src[e];
  }
}

template <bool PRETRAIN, bool FAST>
static bool launch_sample_reg(const float* logits, const float* u, float temperature, int B, int V, int L, int t,
                              float* out, int64_t* ids, const int64_t* forced, const float* embed, int E,
                              float* x_next, cudaStream_t s) {
  const int nv4 = V >> 2;
#define GIC_SAMPLE(NV4_)                                                                                         \
  sample_step_reg_kernel<PRETRAIN, NV4_, FAST><<<B, 256, 0, s>>>(logits, u, temperature, g_t_dev, V, L, t, out, ids, forced, embed, \
                                                           E, x_next)
  if (nv4 <= 256 * 1) GIC_SAMPLE(1);
  else if (nv4 <= 256 * 2) GIC_SAMPLE(2);
  else if (nv4 <= 256 * 4) GIC_SAMPLE(4);
  else if (nv4 <= 256 * 8) GIC_SAMPLE(8);
  else if (nv4 <= 256 * 10) GIC_SAMPLE(10);
  else if (nv4 <= 256 * 16) GIC_SAMPLE(16);
  else return false;
#undef GIC_SAMPLE
  return true;
}

int sample_step(bool pretrain, const float* logits, const float* u, float temperature, int B, int V,
                int L, int t, float* out, int64_t* ids, const int64_t* forced, const float* embed,
                int E, float* x_next, cudaStream_t s, bool fast_math) {
  ProfScope prof(PROF_SAMPLE, 8.0 * B * V, s);     // algorithmic HBM bytes: read u, write probs (SURVEY 8d)
  if ((V % 4 == 0) && aligned16(logits) && aligned16(out) && (pretrain || aligned16(u))) {
    bool done;
    if (pretrain) done = launch_sample_reg<true, false>(logits, u, temperature, B, V, L, t, out, ids, forced, embed, E, x_next, s);
    else if (fast_math) done = launch_sample_reg<false, true>(logits, u, temperature, B, V, L, t, out, ids, forced, embed, E, x_next, s);
    else done = launch_sample_reg<false, false>(logits, u, temperature, B, V, L, t, out, ids, forced, embed, E, x_next, s);
    if (done) return check_launch("sample_step_reg_kernel");
  }
  const size_t smem = (size_t)V * sizeof(float);
  const int in_smem = smem <= 200 * 1024 ? 1 : 0;
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(sample_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(sample_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_set = true;
  }
  const size_t dyn = in_smem ? smem : 0;
  if (pretrain)
    sample_step_kernel<true><<<B, 256, dyn, s>>>(logits, u, temperature, g_t_dev, V, L, t, out, ids, forced, embed, E,
                                               x_next, in_smem);
  else
    sample_step_kernel<false><<<B, 256, dyn, s>>>(logits, u, temperature, g_t_dev, V, L, t, out, ids, forced, embed, E,
                                                x_next, in_smem);
  return check_launch("sample_step_kernel");
}

// ---------------------------------------------------------------------------------------
// EXTENSION (north-star stage 2/3, not in the reference: SURVEY.md 8a row B2): fused vocab softmax + categorical
// sample by inverse CDF from ONE caller-supplied uniform per row.  token = first index whose cumulative probability
// exceeds u (clamped to V-1); also returns log pi(token) for the policy-gradient loss.  Nothing of size [B,V] is
// written unless `out` (raw logits, kept for the backward of the sampled caption) is given.
// One CTA (256 threads) per row.  Order of the cumulative sum: element e belongs to segment e / 128 (a warp's float4
// sweep); segments are summed in index order by one thread, the hit segment is resolved by a warp scan, the hit
// float4 sequentially.  All in unnormalised exp space against the target u * sum.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sample_cdf_kernel(const float* __restrict__ logits, const float* __restrict__ u, int V, int L, int t,
                  long long id_stride /*elements between rows of ids*/, float* __restrict__ out /*[rows,L,V] or null*/,
                  int64_t* __restrict__ ids, float* __restrict__ logp /*[rows,L] or null*/,
                  const int64_t* __restrict__ forced, const float* __restrict__ embed, int E,
                  float* __restrict__ x_next) {
  extern __shared__ float seg_s[];          // [nseg] partial sums, nseg = ceil(V / 128)
  __shared__ float red[32];
  __shared__ int s_seg, s_tok;
  __shared__ float s_before, s_sum, s_max;
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float* lrow = logits + (size_t)b * V;
  const int nseg = (V + 127) >> 7;
  // pass 1: max
  float mx = -INFINITY;
  for (int v = threadIdx.x; v < V; v += blockDim.x) mx = fmaxf(mx, lrow[v]);
  mx = block_max(mx, red);
  // pass 2: per-segment sums of exp (segment = 128 consecutive elements = one warp sweep of 4 per lane)
  float tot = 0.f;
  for (int sgi = warp; sgi < nseg; sgi += 8) {
    const int v0 = sgi * 128 + lane * 4;
    float e = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) if (v0 + j < V) e += expf(lrow[v0 + j] - mx);
    e = warp_sum(e);
    if (lane == 0) seg_s[sgi] = e;
    tot += e;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float S = 0.f;
    for (int i = 0; i < nseg; ++i) S += seg_s[i];
    const float target = u[b] * S;
    float acc = 0.f;
    int hit = -1;
    for (int i = 0; i < nseg; ++i) {
      const float nxt = acc + seg_s[i];
      if (nxt > target) { hit = i; break; }
      acc = nxt;
    }
    s_seg = hit; s_before = acc; s_sum = S; s_max = mx;
    s_tok = (hit < 0) ? V - 1 : min(V - 1, hit * 128 + 127);     // u beyond the total mass -> last token
  }
  __syncthreads();
  (void)tot;
  if (warp == 0 && s_seg >= 0) {
    const int sgi = s_seg;
    const float target = u[b] * s_sum;
    const int v0 = sgi * 128 + lane * 4;
    float e[4];
    float mine = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) { e[j] = (v0 + j < V) ? expf(lrow[v0 + j] - mx) : 0.f; mine += e[j]; }
    float inc = mine;                                            // inclusive warp scan of the lanes' sums
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float y = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += y;
    }
    const bool hit = (s_before + inc > target);
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m != 0u && lane == (__ffs(m) - 1)) {
      float acc = s_before + (inc - mine);
      int tok = min(V - 1, v0 + 3);
      for (int j = 0; j < 4; ++j) {
        acc += e[j];
        if (acc > target) { tok = v0 + j; break; }
      }
      s_tok = min(tok, V - 1);
    }
  }
  __syncthreads();
  const int tok = s_tok;
  if (threadIdx.x == 0) {
    ids[(size_t)b * id_stride + t] = tok;
    if (logp) logp[(size_t)b * L + t] = (lrow[tok] - s_max) - logf(s_sum);
  }
  if (out) {
    float* orow = out + ((size_t)b * L + t) * V;
    for (int v = threadIdx.x; v < V; v += blockDim.x) orow[v] = lrow[v];
  }
  if (x_next) {
    int fed = tok;
    if (forced) {
      const int64_t f = forced[(size_t)b * id_stride + t];
      fed = (f >= 0 && f < V) ? (int)f : 0;
    }
    const float* src = embed + (size_t)fed * E;
    float* dst = x_next + (size_t)b * E;
    for (int e = threadIdx.x; e < E; e += blockDim.x) dst[e] = src[e];
  }
}

int sample_cdf_step(const float* logits, const float* u, int rows, int V, int L, int t, long long id_stride, float* out,
                    int64_t* ids, float* logp, const int64_t* forced, const float* embed, int E, float* x_next,
                    cudaStream_t s) {
  if (rows == 0) return GIC_OK;
  ProfScope prof(PROF_SAMPLE, 4.0 * rows * V, s);
  const size_t smem = (size_t)((V + 127) >> 7) * sizeof(float);
  sample_cdf_kernel<<<rows, 256, smem, s>>>(logits, u, V, L, t, id_stride, out, ids, logp, forced, embed, E, x_next);
  return check_launch("sample_cdf_kernel");
}

// rollout group initialisation (SeqGAN-style Monte-Carlo search): rows of group t replicate the sampled caption's state
// after t steps n times: h <- hs[t][b], c <- cs[t][b], x <- embed(ids[b][t-1]), prefix ids copied.
__global__ void rollout_init_kernel(const float* __restrict__ hs_t, const float* __restrict__ cs_t,
                                    const int64_t* __restrict__ main_ids, const float* __restrict__ embed, int B, int n,
                                    int L, int t, int H, int E, int V, float* __restrict__ h, float* __restrict__ c,
                                    float* __restrict__ x, int64_t* __restrict__ roll_ids) {
  const int r = blockIdx.x;                  // row within the group: b * n + j
  const int b = r / n;
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    h[(size_t)r * H + i] = hs_t[(size_t)b * H + i];
    c[(size_t)r * H + i] = cs_t[(size_t)b * H + i];
  }
  int64_t tok = main_ids[(size_t)b * L + (t - 1)];
  if (tok < 0 || tok >= V) tok = 0;
  for (int i = threadIdx.x; i < E; i += blockDim.x) x[(size_t)r * E + i] = embed[(size_t)tok * E + i];
  for (int i = threadIdx.x; i < t; i += blockDim.x) roll_ids[(size_t)r * L + i] = main_ids[(size_t)b * L + i];
}
int rollout_init(const float* hs_t, const float* cs_t, const int64_t* main_ids, const float* embed, int B, int n, int L,
                 int t, int H, int E, int V, float* h, float* c, float* x, int64_t* roll_ids, cudaStream_t s) {
  rollout_init_kernel<<<B * n, 128, 0, s>>>(hs_t, cs_t, main_ids, embed, B, n, L, t, H, E, V, h, c, x, roll_ids);
  return check_launch("rollout_init_kernel");
}

// ---------------------------------------------------------------------------------------
// softmax backward with temperature: dz = T * p * (dp - sum_v p*dp), one CTA per (b,t) row.
// (autograd of F.softmax(gumbel_t * T), src/generator.py:69; the Gumbel add is a constant.)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
softmax_bwd_kernel(const float* __restrict__ p, const float* dp, float temperature_v, const float* __restrict__ t_dev,
                   int V, float* dz) {   // dz may alias dp
  const float temperature = pick_t(temperature_v, t_dev);
  __shared__ float red[32];
  const size_t row = blockIdx.x;
  const float* pr = p + row * V;
  const float* dr = dp + row * V;
  float* zr = dz + row * V;
  float dot = 0.f;
  for (int v = threadIdx.x; v < V; v += blockDim.x) dot = fmaf(pr[v], dr[v], dot);
  dot = block_sum(dot, red);
  for (int v = threadIdx.x; v < V; v += blockDim.x) zr[v] = temperature * pr[v] * (dr[v] - dot);
}

int softmax_bwd(const float* p, const float* dp, float temperature, int rows, int V, float* dz,
                cudaStream_t s) {
  if (rows == 0) return GIC_OK;
  ProfScope prof(PROF_SOFTMAX_BWD, 12.0 * rows * V, s);               // read p, dp; write dz
  softmax_bwd_kernel<<<rows, 256, 0, s>>>(p, dp, temperature, g_t_dev, V, dz);
  return check_launch("softmax_bwd_kernel");
}

// Softmax backward with the row dot products already known (factored path: dot = <d(emb), emb>): a pure streaming
// elementwise pass dz = T * p * (dp - dot[row]), float4, in place over dp.  12 B of HBM traffic per element.
__global__ void __launch_bounds__(256)
softmax_bwd_dot_kernel(const float4* __restrict__ p, const float4* dp, const float* __restrict__ dot, float temperature_v,
                       const float* __restrict__ t_dev, int V4, size_t n4, float4* dz) {
  const float temperature = pick_t(temperature_v, t_dev);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i0 < n4; i0 += 4 * stride) {
    float4 pv[4], dv[4];
    float dt[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const size_t i = i0 + j * stride;
      if (i < n4) { pv[j] = p[i]; dv[j] = dp[i]; dt[j] = dot[i / V4]; }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const size_t i = i0 + j * stride;
      if (i < n4) {
        float4 z;
        z.x = temperature * pv[j].x * (dv[j].x - dt[j]); z.y = temperature * pv[j].y * (dv[j].y - dt[j]);
        z.z = temperature * pv[j].z * (dv[j].z - dt[j]); z.w = temperature * pv[j].w * (dv[j].w - dt[j]);
        dz[i] = z;
      }
    }
  }
}
__global__ void softmax_bwd_dot_scalar_kernel(const float* __restrict__ p, const float* dp, const float* __restrict__ dot,
                                              float temperature_v, const float* __restrict__ t_dev, int V, size_t n,
                                              float* dz) {
  const float temperature = pick_t(temperature_v, t_dev);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    dz[i] = temperature * p[i] * (dp[i] - dot[i / V]);
}
int softmax_bwd_dot(const float* p, const float* dp, const float* dot, float temperature, int rows, int V, float* dz,
                    cudaStream_t s) {
  if (rows == 0) return GIC_OK;
  ProfScope prof(PROF_SOFTMAX_BWD, 12.0 * rows * V, s);
  const size_t n = (size_t)rows * V;
  if ((V % 4 == 0) && aligned16(p) && aligned16(dp) && aligned16(dz)) {
    const size_t n4 = n / 4;
    const int grid = (int)min((size_t)num_sms() * 8, (n4 + 1023) / 1024);
    softmax_bwd_dot_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(p), reinterpret_cast<const float4*>(dp), dot,
                                               temperature, g_t_dev, V / 4, n4, reinterpret_cast<float4*>(dz));
  } else {
    softmax_bwd_dot_scalar_kernel<<<num_sms() * 8, 256, 0, s>>>(p, dp, dot, temperature, g_t_dev, V, n, dz);
  }
  return check_launch("softmax_bwd_dot_kernel");
}

// bf16-output variant (GIC_GEMM_BF16): dz is only read by tensor-core contractions, so it is written once as bf16 with
// row pitch Vp (8 B per 4 elements instead of 16): 10 B of HBM traffic per element.
__global__ void __launch_bounds__(256)
softmax_bwd_dot_bf16_kernel(const float4* __restrict__ p, const float4* __restrict__ dp, const float* __restrict__ dot,
                            float temperature_v, const float* __restrict__ t_dev, int V4, int Vp, size_t n4,
                            unsigned short* __restrict__ dz) {
  const float temperature = pick_t(temperature_v, t_dev);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i0 = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i0 < n4; i0 += 4 * stride) {
    float4 pv[4], dv[4];
    float dt[4];
    size_t row[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const size_t i = i0 + j * stride;
      if (i < n4) { pv[j] = p[i]; dv[j] = dp[i]; row[j] = i / V4; dt[j] = dot[row[j]]; }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const size_t i = i0 + j * stride;
      if (i < n4) {
        const float z0 = temperature * pv[j].x * (dv[j].x - dt[j]), z1 = temperature * pv[j].y * (dv[j].y - dt[j]);
        const float z2 = temperature * pv[j].z * (dv[j].z - dt[j]), z3 = temperature * pv[j].w * (dv[j].w - dt[j]);
        auto bf = [](float x) { unsigned int u = __float_as_uint(x); u += 0x7fffu + ((u >> 16) & 1u); return u >> 16; };
        uint2 pk;
        pk.x = bf(z0) | (bf(z1) << 16);
        pk.y = bf(z2) | (bf(z3) << 16);
        const size_t c4 = i - row[j] * V4;
        *reinterpret_cast<uint2*>(dz + row[j] * Vp + 4 * c4) = pk;
      }
    }
  }
}
int softmax_bwd_dot_bf16(const float* p, const float* dp, const float* dot, float temperature, int rows, int V, void* dz,
                         int Vp, cudaStream_t s) {
  if (rows == 0) return GIC_OK;
  GIC_REQUIRE((V % 4 == 0) && (Vp % 4 == 0) && aligned16(p) && aligned16(dp) && aligned16(dz), GIC_ERR_SHAPE,
              "softmax_bwd_dot_bf16: V %% 4 != 0 or misaligned operands");
  ProfScope prof(PROF_SOFTMAX_BWD, 10.0 * rows * V, s);
  const size_t n4 = (size_t)rows * V / 4;
  const int grid = (int)min((size_t)num_sms() * 8, (n4 + 1023) / 1024);
  softmax_bwd_dot_bf16_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const float4*>(p), reinterpret_cast<const float4*>(dp), dot,
                                                  temperature, g_t_dev, V / 4, Vp, n4, reinterpret_cast<unsigned short*>(dz));
  return check_launch("softmax_bwd_dot_bf16_kernel");
}

// dot[row] = <a[row, :n], b[row, :n]>, one warp per row.  With a = d(emb), b = emb = p W_e^T of the discriminator's
// soft-caption embedding this is sum_v p[row,v] * d(p)[row,v] of the softmax backward without the dense d(p).
__global__ void rowdot_kernel(const float* __restrict__ a, const float* __restrict__ b, int rows, int n,
                              float* __restrict__ dot) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float s = 0.f;
  for (int j = lane; j < n; j += 32) s = fmaf(a[(size_t)row * n + j], b[(size_t)row * n + j], s);
  s = warp_sum(s);
  if (lane == 0) dot[row] = s;
}
int rowdot(const float* a, const float* b, int rows, int n, float* dot, cudaStream_t s) {
  if (rows == 0) return GIC_OK;
  rowdot_kernel<<<cdiv(rows, 8), 256, 0, s>>>(a, b, rows, n, dot);
  return check_launch("rowdot_kernel");
}

// ---------------------------------------------------------------------------------------
// embedding gradient: dW_emb[tok[b,t-1], :] += dX[t, b, :] for t >= 1 (the token fed back at
// step t-1 is the input of step t); dfeatures[b,:] = dX[0,b,:].  fp32 atomics: the order of
// duplicate-token accumulation differs from the reference (within rtol, not bitwise).
// ---------------------------------------------------------------------------------------
__global__ void embed_scatter_kernel(const float* __restrict__ dX /*[L,B,E]*/, const int64_t* __restrict__ fed /*[B,L]*/,
                                     int B, int L, int E, int V, float* __restrict__ dW_emb,
                                     float* __restrict__ dfeat) {
  const int tb = blockIdx.x;      // t * B + b
  const int t = tb / B, b = tb % B;
  const float* src = dX + (size_t)tb * E;
  if (t == 0) {
    if (dfeat)
      for (int e = threadIdx.x; e < E; e += blockDim.x) dfeat[(size_t)b * E + e] = src[e];
    return;
  }
  int64_t tok = fed[(size_t)b * L + (t - 1)];
  if (tok < 0 || tok >= V) tok = 0;
  float* dst = dW_emb + (size_t)tok * E;
  for (int e = threadIdx.x; e < E; e += blockDim.x) atomicAdd(dst + e, src[e]);
}

int embed_scatter(const float* dX, const int64_t* fed, int B, int L, int E, int V, float* dW_emb,
                  float* dfeat, cudaStream_t s) {
  embed_scatter_kernel<<<L * B, 128, 0, s>>>(dX, fed, B, L, E, V, dW_emb, dfeat);
  return check_launch("embed_scatter_kernel");
}

// ---------------------------------------------------------------------------------------
// BatchNorm1d (train mode, batch statistics, biased variance) forward / backward over [B,E].
// One warp per feature column.  (Encoder.bn, src/generator.py:16,24)
// ---------------------------------------------------------------------------------------
__global__ void bn_fwd_kernel(const float* __restrict__ y, int B, int E, const float* __restrict__ gamma,
                              const float* __restrict__ beta, float eps, float* __restrict__ out,
                              float* __restrict__ save_mean, float* __restrict__ save_rstd) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  float s = 0.f;
  for (int b = lane; b < B; b += 32) s += y[(size_t)b * E + j];
  const float mu = warp_sum(s) / B;
  float q = 0.f;
  for (int b = lane; b < B; b += 32) { const float d = y[(size_t)b * E + j] - mu; q += d * d; }
  const float var = warp_sum(q) / B;
  const float rstd = 1.0f / sqrtf(var + eps);
  for (int b = lane; b < B; b += 32)
    out[(size_t)b * E + j] = (y[(size_t)b * E + j] - mu) * rstd * gamma[j] + beta[j];
  if (lane == 0) { save_mean[j] = mu; save_rstd[j] = rstd; }
}

__global__ void bn_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dout, int B, int E,
                              const float* __restrict__ gamma, const float* __restrict__ save_mean,
                              const float* __restrict__ save_rstd, float* __restrict__ dy,
                              float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  const float mu = save_mean[j], rstd = save_rstd[j];
  float sd = 0.f, sdx = 0.f;
  for (int b = lane; b < B; b += 32) {
    const float d = dout[(size_t)b * E + j];
    const float xh = (y[(size_t)b * E + j] - mu) * rstd;
    sd += d; sdx += d * xh;
  }
  sd = warp_sum(sd); sdx = warp_sum(sdx);
  const float g = gamma[j];
  for (int b = lane; b < B; b += 32) {
    const float d = dout[(size_t)b * E + j];
    const float xh = (y[(size_t)b * E + j] - mu) * rstd;
    dy[(size_t)b * E + j] = g * rstd * (d - sd / B - xh * sdx / B);
  }
  if (lane == 0) { dgamma[j] = sdx; dbeta[j] = sd; }
}

// ---- synchronised BatchNorm (data parallel): the batch statistics are sums over ALL ranks' rows, so each half of the
// BN forward / backward is split into "local sums" and "apply with the all-reduced sums" (SURVEY.md section 8e: the one
// op of the path that is not row-local).  stats = [2][E]; count = global number of rows.
__global__ void bn_stats_kernel(const float* __restrict__ y, int B, int E, float* __restrict__ stats) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  float s = 0.f, q = 0.f;
  for (int b = lane; b < B; b += 32) { const float v = y[(size_t)b * E + j]; s += v; q = fmaf(v, v, q); }
  s = warp_sum(s); q = warp_sum(q);
  if (lane == 0) { stats[j] = s; stats[E + j] = q; }
}
__global__ void bn_apply_kernel(const float* __restrict__ y, int B, int E, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float eps, const float* __restrict__ stats, float count,
                                float* __restrict__ out, float* __restrict__ save_mean, float* __restrict__ save_rstd) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  const float mu = stats[j] / count;
  const float var = fmaxf(stats[E + j] / count - mu * mu, 0.f);        // biased variance, as BatchNorm1d in training mode
  const float rstd = 1.0f / sqrtf(var + eps);
  for (int b = lane; b < B; b += 32)
    out[(size_t)b * E + j] = (y[(size_t)b * E + j] - mu) * rstd * gamma[j] + beta[j];
  if (lane == 0) { save_mean[j] = mu; save_rstd[j] = rstd; }
}
__global__ void bn_bwd_stats_kernel(const float* __restrict__ y, const float* __restrict__ dout, int B, int E,
                                    const float* __restrict__ save_mean, const float* __restrict__ save_rstd,
                                    float* __restrict__ stats) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  const float mu = save_mean[j], rstd = save_rstd[j];
  float sd = 0.f, sdx = 0.f;
  for (int b = lane; b < B; b += 32) {
    const float d = dout[(size_t)b * E + j];
    sd += d; sdx = fmaf(d, (y[(size_t)b * E + j] - mu) * rstd, sdx);
  }
  sd = warp_sum(sd); sdx = warp_sum(sdx);
  if (lane == 0) { stats[j] = sd; stats[E + j] = sdx; }
}
// dgamma / dbeta are written as (global sum) * grad_share so that the later all-reduce(sum) of the flat gradient buffers
// (every rank holds the same value) followed by the 1/world factor of the optimizer gives the global-batch gradient.
__global__ void bn_bwd_apply_kernel(const float* __restrict__ y, const float* __restrict__ dout, int B, int E,
                                    const float* __restrict__ gamma, const float* __restrict__ save_mean,
                                    const float* __restrict__ save_rstd, const float* __restrict__ stats, float count,
                                    float grad_share, float* __restrict__ dy, float* __restrict__ dgamma,
                                    float* __restrict__ dbeta) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= E) return;
  const float mu = save_mean[j], rstd = save_rstd[j], g = gamma[j];
  const float sd = stats[j], sdx = stats[E + j];
  for (int b = lane; b < B; b += 32) {
    const float d = dout[(size_t)b * E + j];
    const float xh = (y[(size_t)b * E + j] - mu) * rstd;
    dy[(size_t)b * E + j] = g * rstd * (d - sd / count - xh * sdx / count);
  }
  if (lane == 0) { dgamma[j] = sdx * grad_share; dbeta[j] = sd * grad_share; }
}
__global__ void vec_add_kernel(const float* __restrict__ a, const float* __restrict__ b, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}
int vec_add(const float* a, const float* b, int n, float* out, cudaStream_t s) {
  vec_add_kernel<<<cdiv(n, 256), 256, 0, s>>>(a, b, n, out);
  return check_launch("vec_add_kernel");
}
// BatchNorm1d bookkeeping of a training-mode forward (src/generator.py:16: momentum 0.01): running_mean / running_var
// move towards the batch mean / UNBIASED batch variance, num_batches_tracked += 1.  count = rows the statistics ran over.
__global__ void bn_running_update_kernel(const float* __restrict__ save_mean, const float* __restrict__ save_rstd, int E,
                                         float eps, float count, float momentum, float* __restrict__ running_mean,
                                         float* __restrict__ running_var, long long* __restrict__ nbt) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0 && nbt) nbt[0] += 1;
  if (j >= E) return;
  const float r = save_rstd[j];
  const float var_b = fmaxf(1.0f / (r * r) - eps, 0.f);                       // biased batch variance
  const float var_u = count > 1.f ? var_b * (count / (count - 1.f)) : var_b;  // what BatchNorm stores
  running_mean[j] = (1.f - momentum) * running_mean[j] + momentum * save_mean[j];
  running_var[j] = (1.f - momentum) * running_var[j] + momentum * var_u;
}
int bn_running_update(const float* save_mean, const float* save_rstd, int E, float eps, float count, float momentum,
                      float* running_mean, float* running_var, long long* nbt, cudaStream_t s) {
  bn_running_update_kernel<<<cdiv(E, 128), 128, 0, s>>>(save_mean, save_rstd, E, eps, count, momentum, running_mean,
                                                        running_var, nbt);
  return check_launch("bn_running_update_kernel");
}
// eval-mode BatchNorm1d (gen.eval() in the reference's validation loops, src/training.py:213): running statistics
__global__ void bn_eval_kernel(const float* __restrict__ y, int B, int E, const float* __restrict__ gamma,
                               const float* __restrict__ beta, float eps, const float* __restrict__ running_mean,
                               const float* __restrict__ running_var, float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * E) return;
  const int j = (int)(i % E);
  out[i] = (y[i] - running_mean[j]) * (1.0f / sqrtf(running_var[j] + eps)) * gamma[j] + beta[j];
}
int bn_eval(const float* y, int B, int E, const float* gamma, const float* beta, float eps, const float* running_mean,
            const float* running_var, float* out, cudaStream_t s) {
  bn_eval_kernel<<<cdiv((long long)B * E, 256), 256, 0, s>>>(y, B, E, gamma, beta, eps, running_mean, running_var, out);
  return check_launch("bn_eval_kernel");
}
int bn_stats(const float* y, int B, int E, float* stats, cudaStream_t s) {
  bn_stats_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, B, E, stats);
  return check_launch("bn_stats_kernel");
}
int bn_apply(const float* y, int B, int E, const float* gamma, const float* beta, float eps, const float* stats,
             float count, float* out, float* save_mean, float* save_rstd, cudaStream_t s) {
  bn_apply_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, B, E, gamma, beta, eps, stats, count, out, save_mean, save_rstd);
  return check_launch("bn_apply_kernel");
}
int bn_bwd_stats(const float* y, const float* dout, int B, int E, const float* save_mean, const float* save_rstd,
                 float* stats, cudaStream_t s) {
  bn_bwd_stats_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, dout, B, E, save_mean, save_rstd, stats);
  return check_launch("bn_bwd_stats_kernel");
}
int bn_bwd_apply(const float* y, const float* dout, int B, int E, const float* gamma, const float* save_mean,
                 const float* save_rstd, const float* stats, float count, float grad_share, float* dy, float* dgamma,
                 float* dbeta, cudaStream_t s) {
  bn_bwd_apply_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, dout, B, E, gamma, save_mean, save_rstd, stats, count, grad_share, dy,
                                                 dgamma, dbeta);
  return check_launch("bn_bwd_apply_kernel");
}

int bn_fwd(const float* y, int B, int E, const float* gamma, const float* beta, float eps, float* out,
           float* save_mean, float* save_rstd, cudaStream_t s) {
  bn_fwd_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, B, E, gamma, beta, eps, out, save_mean, save_rstd);
  return check_launch("bn_fwd_kernel");
}
int bn_bwd(const float* y, const float* dout, int B, int E, const float* gamma, const float* save_mean,
           const float* save_rstd, float* dy, float* dgamma, float* dbeta, cudaStream_t s) {
  bn_bwd_kernel<<<cdiv(E, 4), 128, 0, s>>>(y, dout, B, E, gamma, save_mean, save_rstd, dy, dgamma, dbeta);
  return check_launch("bn_bwd_kernel");
}

int lstm_cell_fwd(const float* gates, const float* c_prev, int B, int H, float* acts, float* c_new,
                  float* h_new, float* htop, int L, int t, cudaStream_t s) {
  lstm_cell_fwd_kernel<<<cdiv((long long)B * H, 256), 256, 0, s>>>(gates, c_prev, B, H, acts, c_new, h_new,
                                                                  htop, L, t);
  return check_launch("lstm_cell_fwd_kernel");
}
int lstm_cell_bwd(const float* acts, const float* c_prev, const float* c_cur, const float* dh_in,
                  long long dh_stride, const float* dh_rec, float* dc_rec, int B, int H, float* dgates,
                  cudaStream_t s) {
  lstm_cell_bwd_kernel<<<cdiv((long long)B * H, 256), 256, 0, s>>>(acts, c_prev, c_cur, dh_in, dh_stride,
                                                                  dh_rec, dc_rec, B, H, dgates);
  return check_launch("lstm_cell_bwd_kernel");
}

}  // namespace gic
