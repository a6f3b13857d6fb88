// extern "C" entry points of libgic_b200.so (declared in include/gic_b200.h) and the host-side
// composition of the decode forward/backward passes.
#include "../../include/gic_b200.h"
#include <stdlib.h>
#include <new>

#include "gic_internal.cuh"

namespace gic {
// decode.cu
int gather_rows(const float*, const int64_t*, int, int, int, float*, cudaStream_t);
int vec_add(const float*, const float*, int, float*, cudaStream_t);
int sample_step(bool, const float*, const float*, float, int, int, int, int, float*, int64_t*, const int64_t*,
                const float*, int, float*, cudaStream_t, bool fast_math = false);
int softmax_bwd(const float*, const float*, float, int, int, float*, cudaStream_t);
int rowdot(const float*, const float*, int, int, float*, cudaStream_t);
int sample_cdf_step(const float*, const float*, int, int, int, int, long long, float*, int64_t*, float*, const int64_t*,
                    const float*, int, float*, cudaStream_t);
int rollout_init(const float*, const float*, const int64_t*, const float*, int, int, int, int, int, int, int, float*,
                 float*, float*, int64_t*, cudaStream_t);
int softmax_bwd_dot(const float*, const float*, const float*, float, int, int, float*, cudaStream_t);
int softmax_bwd_dot_bf16(const float*, const float*, const float*, float, int, int, void*, int, cudaStream_t);
int colsum_bf16(const void*, int, int, int, bool, float*, cudaStream_t);
int embed_scatter(const float*, const int64_t*, int, int, int, int, float*, float*, cudaStream_t);
int bn_fwd(const float*, int, int, const float*, const float*, float, float*, float*, float*, cudaStream_t);
int bn_bwd(const float*, const float*, int, int, const float*, const float*, const float*, float*, float*, float*,
           cudaStream_t);
int lstm_cell_fwd(const float*, const float*, int, int, float*, float*, float*, float*, int, int, cudaStream_t);
int lstm_cell_bwd(const float*, const float*, const float*, const float*, long long, const float*, float*, int, int,
                  float*, cudaStream_t);
// attn.cu
int attn_fwd(const float*, const float*, const float*, const float*, int, int, int, int, float*, float*, cudaStream_t);
int attn_bwd_step(const float*, const float*, const float*, const float*, const float*, const float*, int, int, int, int,
                  float*, float*, cudaStream_t);
int attn_bwd_accum(const float*, const float*, const float*, const float*, const float*, const float*, int, int, int, int, int,
                   float*, float*, float*, cudaStream_t);
// lstm_tcgen05.cu
int bptt_step_tc(const float* dG_t, const float* W_hh, const float* acts_prev, const float* c_prev, const float* c_cur,
                 const float* dh_top, float* dc_rec, float* dG_out, int B, int H, int L, int t, cudaStream_t stream,
                 bool* handled);
int bptt_persistent_tc(float* dG, const float* W_hh, const float* acts, const float* cs, const float* dh_top, const float* dc_in,
                       unsigned int* counter, int B, int H, int L, cudaStream_t stream, bool* handled);
// vocab_sample_tcgen05.cu: fused decode step (projection + sample of step t, recurrent contraction and cell of step t + 1)
bool decode_step_plan(int B, int V, int H);
int decode_step_tc(const float* hs_t1, const float* W_out, const float* b_out, const float* W_hh, const float* EW, float* R, unsigned int* rec_done, const float* u_t, float T,
                   const float* T_dev, int B, int V, int H, int L, int t, int last, float* out, int64_t* ids,
                   const int64_t* forced, const float* embed, int E, float* x_next, const float* c_prev, float* c_out,
                   float* h_out, float* acts, float* htop, float* scratch, cudaStream_t stream, bool* handled);
int lstm_step_tc(const float*, int, const float*, const float*, const float*, const float*, const float*, const float*,
                 int, int, float*, float*, float*, float*, int, int, cudaStream_t, bool*);
// beam_tcgen05.cu
size_t vocab_topk_ws_floats(int M, int V, int K);
int vocab_topk(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K, float* logp,
               int64_t* tokens, float* lse, const uint32_t* ban, float* ws, cudaStream_t s);
size_t decode_beam_ws_floats(int B, int K, int L, int V, int E, int H, int layers, const gic_decode_constraints_t* c);
int decode_beam(int mode, const float* features, const float* W_emb, const float* const* W_ih, const float* const* W_hh,
                const float* const* b_ih, const float* const* b_hh, const float* W_out, const float* b_out, int B, int K,
                int L, int V, int E, int H, int layers, int64_t eos, float length_penalty,
                const gic_decode_constraints_t* c, int64_t* ids, float* scores, int32_t* lengths, int32_t* trace, float* ws,
                cudaStream_t s);
size_t vocab_target_ws_floats(int M, int V);
int vocab_target_scores(int mode, const float* h, const float* W_out, const float* b_out, const int64_t* targets, int M, int V,
                        int H, int L, const int32_t* lengths, float* logp, float* lse, int64_t* argmax, uint8_t* correct,
                        float* caption_logp, float* ws, cudaStream_t s);
int teacher_inputs(const float* features, const int64_t* captions, const float* embed, int B, int L, int E, int V, float* x,
                   cudaStream_t s);
size_t vocab_sample_ws_floats(int M, int V, int top_k);
int vocab_sample(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int t, float T,
                 int top_k, float top_p, int64_t* tokens, float* logp, const SampleDecode* d, const uint32_t* ban, float* ws,
                 cudaStream_t s);
int sample_init(const float* features, int n, int M, const SampleDecode& d, cudaStream_t s);
// disc.cu
int scale_inplace(float*, size_t, float, cudaStream_t);
// loss_optim.cu
int gan_loss(int, const float*, const float*, const float*, int, float*, float*, float*, float*, cudaStream_t);
int grad_sqnorm(const float*, size_t, float*, cudaStream_t);
int rollout_q(const float*, const float*, int, int, int, int, float*, cudaStream_t);
int pg_loss(const float*, const int64_t*, const float*, int, int, int, int, float*, float*, float*, cudaStream_t);
int clip_adam(float*, const float*, float*, float*, size_t, const float*, float, float, int, float, float, float,
              float, const float*, cudaStream_t);
Ctx* ctx_set_current(Ctx*);
void set_temperature_device(const float*);
void set_rng(unsigned long long, unsigned long long, const unsigned long long*);
int philox_uniform(uint32_t, unsigned long long, size_t, float*, cudaStream_t);
int philox_keep_mask(uint32_t, size_t, float, uint8_t*, cudaStream_t);
int bn_stats(const float*, int, int, float*, cudaStream_t);
int bn_running_update(const float*, const float*, int, float, float, float, float*, float*, long long*, cudaStream_t);
int bn_eval(const float*, int, int, const float*, const float*, float, const float*, const float*, float*, cudaStream_t);
int bn_apply(const float*, int, int, const float*, const float*, float, const float*, float, float*, float*, float*, cudaStream_t);
int bn_bwd_stats(const float*, const float*, int, int, const float*, const float*, float*, cudaStream_t);
int bn_bwd_apply(const float*, const float*, int, int, const float*, const float*, const float*, const float*, float, float,
                 float*, float*, float*, cudaStream_t);
int pack_captions(const int32_t*, const int32_t*, int, int, int64_t*, int32_t*, cudaStream_t);
const float* temperature_device();
void disc_set_prepared(const float*);
int disc_prepare(int, const float*, const float*, const float*, int, const float*, const float*, int, float*, cudaStream_t);
const char* last_error();
unsigned long long launch_count();
unsigned long long kernel_launches(const char*);
int kernel_names(char*, int);
void prof_begin();
void prof_end(double*, double*, unsigned long long*);
// disc_api.cu-style wrappers implemented in disc.cu
int disc_fwd_entry(int mode, const float* inp_soft, const int64_t* ids, int N, int L, int V, int De, int R,
                   int n_groups, const int* fs, const int* nf, const float* W_e, const float* const* cw,
                   const float* const* cb, const float* W_h, const float* b_h, const float* W_f, const float* b_f,
                   int Hd, const float* W_o, const float* b_o, int n_heads, const uint8_t* const* keep, float drop_p,
                   float* const* logits, float* saved, float* ws, cudaStream_t s);
int disc_bwd_entry(int mode, const float* dlogits, const uint8_t* keep, float drop_p, const float* inp_soft,
                   const int64_t* ids, int N, int L, int V, int De, int R, int n_groups, const int* fs, const int* nf,
                   const float* W_e, const float* const* cw, const float* const* cb, const float* W_h,
                   const float* W_f, const float* b_f, int Hd, const float* W_o, const float* b_o, const float* saved,
                   float* ws, float* dW_e, float* const* dcw, float* const* dcb, float* dW_h, float* db_h,
                   float* dW_f, float* db_f, float* dW_o, float* db_o, float* dinp, int want_param, int accumulate,
                   cudaStream_t s);

// attention saved layout (floats): Ak[B,P,Da] | Av[B,P,E] | q[L,B,Da] | alpha[L,B,P]
// attention backward workspace:    dAk[B,P,Da] | dAv[B,P,E] | dq[L,B,Da] | ds[L,B,P]
struct AttnLayout {
  size_t Ak, Av, q, alpha, total;      // saved
  size_t dAk, dAv, dq, ds, ws_total;   // workspace
  AttnLayout(int B, int L, int P, int Da, int E) {
    Ak = 0; Av = a4((size_t)B * P * Da); q = Av + a4((size_t)B * P * E); alpha = q + a4((size_t)L * B * Da);
    total = alpha + a4((size_t)L * B * P);
    dAk = 0; dAv = a4((size_t)B * P * Da); dq = dAv + a4((size_t)B * P * E); ds = dq + a4((size_t)L * B * Da);
    ws_total = ds + a4((size_t)L * B * P);
  }
};

// saved-for-backward layout of the decode (floats):
//   xs[L][B][E] | per layer l: hs[l][(L+1)][B][H], cs[l][(L+1)][B][H], acts[l][L][B][4H] | htop[B][L][H]
struct DecodeSaved {
  size_t xs, hs0, cs0, acts0, per_layer, htop, total;
  DecodeSaved(int B, int L, int E, int H, int layers) {
    const size_t BH = (size_t)B * H;
    xs = 0;
    size_t off = a4((size_t)L * B * E);
    hs0 = off;
    cs0 = hs0 + a4((size_t)(L + 1) * BH);
    acts0 = cs0 + a4((size_t)(L + 1) * BH);
    per_layer = 2 * a4((size_t)(L + 1) * BH) + a4((size_t)L * BH * 4);
    htop = off + (size_t)layers * per_layer;
    total = htop + a4((size_t)B * L * H);
  }
  size_t hs(int l) const { return hs0 + (size_t)l * per_layer; }
  size_t cs(int l) const { return cs0 + (size_t)l * per_layer; }
  size_t acts(int l) const { return acts0 + (size_t)l * per_layer; }
};

// One time step of the LSTM stack.  Layer 0 reads x[B,E], layer l > 0 the h that layer l - 1 just wrote.  Tensor-core modes
// run lstm_step_tc (both contractions + the cell update in one tcgen05 kernel); where it declines, and in exact fp32, two
// GEMMs into gates[B,4H] and lstm_cell_fwd.  acts may be NULL; the top layer also writes htop[B,L,H] at step t unless NULL.
struct LstmLayerIO { const float* h_prev; const float* c_prev; float* h_new; float* c_new; float* acts; };
static int lstm_stack_step(int mode, const float* x, const LstmLayerIO* io, int layers, const float* const* W_ih,
                           const float* const* W_hh, const float* const* b_ih, const float* const* b_hh, int B, int E, int H,
                           float* htop, float* gates, int L, int t, cudaStream_t s) {
  for (int l = 0; l < layers; ++l) {
    const float* xin = (l == 0) ? x : io[l - 1].h_new;
    const int In = (l == 0) ? E : H;
    const LstmLayerIO& y = io[l];
    float* ht = (l == layers - 1) ? htop : nullptr;
    bool fused = false;
    if (mode == GEMM_TF32 || mode == GEMM_BF16)
      GIC_TRY(lstm_step_tc(xin, In, y.h_prev, W_ih[l], W_hh[l], b_ih[l], b_hh[l], y.c_prev, B, H, y.acts, y.c_new, y.h_new, ht,
                           L, t, s, &fused));
    if (!fused) {
      // gates = x W_ih^T + b_ih + h W_hh^T + b_hh          (src/generator.py:61)
      GIC_TRY(gemm(mode, false, true, B, 4 * H, In, 1.f, xin, In, W_ih[l], In, 0.f, gates, 4 * H, b_ih[l], s));
      GIC_TRY(gemm(mode, false, true, B, 4 * H, H, 1.f, y.h_prev, H, W_hh[l], H, 1.f, gates, 4 * H, b_hh[l], s));
      GIC_TRY(lstm_cell_fwd(gates, y.c_prev, B, H, y.acts, y.c_new, y.h_new, ht, L, t, s));
    }
  }
  return GIC_OK;
}

// forward workspace of the decode (floats):
//   gates[B][4H] | logits[B][V] | vs_scratch (fused projection + sampler: barrier counters + row statistics)
//   | u_slice[B][V] (uniforms of one step: u == NULL, unfused path)
//   | fused decode step: EW[V][4H] (embed W_ih^T + b_ih + b_hh) | R[B][4H] | rec_done (64 u32 counters) | bsum[4H] (b_ih + b_hh)
struct DecodeFwdWs {
  size_t gates, logits, vs_scratch, u_slice, EW, R, rec_done, bsum, total;
  DecodeFwdWs(int B, int V, int H) {
    const size_t G4 = (size_t)4 * H;
    gates = 0; logits = a4(B * G4); vs_scratch = logits + a4((size_t)B * V);
    u_slice = vs_scratch + a4(vocab_sample_scratch_floats(B, V)); EW = u_slice + a4((size_t)B * V);
    R = EW + V * G4; rec_done = R + B * G4; bsum = rec_done + 64; total = bsum + G4;
  }
};

// pretrain: 0 = Gumbel-softmax (u[L,B,V], out = soft captions), 1 = pretrain (out = logits, greedy), 2 = inverse-CDF
// categorical sampling (EXTENSION: u[L,B], out = logits or NULL, logp[B,L] or NULL)
static int decode_fwd(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                      const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                      const float* W_out, const float* b_out, const float* u, float T, int pretrain,
                      const int64_t* forced, int B, int L, int V, int E, int H, int layers, float* out, int64_t* ids,
                      float* saved, float* ws, cudaStream_t s, float* logp = nullptr, const gic_attn_t* at = nullptr) {
  GIC_REQUIRE(B >= 0 && L >= 1 && V >= 1 && E >= 1 && H >= 1 && layers >= 1 && layers <= 8, GIC_ERR_SHAPE,
              "decode_sample_fwd: bad shape B=%d L=%d V=%d E=%d H=%d layers=%d", B, L, V, E, H, layers);
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(features && W_emb && W_ih && W_hh && b_ih && b_hh && W_out && b_out && (out || pretrain == 2) && ids &&
                  saved && ws, GIC_ERR_NULL, "decode_sample_fwd: NULL pointer");
  GIC_REQUIRE(pretrain != 2 || u, GIC_ERR_NULL, "decode_sample_cdf_fwd: uniforms required");
  // pretrain == 0 with u == NULL: the Gumbel uniforms are drawn by the library (Philox state of gic_set_rng; the fused
  // kernel draws its tile on the fly, the separate sampler reads a [B,V] slice filled by the same generator)
  const DecodeSaved sv(B, L, E, H, layers);
  const DecodeFwdWs w(B, V, H);
  const size_t BH = (size_t)B * H, BE = (size_t)B * E;
  float* gates = ws + w.gates;
  float* logits = ws + w.logits;
  float* vs_scratch = ws + w.vs_scratch;
  float* u_slice = ws + w.u_slice;
  cudaMemcpyAsync(saved + sv.xs, features, BE * sizeof(float), cudaMemcpyDeviceToDevice, s);
  for (int l = 0; l < layers; ++l) {
    cudaMemsetAsync(saved + sv.hs(l), 0, BH * sizeof(float), s);
    cudaMemsetAsync(saved + sv.cs(l), 0, BH * sizeof(float), s);
  }
  const AttnLayout al(B, L, at ? at->P : 1, at ? at->Da : 1, E);
  if (at) {
    GIC_REQUIRE(at->grid && at->W_k && at->W_v && at->W_q && at->w_e && at->saved && at->P >= 1 && at->Cf >= 1 && at->Da >= 1,
                GIC_ERR_NULL, "decode_sample_fwd_attn: incomplete attention block");
    // once per image: key / value projections of the feature grid
    GIC_TRY(gemm(mode, false, true, B * at->P, at->Da, at->Cf, 1.f, at->grid, at->Cf, at->W_k, at->Cf, 0.f, at->saved + al.Ak,
                 at->Da, nullptr, s));
    GIC_TRY(gemm(mode, false, true, B * at->P, E, at->Cf, 1.f, at->grid, at->Cf, at->W_v, at->Cf, 0.f, at->saved + al.Av, E,
                 nullptr, s));
  }
  if (pretrain == 0 && !at && layers == 1 && (mode == GEMM_TF32 || mode == GEMM_BF16) && (E % 4) == 0 && decode_step_plan(B, V, H)) {
    // Tensor-core modes, one layer, Gumbel-softmax sampling: ONE kernel per decode step (vocab_sample_tcgen05.cu).  The
    // LSTM pre-activation of step t + 1 is embed[tok_t] W_ih^T + h_t W_hh^T + biases: the recurrent half needs only h_t, so
    // it runs as extra tiles of step t's projection / sample launch, and the token-dependent half is a row of
    // EW = embed W_ih^T [V, 4H], rebuilt once per decode (the weights change every optimizer step), added in the cell
    // tail of the CTA that sampled the token.  Step 0 (input = features, h = 0) is the stand-alone LSTM kernel.
    float* EW = ws + w.EW;
    float* R = ws + w.R;
    unsigned int* rec_done = reinterpret_cast<unsigned int*>(ws + w.rec_done);
    float* bsum = ws + w.bsum;
    bool ok0 = false;
    GIC_TRY(lstm_step_tc(saved + sv.xs, E, saved + sv.hs(0), W_ih[0], W_hh[0], b_ih[0], b_hh[0], saved + sv.cs(0), B, H,
                         saved + sv.acts(0), saved + sv.cs(0) + BH, saved + sv.hs(0) + BH, saved + sv.htop, L, 0, s, &ok0));
    if (ok0) {
      if (L > 1) {
        GIC_TRY(vec_add(b_ih[0], b_hh[0], 4 * H, bsum, s));
        GIC_TRY(gemm(mode, false, true, V, 4 * H, E, 1.f, W_emb, E, W_ih[0], E, 0.f, EW, 4 * H, bsum, s, PROF_GEMM_DECODE));
      }
      cudaMemsetAsync(rec_done, 0, 64 * sizeof(unsigned int), s);
      for (int t = 0; t < L; ++t) {
        const int last = (t + 1 == L);
        bool done = false;
        ProfScope prof(PROF_VOCAB_SAMPLE, 8.0 * B * V, s);
        GIC_TRY(decode_step_tc(saved + sv.hs(0) + (size_t)(t + 1) * BH, W_out, b_out, W_hh[0], EW, R, rec_done,
                               u ? u + (size_t)t * B * V : nullptr, T, temperature_device(), B, V, H, L, t, last, out, ids, forced,
                               W_emb, E, last ? nullptr : saved + sv.xs + (size_t)(t + 1) * BE,
                               saved + sv.cs(0) + (size_t)(t + 1) * BH, saved + sv.cs(0) + (size_t)(t + 2) * BH,
                               saved + sv.hs(0) + (size_t)(t + 2) * BH, saved + sv.acts(0) + (size_t)(t + 1) * BH * 4,
                               saved + sv.htop, vs_scratch, s, &done));
        GIC_REQUIRE(done, GIC_ERR_UNSUPPORTED, "decode_sample_fwd: fused decode step declined after its plan accepted the shape");
      }
      return GIC_OK;
    }
  }
  for (int t = 0; t < L; ++t) {
    if (at) {
      // q_t = h_{t-1} W_q^T (top... layer 0 state), scores / softmax over the P locations / context added to x_t
      float* q_t = at->saved + al.q + (size_t)t * B * at->Da;
      GIC_TRY(gemm(mode, false, true, B, at->Da, H, 1.f, saved + sv.hs(0) + (size_t)t * BH, H, at->W_q, H, 0.f, q_t, at->Da,
                   nullptr, s));
      GIC_TRY(attn_fwd(at->saved + al.Ak, at->saved + al.Av, q_t, at->w_e, B, at->P, at->Da, E,
                       saved + sv.xs + (size_t)t * BE, at->saved + al.alpha + (size_t)t * B * at->P, s));
    }
    LstmLayerIO io[8];
    for (int l = 0; l < layers; ++l)
      io[l] = {saved + sv.hs(l) + (size_t)t * BH, saved + sv.cs(l) + (size_t)t * BH, saved + sv.hs(l) + (size_t)(t + 1) * BH,
               saved + sv.cs(l) + (size_t)(t + 1) * BH, saved + sv.acts(l) + (size_t)t * BH * 4};
    GIC_TRY(lstm_stack_step(mode, saved + sv.xs + (size_t)t * BE, io, layers, W_ih, W_hh, b_ih, b_hh, B, E, H, saved + sv.htop,
                            gates, L, t, s));
    const float* htop_t = saved + sv.hs(layers - 1) + (size_t)(t + 1) * BH;
    float* x_next = (t + 1 < L) ? saved + sv.xs + (size_t)(t + 1) * BE : nullptr;
    if (pretrain == 0 && (mode == GEMM_TF32 || mode == GEMM_BF16)) {
      // tensor-core modes: projection + Gumbel-softmax + sample + next-token gather in ONE kernel (logits stay on chip)
      bool fused_vs = false;
      {
        ProfScope prof(PROF_VOCAB_SAMPLE, 8.0 * B * V, s);
        GIC_TRY(vocab_sample_tc(htop_t, H, W_out, b_out, u ? u + (size_t)t * B * V : nullptr, T, temperature_device(), B, V, H, L, t, out,
                                ids, forced, W_emb, E, x_next, vs_scratch, s, &fused_vs));
      }
      if (fused_vs) continue;
    }
    GIC_TRY(gemm(mode, false, true, B, V, H, 1.f, htop_t, H, W_out, H, 0.f, logits, V, b_out, s, PROF_GEMM_DECODE));   // :64,68
    if (pretrain == 2)
      GIC_TRY(sample_cdf_step(logits, u + (size_t)t * B, B, V, L, t, L, out, ids, logp, forced, W_emb, E, x_next, s));
    else {
      const float* u_t = nullptr;
      if (!pretrain) {
        if (u) u_t = u + (size_t)t * B * V;
        else { GIC_TRY(philox_uniform(0x47u /*RNG_TAG_GUMBEL*/, (unsigned long long)t * B * V, (size_t)B * V, u_slice, s)); u_t = u_slice; }
      }
      GIC_TRY(sample_step(pretrain != 0, logits, u_t, T, B, V, L, t, out, ids,
                            forced, W_emb, E, x_next, s, /*fast_math=*/mode == GEMM_TF32 || mode == GEMM_BF16));
    }
  }
  return GIC_OK;
}

// teacher-forced scoring workspace (floats): x[L][B][E] | per layer: h[2][B][H] (ping-pong), c[B][H] (updated in place)
// | gates[B][4H] | htop[B][L][H] | target-logit producer
struct ScoreWs {
  size_t x, state, per_layer, gates, htop, prod, total;
  ScoreWs(int B, int L, int V, int E, int H, int layers) {
    const size_t BH = a4((size_t)B * H);
    x = 0;
    state = a4((size_t)L * B * E);
    per_layer = 3 * BH;
    gates = state + (size_t)layers * per_layer;
    htop = gates + a4((size_t)B * 4 * H);
    prod = htop + a4((size_t)B * L * H);
    total = prod + vocab_target_ws_floats(B * L, V);
  }
};

// Teacher-forced log-likelihood of captions[B,L] (gic_score_captions): the LSTM stack over the forced inputs with the
// kernels decode_fwd runs (so the hidden states are Decoder.sample(pretrain=True, forced_ids)'s), then ONE projection of
// all B L rows with the target pick, and one consumer.  No host sync.
static int score_captions(int mode, const float* features, const int64_t* captions, const int32_t* lengths, const float* W_emb,
                          const float* const* W_ih, const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                          const float* W_out, const float* b_out, int B, int L, int V, int E, int H, int layers, float* logp,
                          float* caption_logp, uint8_t* correct, float* ws, cudaStream_t s) {
  const ScoreWs w(B, L, V, E, H, layers);
  const size_t BH = a4((size_t)B * H);
  GIC_TRY(teacher_inputs(features, captions, W_emb, B, L, E, V, ws + w.x, s));
  for (int l = 0; l < layers; ++l) {
    float* st = ws + w.state + (size_t)l * w.per_layer;
    cudaMemsetAsync(st, 0, (size_t)B * H * sizeof(float), s);                    // h of step -1
    cudaMemsetAsync(st + 2 * BH, 0, (size_t)B * H * sizeof(float), s);          // c
  }
  for (int t = 0; t < L; ++t) {
    LstmLayerIO io[8];
    for (int l = 0; l < layers; ++l) {
      float* st = ws + w.state + (size_t)l * w.per_layer;
      io[l] = {st + (t & 1) * BH, st + 2 * BH, st + ((t + 1) & 1) * BH, st + 2 * BH, nullptr};
    }
    GIC_TRY(lstm_stack_step(mode, ws + w.x + (size_t)t * B * E, io, layers, W_ih, W_hh, b_ih, b_hh, B, E, H, ws + w.htop,
                            ws + w.gates, L, t, s));
  }
  return vocab_target_scores(mode, ws + w.htop, W_out, b_out, captions, B * L, V, H, L, lengths, logp, nullptr, nullptr,
                             correct, caption_logp, ws + w.prod, s);
}

// sampled-caption workspace (floats): x[M][E] | per layer: h[2][M][H] (ping-pong), c[M][H] (updated in place)
// | gates[M][4H] | fin[M] | sampling-step workspace | ban bitmaps (BanWs, size 0 unconstrained), M = B n
struct SampleCaptionsWs {
  size_t x, state, per_layer, gates, fin, step, ban, total;
  SampleCaptionsWs(int M, int V, int E, int H, int layers, int top_k, int L = 1, const gic_decode_constraints_t* c = nullptr) {
    const size_t MH = a4((size_t)M * H);
    x = 0;
    state = a4((size_t)M * E);
    per_layer = 3 * MH;
    gates = state + (size_t)layers * per_layer;
    fin = gates + a4((size_t)M * 4 * H);
    step = fin + a4((size_t)M);
    ban = step + vocab_sample_ws_floats(M, V, top_k);
    total = ban + BanWs(M, V, L, c).total;
  }
};

// n sampled captions per image (gic_sample_captions): rows m = b n + j start from features[b] with h = c = 0; every step
// runs the LSTM stack (lstm_stack_step, as scoring does), the producer and sample_rows_kernel, which appends the token and
// writes the next input.  Always L steps, no host sync.  With constraints (c != NULL) ban_rows_kernel rebuilds the rows'
// ban bitmaps before the producer of every step.
static int sample_captions(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                           const float* const* W_hh, const float* const* b_ih, const float* const* b_hh, const float* W_out,
                           const float* b_out, int B, int n, int L, int V, int E, int H, int layers, int eos, float T,
                           int top_k, float top_p, const gic_decode_constraints_t* c, int64_t* ids, float* caption_logp,
                           int32_t* lengths, float* ws, cudaStream_t s) {
  const int M = B * n;
  const SampleCaptionsWs w(M, V, E, H, layers, top_k, L, c);
  const BanWs bw(M, V, L, c);
  const size_t MH = a4((size_t)M * H);
  SampleDecode d = {ids, reinterpret_cast<int*>(ws + w.fin), lengths, caption_logp, ws + w.x, W_emb, L, E, eos};
  GIC_TRY(sample_init(features, n, M, d, s));
  for (int l = 0; l < layers; ++l) {
    float* st = ws + w.state + (size_t)l * w.per_layer;
    cudaMemsetAsync(st, 0, (size_t)M * H * sizeof(float), s);                    // h of step -1
    cudaMemsetAsync(st + 2 * MH, 0, (size_t)M * H * sizeof(float), s);          // c
  }
  if (c) GIC_TRY(ban_base(c, V, bw, ws + w.ban, s));
  for (int t = 0; t < L; ++t) {
    LstmLayerIO io[8];
    for (int l = 0; l < layers; ++l) {
      float* st = ws + w.state + (size_t)l * w.per_layer;
      io[l] = {st + (t & 1) * MH, st + 2 * MH, st + ((t + 1) & 1) * MH, st + 2 * MH, nullptr};
    }
    GIC_TRY(lstm_stack_step(mode, ws + w.x, io, layers, W_ih, W_hh, b_ih, b_hh, M, E, H, nullptr, ws + w.gates, L, t, s));
    if (c) GIC_TRY(ban_rows(c, M, V, L, t, eos, d.fin, ids, nullptr, B, n, bw, ws + w.ban, s));
    GIC_TRY(vocab_sample(mode, io[layers - 1].h_new, W_out, b_out, M, V, H, t, T, top_k, top_p, nullptr, nullptr, &d,
                         c ? reinterpret_cast<const uint32_t*>(ws + w.ban + bw.ban) : nullptr, ws + w.step, s));
  }
  return GIC_OK;
}

// backward workspace (floats):
//   dlogits[B*L*V] | dHtop[B*L*H] | dG[layers][L][B][4H] | dh_rec[layers][B][H] | dc_rec[layers][B][H]
//   | dxin[B][H] | dX[L][B][E] | dot[B*L] | bf16 copies for GIC_GEMM_BF16: dz[B*L][Vp], htop[B*L][H], W_out[V][H]
struct DecodeBwdWs {
  size_t dlogits, dhtop, dG, dhrec, dcrec, dxin, dX, dot, dz_bf, htop_bf, wout_bf, total;
  int Vp;
  DecodeBwdWs(int B, int L, int V, int E, int H, int layers) {
    const size_t BH = (size_t)B * H;
    dlogits = 0;
    dhtop = a4((size_t)B * L * V);
    dG = dhtop + a4((size_t)B * L * H);
    dhrec = dG + (size_t)layers * a4((size_t)L * BH * 4);
    dcrec = dhrec + (size_t)layers * a4(BH);
    dxin = dcrec + (size_t)layers * a4(BH);
    dX = dxin + a4(BH);
    dot = dX + a4((size_t)L * B * E);
    Vp = ((V + 63) / 64) * 64;
    dz_bf = dot + a4((size_t)B * L);
    htop_bf = dz_bf + a4((size_t)B * L * Vp / 2);
    wout_bf = htop_bf + a4(((size_t)B * L * H + 1) / 2);
    total = wout_bf + a4(((size_t)V * H + 1) / 2);
  }
};

// dout source: dense dout[B,L,V], or (dout == nullptr) the factored form d(emb)[B*L,De] x W_e[De,V] coming out of the
// discriminator's embedding layer, with emb[B*L,De] = out W_e^T saved by its forward.
//
// Data-parallel hook: dW_out / db_out (40 % of the generator's gradient bytes at c2) are final long before the serial
// BPTT tail.  When the caller registered an event (gic_set_vocab_grads_event) it is recorded on the stream right after
// those two buffers are complete, so their all-reduce can run on another stream underneath the rest of the backward.
static int record_vocab_grads_event(cudaStream_t s) {
  cudaEvent_t ev = ctx().vocab_grads_event;
  if (!ev) return GIC_OK;
  cudaError_t e = cudaEventRecord(ev, s);
  if (e != cudaSuccess) { set_error("cudaEventRecord(vocab grads): %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  return GIC_OK;
}
static int record_embed_grads_event(cudaStream_t s) {
  cudaEvent_t ev = ctx().embed_grads_event;
  if (!ev) return GIC_OK;
  cudaError_t e = cudaEventRecord(ev, s);
  if (e != cudaSuccess) { set_error("cudaEventRecord(embed grads): %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  return GIC_OK;
}
static int decode_bwd(int mode, const float* dout, const float* demb, const float* emb, const float* W_e, int De,
                      const float* out, const int64_t* fed, const float* W_emb,
                      const float* const* W_ih, const float* const* W_hh, const float* W_out, float T, int pretrain,
                      int B, int L, int V, int E, int H, int layers, const float* saved, float* ws, float* dW_emb,
                      float* const* dW_ih, float* const* dW_hh, float* const* db_ih, float* const* db_hh,
                      float* dW_out, float* db_out, float* dfeat, int accumulate, cudaStream_t s,
                      const gic_attn_t* at = nullptr) {
  GIC_REQUIRE(B >= 0 && L >= 1 && V >= 1 && E >= 1 && H >= 1 && layers >= 1 && layers <= 8, GIC_ERR_SHAPE,
              "decode_sample_bwd: bad shape");
  const AttnLayout al(B, L, at ? at->P : 1, at ? at->Da : 1, E);
  if (at) {
    GIC_REQUIRE(at->grid && at->W_k && at->W_v && at->W_q && at->w_e && at->saved && at->ws && at->dW_k && at->dW_v &&
                    at->dW_q && at->dw_e, GIC_ERR_NULL, "decode_sample_bwd_attn: incomplete attention block");
    GIC_REQUIRE(!accumulate, GIC_ERR_UNSUPPORTED, "decode_sample_bwd_attn: accumulate is not supported");
    cudaMemsetAsync(at->dw_e, 0, (size_t)at->Da * sizeof(float), s);               // accumulated with atomics
  }
  if (B == 0) return GIC_OK;
  GIC_REQUIRE((dout || (demb && emb && W_e && De >= 1)) && fed && W_emb && W_ih && W_hh && W_out && saved && ws && dW_emb && dW_ih && dW_hh && db_ih &&
                  db_hh && dW_out && db_out, GIC_ERR_NULL, "decode_sample_bwd: NULL pointer");
  GIC_REQUIRE(pretrain || out, GIC_ERR_NULL, "decode_sample_bwd: soft captions `out` required");
  const DecodeSaved sv(B, L, E, H, layers);
  const DecodeBwdWs w(B, L, V, E, H, layers);
  const size_t BH = (size_t)B * H, BE = (size_t)B * E;
  const float beta = accumulate ? 1.f : 0.f;
  const int BL = B * L;
  const size_t dG_stride = a4((size_t)L * BH * 4);

  // 1. through the tempered softmax (the Gumbel add is a constant)
  bool vocab_done = false;          // GIC_GEMM_BF16: step 2 already done on bf16 operands
  const float* dlogits = dout;
  if (dout == nullptr) {
    GIC_REQUIRE(!pretrain, GIC_ERR_UNSUPPORTED, "decode_sample_bwd: factored dout is the adversarial path only");
    // dz = T p (d(emb) W_e - <d(emb), emb>): d(probs) is never materialised in tensor-core mode
    if (mode == GEMM_FP32) {
      // parity mode keeps the reference's own arithmetic: dense d(probs), then sum_v p dp per row (at T = 100 the
      // softmax saturates and dz is a difference of nearly equal numbers; a different dot product shows up there)
      GIC_TRY(gemm(mode, false, false, BL, V, De, 1.f, demb, De, W_e, V, 0.f, ws + w.dlogits, V, nullptr, s));
      GIC_TRY(softmax_bwd(out, ws + w.dlogits, T, BL, V, ws + w.dlogits, s));
    } else {
      GIC_TRY(rowdot(demb, emb, BL, De, ws + w.dot, s));
      if (mode == GEMM_BF16 && (V % 4 == 0) && (H % 8 == 0)) {
        // bf16 operands for the two 52-GF contractions of the vocab projection's backward: dz is written once as bf16
        // (it is read by nothing else), htop and W_out are converted (2.6 M + 5.1 M elements)
        void* dz_bf = ws + w.dz_bf;
        void* htop_bf = ws + w.htop_bf;
        void* wout_bf = ws + w.wout_bf;
        // one streaming kernel: d(probs) tile in TMEM -> dz (bf16) + db_out; the separate kernels are the fallback
        bool dz_done = false;
        {
          ProfScope prof(PROF_SOFTMAX_BWD, 6.0 * BL * V, s);        // algorithmic HBM bytes: read p (4), write dz (2)
          GIC_TRY(dz_fused_tc(demb, De, W_e, out, ws + w.dot, T, temperature_device(), BL, V, dz_bf, w.Vp, db_out,
                              accumulate, s, &dz_done));
        }
        if (!dz_done) {
          GIC_TRY(gemm(mode, false, false, BL, V, De, 1.f, demb, De, W_e, V, 0.f, ws + w.dlogits, V, nullptr, s));
          GIC_TRY(softmax_bwd_dot_bf16(out, ws + w.dlogits, ws + w.dot, T, BL, V, dz_bf, w.Vp, s));
          GIC_TRY(colsum_bf16(dz_bf, BL, V, w.Vp, accumulate != 0, db_out, s));
        }
        GIC_TRY(f32_to_bf16(saved + sv.htop, BL, H, H, htop_bf, H, s));
        GIC_TRY(f32_to_bf16(W_out, V, H, H, wout_bf, H, s));
        GIC_TRY(gemm_bf16(true, false, V, H, BL, 1.f, dz_bf, w.Vp, htop_bf, H, beta, dW_out, H, nullptr, s));
        GIC_TRY(record_vocab_grads_event(s));
        GIC_TRY(gemm_bf16(false, false, BL, H, V, 1.f, dz_bf, w.Vp, wout_bf, H, 0.f, ws + w.dhtop, H, nullptr, s));
        vocab_done = true;
      }
      if (!vocab_done) {
        GIC_TRY(gemm(mode, false, false, BL, V, De, 1.f, demb, De, W_e, V, 0.f, ws + w.dlogits, V, nullptr, s));
        GIC_TRY(softmax_bwd_dot(out, ws + w.dlogits, ws + w.dot, T, BL, V, ws + w.dlogits, s));
      }
    }
    dlogits = ws + w.dlogits;
  } else if (!pretrain) {
    GIC_TRY(softmax_bwd(out, dout, T, BL, V, ws + w.dlogits, s));
    dlogits = ws + w.dlogits;
  }
  // 2. vocab projection: db_out, dW_out[V,H] = dlogits^T htop, dHtop[B*L,H] = dlogits W_out
  if (!vocab_done) {
    GIC_TRY(colsum_f32(dlogits, BL, V, V, 1.f, accumulate != 0, db_out, s));
    GIC_TRY(gemm(mode, true, false, V, H, BL, 1.f, dlogits, V, saved + sv.htop, H, beta, dW_out, H, nullptr, s));
    GIC_TRY(record_vocab_grads_event(s));
    GIC_TRY(gemm(mode, false, false, BL, H, V, 1.f, dlogits, V, W_out, H, 0.f, ws + w.dhtop, H, nullptr, s));
  }
  // 3. BPTT through (h, c)
  cudaMemsetAsync(ws + w.dhrec, 0, (size_t)2 * layers * a4(BH) * sizeof(float), s);   // dh_rec and dc_rec
  const bool bptt_fusable = (mode == GEMM_TF32 || mode == GEMM_BF16) && layers == 1 && !at;
  bool bptt_fused_prev = false;
  bool bptt_done = false;
  if (bptt_fusable && L >= 2) {
    // the whole recurrence as one persistent launch (bptt_tcgen05.cu): cell backward of the last step first, then
    // dG[L-2 .. 0]; the zeroed dh_rec buffer (no longer needed after the first cell kernel) lends its first word to the
    // grid-wide arrival counter
    const int t = L - 1;
    GIC_TRY(lstm_cell_bwd(saved + sv.acts(0) + (size_t)t * BH * 4, saved + sv.cs(0) + (size_t)t * BH,
                          saved + sv.cs(0) + (size_t)(t + 1) * BH, ws + w.dhtop + (size_t)t * H, (long long)L * H, ws + w.dhrec,
                          ws + w.dcrec, B, H, ws + w.dG + (size_t)t * BH * 4, s));
    GIC_TRY(bptt_persistent_tc(ws + w.dG, W_hh[0], saved + sv.acts(0), saved + sv.cs(0), ws + w.dhtop, ws + w.dcrec,
                               reinterpret_cast<unsigned int*>(ws + w.dhrec), B, H, L, s, &bptt_done));
    bptt_fused_prev = !bptt_done;      // not handled: the loop below continues from the cell backward already done
  }
  for (int t = bptt_done ? -1 : L - 1; t >= 0; --t) {
    for (int l = layers - 1; l >= 0; --l) {
      const bool top = (l == layers - 1);
      const float* dh_in = top ? ws + w.dhtop + (size_t)t * H : ws + w.dxin;
      const long long stride = top ? (long long)L * H : (long long)H;
      float* dG_lt = ws + w.dG + (size_t)l * dG_stride + (size_t)t * BH * 4;
      float* dhrec = ws + w.dhrec + (size_t)l * a4(BH);
      float* dcrec = ws + w.dcrec + (size_t)l * a4(BH);
      if (!bptt_fused_prev)      // else dG of this step (and dc) came out of the fused kernel launched for step t + 1
        GIC_TRY(lstm_cell_bwd(saved + sv.acts(l) + (size_t)t * BH * 4, saved + sv.cs(l) + (size_t)t * BH,
                              saved + sv.cs(l) + (size_t)(t + 1) * BH, dh_in, stride, dhrec, dcrec, B, H, dG_lt, s));
      bptt_fused_prev = false;
      // recurrent gradient for step t-1: dh_rec = dgates W_hh    ([B,4H] x [4H,H])
      if (t > 0) {
        // tensor-core modes, one layer, no attention: contraction (split-K over a cluster, DSMEM reduction) and the cell
        // backward of step t - 1 in ONE kernel (bptt_tcgen05.cu)
        if (bptt_fusable)
          GIC_TRY(bptt_step_tc(dG_lt, W_hh[0], saved + sv.acts(0) + (size_t)(t - 1) * BH * 4, saved + sv.cs(0) + (size_t)(t - 1) * BH,
                               saved + sv.cs(0) + (size_t)t * BH, ws + w.dhtop, dcrec, ws + w.dG + (size_t)(t - 1) * BH * 4, B, H, L, t,
                               s, &bptt_fused_prev));
        if (!bptt_fused_prev)
          GIC_TRY(gemm(mode, false, false, B, H, 4 * H, 1.f, dG_lt, 4 * H, W_hh[l], H, 0.f, dhrec, H, nullptr, s));
      }
      if (at && l == 0) {
        // attention: dx'_t = dG_t W_ih (per step: dq_t feeds the recurrent gradient), then the attention backward
        float* dXt = ws + w.dX + (size_t)t * BE;
        float* dq_t = at->ws + al.dq + (size_t)t * B * at->Da;
        GIC_TRY(gemm(mode, false, false, B, E, 4 * H, 1.f, dG_lt, 4 * H, W_ih[0], E, 0.f, dXt, E, nullptr, s));
        GIC_TRY(attn_bwd_step(dXt, at->saved + al.alpha + (size_t)t * B * at->P, at->saved + al.q + (size_t)t * B * at->Da,
                              at->saved + al.Ak, at->saved + al.Av, at->w_e, B, at->P, at->Da, E, dq_t,
                              at->ws + al.ds + (size_t)t * B * at->P, s));
        if (t > 0)   // q_t = h_{t-1} W_q^T: dh_{t-1} += dq_t W_q
          GIC_TRY(gemm(mode, false, false, B, H, at->Da, 1.f, dq_t, at->Da, at->W_q, H, 1.f, dhrec, H, nullptr, s));
      }
      // gradient to the layer below at the same step
      if (l > 0)
        GIC_TRY(gemm(mode, false, false, B, H, 4 * H, 1.f, dG_lt, 4 * H, W_ih[l], H, 0.f, ws + w.dxin, H, nullptr, s));
    }
  }
  // 4. input gradients first (no attention): dX[L*B,E] = dG[0] W_ih[0]; t = 0 -> dfeatures, t >= 1 -> embedding rows.
  // They need dG only, and dW_emb is 40 % of the generator's gradient bytes: formed BEFORE the weight-gradient GEMMs, its
  // all-reduce (gic_set_embed_grads_event) runs underneath them instead of in the exposed tail of the step.
  if (!at) {
    GIC_TRY(gemm(mode, false, false, L * B, E, 4 * H, 1.f, ws + w.dG, 4 * H, W_ih[0], E, 0.f, ws + w.dX, E, nullptr, s));
    if (!accumulate) cudaMemsetAsync(dW_emb, 0, (size_t)V * E * sizeof(float), s);
    GIC_TRY(embed_scatter(ws + w.dX, fed, B, L, E, V, dW_emb, dfeat, s));
    GIC_TRY(record_embed_grads_event(s));
  }
  // 5. weight gradients, batched over all (t, b)
  for (int l = 0; l < layers; ++l) {
    const float* dG_l = ws + w.dG + (size_t)l * dG_stride;           // [L*B, 4H]
    const int In = (l == 0) ? E : H;
    const float* xin = (l == 0) ? saved + sv.xs : saved + sv.hs(l - 1) + BH;   // inputs of step t, t-major
    GIC_TRY(gemm(mode, true, false, 4 * H, In, L * B, 1.f, dG_l, 4 * H, xin, In, beta, dW_ih[l], In, nullptr, s));
    GIC_TRY(gemm(mode, true, false, 4 * H, H, L * B, 1.f, dG_l, 4 * H, saved + sv.hs(l), H, beta, dW_hh[l], H, nullptr, s));
    // both biases enter the same pre-activation (src/generator.py:61), so their gradients are the same column sums
    GIC_TRY(colsum_f32(dG_l, L * B, 4 * H, 4 * H, 1.f, accumulate != 0, db_ih[l], s));
    if (!accumulate) cudaMemcpyAsync(db_hh[l], db_ih[l], (size_t)4 * H * sizeof(float), cudaMemcpyDeviceToDevice, s);
    else GIC_TRY(colsum_f32(dG_l, L * B, 4 * H, 4 * H, 1.f, true, db_hh[l], s));
  }
  // 6. attention: the per-step dX is already there
  if (at) {
    // dAk, dAv, dw_e: sums over the L steps, formed once (attn.cu)
    GIC_TRY(attn_bwd_accum(at->saved + al.alpha, at->ws + al.ds, at->saved + al.q, ws + w.dX, at->saved + al.Ak, at->w_e, B, L,
                           at->P, at->Da, E, at->ws + al.dAk, at->ws + al.dAv, at->dw_e, s));
    // attention parameter gradients: dW_q = sum_t dq_t^T h_{t-1} (step 0 sees h = 0), dW_k = dAk^T grid, dW_v = dAv^T grid
    GIC_TRY(gemm(mode, true, false, at->Da, H, L * B, 1.f, at->ws + al.dq, at->Da, saved + sv.hs(0), H, 0.f, at->dW_q, H,
                 nullptr, s));
    GIC_TRY(gemm(mode, true, false, at->Da, at->Cf, B * at->P, 1.f, at->ws + al.dAk, at->Da, at->grid, at->Cf, 0.f, at->dW_k,
                 at->Cf, nullptr, s));
    GIC_TRY(gemm(mode, true, false, E, at->Cf, B * at->P, 1.f, at->ws + al.dAv, E, at->grid, at->Cf, 0.f, at->dW_v, at->Cf,
                 nullptr, s));
    if (!accumulate) cudaMemsetAsync(dW_emb, 0, (size_t)V * E * sizeof(float), s);
    GIC_TRY(embed_scatter(ws + w.dX, fed, B, L, E, V, dW_emb, dfeat, s));
    GIC_TRY(record_embed_grads_event(s));
  }
  (void)BE;
  return GIC_OK;
}

// ---------------------------------------------------------------------------------------------------------
// EXTENSION: Monte-Carlo rollouts (SeqGAN-style search; SURVEY.md 8a row B2, not in the reference).
// For every prefix length t = 1..L-1 of the sampled captions main_ids[B,L], n continuations are sampled with the
// generator policy (inverse-CDF sampling, one uniform per row and step).  Row (t-1)*B*n + b*n + j of roll_ids[Mmax,L]
// holds the j-th completed caption of prefix t of image b.  The active set grows by B*n rows per step and is always a
// contiguous prefix of the row space, so every step is ONE batched LSTM step + vocab projection over all live rollouts
// (up to (L-1)*B*n rows): the shapes that make the decode GEMMs tensor-bound.
// workspace: h[2][Mmax,H] | c[Mmax,H] | x[Mmax,E] | gates[Mmax,4H] (fp32 mode) | logits[chunk,V]
// ---------------------------------------------------------------------------------------------------------
struct RolloutWs {
  size_t h0, h1, c, x, gates, logits, total;
  int chunk;
  RolloutWs(int B, int L, int V, int E, int H, int n) {
    const size_t M = (size_t)(L - 1) * B * n;
    chunk = (int)(M < 8192 ? M : 8192);
    h0 = 0; h1 = a4(M * H); c = h1 + a4(M * H); x = c + a4(M * H); gates = x + a4(M * E);
    logits = gates + a4(M * 4 * H);
    total = logits + a4((size_t)chunk * V);
  }
};

static int decode_rollouts(int mode, const float* saved, const int64_t* main_ids, const float* W_emb, const float* W_ih,
                           const float* W_hh, const float* b_ih, const float* b_hh, const float* W_out,
                           const float* b_out, const float* u_roll, int B, int L, int V, int E, int H, int n,
                           int64_t* roll_ids, float* ws, cudaStream_t s) {
  GIC_REQUIRE(B >= 1 && L >= 2 && V >= 1 && E >= 1 && H >= 1 && n >= 1, GIC_ERR_SHAPE, "decode_rollouts: bad shape");
  GIC_REQUIRE(saved && main_ids && W_emb && W_ih && W_hh && b_ih && b_hh && W_out && b_out && u_roll && roll_ids && ws,
              GIC_ERR_NULL, "decode_rollouts: NULL pointer");
  const DecodeSaved sv(B, L, E, H, 1);
  const RolloutWs w(B, L, V, E, H, n);
  const size_t BH = (size_t)B * H, G = (size_t)B * n, Mmax = (size_t)(L - 1) * G;
  float* hbuf[2] = {ws + w.h0, ws + w.h1};
  float* c = ws + w.c;
  float* x = ws + w.x;
  int cur = 0;
  for (int t = 1; t < L; ++t) {
    // group t joins: state after t steps of the sampled caption, next input = embed(token t-1)
    const size_t r0 = (size_t)(t - 1) * G;
    GIC_TRY(rollout_init(saved + sv.hs(0) + (size_t)t * BH, saved + sv.cs(0) + (size_t)t * BH, main_ids, W_emb, B, n, L, t,
                         H, E, V, hbuf[cur] + r0 * H, c + r0 * H, x + r0 * E, roll_ids + r0 * L, s));
    const int M = (int)((size_t)t * G);                       // live rows
    float* hn = hbuf[cur ^ 1];
    bool fused = false;
    if (mode == GEMM_TF32 || mode == GEMM_BF16)
      GIC_TRY(lstm_step_tc(x, E, hbuf[cur], W_ih, W_hh, b_ih, b_hh, c, M, H, nullptr, c, hn, nullptr, L, t, s, &fused));
    if (!fused) {
      float* gates = ws + w.gates;
      GIC_TRY(gemm(mode, false, true, M, 4 * H, E, 1.f, x, E, W_ih, E, 0.f, gates, 4 * H, b_ih, s));
      GIC_TRY(gemm(mode, false, true, M, 4 * H, H, 1.f, hbuf[cur], H, W_hh, H, 1.f, gates, 4 * H, b_hh, s));
      GIC_TRY(lstm_cell_fwd(gates, c, M, H, nullptr, c, hn, nullptr, L, t, s));
    }
    for (int m0 = 0; m0 < M; m0 += w.chunk) {
      const int mc = (M - m0 < w.chunk) ? (M - m0) : w.chunk;
      GIC_TRY(gemm(mode, false, true, mc, V, H, 1.f, hn + (size_t)m0 * H, H, W_out, H, 0.f, ws + w.logits, V, b_out, s));
      GIC_TRY(sample_cdf_step(ws + w.logits, u_roll + (size_t)t * Mmax + m0, mc, V, L, t, L, nullptr,
                              roll_ids + (size_t)m0 * L, nullptr, nullptr, W_emb, E, x + (size_t)m0 * E, s));
    }
    cur ^= 1;
  }
  return GIC_OK;
}

static int require_device() {
  static int cached = -1;
  if (cached == GIC_OK) return GIC_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { set_error("no CUDA device: %s (libgic_b200 has no CPU fallback)", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) { set_error("cudaDeviceGetAttribute: %s", cudaGetErrorString(e)); return GIC_ERR_CUDA; }
  if (major != 10) { set_error("device compute capability %d.x is not sm_100 (B200)", major); return GIC_ERR_ARCH; }
  cached = GIC_OK;
  return GIC_OK;
}

}  // namespace gic

using namespace gic;
#define S(x) reinterpret_cast<cudaStream_t>(x)

extern "C" {

int gic_version(void) { return 100; }
const char* gic_last_error(void) { return last_error(); }
int gic_check_device(void) { return require_device(); }
unsigned long long gic_launch_count(void) { return launch_count(); }
unsigned long long gic_kernel_launches(const char* name) { return kernel_launches(name); }
int gic_kernel_names(char* buf, int cap) { return kernel_names(buf, cap); }
void gic_prof_begin(void) { prof_begin(); }
void gic_prof_end(double* ms, double* work, unsigned long long* calls) { prof_end(ms, work, calls); }

int gic_gemm(int mode, int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda,
             const float* B, int ldb, float beta, float* C, int ldc, const float* bias, gic_stream_t stream) {
  GIC_TRY(require_device());
  return gemm(mode, transA != 0, transB != 0, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, S(stream));
}

int gic_gemm_bf16(int transA, int transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B,
                  int ldb, float beta, float* C, int ldc, const float* bias, gic_stream_t stream) {
  GIC_TRY(require_device());
  return gemm_bf16(transA != 0, transB != 0, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, S(stream));
}

int gic_encoder_fwd(int mode, const float* pooled, int B, int Fin, int E, const float* W, const float* b,
                    const float* gamma, const float* beta, float eps, float* lin_out, float* save_mean,
                    float* save_rstd, float* features, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && Fin >= 1 && E >= 1, GIC_ERR_SHAPE, "encoder_fwd: bad shape");
  GIC_REQUIRE(pooled && W && b && gamma && beta && lin_out && save_mean && save_rstd && features, GIC_ERR_NULL,
              "encoder_fwd: NULL pointer");
  GIC_TRY(gemm(mode, false, true, B, E, Fin, 1.f, pooled, Fin, W, Fin, 0.f, lin_out, E, b, S(stream)));
  return bn_fwd(lin_out, B, E, gamma, beta, eps, features, save_mean, save_rstd, S(stream));
}

int gic_encoder_bwd(int mode, const float* dfeatures, const float* pooled, const float* lin_out,
                    const float* save_mean, const float* save_rstd, const float* W, const float* gamma, int B,
                    int Fin, int E, float* dlin_ws, float* dW, float* db, float* dgamma, float* dbeta, int accumulate,
                    gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && Fin >= 1 && E >= 1, GIC_ERR_SHAPE, "encoder_bwd: bad shape");
  GIC_REQUIRE(dfeatures && pooled && lin_out && save_mean && save_rstd && gamma && dlin_ws && dW && db && dgamma && dbeta,
              GIC_ERR_NULL, "encoder_bwd: NULL pointer");
  GIC_REQUIRE(!accumulate, GIC_ERR_UNSUPPORTED, "encoder_bwd: accumulate is not supported");
  (void)W;
  GIC_TRY(bn_bwd(lin_out, dfeatures, B, E, gamma, save_mean, save_rstd, dlin_ws, dgamma, dbeta, S(stream)));
  GIC_TRY(gemm(mode, true, false, E, Fin, B, 1.f, dlin_ws, E, pooled, Fin, 0.f, dW, Fin, nullptr, S(stream)));
  return colsum_f32(dlin_ws, B, E, E, 1.f, false, db, S(stream));
}

int gic_encoder_bn_running_update(const float* save_mean, const float* save_rstd, int E, float eps, float count,
                                  float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                                  gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(E >= 1 && count >= 1.f && momentum >= 0.f && momentum <= 1.f, GIC_ERR_SHAPE, "encoder_bn_running_update: bad argument");
  GIC_REQUIRE(save_mean && save_rstd && running_mean && running_var, GIC_ERR_NULL, "encoder_bn_running_update: NULL pointer");
  return bn_running_update(save_mean, save_rstd, E, eps, count, momentum, running_mean, running_var,
                           reinterpret_cast<long long*>(num_batches_tracked), S(stream));
}

int gic_encoder_fwd_eval(int mode, const float* pooled, int B, int Fin, int E, const float* W, const float* b,
                         const float* gamma, const float* beta, float eps, const float* running_mean,
                         const float* running_var, float* lin_out, float* features, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && Fin >= 1 && E >= 1, GIC_ERR_SHAPE, "encoder_fwd_eval: bad shape");
  GIC_REQUIRE(pooled && W && b && gamma && beta && running_mean && running_var && lin_out && features, GIC_ERR_NULL,
              "encoder_fwd_eval: NULL pointer");
  GIC_TRY(gemm(mode, false, true, B, E, Fin, 1.f, pooled, Fin, W, Fin, 0.f, lin_out, E, b, S(stream)));
  return bn_eval(lin_out, B, E, gamma, beta, eps, running_mean, running_var, features, S(stream));
}

// ---- synchronised-BatchNorm variant of the encoder projection (data parallel; see decode.cu) ----
int gic_encoder_fwd_stats(int mode, const float* pooled, int B, int Fin, int E, const float* W, const float* b,
                          float* lin_out, float* stats, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && Fin >= 1 && E >= 1, GIC_ERR_SHAPE, "encoder_fwd_stats: bad shape");
  GIC_REQUIRE(pooled && W && b && lin_out && stats, GIC_ERR_NULL, "encoder_fwd_stats: NULL pointer");
  GIC_TRY(gemm(mode, false, true, B, E, Fin, 1.f, pooled, Fin, W, Fin, 0.f, lin_out, E, b, S(stream)));
  return bn_stats(lin_out, B, E, stats, S(stream));
}
int gic_encoder_fwd_apply(const float* lin_out, int B, int E, const float* gamma, const float* beta, float eps,
                          const float* stats, float count, float* save_mean, float* save_rstd, float* features,
                          gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && E >= 1 && count >= 1.f, GIC_ERR_SHAPE, "encoder_fwd_apply: bad shape");
  GIC_REQUIRE(lin_out && gamma && beta && stats && save_mean && save_rstd && features, GIC_ERR_NULL, "encoder_fwd_apply: NULL pointer");
  return bn_apply(lin_out, B, E, gamma, beta, eps, stats, count, features, save_mean, save_rstd, S(stream));
}
int gic_encoder_bwd_stats(const float* dfeatures, const float* lin_out, const float* save_mean, const float* save_rstd,
                          int B, int E, float* stats, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && E >= 1, GIC_ERR_SHAPE, "encoder_bwd_stats: bad shape");
  GIC_REQUIRE(dfeatures && lin_out && save_mean && save_rstd && stats, GIC_ERR_NULL, "encoder_bwd_stats: NULL pointer");
  return bn_bwd_stats(lin_out, dfeatures, B, E, save_mean, save_rstd, stats, S(stream));
}
int gic_encoder_bwd_apply(int mode, const float* dfeatures, const float* pooled, const float* lin_out,
                          const float* save_mean, const float* save_rstd, const float* gamma, int B, int Fin, int E,
                          const float* stats, float count, float grad_share, float* dlin_ws, float* dW, float* db,
                          float* dgamma, float* dbeta, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 1 && Fin >= 1 && E >= 1 && count >= 1.f, GIC_ERR_SHAPE, "encoder_bwd_apply: bad shape");
  GIC_REQUIRE(dfeatures && pooled && lin_out && save_mean && save_rstd && gamma && stats && dlin_ws && dW && db && dgamma && dbeta,
              GIC_ERR_NULL, "encoder_bwd_apply: NULL pointer");
  GIC_TRY(bn_bwd_apply(lin_out, dfeatures, B, E, gamma, save_mean, save_rstd, stats, count, grad_share, dlin_ws, dgamma, dbeta,
                       S(stream)));
  GIC_TRY(gemm(mode, true, false, E, Fin, B, 1.f, dlin_ws, E, pooled, Fin, 0.f, dW, Fin, nullptr, S(stream)));
  return colsum_f32(dlin_ws, B, E, E, 1.f, false, db, S(stream));
}

int gic_sample_step(int pretrain, const float* logits, const float* u, float temperature, int B, int V, int L, int t,
                    float* out, int64_t* ids, const int64_t* forced_ids, const float* embed, int E, float* x_next,
                    gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 0 && V >= 1 && L >= 1 && t >= 0 && t < L, GIC_ERR_SHAPE, "sample_step: bad shape");
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(logits && out && ids && (pretrain || u), GIC_ERR_NULL, "sample_step: NULL pointer");
  GIC_REQUIRE(!x_next || embed, GIC_ERR_NULL, "sample_step: embed table required for x_next");
  return sample_step(pretrain != 0, logits, u, temperature, B, V, L, t, out, ids, forced_ids, embed, E, x_next,
                     S(stream));
}

size_t gic_attn_saved_floats(int B, int L, int P, int Da, int E) { return AttnLayout(B, L, P, Da, E).total; }
size_t gic_attn_bwd_workspace_floats(int B, int L, int P, int Da, int E) { return AttnLayout(B, L, P, Da, E).ws_total; }

int gic_decode_sample_fwd_attn(const gic_attn_t* attn, int mode, const float* features, const float* W_emb,
                               const float* const* W_ih, const float* const* W_hh, const float* const* b_ih,
                               const float* const* b_hh, const float* W_out, const float* b_out, const float* u,
                               float temperature, int pretrain, const int64_t* forced_ids, int B, int L, int V, int E,
                               int H, int layers, float* out, int64_t* ids, float* saved, float* workspace,
                               gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(attn, GIC_ERR_NULL, "decode_sample_fwd_attn: NULL attention block");
  return decode_fwd(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, u, temperature, pretrain, forced_ids,
                    B, L, V, E, H, layers, out, ids, saved, workspace, S(stream), nullptr, attn);
}

int gic_decode_sample_bwd_attn(const gic_attn_t* attn, int mode, const float* dout, const float* demb, const float* emb,
                               const float* W_e, int De, const float* out, const int64_t* fed_ids, const float* W_emb,
                               const float* const* W_ih, const float* const* W_hh, const float* W_out,
                               float temperature, int pretrain, int B, int L, int V, int E, int H, int layers,
                               const float* saved, float* workspace, float* dW_emb, float* const* dW_ih,
                               float* const* dW_hh, float* const* db_ih, float* const* db_hh, float* dW_out,
                               float* db_out, float* dfeatures, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(attn, GIC_ERR_NULL, "decode_sample_bwd_attn: NULL attention block");
  return decode_bwd(mode, dout, demb, emb, W_e, De, out, fed_ids, W_emb, W_ih, W_hh, W_out, temperature, pretrain, B, L,
                    V, E, H, layers, saved, workspace, dW_emb, dW_ih, dW_hh, db_ih, db_hh, dW_out, db_out, dfeatures, 0,
                    S(stream), attn);
}

int gic_sample_cdf_step(const float* logits, const float* u, int B, int V, int L, int t, float* out, int64_t* ids,
                        float* logp, const int64_t* forced_ids, const float* embed, int E, float* x_next,
                        gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 0 && V >= 1 && L >= 1 && t >= 0 && t < L, GIC_ERR_SHAPE, "sample_cdf_step: bad shape");
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(logits && u && ids, GIC_ERR_NULL, "sample_cdf_step: NULL pointer");
  GIC_REQUIRE(!x_next || embed, GIC_ERR_NULL, "sample_cdf_step: embed table required for x_next");
  return sample_cdf_step(logits, u, B, V, L, t, L, out, ids, logp, forced_ids, embed, E, x_next, S(stream));
}

size_t gic_decode_saved_floats(int B, int L, int E, int H, int layers) { return DecodeSaved(B, L, E, H, layers).total; }
size_t gic_decode_fwd_workspace_floats(int B, int V, int H) { return DecodeFwdWs(B, V, H).total; }
size_t gic_decode_bwd_workspace_floats(int B, int L, int V, int E, int H, int layers) {
  return DecodeBwdWs(B, L, V, E, H, layers).total;
}

int gic_decode_sample_fwd(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                          const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                          const float* W_out, const float* b_out, const float* u, float temperature, int pretrain,
                          const int64_t* forced_ids, int B, int L, int V, int E, int H, int layers, float* out,
                          int64_t* ids, float* saved, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  return decode_fwd(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, u, temperature, pretrain, forced_ids,
                    B, L, V, E, H, layers, out, ids, saved, workspace, S(stream));
}

int gic_decode_sample_bwd(int mode, const float* dout, const float* out, const int64_t* fed_ids, const float* W_emb,
                          const float* const* W_ih, const float* const* W_hh, const float* W_out, float temperature,
                          int pretrain, int B, int L, int V, int E, int H, int layers, const float* saved,
                          float* workspace, float* dW_emb, float* const* dW_ih, float* const* dW_hh,
                          float* const* db_ih, float* const* db_hh, float* dW_out, float* db_out, float* dfeatures,
                          int accumulate, gic_stream_t stream) {
  GIC_TRY(require_device());
  return decode_bwd(mode, dout, nullptr, nullptr, nullptr, 0, out, fed_ids, W_emb, W_ih, W_hh, W_out, temperature,
                    pretrain, B, L, V, E, H, layers, saved, workspace, dW_emb, dW_ih, dW_hh, db_ih, db_hh, dW_out, db_out,
                    dfeatures, accumulate, S(stream));
}

int gic_decode_sample_bwd_factored(int mode, const float* demb, const float* emb, const float* W_e, int De,
                                   const float* out, const int64_t* fed_ids, const float* W_emb,
                                   const float* const* W_ih, const float* const* W_hh, const float* W_out,
                                   float temperature, int B, int L, int V, int E, int H, int layers, const float* saved,
                                   float* workspace, float* dW_emb, float* const* dW_ih, float* const* dW_hh,
                                   float* const* db_ih, float* const* db_hh, float* dW_out, float* db_out,
                                   float* dfeatures, int accumulate, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(demb && emb && W_e && De >= 1, GIC_ERR_NULL, "decode_sample_bwd_factored: NULL factor");
  return decode_bwd(mode, nullptr, demb, emb, W_e, De, out, fed_ids, W_emb, W_ih, W_hh, W_out, temperature, 0, B, L, V,
                    E, H, layers, saved, workspace, dW_emb, dW_ih, dW_hh, db_ih, db_hh, dW_out, db_out, dfeatures,
                    accumulate, S(stream));
}

size_t gic_disc_bwd_demb_offset_floats(int N, int L, int De, int R, int F) { return DiscBwdWs(N, L, De, R, F).demb; }

int gic_decode_sample_cdf_fwd(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                              const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                              const float* W_out, const float* b_out, const float* u, const int64_t* forced_ids, int B,
                              int L, int V, int E, int H, int layers, float* logits_out, int64_t* ids, float* logp,
                              float* saved, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  return decode_fwd(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, u, 1.f, 2, forced_ids, B, L, V, E, H,
                    layers, logits_out, ids, saved, workspace, S(stream), logp);
}

size_t gic_decode_rollouts_workspace_floats(int B, int L, int V, int E, int H, int n_roll) {
  return RolloutWs(B, L, V, E, H, n_roll).total;
}

int gic_decode_rollouts(int mode, const float* saved, const int64_t* main_ids, const float* W_emb, const float* W_ih,
                        const float* W_hh, const float* b_ih, const float* b_hh, const float* W_out,
                        const float* b_out, const float* u_roll, int B, int L, int V, int E, int H, int n_roll,
                        int64_t* roll_ids, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  return decode_rollouts(mode, saved, main_ids, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, u_roll, B, L, V, E, H,
                         n_roll, roll_ids, workspace, S(stream));
}

int gic_rollout_rewards(const float* roll_logits, const float* main_logits, int B, int L, int n_roll, int R, float* Q,
                        gic_stream_t stream) {
  GIC_TRY(require_device());
  return rollout_q(roll_logits, main_logits, B, L, n_roll, R, Q, S(stream));
}

int gic_ce_loss_fwd_bwd(const float* logits, const int64_t* targets, int B, int L, int V, float* loss, float* dlogits,
                        gic_stream_t stream) {
  GIC_TRY(require_device());
  return pg_loss(logits, targets, nullptr, 0, B, L, V, loss, dlogits, nullptr, S(stream));
}

int gic_pg_loss_fwd_bwd(const float* logits, const int64_t* ids, const float* Q, int baseline_mode, int B, int L, int V,
                        float* loss, float* dlogits, float* logp, gic_stream_t stream) {
  GIC_TRY(require_device());
  return pg_loss(logits, ids, Q, baseline_mode, B, L, V, loss, dlogits, logp, S(stream));
}

// Constrained generation: a constraint block with every constraint off is no constraint (NULL).
static const gic_decode_constraints_t* active_constraints(const gic_decode_constraints_t* c) {
  return (c && (c->min_length != 0 || c->no_repeat_ngram_size != 0 || c->n_bad != 0)) ? c : nullptr;
}
// GIC_ERR_SHAPE unless 0 <= min_length <= L, no_repeat_ngram_size >= 0, n_bad >= 0 and every step keeps at least
// max(width, 1) allowed columns; GIC_ERR_NULL for n_bad > 0 without bad_ids
static int constraints_check(const gic_decode_constraints_t* c, int L, int V, int width, const char* who) {
  if (!c) return GIC_OK;
  GIC_REQUIRE(c->min_length >= 0 && c->min_length <= L && c->no_repeat_ngram_size >= 0 && c->n_bad >= 0, GIC_ERR_SHAPE,
              "%s: bad constraints min_length=%d no_repeat_ngram_size=%d n_bad=%d L=%d", who, c->min_length,
              c->no_repeat_ngram_size, c->n_bad, L);
  const long long allowed = (long long)V - c->n_bad - (c->min_length > 0 ? 1 : 0) - (c->no_repeat_ngram_size > 0 ? L - 1 : 0);
  GIC_REQUIRE((width > 1 ? width : 1) <= allowed, GIC_ERR_SHAPE,
              "%s: constraints may leave %lld allowed tokens of V=%d, fewer than %d", who, allowed, V, width > 1 ? width : 1);
  GIC_REQUIRE(c->n_bad == 0 || c->bad_ids, GIC_ERR_NULL, "%s: NULL bad_ids with n_bad=%d", who, c->n_bad);
  return GIC_OK;
}

size_t gic_vocab_topk_workspace_floats(int M, int V, int K) { return vocab_topk_ws_floats(M, V, K); }
int gic_vocab_topk(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K,
                   float* logp, int64_t* tokens, float* lse, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(M >= 0 && V >= 1 && H >= 1 && K >= 1 && K <= 16 && K <= V, GIC_ERR_SHAPE,
              "vocab_topk: bad shape M=%d V=%d H=%d K=%d", M, V, H, K);
  if (M == 0) return GIC_OK;
  GIC_REQUIRE(h && W_out && b_out && logp && tokens && workspace, GIC_ERR_NULL, "vocab_topk: NULL pointer");
  return vocab_topk(mode, h, W_out, b_out, M, V, H, K, logp, tokens, lse, nullptr, workspace, S(stream));
}
int gic_vocab_topk_masked(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K,
                          float* logp, int64_t* tokens, float* lse, const uint32_t* ban, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(M >= 0 && V >= 1 && H >= 1 && K >= 1 && K <= 16 && K <= V, GIC_ERR_SHAPE,
              "vocab_topk_masked: bad shape M=%d V=%d H=%d K=%d", M, V, H, K);
  if (M == 0) return GIC_OK;
  GIC_REQUIRE(h && W_out && b_out && logp && tokens && ban && workspace, GIC_ERR_NULL, "vocab_topk_masked: NULL pointer");
  return vocab_topk(mode, h, W_out, b_out, M, V, H, K, logp, tokens, lse, ban, workspace, S(stream));
}
size_t gic_decode_beam_workspace_floats(int B, int K, int L, int V, int E, int H, int layers) {
  return decode_beam_ws_floats(B, K, L, V, E, H, layers, nullptr);
}
size_t gic_decode_beam_constrained_workspace_floats(int B, int K, int L, int V, int E, int H, int layers,
                                                    const gic_decode_constraints_t* c) {
  return decode_beam_ws_floats(B, K, L, V, E, H, layers, active_constraints(c));
}
int gic_decode_beam(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                    const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                    const float* W_out, const float* b_out, int B, int K, int L, int V, int E, int H, int layers,
                    int64_t eos_id, float length_penalty, int64_t* ids, float* scores, int32_t* lengths, int32_t* trace,
                    float* workspace, gic_stream_t stream) {
  return gic_decode_beam_constrained(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, B, K, L, V, E, H, layers,
                                     eos_id, length_penalty, nullptr, ids, scores, lengths, trace, workspace, stream);
}
int gic_decode_beam_constrained(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                                const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                                const float* W_out, const float* b_out, int B, int K, int L, int V, int E, int H, int layers,
                                int64_t eos_id, float length_penalty, const gic_decode_constraints_t* constraints,
                                int64_t* ids, float* scores, int32_t* lengths, int32_t* trace, float* workspace,
                                gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 0 && K >= 1 && K <= 16 && K <= V && L >= 1 && V >= 1 && E >= 1 && H >= 1 && layers >= 1 && layers <= 8 &&
                  eos_id >= 0 && eos_id < V,
              GIC_ERR_SHAPE, "decode_beam: bad shape B=%d K=%d L=%d V=%d E=%d H=%d layers=%d eos_id=%lld", B, K, L, V, E, H,
              layers, (long long)eos_id);
  const gic_decode_constraints_t* c = active_constraints(constraints);
  GIC_TRY(constraints_check(c, L, V, K, "decode_beam"));
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(features && W_emb && W_ih && W_hh && b_ih && b_hh && W_out && b_out && ids && scores && lengths && workspace,
              GIC_ERR_NULL, "decode_beam: NULL pointer");
  for (int l = 0; l < layers; ++l)
    GIC_REQUIRE(W_ih[l] && W_hh[l] && b_ih[l] && b_hh[l], GIC_ERR_NULL, "decode_beam: NULL weight of layer %d", l);
  return decode_beam(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, B, K, L, V, E, H, layers, eos_id,
                     length_penalty, c, ids, scores, lengths, trace, workspace, S(stream));
}

size_t gic_vocab_target_logp_workspace_floats(int M, int V) { return vocab_target_ws_floats(M, V); }
int gic_vocab_target_logp(int mode, const float* h, const float* W_out, const float* b_out, const int64_t* targets, int M, int V,
                          int H, float* logp, float* lse, int64_t* argmax, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(M >= 0 && V >= 1 && H >= 1, GIC_ERR_SHAPE, "vocab_target_logp: bad shape M=%d V=%d H=%d", M, V, H);
  if (M == 0) return GIC_OK;
  GIC_REQUIRE(h && W_out && b_out && targets && logp && workspace, GIC_ERR_NULL, "vocab_target_logp: NULL pointer");
  return vocab_target_scores(mode, h, W_out, b_out, targets, M, V, H, 1, nullptr, logp, lse, argmax, nullptr, nullptr,
                             workspace, S(stream));
}
static bool sample_args_ok(float temperature, int top_k, float top_p, int V) {
  return isfinite(temperature) && temperature > 0.f && top_p > 0.f && top_p <= 1.f && top_k >= 0 && top_k <= 16 &&
         top_k <= V && !(top_p < 1.f && top_k == 0);
}
size_t gic_vocab_sample_workspace_floats(int M, int V, int top_k) { return vocab_sample_ws_floats(M, V, top_k); }
int gic_vocab_sample(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int step,
                     float temperature, int top_k, float top_p, int64_t* tokens, float* logp, float* workspace,
                     gic_stream_t stream) {
  GIC_REQUIRE(M >= 0 && V >= 1 && H >= 1 && step >= 0, GIC_ERR_SHAPE, "vocab_sample: bad shape M=%d V=%d H=%d step=%d", M, V,
              H, step);
  GIC_REQUIRE(sample_args_ok(temperature, top_k, top_p, V), GIC_ERR_SHAPE,
              "vocab_sample: bad sampling arguments temperature=%g top_k=%d top_p=%g V=%d", temperature, top_k, top_p, V);
  if (M == 0) return GIC_OK;
  GIC_REQUIRE(h && W_out && b_out && tokens && logp && workspace, GIC_ERR_NULL, "vocab_sample: NULL pointer");
  return vocab_sample(mode, h, W_out, b_out, M, V, H, step, temperature, top_k, top_p, tokens, logp, nullptr, nullptr,
                      workspace, S(stream));
}
int gic_vocab_sample_masked(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int step,
                            float temperature, int top_k, float top_p, int64_t* tokens, float* logp, const uint32_t* ban,
                            float* workspace, gic_stream_t stream) {
  GIC_REQUIRE(M >= 0 && V >= 1 && H >= 1 && step >= 0, GIC_ERR_SHAPE, "vocab_sample_masked: bad shape M=%d V=%d H=%d step=%d",
              M, V, H, step);
  GIC_REQUIRE(sample_args_ok(temperature, top_k, top_p, V), GIC_ERR_SHAPE,
              "vocab_sample_masked: bad sampling arguments temperature=%g top_k=%d top_p=%g V=%d", temperature, top_k, top_p,
              V);
  if (M == 0) return GIC_OK;
  GIC_REQUIRE(h && W_out && b_out && tokens && logp && ban && workspace, GIC_ERR_NULL, "vocab_sample_masked: NULL pointer");
  return vocab_sample(mode, h, W_out, b_out, M, V, H, step, temperature, top_k, top_p, tokens, logp, nullptr, ban, workspace,
                      S(stream));
}
size_t gic_sample_captions_workspace_floats(int B, int n, int V, int E, int H, int layers, int top_k) {
  return SampleCaptionsWs(B * n, V, E, H, layers, top_k).total;
}
size_t gic_sample_captions_constrained_workspace_floats(int B, int n, int L, int V, int E, int H, int layers, int top_k,
                                                        const gic_decode_constraints_t* c) {
  return SampleCaptionsWs(B * n, V, E, H, layers, top_k, L, active_constraints(c)).total;
}
int gic_sample_captions(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                        const float* const* W_hh, const float* const* b_ih, const float* const* b_hh, const float* W_out,
                        const float* b_out, int B, int n, int L, int V, int E, int H, int layers, int64_t eos_id,
                        float temperature, int top_k, float top_p, int64_t* ids, float* caption_logp, int32_t* lengths,
                        float* workspace, gic_stream_t stream) {
  return gic_sample_captions_constrained(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, B, n, L, V, E, H, layers,
                                         eos_id, temperature, top_k, top_p, nullptr, ids, caption_logp, lengths, workspace,
                                         stream);
}
int gic_sample_captions_constrained(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                                    const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                                    const float* W_out, const float* b_out, int B, int n, int L, int V, int E, int H,
                                    int layers, int64_t eos_id, float temperature, int top_k, float top_p,
                                    const gic_decode_constraints_t* constraints, int64_t* ids, float* caption_logp,
                                    int32_t* lengths, float* workspace, gic_stream_t stream) {
  GIC_REQUIRE(B >= 0 && n >= 1 && L >= 1 && V >= 1 && E >= 1 && H >= 1 && layers >= 1 && layers <= 8 && eos_id >= 0 &&
                  eos_id < V, GIC_ERR_SHAPE, "sample_captions: bad shape B=%d n=%d L=%d V=%d E=%d H=%d layers=%d eos_id=%lld",
              B, n, L, V, E, H, layers, (long long)eos_id);
  GIC_REQUIRE(sample_args_ok(temperature, top_k, top_p, V), GIC_ERR_SHAPE,
              "sample_captions: bad sampling arguments temperature=%g top_k=%d top_p=%g V=%d", temperature, top_k, top_p, V);
  const gic_decode_constraints_t* c = active_constraints(constraints);
  GIC_TRY(constraints_check(c, L, V, top_k, "sample_captions"));
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(features && W_emb && W_ih && W_hh && b_ih && b_hh && W_out && b_out && ids && caption_logp && lengths &&
                  workspace, GIC_ERR_NULL, "sample_captions: NULL pointer");
  for (int l = 0; l < layers; ++l)
    GIC_REQUIRE(W_ih[l] && W_hh[l] && b_ih[l] && b_hh[l], GIC_ERR_NULL, "sample_captions: NULL weight of layer %d", l);
  return sample_captions(mode, features, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, B, n, L, V, E, H, layers, (int)eos_id,
                         temperature, top_k, top_p, c, ids, caption_logp, lengths, workspace, S(stream));
}

size_t gic_score_captions_workspace_floats(int B, int L, int V, int E, int H, int layers) {
  return ScoreWs(B, L, V, E, H, layers).total;
}
int gic_score_captions(int mode, const float* features, const int64_t* captions, const int32_t* lengths, const float* W_emb,
                       const float* const* W_ih, const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                       const float* W_out, const float* b_out, int B, int L, int V, int E, int H, int layers, float* logp,
                       float* caption_logp, uint8_t* correct, float* workspace, gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(B >= 0 && L >= 1 && V >= 1 && E >= 1 && H >= 1 && layers >= 1 && layers <= 8, GIC_ERR_SHAPE,
              "score_captions: bad shape B=%d L=%d V=%d E=%d H=%d layers=%d", B, L, V, E, H, layers);
  if (B == 0) return GIC_OK;
  GIC_REQUIRE(features && captions && W_emb && W_ih && W_hh && b_ih && b_hh && W_out && b_out && logp && caption_logp &&
                  workspace, GIC_ERR_NULL, "score_captions: NULL pointer");
  for (int l = 0; l < layers; ++l)
    GIC_REQUIRE(W_ih[l] && W_hh[l] && b_ih[l] && b_hh[l], GIC_ERR_NULL, "score_captions: NULL weight of layer %d", l);
  return score_captions(mode, features, captions, lengths, W_emb, W_ih, W_hh, b_ih, b_hh, W_out, b_out, B, L, V, E, H, layers,
                        logp, caption_logp, correct, workspace, S(stream));
}

size_t gic_disc_saved_floats(int N, int L, int De, int R, int F) { return DiscSaved(N, L, De, R, F).total; }
size_t gic_disc_fwd_workspace_floats(int F) { return DiscFwdWs(F).total; }
size_t gic_disc_bwd_workspace_floats(int N, int L, int De, int R, int F) { return DiscBwdWs(N, L, De, R, F).total; }

int gic_disc_fwd(int mode, const float* inp_soft, const int64_t* ids, int N, int L, int V, int De, int R,
                 int n_groups, const int* filter_sizes, const int* num_filters, const float* W_e,
                 const float* const* conv_w, const float* const* conv_b, const float* W_h, const float* b_h,
                 const float* W_f, const float* b_f, int Hd, const float* W_o, const float* b_o, int n_heads,
                 const uint8_t* const* keep, float drop_p, float* const* logits, float* saved, float* workspace,
                 gic_stream_t stream) {
  GIC_TRY(require_device());
  return disc_fwd_entry(mode, inp_soft, ids, N, L, V, De, R, n_groups, filter_sizes, num_filters, W_e, conv_w, conv_b,
                        W_h, b_h, W_f, b_f, Hd, W_o, b_o, n_heads, keep, drop_p, logits, saved, workspace, S(stream));
}

int gic_disc_bwd(int mode, const float* dlogits, const uint8_t* keep, float drop_p, const float* inp_soft,
                 const int64_t* ids, int N, int L, int V, int De, int R, int n_groups, const int* filter_sizes,
                 const int* num_filters, const float* W_e, const float* const* conv_w, const float* const* conv_b,
                 const float* W_h, const float* W_f, const float* b_f, int Hd, const float* W_o, const float* b_o,
                 const float* saved, float* workspace, float* dW_e, float* const* dconv_w, float* const* dconv_b,
                 float* dW_h, float* db_h, float* dW_f, float* db_f, float* dW_o, float* db_o, float* dinp,
                 int want_param, int accumulate, gic_stream_t stream) {
  GIC_TRY(require_device());
  return disc_bwd_entry(mode, dlogits, keep, drop_p, inp_soft, ids, N, L, V, De, R, n_groups, filter_sizes,
                        num_filters, W_e, conv_w, conv_b, W_h, W_f, b_f, Hd, W_o, b_o, saved, workspace, dW_e, dconv_w,
                        dconv_b, dW_h, db_h, dW_f, db_f, dW_o, db_o, dinp, want_param, accumulate, S(stream));
}

int gic_gan_loss_fwd_bwd(int loss_type, const float* d_out_real, const float* d_out_fake, const float* g_out, int n,
                         float* losses, float* dd_real, float* dd_fake, float* dg_out, gic_stream_t stream) {
  GIC_TRY(require_device());
  return gan_loss(loss_type, d_out_real, d_out_fake, g_out, n, losses, dd_real, dd_fake, dg_out, S(stream));
}

int gic_grad_sqnorm(const float* g, size_t n, float* sqnorm, gic_stream_t stream) {
  GIC_TRY(require_device());
  return grad_sqnorm(g, n, sqnorm, S(stream));
}

int gic_clip_adam(float* p, const float* g, float* m, float* v, size_t n, const float* sqnorm, float max_norm,
                  float grad_scale, int step, float lr, float beta1, float beta2, float eps, gic_stream_t stream) {
  GIC_TRY(require_device());
  return clip_adam(p, g, m, v, n, sqnorm, max_norm, grad_scale, step, lr, beta1, beta2, eps, nullptr, S(stream));
}

int gic_clip_adam_dyn(float* p, const float* g, float* m, float* v, size_t n, const float* sqnorm, float max_norm,
                      float grad_scale, const float* bias_corr_dev, float beta1, float beta2, float eps,
                      gic_stream_t stream) {
  GIC_TRY(require_device());
  GIC_REQUIRE(bias_corr_dev, GIC_ERR_NULL, "clip_adam_dyn: NULL bias_corr_dev");
  return clip_adam(p, g, m, v, n, sqnorm, max_norm, grad_scale, 0, 0.f, beta1, beta2, eps, bias_corr_dev, S(stream));
}

void gic_set_temperature_device(const float* t_dev) { set_temperature_device(t_dev); }

size_t gic_disc_prepared_floats(int F) { return DiscFwdWs(F).total; }
int gic_disc_prepare(int mode, const float* W_h, const float* W_f, const float* b_f, int Hd, const float* W_o,
                     const float* b_o, int F, float* prepared, gic_stream_t stream) {
  GIC_TRY(require_device());
  return disc_prepare(mode, W_h, W_f, b_f, Hd, W_o, b_o, F, prepared, S(stream));
}
void gic_disc_set_prepared(const float* prepared) { disc_set_prepared(prepared); }
int gic_pack_captions(const int32_t* tokens, const int32_t* offsets, int B, int max_caption_len, int64_t* captions,
                      int32_t* lengths, gic_stream_t stream) {
  GIC_TRY(require_device());
  return pack_captions(tokens, offsets, B, max_caption_len, captions, lengths, S(stream));
}
void gic_set_rng(unsigned long long seed, unsigned long long offset, const unsigned long long* state_dev) {
  set_rng(seed, offset, state_dev);
}
int gic_philox_uniform(unsigned int tag, size_t n, float* out, gic_stream_t stream) {
  GIC_TRY(require_device());
  return philox_uniform(tag, 0ull, n, out, S(stream));
}
int gic_philox_keep_mask(unsigned int tag, size_t n, float p, uint8_t* out, gic_stream_t stream) {
  GIC_TRY(require_device());
  return philox_keep_mask(tag, n, p, out, S(stream));
}
void gic_set_vocab_grads_event(void* cuda_event) { ctx().vocab_grads_event = reinterpret_cast<cudaEvent_t>(cuda_event); }
void gic_set_embed_grads_event(void* cuda_event) { ctx().embed_grads_event = reinterpret_cast<cudaEvent_t>(cuda_event); }

gic_ctx_t* gic_ctx_create(void) { return reinterpret_cast<gic_ctx_t*>(new (std::nothrow) Ctx()); }
void gic_ctx_destroy(gic_ctx_t* c) {
  Ctx* p = reinterpret_cast<Ctx*>(c);
  if (p && &ctx() == p) ctx_set_current(nullptr);
  delete p;
}
gic_ctx_t* gic_ctx_set_current(gic_ctx_t* c) { return reinterpret_cast<gic_ctx_t*>(ctx_set_current(reinterpret_cast<Ctx*>(c))); }
void gic_trap_info(unsigned long long out[4]) {
  const unsigned long long* p = trap_slot();
  for (int i = 0; i < 4; ++i) out[i] = p ? p[i] : 0ull;
}
int gic_trap_notes(unsigned long long* out, int max_records) {
  const unsigned long long* p = trap_slot();
  int n = 0;
  for (int r = 1; p && r < 32 && n < max_records; ++r)
    if (p[4 * r] != 0ull) { for (int i = 0; i < 4; ++i) out[4 * n + i] = p[4 * r + i]; ++n; }
  return n;
}
int gic_ctx_set_option(const char* name, int value) {
  GIC_REQUIRE(name && *name && strlen(name) < sizeof(Ctx::Opt().name), GIC_ERR_SHAPE, "gic_ctx_set_option: bad option name");
  option_set(name, value);
  GIC_REQUIRE(option_is_set(name), GIC_ERR_UNSUPPORTED, "gic_ctx_set_option: option table full");
  return GIC_OK;
}
void gic_ctx_clear_option(const char* name) { if (name) option_clear(name); }
int gic_ctx_get_option(const char* name, int dflt) { return name ? option(name, dflt) : dflt; }

}  // extern "C"
