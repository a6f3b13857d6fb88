/*
 * gic_b200.h -- C ABI of libgic_b200.so: the B200 (sm_100a) adversarial-captioning hot path.
 *
 * Drop-in boundary for kawshik8/GAN-Image-Captioning.  The reference is pure Python/PyTorch
 * and has no FFI of its own; every entry point below replaces the body of one reference
 * function (cited per function, paths relative to the reference checkout) and is what a
 * ctypes binding inside that function would call (see INTEGRATION.md for the stubs).
 *
 * Conventions
 *  - plain pointers and sizes only; all tensors are dense row-major fp32 unless stated;
 *    token ids are int64 (torch.long); dropout keep-masks are uint8 (0 = dropped, 1 = kept).
 *  - every pointer is a DEVICE pointer owned by the caller (PyTorch's caching allocator);
 *    the library never allocates, frees or synchronises; outputs, "saved" (for backward) and
 *    "workspace" buffers are caller-allocated with the *_floats() sizes below.
 *  - kernels are enqueued on `stream` (a cudaStream_t); no hidden host syncs.
 *  - return value: 0 = ok, non-zero = error (gic_last_error() gives the message); the Python
 *    shim raises RuntimeError / NotImplementedError like the reference's own error paths
 *    (src/utils.py:51).
 *  - all randomness is an input: Gumbel uniforms u[L,B,V], dropout keep-masks.
 *  - there is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef GIC_B200_H_
#define GIC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gic_stream_t; /* cudaStream_t */

/* status codes */
#define GIC_OK 0
#define GIC_ERR_SHAPE 1
#define GIC_ERR_NULL 2
#define GIC_ERR_CUDA 3
#define GIC_ERR_WORKSPACE 4
#define GIC_ERR_ARCH 5
#define GIC_ERR_UNSUPPORTED 6

/* precision of the dense contractions (see DESIGN.md "GEMM modes") */
#define GIC_GEMM_FP32 0   /* CUDA-core FFMA, exact fp32                                   */
#define GIC_GEMM_TF32 1   /* tcgen05 kind::tf32, one pass, fp32 accumulate in TMEM         */
/* (2 is unassigned: a 3-pass TF32 split was planned and never built; the exact mode is GIC_GEMM_FP32) */
#define GIC_GEMM_BF16 3   /* as TF32, with the discriminator's [N*R,F]x[F,F] contractions (highway forward, dx, dW_h) on
                             bf16 operands (tcgen05 kind::f16, fp32 accumulate): "bf16 GEMM inputs, stated separately" */

/* adversarial loss types, src/utils.py:14-50 */
#define GIC_LOSS_STANDARD 0
#define GIC_LOSS_JS 1
#define GIC_LOSS_KL 2
#define GIC_LOSS_HINGE 3
#define GIC_LOSS_TV 4
#define GIC_LOSS_RSGAN 5

int gic_version(void);
const char* gic_last_error(void);
/* 0 if the current device is an sm_100 part, GIC_ERR_ARCH / GIC_ERR_CUDA otherwise. */
int gic_check_device(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches). */
unsigned long long gic_launch_count(void);
/* launches of ONE kernel so far, by its __global__ name without template arguments ("vocab_sample_kernel",
 * "gemm_pair_kernel", "bptt_persistent_kernel", ...; NULL = all).  The tests use it to assert that a fused kernel ran
 * rather than the fallback it replaces.  gic_kernel_names writes the names seen so far, newline separated, into buf
 * (cap bytes) and returns their number. */
unsigned long long gic_kernel_launches(const char* name);
int gic_kernel_names(char* buf, int cap);
/* Optional per-kernel-class device timing for bench.py's roofline: between gic_prof_begin() and gic_prof_end()
 * every launch of a profiled class is bracketed by CUDA events on its own stream.  gic_prof_end (call after the
 * stream is synchronised) fills ms[k], work[k] (algorithmic flops for k=0 GEMM, bytes otherwise) and calls[k] for
 * the GIC_PROF_KINDS classes: 0 GEMM (all other contractions), 1 sample step, 2 conv+pool fwd, 3 softmax bwd, 4 clip+Adam,
 * 5 head fwd, 6 the discriminator's [N*R, F] x [F, F] contractions (highway forward, dx, dW_h: the FLOP-dominant kernel),
 * 7 decode-step contractions (fused LSTM step, vocab projection), 8 the fused vocab projection + Gumbel-softmax +
 * sample kernel (work = its HBM bytes, 8 B V: read u, write probs). */
#define GIC_PROF_KINDS 9
void gic_prof_begin(void);
void gic_prof_end(double* ms, double* work, unsigned long long* calls);

/* ---- dense contraction (nn.Linear / its autograd; src/generator.py:64,68, src/discriminator.py:40,53) ----
 * C[M,N] = alpha * op(A) * op(B) + beta * C + bias[N];  transA: A stored [K,M]; transB: B stored [N,K]. */
int gic_gemm(int mode, int transA, int transB, int M, int N, int K, float alpha, const float* A, int lda,
             const float* B, int ldb, float beta, float* C, int ldc, const float* bias, gic_stream_t stream);

/* same contraction with bf16 operands (A, B: bf16, leading dimensions in elements, multiples of 8; 16-byte aligned),
 * fp32 accumulation in TMEM and fp32 C. */
int gic_gemm_bf16(int transA, int transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B,
                  int ldb, float beta, float* C, int ldc, const float* bias, gic_stream_t stream);

/* ---- Encoder.linear + Encoder.bn, train-mode batch statistics (src/generator.py:15-16,23-24) ---- */
int gic_encoder_fwd(int mode, const float* pooled /*[B,Fin]*/, int B, int Fin, int E, const float* W /*[E,Fin]*/,
                    const float* b, const float* gamma, const float* beta, float eps,
                    float* lin_out /*[B,E] saved*/, float* save_mean /*[E]*/, float* save_rstd /*[E]*/,
                    float* features /*[B,E]*/, gic_stream_t stream);
int gic_encoder_bwd(int mode, const float* dfeatures /*[B,E]*/, const float* pooled, const float* lin_out,
                    const float* save_mean, const float* save_rstd, const float* W, const float* gamma, int B,
                    int Fin, int E, float* dlin_ws /*[B,E] workspace*/, float* dW, float* db, float* dgamma,
                    float* dbeta, int accumulate, gic_stream_t stream);

/* BatchNorm1d bookkeeping of a training-mode forward (nn.BatchNorm1d(E, momentum=0.01), src/generator.py:16): from the
 * save_mean / save_rstd gic_encoder_fwd (or gic_encoder_fwd_apply) left behind, running_mean and running_var move by
 * `momentum` towards the batch mean and the UNBIASED batch variance over `count` rows; *num_batches_tracked (int64, may
 * be NULL) is incremented.  Checkpoints then carry the statistics the reference's would. */
int gic_encoder_bn_running_update(const float* save_mean, const float* save_rstd, int E, float eps, float count,
                                  float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                                  gic_stream_t stream);
/* Encoder.linear + Encoder.bn in eval mode (gen.eval() in the validation loops, src/training.py:213): normalises with
 * the running statistics.  Forward only. */
int gic_encoder_fwd_eval(int mode, const float* pooled, int B, int Fin, int E, const float* W, const float* b,
                         const float* gamma, const float* beta, float eps, const float* running_mean,
                         const float* running_var, float* lin_out /*[B,E] workspace*/, float* features /*[B,E]*/,
                         gic_stream_t stream);

/* ---- one fused sampling step (K4): Gumbel + temperature + vocab softmax + first-max + embedding gather.
 * Decoder.add_gumbel + F.softmax + pred.max(1) + self.embed (src/generator.py:68-76, 84-96).
 * pretrain != 0: out row = raw logits, choice = argmax softmax(logits) (src/generator.py:63-66); u unused. */
int gic_sample_step(int pretrain, const float* logits /*[B,V]*/, const float* u /*[B,V]*/, float temperature,
                    int B, int V, int L, int t, float* out /*[B,L,V], row (b,t) written*/,
                    int64_t* ids /*[B,L], (b,t) written*/, const int64_t* forced_ids /*[B,L] or NULL*/,
                    const float* embed /*[V,E]*/, int E, float* x_next /*[B,E] or NULL*/, gic_stream_t stream);

/* ---- Decoder.sample (src/generator.py:55-81) ----
 * features[B,E] is the step-0 LSTM input; per-layer weight pointers follow nn.LSTM's state_dict
 * (weight_ih_l{k}[4H,In], weight_hh_l{k}[4H,H], bias_ih_l{k}[4H], bias_hh_l{k}[4H], gate order i,f,g,o).
 * u[L,B,V]: uniforms in [0,1) (ignored when pretrain).  forced_ids: teacher forcing for parity runs
 * (token fed back at step t is forced_ids[b,t]; ids still receives this run's own choices).
 * out[B,L,V]: soft captions (or logits when pretrain); ids[B,L]. */
size_t gic_decode_saved_floats(int B, int L, int E, int H, int layers);
size_t gic_decode_fwd_workspace_floats(int B, int V, int H);
int gic_decode_sample_fwd(int mode, const float* features, const float* W_emb /*[V,E]*/,
                          const float* const* W_ih, const float* const* W_hh, const float* const* b_ih,
                          const float* const* b_hh, const float* W_out /*[V,H]*/, const float* b_out /*[V]*/,
                          const float* u, float temperature, int pretrain, const int64_t* forced_ids, int B, int L,
                          int V, int E, int H, int layers, float* out, int64_t* ids, float* saved,
                          float* workspace, gic_stream_t stream);

/* Backward of Decoder.sample: given dout[B,L,V] (gradient w.r.t. the soft captions, or w.r.t. the logits when
 * pretrain) produce the gradients of every decoder parameter and of `features` (SURVEY.md section 3.4).
 * fed_ids[B,L]: the tokens that were fed back (ids, or forced_ids when teacher forcing was used).
 * accumulate != 0 adds into the gradient buffers, else overwrites.  dfeatures may be NULL. */
size_t gic_decode_bwd_workspace_floats(int B, int L, int V, int E, int H, int layers);
int gic_decode_sample_bwd(int mode, const float* dout, const float* out, const int64_t* fed_ids,
                          const float* W_emb, const float* const* W_ih, const float* const* W_hh,
                          const float* W_out, float temperature, int pretrain, int B, int L, int V, int E, int H,
                          int layers, const float* saved, float* workspace, float* dW_emb, float* const* dW_ih,
                          float* const* dW_hh, float* const* db_ih, float* const* db_hh, float* dW_out,
                          float* db_out, float* dfeatures, int accumulate, gic_stream_t stream);

/* Same backward with the incoming gradient in factored form (the fused adversarial step): instead of the dense
 * dout[B,L,V] = d g_loss / d probs it takes demb[B*L,De] = d g_loss / d (probs W_e^T) -- what gic_disc_bwd leaves at
 * workspace + gic_disc_bwd_demb_offset_floats() when called with dinp = NULL -- together with emb[B*L,De] (the first
 * B*L*De floats of the discriminator's saved blob) and W_e[De,V].  dz = T p (demb W_e - <demb, emb>) is produced by one
 * tensor-core kernel with the softmax backward as its epilogue; the dense d(probs) is never written or read.
 * Same autograd semantics as src/generator.py:69 + src/discriminator.py:40. */
int gic_decode_sample_bwd_factored(int mode, const float* demb, const float* emb, const float* W_e, int De,
                                   const float* out, const int64_t* fed_ids, const float* W_emb,
                                   const float* const* W_ih, const float* const* W_hh, const float* W_out,
                                   float temperature, int B, int L, int V, int E, int H, int layers, const float* saved,
                                   float* workspace, float* dW_emb, float* const* dW_ih, float* const* dW_hh,
                                   float* const* db_ih, float* const* db_hh, float* dW_out, float* db_out,
                                   float* dfeatures, int accumulate, gic_stream_t stream);

/* ---- Discriminator.forward (src/discriminator.py:34-62) ----
 * Exactly one of inp_soft[N,L,V] (soft / dense one-hot captions) and ids[N,L] (hard tokens: Linear of a one-hot is
 * a column pick, replacing F.one_hot at src/training.py:158) is non-NULL.  De = disc_embed_dim, R = disc_num_rep,
 * emb_dim_single = De/R.  conv_w[g] is convs.g.weight [n_g,1,f_g,De/R], conv_b[g] its bias.  The trunk
 * (embedding, conv+ReLU+max-pool, highway) is evaluated once and n_heads (<= 4) dropout masks are applied to it:
 * logits[h][N*R] = head(dropout_h(trunk)), keep[h] == NULL meaning eval mode for that head.  The reference's three
 * calls per step (real, fake, gen; src/training.py:162-164) are 2 trunks: real (1 head) and fake (2 heads). */
size_t gic_disc_saved_floats(int N, int L, int De, int R, int F);
size_t gic_disc_fwd_workspace_floats(int F);
int gic_disc_fwd(int mode, const float* inp_soft, const int64_t* ids, int N, int L, int V, int De, int R,
                 int n_groups, const int* filter_sizes, const int* num_filters, const float* W_e /*[De,V]*/,
                 const float* const* conv_w, const float* const* conv_b, const float* W_h /*[F,F]*/,
                 const float* b_h, const float* W_f /*[Hd,F]*/, const float* b_f, int Hd, const float* W_o /*[1,Hd]*/,
                 const float* b_o, int n_heads, const uint8_t* const* keep, float drop_p, float* const* logits,
                 float* saved, float* workspace, gic_stream_t stream);

/* Backward of one head of Discriminator.forward.  dlogits[N*R] is the loss seed for that head, keep its mask
 * (NULL = eval).  want_param: produce parameter gradients (accumulate != 0 adds).  dinp != NULL: also produce the
 * gradient w.r.t. the soft input [N,L,V] (the generator's path, SURVEY.md section 3.4). */
size_t gic_disc_bwd_workspace_floats(int N, int L, int De, int R, int F);
/* offset (floats) of demb[N,L,De] = d loss / d embedding output inside the backward workspace after gic_disc_bwd */
size_t gic_disc_bwd_demb_offset_floats(int N, int L, int De, int R, int F);
int gic_disc_bwd(int mode, const float* dlogits, const uint8_t* keep, float drop_p, const float* inp_soft,
                 const int64_t* ids, int N, int L, int V, int De, int R, int n_groups, const int* filter_sizes,
                 const int* num_filters, const float* W_e, const float* const* conv_w, const float* const* conv_b,
                 const float* W_h, const float* W_f, const float* b_f, int Hd, const float* W_o, const float* b_o,
                 const float* saved, float* workspace, float* dW_e, float* const* dconv_w, float* const* dconv_b,
                 float* dW_h, float* db_h, float* dW_f, float* db_f, float* dW_o, float* db_o, float* dinp,
                 int want_param, int accumulate, gic_stream_t stream);

/* ---- get_losses (src/utils.py:10-53) with the backward seeds ----
 * losses[0] = g_loss, losses[1] = d_loss (the reference returns g first).  dd_real/dd_fake = d d_loss / d logits,
 * dg_out = d g_loss / d g_out; any of the three may be NULL. */
int gic_gan_loss_fwd_bwd(int loss_type, const float* d_out_real, const float* d_out_fake, const float* g_out, int n,
                         float* losses, float* dd_real, float* dd_fake, float* dg_out, gic_stream_t stream);

/* ---- GANInstructor.optimize (src/training.py:194-199): clip_grad_norm_ + Adam over a flat buffer ----
 * gic_grad_sqnorm accumulates sum(g^2) into *sqnorm (caller zeroes it; several buffers may share it).
 * gic_clip_adam reads *sqnorm on the device (no host sync): coef = min(1, max_norm/(sqrt(sqnorm)*grad_scale+1e-6)),
 * then torch.optim.Adam's update (weight_decay 0).  grad_scale = 1/world_size after a summed all-reduce. */
int gic_grad_sqnorm(const float* g, size_t n, float* sqnorm, gic_stream_t stream);
int gic_clip_adam(float* p, const float* g, float* m, float* v, size_t n, const float* sqnorm, float max_norm,
                  float grad_scale, int step, float lr, float beta1, float beta2, float eps, gic_stream_t stream);

/* ---- generator pre-training loss (src/training.py:81-83): nn.CrossEntropyLoss() over ALL B*L positions, PAD
 * included (no ignore_index, SURVEY.md Q8), of the raw logits Decoder.sample(pretrain=True) returns, with its
 * backward seed dlogits = (softmax(logits) - onehot(target)) / (B L).  Feed dlogits to gic_decode_sample_bwd(pretrain=1). */
int gic_ce_loss_fwd_bwd(const float* logits /*[B,L,V]*/, const int64_t* targets /*[B,L]*/, int B, int L, int V,
                        float* loss /*[1]*/, float* dlogits /*[B,L,V] or NULL*/, gic_stream_t stream);

/* ==== EXTENSIONS beyond the reference (north-star stages 2-4; SURVEY.md section 8a rows B2, B3).  The reference has no
 * rollouts, no inverse-CDF sampler and no policy-gradient loss (SURVEY.md section 0): these entry points are defined by
 * this library and its oracle (oracle/ref_ext.py), "parity unpinned by reference". ====
 *
 * gic_decode_sample_cdf_fwd: Decoder.sample's loop (src/generator.py:55-81) with the token drawn by inverse CDF from
 *   softmax(logits) and ONE uniform per row and step, u[L,B]; token = first index whose cumulative probability exceeds
 *   u.  logits_out[B,L,V] (raw logits, for the backward via gic_decode_sample_bwd(pretrain = 1)) and logp[B,L]
 *   (log pi(token)) may be NULL.  saved / workspace sizes as for gic_decode_sample_fwd.
 * gic_decode_rollouts: for every prefix length t = 1..L-1 of main_ids[B,L], n_roll continuations sampled with the same
 *   policy (single-layer decoder).  saved = the blob gic_decode_sample_cdf_fwd filled for those captions.
 *   u_roll[L, Mmax] with Mmax = (L-1)*B*n_roll: row m at step s reads u_roll[s*Mmax + m].  roll_ids[Mmax, L]: row
 *   (t-1)*B*n + b*n + j = j-th completion of prefix t of caption b (positions < t copied from main_ids).
 * gic_rollout_rewards: Q[b,t-1] = mean over rollouts j and representations r of sigmoid(D logit) for prefix length
 *   t < L; Q[b,L-1] = the sampled caption's own mean sigmoid(D logit).  roll_logits[Mmax*R], main_logits[B*R] come
 *   from gic_disc_fwd(ids = ...) in eval mode.
 * gic_pg_loss_fwd_bwd: loss[0] = -(1/(B L)) sum log pi(y_bt) (Q_bt - base_t), base_t = mean_b Q_bt (baseline_mode 1) or
 *   0 (mode 0); dlogits[B,L,V] = d loss / d logits (may be NULL); logp[B,L] optional. */
/* one fused vocab-softmax + inverse-CDF sample step (the kernel gic_decode_sample_cdf_fwd / gic_decode_rollouts run
 * per position): u[B] one uniform per row; out row (b,t) of [B,L,V] = raw logits (NULL: nothing of size V is written);
 * ids[b,t] = token; logp[b,t] = log softmax(logits)[token]; x_next[B,E] = embed[fed token] (NULL to skip). */
int gic_sample_cdf_step(const float* logits, const float* u, int B, int V, int L, int t, float* out, int64_t* ids,
                        float* logp, const int64_t* forced_ids, const float* embed, int E, float* x_next,
                        gic_stream_t stream);
int gic_decode_sample_cdf_fwd(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                              const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                              const float* W_out, const float* b_out, const float* u, const int64_t* forced_ids, int B,
                              int L, int V, int E, int H, int layers, float* logits_out, int64_t* ids, float* logp,
                              float* saved, float* workspace, gic_stream_t stream);
size_t gic_decode_rollouts_workspace_floats(int B, int L, int V, int E, int H, int n_roll);
int gic_decode_rollouts(int mode, const float* saved, const int64_t* main_ids, const float* W_emb, const float* W_ih,
                        const float* W_hh, const float* b_ih, const float* b_hh, const float* W_out,
                        const float* b_out, const float* u_roll, int B, int L, int V, int E, int H, int n_roll,
                        int64_t* roll_ids, float* workspace, gic_stream_t stream);
int gic_rollout_rewards(const float* roll_logits, const float* main_logits, int B, int L, int n_roll, int R, float* Q,
                        gic_stream_t stream);
int gic_pg_loss_fwd_bwd(const float* logits, const int64_t* ids, const float* Q, int baseline_mode, int B, int L, int V,
                        float* loss, float* dlogits, float* logp, gic_stream_t stream);

/* ---- caption generation by beam search (EXTENSION, parity unpinned by reference: the reference has no beam search;
 * oracle/ref_beam.py beam_search defines it).
 * gic_vocab_topk: per row of h[M,H]: lse[m] = logsumexp(h W_out^T + b_out), the K largest log-probabilities logp[M,K]
 *   (descending, ties -> lower token) and their tokens[M,K]; nothing of size V is written in the tensor-core modes.
 *   workspace: gic_vocab_topk_workspace_floats(M, V, K); lse may be NULL.  1 <= K <= 16, K <= V.
 * gic_decode_beam: Decoder.sample's LSTM (any number of layers; step 0's input is features[B,E], h = c = 0) with K beams per
 *   image.  Every step each live beam k offers (k, w) at score_k + log_softmax(h W_out^T + b_out)[w]; a beam that has emitted
 *   eos_id is frozen and offers only (k, PAD = 0) at its own score.  The image keeps its K best candidates (higher score, then
 *   lower parent beam, then lower token); beam 0 starts at 0, beams 1..K-1 at -inf.  Always L steps, no host sync (the call
 *   can be captured into a CUDA graph).  Output, per image, the K beams ordered by score / length^length_penalty (ties ->
 *   lower beam slot): ids[B,K,L] (PAD after EOS), scores[B,K] (raw sums of log-probabilities), lengths[B,K] (tokens up to and
 *   including EOS, L when none).  trace[L,B,K,2] (may be NULL): for step t and slot k the parent slot and token chosen.
 *   K = 1 is greedy decoding.  GIC_ERR_SHAPE: K < 1, K > 16, K > V, L < 1, eos_id outside [0, V), layers outside 1..8. */
size_t gic_vocab_topk_workspace_floats(int M, int V, int K);
int gic_vocab_topk(int mode, const float* h, const float* W_out, const float* b_out, int M, int V, int H, int K,
                   float* logp, int64_t* tokens, float* lse, float* workspace, gic_stream_t stream);
size_t gic_decode_beam_workspace_floats(int B, int K, int L, int V, int E, int H, int layers);
int gic_decode_beam(int mode, const float* features, const float* W_emb, const float* const* W_ih,
                    const float* const* W_hh, const float* const* b_ih, const float* const* b_hh,
                    const float* W_out, const float* b_out, int B, int K, int L, int V, int E, int H, int layers,
                    int64_t eos_id, float length_penalty, int64_t* ids /*[B,K,L]*/, float* scores /*[B,K]*/,
                    int32_t* lengths /*[B,K]*/, int32_t* trace /*[L,B,K,2] (parent, token) or NULL*/,
                    float* workspace, gic_stream_t stream);

/* ---- B1 (EXTENSION, parity unpinned by reference): additive attention over the CNN feature grid in the decode step.
 * The reference feeds one pooled vector at step 0 (src/generator.py:19-25,58) and has no attention.  Definition:
 *   once per image: Ak = grid W_k^T [B,P,Da], Av = grid W_v^T [B,P,E];  every step: q = h_{t-1} W_q^T,
 *   s_l = w_e . tanh(Ak_l + q), alpha = softmax_l(s), LSTM input x'_t = x_t + sum_l alpha_l Av_l.
 * gic_attn_t carries the grid, the four parameters, a saved blob (gic_attn_saved_floats) filled by the forward and,
 * for the backward, a workspace (gic_attn_bwd_workspace_floats) and the four gradient outputs (overwritten).
 * The *_attn entry points take the same arguments as gic_decode_sample_fwd / _bwd (dout, or dout = NULL and the
 * factored demb / emb / W_e / De of gic_decode_sample_bwd_factored). */
typedef struct gic_attn_t {
  const float* grid;      /* [B, P, Cf] CNN feature grid */
  int P, Cf, Da;          /* locations, channels, attention width */
  const float* W_k;       /* [Da, Cf] */
  const float* W_v;       /* [E, Cf]  */
  const float* W_q;       /* [Da, H]  */
  const float* w_e;       /* [Da]     */
  float* saved;           /* gic_attn_saved_floats(B, L, P, Da, E) */
  float* ws;              /* backward only: gic_attn_bwd_workspace_floats(B, L, P, Da, E) */
  float* dW_k;            /* backward only */
  float* dW_v;
  float* dW_q;
  float* dw_e;
} gic_attn_t;
size_t gic_attn_saved_floats(int B, int L, int P, int Da, int E);
size_t gic_attn_bwd_workspace_floats(int B, int L, int P, int Da, int E);
int gic_decode_sample_fwd_attn(const gic_attn_t* attn, int mode, const float* features, const float* W_emb,
                               const float* const* W_ih, const float* const* W_hh, const float* const* b_ih,
                               const float* const* b_hh, const float* W_out, const float* b_out, const float* u,
                               float temperature, int pretrain, const int64_t* forced_ids, int B, int L, int V, int E,
                               int H, int layers, float* out, int64_t* ids, float* saved, float* workspace,
                               gic_stream_t stream);
int gic_decode_sample_bwd_attn(const gic_attn_t* attn, int mode, const float* dout, const float* demb, const float* emb,
                               const float* W_e, int De, const float* out, const int64_t* fed_ids, const float* W_emb,
                               const float* const* W_ih, const float* const* W_hh, const float* W_out,
                               float temperature, int pretrain, int B, int L, int V, int E, int H, int layers,
                               const float* saved, float* workspace, float* dW_emb, float* const* dW_ih,
                               float* const* dW_hh, float* const* db_ih, float* const* db_hh, float* dW_out,
                               float* db_out, float* dfeatures, gic_stream_t stream);

/* ---- contexts: the state behind the four setters below ----
 * gic_set_temperature_device, gic_disc_set_prepared, gic_set_rng and gic_set_vocab_grads_event configure the calls that
 * FOLLOW them.  That state is not process-global: it lives in a context, and every host thread has a current context --
 * a private thread-local default until gic_ctx_set_current installs one the caller created.  Two training loops in one
 * process (or two threads) therefore cannot overwrite each other's temperature pointer, prepared weights, generator state or
 * event: give each its own context and make it current around its calls (the Python mirror's GANInstructor does).
 *   gic_ctx_create        a fresh context (all settings cleared); NULL when out of memory
 *   gic_ctx_set_current   install ctx as the calling thread's current context (NULL = back to the thread's default);
 *                         returns the previous one (NULL if that was the default)
 *   gic_ctx_destroy       free it (it stops being current first) */
typedef struct gic_ctx gic_ctx_t;
gic_ctx_t* gic_ctx_create(void);
gic_ctx_t* gic_ctx_set_current(gic_ctx_t* ctx);
void gic_ctx_destroy(gic_ctx_t* ctx);
/* A/B and tuning switches of the CURRENT context (which kernel variant a launch path takes: GIC_DECODE_STEP, GIC_FUSED_SAMPLE,
 * GIC_GEMM_2CTA, GIC_CONV_MMA, GIC_BPTT_PERSISTENT, GIC_BPTT_FUSED, GIC_FUSED_DZ_BF16, GIC_LSTM_SPLITK, GIC_PDL, ...; the
 * full table is in DESIGN.md).  They are integers held by the context; a switch nobody set is looked up in the process
 * environment under the same name ONCE per context -- the first time a launch path asks -- and remembered, so no launch
 * path calls getenv twice and a running job cannot be re-routed by a later setenv.
 *   gic_ctx_set_option    set name = value (GIC_ERR_SHAPE: empty or too long a name; GIC_ERR_UNSUPPORTED: table full)
 *   gic_ctx_clear_option  forget it: the next lookup consults the environment again, then the built-in default
 *   gic_ctx_get_option    the value a launch path would see (dflt when neither set nor in the environment) */
int gic_ctx_set_option(const char* name, int value);
/* The device-side waits of the library (mbarriers, the decode step's flags, the BPTT grid barrier) are bounded: a wait that
 * lasts seconds traps instead of hanging the GPU, and the CUDA context is lost ("unspecified launch failure").  Before it
 * traps the site writes who it was to host-mapped memory, which survives: out[0] = site (0: no trap happened; 1 mbarrier,
 * 2 token wait, 3 recurrent tiles, 4 row statistics, 5 recurrent flag, 6 BPTT grid barrier), out[1] = site-specific word,
 * out[2] = blockIdx.x << 32 | threadIdx.x, out[3] = %globaltimer. */
void gic_trap_info(unsigned long long out[4]);
/* Notes left by waits that had lasted 2 s when the trap came (one per warp of the stuck kernel: site, word, block/thread, -):
 * up to max_records records of 4 words; returns how many. */
int gic_trap_notes(unsigned long long* out, int max_records);
void gic_ctx_clear_option(const char* name);
int gic_ctx_get_option(const char* name, int dflt);

/* ---- CUDA-graph replay support ----
 * By-value scalars are frozen when a launch is captured into a CUDA graph, but the reference changes two of them every
 * batch: the temperature (update_temperature, src/training.py:183,190-191) and Adam's bias corrections (step count).
 * gic_set_temperature_device(t_dev): while t_dev is non-NULL every entry point that takes `temperature` reads it from
 *   *t_dev when its kernels run and ignores the by-value argument (current context; pass NULL to switch back).
 * gic_clip_adam_dyn: gic_clip_adam with the step-dependent factors read from device memory:
 *   bias_corr_dev[0] = lr / (1 - beta1^t), bias_corr_dev[1] = 1 / sqrt(1 - beta2^t). */
void gic_set_temperature_device(const float* t_dev);
int gic_clip_adam_dyn(float* p, const float* g, float* m, float* v, size_t n, const float* sqnorm, float max_norm,
                      float grad_scale, const float* bias_corr_dev, float beta1, float beta2, float eps,
                      gic_stream_t stream);

/* ---- per-step derived discriminator weights ----
 * One adversarial step calls Discriminator.forward three times and backpropagates through it three times
 * (src/training.py:162-169) on the SAME pre-update weights (SURVEY.md Q1).  The quantities derived from the weights
 * alone -- the collapsed score head w_eff = out2logits.weight * feature2out.weight (src/discriminator.py:58-60) and, in
 * GIC_GEMM_BF16 mode, the bf16 copy of highway.weight -- can therefore be computed once:
 * gic_disc_prepare fills prepared[gic_disc_prepared_floats(F)] from the current weights; while
 * gic_disc_set_prepared(prepared) is non-NULL (current context, NULL switches back) gic_disc_fwd / gic_disc_bwd read it
 * instead of recomputing.  The caller must clear it (or prepare again) before the weights change. */
size_t gic_disc_prepared_floats(int F);
int gic_disc_prepare(int mode, const float* W_h /*[F,F]*/, const float* W_f /*[Hd,F]*/, const float* b_f, int Hd,
                     const float* W_o, const float* b_o, int F, float* prepared, gic_stream_t stream);
void gic_disc_set_prepared(const float* prepared);

/* ---- random draws made by the library when the caller supplies none ----
 * The reference draws fresh uniforms every decode step (Tensor.uniform_, src/generator.py:86-90) and fresh dropout masks
 * (nn.Dropout, src/discriminator.py:30,58).  Parity runs pass them in (u[L,B,V], keep masks); a production step passes
 * u = NULL to gic_decode_sample_fwd and the uniforms are then generated INSIDE the fused decode kernel (Philox4x32-10,
 * counter = element index of the logical u[L,B,V], no 4*L*B*V-byte tensor is written or read).
 * gic_set_rng(seed, offset, state_dev): generator state for the calls that follow (current context).  state_dev != NULL:
 *   {seed, offset} are read from device memory when the kernels run (CUDA-graph replay with a fresh offset per step).
 * gic_philox_uniform(tag, n, out): the first n elements of the logical stream `tag` (GIC_RNG_TAG_GUMBEL: exactly the
 *   uniforms the decode uses for u = NULL, so out[L*B*V] passed back in as `u` reproduces that decode bit for bit).
 * gic_philox_keep_mask(tag, n, p, out): uint8 keep masks out[i] = (u_i >= p) for nn.Dropout(p) (GIC_RNG_TAG_DROPOUT). */
#define GIC_RNG_TAG_GUMBEL 0x47u
#define GIC_RNG_TAG_DROPOUT 0x44u
void gic_set_rng(unsigned long long seed, unsigned long long offset, const unsigned long long* state_dev);
int gic_philox_uniform(unsigned int tag, size_t n, float* out, gic_stream_t stream);
int gic_philox_keep_mask(unsigned int tag, size_t n, float p, uint8_t* out, gic_stream_t stream);

/* ---- synchronised BatchNorm for the encoder projection under data parallelism (SURVEY.md section 8e) ----
 * Encoder.bn (src/generator.py:16,24) is the one op of the path that is not row-local: its training-mode statistics run
 * over the whole batch.  With the batch sharded over ranks each half of gic_encoder_fwd / gic_encoder_bwd is split in
 * two, with an all-reduce(sum) of stats[2*E] by the caller in between; count = rows of the GLOBAL batch.
 *   fwd_stats : lin_out = pooled W^T + b;  stats = [sum_b y | sum_b y^2]                  (local rows)
 *   fwd_apply : mean = s1/count, var = s2/count - mean^2 (biased), features = (y - mean) rstd gamma + beta
 *   bwd_stats : stats = [sum_b dout | sum_b dout * xhat]                                  (local rows)
 *   bwd_apply : dlin = gamma rstd (dout - s1/count - xhat s2/count); dW, db from the local rows; dgamma / dbeta =
 *               (global sums) * grad_share, grad_share = 1/world: every rank holds the same value, so the all-reduce(sum)
 *               of the flat gradients followed by the optimizer's 1/world factor yields the global-batch gradient. */
int gic_encoder_fwd_stats(int mode, const float* pooled, int B, int Fin, int E, const float* W, const float* b,
                          float* lin_out, float* stats, gic_stream_t stream);
int gic_encoder_fwd_apply(const float* lin_out, int B, int E, const float* gamma, const float* beta, float eps,
                          const float* stats, float count, float* save_mean, float* save_rstd, float* features,
                          gic_stream_t stream);
int gic_encoder_bwd_stats(const float* dfeatures, const float* lin_out, const float* save_mean, const float* save_rstd,
                          int B, int E, float* stats, gic_stream_t stream);
int gic_encoder_bwd_apply(int mode, const float* dfeatures, const float* pooled, const float* lin_out,
                          const float* save_mean, const float* save_rstd, const float* gamma, int B, int Fin, int E,
                          const float* stats, float count, float grad_share, float* dlin_ws, float* dW, float* db,
                          float* dgamma, float* dbeta, gic_stream_t stream);

/* ---- batch contract: collate_fn (src/tasks.py:138-158), the step immediately before the path ----
 * The ragged token lists of a batch arrive as tokens[sum(len)] (int32, caption after caption) and offsets[B+1] (int32,
 * offsets[b] = start of caption b); captions[B, max_caption_len] int64 = <S>=1, tokens, <E>=2, <PAD>=0 ... and
 * lengths[B] int32 = len + 2 (may be NULL) are written on the device.  max_caption_len = longest caption + 2 is the
 * host's to compute (the reference returns it as a Python int, src/tasks.py:147,158). */
int gic_pack_captions(const int32_t* tokens, const int32_t* offsets, int B, int max_caption_len, int64_t* captions,
                      int32_t* lengths, gic_stream_t stream);

/* ---- data-parallel overlap hook ----
 * gic_set_vocab_grads_event(ev): while ev (a cudaEvent_t, NULL to clear; current context) is registered,
 * gic_decode_sample_bwd / _bwd_factored / _bwd_attn record it on their stream as soon as dW_out and db_out are final
 * -- before the serial BPTT tail -- so the caller can all-reduce that bucket on another stream underneath the rest of
 * the backward (the reference is single-GPU; SURVEY.md section 8e). */
void gic_set_vocab_grads_event(void* cuda_event);
/* gic_set_embed_grads_event(ev): the same for dW_emb (embed.weight's gradient, another 40 % of the generator's gradient
 * bytes at c2): recorded right after the embedding scatter, which the backward runs BEFORE its weight-gradient GEMMs so
 * that this bucket's all-reduce overlaps them. */
void gic_set_embed_grads_event(void* cuda_event);

/* ---- data-parallel gradient exchange over NVLink / NVSwitch peer memory (SURVEY.md section 8e, "gic_allreduce") ----
 * The reference is single-GPU (--device-ids is parsed and ignored, src/args.py:213-216,276); data parallelism over the
 * image batch needs ONE exchange per step: the sum over ranks of the flat G and D gradients, before clip_grad_norm_
 * (src/training.py:198).  gic_allreduce does it in one kernel over peer memory -- reduce-scatter + all-gather with direct
 * NVLink loads / stores, sums in rank order (bit-identical on every rank), the square norm of the reduced gradient
 * accumulated in the same pass (what gic_grad_sqnorm would compute next) -- see csrc/allreduce.cu.
 *
 * A communicator owns the one allocation this library makes: a symmetric buffer of data_bytes that every rank of the
 * node maps through CUDA IPC.  Gradient buffers to be reduced must live inside it (gic_comm_buffer); one process per GPU.
 *   gic_comm_create       allocate this rank's buffer (device = current device); NULL on error
 *   gic_comm_ipc_handle   write gic_comm_handle_bytes() bytes describing it; the caller all-gathers them by rank
 *   gic_comm_open         map every peer's buffer from the gathered handles (world * gic_comm_handle_bytes() bytes)
 *   gic_allreduce         buf[0..n) (inside the buffer, 16-byte aligned, n % 4 == 0) := sum over ranks, in place, on `stream`;
 *                         every rank must call it with the same offset, n and channel.  channel (0..3): independent flag
 *                         sets -- calls that may overlap in time (different streams) need different channels.  sqnorm
 *                         (device float, may be NULL): += sum of squares of the reduced buf, the same value on every rank.
 *   gic_comm_error        non-zero after a wait on a peer expired (2 s): the ranks lost step
 * In-process group (tests on one GPU): W communicators of one process become each other's peers (gic_comm_local_group)
 * and gic_allreduce_local_group runs all W ranks as ONE launch (the ranks' CTAs are co-resident by construction). */
typedef struct gic_comm gic_comm_t;
gic_comm_t* gic_comm_create(int rank, int world, size_t data_bytes);
size_t gic_comm_handle_bytes(void);
int gic_comm_ipc_handle(gic_comm_t* comm, void* out_handle);
int gic_comm_open(gic_comm_t* comm, const void* handles_by_rank);
void* gic_comm_buffer(gic_comm_t* comm);
size_t gic_comm_buffer_bytes(gic_comm_t* comm);
int gic_comm_error(gic_comm_t* comm);
void gic_comm_destroy(gic_comm_t* comm);
int gic_allreduce(float* buf, size_t n, gic_comm_t* comm, int channel, float* sqnorm, gic_stream_t stream);
int gic_comm_local_group(gic_comm_t* const* comms, int world);
int gic_allreduce_local_group(gic_comm_t* const* comms, float* const* bufs, float* const* sqnorms, size_t n, int world,
                              int channel, gic_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GIC_B200_H_ */
