/* libfact_sm100.so -- C ABI of the B200-native FACT hot path (sm_100a).
 *
 * The reference (google-research/mint) has no FFI: its seam is the Python object contract between mint/ctl and
 * the model (SURVEY.md 8b).  Each entry point below names the reference computation it replaces (file:line
 * relative to the reference tree).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless named host_*; the caller owns every buffer (no hidden allocation);
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), returns 0 or a negative FACT_ERR_*;
 *    fact_last_error() returns a thread-local description of the last failure;
 *  - threading: calls on distinct streams may run from distinct threads.  Process-wide state is limited to (a) the
 *    fact_set_flag developer switches (plain ints: change them only while no call is in flight), (b) mutex-guarded
 *    caches of TMA descriptors and of captured AR frame graphs (the latter owned by a fact_ar_session, see below), and
 *    (c) per-thread, per-device helper streams / events;
 *  - activations are row-major fp32 [tokens, features]; "split" buffers are bf16 row-major, `hi` always present,
 *    `lo` present only in FACT_MODE_PRECISE (x ~= hi + lo, see DESIGN.md "bf16x3");
 *  - Keras weight layout is [in, out] row-major (y = x.W); packed GEMM weights are [out, in] bf16 (K-major);
 *  - mode: FACT_MODE_PRECISE = bf16x3 split products, fp32 accumulate (meets the 1e-3 parity bar);
 *          FACT_MODE_BF16    = single bf16 product (throughput mode, reported separately);
 *          FACT_MODE_FP32_SIMT = CUDA-core fp32 GEMMs (debug cross-check only; attention core stays precise).
 */
#ifndef FACT_SM100_H_
#define FACT_SM100_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FACT_OK 0
#define FACT_ERR_BAD_SHAPE (-1)
#define FACT_ERR_BAD_ALIGN (-2)
#define FACT_ERR_CUDA (-3)
#define FACT_ERR_WORKSPACE (-4)
#define FACT_ERR_UNSUPPORTED (-5)

#define FACT_MODE_PRECISE 0
#define FACT_MODE_BF16 1
#define FACT_MODE_FP32_SIMT 2

#define FACT_ABI_VERSION 4

#if defined(__GNUC__)
#define FACT_API __attribute__((visibility("default")))
#else
#define FACT_API
#endif

FACT_API int fact_abi_version(void);
FACT_API const char* fact_last_error(void);
/* Kernels launched by this library on the calling thread so far (each replay of the captured AR frame graph counts
 * the kernels it contains). */
FACT_API long long fact_launch_count(void);

/* ---- weights -------------------------------------------------------------------------------------------- */

/* One transformer layer = Residual(Norm(Attention)) + Residual(Norm(MLP)), base_models.py:102-106. */
typedef struct fact_layer_weights {
  const float* ln1_gamma;  /* [d]            base_models.py:27  */
  const float* ln1_beta;   /* [d]                               */
  const void* wqkv_hi;     /* bf16 [3d, d]   packed to_qkv kernel (no bias), base_models.py:68 */
  const void* wqkv_lo;     /* bf16 [3d, d] or NULL (FACT_MODE_BF16) */
  const void* wo_hi;       /* bf16 [d, d]    packed to_out kernel, base_models.py:69 */
  const void* wo_lo;
  const float* bo;         /* [d] */
  const float* ln2_gamma;  /* [d] */
  const float* ln2_beta;   /* [d] */
  const void* w1_hi;       /* bf16 [ff, d]   packed MLP dense_0 kernel, base_models.py:51-52 */
  const void* w1_lo;
  const float* b1;         /* [ff] */
  const void* w2_hi;       /* bf16 [d, ff]   packed MLP dense_1 kernel, base_models.py:53 */
  const void* w2_lo;
  const float* b2;         /* [d] */
  /* Keras-layout fp32 kernels, only read in FACT_MODE_FP32_SIMT (may be NULL otherwise) */
  const float* wqkv_f32;   /* [d, 3d] */
  const float* wo_f32;     /* [d, d]  */
  const float* w1_f32;     /* [d, ff] */
  const float* w2_f32;     /* [ff, d] */
  /* Keras-layout ([in, out]) bf16 copies: K-major B operands of the backward dX = dY . W^T GEMMs (training only) */
  const void* wqkv_kl;     /* bf16 [d, 3d] */
  const void* wo_kl;       /* bf16 [d, d]  */
  const void* w1_kl;       /* bf16 [d, ff] */
  const void* w2_kl;       /* bf16 [ff, d] */
} fact_layer_weights;

typedef struct fact_dims {
  int d_model;       /* 800  */
  int n_heads;       /* 10   */
  int d_ff;          /* 3072 */
  int motion_layers; /* 2    */
  int audio_layers;  /* 2    */
  int cross_layers;  /* 12   */
  int motion_seq;    /* 120  */
  int audio_seq;     /* 240  */
  int motion_dim;    /* 225  */
  int audio_dim;     /* 35   */
  int out_dim;       /* 225  */
} fact_dims;

/* All weights of FACTModel (fact_model.py:43-70). Layer arrays are host arrays of structs holding device pointers. */
typedef struct fact_weights {
  const fact_layer_weights* motion_layers; /* host array [motion_layers] */
  const fact_layer_weights* audio_layers;  /* host array [audio_layers]  */
  const fact_layer_weights* cross_layers;  /* host array [cross_layers]  */
  const float* motion_embed_w;             /* [motion_dim, d] Keras layout (base_models.py:135) */
  const float* motion_embed_b;             /* [d] */
  const float* motion_pos;                 /* [motion_seq, d] (base_models.py:148-156) */
  const float* audio_embed_w;              /* [audio_dim, d] */
  const float* audio_embed_b;              /* [d] */
  const float* audio_pos;                  /* [audio_seq, d] */
  const float* out_w;                      /* [d, out_dim] Keras layout fp32 (base_models.py:176-180) */
  const float* out_b;                      /* [out_dim] */
  const void* out_w_hi;                    /* bf16 [out_dim, d] packed, for the all-rows head */
  const void* out_w_lo;
  const void* out_w_kl;                    /* bf16 [d, pad64(out_dim)] Keras layout, zero padded (training only) */
} fact_weights;

/* fp32 gradients, same shapes and Keras layout as the master weights (single_task_trainer.py:163-178). */
typedef struct fact_layer_grads {
  float *ln1_gamma, *ln1_beta, *wqkv, *wo, *bo, *ln2_gamma, *ln2_beta, *w1, *b1, *w2, *b2;
} fact_layer_grads;

typedef struct fact_grads {
  const fact_layer_grads* motion_layers; /* host arrays, like fact_weights */
  const fact_layer_grads* audio_layers;
  const fact_layer_grads* cross_layers;
  float *motion_embed_w, *motion_embed_b, *motion_pos, *audio_embed_w, *audio_embed_b, *audio_pos, *out_w, *out_b;
} fact_grads;

/* Pack a Keras-layout fp32 kernel [k_in, n_out] into K-major bf16 [n_out, k_in]: hi = bf16(w), lo = bf16(w-hi).
 * lo may be NULL. */
FACT_API int fact_pack_weight(const float* w_keras, void* hi, void* lo, int k_in, int n_out, void* stream);

/* The same for `count` kernels in ONE launch (arrays of host pointers / sizes; lo may be NULL, or hold NULL entries):
 * what the training step calls after every optimizer update. */
FACT_API int fact_pack_weights(const float* const* w_keras, void* const* hi, void* const* lo, const int* k_in,
                               const int* n_out, int count, void* stream);

/* ---- building-block kernels (each is also a unit-test seam) ---------------------------------------------- */

/* Norm: y = LayerNorm(x; gamma, beta, eps=1e-5) (base_models.py:27-31), written as bf16 hi (+lo).
 * gamma == NULL means "no normalisation": plain fp32 -> bf16 split of x. */
FACT_API int fact_layernorm_split(const float* x, const float* gamma, const float* beta, void* y_hi, void* y_lo,
                         int rows, int d, void* stream);

/* Epilogues of fact_gemm */
#define FACT_EPI_SPLIT 0           /* out_hi/lo = split(acc * (col < scale_cols ? scale : 1))            */
#define FACT_EPI_BIAS_GELU_SPLIT 1 /* out_hi/lo = split(gelu_tanh(acc + bias))   (base_model_util.py:94) */
#define FACT_EPI_BIAS_RESID_F32 2  /* out_f32[map(row)] = acc + bias + resid[row]                        */
#define FACT_EPI_BIAS_F32 3        /* out_f32 = acc + bias                                               */
#define FACT_EPI_BIAS_GELU_SAVE 4  /* z = acc + bias: out_hi = bf16(gelu_tanh(z)), out_lo = bf16(z) (training fwd)  */
#define FACT_EPI_GELU_GRAD 5       /* out_hi = bf16(acc * gelu_tanh'(aux[row, col]))  (aux = saved z, bf16)          */

typedef struct fact_gemm_epilogue {
  int kind;           /* FACT_EPI_* */
  float* out_f32;     /* [*, ldo] */
  void* out_hi;       /* bf16 [*, ldo] */
  void* out_lo;       /* bf16 or NULL */
  int ldo;            /* output row pitch in elements */
  const float* bias;  /* [n] or NULL */
  const float* resid; /* [m, ldr] or NULL */
  int ldr;
  float scale;        /* FACT_EPI_SPLIT: multiplier of the first scale_cols columns (folds the attention scale) */
  int scale_cols;
  /* output-row remap for zero-copy concat (base_models.py:192-193): out_row = (row / seq_in) * seq_out + seq_off
   * + row % seq_in ; seq_in == 0 disables it */
  int seq_in, seq_out, seq_off;
  const void* aux;    /* FACT_EPI_GELU_GRAD: bf16 [m, ldaux] pre-activation saved by FACT_EPI_BIAS_GELU_SAVE */
  int ldaux;
  /* optional fp32 scratch (16-byte aligned): lets small problems (m <= 1024) deal their K blocks over all SMs; needs
   * splits * m * n * 4 bytes, the library uses as many splits as fit.  NULL = never split. */
  void* splitk_scratch;
  size_t splitk_scratch_bytes;
  /* FACT_EPI_GELU_GRAD, optional: colsum[c] += sum over rows of the bf16 output (the bias gradient of the FFN hidden
   * layer) -- folded into the epilogue instead of a second pass over the [m, n] output.  fp32 [n], NULL = skip. */
  float* colsum;
  /* FACT_EPI_BIAS_RESID_F32, optional: > 0 makes resid a [resid_rows, ldr] table read at row % resid_rows (the
   * position embedding added to every clip, base_models.py:148-156); 0 = resid has one row per output row. */
  int resid_rows;
  /* FACT_EPI_BIAS_RESID_F32 without row remap, optional: after the output rows are final also write
   * LayerNorm(out row; gamma, beta, eps 1e-5) split into bf16 hi / lo [m, n] (pitch n) -- the operand of the GEMM that
   * follows in a pre-norm transformer (base_models.py:27-31).  Small m: fused into the split-K finish kernel; otherwise
   * the LayerNorm launch follows the GEMM inside the call.  ln_hi NULL = off; ln_lo NULL = single bf16. */
  const float* ln_gamma;
  const float* ln_beta;
  void* ln_hi;
  void* ln_lo;
  /* optional with ln_hi: 2 * ((m + 31) / 32 + 1) ints, zero before the first call and left zero by every call.  With it, large
   * problems (CTA-pair path, n a multiple of 160) normalise their rows INSIDE the GEMM launch: dedicated warps wait
   * until all column tiles of a 32-row group have landed (arrival counters in ln_sync) and write the bf16 hi / lo
   * rows while the tensor pipe works on the next tiles -- no LayerNorm launch, no second HBM read of the residual
   * stream.  Calls that share an ln_sync array must be ordered on one stream.  NULL = LayerNorm as its own launch. */
  int* ln_sync;
} fact_gemm_epilogue;

/* C[m,n] = A[m,k] . W[n,k]^T on the tcgen05 tensor path (TMA-staged, TMEM accumulators).
 * a_hi/a_lo: bf16 [m, lda]; w_hi/w_lo: bf16 [n, ldw] (packed).  lo pointers NULL -> single bf16 product.
 * Replaces the Keras Dense matmuls at base_models.py:51-53, 68-69, 176-180. */
FACT_API int fact_gemm(const void* a_hi, const void* a_lo, int lda, const void* w_hi, const void* w_lo, int ldw,
              int m, int n, int k, const fact_gemm_epilogue* epi, void* stream);

/* fp32 CUDA-core GEMM, Keras-layout weight [k, n] (debug mode and the tiny embedding projections). Same epilogues. */
FACT_API int fact_gemm_f32(const float* a, int lda, const float* w_keras, int m, int n, int k,
                  const fact_gemm_epilogue* epi, void* stream);

/* Attention core: softmax(q.k^T) . v per (batch, head), no mask (base_models.py:82-85).  qkv: bf16 [batch*n, 3d],
 * column order (qkv, head, dh) (base_models.py:71-72); q must already carry scale*log2(e) (FACT_EPI_SPLIT scale).
 * out: bf16 [batch*n, d], heads merged "b h n d -> b n (h d)" (base_models.py:73). */
FACT_API int fact_sdpa(const void* qkv_hi, const void* qkv_lo, void* out_hi, void* out_lo, int batch, int n, int heads,
              int head_dim, void* stream);

/* Developer switches (defaults in brackets): "sdpa_legacy" [0] = 1 forces the generic mma.sync attention kernel;
 * "gemm_pair" [1] = 0 forces the 1-SM GEMM, 2 forces the CTA-pair GEMM; "gemm_splitk" [1] = 0 disables split-K; "dual_stream" [1] = 0 keeps both modality encoders on one stream;
 * "gemm_bn" [0] forces the GEMM N tile (128 / 160 / 256); "ar_prune" [1] = 0 runs the full last layer
 * in fact_infer_auto_regressive instead of the row-0 tail. */
FACT_API int fact_set_flag(const char* name, int value);

/* LinearEmbedding + PositionEmbedding (fact_model.py:88-90,94-95; base_models.py:135,156):
 * y[b*n_tok + t, :] = x[b, start + t, :f] . W[f, d] + bias + pos[t, :],  start = step_ptr ? *step_ptr : 0.
 * x is [batch, x_len, f] with batch stride x_batch_stride elements. */
FACT_API int fact_embed(const float* x, long long x_batch_stride, const int* step_ptr, const float* w, const float* bias,
               const float* pos, float* y, int batch, int n_tok, int f, int d, void* stream);

/* Output Dense on selected rows (base_models.py:200 + fact_model.py:128): for b < batch,
 * out[b*out_batch_stride + (*step_ptr)*out_dim + j] = x[b*row_stride*d + :] . W[:, j] + bias[j]. */
FACT_API int fact_head_rows(const float* x, long long row_stride, const float* w_keras, const float* bias, float* out,
                   long long out_batch_stride, const int* step_ptr, int batch, int d, int out_dim, void* stream);

/* MSE loss (fact_model.py:143-148): *loss = mean((target - pred[:, :t_len])^2); if dpred != NULL also writes
 * dpred[B, n, out_dim] = dloss/dpred * loss_scale (zeros beyond t_len). partial: >= 1024 floats of scratch. */
FACT_API int fact_mse(const float* target, const float* pred, float* loss, float* dpred, float* partial, int batch, int t_len,
             int n, int out_dim, float loss_scale, void* stream);

/* Training windows from a device-resident dataset (inputs_util.py:59-107 with the sequences decoded once and motion
 * already padded to motion_dim): for b < batch, m0 = motion_row[b], a0 = audio_row[b]:
 *   motion_out[b, t, :] = motion[m0 + t, :]                 t < motion_len
 *   target_out[b, t, :] = motion[m0 + target_shift + t, :]  t < target_len
 *   audio_out[b, t, :]  = audio[a0 + t, :]                  t < audio_len
 * motion is [rows, motion_dim], audio [rows', audio_dim] (64-bit row arithmetic); the caller guarantees every window
 * lies inside its arena.  batch <= 65535. */
FACT_API int fact_gather_windows(const float* motion, int motion_dim, const float* audio, int audio_dim,
                                 const long long* motion_row, const long long* audio_row, int batch, int motion_len,
                                 int target_shift, int target_len, int audio_len, float* motion_out, float* target_out,
                                 float* audio_out, void* stream);

/* ---- whole-model entry points --------------------------------------------------------------------------- */

FACT_API size_t fact_workspace_bytes(const fact_dims* dims, int batch, int mode);

/* FACTModel.call (fact_model.py:72-101): motion [B, motion_seq, motion_dim], audio [B, audio_seq, audio_dim]
 * -> out [B, motion_seq + audio_seq, out_dim]. */
FACT_API int fact_forward(const fact_dims* dims, const fact_weights* w, const float* motion, const float* audio, float* out,
                 int batch, void* workspace, size_t workspace_bytes, int mode, void* stream);

/* FACTModel.infer_auto_regressive (fact_model.py:103-132), frames [start_frame, start_frame + n_frames).
 * motion_hist: [B, motion_seq + hist_capacity, motion_dim]; the first motion_seq rows hold the seed, generated frames
 * are appended in place (the shift-by-one of fact_model.py:131 is an index offset into this buffer), so a call with
 * start_frame > 0 continues a previous one.  audio: [B, audio_len, audio_dim].
 * start_frame + n_frames must be <= min(hist_capacity, audio_len - audio_seq + 1) (the caller applies the early-stop
 * rule of fact_model.py:125-126).  step_counter: device int scratch.
 * use_graph != 0 replays one captured CUDA graph per frame (needs a non-default stream).
 * session: owner of the captured frame graphs (fact_ar_session_create), NULL = a process-wide default session.  A graph
 * is keyed on everything it bakes in (the whole weight table, dims, buffers, sizes, mode, developer flags, device) and a
 * session keeps at most 12 of them (least recently used evicted one at a time).  Destroy the session before freeing the
 * weights / buffers its graphs point into -- e.g. together with the model object. */
FACT_API int fact_infer_auto_regressive(const fact_dims* dims, const fact_weights* w, float* motion_hist,
                                        int hist_capacity, const float* audio, int audio_len, int batch,
                                        int start_frame, int n_frames, int* step_counter, void* workspace,
                                        size_t workspace_bytes, int mode, int use_graph, void* session, void* stream);

/* Owner of captured AR frame graphs.  create returns NULL on allocation failure; destroy(NULL) is a no-op; destroying a
 * session whose graphs are still running is allowed (resources are released when the launches complete). */
FACT_API void* fact_ar_session_create(void);
FACT_API int fact_ar_session_destroy(void* session);
/* Graphs currently cached by `session` (NULL = the default session): test / diagnostics seam. */
FACT_API int fact_ar_session_graphs(void* session);

/* ---- training blocks (bf16 product path; reference semantics: mint/ctl/single_task_trainer.py:138-199) -------- */

/* Attention core with the per-row log2-sum-exp saved for the backward pass: lse[(b*heads + h)*n + row] (may be NULL).
 * Same contract as fact_sdpa otherwise. */
FACT_API int fact_sdpa_lse(const void* qkv_hi, const void* qkv_lo, void* out_hi, void* out_lo, float* lse, int batch,
                           int n, int heads, int head_dim, void* stream);

/* dW[in_dim, out_dim] += X^T . dY  (Keras-layout gradient of a Dense kernel): x_bf16 [tokens, ldx], dy_bf16 [tokens,
 * ldy], fp32 accumulate with atomics (zero dw first).  tcgen05, both operands MN-major through TMA, split-K. */
FACT_API int fact_wgrad_gemm(const void* x_bf16, int ldx, const void* dy_bf16, int ldy, float* dw, int ldw, int tokens,
                             int in_dim, int out_dim, void* stream);

/* Backward of fact_sdpa: qkv bf16 [batch*n, 3d] as written by the forward QKV epilogue (q pre-scaled), o / d_o bf16
 * [batch*n, d], lse from fact_sdpa_lse; writes dqkv bf16 [batch*n, 3d] = d loss / d (unscaled q, k, v).
 * d_scratch: fp32 [batch*heads*n]; dq_scratch: fp32 [batch*n*d]; scale = d_model^-0.5. */
FACT_API int fact_sdpa_backward(const void* qkv, const void* o, const void* d_o, const float* lse, float* d_scratch,
                                float* dq_scratch, void* dqkv, int batch, int n, int heads, int head_dim, float scale,
                                void* stream);

/* dx = dres + d LayerNorm(x; gamma)^T dy (dres may be NULL, dx may alias dres); dgamma / dbeta accumulate (zero them
 * first).  stats_scratch: 4 * rows floats (16-byte aligned). */
FACT_API int fact_layernorm_backward(const float* x, const float* gamma, const float* dy, const float* dres, float* dx,
                                     float* dgamma, float* dbeta, float* stats_scratch, int rows, int d, void* stream);

/* Gradients of fact_embed: dw[f, d] += x^T dy, dbias[d] += colsum(dy), dpos[n_tok, d] += sum over clips (may be NULL). */
FACT_API int fact_embed_backward(const float* x, long long x_batch_stride, const float* dy, float* dw, float* dbias,
                                 float* dpos, int batch, int n_tok, int f, int d, void* stream);

/* y_bf16[r, 0:ldy] = bf16(x[r, 0:n]) zero padded, colsum[c] += sum_r x[r, c] (either output may be NULL). */
FACT_API int fact_cast_colsum(const float* x, int ldx, void* y_bf16, int ldy, float* colsum, int rows, int n,
                              void* stream);

/* bf16 copy of a Keras-layout kernel [rows, cols] with row pitch ld_out (zero padded): B operand of dX = dY . W^T. */
FACT_API int fact_cast_weight(const float* w_keras, void* out_bf16, int rows, int cols, int ld_out, void* stream);

/* Keras Adam (trainer.py:150; beta1 .9, beta2 .999, epsilon 1e-7 outside the root) on a flat range;
 * g is multiplied by grad_scale first (global-norm clipping). step counts from 1.  w_bf16 (optional, n elements): also
 * receives bf16(w) -- the Keras-layout operand copies of the backward GEMMs, refreshed without another pass. */
FACT_API int fact_adam_step(float* w, const float* g, float* m, float* v, long long n, float lr, float beta1,
                            float beta2, float eps, long long step, float grad_scale, void* w_bf16, void* stream);

/* Data-parallel optimizer step fused with its collective (single_task_trainer.py:186-187 + trainer.py:150): the
 * cross-replica SUM of the gradients, the Keras Adam update and the re-mirroring of the variables in ONE kernel over
 * NVLink peer memory.  Every replica keeps its flat gradient bucket, fp32 master weights and bf16 weight mirror inside
 * one "arena" of symmetric memory (same layout on every rank); peer_base[p] is rank p's arena as mapped into this
 * process (host array of `world` device pointers), grad_off / w_off / wb_off the byte offsets of the three arrays inside
 * it.  mc_base: the NVSwitch multicast mapping of the arenas (multimem.ld_reduce / multimem.st: one load reduces over
 * all replicas in the switch, one store reaches all of them), or NULL to loop over peer_base with P2P loads / stores.
 * This rank updates elements [rank * per, (rank + 1) * per) of the n-element bucket, per = ceil(n / world) rounded up to
 * a multiple of 8: it sums that shard of every replica's gradient, advances ITS shard of m / v (fp32 [n] arrays local
 * to this rank: optimizer state is sharded, the other shards are never touched) and stores the new weights -- fp32 and
 * bf16 -- into every replica.  The caller must put a cross-replica barrier before the call (all gradients final) and
 * after it (all stores landed); world <= 16.  Same arithmetic as fact_adam_step. */
FACT_API int fact_dp_adam_step(void* const* peer_base, void* mc_base, long long grad_off, long long w_off,
                               long long wb_off, float* m, float* v, long long n, int rank, int world, float lr,
                               float beta1, float beta2, float eps, long long step, float grad_scale, void* stream);

/* The same on elements [off, off + count) of the bucket only (off, count multiples of 4): this rank updates
 * off + [rank * per, (rank + 1) * per), per = ceil(count / world) rounded up to a multiple of 8.  A data-parallel host
 * calls it once per slice of the bucket as the backward finishes the slices (fact_train_step's stage events), on a
 * side stream, with a cross-replica barrier in front of every call: the slice's gradient sum, update and broadcast run
 * UNDER the rest of the backward -- which no longer reads that slice's weights -- and only the last slice is exposed.
 * max_blocks > 0 caps the grid (a small grid shares the SMs with the backward's persistent GEMMs instead of taking
 * them); 0 = as many blocks as the range needs. */
FACT_API int fact_dp_adam_range(void* const* peer_base, void* mc_base, long long grad_off, long long w_off,
                                long long wb_off, float* m, float* v, long long off, long long count, int rank,
                                int world, float lr, float beta1, float beta2, float eps, long long step,
                                float grad_scale, int max_blocks, void* stream);

/* *out = sum g^2 (for clip_by_global_norm, single_task_trainer.py:180-183). */
FACT_API int fact_sum_squares(const float* g, long long n, float* out, void* stream);

FACT_API size_t fact_train_workspace_bytes(const fact_dims* dims, int batch);

/* One replica's train step up to the gradients (single_task_trainer.py:145-178): forward with saved activations,
 * *loss_out = FACTModel.loss(target, pred) (unscaled), gradients of loss * loss_scale ACCUMULATED into `g` (zero the
 * gradient buffers first; loss_scale = 1 / num_replicas as in :157-158).  bf16 products, fp32 everything else.
 * target: [B, target_len, out_dim].
 * stage_events (optional, NULL = none): host array of n_stage_events cudaEvent_t (entries may be NULL).  The backward
 * finishes the gradient bucket in stages and records stage_events[i] on `stream` when stage i is final:
 *   0                      the output head (out_w, out_b)
 *   1 .. Lc                cross-modal layers Lc-1, Lc-2, ..., 0
 *   Lc+1 .. Lc+Lm          motion layers Lm-1, ..., 0 (the last one also covers motion_pos and the motion embedding)
 *   Lc+Lm+1 .. Lc+Lm+La    audio layers La-1, ..., 0 (the last one also covers audio_pos and the audio embedding; it is
 *                          recorded after all work of the call)
 * A data-parallel host starts the cross-replica sum of a finished slice of its gradient bucket on another stream while
 * the rest of the backward runs (mint_b200/trainer.py). */
FACT_API int fact_train_step(const fact_dims* dims, const fact_weights* w, const fact_grads* g, const float* motion,
                             const float* audio, const float* target, int target_len, int batch, float loss_scale,
                             float* loss_out, void* workspace, size_t workspace_bytes, void* const* stage_events,
                             int n_stage_events, void* stream);

/* g[i] *= clip_norm / max(sqrt(*sum_squares), clip_norm) -- tf.clip_by_global_norm (single_task_trainer.py:180-183)
 * with the squared global norm read from DEVICE memory (fact_sum_squares output): no host synchronisation. */
FACT_API int fact_clip_scale(float* g, long long n, const float* sum_squares, float clip_norm, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FACT_SM100_H_ */
