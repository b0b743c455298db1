/*
 * psvae_b200.h -- C-ABI of the B200-native hot path of pseudo_speaker_VAE.
 *
 * The reference has no FFI layer: its boundary for this path is the Python module API
 * (SURVEY.md 8(b)).  The host package `pseudo_speaker_vae_b200` keeps that API (same class names,
 * signatures, state_dict keys, metric names) and binds the entry points below with ctypes
 * (pseudo_speaker_vae_b200/_lib.py; the stub a maintainer of the reference would add is shown in
 * INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says "host".
 *   - the caller allocates everything (parameters, gradients, workspace, outputs); the library never
 *     allocates device memory and keeps no pointer past the call (TMA descriptors are cached by
 *     (pointer, shape) and hold no ownership).
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*); no host sync inside.
 *   - return 0 = ok; < 0 = argument / shape / alignment / unsupported (text via
 *     psvae_last_error_string()); > 0 = a cudaError_t.  No exceptions cross the boundary.
 *   - there is no CPU fallback: without an sm_100 device the compute entry points return an error.
 *   - tensors are contiguous row-major; `Linear` weights are W[out][in] fp32 inside one flat
 *     parameter buffer whose layout `psvae_model_desc_init` defines (so Adam and the DDP-style
 *     gradient all-reduce are single-buffer operations).
 */
#ifndef PSVAE_B200_H_
#define PSVAE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSVAE_ABI_VERSION 5      /* 4: + psvae_adam_step_ex (amsgrad / maximize); 5: + device step counters (CUDA-graph replay) */
#define PSVAE_MAX_LAYERS 8      /* Linear layers per MLP (num_hidden + 1) */
#define PSVAE_MAX_CLF_TRUNK 4   /* hidden Linear layers of the latent classifier */
#define PSVAE_MAX_CLF_HEADS 4   /* output heads of the latent classifier */
#define PSVAE_NUM_LOSSES 16

/* precision of the GEMM chains */
#define PSVAE_FP32 0 /* CUDA-core FFMA, fp32 storage: the 1e-5 parity mode                       */
#define PSVAE_BF16 1 /* tcgen05 kind::f16 (bf16 operands, fp32 accumulate in TMEM), bf16 storage */

/* element type of the input batch x: the reference's DataLoader yields fp32 (ps_vae/data/cv.py:51-76); a bf16 embedding store
 * (pseudo_speaker_vae_b200/data.py) hands its rows over as they are (tensor-core mode only: no cast pass, half the H2D bytes) */
#define PSVAE_X_F32 0
#define PSVAE_X_BF16 1

/* classifier activations (ps_vae/latent_classifier.py:18-23) */
#define PSVAE_ACT_RELU 0
#define PSVAE_ACT_TANH 1
#define PSVAE_ACT_SIGMOID 2
#define PSVAE_ACT_LEAKY_RELU 3

/* slots of the `losses` output (names follow the train_ / val_ metric names of ps_vae/lightning.py:82-83,127-129) */
#define PSVAE_LOSS_TOTAL 0
#define PSVAE_LOSS_RECON 1
#define PSVAE_LOSS_KL 2
#define PSVAE_LOSS_CLF 3       /* mean over heads of the cross entropies                      */
#define PSVAE_LOSS_CLF_HEAD0 4 /* +h : cross entropy of head h                                */
#define PSVAE_LOSS_ACC_HEAD0 8 /* +h : accuracy of head h (argmax == y)                       */
#define PSVAE_LOSS_CONS 12     /* cross entropy of the consistency classifier on x_hat (train_consistency_loss, lightning.py:100-108) */
#define PSVAE_LOSS_CONS_ACC 13 /* its accuracy (train_consistency)                            */

/* Shape of the model plus the layout of the flat fp32 parameter buffer (element offsets).
 * VAEModel: ps_vae/model.py:8-36 generalised by hidden_dim / num_hidden (reference: 512 / 2).
 * LatentClassifier: ps_vae/latent_classifier.py:7-56.  `clf_num_heads == 0` means no classifier;
 * single-label mode is one head whose Linear is the last entry of the reference's `layers`. */
typedef struct psvae_model_desc {
  int32_t input_dim;         /* D  (multiple of 8)            */
  int32_t latent_dim;        /* L  (multiple of 8, <= 256)    */
  int32_t hidden_dim;        /* H  (multiple of 64)           */
  int32_t num_hidden;        /* hidden layers per MLP, >= 1   */
  int32_t normalize_decoder; /* model.py:60-61                */
  int32_t clf_num_trunk;     /* hidden Linear layers (num_layers - 1) */
  int32_t clf_hidden;
  int32_t clf_activation;
  int32_t clf_num_heads;
  int32_t clf_single_label;
  int32_t clf_head_classes[PSVAE_MAX_CLF_HEADS];
  int32_t reserved_[2];
  /* layer j of both encoders sits side by side: W_mu_j at enc_w[j], W_sigma_j right behind it
   * (enc_w[j] + out_j*in_j); same for the biases.  That makes layer 0 of the two encoders one
   * [2H, D] matrix. */
  int64_t enc_w[PSVAE_MAX_LAYERS];
  int64_t enc_b[PSVAE_MAX_LAYERS];
  int64_t dec_w[PSVAE_MAX_LAYERS];
  int64_t dec_b[PSVAE_MAX_LAYERS];
  int64_t clf_trunk_w[PSVAE_MAX_CLF_TRUNK];
  int64_t clf_trunk_b[PSVAE_MAX_CLF_TRUNK];
  int64_t clf_head_w[PSVAE_MAX_CLF_HEADS];
  int64_t clf_head_b[PSVAE_MAX_CLF_HEADS];
  int64_t vae_numel;   /* elements [0, vae_numel) hold the VAE, classifier follows */
  int64_t total_numel; /* length of the flat buffer (padded; padding stays zero)  */
} psvae_model_desc;

/* The frozen EmbeddingClassifier the reference loads as `consistency_classifier` (ps_vae/lightning.py:44-52;
 * ps_vae/embedding_classifier/embedding_classifier.py:29-62): fc1 [hidden, input] -> ReLU -> fc2 [hidden, hidden]
 * -> ReLU -> fc3 [classes, hidden], in its own flat fp32 buffer (element offsets below).  It receives no gradient. */
typedef struct psvae_consistency_desc {
  int32_t input_dim;   /* = psvae_model_desc.input_dim (multiple of 4) */
  int32_t hidden_dim;  /* multiple of 4                                 */
  int32_t num_classes; /* >= 2                                          */
  int32_t reserved_;
  int64_t w[3];
  int64_t b[3];
  int64_t total_numel;
} psvae_consistency_desc;

/* ---- host-only helpers (work without a GPU) ------------------------------------------------- */
int psvae_abi_version(void);
const char* psvae_last_error_string(void);
/* Fill `desc` (shape fields + canonical offsets).  clf_num_heads = 0 for "no classifier". */
int psvae_model_desc_init(psvae_model_desc* desc, int32_t input_dim, int32_t latent_dim, int32_t hidden_dim,
                          int32_t num_hidden, int32_t normalize_decoder, int32_t clf_num_trunk, int32_t clf_hidden,
                          int32_t clf_activation, int32_t clf_num_heads, int32_t clf_single_label,
                          const int32_t* clf_head_classes);
/* bytes of scratch a call needs for `rows` rows at `precision`; mode: PSVAE_MODE_* (decode works through
 * its rows in chunks of the "decode_chunk" option, so its scratch stops growing there) */
#define PSVAE_MODE_TRAIN 0
#define PSVAE_MODE_FORWARD 1
#define PSVAE_MODE_DECODE 2
/* the classifier-only train step (psvae_train_fwd_bwd_scoped with PSVAE_GRAD_CLASSIFIER): the forward buffers plus the classifier's
 * backward buffers -- none of the VAE backward's */
#define PSVAE_MODE_TRAIN_CLASSIFIER 3
int64_t psvae_workspace_bytes(const psvae_model_desc* desc, int64_t rows, int32_t precision, int32_t mode);
/* bytes of the bf16 shadow copy of the parameters (PSVAE_BF16 only) */
int64_t psvae_shadow_bytes(const psvae_model_desc* desc);
/* algorithmic FLOPs per sample (2 x MAC; SURVEY 8(d)): mode 0 = train fwd+bwd, 1 = forward, 2 = decode */
int64_t psvae_flops_per_sample(const psvae_model_desc* desc, int32_t mode);

/* Tuning knobs (process-wide, set before sizing workspaces; defaults in parentheses): "decode_chunk" rows per pass of the per-layer decode
 * path (131072), "decode_chain" (1: psvae_decode runs the chained decoder kernel where the shape allows), "train_chain" (0), "wgrad_split_cap",
 * "colsum_rows", "deterministic" (0; 1: ordered two-stage sums instead of TMA reduce-add / atomics), "pdl" (1: programmatic dependent launch),
 * "tc_two_cta" (1: CTA pairs, tcgen05 cta_group::2), "tc_grouped" (1), "tc_epi_groups" (1) / "tc_epi_groups_max_k", "fused_head" (1),
 * "clf_grad_in_bwd" (0), "tc_merged_wgrad" (1) / "wgrad_order" (1) / "wgrad_splits" (0 = auto), "tc_bn_rounds" (1), "tc_max_stages" (0 = what fits),
 * "tc_trace_ptr" (0) / "tc_trace_skip", and for tests "tc_force_bn"
 * (0|64|128|256), "tc_grid_limit", "langevin_generic".  INTEGRATION.md lists what each one does.  Env PSVAE_OPT_<NAME>=<int> sets them at load. */
int psvae_set_option(const char* name, int64_t value);
int64_t psvae_get_option(const char* name);

/* ---- optimiser: replaces torch.optim.Adam.step() driven by ps_vae/lightning.py:204-205 ------- */
/* One vectorised pass over the flat buffers (28 B/param).  `step` is the 1-based count after increment;
 * g is read as g*grad_scale (1/world_size after a sum all-reduce).  If shadow_bf16 != NULL the updated
 * parameter is also written there as bf16 (the tcgen05 operand copy).  The hyper-parameters are doubles because torch
 * derives its fp32 scalars (1-beta, lr/(1-beta1^t), sqrt(1-beta2^t)) from python doubles; passing floats would not
 * reproduce them. */
int psvae_adam_step(float* p, const float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int64_t step, double grad_scale, void* shadow_bf16, void* stream);
/* The same update with the two torch.optim.Adam switches that `Adam(self.parameters(), **self.hparams["optimizer"])` (lightning.py:205) can
 * reach: amsgrad (vmax = running maximum of v, [n] fp32, caller-allocated and zero-initialised; the denominator uses it) and maximize
 * (the gradient is negated).  With both off this is psvae_adam_step. */
int psvae_adam_step_ex(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, double lr, double beta1,
                       double beta2, double eps, double weight_decay, int64_t step, double grad_scale, int32_t amsgrad,
                       int32_t maximize, void* shadow_bf16, void* stream);

/* ---- generator: replaces torch.randn / randn_like (model.py:57, inference.py:23,73,95) -------- */
int psvae_philox_uint32(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, int64_t first_elem, void* stream);
int psvae_philox_normal(float* out, int64_t n_rows, int32_t n_cols, uint64_t seed, uint64_t offset, int64_t row0,
                        void* stream);

/* ---- batch assembly out of an HBM-resident packed store: replaces the DataLoader collate of ps_vae/data/cv.py:73-76, :111-123 ---- */
/* dst[i][:] = src[idx[i]][:], rows of row_bytes bytes (a multiple of 16; src and dst 16-byte aligned), idx a DEVICE int64 array of n
 * entries (an index outside [0, src_rows) gives a zero row).  The whole Common Voice train split is 345 MB in bf16: it lives in HBM
 * and the per-step traffic over PCIe is the index list. */
int psvae_gather_rows(const void* src, int64_t src_rows, int64_t row_bytes, const int64_t* idx, int64_t n, void* dst, void* stream);

/* ---- bf16 operand copy of the parameters (call after any out-of-band parameter change) -------- */
int psvae_refresh_shadow(const psvae_model_desc* desc, const float* params, void* shadow_bf16, void* stream);

/* ---- VAEModel.forward (ps_vae/model.py:38-63) -------------------------------------------------- */
/* eps == NULL: in-kernel Philox draw with (seed, offset), element index (row0 + r)*L + c. */
int psvae_forward(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, const void* x, int32_t x_dtype,
                  const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, int32_t precision,
                  float* x_hat, float* mu, float* log_sigma, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- VAEModel.decode (model.py:65-69) and unconditional_synthesis (inference.py:10-27) -------- */
/* z == NULL: z ~ N(0, I) from Philox (seed, offset, row0); z_out (optional) receives the z used. */
int psvae_decode(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, const float* z,
                 uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, int32_t precision, float* x_hat,
                 float* z_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- PseudoSpeakerVAE.training_step + loss.backward() (lightning.py:67-131 + autograd) -------- */
/* Computes the losses and ALL parameter gradients (written, not accumulated, into `grads`, same layout
 * as `params`).  y: int64 [num_heads][rows] (NULL without classifier).  use_cos_loss: lightning.py:110-111.
 * compute_grads = 0 gives validation_step (lightning.py:133-197).  x_hat / mu / log_sigma are optional.
 * x: [rows][D] fp32 (x_dtype = PSVAE_X_F32) or bf16 (PSVAE_X_BF16: precision PSVAE_BF16 and the plain MSE tail only -- the bf16
 * values are then both the first GEMM's operand and the reconstruction target).
 * A class label outside [0, classes) makes the classifier loss (and the total) NaN, where torch's cross_entropy raises. */
int psvae_train_fwd_bwd(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads,
                        const void* x, int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset,
                        int64_t row0, int64_t rows, float kl_weight, float clf_weight, int32_t use_cos_loss,
                        int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma,
                        float* losses, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- backward of VAEModel.forward for a caller's OWN loss (autograd through ps_vae/model.py:38-63) --------- */
/* Recomputes the forward pass (same x, same eps or the same (seed, offset, row0) Philox draw as the psvae_forward call it mirrors) and
 * back-propagates the given d loss / d x_hat [rows][D], d loss / d mu, d loss / d log_sigma [rows][L] (each may be NULL = zero) into
 * `grads` (written, not accumulated; the classifier's entries stay zero).  No loss term is added inside.  workspace >=
 * psvae_workspace_bytes(desc, rows, precision, PSVAE_MODE_TRAIN). */
int psvae_vae_backward(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                       int32_t x_dtype, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows, int32_t precision,
                       const float* g_x_hat, const float* g_mu, const float* g_log_sigma, void* workspace, int64_t workspace_bytes,
                       void* stream);

/* ---- the same step with the consistency term (lightning.py:44-52, 100-108, 119-124) ------------ */
int psvae_consistency_desc_init(psvae_consistency_desc* cons, int32_t input_dim, int32_t hidden_dim, int32_t num_classes);
/* scratch the consistency chain needs ON TOP of psvae_workspace_bytes(...) for the same rows / mode (TRAIN or FORWARD) */
int64_t psvae_consistency_workspace_bytes(const psvae_consistency_desc* cons, int64_t rows, int32_t mode);
/* EmbeddingClassifier.forward (embedding_classifier.py:50-62): logits [rows][num_classes] = fc3(relu(fc2(relu(fc1(x))))); fp32 on
 * the CUDA cores.  workspace >= psvae_consistency_workspace_bytes(cons, rows, PSVAE_MODE_FORWARD). */
int psvae_consistency_forward(const psvae_consistency_desc* cons, const float* cons_params, const float* x, int64_t rows,
                              float* logits, void* workspace, int64_t workspace_bytes, void* stream);
/* The stand-alone trainer of the same classifier (embedding_classifier.py:64-100: training_step / validation_step): logits,
 * CrossEntropyLoss (mean) and multiclass accuracy, and -- compute_grads != 0 -- the gradients of the six tensors in the layout of
 * psvae_consistency_desc (written, not accumulated).  losses[0] = the cross entropy, losses[13] = the accuracy (losses has
 * PSVAE_NUM_LOSSES slots).  logits_out (optional) [rows][num_classes].  fp32 on the CUDA cores.
 * workspace >= psvae_embedding_classifier_workspace_bytes(cons, rows).  A label outside [0, num_classes) gives a NaN loss. */
int64_t psvae_embedding_classifier_workspace_bytes(const psvae_consistency_desc* cons, int64_t rows);
int psvae_embedding_classifier_step(const psvae_consistency_desc* cons, const float* params, float* grads, const float* x,
                                    const int64_t* y, int64_t rows, int32_t compute_grads, float* logits_out, float* losses,
                                    void* workspace, int64_t workspace_bytes, void* stream);
/* psvae_train_fwd_bwd plus  cons_weight * CE(consistency_classifier(x_hat), cons_y)  in the total loss; its gradient reaches the
 * decoder through x_hat (through the L2 normalisation when normalize_decoder is set).  cons_y: int64 [rows] (the single-label y of
 * the batch).  losses[PSVAE_LOSS_CONS], [PSVAE_LOSS_CONS_ACC] are filled.  workspace >= psvae_workspace_bytes(...) +
 * psvae_consistency_workspace_bytes(...).  The classifier runs in fp32 on the CUDA cores in both precisions. */
int psvae_train_fwd_bwd_consistency(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads,
                                    const void* x, int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset,
                                    int64_t row0, int64_t rows, float kl_weight, float clf_weight, int32_t use_cos_loss,
                                    int32_t compute_grads, int32_t precision, float* x_hat, float* mu, float* log_sigma,
                                    float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                                    const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y,
                                    float cons_weight);

/* ---- the train step with its per-step scalars in device memory (a CUDA graph replays it unchanged) ---------------------------------
 * A captured launch freezes its kernel arguments, so the three values that change every step -- the Philox offset of the eps draw, Adam's
 * step count and the learning rate -- are read from caller-allocated device memory instead.  The caller keeps one counter block per
 * parameter group it steps together and one fp64 lr per group, writes them (cudaMemcpyAsync) whenever its own host copies change, and
 * ends each step with psvae_step_counters_advance. */
typedef struct psvae_step_counters {
  uint64_t rng_offset; /* Philox offset of the next train step's eps draw                        */
  int64_t adam_step;   /* Adam steps taken so far (the next update uses t = adam_step + 1)       */
  int64_t reserved_[2];
} psvae_step_counters;
/* psvae_train_fwd_bwd_consistency (cons may be NULL: no consistency term) whose in-kernel Philox draw takes its offset from
 * counters->rng_offset (`offset` is then ignored).  counters == NULL: exactly psvae_train_fwd_bwd(_consistency). */
int psvae_train_fwd_bwd_dc(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                           int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows,
                           float kl_weight, float clf_weight, int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat,
                           float* mu, float* log_sigma, float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                           const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y, float cons_weight,
                           const psvae_step_counters* counters);
/* psvae_adam_step_ex with t = counters->adam_step + 1 and the learning rate *lr (fp64, device) read on the device: for the same t and lr
 * the update is bit-identical (lr / (1 - beta1^t) and sqrt(1 - beta2^t) formed in fp64 with the same expressions, each rounded to fp32
 * once).  Does not advance the counters. */
int psvae_adam_step_dc(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, const double* lr,
                       const psvae_step_counters* counters, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                       int32_t amsgrad, int32_t maximize, void* shadow_bf16, void* stream);
/* rng_offset += 1, adam_step += 1 (one thread); enqueue after the step's last reader of the block */
int psvae_step_counters_advance(psvae_step_counters* counters, void* stream);

/* ---- step-level training options: gradient accumulation and clipping (Lightning's accumulate_grad_batches, gradient_clip_val /
 * gradient_clip_algorithm), device-side so that a CUDA graph replays them unchanged.  Additive to ABI 5. */
/* psvae_train_fwd_bwd_dc plus `accumulate`: accumulate != 0 (with compute_grads != 0) ADDS this call's gradients to what `grads` holds
 * instead of overwriting them: the gradients are computed into grad_scratch (total_numel floats, 16-byte aligned, not `grads`) exactly as
 * the non-accumulating call computes them, then grads[i] += grad_scratch[i] (one fp32 addition per element; padding adds zero).
 * accumulate == 0: exactly psvae_train_fwd_bwd_dc (grad_scratch unused). */
int psvae_train_fwd_bwd_acc(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                            int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows,
                            float kl_weight, float clf_weight, int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat,
                            float* mu, float* log_sigma, float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                            const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y, float cons_weight,
                            const psvae_step_counters* counters, int32_t accumulate, float* grad_scratch);
/* ---- gradient scope (additive to ABI 5).  PSVAE_GRAD_ALL: every parameter, exactly psvae_train_fwd_bwd_acc.  PSVAE_GRAD_CLASSIFIER: the
 * second stage of a two-stage run (frozen VAE, lightning.py freeze_vae): the full forward and every loss term, as the full step computes
 * them, but only the latent classifier's gradients -- no VAE backward.  Only the classifier span of `grads`, [vae_numel, total_numel),
 * is written (cleared, then written; with accumulate != 0: grads[i] += grad_scratch[i] over that span only); every element outside it
 * keeps its value.  workspace >= psvae_workspace_bytes(desc, rows, precision, PSVAE_MODE_TRAIN_CLASSIFIER) (+
 * psvae_consistency_workspace_bytes(cons, rows, PSVAE_MODE_FORWARD) with a consistency term).  A model without a classifier, or an
 * unknown scope, is an argument error. */
#define PSVAE_GRAD_ALL 0
#define PSVAE_GRAD_CLASSIFIER 1
int psvae_train_fwd_bwd_scoped(const psvae_model_desc* desc, const float* params, const void* shadow_bf16, float* grads, const void* x,
                               int32_t x_dtype, const int64_t* y, const float* eps, uint64_t seed, uint64_t offset, int64_t row0, int64_t rows,
                               float kl_weight, float clf_weight, int32_t use_cos_loss, int32_t compute_grads, int32_t precision, float* x_hat,
                               float* mu, float* log_sigma, float* losses, void* workspace, int64_t workspace_bytes, void* stream,
                               const psvae_consistency_desc* cons, const float* cons_params, const int64_t* cons_y, float cons_weight,
                               const psvae_step_counters* counters, int32_t accumulate, float* grad_scratch, int32_t grad_scope);
#define PSVAE_GRAD_NORM_MAX_SPANS 16
#define PSVAE_GRAD_NORM_SCRATCH_BYTES 4096
/* total_norm = || g * grad_scale ||_2 over the n_spans [a, b) spans (host int64 array {a0, b0, a1, b1, ...}) of the flat gradient, and
 * coef = min(fp32(max_norm) / (total_norm + 1e-6f), 1.0f) -- torch.nn.utils.clip_grad_norm_ (norm_type 2).  Both are fp32 device scalars.
 * Squares are summed in fp64 in a fixed order on a fixed grid: bit-identical from run to run.  scratch: PSVAE_GRAD_NORM_SCRATCH_BYTES of
 * caller-allocated device memory, 8-byte aligned, zeroed once before the first call (the kernel leaves it ready for the next).  No host
 * synchronisation: capturable. */
int psvae_grad_norm(const float* g, const int64_t* spans, int32_t n_spans, double grad_scale, double max_norm, float* total_norm, float* coef,
                    void* scratch, int64_t scratch_bytes, void* stream);
#define PSVAE_CLIP_NONE 0
#define PSVAE_CLIP_NORM 1  /* g_eff = g * fp32(grad_scale * *clip_coef)     (clip_coef from psvae_grad_norm; coef = 1 is the unclipped step) */
#define PSVAE_CLIP_VALUE 2 /* g_eff = clamp(g * grad_scale, -clip_value, clip_value)  (torch.nn.utils.clip_grad_value_) */
/* Adam with gradient clipping, applied before weight_decay is added and before maximize negates (where torch clips: before
 * optimizer.step()).  counters == NULL: the host-scalar form (lr, step as psvae_adam_step_ex); counters != NULL: the device form
 * (lr_dev, counters as psvae_adam_step_dc; lr and step ignored).  clip_mode PSVAE_CLIP_NONE is exactly psvae_adam_step_ex / _dc. */
int psvae_adam_step_clip(float* p, const float* g, float* m, float* v, float* vmax, int64_t n, double lr, int64_t step, const double* lr_dev,
                         const psvae_step_counters* counters, double beta1, double beta2, double eps, double weight_decay, double grad_scale,
                         int32_t amsgrad, int32_t maximize, int32_t clip_mode, const float* clip_coef, double clip_value, void* shadow_bf16,
                         void* stream);
/* rng_offset += rng_delta, adam_step += step_delta (one thread): a micro-batch that does not step the optimiser advances the offset only */
int psvae_step_counters_advance_by(psvae_step_counters* counters, uint64_t rng_delta, int64_t step_delta, void* stream);

/* ---- conditional_synthesis Langevin loop (ps_vae/inference.py:72-103) --------------------------- */
/* z_io [rows][L]: z0 == NULL-initialised by the caller or (init_from_philox != 0) drawn in-kernel with
 * offset `offset0`; step s uses offset `offset0 + 1 + s` unless `noise` ([num_steps][rows][L]) is given.
 * targets[h] = class index of head h, or -1 to leave head h out (a dict target naming only some labels).
 * history (optional) receives z after every step: [num_steps][rows][L].  stats (optional) [num_steps][2] =
 * mean log p(z|y), mean p(y|z) as printed by the reference's progress bar (inference.py:103).
 * The variant of analysis/sample_gender_transformation.py:61-99 uses the same loop with three differences, all arguments here:
 * prior_weight scales the log p(z) term (PRIOR_WEIGHT; 1 for inference.py), threshold > 0 stops a sample after the update of the
 * first step whose p(y|z) exceeded it (THRESHOLD; 0 = never), and the start latent is the caller's (z_io = the encoder mean of a real
 * embedding, init_from_philox = 0).  stop_step (optional, int32 [rows]) = that step, num_steps if the sample never stopped;
 * last_prob (optional, [rows]) = p(y|z) of the sample's last evaluated step. */
int psvae_langevin(const psvae_model_desc* desc, const float* params, float* z_io, int64_t rows,
                   const int32_t* targets_host, float step_size, int32_t num_steps, float noise_weight,
                   uint64_t seed, uint64_t offset0, int64_t row0, int32_t init_from_philox, const float* noise,
                   float* history, float* stats, float prior_weight, float threshold, int32_t* stop_step, float* last_prob,
                   void* stream);

/* The same loop with a classifier target per row (additive to ABI 5).  Exactly one of:
 *  - row_targets: device int32 [n_heads][rows], row r's class for head h at [h][r], -1 to leave head h out for that row.  A row with a
 *    target outside [-1, classes) or naming no head gets NaN in z_io, its history rows and last_prob; the other rows are unaffected.
 *  - a target mix of n_mix (1..PSVAE_MAX_TARGET_MIX) entries: mix_targets_host [n_mix][PSVAE_MAX_CLF_HEADS] (class or -1 per head, each
 *    entry naming at least one head) and n_mix - 1 non-decreasing mix_thresholds_host.  Row r takes word row0 + r of the uint32 Philox
 *    stream at offset offset0 + num_steps + 1 (psvae_philox_uint32 with first_elem = row0), u, and picks the first entry k < n_mix - 1 with
 *    u < thresholds[k], else the last; entry k is drawn with probability (thresholds[k] - thresholds[k - 1]) / 2^32.  The drawn targets go to
 *    row_targets_out (required), device int32 [n_heads][rows].  The draw depends on the global row only, so a sharded run draws what one
 *    call over all rows draws.
 * Every row computes exactly what psvae_langevin computes for it with its own target as the shared one (same seed, offset0, row0).
 * Argument errors (no classifier, both or neither target form, n_mix > PSVAE_MAX_TARGET_MIX, a bad mix entry, decreasing thresholds, a mix
 * without row_targets_out) are reported before the device is looked at. */
#define PSVAE_MAX_TARGET_MIX 64
int psvae_langevin_rows(const psvae_model_desc* desc, const float* params, float* z_io, int64_t rows, const int32_t* row_targets,
                        int32_t n_mix, const int32_t* mix_targets_host, const uint32_t* mix_thresholds_host, int32_t* row_targets_out,
                        float step_size, int32_t num_steps, float noise_weight, uint64_t seed, uint64_t offset0, int64_t row0,
                        int32_t init_from_philox, const float* noise, float* history, float* stats, float prior_weight, float threshold,
                        int32_t* stop_step, float* last_prob, void* stream);

/* ---- cosine top-k search between two embedding sets (additive to ABI 5) ----------------------------
 * For every query row i of q [nq][dim] the k keys j of keys [nk][dim] with the highest (default) or lowest (PSVAE_TOPK_SMALLEST) cosine
 * similarity sim = q.x / (max(|q|, 1e-8) max(|x|, 1e-8)) (torch's F.cosine_similarity: a zero row scores 0).  Each set is fp32
 * (PSVAE_X_F32) or bf16 (PSVAE_X_BF16), contiguous, 1 <= k <= 16, dim a multiple of 8 and <= 512; q and keys may be the same array.
 * Candidates are selected from bf16-rounded unit vectors (fp32 accumulation on the tensor cores), the best 2k per row are re-scored in
 * fp32 from the inputs, and the best k of those are returned: out_sim fp32 [nq][k], out_idx int64 [nq][k] (global: k_row0 + j).  Equal
 * similarities go to the lower key index; a NaN similarity is never chosen; a slot without a candidate holds -1 / NaN.  With
 * PSVAE_TOPK_EXCLUDE_SELF the pairs q_row0 + i == k_row0 + j are skipped (k <= nk - 1).  The result is bit-identical from run to run, for
 * any sharding of the queries (q_row0) and any split of the key range (option "topk_key_splits").
 * workspace: psvae_cosine_topk_workspace_bytes(nq, nk, dim, k) bytes, 256-byte aligned (it depends on the option "topk_key_splits").
 * Argument errors are reported before the device is looked at. */
#define PSVAE_TOPK_SMALLEST 1
#define PSVAE_TOPK_EXCLUDE_SELF 2
int64_t psvae_cosine_topk_workspace_bytes(int64_t nq, int64_t nk, int32_t dim, int32_t k);
int psvae_cosine_topk(const void* q, int32_t q_dtype, int64_t nq, int64_t q_row0, const void* keys, int32_t k_dtype, int64_t nk,
                      int64_t k_row0, int32_t dim, int32_t k, int32_t flags, float* out_sim, int64_t* out_idx, void* workspace,
                      int64_t workspace_bytes, void* stream);

/* ---- building block exposed for tests and profiling: C = A[M,K] * B[N,K]^T (+bias) ------------- */
/* a_mn / b_mn: operand stored MN-major (A as [K][M], B as [K][N]).  bf16 in, fp32 out, tcgen05. */
int psvae_gemm_bf16(const void* a_bf16, const void* b_bf16, const float* bias, float* c, int64_t m, int32_t n,
                    int64_t k, int32_t a_mn, int32_t b_mn, int32_t relu, int32_t split_k, void* workspace,
                    int64_t workspace_bytes, void* stream);
/* profiling probe: the two hot epilogue forms of the train step on free-standing operands.
 * form 0: out = relu(A[m,k] W[n,k]^T + bias) in bf16 (+ 1-bit ReLU mask [n/32][m] when mask != NULL);
 * form 1: out = (A[m,k] W[k,n]) .* mask in bf16 (+ column sums accumulated into colsum[n] when != NULL).
 * form 2: wgrad, out[n][k] (fp32) += A[m,n]^T W[m,k] (contraction over the m batch rows, split-K with TMA reduce-add).
 * out == NULL skips the store (forms 0, 1). */
int psvae_gemm_probe(const void* a_bf16, const void* w_bf16, const float* bias, void* out_bf16, uint32_t* mask,
                     float* colsum, int64_t m, int32_t n, int64_t k, int32_t form, void* stream);
/* same contract on the CUDA cores in fp32 (the parity engine) */
int psvae_gemm_fp32(const float* a, const float* b, const float* bias, float* c, int64_t m, int32_t n, int64_t k,
                    int32_t a_mn, int32_t b_mn, int32_t relu, void* stream);

/* number of kernels this library launched since load (bench.py's "gpu_launches") */
int64_t psvae_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PSVAE_B200_H_ */
