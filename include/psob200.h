/*
 * psob200.h -- C ABI of the B200-native (sm_100a) PSO training-step hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8 row b4).  The reference
 * (yaramohamadi/Pairwise_Sample_Optimization) is pure Python/PyTorch and has no FFI
 * of its own; each entry point below names the reference code it replaces
 * (paths relative to the reference root):
 *
 *   TS = human_preference_tuning/pso_pytorch/diffusers_patch/turbo_inference_with_logprob.py
 *   DS = human_preference_tuning/pso_pytorch/diffusers_patch/distilled_inference_with_logprob.py
 *   TP = human_preference_tuning/pso_pytorch/diffusers_patch/sdxl_turbo_with_logprob.py
 *   DP = human_preference_tuning/pso_pytorch/diffusers_patch/sdxl_dmd_with_logprob.py
 *   T  = human_preference_tuning/train_online_pso_sdxl_turbo.py
 *   D  = human_preference_tuning/train_online_pso_sdxl_dmd2.py
 *   P  = personalization/train_pso_sdxl_turbo_dreambooth.py
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer on the
 *     current CUDA device; tensors are dense row-major ("NCHW contiguous"), a sample
 *     is N = C*H*W consecutive elements;
 *   - `stream` is a cudaStream_t passed as void*; work is stream-ordered;
 *   - functions never allocate, never synchronise, never throw; scratch memory is a
 *     caller-provided workspace;
 *   - return 0 on success, a negative PSOB200_ERR_* otherwise (psob200_strerror());
 *   - data-dependent failures that only the device can see (a timestep that is not in
 *     the schedule: TS:63 raises IndexError there) set bits in `*status` (device int,
 *     may be NULL) and poison the affected outputs with NaN.
 */
#ifndef PSOB200_H
#define PSOB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PSOB200_ABI_VERSION 2

#if defined(__GNUC__)
#define PSOB200_API __attribute__((visibility("default")))
#else
#define PSOB200_API
#endif

/* element types */
enum { PSOB200_F32 = 0, PSOB200_BF16 = 1, PSOB200_F16 = 2 };
/* timestep element types */
enum { PSOB200_TS_I64 = 0, PSOB200_TS_F32 = 1, PSOB200_TS_I32 = 2 };
/* scheduler families */
enum { PSOB200_SCHED_TURBO = 0, PSOB200_SCHED_DMD = 1, PSOB200_SCHED_AFFINE = 2 };
/* DreamBooth loss types (P:1924-1929) */
enum { PSOB200_DB_PSO = 0, PSOB200_DB_PSO_DB = 1 };

/* error codes */
enum {
  PSOB200_OK = 0,
  PSOB200_ERR_INVALID_ARG = -1,
  PSOB200_ERR_DTYPE = -2,
  PSOB200_ERR_ALIGNMENT = -3,
  PSOB200_ERR_LAUNCH = -4,
  PSOB200_ERR_SHAPE = -5,
  PSOB200_ERR_WORKSPACE = -6,
  PSOB200_ERR_DRIVER = -7
};

/* bits set in *status by kernels */
#define PSOB200_STATUS_TIMESTEP_NOT_IN_SCHEDULE 1
#define PSOB200_STATUS_NONFINITE_COEFFICIENT 2

/*
 * How per-sample step coefficients are obtained.  Both reference step functions are the
 * affine Gaussian  x' ~ N(k*x + a*eps, s^2)  (SURVEY.md App. A.2):
 *   TURBO  (TS:61-92):  idx = first i with sched_timesteps[i] == t  (TS:63);
 *                       sigma = table[idx], sigma_to = table[idx+1]   (TS:77-78)
 *                       k = 1, a = sigma_down - sigma, s = sigma_up    (TS:79-92)
 *   DMD    (DS:36-42,102-112): abar_t = table[t], abar_p = table[t_prev] (negative
 *                       indices wrap like torch indexing);
 *                       k = sqrt(abar_p/abar_t), a = -sqrt(abar_p (1-abar_t)/abar_t),
 *                       s = sqrt(1-abar_p)
 *   AFFINE: k, a, s given directly as device float arrays of length B.
 */
typedef struct psob200_schedule {
  int32_t kind;                 /* PSOB200_SCHED_*                                         */
  int32_t n_table;              /* TURBO: number of timesteps (table has n_table+1 sigmas);
                                   DMD: length of alphas_cumprod                           */
  const float* sched_timesteps; /* TURBO: device float[n_table] (diffusers keeps fp32)     */
  const float* table;           /* TURBO: sigmas; DMD: alphas_cumprod (device float)       */
  int32_t ts_dtype;             /* PSOB200_TS_* of the per-sample timestep arrays          */
  int32_t reserved;
} psob200_schedule;

PSOB200_API int psob200_abi_version(void);
PSOB200_API const char* psob200_strerror(int rc);
/* What the CUDA runtime reported for this thread's most recent PSOB200_ERR_LAUNCH ("" if none). */
PSOB200_API const char* psob200_last_error_detail(void);
/* Number of SMs / compute capability the library was queried with; -1 if no device. */
PSOB200_API int psob200_device_sm_count(void);
/* Kernels this library has launched successfully in this process (monotonic; for launch accounting). */
PSOB200_API long long psob200_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Workspace for the pair-loss kernels: >= psob200_pair_loss_workspace_bytes(B) bytes,
 * 16-byte aligned, ZERO-INITIALISED once by the caller; the kernels leave it zeroed.
 * One workspace must not be shared by launches that may run concurrently.
 */
PSOB200_API size_t psob200_pair_loss_workspace_bytes(int64_t B);

/*
 * Fused online-PSO loss + gradient: replaces the four step-with-logprob calls, the
 * inline loss and its autograd backward of one training micro-step
 * (T:810-850 + T:857, D:812-854 + D:859) with ONE kernel launch:
 *
 *   logp_{m,k}[b] = mean_CHW[-(next_k - mu_{m,k})^2/(2 s^2) - log s - 0.5 log 2pi],
 *                   m in {policy, ref}, k in {0,1}                        (TS:108-114, DS:129-135)
 *   ratio_k = clamp(exp(logp_pol,k - logp_ref,k), 1-eps, 1+eps)           (T:844-845)
 *   loss    = loss_scale * mean_b[-log sigmoid(beta*(h0*log ratio_0 + h1*log ratio_1))]   (T:847-850)
 *   grad_k  = d loss / d pred_k   (dtype of pred)                         (T:857 autograd)
 *
 * pred_k/ref_k: policy / frozen-reference UNet outputs, [B,N] of `pred_dtype`.
 * sample_k/next_k: current latent and stored next latent, [B,N] of `latent_dtype`.
 * ts_k (and ts_prev_k for DMD): per-sample timesteps [B]; for AFFINE, coef_k points to
 * float[3*B] = k[B], a[B], s[B] and ts_* are ignored.
 * human_prefer: float[B*2] rows (h0,h1) as produced by T:401-416 / D:420-434.
 * Outputs: grad_k [B,N] pred_dtype; loss float[1]; stats float[B*8] (may be NULL) =
 *   (logp_pol0, logp_ref0, logp_pol1, logp_ref1, delta0, delta1, z, pair_loss) per pair.
 * tune_threads: 0 = library heuristics (the tensor-memory kernel when N is a multiple of 8 and everything is 16-byte
 *   aligned, else the general kernel); 1 = the TMA-ring kernel (kept for A/B timing); >= 32 = the general kernel with
 *   that many threads.  tune_cluster: CTAs per pair (1, 2, 4, 8), 0 = heuristics.
 */
typedef struct psob200_online_pso_args {
  const void* pred[2];
  const void* ref[2];
  const void* sample[2];
  const void* next[2];
  const void* ts[2];
  const void* ts_prev[2];
  const float* coef[2];
  const float* human_prefer;
  /* element stride between consecutive samples of each input (0 = dense, i.e. N); lets the
     trainers' views `latents[:, j]` of a [B,T,C,H,W] tensor be consumed without a copy */
  int64_t stride_pred[2];
  int64_t stride_ref[2];
  int64_t stride_sample[2];
  int64_t stride_next[2];
  void* grad[2];
  float* loss;
  float* stats;
  int32_t* status;
  void* workspace;
  size_t workspace_bytes;
  int64_t B;
  int64_t N;
  int32_t pred_dtype;
  int32_t latent_dtype;
  float beta;
  float eps;
  float loss_scale;
  int32_t tune_threads;
  int32_t tune_cluster;
  int32_t reserved;
} psob200_online_pso_args;

PSOB200_API int psob200_online_pso_loss_grad(const psob200_schedule* sched, const psob200_online_pso_args* args,
                                 void* stream);

/*
 * Dynamic loss scaling on the device: the state of torch's GradScaler, which accelerate wraps around every step of the
 * fp16 recipes (mixed_precision="fp16", T:126; scaler.scale(loss).backward() T:857, unscale_ + clip_grad_norm_ T:859,
 * scaler.step + scaler.update() T:860).  scale (S) and growth_tracker are DEVICE scalars; nothing reads them on the host.
 *   loss entry points (*_loss_grad_scaled): the per-pair gradient multiplier is multiplied by *scale before the
 *     elementwise pass, so grad = S * d loss / d pred is rounded to the prediction dtype once, already scaled; loss and
 *     stats stay unscaled.  Only `scale` is read.
 *   optimizer entry points (psob200_flat_adamw*_step_scaled): the unscale factor is (float)(1 / (double)*scale) times
 *     grad_scale (fp32), used where grad_scale is used without a scaler; the norm is always computed; the last block
 *     updates S and growth_tracker as torch._amp_update_scale_ does, with found_inf = "the norm is not finite":
 *       found_inf:  S = (float)(S * backoff_factor), tracker = 0
 *       else:       t = tracker + 1; t == growth_interval ? (S' = (float)(S * growth_factor), S = S' if finite, tracker = 0)
 *                                                         : tracker = t          (products in double)
 *     growth_factor > 1, 0 < backoff_factor < 1, growth_interval > 0, else PSOB200_ERR_INVALID_ARG.
 */
typedef struct psob200_loss_scaler {
  float* scale;            /* device float[1] */
  int32_t* growth_tracker; /* device int32[1]; unused by the loss entry points (may be NULL there) */
  double growth_factor;
  double backoff_factor;
  int32_t growth_interval;
  int32_t reserved;
} psob200_loss_scaler;

/* psob200_online_pso_loss_grad with the gradient scaled by the device loss scale (T:857 under GradScaler). */
PSOB200_API int psob200_online_pso_loss_grad_scaled(const psob200_schedule* sched, const psob200_online_pso_args* args,
                                                    const psob200_loss_scaler* scaler, void* stream);

/*
 * Fused DreamBooth-PSO loss + gradient: replaces P:1847-1865 (EDM-style epsilon
 * preconditioning, non-EDM scheduler) + P:1881-1935 + the autograd backward (P:1953).
 * model_pred/ref_pred: raw UNet outputs [2b,N] (`pred_dtype`), rows [0,b) = win images,
 * [b,2b) = lose images; ref_pred is ignored (may be NULL) for PSOB200_DB_PSO_DB.
 * noisy/target: noisy_model_input and model_input [2b,N] (`latent_dtype`);
 * sigmas: float[2b].
 *   x0_hat = -sigma*pred + noisy ; L_i = mean_CHW(sigma^-2 (x0_hat - target)^2)
 *   logits = (Lref_w - nu Lref_l) - (L_w - nu L_l)        (pso)   | -(L_w - nu L_l)  (pso_db)
 *   loss   = mean -logsigmoid(beta logits)                (pso)   | mean relu(1 - beta logits)
 *            + lambda * mean(L_l)   if lambda > 0
 * Outputs: grad [2b,N]; loss float[1]; stats float[b*8] (may be NULL) =
 *   (L_w, L_l, Lref_w, Lref_l, logits, pair_loss, 0, 0).
 */
typedef struct psob200_dreambooth_args {
  const void* model_pred;
  const void* ref_pred;
  const void* noisy;
  const void* target;
  const float* sigmas;
  void* grad;
  float* loss;
  float* stats;
  int32_t* status;
  void* workspace;
  size_t workspace_bytes;
  int64_t b; /* pairs; tensors have 2*b rows */
  int64_t N;
  int32_t pred_dtype;
  int32_t latent_dtype;
  int32_t loss_type;
  float beta_pso;
  float neg_defactor;
  float prior_loss_weight;
  float loss_scale;
  int32_t tune_threads;
  int32_t tune_cluster;
  int32_t reserved;
} psob200_dreambooth_args;

PSOB200_API int psob200_dreambooth_pso_loss_grad(const psob200_dreambooth_args* args, void* stream);
/* psob200_dreambooth_pso_loss_grad with the gradient scaled by the device loss scale (P:1953 under GradScaler). */
PSOB200_API int psob200_dreambooth_pso_loss_grad_scaled(const psob200_dreambooth_args* args,
                                                        const psob200_loss_scaler* scaler, void* stream);

/* ------------------------------------------------------------------------------------
 * One scheduler update + Gaussian log-prob: the body of turbo_step_with_logprob
 * (TS:24-116) and distilled_step_with_logprob (DS:45-137).
 *
 * Scoring mode (prev_sample != NULL, noise == NULL): log_prob[b] of the given
 * prev_sample (TS:100-114, DS:129-135).
 * Sampling mode (prev_sample == NULL, noise != NULL): prev_out = mu + s*noise
 * (TS:94-99, DS:121-126) and its log_prob.  noise is [noise_rows,N] with noise_rows == B
 * (turbo) or 1 (DMD: one draw shared by the batch, DS:123-124), of `out_dtype`.
 * prev_out [B,N] `out_dtype` (model_output dtype for turbo TS:116, sample dtype for DMD
 * DS:137).  scaled_next_out (may be NULL) = prev_out_fp32 / sqrt(sigma_next^2+1), the
 * next UNet input of the turbo sampler (TP:120-121), `out_dtype`.
 * Throughput mode (prev_sample == NULL, noise == NULL, use_philox != 0): the N(0,1) draws come from a counter-based
 * generator inside the kernel (Philox4x32-10 + Box-Muller; four draws per counter (q, philox_offset), q = index of the
 * 4-element group inside the [noise_rows, N] noise tensor, key = philox_seed; values rounded through `out_dtype` as
 * randn(dtype=...) would), so no noise tensor is written or read.  torch's own generator stream is not reproduced: pass
 * `noise` when the draws must be the caller's.  Advance philox_offset by 1 per call.
 */
typedef struct psob200_step_args {
  const void* model_output; /* [B,N] pred_dtype   */
  const void* sample;       /* [B,N] latent_dtype */
  const void* prev_sample;  /* [B,N] latent_dtype, scoring mode */
  const void* noise;        /* [noise_rows,N] out_dtype, sampling mode */
  const void* ts;           /* [B] or [1] (ts_rows) */
  const void* ts_prev;      /* DMD only */
  const float* coef;        /* AFFINE only: k[B], a[B], s[B] */
  void* prev_out;           /* sampling mode */
  void* scaled_next_out;    /* sampling mode, optional */
  float* log_prob;          /* [B] */
  int32_t* status;
  int64_t B;
  int64_t N;
  int64_t noise_rows;
  int64_t ts_rows; /* B, or 1 to broadcast one timestep over the batch (TP:139) */
  int64_t stride_model_output; /* element strides between samples, 0 = dense */
  int64_t stride_sample;
  int64_t stride_prev_sample;
  int32_t pred_dtype;
  int32_t latent_dtype;
  int32_t out_dtype;
  int32_t tune_threads;
  int32_t tune_cluster;
  int32_t use_philox;
  uint64_t philox_seed;
  uint64_t philox_offset;
} psob200_step_args;

PSOB200_API int psob200_step_logprob(const psob200_schedule* sched, const psob200_step_args* args, void* stream);

/*
 * Backward of the scoring-mode log-prob into model_output (autograd of TS:108-114 /
 * DS:129-135 as run by T:857):  grad[b,:] = grad_log_prob[b] * a/(s^2 N) * (prev - mu).
 */
typedef struct psob200_step_bwd_args {
  const void* model_output;
  const void* sample;
  const void* prev_sample;
  const void* ts;
  const void* ts_prev;
  const float* coef;
  const float* grad_log_prob; /* [B] */
  void* grad_model_output;    /* [B,N] pred_dtype */
  int32_t* status;
  int64_t B;
  int64_t N;
  int64_t ts_rows;
  int64_t stride_model_output; /* element strides between samples, 0 = dense */
  int64_t stride_sample;
  int64_t stride_prev_sample;
  int32_t pred_dtype;
  int32_t latent_dtype;
  int32_t reserved0;
  int32_t reserved1;
} psob200_step_bwd_args;

PSOB200_API int psob200_step_logprob_backward(const psob200_schedule* sched, const psob200_step_bwd_args* args,
                                  void* stream);

/*
 * x0 = (sample - sqrt(1-abar_t) * model_output) / sqrt(abar_t)   (DS:36-42; the last DMD
 * sampler step, DP:158-162).  Output dtype = out_dtype.
 */
PSOB200_API int psob200_dmd_x0_from_noise(const float* alphas_cumprod, int32_t n_table, const void* model_output,
                              const void* sample, const void* ts, int32_t ts_dtype, int64_t ts_rows,
                              void* x0_out, int64_t B, int64_t N, int32_t pred_dtype,
                              int32_t latent_dtype, int32_t out_dtype, int32_t* status, void* stream);

/*
 * out = in * scale[0 or b]  -- the sampler's elementwise glue:  latents*init_noise_sigma
 * (TP:99, DP:49) and latents/sqrt(sigma^2+1) (TP:121, P:1796).  scale is a HOST float.
 */
PSOB200_API int psob200_scale(const void* in, void* out, int64_t count, float scale, int32_t in_dtype,
                  int32_t out_dtype, void* stream);

/*
 * data[i] *= scale_dev[0] for a DEVICE-resident scalar; returns immediately on the device
 * when the scalar is exactly 1.0f.  Used to apply autograd's upstream gradient of the loss
 * to gradients that the fused kernels already produced (T:857: accelerate hands
 * loss/gradient_accumulation_steps to backward()).
 */
PSOB200_API int psob200_scale_inplace_by_device_scalar(void* data, int64_t count, int32_t dtype,
                                                       const float* scale_dev, void* stream);

/* ------------------------------------------------------------------------------------
 * LoRA projection GEMMs on the tcgen05 tensor cores (TMA-fed, accumulators in tensor memory).
 *
 *   D[M,N] = alpha * ( A1[M,K1] * B1[N,K1]^T  +  A2[M,K2] * B2[N,K2]^T ) + bias[N]
 *
 * replaces the three library GEMMs + scale + add that peft==0.11.1 `lora.Linear.forward` issues per
 * wrapped projection (installed by `unet.add_adapter`, T:338-345, D:361-368, P:1319-1326) and their
 * autograd backward (T:857).  All operands are 16-bit (`ab_dtype` = PSOB200_BF16 or PSOB200_F16),
 * row-major with the reduction dimension contiguous ("K-major"), leading dimensions in elements and a
 * multiple of 8, base pointers 16-byte aligned; M, N, K1, K2 are otherwise arbitrary (tails are
 * zero-filled by the TMA unit).  K2 == 0 disables the second segment.
 *
 * a_reduction_major != 0: A1 is given as [K1, M] row-major (the output-row index contiguous), i.e. the
 *   product A1^T-as-stored: used for the weight-gradient reductions dA = U^T X, dB = dY^T T where the
 *   activations are only available token-major.  Requires K2 == 0.
 * b_reduction_major != 0: B1 (and B2) are given as [K, N] row-major (the output-column index contiguous):
 *   lets the backward dX = dY W + U A and U = s dY B consume W [N_out,K_in], lora_A [r,K] and lora_B [N,r]
 *   in the layout the reference stores them, with no transposed copies.
 * d / dt: row-major output [M,N] (leading dimension ldd) and / or its transpose [N,M] (lddt);
 *   element type d_dtype.  accumulate != 0: fp32 outputs are accumulated with atomic adds (gradient
 *   accumulation into .grad) and the reduction may be split over CTAs (split_k: 0 = heuristics).
 * bias: optional [N] of bias_dtype.  tune_bn: tile width (multiple of 16, <= 256), 0 = heuristics.
 */
typedef struct psob200_gemm_args {
  const void* a1;
  const void* b1;
  const void* a2;
  const void* b2;
  const void* bias;
  void* d;
  void* dt;
  int64_t lda1, ldb1, lda2, ldb2, ldd, lddt;
  int64_t M, N, K1, K2;
  float alpha;
  int32_t ab_dtype;
  int32_t d_dtype;
  int32_t bias_dtype;
  int32_t a_reduction_major;
  int32_t b_reduction_major;
  int32_t accumulate;
  int32_t split_k;
  int32_t tune_bn;
  int32_t pdl;  /* programmatic dependent launch: 1 = let the next launch on the stream start early (this grid signals
                   at its start); 2 = this launch may start before the previous one has finished and waits for it only
                   before reading the second K segment (a2); 6 = ... waits before its first load; 8 = independent of the
                   previous launch, may overlap it entirely (waits for it only before exiting).  0 = plain launch */
  int32_t diag; /* timing experiments only (results are then wrong): bit 0 skip the MMAs, bit 1 skip the stores,
                   bits 2-3 skip the operand loads, bit 18 (0x40000) record the per-CTA timeline; A/B switches with
                   correct results: bit 16 force / bit 17 forbid the CTA-pair kernel, bit 19 (0x80000) no interleaving of a
                   pair's first two waiting tiles.  PSOB200_GEMM_DIAG in the environment is OR-ed into every launch */
} psob200_gemm_args;

PSOB200_API int psob200_lora_gemm(const psob200_gemm_args* args, void* stream);

/* Diagnostics only (tools/diag_timeline.py): after a CTA-pair launch with diag bit 0x40000, copies that launch's per-CTA time
 * stamps to `host_out` (synchronous): [cta][slot 0..7][globaltimer ns, SM cycle counter], 512 CTAs.  Slots: 0 entry, 1 prologue
 * done, 2 first operands landed (leader CTA), 3 / 5 first / last accumulator complete, 4 / 6 first / last tile drained, 7 exit.
 * Returns the number of values written (8192) or a negative error code. */
PSOB200_API int psob200_lora_gemm_timeline(unsigned long long* host_out, long long capacity);

/*
 * The LoRA-wrapped projection as the reference's stack runs it (peft==0.11.1 lora.Linear, created by
 * unet.add_adapter at T:338-345 / D:361-368 / P:1319-1326 on to_q, to_k, to_v, to_out.0), forward and backward,
 * each a short sequence of psob200_lora_gemm launches on `stream`:
 *
 *   forward   t  = scaling * x A^T               [M,r]  (skinny pass; also tt = t^T when tt != NULL)
 *             y  = x W^T + bias + t B^T          [M,N]  (ONE pass over W: second K segment = the adapter)
 *             adapters_enabled == 0 (disable_adapters(), T:790): y = x W^T + bias only
 *   backward  u  = scaling * dy B                [M,r]  (+ ut = u^T)
 *             dx = dy W + u A                    [M,K]  (skipped when dx == NULL)
 *             dA += u^T x  [r,K]   dB += dy^T t  [N,r]  (fp32, accumulated: gradient accumulation T:232)
 *
 * x [M,K], w [N,K], lora_a [r,K], lora_b [N,r], dy [M,N] are 16-bit (`dtype`), in the layouts the reference keeps
 * them (nn.Linear weight [out,in]); no transposed copies are needed.  Leading dimensions are in elements,
 * multiples of 8 (so lora_b, t, u are stored with ld >= r rounded up to 8).  t/tt (forward) and u/ut (backward)
 * are caller-provided scratch; tt must be kept for the backward.  r <= 256.
 * forward_phases / backward_phases: 0 = every launch of the sequence; else a mask of the launches to issue, so that a
 * caller can put them on different streams or bracket each with its own events (outputs of the omitted launches must be
 * in place from an earlier call): PSOB200_FWD_DOWN (t), PSOB200_FWD_MAIN (y); PSOB200_BWD_U (u, ut), PSOB200_BWD_DX,
 * PSOB200_BWD_DA, PSOB200_BWD_DB.  Nothing downstream of a layer waits for dA / dB, hence PSOB200_BWD_WEIGHT_GRAD.
 */
#define PSOB200_FWD_DOWN 1
#define PSOB200_FWD_MAIN 2
#define PSOB200_BWD_U 1
#define PSOB200_BWD_DX 2
#define PSOB200_BWD_DA 4
#define PSOB200_BWD_DB 8
#define PSOB200_BWD_INPUT_GRAD (PSOB200_BWD_U | PSOB200_BWD_DX)
#define PSOB200_BWD_WEIGHT_GRAD (PSOB200_BWD_DA | PSOB200_BWD_DB)
typedef struct psob200_lora_linear_args {
  const void* x;
  const void* w;
  const void* bias; /* [N] of bias_dtype, may be NULL */
  const void* lora_a;
  const void* lora_b;
  void* y;
  void* t;
  void* tt;
  const void* dy;
  void* dx;
  void* u;
  void* ut;
  float* d_lora_a; /* [r, ld_da] fp32, accumulated into; may be NULL */
  float* d_lora_b; /* [N, ld_db] fp32, accumulated into; may be NULL */
  int64_t ldx, ldw, lda, ldb, ldy, ldt, ldtt, lddy, lddx, ldu, ldut, ld_da, ld_db;
  int64_t M, K, N, r;
  float scaling;
  int32_t dtype;
  int32_t bias_dtype;
  int32_t adapters_enabled;
  int32_t backward_phases;
  int32_t forward_phases;
  /* Optional zeroed int32 workspace (>= ceil(M / 128) + 1 entries, left zeroed): when given, and all phases of a direction
   * are requested, t (u) becomes a problem of the SAME launch as y (dx) -- its tiles release a flag per row block and the
   * adapter segment of the main problem waits for it -- so the forward is ONE launch and the backward two (input
   * gradients; weight gradients).  One workspace per stream. */
  int32_t* flags;
  int64_t flags_len;
} psob200_lora_linear_args;

PSOB200_API int psob200_lora_linear_forward(const psob200_lora_linear_args* args, void* stream);
PSOB200_API int psob200_lora_linear_backward(const psob200_lora_linear_args* args, void* stream);

/*
 * G LoRA-wrapped projections that share their input, STACKED (attention to_q / to_k / to_v, cross-attention to_k / to_v;
 * G = 1 is psob200_lora_linear_*): the frozen weights are one matrix w [G N, K], the adapters lora_a [G r, K] and
 * lora_b [G N, r] (projection g owns rows [g r, (g+1) r) resp. [g N, (g+1) N)), the output is y [M, G N] whose column
 * group g is projection g (the reference runs G separate peft lora.Linear modules: attn.to_q / to_k / to_v in diffusers
 * AttnProcessor2_0, wrapped at T:338-345).  Launches on `stream`:
 *
 *   forward  (1 launch with `flags`, else 2)   t = scaling * x lora_a^T  [M, G r]  (+ tt = t^T);   y = x w^T + t_g B_g^T
 *   backward (2 launches with `flags`)         u_g = scaling * dy_g B_g  (+ ut);   dx = sum_g dy_g W_g + u lora_a
 *                                              dA += u^T x  [G r, K];   dB_g += dy_g^T t_g  [N, r]   (fp32, accumulated)
 *
 * With `flags` the tiles of the main problem SPIN until the tiles of t (u) of the same launch have published their rows: every
 * CTA of the launch must be able to become resident, so keep at most one such launch in flight per device (issue the
 * LoRA-enabled passes of a device from ONE stream; launches without adapters, and the weight-gradient launch, never wait).
 * dy[g] are G separate [M, N] gradients (their own row pitches lddy[g]); dx may be NULL (cross-attention k / v: the prompt
 * embeddings need no gradient).  G > 1 needs r_stride % 8 == 0 (see r_stride).  bias only for G = 1.  Phases and scratch as psob200_lora_linear_args.
 * The BACKWARD takes at most PSOB200_MAX_GROUP projections (dy[] pointers); the FORWARD any G with G N < 2^31: the k / v
 * projections of EVERY cross-attention layer read the same prompt embeddings (TP:136, T:775-805 pass one encoder_hidden_states to
 * all 70 blocks), so one forward launch can produce all of them (lora.CrossKVBank), the backward staying per layer.
 */
#define PSOB200_MAX_GROUP 3
typedef struct psob200_lora_group_args {
  const void* x;
  const void* w;
  const void* bias;
  const void* lora_a;
  const void* lora_b;
  void* y;
  void* t;
  void* tt;
  const void* dy[PSOB200_MAX_GROUP];
  void* dx;
  void* u;
  void* ut;
  float* d_lora_a;
  float* d_lora_b;
  int32_t* flags;
  int64_t flags_len;
  int64_t ldx, ldw, lda, ldb, ldy, ldt, ldtt, lddy[PSOB200_MAX_GROUP], lddx, ldu, ldut, ld_da, ld_db;
  int64_t M, K, N, r;
  int32_t G;
  float scaling;
  int32_t dtype;
  int32_t bias_dtype;
  int32_t adapters_enabled;
  int32_t forward_phases;
  int32_t backward_phases;
  /* bit 0: launch every kernel of the call with programmatic stream serialization; its TMA producer then executes
   * griddepcontrol.wait before its first load, so that the launch latency and the prologue (barriers, tensor-memory
   * allocation, tensor-map fetch) overlap the tail of WHATEVER kernel precedes it on the stream.  Safe for any predecessor:
   * nothing is read or written before the wait has returned.
   * bit 1: DETERMINISTIC weight gradients: the dA / dB reductions are not split over CTAs, so every element of the fp32
   * gradient receives exactly one accumulation per launch (launches on a stream are ordered): bit-reproducible adapter
   * gradients at the price of a less parallel launch (10-40 tiles instead of one wave of split tiles). */
  int32_t launch_flags;
  /* Stride of the G column groups inside the stacked t / u (and of the row groups inside lora_a, tt, ut); 0 = r.  A rank that is
   * not a multiple of 8 is stacked with r_stride = r rounded up to 8: lora_a is then [G r_stride, K] with ZERO rows behind each
   * projection's r rows, t / u / tt / ut are G r_stride wide / tall; lora_b stays [G N, r] and the gradients d_lora_a
   * [G r, K] / d_lora_b [G N, r] stay packed. */
  int64_t r_stride;
} psob200_lora_group_args;

PSOB200_API int psob200_lora_group_forward(const psob200_lora_group_args* args, void* stream);
PSOB200_API int psob200_lora_group_backward(const psob200_lora_group_args* args, void* stream);

/*
 * Optimizer boundary over the FLAT LoRA buffers (one fp32 buffer each for parameters, gradients and the two Adam
 * moments; every adapter matrix is a slice): global-norm clipping (accelerate clip_grad_norm_, T:859), AdamW
 * (T:428-448: lr, betas, weight_decay, eps) with torch.optim.AdamW's update rule, zero_grad, and the refresh of the
 * 16-bit operand copies the GEMM kernels read -- two launches instead of thousands.
 *   norm  = grad_scale * ||grad||_2 ;  coef = max_grad_norm > 0 ? min(1, max_grad_norm / (norm + 1e-6)) : 1
 *   g     = grad * grad_scale * coef   (grad_scale folds the 1/world of a summed all-reduce, or 1)
 * operand (may be NULL): 16-bit copy of the updated parameters, same flat layout.  norm_out (may be NULL): float[1].
 * workspace: 16 bytes, 16-byte aligned, zero-initialised once; left zeroed.  step: 1-based optimizer step count.
 * Overflow handling (fp16 loss scaling: accelerate's GradScaler around T:857-860, mixed_precision="fp16" T:126): grad_scale
 * is the UNSCALE factor (1 / loss scale, times 1 / world for a summed all-reduce).  When the norm is not finite the whole
 * update is SKIPPED -- parameters, moments and operand copies untouched, the gradient still zeroed (the trainer calls
 * zero_grad either way, T:861) -- norm_out receives the non-finite norm and found_inf (may be NULL: float[1]) 1.0f, else
 * 0.0f.  step_dev (may be NULL: int64[1] on the device, starts at 0): when given, the bias corrections use *step_dev + 1
 * and the counter advances only for applied updates, so that a skipped step does not age the moments (`step` is then ignored).
 */
typedef struct psob200_flat_adamw_args {
  float* param;
  float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  void* operand;
  float* norm_out;
  void* workspace;
  int64_t n;
  int64_t step;
  float lr, beta1, beta2, eps, weight_decay, max_grad_norm, grad_scale;
  int32_t operand_dtype;
  /* n_sumsq_parts > 0: the gradient's sum of squares was already produced in n_sumsq_parts pieces (double[], LOCAL
   * address) by psob200_flat_allreduce_sumsq -- the norm launch is skipped; the pieces are left zeroed. */
  int32_t n_sumsq_parts;
  double* sumsq_parts;
  float* found_inf;
  long long* step_dev;
} psob200_flat_adamw_args;

PSOB200_API int psob200_flat_adamw_step(const psob200_flat_adamw_args* args, void* stream);
/* psob200_flat_adamw_step unscaled by, and updating, a device loss scaler (GradScaler unscale_ / step / update, T:859-860). */
PSOB200_API int psob200_flat_adamw_step_scaled(const psob200_flat_adamw_args* args, const psob200_loss_scaler* scaler,
                                               void* stream);

/*
 * The same optimizer boundary with bitsandbytes' blockwise 8-bit AdamW state (the Turbo recipe's `use_8bit_adam`:
 * "AdamW(8bit)" over the LoRA parameters, T:428-448; Dettmers et al. 2022, "8-bit Optimizers via Block-wise Quantization").
 * Clipping, grad_scale, the overflow skip, found_inf, step_dev, norm_out, workspace, sumsq_parts, zero_grad and the operand
 * refresh are those of psob200_flat_adamw_step; only the moment storage and the update rule differ.
 *
 * 8-bit blocks (blocks8: n_blocks8 pairs {flat offset, length}, 0 < length <= block_size, offset a multiple of 8): block b
 * keeps one fp32 absmax per moment (absmax1[b], absmax2[b]) and one uint8 code per element and moment, at the element's FLAT
 * position in code1 / code2 (n bytes each).  map1 (signed, first moment) / map2 (unsigned, second moment): 256 sorted
 * floats each.  Per element, every operation fp32 and rounded separately (no contraction):
 *   g  = grad * coef                                  (coef as in psob200_flat_adamw_step)
 *   m  = map1[c1] * absmax1 ;  v = map2[c2] * absmax2
 *   m  = m * beta1 + (1 - beta1) * g ;  v = v * beta2 + (1 - beta2) * g * g
 *   bc1 = (float)(1 - beta1^t), bc2 = (float)sqrt(1 - beta2^t)   (double; t = *step_dev + 1, or `step`)
 *   p  = p + ((-lr * bc2) / bc1) * (m / (sqrt(v) + eps * bc2)) ;  if weight_decay > 0: p = p * (1 - lr * weight_decay)
 *   absmax = max |m| (max |v|) over the block ;  x = absmax > 0 ? m / absmax : 0
 *   code   = number of the 255 midpoints (map[i] + map[i+1]) * 0.5 strictly below x ;
 *   first moment only: when the sign bit of map1[code] differs from that of m, the code steps one towards m's side.
 * fp32-class ranges (chunks32: n_chunks32 triples {flat offset, length, compact offset}, 0 < length <= block_size, both
 * offsets multiples of 8): the same formulas with fp32 m / v at exp_avg32 / exp_avg_sq32 [compact offset + i].
 * The gradient is zeroed over every block and range, rounded up to whole 8-element groups (at most up to n); flat elements
 * outside them are not touched.  block_size: 256 (one warp per block) or 2048 (one 256-thread CTA per block), else
 * PSOB200_ERR_SHAPE.  param, grad, operand, code1, code2, exp_avg32, exp_avg_sq32 16-byte aligned, else PSOB200_ERR_ALIGNMENT.
 * One update launch (plus the norm launch when the norm is not supplied); deterministic; no allocation, no host sync.
 */
typedef struct psob200_flat_adamw8_args {
  float* param;
  float* grad;
  uint8_t* code1;
  uint8_t* code2;
  float* absmax1;
  float* absmax2;
  const float* map1;
  const float* map2;
  const int64_t* blocks8;
  int64_t n_blocks8;
  const int64_t* chunks32;
  int64_t n_chunks32;
  float* exp_avg32;
  float* exp_avg_sq32;
  void* operand;
  float* norm_out;
  void* workspace;
  int64_t n;
  int64_t step;
  float lr, beta1, beta2, eps, weight_decay, max_grad_norm, grad_scale;
  int32_t operand_dtype;
  int32_t n_sumsq_parts;
  int32_t block_size;
  double* sumsq_parts;
  float* found_inf;
  long long* step_dev;
} psob200_flat_adamw8_args;

PSOB200_API int psob200_flat_adamw8_step(const psob200_flat_adamw8_args* args, void* stream);
/* psob200_flat_adamw8_step unscaled by, and updating, a device loss scaler (GradScaler around the 8-bit AdamW, T:859-860). */
PSOB200_API int psob200_flat_adamw8_step_scaled(const psob200_flat_adamw8_args* args, const psob200_loss_scaler* scaler,
                                                void* stream);

/*
 * The data-parallel exchange of the training step (DDP's gradient all-reduce behind accelerator.prepare, T:491, sync
 * gate T:858) fused with the norm pass of clip_grad_norm_ (T:859), over NVLink SHARP: ONE launch per rank, no NCCL call.
 * The flat fp32 gradient buffer is symmetric memory (same size on every rank of the group) and grad_multicast is its
 * MULTICAST address (cuMulticast* / torch.distributed._symmetric_memory): rank r load-reduces its 1/world slice through
 * the NVSwitch (multimem.ld_reduce.add.v4.f32), multiplies by `scale` (1/world for the mean), stores the result into every
 * rank's copy (multimem.st) and adds the slice's sum of squares into sumsq_multicast[rank] on every rank
 * (multimem.red.add.f64; sumsq_multicast = multicast address of a zero-initialised double[world]).
 * Contract: the caller places a cross-rank barrier on the stream BEFORE this launch (every rank's backward has finished
 * accumulating) and AFTER it (every slice has landed) -- then all ranks hold bitwise-identical gradients, and
 * psob200_flat_adamw_step(n_sumsq_parts = world, sumsq_parts = the LOCAL address of that array) finishes the boundary.
 * n must be a multiple of 4; grad_multicast 16-byte aligned.
 */
typedef struct psob200_flat_allreduce_args {
  float* grad_multicast;
  double* sumsq_multicast;
  int64_t n;
  int32_t rank, world;
  float scale;
} psob200_flat_allreduce_args;

PSOB200_API int psob200_flat_allreduce_sumsq(const psob200_flat_allreduce_args* args, void* stream);

/*
 * Gated GELU of the transformer feed-forward that sits between the LoRA-wrapped attention blocks (diffusers==0.27.0
 * GEGLU.forward: `hidden, gate = self.proj(x).chunk(2, dim=-1); return hidden * F.gelu(gate)`), forward and backward
 * in one launch each.  Not a row of the PSO hot path (SURVEY.md section 8): it is here because the stock lowering of that
 * line was the largest single item of the measured micro-step.
 *   proj  [M, 2 I] (row pitch ld_proj): first I columns = hidden, last I = gate.
 *   forward:  out[M, I]   = hidden * gelu(gate)                 (exact erf GELU, fp32 arithmetic)
 *   backward: dproj[M, 2 I] = [ dout * gelu(gate) | dout * hidden * gelu'(gate) ]
 * I and the row pitches must be multiples of 16 bytes worth of elements; pointers 16-byte aligned.
 */
typedef struct psob200_geglu_args {
  const void* proj;
  void* out;
  const void* dout;
  void* dproj;
  int64_t M, I;
  int64_t ld_proj, ld_out, ld_dout, ld_dproj;
  int32_t dtype;
} psob200_geglu_args;

PSOB200_API int psob200_geglu_forward(const psob200_geglu_args* args, void* stream);
PSOB200_API int psob200_geglu_backward(const psob200_geglu_args* args, void* stream);

/*
 * LayerNorm over the last dimension (torch.nn.LayerNorm with one normalised dimension: the norm1 / norm2 / norm3 of every
 * diffusers==0.27.0 BasicTransformerBlock), forward and backward, one launch each.  Not a row of the PSO hot path
 * (SURVEY.md section 8): the stock norm kernels were the largest stock item after the attention core.
 *   x [rows, C] of dtype (row pitch ld_x); weight / bias [C] of param_dtype, each may be NULL (1 resp. 0).
 *   forward:  y = (x - mean) rstd weight + bias   [rows, C] of out_dtype;  mean, rstd: float[rows]
 *             mean = sum x / C,  rstd = 1 / sqrt(sum (x - mean)^2 / C + eps)   (fp32, centred two-pass)
 *   backward: dx = rstd (g - mean_C g - xhat mean_C(g xhat)),  g = dy weight,  xhat = (x - mean) rstd   (dy of out_dtype,
 *             dx of dtype; no weight / bias gradient: the base model is frozen)
 * dtype F32 / BF16 / F16; out_dtype = dtype, or F32 (autocast: layer_norm runs in fp32 on 16-bit input).  C a multiple of 8,
 * at most 2048; row pitches multiples of 8 elements; x, y, dy, dx 16-byte aligned.  Deterministic.
 */
typedef struct psob200_layer_norm_args {
  const void* x;
  void* y;
  const void* dy;
  void* dx;
  const void* weight;
  const void* bias;
  float* mean;
  float* rstd;
  int64_t rows, C;
  int64_t ld_x, ld_y, ld_dy, ld_dx;
  float eps;
  int32_t dtype;
  int32_t out_dtype;
  int32_t param_dtype;
} psob200_layer_norm_args;

PSOB200_API int psob200_layer_norm_forward(const psob200_layer_norm_args* args, void* stream);
PSOB200_API int psob200_layer_norm_backward(const psob200_layer_norm_args* args, void* stream);

/*
 * GroupNorm over contiguous NCHW (torch.nn.GroupNorm), optionally fused with what surrounds it in diffusers==0.27.0
 * ResnetBlock2D.forward: `nonlinearity(norm1(x))` (silu != 0) and `nonlinearity(norm2(h + time_emb_proj(temb)[:, :, None,
 * None]))` (silu != 0 and channel_add = the [N, C] projection).  Forward and backward, two launches each.
 *   x [N, C, HW] of dtype; channel_add [N, C] of dtype or NULL: xs = round_to_dtype(x + channel_add[n, c]) is what is
 *   normalised (the stock add's rounding; the backward recomputes it); weight / bias [C] of param_dtype or NULL.
 *   Group g of sample n = channels [g C / G, (g + 1) C / G), one contiguous span of S = (C / G) HW elements.
 *   forward:  z = (xs - mean) rstd weight[c] + bias[c];  y = silu ? z sigmoid(z) : z   ([N, C, HW] of out_dtype)
 *             mean, rstd: float[N G] (biased variance, Chan's pairwise merge of per-part moments)
 *   backward: g = dy (silu ? silu'(z) : 1) weight[c];  dx = rstd (g - mean_S g - xhat mean_S(g xhat))   (dx of dtype; no
 *             weight / bias / channel_add gradient: the base model is frozen)
 * Any HW >= 1 and any C divisible by G (else PSOB200_ERR_SHAPE).  workspace: >= psob200_group_norm_workspace_bytes(N, C, HW,
 * G) bytes, 16-byte aligned, no initialisation needed (cross-CTA partials of one call; one workspace per stream).
 * x, y, dy, dx 16-byte aligned.  dtype / out_dtype as psob200_layer_norm_args.  Deterministic: every group is cut into parts
 * that depend on the shape only, and the parts are combined in a fixed order.
 */
typedef struct psob200_group_norm_args {
  const void* x;
  const void* channel_add;
  void* y;
  const void* dy;
  void* dx;
  const void* weight;
  const void* bias;
  float* mean;
  float* rstd;
  void* workspace;
  size_t workspace_bytes;
  int64_t N, C, HW;
  int32_t G;
  float eps;
  int32_t dtype;
  int32_t out_dtype;
  int32_t param_dtype;
  int32_t silu;
} psob200_group_norm_args;

PSOB200_API size_t psob200_group_norm_workspace_bytes(int64_t N, int64_t C, int64_t HW, int32_t G);
PSOB200_API int psob200_group_norm_forward(const psob200_group_norm_args* args, void* stream);
PSOB200_API int psob200_group_norm_backward(const psob200_group_norm_args* args, void* stream);

/*
 * Reward-side image preprocessing on the device (SURVEY.md section 8f rank 4).  Replaces, in one launch, the round trip the
 * trainers make before every reward call (train_online_pso_sdxl_turbo.py:632-640, pso_pytorch/pickscore_utils.py:24-33):
 *     ((images + 1) * 127.5).clamp(0, 255).to(uint8).permute(0,2,3,1).cpu().numpy() -> PIL.Image.fromarray -> CLIPImageProcessor
 *     (resize shortest edge to `size` with PIL BICUBIC, centre crop, * 1/255, (x - mean) / std, channels first) -> .to(device)
 * bit-exactly: the resize is Pillow's two-pass fixed-point convolution (libImaging/Resample.c, 8 bits per channel: bicubic
 * a = -0.5 with the support stretched by the down-scale factor, coefficients rounded to 22 fractional bits, horizontal pass
 * rounded to uint8 before the vertical pass); rescale + normalise are a 3 x 256 entry table built with numpy's rounding.
 *
 * psob200_resample_taps / psob200_resample_plan (HOST only, no CUDA call): the coefficient table of one axis.  For output
 * index j (0 <= j < out_size): bounds[2j] = first input index, bounds[2j+1] = tap count, coeffs[j*taps .. ] = fixed-point
 * weights (the rest zero); `taps` = psob200_resample_taps(in_size, out_size).  The caller uploads both tables.
 * psob200_clip_norm_table (HOST only): table[c*256 + v] = float32((float32(v * rescale) - mean[c]) / std[c]).
 *
 * psob200_clip_preprocess: src is uint8 NHWC [B, in_h, in_w, 3] (src_dtype = PSOB200_U8) or the decoded image itself,
 * float NCHW [B, 3, in_h, in_w] in [-1, 1] (src_dtype F32 / BF16 / F16; quantised like the trainer's expression above, in
 * the tensor's own arithmetic type).  The image is resized to [rs_h, rs_w] (the tables' out sizes) and the window
 * [crop_top, crop_top + out_h) x [crop_left, crop_left + out_w) is written as dst [B, 3, out_h, out_w] (F32 / BF16 / F16).
 */
#define PSOB200_U8 3
PSOB200_API int psob200_resample_taps(int64_t in_size, int64_t out_size);
PSOB200_API int psob200_resample_plan(int64_t in_size, int64_t out_size, int32_t* bounds, int32_t* coeffs);
PSOB200_API int psob200_clip_norm_table(double rescale, const float* mean3, const float* std3, float* table768);

typedef struct psob200_clip_preprocess_args {
  const void* src;
  void* dst;
  const int32_t* bounds_h; /* device: horizontal (x) axis tables, out size rs_w */
  const int32_t* coeffs_h;
  const int32_t* bounds_v; /* device: vertical (y) axis tables, out size rs_h */
  const int32_t* coeffs_v;
  const float* norm_table; /* device: 768 floats */
  int64_t B, in_h, in_w, rs_h, rs_w, out_h, out_w, crop_top, crop_left;
  int32_t taps_h, taps_v;
  int32_t src_dtype, dst_dtype;
} psob200_clip_preprocess_args;

PSOB200_API int psob200_clip_preprocess(const psob200_clip_preprocess_args* args, void* stream);

/* sizeof() of the argument structs as compiled into the library, for FFI bindings to
 * verify their mirror of this header: which = 0 schedule, 1 online_pso_args,
 * 2 dreambooth_args, 3 step_args, 4 step_bwd_args, 5 gemm_args,
 * 6 lora_linear_args, 7 flat_adamw_args, 8 geglu_args,
 * 9 flat_allreduce_args, 10 clip_preprocess_args, 11 lora_group_args,
 * 12 flat_adamw8_args, 13 loss_scaler, 14 layer_norm_args, 15 group_norm_args.
 * Returns 0 for unknown ids. */
PSOB200_API size_t psob200_struct_size(int which);

#ifdef __cplusplus
}
#endif
#endif /* PSOB200_H */
