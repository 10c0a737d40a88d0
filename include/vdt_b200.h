/* vdt_b200.h — C ABI of the B200-native sampling hot path for tqch/v-diffusion-torch.
 *
 * The reference has no FFI: its boundary for this path is a Python object protocol
 * (SURVEY.md §8b).  Each entry point below names the reference interface it stands in for;
 * the Python shim in v-diffusion-torch_b200/ (UNet, GaussianDiffusion) binds them with ctypes
 * and INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success, non-zero on error (vdt_last_error() gives the
 * message, thread-local).  Unless the name ends in _host, data pointers are DEVICE pointers on the
 * current CUDA device and the call is stream-ordered on `stream` (a cudaStream_t, may be NULL).
 * A plan owns its workspace; calls on one plan must not overlap in time.
 */
#ifndef VDT_B200_H
#define VDT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDT_MAX_LEVELS 8

/* UNet constructor integers — v_diffusion/models/unet.py:155-171 (UNet.__init__), as they arrive from
 * config["model"] after the defaults merge (generate.py:86-91).  head_dim / num_heads: 0 = None. */
typedef struct vdt_unet_config {
    int32_t in_channels;
    int32_t hid_channels;
    int32_t out_channels;
    int32_t num_levels;
    int32_t ch_multipliers[VDT_MAX_LEVELS];
    int32_t num_res_blocks;
    int32_t apply_attn[VDT_MAX_LEVELS];
    int32_t embedding_dim;        /* 0 = 4 * hid_channels */
    int32_t head_dim;
    int32_t num_heads;
    int32_t num_classes;
    int32_t multitags;            /* 1: labels are fp32 multi-hot [B, num_classes] (CelebA attributes, unet.py:209-210, 290-294) */
    int32_t resolution;           /* H = W of the images this plan serves (DATA_INFO[...]["resolution"]) */
    int32_t max_rows;             /* UNet batch rows processed per pass; larger batches are chunked */
    int32_t operand_dtype;        /* 16-bit tensor-core operand format: 0 = fp16 (default), 1 = bf16; accumulation,
                                     GroupNorm statistics, softmax and the residual stream are fp32 either way.
                                     2 = split-precision validation mode: every operand is an fp16 hi/lo pair and every
                                     product three K segments (hi*hi + lo*hi + hi*lo, ~22-bit mantissa) on the same
                                     tcgen05 kernels; attention runs in fp32 on CUDA cores. ~3x slower. */
} vdt_unet_config;

/* GaussianDiffusion constructor + get_logsnr_schedule arguments — diffusion.py:260-291, 42-112. */
enum { VDT_OUT_X0 = 0, VDT_OUT_EPS = 1, VDT_OUT_BOTH = 2, VDT_OUT_V = 3 };
enum { VDT_VAR_FIXED_SMALL = 0, VDT_VAR_FIXED_LARGE = 1, VDT_VAR_FIXED_MEDIUM = 2 };
enum { VDT_SCHED_COSINE = 0, VDT_SCHED_LINEAR = 1, VDT_SCHED_SIGMOID = 2, VDT_SCHED_LEGACY = 3 };
/* Solver of the reverse loop.  FIRST_ORDER: the reference's DDIM / ancestral step.  DPMPP_2M: DPM-Solver++(2M) (Lu et al.,
 * 2022) on the same time grid t = i/T, DDIM only (use_ddim = 1, x0eps_coef = 0): the first step is DDIM, every later step
 * but the last adds c2k * (pred_x0 - pred_x0 of the previous step) to the DDIM mean (vdt_step_coefficients slot 15), and
 * the last step returns the guided x0 like DDIM. */
enum { VDT_SOLVER_FIRST_ORDER = 0, VDT_SOLVER_DPMPP_2M = 1 };
typedef struct vdt_sampler_config {
    int32_t sample_timesteps;     /* T */
    int32_t model_out_type;       /* VDT_OUT_* */
    int32_t model_var_type;       /* VDT_VAR_* */
    int32_t logsnr_schedule;      /* VDT_SCHED_* */
    int32_t use_ddim;             /* p_sample(..., use_ddim=) */
    int32_t x0eps_coef;           /* GaussianDiffusion(x0eps_coef=): posterior mean as c1*eps + c2*x0 (diffusion.py:137-140, 335-343) */
    int32_t t_fp32;               /* 1: the step tensor is fp32 as in p_sample_progressive (diffusion.py:421): s, t are fp32
                                     quotients and the timestep embedding is evaluated in fp32; 0: fp64 as in p_sample (:399) */
    int32_t solver;               /* VDT_SOLVER_*; 0 = the reference's first-order step */
    double intp_frac;
    double logsnr_min, logsnr_max;
    double w_guide;
    uint64_t seed;                /* on-device noise stream for ancestral sampling without injected noise */
} vdt_sampler_config;

typedef struct vdt_plan vdt_plan;

const char* vdt_last_error(void);
int vdt_version(void);

/* UNet(...) — unet.py:155-283.  Builds the block list, the weight table and (lazily) the workspace. */
int vdt_plan_create(const vdt_unet_config* cfg, vdt_plan** out);
void vdt_plan_destroy(vdt_plan* plan);

/* state_dict layout — SURVEY §8b.  Enumerate the expected keys / shapes (OIHW fp32 like the reference). */
int vdt_plan_num_weights(const vdt_plan* plan);
const char* vdt_plan_weight_name(const vdt_plan* plan, int index);
int vdt_plan_weight_shape(const vdt_plan* plan, int index, int64_t* shape4, int* ndim);

/* load_state_dict — generate.py:92-98.  `data` is contiguous fp32 with the reference's shape;
 * on_device != 0: device pointer, else host pointer.  Re-loading a key re-packs it. */
int vdt_plan_load_weight(vdt_plan* plan, const char* key, const float* data, int64_t numel, int on_device);
/* After all keys are loaded: pack bf16 GEMM operands.  Fails listing the first missing key. */
int vdt_plan_finalize(vdt_plan* plan);

/* UNet.forward(x, t, y) — unet.py:286-322.  x fp32 NCHW [B, in, R, R]; t fp64 [B]; y NULL, int64 [B] class ids
 * (0 = none), or fp32 multi-hot [B, num_classes] when the plan was created with multitags; out fp32 NCHW [B, out, R, R]. */
int vdt_unet_forward(vdt_plan* plan, const float* x, const double* t, const void* y, float* out, int32_t batch,
                     void* stream);

/* UNet.forward in .train() mode: the same network with nn.Dropout(drop_rate, inplace=True) active between act2 and conv2 of
 * every ResidualBlock (unet.py:135, 146).  The masks come from this library's Philox4x32-10 stream keyed by (seed, block,
 * element); drop_rate = 0 is bit-identical to vdt_unet_forward.  Forward only (the plan keeps no activations): the differentiable path is
 * the kernel tape of v-diffusion-torch_b200/training.py over the vdt_op_* entry points below. */
int vdt_unet_forward_train(vdt_plan* plan, const float* x, const double* t, const void* y, float* out, int32_t batch,
                           float drop_rate, uint64_t seed, void* stream);

/* GaussianDiffusion.p_sample(denoise_fn=UNet, shape, noise, label, use_ddim) — diffusion.py:394-414,
 * with p_sample_step (360-392) and p_mean_var (317-356) fused into one kernel per step and the step
 * captured as a CUDA graph.  noise fp32 [B, C, R, R] (x_T); label NULL, int64 [B], or fp32 multi-hot [B, num_classes] (multitags); step_noise NULL or
 * fp32 [T, B, C, R, R] (the per-step normal draws of diffusion.py:389, indexed by step); out fp32 [B, C, R, R]. */
int vdt_p_sample(vdt_plan* plan, const vdt_sampler_config* sc, const float* noise, const void* label,
                 const float* step_noise, float* out, int32_t batch, void* stream);
/* A slice of the same loop, in place on x (fp32 [B, C, R, R]): runs `num_steps` consecutive steps starting
 * at step index `first_step` (T-1 is the first step of a trajectory) — p_sample_step (diffusion.py:360-392)
 * applied num_steps times.  vdt_p_sample == copy noise, range(T-1, T), copy out.  Used by bench.py to time
 * K denoising steps of the real loop. */
int vdt_p_sample_range(vdt_plan* plan, const vdt_sampler_config* sc, float* x, const void* label,
                       const float* step_noise, int32_t batch, int32_t first_step, int32_t num_steps,
                       float* pred_x0 /* optional [B, C, R, R]: guided x0 prediction of the last step run
                                         (p_sample_step(return_pred=True); used by p_sample_progressive, 416-441).
                                         solver = DPMPP_2M: in/out -- on entry the guided x0 of step first_step + 1,
                                         read when first_step < T-1 (then it must be given) */,
                       void* stream);
/* Inpainting by replacement (Song et al., 2021, "Score-based generative modeling through SDEs", App. I; RePaint without
 * resampling).  known fp32 [B, C, R, R]: the image in model space ([-1, 1]); mask fp32 [B, C, R, R] in [0, 1], 1 = known
 * (the Python layer expands a [B, 1, R, R] mask over channels); known_noise NULL or fp32 [T, B, C, R, R], indexed by step
 * like step_noise.  known and mask come together; known_noise needs both.  Device pointers, any 4-byte alignment.
 * After step i has produced x_s (and stored the guided x0 in pred_x0, which is never replaced):
 *   i > 0:  x_s = m * k_s + (1 - m) * x_s,  k_s = alpha_s * known + sigma_s * z', with alpha_s, sigma_s = slots 0, 1 of
 *           coefficient row i - 1 (whose t is this step's s) and z' = known_noise[i], or else a standard normal from this
 *           library's Philox4x32-10 stream keyed by sc->seed with counter word 3 = 1 (the ancestral draws use 0);
 *   i = 0:  x_0 = m * known + (1 - m) * x_0.
 * m = 0 leaves x_s unchanged and m = 1 gives k_s exactly.  x_T is the caller's noise.  Every solver and output type is
 * allowed.  Under DDIM without known_noise the caller picks the seed of the z' stream. */
typedef struct vdt_inpaint {
    const float* known;
    const float* mask;
    const float* known_noise;
} vdt_inpaint;
/* vdt_p_sample / vdt_p_sample_range with inpainting; inpaint = NULL (or all three NULL) is the plain call. */
int vdt_p_sample_inpaint(vdt_plan* plan, const vdt_sampler_config* sc, const vdt_inpaint* inpaint, const float* noise,
                         const void* label, const float* step_noise, float* out, int32_t batch, void* stream);
int vdt_p_sample_range_inpaint(vdt_plan* plan, const vdt_sampler_config* sc, const vdt_inpaint* inpaint, float* x,
                               const void* label, const float* step_noise, int32_t batch, int32_t first_step,
                               int32_t num_steps, float* pred_x0, void* stream);
/* Sampling from an intermediate time (SDEdit, Meng et al., 2022; re-sampling an inverted latent): x (in place, fp32
 * [B, C, R, R]) is x at t = (first_step + 1) / T, and steps first_step ... 0 run as a fresh trajectory -- under
 * DPM-Solver++(2M) step first_step is first-order, as step T-1 is for a whole trajectory.  DDIM, ancestral sampling, CFG and
 * inpainting work unchanged; step_noise and known_noise stay [T, B, C, R, R], indexed by step.  first_step = T-1 is
 * vdt_p_sample_inpaint (in place).  0 <= first_step < T. */
int vdt_p_sample_from(vdt_plan* plan, const vdt_sampler_config* sc, const vdt_inpaint* inpaint /* nullable */, float* x,
                      const void* label, const float* step_noise, int32_t batch, int32_t first_step, void* stream);
/* DDIM inversion (Song et al., DDIM, section 4.3): the deterministic DDIM ODE walked forward in time to encode an image.
 * Inversion step j (0 <= j < T) maps x at s = j/T to x at t = (j+1)/T, the (s, t) pair of sampler step j:
 *   - the model is evaluated at the input's own time s (fp64 t = j/T; t = 0 at j = 0, where lambda = logsnr_max);
 *   - x0 comes from the raw model output through the converters of every model_out_type at lambda_s, NOT clipped (a clip
 *     would make the step impossible to invert); under CFG (w_guide > 0 and labels; rows 2i conditional, 2i+1
 *     unconditional) the guided x0 = x0c + w (x0c - x0u) -- the step is linear in x0, so this is the sampler's guidance on
 *     the means without its per-branch clip;
 *   - x_t = c1' x_s + c2' x0, c1' = sigma_t / sigma_s = exp((logsigmoid(-l_t) - logsigmoid(-l_s)) / 2),
 *     c2' = alpha_t - alpha_s c1' = -alpha_t expm1((l_s - l_t) / 2), in fp64 from the fp32-rounded log-SNRs, rounded once.
 * For an x0-type model the first step multiplies the model's error at t = 0 by sigma_t / sigma_s (about 350 at T = 100 on
 * the cosine +-20 schedule); v, eps and both are benign there, because x0 at lambda = logsnr_max reduces to x.
 * Refused (vdt_last_error): use_ddim = 0, x0eps_coef = 1, solver != FIRST_ORDER, t_fp32 = 1, steps outside [0, T).
 * vdt_invert_coefficients: out [T][16] in the vdt_step_coefficients layout -- slots 0-5 and 12-13 the converters at
 * lambda_s, 6-7 c1' and c2', 10-11 l_s and l_t, every other slot 0.
 * vdt_ddim_invert_range: in place on x (fp32 [B, C, R, R]), steps first_step ... first_step + num_steps - 1. */
int vdt_invert_coefficients(const vdt_sampler_config* sc, float* out);
int vdt_ddim_invert_range(vdt_plan* plan, const vdt_sampler_config* sc, float* x, const void* label, int32_t batch,
                          int32_t first_step, int32_t num_steps, void* stream);
/* Likelihood evaluation: the negative ELBO in bits per dimension (Ho et al., 2020, section 3.3; Nichol & Dhariwal, 2021,
 * _vb_terms_bpd / calc_bpd_loop), on this library's time grid and coefficient table.  It follows that standard definition;
 * it is not pinned to the reference's own likelihood code, which could not be compared.  For step i = 0 ... T-1 with
 * s = i/T, t = (i+1)/T (the sampler's pair of step i) and x0 in model space ([-1, 1]):
 *   - eps_i ~ N(0, I), fresh per step: noise[i] (injected, fp32 [T, B, C, R, R]) or else this library's Philox4x32-10 stream
 *     keyed by sc->seed with counter word 3 = 2 (0 is the ancestral noise, 1 inpainting's z');
 *   - x_t = alpha_t x0 + sigma_t eps_i (two fp32 products and a sum, rounded like vdt_q_sample); the model sees x_t at
 *     fp64 time t, as p_sample's does;
 *   - x0_hat from the raw output at lambda_t through the converters of every model_out_type, clipped to [-1, 1] iff
 *     clip_denoised; mse_i = mean over C*H*W of (x0_hat - x0)^2 (fp32 products, per-tile sums in fp64);
 *   - i > 0: term_i = KL(q(x_s | x_t, x0) || p(x_s | x_t)) / ln 2 as a mean over C*H*W.  Both are Gaussians with means
 *     c1 x_t + c2 x0 and c1 x_t + c2 x0_hat (c1, c2 the ancestral posterior's), log-variances lv_q = fixed_small's and
 *     lv_p = the configured model_var_type's, so term_i = K_i + k_i mse_i with K_i = (-1 + lv_p - lv_q + e^(lv_q - lv_p)) /
 *     (2 ln 2) and k_i = c2^2 e^(-lv_p) / (2 ln 2) (K_i = 0 under fixed_small);
 *   - i = 0: term_0 = -mean over C*H*W of log p(x0 | x0_hat) / ln 2 for the 8-bit discretized Gaussian decoder with
 *     log-scale lv_p(row 0) / 2: bins of half-width 1/255, CDF 0.5 (1 + tanh(sqrt(2/pi) (u + 0.044715 u^3))), open edge
 *     bins (x0 < -0.999: log CDF(plus); x0 > 0.999: log(1 - CDF(min))), every log clamped at 1e-12, in fp32.  Under
 *     fixed_small lv_p(row 0) is about -20 on the +-20 cosine schedule, so the decoder is a near-delta and term_0 is large
 *     unless x0_hat is within a bin of x0; IDDPM's clip of that variance is not reproduced;
 *   - prior_bpd = mean over C*H*W of (-1 - lv_1 + e^(lv_1) + alpha_1^2 x0^2) / (2 ln 2), alpha_1^2 = sigmoid(l1),
 *     lv_1 = logsigmoid(-l1), l1 = lambda(1) rounded to fp32;
 *   - total_bpd = sum over i of term_i (in order, fp64) + prior_bpd (the Python layer adds them).
 * Guidance plays no part (a guided model has no ELBO): labels condition the model, w_guide is ignored, as are use_ddim and
 * solver.  Refused (vdt_last_error): x0eps_coef = 1, t_fp32 = 1, model_var_type outside the three fixed types, steps outside
 * [0, T).
 * vdt_bpd_coefficients: out [T][16] in the vdt_step_coefficients layout with use_ddim = 0 -- slots 0-5 and 12-13 the
 * converters at lambda_t, 6-7 c1 and c2, 8-11 as in vdt_step_coefficients (9 = lv_p) -- with slot 14 = K_i and slot 15 = k_i
 * in place of the x0eps flag and c2k, which this path never uses.  Row 0's K_0, k_0 are the formula's and unused.
 * vdt_calc_bpd_range: x0 fp32 [B, C, R, R] (read only), label as for vdt_p_sample; fills columns first_step ...
 * first_step + num_steps - 1 of terms and mse, fp64 [B, T].  Each step is independent of the others, and per-sample sums run
 * over fixed tiles, so results are bit-identical however the range is split and the batch chunked.
 * vdt_bpd_prior: out fp64 [B], x0 fp32 [B, chw]. */
int vdt_bpd_coefficients(const vdt_sampler_config* sc, float* out);
int vdt_calc_bpd_range(vdt_plan* plan, const vdt_sampler_config* sc, const float* x0, const void* label,
                       const float* noise /* nullable, [T, B, C, R, R] */, int32_t clip_denoised, int32_t batch,
                       int32_t first_step, int32_t num_steps, double* terms, double* mse, void* stream);
int vdt_bpd_prior(const vdt_sampler_config* sc, const float* x0, int32_t batch, int32_t chw, double* out, void* stream);
/* Same with HOST buffers (pinned or pageable); copies in/out inside the call and synchronises. */
int vdt_p_sample_host(vdt_plan* plan, const vdt_sampler_config* sc, const float* noise, const void* label,
                      const float* step_noise, float* out, int32_t batch);

/* ---- training step: GaussianDiffusion.train_loss around the model call (diffusion.py:492-545) ------- */
enum { VDT_REWEIGHT_CONSTANT = 0, VDT_REWEIGHT_SNR = 1, VDT_REWEIGHT_SNR_TRUNC = 2, VDT_REWEIGHT_SNR_1PLUS = 3 };
/* Per-sample scalars from continuous times t in [0, 1] (HOST fp64 [B], Trainer.loss train_utils.py:137-147): out HOST
 * [B][16] floats, the vdt_step_coefficients slots 0-5, 11-13 (alpha, sigma, rsqrt(sigmoid l), exp(-l/2), sigmoid l,
 * sigmoid -l, l, rsqrt(sigmoid -l), exp(l/2)); only the schedule fields of sc are read. */
int vdt_train_coefficients(const vdt_sampler_config* sc, const double* t_host, int32_t batch, float* out);
/* q_sample (diffusion.py:242-245): x_t = x_0 * alpha_t + eps * sigma_t; device fp32 [B, C*H*W]; coef_dev = the table above on the device. */
int vdt_q_sample(const float* x0, const float* noise, const float* coef_dev, float* x_t, int32_t batch, int32_t chw, void* stream);
/* from_model_out_to_pred + the re-weighted MSE (diffusion.py:466-490, 518-541): loss fp32 [B]; grad_out (optional, shaped
 * like model_out) receives d loss.mean() / d model_out, the tensor autograd would hand to the UNet's backward pass. */
int vdt_train_loss(const float* model_out, const float* x0, const float* noise, const float* x_t, const float* coef_dev,
                   float* loss, float* grad_out, int32_t batch, int32_t c, int32_t hw, int32_t model_out_type,
                   int32_t reweight_type, void* stream);

/* ---- progressive distillation (Salimans & Ho, 2022, Algorithm 2) ------------------------------------------------------
 * A student sampled with N DDIM steps learns to match a teacher with 2N.  Per sample a step index i in [0, N) gives the times
 * t = (i+1)/N, t' = (2i+1)/(2N), t'' = i/N (fp64: the sampler's (t, s) grid at N and at 2N) and z_t = alpha_t x + sigma_t eps.
 * The teacher takes two DDIM steps t -> t' -> t'', each the fused sampler's DDIM step with this sample's coefficients:
 *   x1 = the guided x0 at t (per branch clipped to [-1, 1], then x0c + w (x0c - x0u); rows 2b conditional, 2b+1
 *   unconditional), z_t' = c1 z_t + c2 x1; x2 = the same at t' from z_t', z_t'' = c1' z_t' + c2' x2 (= x2 when t'' = 0).
 * Algorithm 2's target x~ = (z_t'' - (sigma_t''/sigma_t) z_t) / (alpha_t'' - (sigma_t''/sigma_t) alpha_t), the x0 with which one
 * student DDIM step from z_t lands on z_t''.  Substituting the two steps, z_t cancels exactly:
 *   z_t'' = (sigma_t''/sigma_t) z_t + sigma_t'' (alpha_t'/sigma_t' - alpha_t/sigma_t) x1 + (alpha_t'' - sigma_t'' alpha_t'/sigma_t') x2,
 * and with alpha/sigma = e^(l/2) (l = log-SNR) and every term divided by alpha_t'':
 *   x~ = c_a x1 + c_b x2,  c_b = expm1((l_t' - l_t'')/2) / expm1((l_t - l_t'')/2),
 *                          c_a = 1 - c_b = e^((l_t' - l_t'')/2) expm1((l_t - l_t')/2) / expm1((l_t - l_t'')/2),
 * both in [0, 1] since l_t < l_t' < l_t''.  At t'' = 0 the student's own last step returns its x0, so c_a = 0, c_b = 1.
 * The form never subtracts nearly equal z's, so the low-SNR end (sigma_t''/sigma_t -> 1) stays well conditioned.  The student
 * loss is vdt_train_loss unchanged with x0 := x~, noise := eps~ = z_t / sigma_t - x~ alpha_t / sigma_t, x_t := z_t and plane 0
 * below as its table, so every model_out_type and reweight_type works as in training.
 * vdt_distill_coefficients: sc->sample_timesteps is the student's N; only it, x0eps_coef and the schedule fields are read.
 * step_host HOST int32 [B]; out HOST [2][B][16]:
 *   plane 0 (t):  vdt_train_coefficients at t bit for bit, with slots 6-7 = the DDIM c1, c2 of t -> t' (sampler row 2i+1 at
 *                 2N).  It also serves vdt_q_sample and vdt_train_loss;
 *   plane 1 (t'): vdt_train_coefficients at t', with slots 6-7 = c1, c2 of t' -> t'' (sampler row 2i at 2N; 0 and 1 when
 *                 t'' = 0), 8-9 = c_a, c_b and 10 = l_t''.
 * c_a, c_b are fp64 from the fp32-rounded log-SNRs, rounded once.  Refused (vdt_last_error): x0eps_coef = 1, N < 1, steps
 * outside [0, N).
 * vdt_op_distill_step: teacher_out fp32 [B*(1+cfg), Cm, H, W] at t, z_t fp32 [B, C, H, W] -> z_mid = z_t', x0_hat = x1.
 * vdt_op_distill_target: teacher_out at t', z_mid, x0_hat, z_t -> x_target = x~, eps_target = eps~.
 * coef_dev: the table above on the device (16-byte aligned).  Image tensors at any 4-byte alignment; asynchronous on stream. */
int vdt_distill_coefficients(const vdt_sampler_config* sc, const int32_t* step_host, int32_t batch, float* out);
int vdt_op_distill_step(const float* teacher_out, const float* z_t, float* z_mid, float* x0_hat, const float* coef_dev,
                        int32_t batch, int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, float w, void* stream);
int vdt_op_distill_target(const float* teacher_out, const float* z_mid, const float* x0_hat, const float* z_t, float* x_target,
                          float* eps_target, const float* coef_dev, int32_t batch, int32_t c, int32_t hw, int32_t cfg,
                          int32_t model_out_type, float w, void* stream);

/* The tail of generate.py's batch loop (generate.py:149): fp32 NCHW samples -> uint8 NHWC pixels,
 * (x * 127.5 + 127.5).clamp(0, 255).to(uint8).permute(0, 2, 3, 1).  x fp32 [B, C, HW], out uint8 [B, HW, C]; device pointers. */
int vdt_images_to_uint8(const float* x_nchw, uint8_t* out_nhwc, int32_t batch, int32_t c, int32_t hw, void* stream);

/* logsnr schedule + posterior coefficients — diffusion.py:42-112, 126-203 (host, fp64 with the reference's
 * fp32 rounding points).  out: [T][16] floats: alpha_t, sigma_t, rsqrt(sigmoid l_t), exp(-l_t/2), sigmoid(l_t),
 * sigmoid(-l_t), c1, c2, std, logvar, logsnr_s, logsnr_t, rsqrt(sigmoid -l_t), exp(l_t/2), x0eps_coef (0/1), c2k.
 * c2k (slot 15) is 0 unless solver = DPMPP_2M; there, for 0 < i < T-1, c2k = c2 * h_i / (2 h_{i+1}) with h_i = (l_s - l_t)/2
 * of step i (fp64 from the fp32-rounded log-SNRs, rounded once), and 0 in rows 0 and T-1.  The solver is refused for
 * use_ddim = 0 and for x0eps_coef = 1.
 * With x0eps_coef and DDIM, c1/c2 are the LOGARITHMS 0.5*logsigmoid(-+l_s): the reference only exponentiates
 * them for eta != 0 (diffusion.py:180-182 vs 199) and p_sample always runs eta = 0; reproduced as is. */
int vdt_step_coefficients(const vdt_sampler_config* sc, float* out);

/* fp16 range monitor.  With fp16 operands (operand_dtype 0 / 2) every conversion of an unbounded value -- the raw
 * residual stream copied as the skip conv's operand, conv1 / q / k / v outputs kept in 16 bits -- saturates at +-65504
 * instead of overflowing to inf.  This returns how many (warp, 32x32-chunk) / thread events clamped a value since the
 * plan was finalized (or since the last call with reset != 0).  Non-zero means the checkpoint's activations leave the
 * fp16 range: use operand_dtype = 1 (bf16, fp32 exponent range) for it.  Synchronises the plan's stream. */
int vdt_plan_saturations(vdt_plan* plan, uint64_t* count, int reset);

/* Counters: kernels launched by this library since process start (graph replays count their nodes). */
uint64_t vdt_kernel_launches(void);

/* Algorithmic FLOPs (1 MAC = 2 FLOP) of one UNet.forward batch row, split like SURVEY §6:
 * convolutions (incl. 1x1), attention matmuls, embedding linears. */
int vdt_plan_flops(const vdt_plan* plan, double* conv, double* attn, double* linear);
/* FLOPs per UNet row the conv kernels execute (padded in_conv / out_conv GEMMs, sub-pixel upsampling convs; with
 * cfg_rows != 0 the label-independent prefix -- in_conv and conv1 of block 0 -- counted once per CFG row pair). */
int vdt_plan_conv_flops_executed(const vdt_plan* plan, int32_t cfg_rows, double* out);

/* Per-kernel-family device timing.  While enabled, steps run eagerly (no graph) with a CUDA-event pair
 * around every launch on the launching stream; vdt_profile_read returns accumulated milliseconds and launch
 * counts for VDT_PROF_* families and resets them. */
enum { VDT_PROF_CONV = 0, VDT_PROF_GROUPNORM = 1, VDT_PROF_ATTENTION = 2, VDT_PROF_OTHER = 3, VDT_PROF_FAMILIES = 4 };
int vdt_profile_enable(int on);
int vdt_profile_read(double* ms4, uint64_t* launches4);

/* ---- optimizer step of the reference trainer (train_utils.py:159-166) -------------------------------------------
 * nn.utils.clip_grad_norm_(params, max_norm) -> torch.optim.AdamW.step() (train.py:158) -> EMA.update() (utils.py:144-149),
 * without a host sync: vdt_grad_sq_accumulate adds one gradient tensor's sum of squares to a device double (zero it once
 * per step; fixed summation order), vdt_adamw_ema_step then updates one parameter tensor in place: g *= min(1, max_norm /
 * (sqrt(total) + 1e-6)) (skipped when grad_sq_total is null or max_norm <= 0), p *= 1 - lr * wd, Adam moments, bias-corrected
 * update with `step` = the 1-based step count, and shadow += (1 - ema_decay) * (p - shadow) when ema_shadow is given
 * (ema_decay = min(decay, (1 + num_updates) / (10 + num_updates)) is the caller's, utils.py:146). */
int64_t vdt_grad_sq_scratch_bytes(int64_t n);
int vdt_grad_sq_accumulate(const float* grad, int64_t n, void* scratch, int64_t scratch_bytes, double* sq_accum, void* stream);
int vdt_adamw_ema_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema_shadow, int64_t n,
                       double lr, double beta1, double beta2, double eps, double weight_decay, int32_t step,
                       const double* grad_sq_total, double max_norm, double ema_decay, void* stream);

/* ---- kernel-level entry points (used by the parity tests; device pointers) ------------------------- */
/* f16: 1 = fp16 operands, 0 = bf16.  conv2d(k x k, pad k/2) on 16-bit NHWC input with fp32 OIHW weights -> fp32 NHWC
 * (+bias, +residual), or 16-bit NHWC when out16 is given.  stats_out (optional): GroupNorm partial statistics,
 * float2 (sum, sum of squares) per (slab of 32 rows, stat_cols = 4 or 2 columns): [rows/32][cout/stat_cols]. */
int vdt_op_conv(const void* x_16_nhwc, int32_t batch, int32_t h, int32_t w, int32_t cin, const float* w_oihw,
                int32_t cout, int32_t ksize, const float* bias, const float* residual, float* out_nhwc, int32_t f16,
                void* out16, void* stats_out, int32_t stat_cols, void* stream);
/* One conv of the UNet plan in any of the modes the sampler runs, packed by the plan's own weight packers and launched
 * through the same setup: sub-pixel 2x-upsampling conv (ups), fused 1x1 skip conv (a1 / w1 appended as extra K),
 * split-precision operands (a3_lo / a1_lo, operand_dtype 2), upsampled or pair-shared residuals, 16-bit output, GroupNorm
 * statistics and the fp16 saturation counter.  H, W = 2h, 2w when ups = 1, else h, w.  Refused (before any CUDA call):
 * ups with a1 or a residual; resid_mode 1 with odd H or W; resid_mode 2 with an odd batch; a3_lo without a1_lo when a1 is
 * given, or the reverse; c3, c1 or cout off the multiples of 64; stats where vdt_op_conv has no layout for H x W, and for
 * ups also where 4 * slabs(h, w) != slabs(H, W) (e.g. 14 -> 28). */
typedef struct vdt_conv_op {
    const void* a3;               /* 16-bit NHWC [batch, h, w, c3]: the 3x3 operand (the low-resolution input when ups = 1) */
    const void* a3_lo;            /* NULL, or the lo halves of a3: split-precision mode, round16(x - round16(x)) */
    const void* a1;               /* NULL, or 16-bit NHWC [batch, H, W, c1]: operand of the fused 1x1 skip conv */
    const void* a1_lo;            /* lo halves of a1, given exactly when a1 and a3_lo are */
    const float* w3;              /* fp32 OIHW [cout, c3, 3, 3] */
    const float* w1;              /* fp32 OIHW [cout, c1, 1, 1], given exactly when a1 is */
    const float* bias;            /* fp32 [cout]: the conv bias (plus the skip conv's, which the plan adds into it) */
    const float* residual;        /* NULL or fp32 NHWC, read per resid_mode */
    float* out_f32;               /* fp32 NHWC [batch, H, W, cout]; exactly one of out_f32 and out16 */
    void* out16;                  /* 16-bit NHWC [batch, H, W, cout] in the operand format (fp16 saturates at +-65504) */
    void* stats;                  /* NULL or float2 [batch * vdt_stat_slabs_per_image(H, W) + 4][cout / stat_cols] */
    uint64_t* sat_count;          /* NULL or a device counter: +1 per (warp, 32x32 chunk) whose fp16 store saturated */
    int32_t batch, h, w;          /* a3's shape */
    int32_t c3, c1, cout;
    int32_t ups;                  /* 1: conv3x3(nearest_upsample_2x(a3)) in the sub-pixel form */
    int32_t resid_mode;           /* 0: residual [batch, H, W, cout]; 1: [batch, H/2, W/2, cout], output pixel (y, x) adds
                                     (y/2, x/2); 2: [batch/2, H, W, cout], output image i adds residual image i/2 */
    int32_t stat_cols;            /* 4 or 2 columns per statistics entry */
    int32_t f16;                  /* 1 fp16 operands, 0 bf16 */
} vdt_conv_op;
int vdt_op_conv_ex(const vdt_conv_op* op, void* stream);
/* The network's first conv as the plan runs it (im2col into 64 patch columns, then a pointwise GEMM): x fp32 NCHW
 * [batch, c, h, w] with 1 <= c <= 7, w fp32 OIHW [hid, c, 3, 3], bias [hid] -> out fp32 NHWC [batch * rep, h, w, hid], where
 * output image i reads input image i / rep (rep = 2: the CFG pair interleave); stats_out as for vdt_op_conv. */
int vdt_op_in_conv(const float* x_nchw, int32_t batch, int32_t rep, int32_t c, int32_t h, int32_t w, const float* w_oihw,
                   const float* bias, int32_t hid, float* out_nhwc, void* stats_out, int32_t stat_cols, int32_t f16, void* stream);
/* The network's last conv as the plan runs it (a pointwise GEMM over tap-major weight rows, then a tap-sum gather): a 16-bit
 * NHWC [batch, h, w, c0], w fp32 OIHW [cout, c0, 3, 3] with 1 <= cout <= 16, bias [cout] -> out fp32 NCHW [batch, cout, h, w]. */
int vdt_op_out_conv(const void* a_16_nhwc, int32_t batch, int32_t h, int32_t w, int32_t c0, const float* w_oihw, int32_t cout,
                    const float* bias, float* out_nchw, int32_t f16, void* stream);
/* Backward of a conv layer (F.conv2d under autograd, modules.py:141-144).
 * dgrad: dX fp32 NHWC [B, H, W, cin] = conv(dY, W rotated 180 degrees with its channel axes swapped) on the forward kernel;
 *        dy 16-bit NHWC [B, H, W, cout], w fp32 OIHW [cout, cin, k, k].
 * wgrad: dW fp32 OIHW [cout, cin, k, k] = sum over pixels of dY[p][co] * X[p + tap][ci] (tcgen05, both operands MN-major,
 *        K split over CTAs with a fixed-order reduction); optional dbias fp32 [cout] = sum over pixels of dY.  x, dy 16-bit
 *        NHWC.  Needs cout % 64 == 0 and cin % 64 == 0; takes any feature map the forward conv takes (width <= 128), including
 *        those whose tile holds fewer than 128 pixels (28x28, 14x14, 7x7, ...). */
int vdt_op_conv_dgrad(const void* dy_16_nhwc, int32_t batch, int32_t h, int32_t w, int32_t cin, const float* w_oihw, int32_t cout,
                      int32_t ksize, float* dx_nhwc, int32_t f16, void* stream);
int vdt_op_conv_wgrad(const void* x_16_nhwc, const void* dy_16_nhwc, int32_t batch, int32_t h, int32_t w, int32_t cin, int32_t cout,
                      int32_t ksize, float* dw_oihw, float* dbias, int32_t f16, void* stream);
/* Rows of the statistics table vdt_op_conv writes per image: stats_out is [batch * slabs (+ 4 rows of slack: the last
 * M tile always writes its four quarters)][cout / stat_cols] (sum, sumsq)
 * float2, one slab per 32-row quarter of an M tile of the conv kernel's image-aligned tiling; 0 = this feature-map size
 * has no such layout (the GroupNorm then makes its own statistics pass). */
int vdt_stat_slabs_per_image(int32_t h, int32_t w);
/* GroupNorm(32, 1e-6) [+FiLM] [+SiLU] [+resample 0 none / 1 avgpool2 / 2 nearest x2] over concat(src1, src2).
 * stats1/stats2 (optional): partial statistics from vdt_op_conv for src1/src2 -> single-pass kernel;
 * in16: src1 is 16-bit (needs stats1). */
int vdt_op_groupnorm(const void* src1, int32_t c1, const float* src2, int32_t c2, int32_t batch, int32_t h, int32_t w,
                     const float* gamma, const float* beta, const float* film, int32_t film_stride, int32_t film_off,
                     int32_t silu, int32_t resample, void* out_act_16, void* out_raw_16, float* out_res,
                     int32_t f16, const void* stats1, const void* stats2, int32_t stat_cols, int32_t in16, void* stream);
/* GroupNorm + SiLU with training dropout on a plain fp32 NHWC tensor (two-pass statistics): the op norm2 -> act2 -> dropout
 * of a ResidualBlock in .train() mode, exposed for the mask-statistics test. */
int vdt_op_groupnorm_dropout(const void* src1, int32_t c1, int32_t batch, int32_t h, int32_t w, const float* gamma,
                             const float* beta, int32_t silu, void* out_act_16, int32_t f16, float drop_p, uint64_t seed,
                             int32_t layer, void* stream);
/* Backward of norm -> FiLM -> SiLU -> dropout (the activation chain of a ResidualBlock, unet.py:131-135, 143-146): x and
 * grad_out fp32 [batch, h*w, c] (c % 64 == 0, c <= 2048), grad_out = gradient at the activation; film = null or
 * [batch][2c] (shift | scale per sample); (drop_p, seed, layer) name the forward's dropout stream (drop_p = 0: none).
 * Writes grad_x [batch, h*w, c], grad_gamma / grad_beta [c] and, when given, grad_film [batch][2c] (d shift | d scale).
 * Replaces autograd through F.group_norm / F.silu / F.dropout (torch/nn/functional.py) on this chain. */
int vdt_op_groupnorm_backward(const float* x, const float* grad_out, int32_t c, int32_t batch, int32_t h, int32_t w,
                              const float* gamma, const float* beta, const float* film, int32_t silu, float drop_p,
                              uint64_t seed, int32_t layer, float* grad_x, float* grad_gamma, float* grad_beta,
                              float* grad_film, void* stream);
/* The same GroupNorm kernel with the FiLM table and the training dropout stream both given: norm2 -> FiLM -> act2 -> dropout
 * of a ResidualBlock in .train() mode (unet.py:143-146) on a plain fp32 NHWC tensor; drop_p = 0: no dropout.  The mask is the
 * one vdt_op_groupnorm_backward regenerates from (seed, layer). */
int vdt_op_groupnorm_train(const void* src1, int32_t c1, int32_t batch, int32_t h, int32_t w, const float* gamma,
                           const float* beta, const float* film, int32_t film_stride, int32_t film_off, int32_t silu,
                           void* out_act_16, int32_t f16, float drop_p, uint64_t seed, int32_t layer, void* stream);
/* F.linear(x, W, b) [+ SiLU] in fp32 (modules.py:77-78; time_embed, class_embed and every ResidualBlock.fc, unet.py:142,
 * 287-295): x [rows, K], W [N, K], b [N] (required) -> out [rows, N]; K <= 1536.  The composed training step also forms the
 * backward products with it (dX = dY W: pass W^T; dW = dY^T X: pass the transposed operands). */
int vdt_op_linear(const float* x, const float* w, const float* b, float* out, int32_t rows, int32_t k, int32_t n,
                  int32_t silu_out, void* stream);
/* get_timestep_embedding(t, dim) (functions.py:10-29) for fp64 t [rows] -> fp32 [rows, dim] (sin | cos halves). */
int vdt_op_timestep_embedding(const double* t, float* out, int32_t rows, int32_t dim, void* stream);
/* The conditioning path one kernel at a time, as the plan launches it (refused before any CUDA call: null pointers, shapes
 * outside the ranges below, element counts past 2^31 - 1).
 * vdt_op_timestep_embedding_ex: the same with the plan's fp32-t switch (vdt_sampler_config.t_fp32): fp32_t = 1 rounds every
 *   op of functions.py:20-25 to fp32, as p_sample_progressive's fp32 step tensor does; 0 is vdt_op_timestep_embedding.
 * vdt_op_class_embed: out [rows, E] = SiLU(e + class term) with e [rows, E] (the time MLP's output), w [E, num_classes],
 *   b [E]; exactly one label form: y int64 [rows] (OneHot(exclude_zero=True) + Linear: id c in 1..num_classes adds
 *   b + w[:, c-1], id 0 adds b; ids below 0 add b and ids above num_classes are clamped to num_classes) or y_multihot fp32
 *   [rows, num_classes] (adds w y / sqrt(max(1, nonzeros of y)) + b, unet.py:290-294).
 * vdt_op_film_rows: the sampler's FiLM-table row per UNet row: out int32 [rows], row i reads label[i / rep], except that the
 *   odd rows of rep = 2 (CFG's unconditional half) and a NULL label give 0; ids are clamped to [0, ncls].
 * vdt_op_multitag_rows: its multitag twin: out fp32 [rows, ncls] = label[i / rep] (fp32 [rows / rep, ncls]), odd rows of
 *   rep = 2 all zero.
 * vdt_op_attention_f32: the split-precision mode's attention (operand_dtype 2), fp32 on CUDA cores: qkv fp32 [B*N, 3*hid]
 *   in vdt_op_attention's layout, d in {64, 128, 192, 256} -> out_hi 16-bit [B*N, hid] = round16(o), out_lo 16-bit =
 *   round16(o - out_hi). */
int vdt_op_timestep_embedding_ex(const double* t, float* out, int32_t rows, int32_t dim, int32_t fp32_t, void* stream);
int vdt_op_class_embed(const float* e, const int64_t* y, const float* y_multihot, const float* w, const float* b,
                       int32_t num_classes, float* out, int32_t rows, int32_t E, void* stream);
int vdt_op_film_rows(const int64_t* label, int32_t rows, int32_t rep, int32_t ncls, int32_t* out, void* stream);
int vdt_op_multitag_rows(const float* label, int32_t rows, int32_t rep, int32_t ncls, float* out, void* stream);
int vdt_op_attention_f32(const float* qkv, void* out_hi, void* out_lo, int32_t batch, int32_t n, int32_t heads, int32_t d,
                         int32_t f16, void* stream);
/* attention on qkv 16-bit [B*N, 3*hid] (q | k | v thirds, heads contiguous inside each, the layout proj_in writes)
 * -> 16-bit [B*N, hid]; any N >= 1 (ragged last key / query tiles are masked) */
int vdt_op_attention(const void* qkv_16, void* out_16, int32_t batch, int32_t n, int32_t heads,
                     int32_t d, int32_t f16, void* stream);
/* Backward of the attention core (autograd through the einsum / softmax / einsum of unet.py:55-64), reference-grade: fp32 on
 * CUDA cores, two passes (per query row: softmax statistics, D = dO . O, dQ; per key row: dK, dV), nothing N x N stored.
 * qkv fp32 [B*N, 3*hid] (q | k | v thirds, heads contiguous), grad_out fp32 [B*N, hid] -> grad_qkv fp32 [B*N, 3*hid]. */
int vdt_op_attention_backward(const float* qkv, const float* grad_out, float* grad_qkv, int32_t batch, int32_t n, int32_t heads,
                              int32_t d, void* stream);
/* one sampler update with explicit step index; coef = one row of vdt_step_coefficients (host pointer). */
int vdt_op_sampler_step(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                        int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step, const float* coef_host,
                        float w, void* stream);
/* The same update with a history buffer, for DPM-Solver++(2M) rows: pred_hist fp32 [B, C, H, W] holds the guided x0 of
 * the previous step on entry when coef[15] != 0 (it is not read otherwise) and this step's guided x0 on return.
 * vdt_op_sampler_step refuses a row with coef[15] != 0. */
int vdt_op_sampler_step_hist(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                             int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step, const float* coef_host,
                             float w, float* pred_hist, void* stream);
/* The same update followed by the inpainting replacement of vdt_inpaint: known, mask fp32 [B, C, H, W]; known_noise this
 * step's z' [B, C, H, W] or NULL (then the Philox stream 1 keyed by seed); coef_prev_host = coefficient row step - 1 (host;
 * NULL at step 0).  pred_hist may be NULL for a first-order row.  known = mask = NULL is the plain step. */
int vdt_op_sampler_step_known(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                              int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step, const float* coef_host,
                              float w, float* pred_hist, const float* known, const float* mask, const float* known_noise,
                              uint64_t seed, const float* coef_prev_host, void* stream);
/* One DDIM inversion step (vdt_ddim_invert_range) for a generic denoise_fn: x fp32 [B, C, H, W] at s -> x_next at t (may
 * alias x); model_out as for vdt_op_sampler_step; coef_host = one row of vdt_invert_coefficients (host). */
int vdt_op_invert_step(const float* model_out, const float* x, float* x_next, int32_t batch, int32_t c, int32_t hw, int32_t cfg,
                       int32_t model_out_type, const float* coef_host, float w, void* stream);
/* One step of vdt_calc_bpd_range for a generic denoise_fn: model_out fp32 [B, Cm, H, W] (no CFG rows) computed from x_t fp32
 * [B, C, H, W], x0 fp32 [B, C, H, W]; coef_host = row `step` of vdt_bpd_coefficients (host).  Writes terms[b][step] and
 * mse[b][step] of fp64 [B, num_steps] outputs.  Any 4-byte alignment. */
int vdt_op_bpd_term(const float* model_out, const float* x_t, const float* x0, int32_t batch, int32_t c, int32_t hw,
                    int32_t model_out_type, int32_t step, int32_t num_steps, const float* coef_host, int32_t clip_denoised,
                    double* terms, double* mse, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VDT_B200_H */
