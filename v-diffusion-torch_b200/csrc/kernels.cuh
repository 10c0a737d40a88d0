// Launch-parameter structs and launcher prototypes shared by the kernels (.cu) and the host
// runtime (plan.cu).  All pointers are device pointers; all launchers are stream-ordered and
// return the cudaError_t of the launch.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace vdt {

constexpr int kMaxDevices = 64;   // per-device launch state (function attributes) is indexed by device ordinal
typedef uint16_t h16;   // storage of a 16-bit GEMM operand: IEEE fp16 (default) or bf16, per the launch's `f16` flag

// ------------------------------------------------------------------------------------------------
// Implicit-GEMM convolution / linear layer on tcgen05 (conv_gemm.cu)
//   D[M, Cout] = sum over K-segments  A_seg[M, taps*Cin_seg] * W[Cout, K_total]^T  (+ epilogue)
// M rows are NHWC pixels (or batch rows for a linear layer).  A tile of 128 rows is `box_n` images
// x `box_h` image rows x W pixels; a 3x3 tap is a shifted TMA box whose out-of-bounds part the
// hardware zero-fills (= the conv padding).
// ------------------------------------------------------------------------------------------------
constexpr int kConvMaxSegs = 6;   // 3x3 body + 1x1 skip, each x3 in the split-precision validation mode

enum ConvOutMode : int {
    kOutF32 = 0,        // fp32 [M, ld]            (+bias, +residual, optional SiLU)
    kOutBF16 = 1,       // 16-bit [M, ld]
};

struct alignas(64) ConvParams {
    CUtensorMap a_map[kConvMaxSegs];   // 4-D (C, W, H, N) bf16, box (64, W, box_h, box_n), SWIZZLE_128B
    CUtensorMap b_map;                 // 2-D (K_total, Cout) 16-bit, box (64, block_n / 2), SWIZZLE_128B
    int num_segs;
    int seg_taps[kConvMaxSegs];        // 9 (3x3, pad 1) or 1 (pointwise)
    int seg_kblocks[kConvMaxSegs];     // Cin_seg / 64
    int pointwise;                     // 1: A is a plain [M, C] matrix, tile row origin = m_tile * 128
    int tiles_per_image;               // H / box_h  (when box_n == 1), else 1
    int box_h, box_n;
    int rows_per_tile;                 // box_n * box_h * W  (<= 128)
    int num_m_tiles, num_n_tiles, block_n;
    int M, Cout;                       // valid rows / columns
    int out_mode;
    int ld;                            // row stride (elements) of out_f32 / out_bf16 / residual
    int HW;
    int act_silu;
    int f16;                           // operand / 16-bit output format: 1 fp16, 0 bf16
    const float* bias;                 // [Cout]
    const float* residual;             // fp32 [M, ld] or null
    int pair_tiles;                    // tiles per image when a CTA pair works on the same tile of two consecutive images, else 0
    int resid_rep;                     // > 1: output image i adds residual image i / resid_rep ([M / resid_rep, ld]; CFG row pairs
                                       // share the residual computed before the first FiLM); power-of-two HW takes the fast epilogue
    float* out_f32;
    h16* out_bf16;
    // optional GroupNorm partial statistics of the row-major output (after bias/residual): for every slab of
    // 32 consecutive rows and every stat_cols (4 or 2) consecutive columns, (sum, sum of squares):
    // stats[slab * Cout/stat_cols + col/stat_cols], slab = m_tile * 4 + (row in tile) / 32
    float2* stats;
    int stat_cols;
    // Sub-pixel form of "3x3 conv on a 2x nearest-upsampled input" (unet.py:127-128, 141 of an upsampling
    // ResidualBlock): ups = 1 -> the A operand is the LOW-resolution tensor [n, h, w, c]; each work item also carries a
    // parity class (py, px) of output pixels (2y + py, 2x + px), for which only a 2x2 neighbourhood of low-resolution
    // pixels contributes, with the 3x3 weights that fall on the same source pixel pre-summed: 4 parities x 4 taps instead
    // of 9 taps on 4x the pixels (16/36 of the MACs, the upsampled tensor never exists).  Packed weight columns:
    // [parity][segment][tap = ty * 2 + tx][cin]; tap (ty, tx) of parity (py, px) reads low-res pixel (y + ty - 1 + py,
    // x + tx - 1 + px).  Output rows are scattered to their high-resolution positions; M, HW, the tiling and the
    // statistics slabs count LOW-resolution pixels (slab of parity p: ((img * 4 + p) * stat_slabs_img + slab in image)).
    int ups, ups_w, stat_slabs_img;
    // resid_up = 1: `residual` is the low-resolution fp32 tensor [M/4, ld] of an upsampling block's identity skip
    // (unet.py:138): output pixel (y, x) of an out_w-wide image adds pixel (y >> 1, x >> 1)
    int resid_up, out_w;
    int map_shift;                     // log2 of ups_w (ups) / out_w (resid_up) when the map is square with power-of-two
                                       // sides (the fast epilogues then remap rows with shifts), else -1 (generic epilogue)
    // optional device counter of fp16 range events: incremented (once per warp and 32x32 chunk) when a value written in
    // the fp16 operand format had |x| > 65504 and was clamped by the saturating conversion
    unsigned long long* sat_count;
};
constexpr int kStatRows = 32;   // rows per statistics slab: one epilogue warp's quarter of an M tile (slab = m_tile * 4 + quarter)
// Statistics slabs per image for an h x w feature map under the conv kernel's tiling, 0 when a slab could mix two
// images: whole-image-row tiles (one image per tile) give 4 slabs per tile, partly or entirely empty when the tile
// uses fewer than 128 rows; several images per tile need images of 32 or 64 pixels.
inline int stat_slabs_per_image(int h, int w) {
    if (w < 1 || h < 1 || w > 128) return 0;
    if (2 * w * h > 128) {
        int bh = 0;
        for (int d = 1; d <= h; ++d)
            if (h % d == 0 && d * w <= 128) bh = d;
        return bh ? 4 * (h / bh) : 0;
    }
    return ((w * h) % kStatRows == 0 && 128 % (w * h) == 0) ? (w * h) / kStatRows : 0;
}
cudaError_t launch_conv_gemm(const ConvParams& p, int num_sms, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// GroupNorm(32, eps 1e-6) [+ FiLM (1+scale)*y+shift] [+ SiLU] [+ 2x avg-pool | 2x nearest upsample]
// over an fp32 NHWC tensor that may be the channel concat of two tensors (groupnorm.cu).
// ------------------------------------------------------------------------------------------------
enum Resample : int { kResNone = 0, kResDown = 1, kResUp = 2 };

struct GroupNormParams {
    const void* src1; int C1;          // fp32 (or 16-bit when in16) [B, HW, C1]
    const float* src2; int C2;         // fp32 [B, HW, C2] or null: channels C1..C1+C2 (virtual concat)
    int in16;                          // src1 holds 16-bit values in the launch's operand format (C2 must be 0)
    // rep1 / rep2 > 1: output sample b reads image b / rep of that source (and its statistics): under CFG the cond /
    // uncond rows of a sample share every tensor computed before the first FiLM (in_conv, norm1 + conv1 of block 0)
    int rep1, rep2;
    // partial statistics written by the producing conv epilogue (ConvParams::stats); when stats1 is set the
    // kernel is a single streaming pass (after a tiny finalize launch that combines the partials of every image into the
    // 32 (mean, rstd) pairs in a fixed order), otherwise it makes a statistics pass of its own
    const float2* stats1; const float2* stats2;
    int stat_cols;                     // columns per statistics entry (4, or 2 when groups are not a multiple of 4 channels)
    int stat_slabs;                    // statistics slabs per image = stat_slabs_per_image(H, W)
    float2* meanrstd;                  // scratch [B][32] (mean, rstd), required when stats1 is set
    int B, H, W;
    const float* gamma; const float* beta;   // [C1 + C2]
    const float* film;                 // null or fp32 table; row r holds [shift(C) | scale(C)] at film_off
    const int* film_row;               // [B] row index per sample (null: row = sample index)
    int film_stride, film_off;
    int silu;
    int f16;                           // 16-bit output format: 1 fp16, 0 bf16
    int resample;                      // applied after norm+act (unet.py:141)
    h16* out_act;                     // 16-bit [B, H'W', C]   normalised (+FiLM, +SiLU), resampled
    h16* out_raw;                     // optional 16-bit [B, HW, C]: the un-normalised concat (skip-conv operand)
    h16* out_act_lo;                  // split-precision mode: second halves, lo = round16(x - float(round16(x)))
    h16* out_raw_lo;
    float* out_res;                    // optional fp32 [B, H'W', C]: resampled raw input (identity-skip residual)
    // training-mode dropout on the output activation (nn.Dropout(p, inplace=True) between act2 and conv2, unet.py:135,
    // 146): element (sample, pixel, channel) is zeroed when its Philox4x32-10 word, keyed by (*drop_seed, drop_layer),
    // falls below drop_p * 2^32, and scaled by 1 / (1 - drop_p) otherwise.  drop_p = 0: no dropout (sampling path).
    float drop_p;
    const unsigned long long* drop_seed;   // device word: rewritten before every training forward, read by the captured graph
    int drop_layer;
    unsigned long long* sat_count;     // optional device counter of fp16 range events (see ConvParams::sat_count): raw
                                       // stream values clamped by out_raw's conversion, saturated 16-bit inputs read
};
cudaError_t launch_groupnorm(const GroupNormParams& p, cudaStream_t stream);

// Backward of GroupNorm -> FiLM -> SiLU -> dropout (gn_backward.cu) for an fp32 [B, HW, C] input with C % 64 == 0,
// C <= 2048; grad_out is the gradient at the activation (the forward's 16-bit rounding is straight-through).
struct GroupNormBwdParams {
    const float* x; const float* grad_out;
    const float* gamma; const float* beta;
    const float* film;                 // null or [B][2C]: shift(C) | scale(C) of every sample
    int B, HW, C, silu;
    float drop_p; unsigned long long drop_seed; int drop_layer;   // the forward's dropout stream (GroupNormParams)
    void* scratch;                     // groupnorm_backward_scratch_bytes(B, HW, C)
    float* grad_x;                     // [B, HW, C]
    float* grad_gamma; float* grad_beta;   // [C]
    float* grad_film;                  // null or [B][2C]: d shift | d scale
};
size_t groupnorm_backward_scratch_bytes(int B, int HW, int C, int* slabs_out = nullptr);
cudaError_t launch_groupnorm_backward(const GroupNormBwdParams& p, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Self-attention softmax(q^T k / sqrt(d)) v per image and head, flash-style on tcgen05 (attention.cu)
// ------------------------------------------------------------------------------------------------
struct alignas(64) AttnParams {
    CUtensorMap q_map;                 // 2-D (3*hid, B*N) 16-bit, box (64, 128): q | k | v thirds, heads contiguous in each
    CUtensorMap kv_map;                // same tensor, box (64, 64): K tiles at column hid + h*d, V tiles at 2*hid + h*d
    int B, N, heads, d, hid;
    int f16;
    float scale_log2e;                 // log2(e) / sqrt(d)
    h16* out;                         // 16-bit [B*N, hid]
};
cudaError_t launch_attention(const AttnParams& p, int num_sms, cudaStream_t stream);
// backward of the attention core in fp32 on CUDA cores (attention_bwd.cu; reference-grade, not the tensor-core kernel):
// qkv fp32 [B*N, 3*hid], dout fp32 [B*N, hid] -> dqkv fp32 [B*N, 3*hid]; stat_scratch = B*N*heads float2
cudaError_t launch_attention_backward_f32(const float* qkv, const float* dout, float* dqkv, void* stat_scratch, int B, int N, int heads,
                                          int d, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Small kernels (pointwise.cu)
// ------------------------------------------------------------------------------------------------
// x fp32 NCHW [B, C, H, W] (9*C <= 64) -> 16-bit patch matrix [B*rep*H*W, 64]: column (r*3+s)*C + c =
// x[b, c, h+r-1, w+s-1] (zero outside); output image i reads input image i / rep (the CFG
// repeat-interleave of diffusion.py:30-35, 370).
cudaError_t launch_im2col3x3(const float* x, h16* out, h16* out_lo, int B, int rep, int C, int H, int W, int f16,
                             cudaStream_t stream);

// fp32 CUDA-core attention for the split-precision validation mode: qkv fp32 [B*N, 3*hid] (q | k | v, heads
// contiguous) -> O as a 16-bit hi/lo pair [B*N, hid].  One warp per query, online softmax.
cudaError_t launch_attention_f32(const float* qkv, h16* out_hi, h16* out_lo, int B, int N, int heads, int d, int f16,
                                 cudaStream_t stream);

// sinusoidal embedding evaluated in fp64 like functions.py:11-29 -> fp32 [rows, dim]
// fp32_flag (optional device int): non-zero -> the arithmetic runs in fp32 like the reference's when it is handed an
// fp32 t (functions.py:20-25 computes in the dtype of `timesteps`; p_sample_progressive passes fp32, diffusion.py:421)
cudaError_t launch_timestep_embedding(const double* t, float* out, int rows, int dim, const int* fp32_flag, cudaStream_t stream);

// out[r, n] = act( sum_k x[r, k] * W[n, k] + b[n] )   fp32 CUDA-core path for the embedding MLP
// (time_embed, fc of every ResidualBlock: unet.py:201-205, 122, 142); rows are few (one per distinct
// (t, class) pair in the sampler), so this is weight-bandwidth bound and kept in exact fp32.
cudaError_t launch_linear_f32(const float* x, const float* W, const float* b, float* out, int rows, int K, int N,
                              int silu_out, cudaStream_t stream);

// e[r, :] = SiLU( e[r, :] + (y ? (y[r] > 0 ? W_cls[:, y[r]-1] : 0) + b_cls : 0) )   (unet.py:289-295, modules.py:184-201;
// the SiLU is the act1 applied before every fc, unet.py:142)
cudaError_t launch_class_embed_silu(const float* e, const int64_t* y, const float* w_cls, const float* b_cls,
                                    int num_classes, float* out, int rows, int E, cudaStream_t stream);

// multitag labels (unet.py:290-294): y fp32 multi-hot [rows, num_classes]; e[r, :] = SiLU(e[r, :] + W (y[r] /
// sqrt(max(nnz(y[r]), 1))) + b) with W the stock nn.Linear weight [E, num_classes] (y == nullptr: SiLU only)
cudaError_t launch_class_embed_multitag_silu(const float* e, const float* y, const float* w_cls, const float* b_cls,
                                             int num_classes, float* out, int rows, int E, cudaStream_t stream);

// out[img, co, y, x] = bias[co] + sum over the 9 taps of y[pixel shifted by the tap, tap * Cout + co] (zero padding):
// the gather half of the network's last 3x3 conv, whose GEMM half is a pointwise GEMM with N = 9 * Cout (pointwise.cu)
cudaError_t launch_tapsum3x3(const float* y, const float* bias, float* out, int B, int H, int W, int Cout, int ld,
                             cudaStream_t stream);

// generate.py:149: fp32 NCHW images in [-1, 1] -> uint8 NHWC, (x * 127.5 + 127.5).clamp(0, 255) truncated
cudaError_t launch_images_to_uint8(const float* x, uint8_t* out, int B, int C, int HW, cudaStream_t stream);

// Per-step device-side sampler state: everything that changes from step to step -- and everything that changes from
// call to call (noise tensor, seed) -- lives here, so one captured CUDA graph is replayed for every step of every call.
struct SamplerState {
    int next_step;                     // step index the next begin_step will consume (T-1 .. 0; 0 .. T-1 for inversion)
    int step;                          // step index of the step in flight
    int img0;                          // first image of the current chunk (offset into injected noise)
    int t_fp32;                        // 1: t = (step+1)/T and the sinusoidal embedding are evaluated in fp32, as
                                       // p_sample_progressive does (diffusion.py:421: `t = torch.empty(B)`)
    const float* noise;                // injected per-step noise [T, Btotal, C, HW] or null
    long long noise_step_stride;       // elements between steps (Btotal*C*HW)
    unsigned long long seed;           // on-device Philox noise when `noise` is null and std > 0; stream 1 of the same key
                                       // gives the inpainting draws when `known_noise` is null
    float known_a, known_s;            // inpainting: alpha_s, sigma_s of this step's s (slots 0, 1 of row step - 1)
    float coef[16];                    // one row of vdt_step_coefficients (include/vdt_b200.h)
    // Inpainting by replacement (include/vdt_b200.h vdt_inpaint): null mask = off.  Full-batch tensors indexed like
    // `noise` (img0 * CHW + element; known_noise also by step * noise_step_stride), possibly at odd offsets.
    const float* known;                // [Btotal, C, HW] known image in model space
    const float* mask;                 // [Btotal, C, HW] in [0, 1], 1 = known
    const float* known_noise;          // [T, Btotal, C, HW] injected z' or null
    // first step of the call's trajectory: the begin-step zeroes c2k (slot 15) there, so DPM-Solver++(2M) starts with a
    // first-order step when sampling starts at an intermediate time.  T-1 for a whole trajectory (where c2k is 0 already)
    // and for a range of one.  Kept last: coef must stay 16-byte aligned for the step kernel's float4 reads.
    int start_step;
};
constexpr int kCoefStride = 16;
// single-thread kernel: st->step = st->next_step--, copies the coefficient row (and slots 0, 1 of row step - 1 into
// known_a / known_s when step > 0; c2k zeroed when step == start_step), writes t_rows[r] = (step+1)/T
cudaError_t launch_sampler_begin_step(SamplerState* st, const float* coef_table, double* t_rows, int nrows, int T,
                                      cudaStream_t stream);
// the same for DDIM inversion, which walks upwards: st->step = st->next_step++, copies row step of the inversion table
// (vdt_invert_coefficients), writes t_rows[r] = step/T (fp64): the model sees the input's own time
cudaError_t launch_invert_begin_step(SamplerState* st, const float* coef_table, double* t_rows, int nrows, int T,
                                     cudaStream_t stream);

struct SamplerStepParams {
    const float* model_out;            // fp32 NCHW [B*(1+cfg), Cm, HW]; cond rows even, uncond rows odd
    const float* x_t;                  // fp32 NCHW [B, C, HW]
    float* x_s;                        // fp32 NCHW [B, C, HW]  (may alias x_t)
    float* pred_x0;                    // optional fp32 NCHW [B, C, HW]: the (guided) x0 prediction of this step
                                       // (p_sample_step(return_pred=True), diffusion.py:385, 392).  Required when the
                                       // coefficient row's c2k (slot 15, DPM-Solver++(2M)) is non-zero: it then holds the
                                       // previous step's prediction on entry
    const SamplerState* st;            // step index, coefficient row, injected noise / seed of this call
    int B, C, HW;
    int cfg;                           // 1: classifier-free guidance pair per sample
    int model_out_type;                // 0 x0, 1 eps, 2 both, 3 v
    float w;
    int x0eps;                         // posterior mean = c1 * eps + c2 * x0, eps re-derived from the clipped x0
};
cudaError_t launch_sampler_step(const SamplerStepParams& p, cudaStream_t stream);
// One DDIM inversion step x_s -> x_t on the same parameters: x_t (the input, at s) -> x_s (the output, at t, may alias),
// x_t = c1' x_s + c2' x0 with the unclipped (guided) x0 and the coefficient row in st->coef; pred_x0, x0eps and the state's
// noise and inpainting fields are not read.
cudaError_t launch_invert_step(const SamplerStepParams& p, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Training-step kernels (train.cu): GaussianDiffusion.train_loss around the model call (diffusion.py:492-545)
// ------------------------------------------------------------------------------------------------
// coef: device [B][kCoefStride] rows of vdt_train_coefficients.  x_t = x_0 * alpha_t + eps * sigma_t per sample.
cudaError_t launch_q_sample(const float* x0, const float* eps, const float* coef, float* x_t, int B, int chw, cudaStream_t stream);
// per-sample re-weighted MSE (type: 0 x0, 1 eps, 2 both, 3 v; reweight: 0 constant, 1 snr, 2 snr_trunc, 3 snr_1plus) and,
// when grad_out is given, d loss.mean() / d model_out
cudaError_t launch_train_loss(const float* model_out, const float* x0, const float* noise, const float* x_t, const float* coef,
                              float* loss, float* grad_out, int B, int C, int HW, int type, int reweight, cudaStream_t stream);

// optimizer step of the reference trainer (train_utils.py:159-166): sum of squared gradients of one tensor added to *accum
// (deterministic), then clip + AdamW + EMA for one parameter tensor; scratch = grad_sq_scratch_bytes(n)
size_t grad_sq_scratch_bytes(long long n);
cudaError_t launch_grad_sq(const float* g, long long n, void* scratch, double* accum, cudaStream_t stream);
cudaError_t launch_adamw_ema(float* p, const float* g, float* m, float* v, float* shadow, long long n, double lr, double beta1,
                             double beta2, double eps, double wd, int step, const double* grad_sq_total, float max_norm,
                             double ema_decay, cudaStream_t stream);

// weight gradient of a 3x3 / 1x1 conv (wgrad.cu): dW[co][ci][tap] = sum_p dY[p][co] * X[p + shift(tap)][ci]
struct alignas(64) WgradParams {
    CUtensorMap dy_map;                // 4-D (Cout, W, H, N) 16-bit, box (64, W, box_h, box_n), SWIZZLE_128B
    CUtensorMap x_map;                 // 4-D (Cin, W, H, N) 16-bit, same box
    int taps;                          // 9 or 1
    int Cout, Cin;
    int co_blocks;                     // ceil(Cout / 128); with Cout % 128 == 64 the last block holds 64 channels
    int ci_block, ci_blocks;           // input channels per accumulator (<= 256, multiple of 64), Cin / ci_block
    int tap_groups;                    // ceil(taps / 2): two taps' accumulators fill TMEM
    int splits;                        // K splits (pixel-tile ranges)
    int num_tiles, tiles_per_image, box_h, box_n, rows_per_tile;   // the forward conv's 128-pixel tiling (rows_per_tile <= 128)
    int f16;
    float* partial;                    // fp32 [splits][taps][Cout][Cin]
};
int wgrad_splits(const WgradParams& p, int num_sms);
// runs the GEMM, the fixed-order split reduction into dw (fp32 OIHW) and, when dbias is given, db[co] = sum_p dY[p][co]
cudaError_t launch_wgrad(const WgradParams& p, float* dw, float* dbias, const h16* dy, long long rows, cudaStream_t stream);

}  // namespace vdt
