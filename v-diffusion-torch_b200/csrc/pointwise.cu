// Small kernels around the UNet: input patch extraction, timestep/class embedding MLP (fp32),
// and the fused per-step sampler update (v/eps/x0 -> x0, clip, DDIM / ancestral posterior mean,
// classifier-free-guidance combine, noise injection).
#include "kernels.cuh"
#include "ptx.cuh"
#include "sampler_math.cuh"

namespace vdt {
namespace {

// ------------------------------------------------------------------------------------------ im2col
__global__ void im2col3x3_kernel(const float* __restrict__ x, h16* __restrict__ out, h16* __restrict__ out_lo, int B,
                                 int rep, int C, int H, int W, int f16) {
    const long long row = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long rows = static_cast<long long>(B) * rep * H * W;
    if (row >= rows) return;
    const int HW = H * W;
    const int img = static_cast<int>(row / HW), pix = static_cast<int>(row % HW);
    const int h = pix / W, w = pix % W;
    const float* xi = x + static_cast<size_t>(img / rep) * C * HW;
    float v[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) v[i] = 0.f;
    for (int tap = 0; tap < 9; ++tap) {
        const int hh = h + tap / 3 - 1, ww = w + tap % 3 - 1;
        if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
        for (int c = 0; c < C; ++c) v[tap * C + c] = __ldg(xi + static_cast<size_t>(c) * HW + hh * W + ww);
    }
    uint4* dst = reinterpret_cast<uint4*>(out + row * 64);
#pragma unroll
    for (int j = 0; j < 8; ++j)
        dst[j] = make_uint4(pack_16(v[8 * j], v[8 * j + 1], f16), pack_16(v[8 * j + 2], v[8 * j + 3], f16),
                            pack_16(v[8 * j + 4], v[8 * j + 5], f16), pack_16(v[8 * j + 6], v[8 * j + 7], f16));
    if (out_lo) {                                    // split-precision mode: lo = round16(v - round16(v))
#pragma unroll
        for (int i = 0; i < 64; ++i) {
            const uint16_t h = cvt_16(v[i], f16);
            v[i] -= f16 ? __half2float(*reinterpret_cast<const __half*>(&h)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&h));
        }
        uint4* dl = reinterpret_cast<uint4*>(out_lo + row * 64);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            dl[j] = make_uint4(pack_16(v[8 * j], v[8 * j + 1], f16), pack_16(v[8 * j + 2], v[8 * j + 3], f16),
                               pack_16(v[8 * j + 4], v[8 * j + 5], f16), pack_16(v[8 * j + 6], v[8 * j + 7], f16));
    }
}

// ------------------------------------------------------------------------------------------ fp32 attention
// Validation-mode attention (scaled_dot_product, unet.py:55-64) entirely in fp32 on CUDA cores: one warp per
// query row, lane l owns features l, l+32, ...; online softmax over the keys of the same image and head.
template <int DPL>   // features per lane = d / 32
__global__ void __launch_bounds__(256) attention_f32_kernel(const float* __restrict__ qkv, h16* __restrict__ out_hi,
                                                            h16* __restrict__ out_lo, int B, int N, int heads, int f16) {
    const int d = DPL * 32, hid = heads * d;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long qrow = (static_cast<long long>(blockIdx.x) * 8 + warp) / heads;      // global query row
    const int h = static_cast<int>((static_cast<long long>(blockIdx.x) * 8 + warp) % heads);
    if (qrow >= static_cast<long long>(B) * N) return;
    const long long img = qrow / N;
    const float* qp = qkv + qrow * 3 * hid + h * d;
    float q[DPL], o[DPL];
    const float scale = rsqrtf(static_cast<float>(d));
#pragma unroll
    for (int i = 0; i < DPL; ++i) { q[i] = qp[lane + 32 * i] * scale; o[i] = 0.f; }
    float m = -INFINITY, l = 0.f;
    for (int k = 0; k < N; ++k) {
        const float* kp = qkv + (img * N + k) * 3 * hid + hid + h * d;
        const float* vp = kp + hid;
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < DPL; ++i) s = fmaf(q[i], __ldg(kp + lane + 32 * i), s);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        const float mn = fmaxf(m, s);
        const float corr = expf(m - mn), pr = expf(s - mn);
        l = l * corr + pr;
#pragma unroll
        for (int i = 0; i < DPL; ++i) o[i] = fmaf(o[i], corr, pr * __ldg(vp + lane + 32 * i));
        m = mn;
    }
    const float inv = 1.f / l;
#pragma unroll
    for (int i = 0; i < DPL; ++i) {
        const float v = o[i] * inv;
        const uint16_t hi = cvt_16(v, f16);
        const float hf = f16 ? __half2float(*reinterpret_cast<const __half*>(&hi)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&hi));
        out_hi[qrow * hid + h * d + lane + 32 * i] = hi;
        out_lo[qrow * hid + h * d + lane + 32 * i] = cvt_16(v - hf, f16);
    }
}

// ------------------------------------------------------------------------------------------ embedding
__global__ void timestep_embedding_kernel(const double* __restrict__ t, float* __restrict__ out, int rows, int dim,
                                          const int* __restrict__ fp32_flag) {
    const int half = dim / 2;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * half) return;
    const int r = idx / half, k = idx % half;
    const double c = log(10000.0) / static_cast<double>(half - 1);
    float sn, cs;
    if (fp32_flag != nullptr && *fp32_flag != 0) {
        // fp32 `timesteps` (p_sample_progressive, diffusion.py:421): every op of functions.py:20-25 rounds to fp32
        const float ts = __fmul_rn(1000.0f, static_cast<float>(t[r]));
        const float fr = expf(__fmul_rn(-static_cast<float>(k), static_cast<float>(c)));
        const float ang = __fmul_rn(ts, fr);
        sn = sinf(ang); cs = cosf(ang);
    } else {
        const double ang = (1000.0 * t[r]) * exp(-static_cast<double>(k) * c);
        sn = static_cast<float>(sin(ang)); cs = static_cast<float>(cos(ang));
    }
    out[static_cast<size_t>(r) * dim + k] = sn;
    out[static_cast<size_t>(r) * dim + half + k] = cs;
    if ((dim & 1) && k == 0) out[static_cast<size_t>(r) * dim + dim - 1] = 0.f;
}

constexpr int kLinRows = 8;
// one warp per output feature n, kLinRows rows at a time
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ x, const float* __restrict__ W,
                                                         const float* __restrict__ b, float* __restrict__ out,
                                                         int rows, int K, int N, int silu_out) {
    extern __shared__ float xs[];                    // [kLinRows][K]
    const int r0 = blockIdx.y * kLinRows;
    const int nr = min(kLinRows, rows - r0);
    for (int i = threadIdx.x; i < kLinRows * K; i += blockDim.x) {
        const int r = i / K;
        xs[i] = (r < nr) ? x[static_cast<size_t>(r0 + r) * K + (i % K)] : 0.f;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = blockIdx.x * 8 + warp;
    if (n >= N) return;
    float acc[kLinRows];
#pragma unroll
    for (int r = 0; r < kLinRows; ++r) acc[r] = 0.f;
    const float* w = W + static_cast<size_t>(n) * K;
    for (int k = lane; k < K; k += 32) {
        const float wv = __ldg(w + k);
#pragma unroll
        for (int r = 0; r < kLinRows; ++r) acc[r] = fmaf(wv, xs[r * K + k], acc[r]);
    }
#pragma unroll
    for (int r = 0; r < kLinRows; ++r) {
        float v = acc[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        acc[r] = v;
    }
    if (lane < nr) {
        float v = 0.f;
#pragma unroll
        for (int r = 0; r < kLinRows; ++r) if (lane == r) v = acc[r];
        v += __ldg(b + n);
        if (silu_out) v = v / (1.f + expf(-v));
        out[static_cast<size_t>(r0 + lane) * N + n] = v;
    }
}

__global__ void class_embed_silu_kernel(const float* __restrict__ e, const int64_t* __restrict__ y,
                                        const float* __restrict__ w_cls, const float* __restrict__ b_cls,
                                        int num_classes, float* __restrict__ out, int rows, int E) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * E) return;
    const int r = idx / E, j = idx % E;
    float v = e[idx];
    if (y != nullptr) {
        // ids above num_classes are clamped like film_rows_kernel's (plan.cu), so that a C caller's label never reads past
        // w_cls; ids <= 0 add the bias only
        const long long id = y[r];
        const long long cls = id > num_classes ? num_classes : id;
        float add = b_cls[j];
        if (cls > 0) add += w_cls[static_cast<size_t>(j) * num_classes + (cls - 1)];
        v += add;
    }
    out[idx] = v / (1.f + expf(-v));
}

__global__ void class_embed_multitag_silu_kernel(const float* __restrict__ e, const float* __restrict__ y,
                                                 const float* __restrict__ w_cls, const float* __restrict__ b_cls,
                                                 int num_classes, float* __restrict__ out, int rows, int E) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * E) return;
    const int r = idx / E, j = idx % E;
    float v = e[idx];
    if (y != nullptr) {
        const float* yr = y + static_cast<size_t>(r) * num_classes;
        float nnz = 0.f, s = 0.f;
        for (int k = 0; k < num_classes; ++k) {
            const float yk = yr[k];
            nnz += (yk != 0.f) ? 1.f : 0.f;
            s = fmaf(w_cls[static_cast<size_t>(j) * num_classes + k], yk, s);
        }
        v += s / sqrtf(fmaxf(nnz, 1.f)) + b_cls[j];
    }
    out[idx] = v / (1.f + expf(-v));
}

// ------------------------------------------------------------------------------------------ sampler
__global__ void sampler_begin_step_kernel(SamplerState* st, const float* __restrict__ coef_table, double* t_rows,
                                          int nrows, int T) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const int step = st->next_step;
        st->step = step;
        st->next_step = step - 1;
        for (int i = 0; i < kCoefStride; ++i) st->coef[i] = coef_table[step * kCoefStride + i];
        // a trajectory that starts at this step (sampling from an intermediate time) has no previous guided x0 for 2M
        if (step == st->start_step) st->coef[15] = 0.f;
        // inpainting: the known image is diffused to this step's s = step / T, which is row step - 1's t (in both t modes)
        if (step > 0) {
            st->known_a = coef_table[(step - 1) * kCoefStride + 0];
            st->known_s = coef_table[(step - 1) * kCoefStride + 1];
        }
        // t = (step + 1) / T: fp64 in p_sample (diffusion.py:399, 364), fp32 in p_sample_progressive (diffusion.py:421)
        const double t = st->t_fp32 ? static_cast<double>(__fdiv_rn(static_cast<float>(step + 1), static_cast<float>(T)))
                                    : static_cast<double>(step + 1) / static_cast<double>(T);
        for (int r = 0; r < nrows; ++r) t_rows[r] = t;
    }
}

// Inversion walks the steps upwards: st->step = st->next_step++, and the model sees the input's own time s = step / T (fp64;
// the table of an inversion exec is vdt_invert_coefficients, which refuses the fp32-t mode)
__global__ void invert_begin_step_kernel(SamplerState* st, const float* __restrict__ coef_table, double* t_rows, int nrows, int T) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const int step = st->next_step;
        st->step = step;
        st->next_step = step + 1;
        for (int i = 0; i < kCoefStride; ++i) st->coef[i] = coef_table[step * kCoefStride + i];
        const double t = static_cast<double>(step) / static_cast<double>(T);
        for (int r = 0; r < nrows; ++r) t_rows[r] = t;
    }
}

__device__ __forceinline__ float pred_x0(int type, float x, float o, float o2, const float* cf) {
    return fminf(fmaxf(pred_x0_raw(type, x, o, o2, cf), -1.f), 1.f);   // clip_denoised (diffusion.py:327)
}

template <int VEC> struct SVec;
template <> struct SVec<4> { typedef float4 type; };
template <> struct SVec<1> { typedef float type; };

// One thread owns VEC (4 or 1) consecutive elements of one image: every tensor is read / written once with 16-byte
// (VEC = 4) fully coalesced accesses; the per-step scalars come from the device-side SamplerState.
// Six 256-thread blocks per SM (<= 42 registers): the occupancy the kernel had before inpainting added its branch, which a
// memory-bound kernel needs to keep its latency hidden (without the bound: 48 registers, five blocks, ~12 % slower).
template <int VEC>
__global__ void __launch_bounds__(256, 6) sampler_step_kernel(const SamplerStepParams p) {
    typedef typename SVec<VEC>::type vec_t;
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * VEC;
    if (i >= n) return;
    const SamplerState* st = p.st;
    float cf[kCoefStride];
#pragma unroll
    for (int k = 0; k < kCoefStride; k += 4) {
        const float4 c4 = *reinterpret_cast<const float4*>(st->coef + k);
        cf[k] = c4.x; cf[k + 1] = c4.y; cf[k + 2] = c4.z; cf[k + 3] = c4.w;
    }
    const int step = st->step;
    // read with the other state fields: the stores below may alias *st, so a later read could not be hoisted above them
    const float* const mask = st->mask;
    const int chw = p.C * p.HW;
    const int b = static_cast<int>(i / chw), e = static_cast<int>(i % chw);
    const int Cm = (p.model_out_type == 2) ? 2 * p.C : p.C;
    const int rep = 1 + p.cfg;
    const float* mo = p.model_out + static_cast<size_t>(b) * rep * Cm * p.HW + e;
    const size_t second = static_cast<size_t>(p.C) * p.HW;           // "both": eps half follows the x0 half
    float x[VEC], o[VEC], o2[VEC], u[VEC], u2[VEC], out[VEC], pr[VEC];
    auto ldv = [](const float* q, float (&v)[VEC]) {
        const vec_t t = *reinterpret_cast<const vec_t*>(q);
        const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[k] = f[k];
    };
    auto stv = [](float* q, const float (&v)[VEC]) {
        vec_t t;
        float* f = reinterpret_cast<float*>(&t);
#pragma unroll
        for (int k = 0; k < VEC; ++k) f[k] = v[k];
        *reinterpret_cast<vec_t*>(q) = t;
    };
    auto ldu = [&ldv](const float* q, float (&v)[VEC]) {            // caller-owned tensors may sit at odd offsets
        if (VEC == 1 || (reinterpret_cast<uintptr_t>(q) & 15u) == 0) {
            ldv(q, v);
        } else {
#pragma unroll
            for (int k = 0; k < VEC; ++k) v[k] = q[k];
        }
    };
    ldv(p.x_t + i, x);
    ldv(mo, o);
    if (p.model_out_type == 2) ldv(mo + second, o2);
    if (p.cfg) {
        ldv(mo + static_cast<size_t>(Cm) * p.HW, u);
        if (p.model_out_type == 2) ldv(mo + static_cast<size_t>(Cm) * p.HW + second, u2);
    }
    const float c1 = cf[6], c2 = cf[7], sd = cf[8];
    const bool last = (step == 0);
    const bool noisy = !last && sd > 0.f;
    float z[VEC];
    const long long gi = static_cast<long long>(st->img0) * chw + i;          // element index inside the whole batch
    if (noisy) {
        if (st->noise) {
            ldu(st->noise + static_cast<long long>(step) * st->noise_step_stride + gi, z);
        } else {
            const float4 g = philox_normal4(st->seed, static_cast<uint32_t>(step), static_cast<unsigned long long>(gi) >> 2);
            const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
            for (int k = 0; k < VEC; ++k) z[k] = gv[(VEC == 4) ? k : static_cast<int>(gi & 3)];
        }
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        const float x0c = pred_x0(p.model_out_type, x[k], o[k], (p.model_out_type == 2) ? o2[k] : 0.f, cf);
        // x0eps_coef: the mean's first argument is eps re-derived from the clipped x0 (diffusion.py:335-343, 222-223)
        const float a_c = p.x0eps ? x[k] * cf[12] - x0c * cf[13] : x[k];
        float mean = last ? x0c : c1 * a_c + c2 * x0c;               // where(cond, mean, pred_x_0)  (diffusion.py:378)
        float pred = x0c;
        if (p.cfg) {
            const float x0u = pred_x0(p.model_out_type, x[k], u[k], (p.model_out_type == 2) ? u2[k] : 0.f, cf);
            const float a_u = p.x0eps ? x[k] * cf[12] - x0u * cf[13] : x[k];
            const float mean_u = last ? x0u : c1 * a_u + c2 * x0u;
            mean = mean + p.w * (mean - mean_u);                     // guided, not re-clipped (diffusion.py:384)
            pred = x0c + p.w * (x0c - x0u);                          // diffusion.py:385
        }
        if (noisy) mean += sd * z[k];
        out[k] = mean; pr[k] = pred;
    }
    // DPM-Solver++(2M): x_s = DDIM mean + c2k (pred - pred of the previous step), i.e. c1 x_t + c2 D with
    // D = pred + k (pred - pred_prev).  The previous pred is read only for a non-zero c2k: the buffer may hold stale values
    // from another chunk or call (0 * NaN is NaN), and DDIM / ancestral rows (c2k = 0) keep exactly their instructions.
    // This thread owns these elements, so the read precedes the store below without a race.
    const float c2k = cf[15];
    if (c2k != 0.f) {
        float pp[VEC];
        ldv(p.pred_x0 + i, pp);
#pragma unroll
        for (int k = 0; k < VEC; ++k) out[k] = fmaf(c2k, pr[k] - pp[k], out[k]);
    }
    if (p.pred_x0) stv(p.pred_x0 + i, pr);
    // Inpainting by replacement (Song et al., 2021, App. I): x_s = m k_s + (1 - m) x_s with k_s = alpha_s known + sigma_s z'
    // (z' fresh per step, independent of the ancestral draws), and k_0 = known at the last step.  Written as m k + (1 - m) x
    // so m = 0 returns x_s and m = 1 returns k_s bit for bit.  pred (above) stays the model's guided x0.
    if (mask) {
        float m[VEC], kn[VEC];
        ldu(mask + gi, m);
        ldu(st->known + gi, kn);
        if (!last) {
            float zk[VEC];
            if (st->known_noise) {
                ldu(st->known_noise + static_cast<long long>(step) * st->noise_step_stride + gi, zk);
            } else {
                const float4 g = philox_normal4(st->seed, static_cast<uint32_t>(step), static_cast<unsigned long long>(gi) >> 2, 1u);
                const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
                for (int k = 0; k < VEC; ++k) zk[k] = gv[(VEC == 4) ? k : static_cast<int>(gi & 3)];
            }
            const float a = st->known_a, s = st->known_s;
#pragma unroll
            for (int k = 0; k < VEC; ++k) kn[k] = fmaf(a, kn[k], s * zk[k]);
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) out[k] = fmaf(m[k], kn[k], (1.f - m[k]) * out[k]);
    }
    stv(p.x_s + i, out);
}

// DDIM inversion (Song et al., DDIM, section 4.3): one step of the deterministic DDIM ODE forward in time, x at s -> x at t,
// x_t = c1' x_s + c2' x0 with the UNCLIPPED x0 at lambda_s and, under CFG, the guided x0c + w (x0c - x0u) (the step is linear in
// x0).  A kernel of its own rather than a mode of sampler_step_kernel, whose register budget (six blocks per SM) a branch for
// this caller would spend.  p.x_t is the input x_s, p.x_s the output x_t; the coefficient row is one of vdt_invert_coefficients.
template <int VEC>
__global__ void __launch_bounds__(256) invert_step_kernel(const SamplerStepParams p) {
    typedef typename SVec<VEC>::type vec_t;
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * VEC;
    if (i >= n) return;
    float cf[kCoefStride];
#pragma unroll
    for (int k = 0; k < kCoefStride; k += 4) {
        const float4 c4 = *reinterpret_cast<const float4*>(p.st->coef + k);
        cf[k] = c4.x; cf[k + 1] = c4.y; cf[k + 2] = c4.z; cf[k + 3] = c4.w;
    }
    const int chw = p.C * p.HW;
    const int b = static_cast<int>(i / chw), e = static_cast<int>(i % chw);
    const int Cm = (p.model_out_type == 2) ? 2 * p.C : p.C;
    const int rep = 1 + p.cfg;
    const float* mo = p.model_out + static_cast<size_t>(b) * rep * Cm * p.HW + e;
    const size_t second = static_cast<size_t>(p.C) * p.HW;           // "both": eps half follows the x0 half
    float x[VEC], o[VEC], o2[VEC], u[VEC], u2[VEC], out[VEC];
    auto ldv = [](const float* q, float (&v)[VEC]) {
        const vec_t t = *reinterpret_cast<const vec_t*>(q);
        const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[k] = f[k];
    };
    ldv(p.x_t + i, x);
    ldv(mo, o);
    if (p.model_out_type == 2) ldv(mo + second, o2);
    if (p.cfg) {
        ldv(mo + static_cast<size_t>(Cm) * p.HW, u);
        if (p.model_out_type == 2) ldv(mo + static_cast<size_t>(Cm) * p.HW + second, u2);
    }
    const float c1 = cf[6], c2 = cf[7];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        float x0 = pred_x0_raw(p.model_out_type, x[k], o[k], (p.model_out_type == 2) ? o2[k] : 0.f, cf);
        if (p.cfg) {
            const float x0u = pred_x0_raw(p.model_out_type, x[k], u[k], (p.model_out_type == 2) ? u2[k] : 0.f, cf);
            x0 = x0 + p.w * (x0 - x0u);
        }
        out[k] = c1 * x[k] + c2 * x0;
    }
    vec_t t;
    float* f = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) f[k] = out[k];
    *reinterpret_cast<vec_t*>(p.x_s + i) = t;
}

// ------------------------------------------------------------------------------------------ out_conv tap sum
// The network's last 3x3 conv has only Cout = out_channels (3 / 6 / 1) output channels: as an implicit GEMM its A operand
// would be fetched nine times (once per tap) for an N tile of 16 columns.  It is computed instead as ONE pointwise GEMM
// Y[p, tap * Cout + co] = sum_c act[p, c] * W[co, c, tap] (A read once) followed by this gather:
//   out[img, co, y, x] = bias[co] + sum_tap Y[pixel (y + dy, x + dx), tap * Cout + co]   (taps outside the image drop out)
// One thread per output pixel; consecutive threads own consecutive pixels, so the NCHW stores are coalesced and the nine
// gathered rows of a warp are 32 consecutive 128-byte (ld = 32) rows each.
__global__ void __launch_bounds__(256) tapsum3x3_kernel(const float* __restrict__ y, const float* __restrict__ bias,
                                                        float* __restrict__ out, long long pixels, int H, int W, int Cout, int ld) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= pixels) return;
    const int HW = H * W;
    const long long img = i / HW;
    const int pix = static_cast<int>(i - img * HW);
    const int yy = pix / W, xx = pix - yy * W;
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = (c < Cout) ? __ldg(bias + c) : 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
        const int dy = tap / 3 - 1, dx = tap % 3 - 1;
        const int y2 = yy + dy, x2 = xx + dx;
        if (y2 < 0 || y2 >= H || x2 < 0 || x2 >= W) continue;
        const float* src = y + (img * HW + y2 * W + x2) * ld + tap * Cout;
#pragma unroll
        for (int c = 0; c < 16; ++c)
            if (c < Cout) acc[c] += __ldg(src + c);
    }
    float* dst = out + img * Cout * HW + pix;
#pragma unroll
    for (int c = 0; c < 16; ++c)
        if (c < Cout) dst[static_cast<size_t>(c) * HW] = acc[c];
}

// ------------------------------------------------------------------------------------------ uint8 tail
// generate.py:149: (x * 127.5 + 127.5).clamp(0, 255).to(uint8).permute(0, 2, 3, 1) -- one thread per pixel: C coalesced
// channel-plane reads, C consecutive bytes written
__global__ void images_to_uint8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, long long pixels, int C, int HW) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i >= pixels) return;
    const long long b = i / HW;
    const int pix = static_cast<int>(i - b * HW);
    const float* xp = x + b * C * HW + pix;
    uint8_t* op = out + i * C;
    for (int c = 0; c < C; ++c) {
        // torch evaluates x * 127.5 + 127.5 as two roundings: no FMA contraction here
        float v = __fadd_rn(__fmul_rn(xp[static_cast<size_t>(c) * HW], 127.5f), 127.5f);
        v = fminf(fmaxf(v, 0.f), 255.f);
        op[c] = static_cast<uint8_t>(v);                                      // .to(uint8) truncates
    }
}

}  // namespace

cudaError_t launch_tapsum3x3(const float* y, const float* bias, float* out, int B, int H, int W, int Cout, int ld,
                             cudaStream_t stream) {
    const long long pixels = static_cast<long long>(B) * H * W;
    if (pixels == 0) return cudaSuccess;
    if (Cout > 16) return cudaErrorInvalidValue;
    tapsum3x3_kernel<<<static_cast<unsigned>((pixels + 255) / 256), 256, 0, stream>>>(y, bias, out, pixels, H, W, Cout, ld);
    return cudaGetLastError();
}

cudaError_t launch_images_to_uint8(const float* x, uint8_t* out, int B, int C, int HW, cudaStream_t stream) {
    const long long pixels = static_cast<long long>(B) * HW;
    if (pixels == 0) return cudaSuccess;
    images_to_uint8_kernel<<<static_cast<unsigned>((pixels + 255) / 256), 256, 0, stream>>>(x, out, pixels, C, HW);
    return cudaGetLastError();
}

cudaError_t launch_im2col3x3(const float* x, h16* out, h16* out_lo, int B, int rep, int C, int H, int W, int f16,
                             cudaStream_t stream) {
    if (9 * C > 64) return cudaErrorInvalidValue;
    const long long rows = static_cast<long long>(B) * rep * H * W;
    if (rows == 0) return cudaSuccess;
    im2col3x3_kernel<<<static_cast<unsigned>((rows + 127) / 128), 128, 0, stream>>>(x, out, out_lo, B, rep, C, H, W, f16);
    return cudaGetLastError();
}

cudaError_t launch_attention_f32(const float* qkv, h16* out_hi, h16* out_lo, int B, int N, int heads, int d, int f16,
                                 cudaStream_t stream) {
    const long long warps = static_cast<long long>(B) * N * heads;
    if (warps == 0) return cudaSuccess;
    const unsigned grid = static_cast<unsigned>((warps + 7) / 8);
    switch (d) {
        case 64: attention_f32_kernel<2><<<grid, 256, 0, stream>>>(qkv, out_hi, out_lo, B, N, heads, f16); break;
        case 128: attention_f32_kernel<4><<<grid, 256, 0, stream>>>(qkv, out_hi, out_lo, B, N, heads, f16); break;
        case 192: attention_f32_kernel<6><<<grid, 256, 0, stream>>>(qkv, out_hi, out_lo, B, N, heads, f16); break;
        case 256: attention_f32_kernel<8><<<grid, 256, 0, stream>>>(qkv, out_hi, out_lo, B, N, heads, f16); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t launch_timestep_embedding(const double* t, float* out, int rows, int dim, const int* fp32_flag, cudaStream_t stream) {
    const int n = rows * (dim / 2);
    if (n == 0) return cudaSuccess;
    timestep_embedding_kernel<<<(n + 127) / 128, 128, 0, stream>>>(t, out, rows, dim, fp32_flag);
    return cudaGetLastError();
}

cudaError_t launch_linear_f32(const float* x, const float* W, const float* b, float* out, int rows, int K, int N,
                              int silu_out, cudaStream_t stream) {
    if (rows == 0) return cudaSuccess;
    const size_t smem = static_cast<size_t>(kLinRows) * K * sizeof(float);
    if (smem > 48 * 1024) return cudaErrorInvalidValue;
    dim3 grid((N + 7) / 8, (rows + kLinRows - 1) / kLinRows);
    linear_f32_kernel<<<grid, 256, smem, stream>>>(x, W, b, out, rows, K, N, silu_out);
    return cudaGetLastError();
}

cudaError_t launch_class_embed_silu(const float* e, const int64_t* y, const float* w_cls, const float* b_cls,
                                    int num_classes, float* out, int rows, int E, cudaStream_t stream) {
    const int n = rows * E;
    if (n == 0) return cudaSuccess;
    class_embed_silu_kernel<<<(n + 255) / 256, 256, 0, stream>>>(e, y, w_cls, b_cls, num_classes, out, rows, E);
    return cudaGetLastError();
}

cudaError_t launch_class_embed_multitag_silu(const float* e, const float* y, const float* w_cls, const float* b_cls,
                                             int num_classes, float* out, int rows, int E, cudaStream_t stream) {
    const int n = rows * E;
    if (n == 0) return cudaSuccess;
    class_embed_multitag_silu_kernel<<<(n + 255) / 256, 256, 0, stream>>>(e, y, w_cls, b_cls, num_classes, out, rows, E);
    return cudaGetLastError();
}

cudaError_t launch_sampler_begin_step(SamplerState* st, const float* coef_table, double* t_rows, int nrows, int T,
                                      cudaStream_t stream) {
    sampler_begin_step_kernel<<<1, 32, 0, stream>>>(st, coef_table, t_rows, nrows, T);
    return cudaGetLastError();
}

cudaError_t launch_invert_begin_step(SamplerState* st, const float* coef_table, double* t_rows, int nrows, int T,
                                     cudaStream_t stream) {
    invert_begin_step_kernel<<<1, 32, 0, stream>>>(st, coef_table, t_rows, nrows, T);
    return cudaGetLastError();
}

cudaError_t launch_invert_step(const SamplerStepParams& p, cudaStream_t stream) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    if (n == 0) return cudaSuccess;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
    // caller tensors at odd offsets (or planes of a size not divisible by 4) take the scalar kernel
    const bool vec4 = (p.HW % 4 == 0) && al16(p.model_out) && al16(p.x_t) && al16(p.x_s);
    if (vec4) invert_step_kernel<4><<<static_cast<unsigned>((n / 4 + 255) / 256), 256, 0, stream>>>(p);
    else invert_step_kernel<1><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_sampler_step(const SamplerStepParams& p, cudaStream_t stream) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    if (n == 0) return cudaSuccess;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
    // 16-byte accesses need whole quads per image plane and aligned bases (an injected-noise tensor at an odd offset
    // is read with scalar loads inside the kernel)
    const bool vec4 = (p.HW % 4 == 0) && al16(p.model_out) && al16(p.x_t) && al16(p.x_s) && (p.pred_x0 == nullptr || al16(p.pred_x0));
    if (vec4) sampler_step_kernel<4><<<static_cast<unsigned>((n / 4 + 255) / 256), 256, 0, stream>>>(p);
    else sampler_step_kernel<1><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace vdt
