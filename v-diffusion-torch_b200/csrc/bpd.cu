// Likelihood evaluation (include/vdt_b200.h vdt_calc_bpd_range): the per-step kernels around the model call of the variational
// bound in bits/dim (Ho et al., 2020, section 3.3; Nichol & Dhariwal, 2021, _vb_terms_bpd / calc_bpd_loop).
//
//   bpd_qsample_kernel   x_t = alpha_t x0 + sigma_t eps_i, rounded like q_sample_kernel (train.cu)
//   bpd_term_kernel      per-(sample, tile) sums of (x0_hat - x0)^2 and, at step 0, of the discretized-Gaussian decoder's
//                        log-likelihood, x0_hat from the raw model output (clipped when st->bpd_clip)
//   bpd_finalize_kernel  the tiles of each sample added in index order (fp64): mse_i and term_i = K_i + k_i mse_i (i > 0) or
//                        the decoder's negative log-likelihood (i = 0), in bits per dimension
//
// Kernels of their own rather than modes of sampler_step_kernel, whose register budget (six blocks per SM) a branch for this
// caller would spend.  Every per-step scalar comes from the SamplerState's copy of one vdt_bpd_coefficients row.
#include "kernels.cuh"
#include "sampler_math.cuh"

namespace vdt {
namespace {

constexpr int kBpdBlock = 256;
constexpr double kLn2 = 0.69314718055994530942;

template <int VEC> struct BVec;
template <> struct BVec<4> { typedef float4 type; };
template <> struct BVec<1> { typedef float type; };

template <int VEC>
__device__ __forceinline__ void ld_vec(const float* q, float (&v)[VEC]) {
    const typename BVec<VEC>::type t = *reinterpret_cast<const typename BVec<VEC>::type*>(q);
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = f[k];
}

// injected noise is a caller tensor that may sit at any 4-byte offset
template <int VEC>
__device__ __forceinline__ void ld_any(const float* q, float (&v)[VEC]) {
    if (VEC == 1 || (reinterpret_cast<uintptr_t>(q) & 15u) == 0) {
        ld_vec<VEC>(q, v);
    } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[k] = q[k];
    }
}

template <int VEC>
__global__ void __launch_bounds__(kBpdBlock) bpd_qsample_kernel(const BpdParams p) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * VEC;
    if (i >= n) return;
    const SamplerState* st = p.st;
    const int step = st->step;
    const float a = st->coef[0], s = st->coef[1];
    const long long gi = static_cast<long long>(st->img0) * p.C * p.HW + i;      // element index inside the whole batch
    float x[VEC], z[VEC], out[VEC];
    ld_vec<VEC>(p.x0 + i, x);
    if (st->noise) {
        ld_any<VEC>(st->noise + static_cast<long long>(step) * st->noise_step_stride + gi, z);
    } else {
        const float4 g = philox_normal4(st->seed, static_cast<uint32_t>(step), static_cast<unsigned long long>(gi) >> 2, 2u);
        if constexpr (VEC == 4) {
            z[0] = g.x; z[1] = g.y; z[2] = g.z; z[3] = g.w;
        } else {
            const int r = static_cast<int>(gi & 3);
            z[0] = r == 0 ? g.x : r == 1 ? g.y : r == 2 ? g.z : g.w;
        }
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) out[k] = __fadd_rn(__fmul_rn(x[k], a), __fmul_rn(z[k], s));
    typename BVec<VEC>::type t;
    float* f = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) f[k] = out[k];
    *reinterpret_cast<typename BVec<VEC>::type*>(p.x_t + i) = t;
}

// 0.5 (1 + tanh(sqrt(2/pi) (u + 0.044715 u^3))): the tanh approximation of the standard normal CDF (approx_std_normal_cdf)
__device__ __forceinline__ float approx_cdf(float u) {
    return 0.5f * (1.0f + tanhf(0.7978845608028654f * (u + 0.044715f * u * u * u)));
}

// log-likelihood of the 8-bit bin of x (bin half-width 1/255) under N(mean, e^(2 log_scale)), inv_stdv = e^(-log_scale);
// the edge bins are open (x < -0.999: log CDF(plus); x > 0.999: log(1 - CDF(min))) and every log is clamped at 1e-12
__device__ __forceinline__ float decoder_ll(float x, float mean, float inv_stdv) {
    const float c = x - mean;
    const float cdf_plus = approx_cdf(inv_stdv * (c + 1.0f / 255.0f));
    const float cdf_min = approx_cdf(inv_stdv * (c - 1.0f / 255.0f));
    if (x < -0.999f) return logf(fmaxf(cdf_plus, 1e-12f));
    if (x > 0.999f) return logf(fmaxf(1.0f - cdf_min, 1e-12f));
    return logf(fmaxf(cdf_plus - cdf_min, 1e-12f));
}

// fixed-shape fp64 tree over the block: the same result whatever the grid
__device__ __forceinline__ void block_sum2(double& a, double& b, double* red) {
    red[threadIdx.x] = a;
    red[kBpdBlock + threadIdx.x] = b;
    __syncthreads();
    for (int o = kBpdBlock / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            red[threadIdx.x] += red[threadIdx.x + o];
            red[kBpdBlock + threadIdx.x] += red[kBpdBlock + threadIdx.x + o];
        }
        __syncthreads();
    }
    a = red[0];
    b = red[kBpdBlock];
}

// grid (tiles, B): block (tile, b) sums over elements [tile * kBpdTile, (tile + 1) * kBpdTile) of sample b
template <int VEC>
__global__ void __launch_bounds__(kBpdBlock) bpd_term_kernel(const BpdParams p) {
    __shared__ double red[2 * kBpdBlock];
    const SamplerState* st = p.st;
    float cf[kCoefStride];
#pragma unroll
    for (int k = 0; k < kCoefStride; k += 4) {
        const float4 c4 = *reinterpret_cast<const float4*>(st->coef + k);
        cf[k] = c4.x; cf[k + 1] = c4.y; cf[k + 2] = c4.z; cf[k + 3] = c4.w;
    }
    const bool decoder = st->step == 0;
    const bool clip = st->bpd_clip != 0;
    const float inv_stdv = expf(-0.5f * cf[9]);                      // log_scale = lv_p / 2 of row 0
    const int chw = p.C * p.HW;
    const int b = blockIdx.y;
    const int lo = blockIdx.x * kBpdTile, hi = min(chw, lo + kBpdTile);
    const int Cm = (p.model_out_type == 2) ? 2 * p.C : p.C;
    const size_t base = static_cast<size_t>(b) * chw;
    const float* mo = p.model_out + static_cast<size_t>(b) * Cm * p.HW;
    float sse = 0.f, ll = 0.f;
    for (int e = lo + threadIdx.x * VEC; e < hi; e += kBpdBlock * VEC) {
        float x[VEC], x0[VEC], o[VEC], o2[VEC];
        ld_vec<VEC>(p.x_t + base + e, x);
        ld_vec<VEC>(p.x0 + base + e, x0);
        ld_vec<VEC>(mo + e, o);
        if (p.model_out_type == 2) ld_vec<VEC>(mo + chw + e, o2);     // "both": eps half follows the x0 half
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
            float xh = pred_x0_raw(p.model_out_type, x[k], o[k], (p.model_out_type == 2) ? o2[k] : 0.f, cf);
            if (clip) xh = fminf(fmaxf(xh, -1.f), 1.f);
            const float d = xh - x0[k];
            sse = fmaf(d, d, sse);
            if (decoder) ll += decoder_ll(x0[k], xh, inv_stdv);
        }
    }
    double a = sse, c = ll;
    block_sum2(a, c, red);
    if (threadIdx.x == 0) {
        double* out = p.partial + (static_cast<size_t>(b) * gridDim.x + blockIdx.x) * 2;
        out[0] = a;
        out[1] = c;
    }
}

__global__ void __launch_bounds__(128) bpd_finalize_kernel(const double* __restrict__ partial, const SamplerState* st, int B,
                                                           int chw, int tiles) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double sse = 0.0, ll = 0.0;
    for (int t = 0; t < tiles; ++t) {
        sse += partial[(static_cast<size_t>(b) * tiles + t) * 2];
        ll += partial[(static_cast<size_t>(b) * tiles + t) * 2 + 1];
    }
    const int step = st->step;
    const double mse = sse / chw;
    const double term = step == 0 ? -(ll / chw) / kLn2 : static_cast<double>(st->coef[14]) + static_cast<double>(st->coef[15]) * mse;
    const size_t at = static_cast<size_t>(st->img0 + b) * st->bpd_ld + step;
    st->bpd_terms[at] = term;
    st->bpd_mse[at] = mse;
}

__global__ void __launch_bounds__(kBpdBlock) bpd_prior_kernel(const float* __restrict__ x0, int chw, double c0, double c1,
                                                              double* __restrict__ out) {
    __shared__ double red[2 * kBpdBlock];
    const float* x = x0 + static_cast<size_t>(blockIdx.x) * chw;
    double s = 0.0, unused = 0.0;
    for (int e = threadIdx.x; e < chw; e += kBpdBlock) {
        const double v = x[e];
        s += v * v;
    }
    block_sum2(s, unused, red);
    if (threadIdx.x == 0) out[blockIdx.x] = c0 + c1 * (s / chw);
}

bool al16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

}  // namespace

cudaError_t launch_bpd_qsample(const BpdParams& p, cudaStream_t stream) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    if (n == 0) return cudaSuccess;
    // caller tensors at odd offsets (or sample sizes not divisible by 4) take the scalar kernel
    if ((static_cast<long long>(p.C) * p.HW) % 4 == 0 && al16(p.x0) && al16(p.x_t))
        bpd_qsample_kernel<4><<<static_cast<unsigned>((n / 4 + kBpdBlock - 1) / kBpdBlock), kBpdBlock, 0, stream>>>(p);
    else
        bpd_qsample_kernel<1><<<static_cast<unsigned>((n + kBpdBlock - 1) / kBpdBlock), kBpdBlock, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_bpd_term(const BpdParams& p, cudaStream_t stream) {
    if (p.B == 0) return cudaSuccess;
    const int chw = p.C * p.HW;
    const int tiles = bpd_tiles(chw);
    const dim3 grid(tiles, p.B);
    if (p.HW % 4 == 0 && al16(p.x0) && al16(p.x_t) && al16(p.model_out))
        bpd_term_kernel<4><<<grid, kBpdBlock, 0, stream>>>(p);
    else
        bpd_term_kernel<1><<<grid, kBpdBlock, 0, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    bpd_finalize_kernel<<<(p.B + 127) / 128, 128, 0, stream>>>(p.partial, p.st, p.B, chw, tiles);
    return cudaGetLastError();
}

cudaError_t launch_bpd_prior(const float* x0, int B, int chw, double c0, double c1, double* out, cudaStream_t stream) {
    if (B == 0) return cudaSuccess;
    bpd_prior_kernel<<<B, kBpdBlock, 0, stream>>>(x0, chw, c0, c1, out);
    return cudaGetLastError();
}

}  // namespace vdt
