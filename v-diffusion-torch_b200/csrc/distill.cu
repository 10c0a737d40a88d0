// Progressive distillation (Salimans & Ho, 2022, Algorithm 2; include/vdt_b200.h vdt_distill_coefficients): the per-sample
// coefficient rows and the two kernels between the teacher's forwards.
//
//   distill_step_kernel    teacher output at t and z_t -> x1 = the guided, clipped x0 at t, and z_t' = c1 z_t + c2 x1, the
//                          fused sampler's DDIM step t -> t' with the sample's own row
//   distill_target_kernel  teacher output at t' and z_t' -> x2 (as x1); the student's target x~ = c_a x1 + c_b x2 and
//                          eps~ = z_t / sigma_t - x~ alpha_t / sigma_t
//
// Kernels of their own rather than modes of sampler_step_kernel, whose register budget (six blocks per SM) a branch for this
// caller would spend.  Both are HBM-bound: every tensor is read or written once, with 16-byte accesses where the layout
// allows.  The rows come from a device copy of vdt_distill_coefficients ([2][B][16]: plane 0 at t, plane 1 at t').
#include <cmath>
#include <vector>

#include "../../include/vdt_b200.h"
#include "kernels.cuh"
#include "sampler_math.cuh"

namespace vdt {
namespace {

template <int VEC> struct DVec;
template <> struct DVec<4> { typedef float4 type; };
template <> struct DVec<1> { typedef float type; };

template <int VEC>
__device__ __forceinline__ void dld(const float* q, float (&v)[VEC]) {
    const typename DVec<VEC>::type t = *reinterpret_cast<const typename DVec<VEC>::type*>(q);
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = f[k];
}

template <int VEC>
__device__ __forceinline__ void dst(float* q, const float (&v)[VEC]) {
    typename DVec<VEC>::type t;
    float* f = reinterpret_cast<float*>(&t);
#pragma unroll
    for (int k = 0; k < VEC; ++k) f[k] = v[k];
    *reinterpret_cast<typename DVec<VEC>::type*>(q) = t;
}

__device__ __forceinline__ void load_row(const float* __restrict__ row, float (&cf)[kCoefStride]) {
#pragma unroll
    for (int k = 0; k < kCoefStride; k += 4) {
        const float4 c4 = __ldg(reinterpret_cast<const float4*>(row + k));
        cf[k] = c4.x; cf[k + 1] = c4.y; cf[k + 2] = c4.z; cf[k + 3] = c4.w;
    }
}

struct DistillParams {
    const float* teacher_out;          // fp32 [B*(1+cfg), Cm, HW]; cond rows even, uncond rows odd
    const float* z;                    // step: z_t; target: z_t'
    const float* x1;                   // target: the teacher's x0 at t
    const float* z_t;                  // target: z_t
    float* out_a;                      // step: z_t'; target: x~
    float* out_b;                      // step: x1;   target: eps~
    const float* coef;                 // device [2][B][16]
    int B, C, HW, cfg, model_out_type;
    float w;
};

// the teacher's x0 at this element: per branch from the raw output and clipped to [-1, 1] (clip_denoised), then guided
template <int VEC>
__device__ __forceinline__ void teacher_x0(const DistillParams& p, long long i, int b, int e, const float (&x)[VEC],
                                           const float (&cf)[kCoefStride], float (&x0)[VEC]) {
    const int Cm = (p.model_out_type == 2) ? 2 * p.C : p.C;
    const float* mo = p.teacher_out + static_cast<size_t>(b) * (1 + p.cfg) * Cm * p.HW + e;
    const size_t second = static_cast<size_t>(p.C) * p.HW;           // "both": eps half follows the x0 half
    float o[VEC], o2[VEC], u[VEC], u2[VEC];
    dld<VEC>(mo, o);
    if (p.model_out_type == 2) dld<VEC>(mo + second, o2);
    if (p.cfg) {
        dld<VEC>(mo + static_cast<size_t>(Cm) * p.HW, u);
        if (p.model_out_type == 2) dld<VEC>(mo + static_cast<size_t>(Cm) * p.HW + second, u2);
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        const float xc = fminf(fmaxf(pred_x0_raw(p.model_out_type, x[k], o[k], (p.model_out_type == 2) ? o2[k] : 0.f, cf), -1.f), 1.f);
        x0[k] = xc;
        if (p.cfg) {
            const float xu = fminf(fmaxf(pred_x0_raw(p.model_out_type, x[k], u[k], (p.model_out_type == 2) ? u2[k] : 0.f, cf), -1.f), 1.f);
            x0[k] = xc + p.w * (xc - xu);
        }
    }
}

template <int VEC>
__global__ void __launch_bounds__(256) distill_step_kernel(const DistillParams p) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * VEC;
    if (i >= n) return;
    const int chw = p.C * p.HW;
    const int b = static_cast<int>(i / chw), e = static_cast<int>(i % chw);
    float cf[kCoefStride];
    load_row(p.coef + static_cast<size_t>(b) * kCoefStride, cf);
    float x[VEC], x0[VEC], zs[VEC];
    dld<VEC>(p.z + i, x);
    teacher_x0<VEC>(p, i, b, e, x, cf, x0);
#pragma unroll
    for (int k = 0; k < VEC; ++k) zs[k] = cf[6] * x[k] + cf[7] * x0[k];
    dst<VEC>(p.out_a + i, zs);
    dst<VEC>(p.out_b + i, x0);
}

template <int VEC>
__global__ void __launch_bounds__(256) distill_target_kernel(const DistillParams p) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    const long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * VEC;
    if (i >= n) return;
    const int chw = p.C * p.HW;
    const int b = static_cast<int>(i / chw), e = static_cast<int>(i % chw);
    float cf0[kCoefStride], cf1[kCoefStride];
    load_row(p.coef + static_cast<size_t>(b) * kCoefStride, cf0);
    load_row(p.coef + (static_cast<size_t>(p.B) + b) * kCoefStride, cf1);
    float x[VEC], x2[VEC], x1[VEC], z[VEC], xt[VEC], et[VEC];
    dld<VEC>(p.z + i, x);
    teacher_x0<VEC>(p, i, b, e, x, cf1, x2);
    dld<VEC>(p.x1 + i, x1);
    dld<VEC>(p.z_t + i, z);
    const float ca = cf1[8], cb = cf1[9];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        xt[k] = __fadd_rn(__fmul_rn(ca, x1[k]), __fmul_rn(cb, x2[k]));
        et[k] = __fsub_rn(__fmul_rn(z[k], cf0[12]), __fmul_rn(xt[k], cf0[13]));   // pred_eps_from_x0 at lambda_t (train.cu)
    }
    dst<VEC>(p.out_a + i, xt);
    dst<VEC>(p.out_b + i, et);
}

bool al16(const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

template <bool kTarget>
cudaError_t launch_distill(const DistillParams& p, cudaStream_t stream) {
    const long long n = static_cast<long long>(p.B) * p.C * p.HW;
    if (n == 0) return cudaSuccess;
    // caller tensors at odd offsets (or samples of a size not divisible by 4) take the scalar kernel
    const bool vec4 = (static_cast<long long>(p.C) * p.HW) % 4 == 0 && al16(p.teacher_out) && al16(p.z) && al16(p.x1) &&
                      al16(p.z_t) && al16(p.out_a) && al16(p.out_b);
    if (vec4) {
        const unsigned grid = static_cast<unsigned>((n / 4 + 255) / 256);
        if (kTarget) distill_target_kernel<4><<<grid, 256, 0, stream>>>(p);
        else distill_step_kernel<4><<<grid, 256, 0, stream>>>(p);
    } else {
        const unsigned grid = static_cast<unsigned>((n + 255) / 256);
        if (kTarget) distill_target_kernel<1><<<grid, 256, 0, stream>>>(p);
        else distill_step_kernel<1><<<grid, 256, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

int check_args(const float* teacher_out, const float* coef_dev, int32_t batch, int32_t c, int32_t hw, int32_t model_out_type) {
    if (!teacher_out || !coef_dev) return api_fail("null argument");
    if (model_out_type < 0 || model_out_type > 3) return api_fail("unknown model_out_type %d", model_out_type);
    if (batch < 0 || c < 1 || hw < 1) return api_fail("bad image shape (%d, %d, %d)", batch, c, hw);
    if ((reinterpret_cast<uintptr_t>(coef_dev) & 15u) != 0) return api_fail("the coefficient table must be 16-byte aligned");
    return 0;
}

}  // namespace
}  // namespace vdt

using namespace vdt;

extern "C" int vdt_distill_coefficients(const vdt_sampler_config* scp, const int32_t* step_host, int32_t batch, float* out) {
    if (!scp || !step_host || !out) return api_fail("null argument");
    const int N = scp->sample_timesteps;
    if (N < 1) return api_fail("sample_timesteps (the student's N) must be >= 1, got %d", N);
    if (N > (1 << 29)) return api_fail("sample_timesteps %d is too large", N);
    if (scp->x0eps_coef)
        return api_fail("distillation needs x0eps_coef = 0 (under DDIM the reference's (eps, x0) coefficients are logarithms)");
    if (batch < 0) return api_fail("batch must be >= 0, got %d", batch);
    for (int b = 0; b < batch; ++b)
        if (step_host[b] < 0 || step_host[b] >= N) return api_fail("step %d of sample %d lies outside [0, %d)", step_host[b], b, N);
    // the teacher's DDIM table on the 2N grid: row 2i+1 is t -> t', row 2i is t' -> t'' (the p_sample fp64 time grid)
    vdt_sampler_config tc = *scp;
    tc.sample_timesteps = 2 * N;
    tc.use_ddim = 1;
    tc.solver = VDT_SOLVER_FIRST_ORDER;
    tc.t_fp32 = 0;
    std::vector<float> tab(static_cast<size_t>(2 * N) * kCoefStride);
    if (vdt_step_coefficients(&tc, tab.data()) != 0) return 1;
    for (int b = 0; b < batch; ++b) {
        const int i = step_host[b];
        float* o0 = out + static_cast<size_t>(b) * kCoefStride;
        float* o1 = out + (static_cast<size_t>(batch) + b) * kCoefStride;
        const double t = static_cast<double>(i + 1) / static_cast<double>(N);
        const double tm = static_cast<double>(2 * i + 1) / static_cast<double>(2 * N);
        if (vdt_train_coefficients(scp, &t, 1, o0) != 0) return 1;
        if (vdt_train_coefficients(scp, &tm, 1, o1) != 0) return 1;
        const float* r1 = tab.data() + static_cast<size_t>(2 * i + 1) * kCoefStride;     // t -> t'
        const float* r0 = tab.data() + static_cast<size_t>(2 * i) * kCoefStride;         // t' -> t''
        o0[6] = r1[6];
        o0[7] = r1[7];
        const double lt = r1[11], lm = r1[10], ls = r0[10];                               // fp32-rounded l_t, l_t', l_t''
        if (i == 0) {                    // t'' = 0: the teacher's second step and the student's step both return x0
            o1[6] = 0.0f; o1[7] = 1.0f; o1[8] = 0.0f; o1[9] = 1.0f;
        } else {
            o1[6] = r0[6];
            o1[7] = r0[7];
            const double den = std::expm1(0.5 * (lt - ls));
            o1[8] = static_cast<float>(std::exp(0.5 * (lm - ls)) * std::expm1(0.5 * (lt - lm)) / den);
            o1[9] = static_cast<float>(std::expm1(0.5 * (lm - ls)) / den);
        }
        o1[10] = static_cast<float>(ls);
    }
    return 0;
}

extern "C" int vdt_op_distill_step(const float* teacher_out, const float* z_t, float* z_mid, float* x0_hat, const float* coef_dev,
                                   int32_t batch, int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, float w,
                                   void* stream) {
    if (check_args(teacher_out, coef_dev, batch, c, hw, model_out_type) != 0) return 1;
    if (!z_t || !z_mid || !x0_hat) return api_fail("null argument");
    DistillParams p{};
    p.teacher_out = teacher_out; p.z = z_t; p.out_a = z_mid; p.out_b = x0_hat; p.coef = coef_dev;
    p.B = batch; p.C = c; p.HW = hw; p.cfg = cfg ? 1 : 0; p.model_out_type = model_out_type; p.w = w;
    const cudaError_t e = launch_distill<false>(p, reinterpret_cast<cudaStream_t>(stream));
    api_count_launch();
    if (e != cudaSuccess) return api_fail("distill_step launch failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_op_distill_target(const float* teacher_out, const float* z_mid, const float* x0_hat, const float* z_t,
                                     float* x_target, float* eps_target, const float* coef_dev, int32_t batch, int32_t c,
                                     int32_t hw, int32_t cfg, int32_t model_out_type, float w, void* stream) {
    if (check_args(teacher_out, coef_dev, batch, c, hw, model_out_type) != 0) return 1;
    if (!z_mid || !x0_hat || !z_t || !x_target || !eps_target) return api_fail("null argument");
    DistillParams p{};
    p.teacher_out = teacher_out; p.z = z_mid; p.x1 = x0_hat; p.z_t = z_t; p.out_a = x_target; p.out_b = eps_target;
    p.coef = coef_dev; p.B = batch; p.C = c; p.HW = hw; p.cfg = cfg ? 1 : 0; p.model_out_type = model_out_type; p.w = w;
    const cudaError_t e = launch_distill<true>(p, reinterpret_cast<cudaStream_t>(stream));
    api_count_launch();
    if (e != cudaSuccess) return api_fail("distill_target launch failed: %s", cudaGetErrorString(e));
    return 0;
}
