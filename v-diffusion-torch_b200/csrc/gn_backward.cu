// Backward of the fused GroupNorm(32, eps 1e-6) -> FiLM -> SiLU -> dropout activation of a ResidualBlock
// (unet.py:106-148; forward: groupnorm.cu).  HBM-bound: two streaming passes over (x, dA), everything else is tiny.
//
//   xhat = (x - mean_g) * rstd_g,  y = gamma * xhat + beta,  z = (1 + scale_b) * y + shift_b,  a = drop(silu(z))
//
//   dz        = dA * mask / (1 - p) * silu'(z)
//   A[b, c]   = sum_hw dz              Bc[b, c] = sum_hw dz * xhat               (pass 1, per-sample slabs, fixed order)
//   dshift    = A                      dscale   = gamma * Bc + beta * A
//   dgamma[c] = sum_b (1 + scale) Bc   dbeta[c] = sum_b (1 + scale) A
//   m1[b, g]  = mean over the group of dxhat = sum_c gamma (1 + scale) A / n,    m2 = the same with Bc
//   dx        = rstd * (gamma (1 + scale) dz - m1 - xhat * m2)                   (pass 2)
//
// The 16-bit rounding of the forward output is treated as the identity (straight-through).  The dropout mask is
// regenerated from the forward's Philox stream (same counter / key / word per element), never stored.
// All reductions run in a fixed order: results are bit-reproducible run to run.
//
// Channel layout (as the forward, groupnorm.cu: launch_groupnorm): a thread owns VEC channels of one group -- 4 when the
// group width is a multiple of 4, else 2 -- and a row of CV = CB / VEC threads covers one channel block of CB channels
// (whole groups); the kThreads / CV rows of a CTA stride over the pixels.  C up to 256 four-wide vectors is one channel
// block; wider C, or a row that would leave more than a quarter of the CTA idle, is split over gridDim.z channel blocks.
#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {
namespace {

constexpr int kGroups = 32;
constexpr float kEps = 1e-6f;
constexpr int kThreads = 256;

template <int VEC>
__device__ __forceinline__ void load_vec(const float* src, float (&v)[VEC]) {
    if constexpr (VEC == 4) {
        const float4 t = *reinterpret_cast<const float4*>(src);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
        const float2 t = *reinterpret_cast<const float2*>(src);
        v[0] = t.x; v[1] = t.y;
    }
}

// (mean, rstd) of every group of one channel block of one sample: fp32 partial sums per thread, combined in fp64 (as the
// forward's fallback pass).  grid (B, channel blocks)
template <int VEC>
__global__ void __launch_bounds__(kThreads) gn_stats_kernel(const float* __restrict__ x, float2* __restrict__ meanrstd, int HW, int C, int CB) {
    extern __shared__ float2 part[];                       // [kThreads]
    const int b = blockIdx.x, tid = threadIdx.x;
    const int CV = CB / VEC, PPH = kThreads / CV;          // channel vectors, pixel phases (host: CV <= kThreads)
    const int cv = tid % CV, pp = tid / CV;
    const float* src = x + static_cast<size_t>(b) * HW * C + blockIdx.y * CB + cv * VEC;
    float s = 0.f, ss = 0.f;
    if (pp < PPH)
        for (int pix = pp; pix < HW; pix += PPH) {
            float v[VEC];
            load_vec<VEC>(src + static_cast<size_t>(pix) * C, v);
            if constexpr (VEC == 4) {
                s += (v[0] + v[1]) + (v[2] + v[3]);
                ss = fmaf(v[0], v[0], fmaf(v[1], v[1], fmaf(v[2], v[2], fmaf(v[3], v[3], ss))));
            } else {
                s += v[0] + v[1];
                ss = fmaf(v[0], v[0], fmaf(v[1], v[1], ss));
            }
        }
    part[tid] = make_float2(s, ss);
    __syncthreads();
    const int cpg = C / kGroups, vpg = cpg / VEC, G = CB / cpg;
    if (tid < G) {
        double ds = 0.0, dss = 0.0;
        for (int ph = 0; ph < PPH; ++ph)
            for (int j = 0; j < vpg; ++j) {
                const float2 t = part[ph * CV + tid * vpg + j];
                ds += t.x; dss += t.y;
            }
        const double n = static_cast<double>(cpg) * HW;
        const double mean = ds / n;
        double var = dss / n - mean * mean;
        if (var < 0.0) var = 0.0;
        meanrstd[b * kGroups + blockIdx.y * G + tid] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + static_cast<double>(kEps))));
    }
}

template <int VEC>
struct Elem { float xhat[VEC], dz[VEC]; };

// The per-element chain shared by both passes: recompute xhat, z and the activation's derivative, apply the mask.
template <int VEC>
struct Chain {
    float rstd, mean;
    float ga[VEC], be[VEC], fs[VEC], fb[VEC];
    int silu;
    int word0;                  // 2-wide vectors: 1 -> Philox words 2, 3 (word ((c >> 1) & 1) * 2 + i, as groupnorm.cu)
    bool drop; uint32_t thr; float dscale; unsigned long long seed; int layer;
    // e: element index of the vector's first channel; one Philox call per 4 elements (counter e >> 2) as in the forward
    __device__ __forceinline__ Elem<VEC> eval(const float (&x)[VEC], const float (&g)[VEC], unsigned long long e) const {
        uint32_t w[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        if (drop) {
            const uint4 r = philox4x32(make_uint4(static_cast<uint32_t>(e >> 2), static_cast<uint32_t>(e >> 34), static_cast<uint32_t>(layer), 0x44524f50u),
                                       make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
            w[0] = r.x; w[1] = r.y; w[2] = r.z; w[3] = r.w;
            if (VEC == 2 && word0) { w[0] = r.z; w[1] = r.w; }
        }
        Elem<VEC> o;
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            o.xhat[i] = (x[i] - mean) * rstd;
            const float z = fs[i] * (ga[i] * o.xhat[i] + be[i]) + fb[i];
            float d = g[i];
            if (drop) d = (w[i] < thr) ? 0.f : d * dscale;
            if (silu) {
                const float sg = 1.f / (1.f + expf(-z));
                d *= sg * (1.f + z * (1.f - sg));
            }
            o.dz[i] = d;
        }
        return o;
    }
};

struct BwdArgs {
    const float* x; const float* grad_out; const float2* meanrstd;
    const float* gamma; const float* beta; const float* film;      // film: [B][2C] (shift | scale) or null
    int B, HW, C, CB, silu, slabs;                                 // CB: channels of one channel block (gridDim.z = C / CB)
    float drop_p; unsigned long long seed; int layer;
    float2* partial;            // [B][slabs][C] (sum dz, sum dz * xhat)
    float2* ab;                 // [B][C] the same, summed over the slabs
    float2* m12;                // [B][32]
    float* grad_x; float* grad_gamma; float* grad_beta; float* grad_film;
};

template <int VEC>
__device__ __forceinline__ Chain<VEC> make_chain(const BwdArgs& p, int b, int c) {
    Chain<VEC> ch;
    const float2 st = p.meanrstd[b * kGroups + c / (p.C / kGroups)];
    ch.mean = st.x; ch.rstd = st.y;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
        ch.ga[i] = p.gamma[c + i]; ch.be[i] = p.beta[c + i];
        ch.fb[i] = p.film ? p.film[static_cast<size_t>(b) * 2 * p.C + c + i] : 0.f;
        ch.fs[i] = p.film ? 1.f + p.film[static_cast<size_t>(b) * 2 * p.C + p.C + c + i] : 1.f;
    }
    ch.silu = p.silu;
    ch.word0 = VEC == 4 ? 0 : (c >> 1) & 1;
    ch.drop = p.drop_p > 0.f;
    ch.thr = ch.drop ? static_cast<uint32_t>(fminf(p.drop_p, 0.99999994f) * 4294967296.0f) : 0u;
    ch.dscale = ch.drop ? 1.f / (1.f - p.drop_p) : 1.f;
    ch.seed = p.seed; ch.layer = p.layer;
    return ch;
}

// pass 1: grid (slabs, B, channel blocks); a CTA owns the pixels [slab * HW / slabs, ...) of one sample's channel block
template <int VEC>
__global__ void __launch_bounds__(kThreads) gn_bwd_reduce_kernel(const BwdArgs p) {
    extern __shared__ float2 red[];                        // [kThreads][VEC]
    const int b = blockIdx.y, slab = blockIdx.x, tid = threadIdx.x;
    const int CV = p.CB / VEC, PPH = kThreads / CV;
    const int cv = tid % CV, pp = tid / CV, c = blockIdx.z * p.CB + cv * VEC;
    const int p0 = static_cast<int>(static_cast<long long>(slab) * p.HW / p.slabs), p1 = static_cast<int>(static_cast<long long>(slab + 1) * p.HW / p.slabs);
    float a[VEC], bc[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) { a[i] = 0.f; bc[i] = 0.f; }
    if (pp < PPH) {
        const Chain<VEC> ch = make_chain<VEC>(p, b, c);
        for (int pix = p0 + pp; pix < p1; pix += PPH) {
            const size_t off = (static_cast<size_t>(b) * p.HW + pix) * p.C + c;
            float xv[VEC], gv[VEC];
            load_vec<VEC>(p.x + off, xv);
            load_vec<VEC>(p.grad_out + off, gv);
            const Elem<VEC> e = ch.eval(xv, gv, off);
#pragma unroll
            for (int i = 0; i < VEC; ++i) { a[i] += e.dz[i]; bc[i] = fmaf(e.dz[i], e.xhat[i], bc[i]); }
        }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) red[tid * VEC + i] = make_float2(a[i], bc[i]);
    __syncthreads();
    if (tid < CV) {                                        // fixed order over the pixel phases
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float sa = 0.f, sb = 0.f;
            for (int ph = 0; ph < PPH; ++ph) { const float2 t = red[(ph * CV + tid) * VEC + i]; sa += t.x; sb += t.y; }
            p.partial[(static_cast<size_t>(b) * p.slabs + slab) * p.C + c + i] = make_float2(sa, sb);
        }
    }
}

// per sample: slab sums -> ab[b][c], FiLM gradients, group means m1 / m2
__global__ void __launch_bounds__(kThreads) gn_bwd_finalize_kernel(const BwdArgs p) {
    extern __shared__ double2 gsum[];                      // [C] gamma (1 + scale) (A, Bc)
    const int b = blockIdx.x;
    for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
        double sa = 0.0, sb = 0.0;
        for (int s = 0; s < p.slabs; ++s) {
            const float2 t = p.partial[(static_cast<size_t>(b) * p.slabs + s) * p.C + c];
            sa += t.x; sb += t.y;
        }
        p.ab[static_cast<size_t>(b) * p.C + c] = make_float2(static_cast<float>(sa), static_cast<float>(sb));
        const double g = p.gamma[c], be = p.beta[c];
        const double fs = p.film ? 1.0 + p.film[static_cast<size_t>(b) * 2 * p.C + p.C + c] : 1.0;
        if (p.grad_film) {
            p.grad_film[static_cast<size_t>(b) * 2 * p.C + c] = static_cast<float>(sa);                  // d shift
            p.grad_film[static_cast<size_t>(b) * 2 * p.C + p.C + c] = static_cast<float>(g * sb + be * sa);   // d scale
        }
        gsum[c] = make_double2(g * fs * sa, g * fs * sb);
    }
    __syncthreads();
    if (threadIdx.x < kGroups) {
        const int cpg = p.C / kGroups;
        double m1 = 0.0, m2 = 0.0;
        for (int j = 0; j < cpg; ++j) { m1 += gsum[threadIdx.x * cpg + j].x; m2 += gsum[threadIdx.x * cpg + j].y; }
        const double n = static_cast<double>(cpg) * p.HW;
        p.m12[b * kGroups + threadIdx.x] = make_float2(static_cast<float>(m1 / n), static_cast<float>(m2 / n));
    }
}

// d gamma / d beta: one warp per channel, lanes stride over the samples, fixed shuffle tree (deterministic)
__global__ void __launch_bounds__(256) gn_bwd_param_kernel(const BwdArgs p) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= p.C) return;
    double dg = 0.0, db = 0.0;
    for (int b = lane; b < p.B; b += 32) {
        const float2 t = p.ab[static_cast<size_t>(b) * p.C + c];
        const double fs = p.film ? 1.0 + p.film[static_cast<size_t>(b) * 2 * p.C + p.C + c] : 1.0;
        db += fs * t.x; dg += fs * t.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { dg += __shfl_xor_sync(0xffffffffu, dg, o); db += __shfl_xor_sync(0xffffffffu, db, o); }
    if (lane == 0) { p.grad_gamma[c] = static_cast<float>(dg); p.grad_beta[c] = static_cast<float>(db); }
}

// pass 2: dx; grid as pass 1
template <int VEC>
__global__ void __launch_bounds__(kThreads) gn_bwd_apply_kernel(const BwdArgs p) {
    const int b = blockIdx.y, slab = blockIdx.x, tid = threadIdx.x;
    const int CV = p.CB / VEC, PPH = kThreads / CV;
    const int cv = tid % CV, pp = tid / CV, c = blockIdx.z * p.CB + cv * VEC;
    if (pp >= PPH) return;
    const int p0 = static_cast<int>(static_cast<long long>(slab) * p.HW / p.slabs), p1 = static_cast<int>(static_cast<long long>(slab + 1) * p.HW / p.slabs);
    const Chain<VEC> ch = make_chain<VEC>(p, b, c);
    const float2 m = p.m12[b * kGroups + c / (p.C / kGroups)];
    float k[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) k[i] = ch.ga[i] * ch.fs[i];
    for (int pix = p0 + pp; pix < p1; pix += PPH) {
        const size_t off = (static_cast<size_t>(b) * p.HW + pix) * p.C + c;
        float xv[VEC], gv[VEC];
        load_vec<VEC>(p.x + off, xv);
        load_vec<VEC>(p.grad_out + off, gv);
        const Elem<VEC> e = ch.eval(xv, gv, off);
        if constexpr (VEC == 4) {
            float4 o;
            o.x = ch.rstd * (k[0] * e.dz[0] - m.x - e.xhat[0] * m.y);
            o.y = ch.rstd * (k[1] * e.dz[1] - m.x - e.xhat[1] * m.y);
            o.z = ch.rstd * (k[2] * e.dz[2] - m.x - e.xhat[2] * m.y);
            o.w = ch.rstd * (k[3] * e.dz[3] - m.x - e.xhat[3] * m.y);
            *reinterpret_cast<float4*>(p.grad_x + off) = o;
        } else {
            float2 o;
            o.x = ch.rstd * (k[0] * e.dz[0] - m.x - e.xhat[0] * m.y);
            o.y = ch.rstd * (k[1] * e.dz[1] - m.x - e.xhat[1] * m.y);
            *reinterpret_cast<float2*>(p.grad_x + off) = o;
        }
    }
}

// Vector width and channel block of a width C (C % 64 == 0: whole, even-width groups): the fewest channel blocks (whole
// groups, at most kThreads vectors wide) whose pixel-phase rows keep at least 3/4 of a CTA's threads busy.  C = 128, 256,
// 512 and 1024 (four-wide vectors dividing kThreads) take one block, the layout this kernel had before wider C existed.
struct BwdLayout { int vec, cb; };
BwdLayout bwd_layout(int C) {
    const int cpg = C / kGroups, vec = (cpg % 4 == 0) ? 4 : 2;
    int nblk = 1;
    for (; nblk < kGroups; nblk *= 2) {
        const int cv = C / nblk / vec;
        if (cv <= kThreads && (kThreads / cv) * cv * 4 >= kThreads * 3) break;
    }
    return BwdLayout{vec, C / nblk};
}

template <int VEC>
void launch_passes(const BwdArgs& p, const float* x, float2* mr, int nblk, cudaStream_t stream) {
    gn_stats_kernel<VEC><<<dim3(p.B, nblk), kThreads, kThreads * sizeof(float2), stream>>>(x, mr, p.HW, p.C, p.CB);
    gn_bwd_reduce_kernel<VEC><<<dim3(p.slabs, p.B, nblk), kThreads, kThreads * VEC * sizeof(float2), stream>>>(p);
    gn_bwd_finalize_kernel<<<p.B, kThreads, p.C * sizeof(double2), stream>>>(p);
    gn_bwd_param_kernel<<<(p.C + 7) / 8, 256, 0, stream>>>(p);
    gn_bwd_apply_kernel<VEC><<<dim3(p.slabs, p.B, nblk), kThreads, 0, stream>>>(p);
}

}  // namespace

size_t groupnorm_backward_scratch_bytes(int B, int HW, int C, int* slabs_out) {
    int slabs = 1;
    while (slabs < 16 && HW / (slabs * 2) >= 64) slabs *= 2;       // at least 64 pixels per CTA
    if (slabs_out) *slabs_out = slabs;
    return (static_cast<size_t>(B) * slabs * C + static_cast<size_t>(B) * C + 2 * static_cast<size_t>(B) * kGroups) * sizeof(float2);
}

cudaError_t launch_groupnorm_backward(const GroupNormBwdParams& q, cudaStream_t stream) {
    // every width the forward takes from one source: groups of an even channel count, at most 2048 channels
    if (q.C < 2 * kGroups || q.C % (2 * kGroups) != 0 || q.C > 2048) return cudaErrorInvalidValue;
    const BwdLayout lay = bwd_layout(q.C);
    int slabs = 1;
    groupnorm_backward_scratch_bytes(q.B, q.HW, q.C, &slabs);
    BwdArgs p{};
    p.x = q.x; p.grad_out = q.grad_out; p.gamma = q.gamma; p.beta = q.beta; p.film = q.film;
    p.B = q.B; p.HW = q.HW; p.C = q.C; p.CB = lay.cb; p.silu = q.silu; p.slabs = slabs;
    p.drop_p = q.drop_p; p.seed = q.drop_seed; p.layer = q.drop_layer;
    float2* s = static_cast<float2*>(q.scratch);
    p.partial = s; s += static_cast<size_t>(q.B) * slabs * q.C;
    p.ab = s; s += static_cast<size_t>(q.B) * q.C;
    p.m12 = s; s += static_cast<size_t>(q.B) * kGroups;
    float2* mr = s;
    p.meanrstd = mr;
    p.grad_x = q.grad_x; p.grad_gamma = q.grad_gamma; p.grad_beta = q.grad_beta; p.grad_film = q.grad_film;
    const int nblk = q.C / lay.cb;
    if (lay.vec == 4) launch_passes<4>(p, q.x, mr, nblk, stream);
    else launch_passes<2>(p, q.x, mr, nblk, stream);
    return cudaGetLastError();
}

}  // namespace vdt
