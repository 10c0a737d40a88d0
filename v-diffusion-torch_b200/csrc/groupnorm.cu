// Fused GroupNorm(32 groups, eps 1e-6) + optional FiLM (1+scale)*y+shift + optional SiLU + optional
// 2x average-pool / 2x nearest-upsample, fp32 NHWC in -> bf16 NHWC out (the next conv's operand).
//
// Replaces nn.GroupNorm + SiLU + (1+scale)*x+shift + AvgPool2d/Upsample of the reference
// (unet.py:28-30, 119-124, 127-132, 141-146; AttentionBlock.norm unet.py:52,76; out_conv unet.py:229-231)
// and the channel concat feeding it (unet.py:315) by reading two sources.
//
// Statistics: normally the producing conv epilogue has already written per-(32-row slab, 4-channel)
// partial (sum, sum of squares) next to the tensor (ConvParams::stats); a tiny finalize launch combines the
// partials of every image in a fixed order (deterministic, fp64) and the apply kernel is then a single
// streaming pass: read fp32 (or 16-bit) once, write the 16-bit operand once.  Images are split over several CTAs.
// Fallback (groups that are not a multiple of 4 channels, or a concat seam inside a group): one CTA
// per sample makes its own statistics pass first (thread t owns VEC consecutive channels of one
// group and every PPH-th pixel; private fp32 partials combined once through shared memory).
// Optionally also writes the raw concat in 16 bits (operand of the 1x1 skip conv) and the resampled
// raw input in fp32 (identity-skip residual of a resampling block).
#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {
namespace {

constexpr int kGroups = 32;
constexpr float kEps = 1e-6f;

template <int VEC> struct VecT;
template <> struct VecT<4> { typedef float4 type; };
template <> struct VecT<2> { typedef float2 type; };

template <int VEC>
__device__ __forceinline__ void load_vec(const float* p, float (&v)[VEC]) {
    typename VecT<VEC>::type t = __ldg(reinterpret_cast<const typename VecT<VEC>::type*>(p));
    const float* f = reinterpret_cast<const float*>(&t);
#pragma unroll
    for (int i = 0; i < VEC; ++i) v[i] = f[i];
}
// 16-bit source (conv1 output kept in the operand format): VEC == 4 only
__device__ __forceinline__ void load_vec16(const h16* p, float (&v)[4], int f16) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    if (f16) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    } else {
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
}
__device__ __forceinline__ void load_vec16(const h16* p, float (&v)[2], int f16) {
    const uint32_t t = __ldg(reinterpret_cast<const uint32_t*>(p));
    const float2 a = f16 ? __half22float2(*reinterpret_cast<const __half2*>(&t)) : __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t));
    v[0] = a.x; v[1] = a.y;
}

// the same in two steps, so that a deeper batch of loads can stay packed in registers until it is consumed
template <int VEC> struct RawT;
template <> struct RawT<4> { typedef uint2 type; };
template <> struct RawT<2> { typedef uint32_t type; };
__device__ __forceinline__ void unpack16(const uint2& t, float (&v)[4], int f16) {
    if (f16) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    } else {
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
}
__device__ __forceinline__ void unpack16(const uint32_t& t, float (&v)[2], int f16) {
    const float2 a = f16 ? __half22float2(*reinterpret_cast<const __half2*>(&t)) : __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t));
    v[0] = a.x; v[1] = a.y;
}

template <int VEC>
__device__ __forceinline__ void store_16(h16* p, const float (&v)[VEC], int f16) {      // saturating (raw stream values)
    if (VEC == 4) {
        *reinterpret_cast<uint2*>(p) = make_uint2(pack_16(v[0], v[1], f16), pack_16(v[2], v[3], f16));
    } else {
        *reinterpret_cast<uint32_t*>(p) = pack_16(v[0], v[1], f16);
    }
}
template <int VEC>
__device__ __forceinline__ void store_16n(h16* p, const float (&v)[VEC], int f16) {     // normalised values: in range
    if (VEC == 4) {
        *reinterpret_cast<uint2*>(p) = make_uint2(pack_16_inrange(v[0], v[1], f16), pack_16_inrange(v[2], v[3], f16));
    } else {
        *reinterpret_cast<uint32_t*>(p) = pack_16_inrange(v[0], v[1], f16);
    }
}
// hi/lo pair for the split-precision mode: hi = round16(v), lo = round16(v - hi)
template <int VEC>
__device__ __forceinline__ void store_lo(h16* p, const float (&v)[VEC], int f16) {
    float r[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
        const uint16_t h = cvt_16(v[i], f16);
        const float hf = f16 ? __half2float(*reinterpret_cast<const __half*>(&h)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&h));
        r[i] = v[i] - hf;
    }
    if (VEC == 4) {
        *reinterpret_cast<uint2*>(p) = make_uint2(pack_16(r[0], r[1], f16), pack_16(r[2], r[3], f16));
    } else {
        *reinterpret_cast<uint32_t*>(p) = pack_16(r[0], r[1], f16);
    }
}
template <int VEC>
__device__ __forceinline__ void store_f32(float* p, const float (&v)[VEC]) {
    if (VEC == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    }
}

// Combines the conv epilogue's partial statistics of one image into (mean, rstd) of group g: the eight threads
// part8 = 0..7 of an aligned 8-lane group each walk every eighth entry in a fixed order (fp64), then combine with a
// fixed shuffle tree -- deterministic, independent of how the image is split over CTAs.  Works for any channels-per-
// group that is a multiple of stat_cols and for groups that straddle the seam of a channel concat.  All 8 lanes return
// the result.
__device__ __forceinline__ float2 group_mean_rstd(const GroupNormParams& p, int b, int g, int part8) {
    const int C = p.C1 + p.C2, HW = p.H * p.W, cpg = C / kGroups;
    // entries of stat_cols channels; a group may straddle the concat seam, so each entry picks its source
    const int sc = p.stat_cols, sub = cpg / sc, slabs = p.stat_slabs;
    const int e1 = p.C1 / sc, e2 = p.C2 / sc;              // entries per slab in source 1 / 2
    const int b1 = p.rep1 > 1 ? b / p.rep1 : b, b2 = p.rep2 > 1 ? b / p.rep2 : b;     // shared sources (GroupNormParams::rep1)
    const float2* s1 = p.stats1 + static_cast<size_t>(b1) * slabs * e1;
    const float2* s2 = p.stats2 ? p.stats2 + static_cast<size_t>(b2) * slabs * e2 : nullptr;
    double ds = 0.0, dss = 0.0;
    const int ent0 = g * sub;                                // first entry of this group over the concatenated channels
    if (ent0 + sub <= e1 || ent0 >= e1) {
        // the whole group lies in one source (always the case without a concat): plain strided walk
        const bool in1 = ent0 < e1;
        const int es = in1 ? e1 : e2;
        const float2* base = (in1 ? s1 : s2) + (in1 ? ent0 : ent0 - e1);
        for (int e0 = 0; e0 < slabs * sub; e0 += 32) {       // 4 independent loads in flight per thread
            float2 t[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * 8 + part8;
                t[u] = (e < slabs * sub) ? __ldg(base + static_cast<size_t>(e / sub) * es + (e % sub)) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) { ds += t[u].x; dss += t[u].y; }
        }
    } else {
        // the group straddles the concat seam: every entry picks its source
        for (int e = part8; e < slabs * sub; e += 8) {
            const int slab = e / sub, ent = ent0 + (e % sub);
            const float2 t = (ent < e1) ? __ldg(s1 + static_cast<size_t>(slab) * e1 + ent)
                                        : __ldg(s2 + static_cast<size_t>(slab) * e2 + (ent - e1));
            ds += t.x; dss += t.y;
        }
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) { ds += __shfl_xor_sync(0xffffffffu, ds, o); dss += __shfl_xor_sync(0xffffffffu, dss, o); }
    const double n = static_cast<double>(cpg) * HW;
    const double mean = ds / n;
    double var = dss / n - mean * mean;
    if (var < 0.0) var = 0.0;
    return make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + static_cast<double>(kEps))));
}

// One 256-thread CTA per image: (mean, rstd) of the 32 groups from the conv epilogue's partials.  A separate, tiny launch:
// folding this into every CTA of the apply kernel was measured slower (+6 ms per step: the dependent prologue delays each
// CTA's first loads) than the 73 launch latencies it saves.
__global__ void __launch_bounds__(256) groupnorm_finalize_kernel(const GroupNormParams p) {
    const int b = blockIdx.x, tid = threadIdx.x;
    const float2 mr = group_mean_rstd(p, b, tid >> 3, tid & 7);
    if ((tid & 7) == 0) p.meanrstd[b * kGroups + (tid >> 3)] = mr;
}

template <int VEC, bool FUSED, bool IN16, bool F16>
__global__ void __launch_bounds__(1024, 1) groupnorm_kernel(const GroupNormParams p, int CV, int PPH) {
    extern __shared__ float2 part[];                 // [CV * PPH] partial (sum, sumsq) (fallback statistics pass)
    __shared__ float2 stat[kGroups];
    const int b = blockIdx.x;
    const int C = p.C1 + p.C2;
    const int HW = p.H * p.W;
    const int cpg = C / kGroups;
    const int tid = threadIdx.x;
    const bool active = tid < CV * PPH;
    const int cv = active ? tid % CV : 0;
    const int pp = active ? tid / CV : 0;
    const int c = cv * VEC;                          // first channel owned by this thread
    const bool from1 = c < p.C1;
    const int b1 = p.rep1 > 1 ? b / p.rep1 : b, b2 = p.rep2 > 1 ? b / p.rep2 : b;     // rows that share a source image
    const float* src = from1 ? static_cast<const float*>(p.src1) + static_cast<size_t>(b1) * HW * p.C1 + c
                             : p.src2 + static_cast<size_t>(b2) * HW * p.C2 + (c - p.C1);
    const h16* src16 = static_cast<const h16*>(p.src1) + static_cast<size_t>(b1) * HW * p.C1 + c;   // IN16 only
    const int sC = from1 ? p.C1 : p.C2;
    float amax = 0.f;                                // fp16 range events seen by this thread (see GroupNormParams::sat_count)
    auto load_px = [&](int pix, float (&v)[VEC]) {
        if (IN16) {
            load_vec16(src16 + static_cast<size_t>(pix) * sC, v, (F16 ? 1 : 0));
            if (F16) {
#pragma unroll
                for (int i = 0; i < VEC; ++i) amax = fmaxf(amax, fabsf(v[i]));
            }
        } else {
            load_vec<VEC>(src + static_cast<size_t>(pix) * sC, v);
        }
    };

    // ---- fallback pass 1: statistics
    float s = 0.f, ss = 0.f;
    if (!FUSED && active) {
        int pix = pp;
        for (; pix + 3 * PPH < HW; pix += 4 * PPH) {
            float v0[VEC], v1[VEC], v2[VEC], v3[VEC];
            load_vec<VEC>(src + static_cast<size_t>(pix) * sC, v0);
            load_vec<VEC>(src + static_cast<size_t>(pix + PPH) * sC, v1);
            load_vec<VEC>(src + static_cast<size_t>(pix + 2 * PPH) * sC, v2);
            load_vec<VEC>(src + static_cast<size_t>(pix + 3 * PPH) * sC, v3);
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                s += (v0[i] + v1[i]) + (v2[i] + v3[i]);
                ss += (v0[i] * v0[i] + v1[i] * v1[i]) + (v2[i] * v2[i] + v3[i] * v3[i]);
            }
        }
        for (; pix < HW; pix += PPH) {
            float v0[VEC];
            load_vec<VEC>(src + static_cast<size_t>(pix) * sC, v0);
#pragma unroll
            for (int i = 0; i < VEC; ++i) { s += v0[i]; ss += v0[i] * v0[i]; }
        }
        part[tid] = make_float2(s, ss);
    }
    if (!FUSED) __syncthreads();
    if (!FUSED && tid < kGroups) {
        const int vpg = cpg / VEC;                   // vectors per group per pixel
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
        stat[tid] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + static_cast<double>(kEps))));
    }
    if (!FUSED) __syncthreads();
    if (!active) return;

    // ---- pass 2: apply
    const float2 st = FUSED ? __ldg(p.meanrstd + b * kGroups + c / cpg) : stat[c / cpg];
    float ga[VEC], be[VEC], fs[VEC], fb[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
        const float g = __ldg(p.gamma + c + i) * st.y;
        ga[i] = g;
        be[i] = __ldg(p.beta + c + i) - st.x * g;
        fs[i] = 1.f; fb[i] = 0.f;
    }
    if (p.film) {
        const int r = p.film_row ? __ldg(p.film_row + b) : b;
        const float* f = p.film + static_cast<size_t>(r) * p.film_stride + p.film_off;
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            fb[i] = __ldg(f + c + i);                // shift first, scale second (unet.py:145)
            fs[i] = 1.f + __ldg(f + C + c + i);
        }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) { ga[i] *= fs[i]; be[i] = be[i] * fs[i] + fb[i]; }

    auto norm_act = [&](const float (&x)[VEC], float (&y)[VEC]) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const float t = x[i] * ga[i] + be[i];
            y[i] = p.silu ? __fdividef(t, 1.f + __expf(-t)) : t;     // 16-bit output: fast-math error is far below its rounding
        }
    };

    // training dropout (only ever on an un-resampled norm2 output): one Philox call per (pixel, 4-channel vector)
    const bool drop = p.drop_p > 0.f;
    const uint32_t drop_thr = drop ? static_cast<uint32_t>(fminf(p.drop_p, 0.99999994f) * 4294967296.0f) : 0u;
    const float drop_scale = drop ? 1.f / (1.f - p.drop_p) : 1.f;
    const unsigned long long dseed = drop ? *p.drop_seed : 0ull;
    auto dropout = [&](float (&y)[VEC], int pix) {
        const unsigned long long e = (static_cast<unsigned long long>(b) * HW + pix) * C + c;      // first element of the vector
        const uint4 r = philox4x32(make_uint4(static_cast<uint32_t>(e >> 2), static_cast<uint32_t>(e >> 34), static_cast<uint32_t>(p.drop_layer), 0x44524f50u),
                                   make_uint2(static_cast<uint32_t>(dseed), static_cast<uint32_t>(dseed >> 32)));
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < VEC; ++i) y[i] = (w[(VEC == 4) ? i : ((c >> 1) & 1) * 2 + i] < drop_thr) ? 0.f : y[i] * drop_scale;
    };

    if (p.resample == kResDown) {
        const int Wo = p.W / 2, HWo = HW / 4;
        h16* oa = p.out_act + static_cast<size_t>(b) * HWo * C + c;
        h16* oa_lo = p.out_act_lo ? p.out_act_lo + static_cast<size_t>(b) * HWo * C + c : nullptr;
        float* orr = p.out_res ? p.out_res + static_cast<size_t>(b) * HWo * C + c : nullptr;
        for (int po = pp; po < HWo; po += PPH) {
            const int ho = po / Wo, wo = po % Wo;
            float acc[VEC], racc[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) { acc[i] = 0.f; racc[i] = 0.f; }
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const int pix = (2 * ho + (d >> 1)) * p.W + 2 * wo + (d & 1);
                float x[VEC], y[VEC];
                load_px(pix, x);
                norm_act(x, y);
#pragma unroll
                for (int i = 0; i < VEC; ++i) { acc[i] += y[i]; racc[i] += x[i]; }
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) { acc[i] *= 0.25f; racc[i] *= 0.25f; }
            store_16n<VEC>(oa + static_cast<size_t>(po) * C, acc, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(po) * C, acc, (F16 ? 1 : 0));
            if (orr) store_f32<VEC>(orr + static_cast<size_t>(po) * C, racc);
        }
    } else if (p.resample == kResUp) {
        const int Wo = p.W * 2;
        h16* oa = p.out_act + static_cast<size_t>(b) * HW * 4 * C + c;
        h16* oa_lo = p.out_act_lo ? p.out_act_lo + static_cast<size_t>(b) * HW * 4 * C + c : nullptr;
        float* orr = p.out_res ? p.out_res + static_cast<size_t>(b) * HW * 4 * C + c : nullptr;
        for (int pix = pp; pix < HW; pix += PPH) {
            const int h = pix / p.W, w = pix % p.W;
            float x[VEC], y[VEC];
            load_px(pix, x);
            norm_act(x, y);
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const size_t po = static_cast<size_t>(2 * h + (d >> 1)) * Wo + 2 * w + (d & 1);
                store_16n<VEC>(oa + po * C, y, (F16 ? 1 : 0));
                if (oa_lo) store_lo<VEC>(oa_lo + po * C, y, (F16 ? 1 : 0));
                if (orr) store_f32<VEC>(orr + po * C, x);
            }
        }
    } else {
        h16* oa = p.out_act + static_cast<size_t>(b) * HW * C + c;
        h16* oa_lo = p.out_act_lo ? p.out_act_lo + static_cast<size_t>(b) * HW * C + c : nullptr;
        h16* ow = p.out_raw ? p.out_raw + static_cast<size_t>(b) * HW * C + c : nullptr;
        h16* ow_lo = (p.out_raw && p.out_raw_lo) ? p.out_raw_lo + static_cast<size_t>(b) * HW * C + c : nullptr;
        // FUSED: the image is split over gridDim.y CTAs
        const int span = HW / gridDim.y, pix_end = (blockIdx.y + 1) * span;
        int pix = blockIdx.y * span + pp;
        if (IN16 && !ow && !oa_lo) {
            // 16-bit input: eight 8-byte loads in flight per thread, kept packed (16 registers) until consumed --
            // the 4-deep loop below leaves this variant latency-bound at ~2/3 of the HBM rate
            typedef typename RawT<VEC>::type raw_t;
            for (; pix + 7 * PPH < pix_end; pix += 8 * PPH) {
                raw_t r[8];
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    r[u] = __ldg(reinterpret_cast<const raw_t*>(src16 + static_cast<size_t>(pix + u * PPH) * sC));
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    float x[VEC], y[VEC];
                    unpack16(r[u], x, (F16 ? 1 : 0));
                    if (F16) {
#pragma unroll
                        for (int i = 0; i < VEC; ++i) amax = fmaxf(amax, fabsf(x[i]));
                    }
                    norm_act(x, y);
                    if (drop) dropout(y, pix + u * PPH);
                    store_16n<VEC>(oa + static_cast<size_t>(pix + u * PPH) * C, y, (F16 ? 1 : 0));
                }
            }
        }
        for (; pix + 3 * PPH < pix_end; pix += 4 * PPH) {     // four independent 16-byte loads in flight per thread
            float x0[VEC], x1[VEC], x2[VEC], x3[VEC], y[VEC];
            load_px(pix, x0);
            load_px(pix + PPH, x1);
            load_px(pix + 2 * PPH, x2);
            load_px(pix + 3 * PPH, x3);
            norm_act(x0, y); if (drop) dropout(y, pix); store_16n<VEC>(oa + static_cast<size_t>(pix) * C, y, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(pix) * C, y, (F16 ? 1 : 0));
            norm_act(x1, y); if (drop) dropout(y, pix + PPH); store_16n<VEC>(oa + static_cast<size_t>(pix + PPH) * C, y, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(pix + PPH) * C, y, (F16 ? 1 : 0));
            norm_act(x2, y); if (drop) dropout(y, pix + 2 * PPH); store_16n<VEC>(oa + static_cast<size_t>(pix + 2 * PPH) * C, y, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(pix + 2 * PPH) * C, y, (F16 ? 1 : 0));
            norm_act(x3, y); if (drop) dropout(y, pix + 3 * PPH); store_16n<VEC>(oa + static_cast<size_t>(pix + 3 * PPH) * C, y, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(pix + 3 * PPH) * C, y, (F16 ? 1 : 0));
            if (ow) {
                if (F16) {
#pragma unroll
                    for (int i = 0; i < VEC; ++i) amax = fmaxf(fmaxf(amax, fmaxf(fabsf(x0[i]), fabsf(x1[i]))), fmaxf(fabsf(x2[i]), fabsf(x3[i])));
                }
                store_16<VEC>(ow + static_cast<size_t>(pix) * C, x0, (F16 ? 1 : 0));
                if (ow_lo) store_lo<VEC>(ow_lo + static_cast<size_t>(pix) * C, x0, (F16 ? 1 : 0));
                store_16<VEC>(ow + static_cast<size_t>(pix + PPH) * C, x1, (F16 ? 1 : 0));
                if (ow_lo) store_lo<VEC>(ow_lo + static_cast<size_t>(pix + PPH) * C, x1, (F16 ? 1 : 0));
                store_16<VEC>(ow + static_cast<size_t>(pix + 2 * PPH) * C, x2, (F16 ? 1 : 0));
                if (ow_lo) store_lo<VEC>(ow_lo + static_cast<size_t>(pix + 2 * PPH) * C, x2, (F16 ? 1 : 0));
                store_16<VEC>(ow + static_cast<size_t>(pix + 3 * PPH) * C, x3, (F16 ? 1 : 0));
                if (ow_lo) store_lo<VEC>(ow_lo + static_cast<size_t>(pix + 3 * PPH) * C, x3, (F16 ? 1 : 0));
            }
        }
        for (; pix < pix_end; pix += PPH) {
            float x0[VEC], y0[VEC];
            load_px(pix, x0);
            norm_act(x0, y0);
            if (drop) dropout(y0, pix);
            store_16n<VEC>(oa + static_cast<size_t>(pix) * C, y0, (F16 ? 1 : 0));
            if (oa_lo) store_lo<VEC>(oa_lo + static_cast<size_t>(pix) * C, y0, (F16 ? 1 : 0));
            if (ow) {
                if (F16) {
#pragma unroll
                    for (int i = 0; i < VEC; ++i) amax = fmaxf(amax, fabsf(x0[i]));
                }
                store_16<VEC>(ow + static_cast<size_t>(pix) * C, x0, (F16 ? 1 : 0));
            }
            if (ow_lo) store_lo<VEC>(ow_lo + static_cast<size_t>(pix) * C, x0, (F16 ? 1 : 0));
        }
    }
    // a 16-bit input that sits at the fp16 maximum was clamped by the conv epilogue that wrote it; a raw stream value
    // above it was clamped by out_raw's conversion just now
    if (F16 && p.sat_count != nullptr && amax >= 65504.f) atomicAdd(p.sat_count, 1ull);
}

}  // namespace

cudaError_t launch_groupnorm(const GroupNormParams& p, cudaStream_t stream) {
    const int C = p.C1 + p.C2;
    if (C % kGroups != 0 || p.B <= 0) return cudaErrorInvalidValue;
    const int cpg = C / kGroups;
    const int vec = (cpg % 4 == 0 && p.C1 % 4 == 0) ? 4 : 2;
    if (cpg % vec != 0 || p.C1 % vec != 0) return cudaErrorInvalidValue;
    const int CV = C / vec;
    if (CV > 1024) return cudaErrorInvalidValue;
    const int HW = p.H * p.W;
    const bool fused = p.stats1 != nullptr;
    if (fused && (p.stat_slabs != stat_slabs_per_image(p.H, p.W) || p.stat_slabs <= 0 || (p.stat_cols != 2 && p.stat_cols != 4) || cpg % p.stat_cols != 0 ||
                  p.C1 % p.stat_cols != 0 || (p.C2 > 0 && p.stats2 == nullptr))) return cudaErrorInvalidValue;
    if (p.in16 && (p.C2 != 0 || !fused)) return cudaErrorInvalidValue;
    if (p.drop_p > 0.f && (p.resample != kResNone || p.drop_seed == nullptr || p.drop_p >= 1.f)) return cudaErrorInvalidValue;
    // threads per CTA: 256 (16 K registers, ~1 KB of shared memory), so that a GroupNorm CTA fits on an SM next to a
    // resident conv / attention CTA of the other lane (plan.cu: vdt_plan::kLanes)
    constexpr int max_threads = 256;
    int PPH = (max_threads > CV ? max_threads : CV) / CV;
    const int work = (p.resample == kResDown) ? HW / 4 : HW;
    if (PPH > work) PPH = work;
    if (PPH > 8) PPH = 8;                             // >= 8 pixels of work per thread at 32x32 / 256 ch
    if (PPH < 1) PPH = 1;
    int threads = ((CV * PPH + 31) / 32) * 32;
    const size_t smem = fused ? 0 : static_cast<size_t>(CV) * PPH * sizeof(float2);
    // split an image over several CTAs when the statistics are already known (no resampling: pixel ranges are trivial)
    int split = 1;
    if (fused && p.resample == kResNone)
        while (split < 8 && (HW / (split * 2)) >= 2 * PPH * 8 && (HW % (split * 2)) == 0) split *= 2;
    dim3 grid(p.B, split);
    // the 16-bit format is a template parameter: the kernel is issue-bound, and a run-time format flag costs a
    // second conversion plus a select per packed pair
    if (fused) {
        if (p.meanrstd == nullptr) return cudaErrorInvalidValue;
        groupnorm_finalize_kernel<<<p.B, 256, 0, stream>>>(p);
        if (vec == 4) {
            if (p.in16 && p.f16) groupnorm_kernel<4, true, true, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else if (p.in16) groupnorm_kernel<4, true, true, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else if (p.f16) groupnorm_kernel<4, true, false, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else groupnorm_kernel<4, true, false, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
        } else {
            if (p.in16 && p.f16) groupnorm_kernel<2, true, true, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else if (p.in16) groupnorm_kernel<2, true, true, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else if (p.f16) groupnorm_kernel<2, true, false, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
            else groupnorm_kernel<2, true, false, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
        }
    } else if (vec == 4) {
        if (p.f16) groupnorm_kernel<4, false, false, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
        else groupnorm_kernel<4, false, false, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
    } else {
        if (p.f16) groupnorm_kernel<2, false, false, true><<<grid, threads, smem, stream>>>(p, CV, PPH);
        else groupnorm_kernel<2, false, false, false><<<grid, threads, smem, stream>>>(p, CV, PPH);
    }
    return cudaGetLastError();
}

}  // namespace vdt
