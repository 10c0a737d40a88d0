// Device helpers shared by the sampler kernels (pointwise.cu) and the likelihood kernels (bpd.cu).
#pragma once
#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {
namespace {

// Philox4x32-10 counter RNG + Box-Muller for on-device ancestral noise (used only when no noise
// tensor is injected; the stream is this library's own, not torch's).  One counter value yields the four
// normals of elements 4q .. 4q+3.  Counter word 3 selects the stream: 0 ancestral noise, 1 inpainting's z', 2 the
// likelihood evaluation's q-sample draws.
__device__ __forceinline__ float4 philox_normal4(unsigned long long seed, uint32_t step, unsigned long long quad,
                                                 uint32_t stream = 0u) {
    const uint4 r = philox4x32(make_uint4(static_cast<uint32_t>(quad), static_cast<uint32_t>(quad >> 32), step, stream),
                               make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32)));
    const float k = 1.0f / 16777216.0f;
    const float u1 = (static_cast<float>(r.x >> 8) + 0.5f) * k, u2 = (static_cast<float>(r.y >> 8) + 0.5f) * k;
    const float u3 = (static_cast<float>(r.z >> 8) + 0.5f) * k, u4 = (static_cast<float>(r.w >> 8) + 0.5f) * k;
    const float ra = sqrtf(-2.0f * logf(u1)), rb = sqrtf(-2.0f * logf(u3));
    float sa, ca, sb, cb;
    sincosf(6.283185307179586f * u2, &sa, &ca);
    sincosf(6.283185307179586f * u4, &sb, &cb);
    return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
}

// x0 from the raw model output, unclipped: the inversion step needs it so (a clip would make the step impossible to invert)
__device__ __forceinline__ float pred_x0_raw(int type, float x, float o, float o2, const float* cf) {
    float x0;
    if (type == 3) x0 = x * cf[0] - o * cf[1];                       // v   (diffusion.py:233-234)
    else if (type == 0) x0 = o;                                      // x0
    else if (type == 1) x0 = x * cf[2] - o * cf[3];                  // eps (diffusion.py:207-208)
    else { const float xe = x * cf[2] - o2 * cf[3]; x0 = o * cf[5] + xe * cf[4]; }   // both (211-214)
    return x0;
}

}  // namespace
}  // namespace vdt
