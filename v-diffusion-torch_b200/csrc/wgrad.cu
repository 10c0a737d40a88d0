// Weight gradient of a 3x3 (pad 1) or 1x1 convolution on tcgen05 -- backward half of F.conv2d with respect to the
// weight (modules.py:141-144 under autograd), first slice of the training step (SURVEY §8 f2):
//
//   dW[co][ci][tap] = sum over pixels p of dY[p][co] * X[p + shift(tap)][ci]          (zero padding outside the image)
//
// One GEMM per filter tap with the PIXELS as the contraction dimension.  Both tensors are NHWC, so for this product
// both operands are MN-major (the output-channel / input-channel index is the contiguous one, pixels are the rows):
// the same TMA boxes the forward conv uses for its A operand land as 128-byte-swizzled [pixel][64 channels] tiles, and
// UMMA reads them through MN-major descriptors (tcgen05 transposes on the fly; nothing is transposed in memory).
//
// Work item = (block of 128 output channels, block of <= 256 input channels, group of <= 2 taps, K split): the CTA walks
// its share of the (up to) 128-pixel tiles; per tile the dY tile is fetched once and one X tile per tap (shifted box, out-of-
// bounds zero fill = padding); the two taps' 128 x 256 fp32 accumulators fill TMEM's 512 columns.  Partial sums go to
// partial[split][tap][co][ci]; a second kernel adds the splits in a fixed order (deterministic) and writes OIHW.
//
// Cout % 128 == 64 (192, 576, ...): the last output-channel block holds 64 channels.  Its CTAs never load the second
// 64-channel dY chunk; that chunk's shared memory is zeroed once in both stages, so the M = 128 MMA multiplies zero rows
// (half of that block's tensor work is spent on zeros) and the epilogue warps of the missing channels write nothing.
//
// Ragged K tiles (28x28, 14x14, 7x7, 24x24, 5x5 ...: the forward conv's box holds rows_per_tile < 128 pixels): the pixels
// are the contraction, so a stale row would be multiplied into every dW entry (in both operands: 0 * NaN is NaN).  Rows
// rows_per_tile .. 127 of every dY and X chunk are zeroed once per CTA in both stages: TMA fills exactly rows_per_tile rows
// and never touches them, and zeroing whole 128-byte rows commutes with the 128B swizzle, which permutes 16-byte pieces
// within a row.  Each tap issues ceil(rows_per_tile / 16) MMAs instead of 8.  Boxes past the batch end are zero-filled by
// TMA, as in the forward conv.
//
//   warp 0   TMA producer      warp 1   MMA issuer      warps 2-5   epilogue (TMEM -> partial sums)
#include <atomic>

#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {
namespace {

constexpr int kPix = 128;                        // pixels per K tile (one TMA box of whole image rows / images)
constexpr int kChunk = kPix * 128;               // bytes of one [128 pixels][64 channels] tile
constexpr int kABytes = 2 * kChunk;              // dY tile: 128 output channels
constexpr int kBBytesMax = 4 * kChunk;           // X tile: up to 256 input channels
constexpr int kWgThreads = 32 * 6;
constexpr int kWgSmem = 2 * kABytes + 2 * kBBytesMax + 1024 + 256;

// kRagged: rows_per_tile < kPix.  A separate instantiation, so full tiles keep their instruction stream unchanged
template <bool F16, bool kRagged>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_kernel(const __grid_constant__ WgradParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* a_smem = smem;                                   // [2][kABytes]
    uint8_t* b_smem = smem + 2 * kABytes;                     // [2][kBBytesMax]
    uint64_t* bars = reinterpret_cast<uint64_t*>(b_smem + 2 * kBBytesMax);
    uint64_t *a_full = bars, *a_empty = bars + 2, *b_full = bars + 4, *b_empty = bars + 6, *acc_full = bars + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // blockIdx.x -> (split, tap group, ci block, co block)
    int w = blockIdx.x;
    const int co_blk = w % p.co_blocks; w /= p.co_blocks;
    const int ci_blk = w % p.ci_blocks; w /= p.ci_blocks;
    const int tg = w % p.tap_groups; w /= p.tap_groups;
    const int split = w;
    const int tap0 = tg * 2, ntaps = min(2, p.taps - tap0);
    const int t_begin = static_cast<int>(static_cast<long long>(split) * p.num_tiles / p.splits);
    const int t_end = static_cast<int>(static_cast<long long>(split + 1) * p.num_tiles / p.splits);
    const int bn = p.ci_block, bchunks = bn / 64;
    const int achunks = (co_blk * 128 + 128 <= p.Cout) ? 2 : 1;         // 1: tail block of 64 output channels

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        mbar_init(acc_full, 1);
        fence_mbar_init();
        tma_prefetch_desc(&p.dy_map); tma_prefetch_desc(&p.x_map);
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    if (achunks == 1) {                                       // zero rows for the missing 64 output channels, both stages
        for (int i = threadIdx.x; i < kChunk / 16; i += blockDim.x) {
            reinterpret_cast<uint4*>(a_smem + kChunk)[i] = make_uint4(0u, 0u, 0u, 0u);
            reinterpret_cast<uint4*>(a_smem + kABytes + kChunk)[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        fence_proxy_async_smem();                             // generic-proxy writes -> visible to UMMA after the barrier
    }
    if (kRagged) {                                            // zero pixel rows rows_per_tile .. 127 of every loaded chunk
        const int tail16 = (kPix - p.rows_per_tile) * 8;      // 16-byte pieces per chunk
        const int per_stage = achunks + bchunks;              // dY chunks (a missing one is zeroed whole above) + X chunks
        for (int i = threadIdx.x; i < 2 * per_stage * tail16; i += blockDim.x) {
            const int c = i / tail16, s = c / per_stage, j = c % per_stage;
            uint8_t* chunk = (j < achunks) ? a_smem + s * kABytes + j * kChunk : b_smem + s * kBBytesMax + (j - achunks) * kChunk;
            reinterpret_cast<uint4*>(chunk + p.rows_per_tile * 128)[i % tail16] = make_uint4(0u, 0u, 0u, 0u);
        }
        fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        {   // warp-uniform loop; one elected lane issues the copies
            int ia = 0, ib = 0;
            for (int t = t_begin; t < t_end; ++t, ++ia) {
                const int y0 = (t % p.tiles_per_image) * p.box_h, n0 = (t / p.tiles_per_image) * p.box_n;
                const int sa = ia & 1;
                mbar_wait(&a_empty[sa], ((ia >> 1) & 1) ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(&a_full[sa], static_cast<uint32_t>(achunks * p.rows_per_tile * 128));
                    for (int c = 0; c < achunks; ++c)
                        tma_load_4d(a_smem + sa * kABytes + c * kChunk, &p.dy_map, &a_full[sa], co_blk * 128 + c * 64, 0, y0, n0);
                }
                __syncwarp();
                for (int k = 0; k < ntaps; ++k, ++ib) {
                    const int tap = tap0 + k;
                    const int dy = (p.taps == 9) ? tap / 3 - 1 : 0, dx = (p.taps == 9) ? tap % 3 - 1 : 0;
                    const int sb = ib & 1;
                    mbar_wait(&b_empty[sb], ((ib >> 1) & 1) ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(&b_full[sb], static_cast<uint32_t>(bchunks * p.rows_per_tile * 128));
                        for (int c = 0; c < bchunks; ++c)
                            tma_load_4d(b_smem + sb * kBBytesMax + c * kChunk, &p.x_map, &b_full[sb], ci_blk * bn + c * 64, dx, y0 + dy, n0);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        {
            // D[co 128][ci bn] += A^T B with A = dY tile, B = X tile, both MN-major (bits 15 / 16 of the descriptor).  The whole
            // warp walks the loop; one elected lane issues each instruction (ptx.cuh: elect_one)
            const uint32_t idesc = umma_idesc_16(128, bn, (F16 ? 1 : 0)) | kIdescBMajorMN | (1u << 15);
            const int kmma = kRagged ? (p.rows_per_tile + 15) / 16 : kPix / 16;
            int ia = 0, ib = 0;
            for (int t = t_begin; t < t_end; ++t, ++ia) {
                const int sa = ia & 1;
                mbar_wait(&a_full[sa], (ia >> 1) & 1);
                tc_fence_after();
                for (int k = 0; k < ntaps; ++k, ++ib) {
                    const int sb = ib & 1;
                    mbar_wait(&b_full[sb], (ib >> 1) & 1);
                    tc_fence_after();
                    const uint64_t adesc = umma_desc_sw128_mn(smem_u32(a_smem + sa * kABytes), kChunk);
                    const uint64_t bdesc = umma_desc_sw128_mn(smem_u32(b_smem + sb * kBBytesMax), kChunk);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < kmma; ++kk)        // 16 pixels per MMA: +2048 bytes (= 128 descriptor units) in both operands
                            umma_16(tmem_base + static_cast<uint32_t>(k * 256), adesc + static_cast<uint64_t>(kk * 128),
                                    bdesc + static_cast<uint64_t>(kk * 128), idesc, (t > t_begin || kk > 0) ? 1u : 0u);
                        umma_commit(&b_empty[sb]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(&a_empty[sa]);
                __syncwarp();
            }
            if (elect_one()) umma_commit(acc_full);
            __syncwarp();
        }
    } else {
        // ---- epilogue: warp q reads TMEM lanes 32q .. 32q+31 (= output channels), 32 input channels at a time
        const int q = warp & 3;
        mbar_wait(acc_full, 0);
        tc_fence_after();
        if (t_end > t_begin && co_blk * 128 + q * 32 < p.Cout) {     // TMEM lanes of the tail block's missing channels: none
            const int co = co_blk * 128 + q * 32 + lane;
            for (int k = 0; k < ntaps; ++k) {
                float* dst = p.partial + ((static_cast<size_t>(split) * p.taps + tap0 + k) * p.Cout + co) * p.Cin + ci_blk * bn;
                for (int c0 = 0; c0 < bn; c0 += 32) {
                    uint32_t r[32];
                    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(k * 256 + c0), r);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4*>(dst + c0 + 4 * j) = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                                                                                  __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// dW[co][ci][tap] = sum over splits (fixed order) of partial[split][tap][co][ci]; splits that walked no tile wrote nothing
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits, int taps, int Cout, int Cin,
                                    int num_tiles) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long n = static_cast<long long>(taps) * Cout * Cin;
    if (idx >= n) return;
    const int ci = static_cast<int>(idx % Cin);
    const int co = static_cast<int>((idx / Cin) % Cout);
    const int tap = static_cast<int>(idx / (static_cast<long long>(Cin) * Cout));
    float s = 0.f;
    for (int k = 0; k < splits; ++k) {
        const long long b = static_cast<long long>(k) * num_tiles / splits, e = static_cast<long long>(k + 1) * num_tiles / splits;
        if (e > b) s += partial[(static_cast<size_t>(k) * taps + tap) * Cout * Cin + static_cast<size_t>(co) * Cin + ci];
    }
    dw[(static_cast<size_t>(co) * Cin + ci) * taps + tap] = s;
}

// db[co] = sum over pixels of dY[p][co]   (bias gradient; one warp per 32 channels x a slice of the rows, then a fixed-order add)
__global__ void __launch_bounds__(256) bias_grad_kernel(const h16* __restrict__ dy, float* __restrict__ db, long long rows, int Cout, int f16) {
    __shared__ float red[8][32];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31), wq = threadIdx.x >> 5;
    float s = 0.f;
    if (c < Cout)
        for (long long r = wq; r < rows; r += 8) {
            const h16 v = dy[r * Cout + c];
            s += f16 ? __half2float(*reinterpret_cast<const __half*>(&v)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&v));
        }
    red[wq][threadIdx.x & 31] = s;
    __syncthreads();
    if (wq == 0 && c < Cout) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
        db[c] = t;
    }
}

}  // namespace

int wgrad_splits(const WgradParams& p, int num_sms) {
    const int types = p.co_blocks * p.ci_blocks * p.tap_groups;
    int s = num_sms / (types > 0 ? types : 1);
    if (s < 1) s = 1;
    if (s > p.num_tiles) s = p.num_tiles;
    return s;
}

cudaError_t launch_wgrad(const WgradParams& p, float* dw, float* dbias, const h16* dy, long long rows, cudaStream_t stream) {
    static std::atomic<bool> attr_set[kMaxDevices];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(wgrad_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem);
        if (e != cudaSuccess) return e;
        attr_set[dev].store(true, std::memory_order_release);
    }
    const int grid = p.co_blocks * p.ci_blocks * p.tap_groups * p.splits;
    if (grid <= 0 || p.num_tiles <= 0) return cudaErrorInvalidValue;
    const bool ragged = p.rows_per_tile < kPix;
    void (*kernel)(WgradParams) = p.f16 ? (ragged ? wgrad_kernel<true, true> : wgrad_kernel<true, false>)
                                        : (ragged ? wgrad_kernel<false, true> : wgrad_kernel<false, false>);
    kernel<<<grid, kWgThreads, kWgSmem, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const long long n = static_cast<long long>(p.taps) * p.Cout * p.Cin;
    wgrad_reduce_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(p.partial, dw, p.splits, p.taps, p.Cout, p.Cin, p.num_tiles);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (dbias) {
        bias_grad_kernel<<<(p.Cout + 31) / 32, 256, 0, stream>>>(dy, dbias, rows, p.Cout, p.f16);
        e = cudaGetLastError();
    }
    return e;
}

}  // namespace vdt
