// Fused self-attention for sm_100a: softmax(q^T k / sqrt(d)) v per image and head, flash-style.
//
// Replaces BaseAttentionBlock.scaled_dot_product (unet.py:55-64: two einsums + a softmax that
// materialise the N x N score matrix in HBM).  A work item is 128 query rows of one image and head
// (two whole images when N = 64); S = Q K^T and O += P V run on tcgen05 with S and O resident in TMEM,
// the softmax runs in registers (two threads per query row, fp32, exp2 with the 1/sqrt(d) scale folded
// in), P is re-quantised to 16 bits into swizzled shared memory as the A operand of the second MMA.
// O is rescaled lazily (only when a row maximum grows by more than 2^8), so the TMEM round trip is rare.
//
// Operand (written row-major by the proj_in GEMM epilogue): QKV 16-bit [B*N, 3*hid] = q | k | v with the
// heads contiguous inside each third (unet.py:76-78).  Q and K tiles are K-major operands as stored; a V
// tile [64 keys][d] is the B operand of P V in MN-major form (d contiguous), so no transposed copy of V
// is ever written.
//
// Persistent: one CTA per SM loops over work items.  TMEM is allocated and the barriers are initialised
// once; the K / V rings and the S / P buffers run on across items, the next item's Q is fetched as soon
// as the current item's last S = Q K^T has retired, and its first two S tiles are issued while the
// softmax warps are still finishing the current item (per-CTA set-up used to cost ~10 us per 128 rows).
//
//   warp 0     TMA producer for Q (per item) and the 64-key K tiles (ring slot freed when S retires)
//   warp 10    TMA producer for the V tiles (ring slot freed when O += P V retires)
//   warp 1     MMA issuer
//   warps 2-9  softmax + final normalise/store: two threads per query row (= TMEM lane), each owning 32
//              of the tile's 64 key columns (and half of O's columns); row maxima are exchanged through
//              shared memory once per tile between the two warps that share a TMEM lane quarter
#include <atomic>

#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {
namespace {

constexpr int kQRows = 128;
constexpr int kKeys = 64;                      // keys per tile = one 128-byte swizzle row of P
constexpr int kThreads = 64 + 256 + 32;
constexpr float kRescaleThreshold = 8.0f;      // log2 units

constexpr int kStages = 2;                     // K / V ring stages
struct Smem {          // stage pointers are computed, not indexed (no local-memory arrays)
    uint8_t* q; uint8_t* k0; uint8_t* v0; uint8_t* p0;
    int kv_stride;
    uint64_t *q_full, *q_empty, *k_full, *v_full, *k_empty, *v_empty, *s_full, *p_full, *o_empty;   // k_/v_ arrays: [kStages]
    uint32_t* tmem_slot;
    __device__ __forceinline__ uint8_t* k(int s) const { return k0 + s * kv_stride; }
    __device__ __forceinline__ uint8_t* v(int s) const { return v0 + s * kv_stride; }
    __device__ __forceinline__ uint8_t* p(int s) const { return p0 + s * 16384; }
};

__host__ __device__ inline int attn_smem_bytes(int d) {
    // Q d/64 x 16K | K ring d/64 x 16K | V ring d/64 x 16K | P 2 x 16K | barriers | row max / sum exchange
    // (ring = 2 stages of d/64 x 8K)
    return (d / 64) * 16384 + 4 * (d / 64) * 8192 + 2 * 16384 + 256 + 2048;
}

struct Item { int b0, h, qt; };
__device__ __forceinline__ Item decode_item(int w, int qtiles, int heads, int ipc) {
    Item it;
    it.qt = w % qtiles;
    it.h = (w / qtiles) % heads;
    it.b0 = (w / (qtiles * heads)) * ipc;
    return it;
}

template <bool F16>
__global__ void __launch_bounds__(kThreads, 1) attention_kernel(const __grid_constant__ AttnParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];   // 128B-swizzled tiles need 1024-byte alignment
    uint8_t* base = smem_raw;
    if ((smem_u32(base) & 1023u) != 0) __trap();
    const int d = p.d, dch = d / 64;
    Smem sm;
    sm.q = base; base += dch * 16384;
    sm.kv_stride = dch * 8192;
    sm.k0 = base; base += 2 * dch * 8192;
    sm.v0 = base; base += 2 * dch * 8192;
    sm.p0 = base; base += 2 * 16384;
    uint64_t* bars = reinterpret_cast<uint64_t*>(base);
    sm.q_full = bars; sm.q_empty = bars + 1; sm.k_full = bars + 2; sm.v_full = sm.k_full + kStages; sm.k_empty = sm.v_full + kStages;
    sm.v_empty = sm.k_empty + kStages; sm.s_full = sm.v_empty + kStages; sm.p_full = sm.s_full + 2; sm.o_empty = sm.p_full + 2;
    sm.tmem_slot = reinterpret_cast<uint32_t*>(sm.o_empty + 1);
    float* xch = reinterpret_cast<float*>(base + 256);      // [2][2][128]: double-buffered row-max exchange; reused for l

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.N;
    // packed: N == 64 puts two images into one item (each 64-key tile belongs to one of them).  Otherwise one image
    // per item with ceil(N / 128) query tiles and ceil(N / 64) key tiles; rows / keys past the image's N are loaded
    // (they belong to the next image or are zero-filled by TMA) and masked: keys to -inf, query rows at the store.
    const bool packed = (2 * N == kQRows);
    const int ipc = packed ? 2 : 1;                         // images per item
    const int qtiles = packed ? 1 : (N + kQRows - 1) / kQRows;
    const int nt = packed ? 2 : (N + kKeys - 1) / kKeys;    // key tiles per item
    const int groups = (p.B + ipc - 1) / ipc;
    const int total_items = groups * p.heads * qtiles;
    const int cta = blockIdx.x, ncta = gridDim.x;           // persistent: this CTA takes items cta, cta + ncta, ...
    uint32_t tmem_cols = 128; while (tmem_cols < static_cast<uint32_t>(d + 2 * kKeys)) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        mbar_init(sm.q_full, 1); mbar_init(sm.q_empty, 1); mbar_init(sm.o_empty, 8);
        for (int s = 0; s < kStages; ++s) { mbar_init(&sm.k_full[s], 1); mbar_init(&sm.v_full[s], 1); mbar_init(&sm.k_empty[s], 1);
                                            mbar_init(&sm.v_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&sm.p_full[s], 8); mbar_init(&sm.s_full[s], 1); }
        fence_mbar_init();
        tma_prefetch_desc(&p.q_map); tma_prefetch_desc(&p.kv_map);
    }
    if (warp == 1) tmem_alloc(sm.tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sm.tmem_slot;
    const uint32_t tmem_o = tmem_base;                      // columns [0, d)
    const uint32_t tmem_s = tmem_base + static_cast<uint32_t>(d);   // two S buffers: columns [d, d+64) and [d+64, d+128)

    // g = running key-tile counter of this CTA across its items: ring slot g % kStages, barrier parity (g / kStages) & 1
    // (the S / P buffers are double-buffered: slot g & 1, parity (g >> 1) & 1)
    if (warp == 0) {
        // ------------------------------------------------------------------ Q + K producer
        // (warp-uniform loop, one elected lane issues the copies)
        {
            int g = 0, it_n = 0;
            for (int w = cta; w < total_items; w += ncta, ++it_n) {
                const Item it = decode_item(w, qtiles, p.heads, ipc);
                const long long row0 = static_cast<long long>(it.b0) * N + static_cast<long long>(it.qt) * kQRows;
                const long long krow0 = static_cast<long long>(it.b0) * N;
                mbar_wait(sm.q_empty, (it_n & 1) ^ 1);      // the previous item's last S = Q K^T has retired
                if (elect_one()) {
                    mbar_expect_tx(sm.q_full, static_cast<uint32_t>(dch * 16384));
                    for (int c = 0; c < dch; ++c)
                        tma_load_2d(sm.q + c * 16384, &p.q_map, sm.q_full, it.h * d + c * 64, static_cast<int>(row0));
                }
                __syncwarp();
                for (int j = 0; j < nt; ++j, ++g) {
                    const int s = g % kStages;
                    mbar_wait(&sm.k_empty[s], ((g / kStages) & 1) ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(&sm.k_full[s], static_cast<uint32_t>(dch * 8192));
                        for (int c = 0; c < dch; ++c)
                            tma_load_2d(sm.k(s) + c * 8192, &p.kv_map, &sm.k_full[s], p.hid + it.h * d + c * 64,
                                        static_cast<int>(krow0) + j * kKeys);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 10) {
        // ------------------------------------------------------------------ V producer
        {
            int g = 0;
            for (int w = cta; w < total_items; w += ncta) {
                const Item it = decode_item(w, qtiles, p.heads, ipc);
                const long long krow0 = static_cast<long long>(it.b0) * N;
                for (int j = 0; j < nt; ++j, ++g) {
                    const int s = g % kStages;
                    mbar_wait(&sm.v_empty[s], ((g / kStages) & 1) ^ 1);
                    if (elect_one()) {
                        mbar_expect_tx(&sm.v_full[s], static_cast<uint32_t>(dch * 8192));
                        for (int c = 0; c < dch; ++c) {    // chunk c: 64 keys x 64 features, one 128-byte row per key
                            const int col = 2 * p.hid + it.h * d + c * 64;
                            tma_load_2d(sm.v(s) + c * 8192, &p.kv_map, &sm.v_full[s], col, static_cast<int>(krow0) + j * kKeys);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        // The whole warp walks the loop (warp-uniform control flow and operands); one elected lane issues each instruction.
        const uint32_t idesc_s = umma_idesc_16(kQRows, kKeys, (F16 ? 1 : 0));
        const uint32_t idesc_o = umma_idesc_16(kQRows, d, (F16 ? 1 : 0)) | kIdescBMajorMN;
        const uint32_t v_lbo = 8192u;                       // next 64-feature chunk of a V stage
        auto mma = [&](uint32_t dt, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
            if (elect_one()) umma_16(dt, ad, bd, idesc, acc);
        };
        auto commit = [&](uint64_t* bar) {
            if (elect_one()) umma_commit(bar);
        };
        const uint64_t q_desc = umma_desc_sw128(smem_u32(sm.q));
        int g = 0, it_n = 0;
        for (int w = cta; w < total_items; w += ncta, ++it_n) {
            auto issue_s = [&](int j) {                     // tile j of this item = running tile g + j
                const int gj = g + j, s = gj % kStages, sb = gj & 1;
                mbar_wait(&sm.k_full[s], (gj / kStages) & 1);
                tc_fence_after();
                const uint64_t k_desc = umma_desc_sw128(smem_u32(sm.k(s)));
                const uint32_t dst = tmem_s + static_cast<uint32_t>(sb * kKeys);
                for (int c = 0; c < dch; ++c) {             // 64-feature chunk c: 16 KB of Q, 8 KB of K (descriptor units of 16 B)
                    const uint64_t ad = q_desc + static_cast<uint64_t>(c * (16384 >> 4));
                    const uint64_t bd = k_desc + static_cast<uint64_t>(c * (8192 >> 4));
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) mma(dst, ad + 2 * k4, bd + 2 * k4, idesc_s, (c | k4) != 0);
                }
                commit(&sm.k_empty[s]);                   // K_j can be overwritten as soon as S_j has retired
                commit(&sm.s_full[sb]);
                if (j == nt - 1) commit(sm.q_empty);        // ... and so can Q after the item's last S
            };
            mbar_wait(sm.q_full, it_n & 1);
            // the S buffers are free: every softmax tile of the previous item was waited for below (p_full)
            issue_s(0);
            if (nt > 1) issue_s(1);                       // S is double-buffered: S_{j+1} is ready before softmax j ends
            for (int j = 0; j < nt; ++j) {
                const int gj = g + j, s = gj % kStages, sb = gj & 1;
                mbar_wait(&sm.p_full[sb], (gj >> 1) & 1);   // P_j in smem, S_j consumed (its buffer is free), O rescaled if needed
                tc_fence_after();
                if (j + 2 < nt) issue_s(j + 2);
                if (j == 0 && it_n > 0) {                   // O still holds the previous item until its rows have been read out
                    mbar_wait(sm.o_empty, (it_n - 1) & 1);
                    tc_fence_after();
                }
                mbar_wait(&sm.v_full[s], (gj / kStages) & 1);
                tc_fence_after();
                const uint64_t p_desc = umma_desc_sw128(smem_u32(sm.p(sb)));
                const uint64_t v_desc = umma_desc_sw128_mn(smem_u32(sm.v(s)), v_lbo);
#pragma unroll
                for (int kk = 0; kk < kKeys / 16; ++kk)         // 16 keys: +32 bytes in a P row, +2048 bytes (16 rows) in V
                    mma(tmem_o, p_desc + 2 * kk, v_desc + static_cast<uint64_t>(kk * (2048 >> 4)), idesc_o, (j | kk) != 0);
                commit(&sm.v_empty[s]);                   // V_j / P_j free, O updated
            }
            g += nt;
        }
    } else if (warp < 10) {
        // ------------------------------------------------------------------ softmax + output
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;                   // which 32 key columns of the tile (and which half of O's columns)
        const int row = q * 32 + lane;
        const uint32_t lane_off = static_cast<uint32_t>(q * 32) << 16;
        const int bar_id = 1 + q;                           // the two warps of a lane quarter exchange row maxima
        const float c = p.scale_log2e;
        const int dh = d >> 1;                              // O columns owned by this thread: [half*dh, half*dh + dh)
        const int row_img = row / N;                        // only meaningful when packed
        int g = 0, it_n = 0;
        for (int w = cta; w < total_items; w += ncta, ++it_n) {
            const Item it = decode_item(w, qtiles, p.heads, ipc);
            const long long grow = static_cast<long long>(it.b0) * N + static_cast<long long>(it.qt) * kQRows + row;
            const bool row_ok = (grow < static_cast<long long>(p.B) * N) && (packed || it.qt * kQRows + row < N);
            float m_used = -INFINITY, l = 0.f;
            for (int j = 0; j < nt; ++j) {
                const int gj = g + j, sb = gj & 1;
                mbar_wait(&sm.s_full[sb], (gj >> 1) & 1);
                tc_fence_after();
                uint32_t r0[32];
                tmem_ld32(tmem_s + static_cast<uint32_t>(sb * kKeys) + lane_off + half * 32, r0);
                tmem_ld_wait();
                float sv[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) sv[i] = __uint_as_float(r0[i]);
                // packed: a 64-key tile belongs to one image; rows of the other image ignore it entirely
                const bool tile_valid = !packed || (j == row_img);
                if (!packed && (j + 1) * kKeys > N) {       // ragged last key tile (warp-uniform): keys >= N drop out
                    const int first_bad = N - j * kKeys - half * 32;
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (i >= first_bad) sv[i] = -INFINITY;
                }
                float m_half = -INFINITY;
                if (tile_valid) {
#pragma unroll
                    for (int i = 0; i < 32; i += 2) m_half = fmaxf(m_half, fmaxf(sv[i], sv[i + 1]));
                }
                float* xm = xch + sb * 256;
                xm[half * 128 + row] = m_half;
                asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
                const float m_tile = fmaxf(m_half, xm[(half ^ 1) * 128 + row]);
                float factor = 1.f;
                bool need = false;
                if (m_tile > m_used) {
                    if (m_used == -INFINITY) {
                        m_used = m_tile;                    // nothing accumulated yet for this row (O row == 0, l == 0)
                    } else if ((m_tile - m_used) * c > kRescaleThreshold) {
                        factor = ex2_approx((m_used - m_tile) * c);
                        m_used = m_tile;
                        need = true;
                    }
                }
                if (__any_sync(0xffffffffu, need)) {
                    // O must be complete through PV_{j-1} before it is rescaled (need implies j >= 1)
                    mbar_wait(&sm.v_empty[(gj - 1) % kStages], ((gj - 1) / kStages) & 1);
                    tc_fence_after();
                    for (int c0 = half * dh; c0 < half * dh + dh; c0 += 32) {
                        uint32_t o[32];
                        tmem_ld32(tmem_o + lane_off + c0, o);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * factor);
                        tmem_st32(tmem_o + lane_off + c0, o);
                    }
                    tmem_st_wait();
                    l *= factor;
                }
                // p = 2^(s*c - m*c); a row that ignores this tile writes zeros (its m may still be -inf)
                const float mc = (m_used == -INFINITY) ? 0.f : m_used * c;
                const float cc = tile_valid ? c : 0.f;
                const float off = tile_valid ? mc : 200.f;  // 2^-200 flushes to exactly 0
                uint32_t pk[16];
                float lsum = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float e0 = ex2_approx(fmaf(sv[2 * i], cc, -off));
                    const float e1 = ex2_approx(fmaf(sv[2 * i + 1], cc, -off));
                    lsum += e0 + e1;
                    pk[i] = pack_16_inrange(e0, e1, (F16 ? 1 : 0));   // p <= 2^8
                }
                l += lsum;
                // P_j goes into the buffer PV_{g-2} read (possibly the previous item's): S_j was issued before that
                // MMA, so s_full alone does not order these stores after its operand reads
                if (gj >= 2) mbar_wait(&sm.v_empty[(gj - 2) % kStages], ((gj - 2) / kStages) & 1);
                uint8_t* prow = sm.p(sb) + row * 128;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch)
                    *reinterpret_cast<uint4*>(prow + (((half * 4 + ch) ^ (row & 7)) << 4)) =
                        make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
                fence_proxy_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.p_full[sb]);
            }
            // ---- final: O / l -> 16-bit.  The two threads of a row add their partial sums.  (The first barrier keeps a
            // fast thread from overwriting a row maximum of the last tile that its partner has not read yet.)
            asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
            xch[half * 128 + row] = l;
            asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
            l += xch[(half ^ 1) * 128 + row];
            const int g_last = g + nt - 1;
            mbar_wait(&sm.v_empty[g_last % kStages], (g_last / kStages) & 1);
            tc_fence_after();
            const float inv_l = (l > 0.f) ? 1.f / l : 0.f;
            for (int c0 = half * dh; c0 < half * dh + dh; c0 += 32) {
                uint32_t o[32];
                tmem_ld32(tmem_o + lane_off + c0, o);
                tmem_ld_wait();
                if (c0 + 32 >= half * dh + dh) {            // this warp's last read of O: the next item may overwrite it
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(sm.o_empty);
                }
                if (row_ok) {
                    uint4* dst = reinterpret_cast<uint4*>(p.out + grow * p.hid + it.h * d + c0);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        dst[i] = make_uint4(pack_16(__uint_as_float(o[8 * i]) * inv_l, __uint_as_float(o[8 * i + 1]) * inv_l, (F16 ? 1 : 0)),
                                            pack_16(__uint_as_float(o[8 * i + 2]) * inv_l, __uint_as_float(o[8 * i + 3]) * inv_l, (F16 ? 1 : 0)),
                                            pack_16(__uint_as_float(o[8 * i + 4]) * inv_l, __uint_as_float(o[8 * i + 5]) * inv_l, (F16 ? 1 : 0)),
                                            pack_16(__uint_as_float(o[8 * i + 6]) * inv_l, __uint_as_float(o[8 * i + 7]) * inv_l, (F16 ? 1 : 0)));
                }
            }
            // the sum exchange above used buffer 0 of xch: the partner must have read it before the next item's first
            // tile (buffer g & 1) may write there
            asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
            g += nt;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

}  // namespace

cudaError_t launch_attention(const AttnParams& p, int num_sms, cudaStream_t stream) {
    if (p.d % 64 != 0 || p.d > 256 || p.N < 1) return cudaErrorInvalidValue;
    const int smem = attn_smem_bytes(p.d);
    // cudaFuncSetAttribute is per device: the configured size is tracked per device ordinal
    static std::atomic<int> smem_set[kMaxDevices];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    if (smem > smem_set[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(attention_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(attention_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        smem_set[dev].store(smem, std::memory_order_release);
    }
    const bool packed = (2 * p.N == kQRows);
    const int ipc = packed ? 2 : 1;
    const int qtiles = packed ? 1 : (p.N + kQRows - 1) / kQRows;
    const int groups = (p.B + ipc - 1) / ipc;
    const long long items = static_cast<long long>(groups) * p.heads * qtiles;
    if (items <= 0) return cudaSuccess;
    // persistent: one CTA per SM: the tiles of a 256-wide head fill the SM's shared memory; the register file holds one
    // CTA of this kernel either way
    long long grid = num_sms;
    if (grid > items) grid = items;
    if (p.f16) attention_kernel<true><<<static_cast<unsigned>(grid), kThreads, smem, stream>>>(p);
    else attention_kernel<false><<<static_cast<unsigned>(grid), kThreads, smem, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace vdt
