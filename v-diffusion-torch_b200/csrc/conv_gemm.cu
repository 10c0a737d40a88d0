// Implicit-GEMM 3x3 / 1x1 convolution and linear layers for sm_100a.
//
// Replaces F.conv2d / F.linear on the reference's hot path (modules.py:79-80, 141-144 as called
// from unet.py:121,125,134,70-71,203-215,217,232).  NHWC bf16 operands, fp32 accumulation in
// TMEM, fused epilogue (bias, residual add, SiLU, 16-bit / NCHW stores).
//
// Persistent warp-specialised kernel, one CTA per SM, 192 threads, CTAs paired (cluster of 2) so
// the tensor cores run in cta_group::2 mode: one 256 x N x 16 MMA spans both SMs, each CTA holding
// its own 128 rows of A, half of the N rows of B and its 128 x N half of the accumulator.  Per SM
// this halves the weight-tile fill (L2 -> smem) and the operand reads (smem -> tensor core) that
// cap a single-CTA 128 x 256 tile at ~2/3 of the MMA rate.
//   warp 0     TMA producer (both CTAs): per K-block one 4-D box of the activation (shifted by the
//                               filter tap; out-of-bounds rows/cols are zero-filled by TMA = conv
//                               padding) and this CTA's half of the packed-weight box, into a
//                               6-stage smem ring; completion is signalled on the leader's barrier
//   warp 1     MMA issuer (leader CTA only): tcgen05.mma.cta_group::2.kind::f16, accumulators
//                               double-buffered in TMEM (2 x 256 columns per CTA)
//   warps 2-9  epilogue (both CTAs): tcgen05.ld -> registers -> smem transposition -> coalesced global
//                               stores (+bias, +residual), overlapping the next tile's main loop
#include <atomic>

#include "kernels.cuh"
#include "ptx.cuh"

namespace vdt {

namespace {

constexpr int kBM = 128;
constexpr int kBK = 64;                       // bf16 elements per K-block = one 128-byte swizzle row
constexpr int kStages = 6;
constexpr int kMaxBN = 256;
constexpr int kABytes = kBM * kBK * 2;        // 16 KiB
constexpr int kBBytes = (kMaxBN / 2) * kBK * 2;   // 16 KiB: this CTA's half of the N rows
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kEpiWarps = 8;                    // two per TMEM lane quarter, alternating 32-column chunks
constexpr int kEpiBytes = kEpiWarps * 32 * 128; // per epilogue warp: 32 rows x 32 fp32 columns transposition tile
constexpr int kSmemBytes = kStages * kStageBytes + kEpiBytes + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int kThreads = 64 + 32 * 8;          // TMA warp + MMA warp + 8 epilogue warps
constexpr int kTmemCols = 512;

struct TileCoord {
    int c1, c2, c3;   // TMA coordinates of the un-shifted tile origin (W, H, N)
};

__device__ __forceinline__ TileCoord tile_origin(const ConvParams& p, int m_tile) {
    TileCoord t;
    if (p.pointwise) {
        t.c1 = m_tile * kBM; t.c2 = 0; t.c3 = 0;
    } else {
        t.c1 = 0;
        t.c2 = (m_tile % p.tiles_per_image) * p.box_h;
        t.c3 = (m_tile / p.tiles_per_image) * p.box_n;
    }
    return t;
}

// work item w -> (M tile of this CTA, N tile, output parity class of the sub-pixel upsampling conv); the parity runs
// fastest so that the four items sharing an A region are in flight together
struct WorkItem { int m_tile, n_tile, par; };
__device__ __forceinline__ WorkItem decode_item(const ConvParams& p, int w, int rank) {
    WorkItem it;
    it.par = 0;
    if (p.ups) { it.par = w & 3; w >>= 2; }
    const int mp = w / p.num_n_tiles;
    // pair_tiles = T > 0: the two CTAs of a pair take tile mp % T of two consecutive images (which share their residual
    // image, ConvParams::resid_rep), so both read the same residual tile at the same time
    it.m_tile = p.pair_tiles > 0 ? (2 * (mp / p.pair_tiles) + rank) * p.pair_tiles + mp % p.pair_tiles : mp * 2 + rank;
    it.n_tile = w % p.num_n_tiles;
    return it;
}

// Row-major epilogue of one 32-row x 32-column chunk after the smem transposition: lane = (row % 4 group rsub,
// 4 columns cq), all 32 rows valid.  Compile-time variants keep the instruction count low (the epilogue warps
// are issue-bound otherwise); ragged tiles and SiLU epilogues take epilogue_rowmajor_generic.
// MAP: 0 rows are stored where they were computed; 1 sub-pixel upsampling conv (ConvParams::ups): row = low-res pixel,
// stored at its high-resolution position of parity `par`; 2 upsampled identity skip (ConvParams::resid_up): the residual
// of output pixel (y, x) is low-res pixel (y >> 1, x >> 1); 3 shared residual (ConvParams::resid_rep == 2): image i adds
// residual image i >> 1.  All three need power-of-two square maps (map_shift).
template <bool F16, bool F32OUT, bool RESID, int STATS, int MAP>   // STATS: 0 none, 4 / 2 = columns per statistics entry
__device__ __forceinline__ void epilogue_rowmajor(const ConvParams& p, uint32_t tile, int lane, long long wrow0, int col0, int slab,
                                                  const float4 b4, int par) {
    const int cq = lane & 7, rsub = lane >> 3;
    const size_t off0 = static_cast<size_t>(wrow0 + rsub) * p.ld + col0 + cq * 4;
    const size_t step = static_cast<size_t>(4) * p.ld;
    // row remaps: a 32-row slab never crosses an image (HW is a power of two >= 32 here)
    const int sh = (MAP != 0) ? p.map_shift : 0, wmask = (1 << sh) - 1;
    const long long img = (MAP != 0) ? (wrow0 >> (2 * sh)) : 0;
    const int pix0 = (MAP != 0) ? static_cast<int>(wrow0 & ((1ll << (2 * sh)) - 1)) + rsub : 0;   // pixel of this lane's first row
    const size_t colo = static_cast<size_t>(col0 + cq * 4);
    // MAP 1: high-res row = img * 4HW + (2y + py) * 2W + 2x + px = base + 4 * pix - 2 * x
    const long long ups_base = (MAP == 1) ? (img << (2 * sh + 2)) + (static_cast<long long>(par >> 1) << (sh + 1)) + (par & 1) : 0;
    float4 res[8];
    if (RESID) {                                             // all eight loads in flight before anything is stored
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (MAP == 2) {
                const int pix = pix0 + 4 * i;
                const int shl = (MAP == 2) ? sh - 1 : 0;           // log2 of the low-resolution width
                const long long src = (img << (2 * shl)) + ((pix >> (sh + 1)) << shl) + ((pix & wmask) >> 1);
                res[i] = ldg_nc_v4_issue(p.residual + static_cast<size_t>(src) * p.ld + colo);
            } else if (MAP == 3) {
                const long long src = ((img >> 1) << (2 * sh)) + (pix0 + 4 * i);
                res[i] = ldg_nc_v4_issue(p.residual + static_cast<size_t>(src) * p.ld + colo);
            } else {
                res[i] = ldg_nc_v4_issue(p.residual + off0 + i * step);
            }
        }
        compiler_fence();
    }
    float ssum = 0.f, ssq = 0.f, ssum1 = 0.f, ssq1 = 0.f;
    float amax = 0.f;                                        // fp16 16-bit outputs: largest magnitude converted
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int rr = i * 4 + rsub;
        float4 o = lds_v4(tile + static_cast<uint32_t>(rr * 8 + (cq ^ (rr & 7))) * 16u);
        o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
        if (RESID) { o.x += res[i].x; o.y += res[i].y; o.z += res[i].z; o.w += res[i].w; }
        {
            size_t off = off0 + i * step;
            if (MAP == 1) {
                const int pix = pix0 + 4 * i;
                off = static_cast<size_t>(ups_base + 4ll * pix - 2 * (pix & wmask)) * p.ld + colo;
            }
            if (F32OUT)
                *reinterpret_cast<float4*>(p.out_f32 + off) = o;
            else {
                *reinterpret_cast<uint2*>(p.out_bf16 + off) = make_uint2(pack_16(o.x, o.y, (F16 ? 1 : 0)), pack_16(o.z, o.w, (F16 ? 1 : 0)));
                if (F16) amax = fmaxf(fmaxf(amax, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
            }
            if (STATS == 4) {
                ssum += (o.x + o.y) + (o.z + o.w);
                ssq = fmaf(o.x, o.x, fmaf(o.y, o.y, fmaf(o.z, o.z, fmaf(o.w, o.w, ssq))));
            } else if (STATS == 2) {
                ssum += o.x + o.y; ssq = fmaf(o.x, o.x, fmaf(o.y, o.y, ssq));
                ssum1 += o.z + o.w; ssq1 = fmaf(o.z, o.z, fmaf(o.w, o.w, ssq1));
            }
        }
    }
    if (F16 && !F32OUT && p.sat_count != nullptr) {         // the saturating pack clamped something: count the event
        if (__any_sync(0xffffffffu, amax > 65504.f) && lane == 0) atomicAdd(p.sat_count, 1ull);
    }
    if (STATS) {                                             // fixed-order reduction over the warp's 32 rows
        ssum += __shfl_xor_sync(0xffffffffu, ssum, 8); ssq += __shfl_xor_sync(0xffffffffu, ssq, 8);
        ssum += __shfl_xor_sync(0xffffffffu, ssum, 16); ssq += __shfl_xor_sync(0xffffffffu, ssq, 16);
        if (STATS == 2) {
            ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, 8); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 8);
            ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, 16); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 16);
        }
        if (rsub == 0) {
            if (MAP == 1) {                                  // the parity classes of an image own consecutive slab groups
                const int simg = slab / p.stat_slabs_img;
                slab = (simg * 4 + par) * p.stat_slabs_img + (slab - simg * p.stat_slabs_img);
            }
            float2* st = p.stats + static_cast<size_t>(slab) * (p.Cout / (STATS ? STATS : 1));
            if (STATS == 4) {
                st[(col0 >> 2) + cq] = make_float2(ssum, ssq);
            } else {
                st[(col0 >> 1) + cq * 2] = make_float2(ssum, ssq);
                st[(col0 >> 1) + cq * 2 + 1] = make_float2(ssum1, ssq1);
            }
        }
    }
}

// Same with every option and bound checked at run time (ragged tiles, SiLU epilogues).
__device__ __noinline__ void epilogue_rowmajor_generic(const ConvParams& p, uint32_t tile, int lane, int q, int m_tile,
                                                       long long wrow0, int col0, const float4 b4, int par) {
    const int cq = lane & 7, rsub = lane >> 3;
    const bool tile_ok = m_tile < p.num_m_tiles;
    float ssum = 0.f, ssq = 0.f, ssum1 = 0.f, ssq1 = 0.f;   // (x, y) and (z, w) halves; merged for 4-column entries
    for (int i = 0; i < 8; ++i) {
        const int rr = i * 4 + rsub;
        const long long g = wrow0 + rr;
        const bool ok = tile_ok && (q * 32 + rr < p.rows_per_tile) && (g < p.M);
        if (!ok) continue;
        float4 o = lds_v4(tile + static_cast<uint32_t>(rr * 8 + (cq ^ (rr & 7))) * 16u);
        long long orow = g;                                  // output row
        if (p.ups) {                                         // low-res pixel (img, y, x) -> high-res pixel (2y + py, 2x + px)
            const long long img = g / p.HW;
            const int pix = static_cast<int>(g - img * p.HW);
            const int y = pix / p.ups_w, x = pix - y * p.ups_w;
            orow = img * 4 * p.HW + static_cast<long long>(2 * y + (par >> 1)) * (2 * p.ups_w) + 2 * x + (par & 1);
        }
        const size_t off = static_cast<size_t>(orow) * p.ld + col0 + cq * 4;
        o.x += b4.x; o.y += b4.y; o.z += b4.z; o.w += b4.w;
        if (p.residual) {
            size_t roff = off;
            if (p.resid_up) {                                // identity skip of an upsampling block: nearest source pixel
                const long long img = g / p.HW;
                const int pix = static_cast<int>(g - img * p.HW);
                const int y = pix / p.out_w, x = pix - y * p.out_w;
                roff = static_cast<size_t>(img * (p.HW >> 2) + static_cast<long long>(y >> 1) * (p.out_w >> 1) + (x >> 1)) * p.ld + col0 + cq * 4;
            } else if (p.resid_rep > 1) {                    // rows of resid_rep consecutive images share one residual image
                const long long img = g / p.HW;
                roff = static_cast<size_t>((img / p.resid_rep) * p.HW + (g - img * p.HW)) * p.ld + col0 + cq * 4;
            }
            const float4 r4 = __ldg(reinterpret_cast<const float4*>(p.residual + roff));
            o.x += r4.x; o.y += r4.y; o.z += r4.z; o.w += r4.w;
        }
        if (p.act_silu) { o.x = silu_f(o.x); o.y = silu_f(o.y); o.z = silu_f(o.z); o.w = silu_f(o.w); }
        if (p.out_mode == kOutF32)
            *reinterpret_cast<float4*>(p.out_f32 + off) = o;
        else {
            *reinterpret_cast<uint2*>(p.out_bf16 + off) = make_uint2(pack_16(o.x, o.y, p.f16), pack_16(o.z, o.w, p.f16));
            if (p.f16 && p.sat_count != nullptr && fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w))) > 65504.f)
                atomicAdd(p.sat_count, 1ull);
        }
        ssum += o.x + o.y; ssq = fmaf(o.x, o.x, fmaf(o.y, o.y, ssq));
        ssum1 += o.z + o.w; ssq1 = fmaf(o.z, o.z, fmaf(o.w, o.w, ssq1));
    }
    if (p.stats) {
        ssum += __shfl_xor_sync(0xffffffffu, ssum, 8); ssq += __shfl_xor_sync(0xffffffffu, ssq, 8);
        ssum += __shfl_xor_sync(0xffffffffu, ssum, 16); ssq += __shfl_xor_sync(0xffffffffu, ssq, 16);
        ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, 8); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 8);
        ssum1 += __shfl_xor_sync(0xffffffffu, ssum1, 16); ssq1 += __shfl_xor_sync(0xffffffffu, ssq1, 16);
        if (rsub == 0 && tile_ok) {                          // a quarter without valid rows still writes its zeros
            int slab = m_tile * 4 + q;
            bool real = true;
            if (p.ups) {                                     // the parity classes of an image own consecutive slab groups
                const int img = slab / p.stat_slabs_img;
                real = img < p.M / p.HW;                     // the zero-filled images of a ragged last tile own no slabs here
                slab = (img * 4 + par) * p.stat_slabs_img + (slab - img * p.stat_slabs_img);
            }
            float2* st = p.stats + static_cast<size_t>(slab) * (p.Cout / p.stat_cols);
            if (!real) {
            } else if (p.stat_cols == 4) {
                st[(col0 >> 2) + cq] = make_float2(ssum + ssum1, ssq + ssq1);
            } else {
                st[(col0 >> 1) + cq * 2] = make_float2(ssum, ssq);
                st[(col0 >> 1) + cq * 2 + 1] = make_float2(ssum1, ssq1);
            }
        }
    }
}

template <bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv_gemm_kernel(const __grid_constant__ ConvParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* epi_smem = smem + kStages * kStageBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem + kEpiBytes);
    uint64_t* full_bar = bars;                    // [kStages] TMA -> MMA
    uint64_t* empty_bar = bars + kStages;         // [kStages] MMA -> TMA
    uint64_t* acc_full = bars + 2 * kStages;      // [2] MMA -> epilogue
    uint64_t* acc_empty = bars + 2 * kStages + 2; // [2] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int rank = static_cast<int>(cluster_ctarank());   // 0 / 1 inside the pair
    const int pair = blockIdx.x >> 1, num_pairs_resident = gridDim.x >> 1;

    if (threadIdx.x == 0) {
        // full / acc_empty are only used in the leader CTA (rank 0); empty / acc_full in both
        for (int s = 0; s < kStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 2 * kEpiWarps); }   // one arrival per epilogue warp of both CTAs
        fence_mbar_init();
        for (int s = 0; s < p.num_segs; ++s) tma_prefetch_desc(&p.a_map[s]);
        tma_prefetch_desc(&p.b_map);
    }
    if (warp == 1) tmem_alloc_2cta(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                      // peer's barriers are initialised before any multicast
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // work item w = (pair of M tiles, N tile); this CTA takes M tile 2*mp + rank (a phantom tile past the
    // end is all zero-filled loads and masked stores)
    const int total_items = ((p.num_m_tiles + 1) >> 1) * p.num_n_tiles * (p.ups ? 4 : 1);
    int kblocks_total = 0;
    for (int s = 0; s < p.num_segs; ++s) kblocks_total += p.seg_taps[s] * p.seg_kblocks[s];

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        // (the whole warp walks the loop, one elected lane issues: coordinates and descriptors stay warp-uniform)
        {
            int stage = 0; uint32_t phase = 0;
            const int half_n = p.block_n >> 1;
            // both CTAs' boxes complete on the leader's barrier
            const uint32_t tx_bytes = 2u * static_cast<uint32_t>(p.rows_per_tile * kBK * 2 + half_n * kBK * 2);
            for (int w = pair; w < total_items; w += num_pairs_resident) {
                const WorkItem it = decode_item(p, w, rank);
                const int n_tile = it.n_tile, py = it.par >> 1, px = it.par & 1;
                const TileCoord o = tile_origin(p, it.m_tile);
                int kcol = it.par * kblocks_total * kBK;   // sub-pixel conv: every parity class has its own weight columns
                for (int s = 0; s < p.num_segs; ++s) {
                    const int taps = p.seg_taps[s];
                    for (int tap = 0; tap < taps; ++tap) {
                        // 9: 3x3, pad 1; 4: the 2x2 neighbourhood of a parity class of the sub-pixel upsampling conv; 1: pointwise
                        const int dy = (taps == 9) ? tap / 3 - 1 : (taps == 4) ? (tap >> 1) - 1 + py : 0;
                        const int dx = (taps == 9) ? tap % 3 - 1 : (taps == 4) ? (tap & 1) - 1 + px : 0;
                        for (int kb = 0; kb < p.seg_kblocks[s]; ++kb) {
                            mbar_wait(&empty_bar[stage], phase ^ 1);
                            uint8_t* a_dst = smem + stage * kStageBytes;
                            uint8_t* b_dst = a_dst + kABytes;
                            if (elect_one()) {
                                if (rank == 0) mbar_expect_tx(&full_bar[stage], tx_bytes);
                                tma_load_4d_2cta(a_dst, &p.a_map[s], &full_bar[stage], kb * kBK, o.c1 + dx, o.c2 + dy, o.c3);
                                tma_load_2d_2cta(b_dst, &p.b_map, &full_bar[stage], kcol, n_tile * p.block_n + rank * half_n);
                            }
                            __syncwarp();
                            kcol += kBK;
                            if (++stage == kStages) { stage = 0; phase ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA)
        // The whole warp walks the loop (warp-uniform control flow and operands); one elected lane issues each
        // instruction, so the descriptors stay in uniform registers (ptx.cuh: elect_one).
        if (rank == 0) {
            const uint32_t idesc = umma_idesc_16(2 * kBM, p.block_n, (F16 ? 1 : 0));
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int w = pair; w < total_items; w += num_pairs_resident) {
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * kMaxBN);
                for (int kb = 0; kb < kblocks_total; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
                    const uint64_t adesc = umma_desc_sw128(a_addr);
                    const uint64_t bdesc = umma_desc_sw128(a_addr + kABytes);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < kBK / 16; ++k)
                            umma_16_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
                        umma_commit_2cta(&empty_bar[stage], static_cast<uint16_t>(3));        // frees the slot in both CTAs
                    }
                    __syncwarp();
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                if (elect_one()) umma_commit_2cta(&acc_full[acc], static_cast<uint16_t>(3));       // both halves complete -> both epilogues
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue (warps 2..5)
        const int q = warp & 3;                              // TMEM lane quarter this warp may access
        const int chunk_par = (warp - 2) >> 2;               // this warp takes the 32-column chunks of this parity
        const int row = q * 32 + lane;
        const uint32_t epi_base = smem_u32(epi_smem);
        // which compile-time epilogue serves this launch (the same for every tile): -1 = generic (SiLU epilogues, row
        // remaps on maps that are not power-of-two squares, 16-bit output with a residual)
        int variant = -1;
        {
            const bool f32o = p.out_mode == kOutF32, resid = p.residual != nullptr;
            const int sti = (p.stats == nullptr) ? 2 : (p.stat_cols == 4 ? 0 : 1);
            const bool mapped = p.ups || p.resid_up || p.resid_rep > 1;
            if (p.act_silu || (mapped && p.map_shift < 3) || (!f32o && resid)) variant = -1;
            else if (p.ups) variant = (f32o ? 9 : 12) + sti;
            else if (p.resid_up) variant = f32o ? 15 + sti : -1;
            else if (p.resid_rep > 1) variant = (f32o && resid && p.resid_rep == 2) ? 18 + sti : -1;
            else if (f32o) variant = (resid ? 0 : 3) + sti;
            else variant = 6 + sti;
        }
        int acc = 0; uint32_t acc_phase = 0;
        for (int w = pair; w < total_items; w += num_pairs_resident) {
            const WorkItem it = decode_item(p, w, rank);
            const int m_tile = it.m_tile, n_tile = it.n_tile;
            const long long grow = static_cast<long long>(m_tile) * p.rows_per_tile + row;
            const bool row_ok = (row < p.rows_per_tile) && (grow < p.M) && (m_tile < p.num_m_tiles);
            if (p.residual && row_ok && !p.resid_up) {
                // the main loop of this tile is still running: pull this warp's residual lines (one 128-byte line
                // per row and 32-column chunk) into L2 so the epilogue's loads below do not pay DRAM latency
                long long rrow = grow;
                if (p.resid_rep > 1) {                       // shared residual: image i reads image i / resid_rep
                    const long long img = grow / p.HW;
                    rrow = (img / p.resid_rep) * p.HW + (grow - img * p.HW);
                }
                const float* rp = p.residual + static_cast<size_t>(rrow) * p.ld + n_tile * p.block_n;
                for (int c0 = chunk_par * 32; c0 < p.block_n; c0 += 64) prefetch_l2(rp + c0);
            }
            // this warp's bias vectors for its (up to four) chunks of the tile, fetched while the main loop still runs:
            // inside the chunk loop the load's L2 latency would be exposed once per chunk, which is what bounds the
            // epilogue-heavy GEMMs (K = 64 / 256: in_conv, proj_in, proj_out)
            float4 bias_c[4];
            {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int colk = n_tile * p.block_n + chunk_par * 32 + 64 * k;
                    bias_c[k] = (chunk_par * 32 + 64 * k < p.block_n && colk < p.Cout)
                                    ? __ldg(reinterpret_cast<const float4*>(p.bias + colk + (lane & 7) * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * kMaxBN);
            const int nkc = (p.block_n - chunk_par * 32 + 63) / 64;    // 32-column chunks of the tile this warp owns (0 .. 4)
#pragma unroll
            for (int kc = 0; kc < 4; ++kc) {
                const int c0 = chunk_par * 32 + 64 * kc;
                if (c0 >= p.block_n) break;
                const float4 b4 = bias_c[kc];
                uint32_t r[32];
                tmem_ld32(t_row + static_cast<uint32_t>(c0), r);
                tmem_ld_wait();
                if (kc == nkc - 1) {
                    // this warp's last read of the accumulator: hand it back to the MMA thread now, before the stores of
                    // the chunk (relaxed arrive: a release fence here would stall the warp until its global stores drained)
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster_relaxed(&acc_empty[acc], 0);   // the leader waits for both CTAs' drains
                }
                const int col0 = n_tile * p.block_n + c0;
                if (col0 >= p.Cout) continue;                // warp-uniform
                {
                    // thread-per-row registers -> swizzled smem tile -> lane = (row % 4 group, 4 columns): every
                    // global access below is 4 rows x 128 (fp32) / 64 (16-bit) contiguous bytes per warp instruction
                    const uint32_t tile = epi_base + static_cast<uint32_t>(warp - 2) * (32u * 128u);
#pragma unroll
                    for (int j = 0; j < 8; ++j)                // (the bias is added after the transposition)
                        sts_v4(tile + static_cast<uint32_t>(lane * 8 + (j ^ (lane & 7))) * 16u,
                               make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                           __uint_as_float(r[4 * j + 3])));
                    __syncwarp();
                    const long long wrow0 = static_cast<long long>(m_tile) * p.rows_per_tile + q * 32;
                    const bool all_valid = (m_tile < p.num_m_tiles) && (q * 32 + 32 <= p.rows_per_tile) && (wrow0 + 32 <= p.M);
                    const int slab = m_tile * 4 + q, par = it.par;
#define VDT_EPI(F32, RES, ST, MAP) epilogue_rowmajor<F16, F32, RES, ST, MAP>(p, tile, lane, wrow0, col0, slab, b4, par); break
                    switch (all_valid ? variant : -1) {      // ragged tiles take the run-time checked generic path
                        case 0: VDT_EPI(true, true, 4, 0);   case 1: VDT_EPI(true, true, 2, 0);   case 2: VDT_EPI(true, true, 0, 0);
                        case 3: VDT_EPI(true, false, 4, 0);  case 4: VDT_EPI(true, false, 2, 0);  case 5: VDT_EPI(true, false, 0, 0);
                        case 6: VDT_EPI(false, false, 4, 0); case 7: VDT_EPI(false, false, 2, 0); case 8: VDT_EPI(false, false, 0, 0);
                        // sub-pixel upsampling conv1: rows scattered to their high-resolution positions, no residual
                        case 9: VDT_EPI(true, false, 4, 1);   case 10: VDT_EPI(true, false, 2, 1);  case 11: VDT_EPI(true, false, 0, 1);
                        case 12: VDT_EPI(false, false, 4, 1); case 13: VDT_EPI(false, false, 2, 1); case 14: VDT_EPI(false, false, 0, 1);
                        // conv2 of an upsampling block: residual gathered from the low-resolution stream
                        case 15: VDT_EPI(true, true, 4, 2);   case 16: VDT_EPI(true, true, 2, 2);   case 17: VDT_EPI(true, true, 0, 2);
                        // conv2 of block 0 under CFG: the cond / uncond rows of a sample share the residual (in_conv's output)
                        case 18: VDT_EPI(true, true, 4, 3);   case 19: VDT_EPI(true, true, 2, 3);   case 20: VDT_EPI(true, true, 0, 3);
                        default: epilogue_rowmajor_generic(p, tile, lane, q, m_tile, wrow0, col0, b4, par); break;
                    }
#undef VDT_EPI
                    __syncwarp();
                }
            }
            if (nkc <= 0) {                                  // a warp without a chunk in this tile still has to arrive
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster_relaxed(&acc_empty[acc], 0);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                      // no CTA exits while its peer may still signal it
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2cta(tmem_base, kTmemCols);
    }
}

}  // namespace

cudaError_t launch_conv_gemm(const ConvParams& p, int num_sms, cudaStream_t stream) {
    // cudaFuncSetAttribute is per device: one flag per device ordinal (a process may drive several GPUs)
    static std::atomic<bool> attr_set[kMaxDevices];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    if (!attr_set[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
        if (e != cudaSuccess) return e;
        attr_set[dev].store(true, std::memory_order_release);
    }
    const int items = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles * (p.ups ? 4 : 1);
    if (items <= 0) return cudaSuccess;
    const int pairs = items < num_sms / 2 ? items : num_sms / 2;
    if (p.f16) conv_gemm_kernel<true><<<2 * pairs, kThreads, kSmemBytes, stream>>>(p);
    else conv_gemm_kernel<false><<<2 * pairs, kThreads, kSmemBytes, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace vdt
