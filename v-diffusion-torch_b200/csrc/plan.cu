// Host runtime behind the C ABI (include/vdt_b200.h): UNet plan (block list mirroring
// unet.py:155-322), weight table with the reference's state_dict keys, 16-bit weight packing,
// TMA tensor maps, per-batch-size execution lists captured as CUDA graphs, and the sampling
// driver (diffusion.py:360-414).  No torch types; device memory via the CUDA runtime.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vdt_b200.h"
#include "kernels.cuh"

using namespace vdt;

// ================================================================================================ errors
static thread_local char g_err[1024] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}
#define CK(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define CKI(expr)                       \
    do {                                \
        int _r = (expr);                \
        if (_r != 0) return _r;         \
    } while (0)

// process-wide profiling switch and accumulators (several plans / host threads may run at once)
static std::atomic<bool> g_profile{false};
static std::mutex g_prof_mu;
static double g_prof_ms[VDT_PROF_FAMILIES] = {0, 0, 0, 0};
static uint64_t g_prof_n[VDT_PROF_FAMILIES] = {0, 0, 0, 0};
extern "C" int vdt_profile_enable(int on) { g_profile.store(on != 0); return 0; }
extern "C" int vdt_profile_read(double* ms4, uint64_t* n4) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int i = 0; i < VDT_PROF_FAMILIES; ++i) {
        if (ms4) ms4[i] = g_prof_ms[i];
        if (n4) n4[i] = g_prof_n[i];
        g_prof_ms[i] = 0; g_prof_n[i] = 0;
    }
    return 0;
}

extern "C" const char* vdt_last_error(void) { return g_err; }
extern "C" int vdt_version(void) { return 1; }
extern "C" uint64_t vdt_kernel_launches(void) { return g_launches.load(); }

// ================================================================================================ tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int get_encoder() {
    if (g_encode) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || fn == nullptr) return fail("cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

// h16 tensor, innermost dimension first; strides in elements for dims 1..rank-1
static int make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                    const uint32_t* box) {   // 2-byte elements; TMA only moves bytes, so fp16 and bf16 share the encoding
    CKI(get_encoder());
    cuuint64_t gdim[4], gstr[3];
    cuuint32_t bdim[4], estr[4];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_elems[i] * 2;
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstr, bdim, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail("cuTensorMapEncodeTiled failed (%d): rank %d dims %llu %llu %llu %llu box %u %u %u %u", (int)r, rank,
                    (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                    (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
                    rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return 0;
}

// A operand of a 3x3 (or geometric 1x1) conv: NHWC h16 [n, h, w, c]
static int make_map_nhwc(CUtensorMap* m, const void* base, int n, int h, int w, int c, int box_h, int box_n) {
    const uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)n};
    const uint64_t str[3] = {(uint64_t)c, (uint64_t)w * c, (uint64_t)h * w * c};
    const uint32_t box[4] = {64, (uint32_t)w, (uint32_t)box_h, (uint32_t)box_n};
    return make_map(m, base, 4, dims, str, box);
}
// plain row-major [rows, ld] matrix viewed through the 4-D path of the conv kernel (cols columns used)
static int make_map_rows4d(CUtensorMap* m, const void* base, long long rows, int cols, int ld) {
    const uint64_t dims[4] = {(uint64_t)cols, (uint64_t)rows, 1, 1};
    const uint64_t str[3] = {(uint64_t)ld, (uint64_t)rows * ld, (uint64_t)rows * ld};
    const uint32_t box[4] = {64, 128, 1, 1};
    return make_map(m, base, 4, dims, str, box);
}
static int make_map_2d(CUtensorMap* m, const void* base, long long rows, int cols, int ld, int box_rows) {
    const uint64_t dims[2] = {(uint64_t)cols, (uint64_t)rows};
    const uint64_t str[1] = {(uint64_t)ld};
    const uint32_t box[2] = {64, (uint32_t)box_rows};
    return make_map(m, base, 2, dims, str, box);
}

// ================================================================================================ pack kernels
__device__ __forceinline__ h16 to_h16(float x, int f16) {
    if (f16) { __half v = __float2half_rn(fminf(fmaxf(x, -65504.f), 65504.f)); return *reinterpret_cast<h16*>(&v); }
    __nv_bfloat16 v = __float2bfloat16(x);
    return *reinterpret_cast<h16*>(&v);
}
__device__ __forceinline__ float h16_to_float(h16 h, int f16) {
    return f16 ? __half2float(*reinterpret_cast<const __half*>(&h)) : __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(&h));
}
// part 0: round16(w); part 1: round16(w - round16(w)) (the "lo" half of the split-precision validation mode)
__global__ void pack_conv_w_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int I, int taps,
                                   int ktot, int koff, int f16, int part) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long n = (long long)O * I * taps;
    if (idx >= n) return;
    const int i = (int)(idx % I);
    const int tap = (int)((idx / I) % taps);
    const int o = (int)(idx / ((long long)I * taps));
    const float w = src[((long long)o * I + i) * taps + tap];
    const h16 hi = to_h16(w, f16);
    dst[(long long)o * ktot + koff + tap * I + i] = part == 0 ? hi : to_h16(w - h16_to_float(hi, f16), f16);
}
// Sub-pixel form of conv3x3(nearest_upsample_2x(x)) (kernels.cuh: ConvParams::ups): for output parity (py, px) the
// 3x3 taps that read the same low-resolution pixel are summed (fp32) into a 2x2 kernel; row r of the 3x3 kernel lands on
// low-res row offset floor((py + r - 1) / 2), i.e. py = 0: {r0} -> ty 0, {r1, r2} -> ty 1; py = 1: {r0, r1} -> ty 0,
// {r2} -> ty 1 (same for columns).  dst columns: par * par_stride + koff + (ty * 2 + tx) * I + i.
__global__ void pack_conv_ups_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int I, int ktot, int par_stride,
                                     int koff, int f16, int part) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long n = (long long)O * I * 16;
    if (idx >= n) return;
    const int i = (int)(idx % I);
    const int t = (int)((idx / I) % 4);
    const int par = (int)((idx / ((long long)I * 4)) % 4);
    const int o = (int)(idx / ((long long)I * 16));
    const int py = par >> 1, px = par & 1, ty = t >> 1, tx = t & 1;
    float w = 0.f;
    for (int r = 0; r < 3; ++r) {
        if (((py + r + 1) >> 1) - 1 + (1 - py) != ty) continue;   // floor((py + r - 1) / 2) relative to the first source row
        for (int c = 0; c < 3; ++c) {
            if (((px + c + 1) >> 1) - 1 + (1 - px) != tx) continue;
            w += src[((long long)o * I + i) * 9 + r * 3 + c];
        }
    }
    const h16 hi = to_h16(w, f16);
    dst[(long long)o * ktot + (long long)par * par_stride + koff + t * I + i] = part == 0 ? hi : to_h16(w - h16_to_float(hi, f16), f16);
}
// data gradient of a conv as a conv: dX = conv(dY, W') with W'[ci][co][tap'] = W[co][ci][taps - 1 - tap'] (transposed
// channels, 180-degree rotated filter); packed like a forward weight whose "output" channels are the conv's inputs
__global__ void pack_conv_dgrad_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int I, int taps, int f16) {
    const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long n = (long long)O * I * taps;
    if (idx >= n) return;
    const int o = (int)(idx % O);
    const int tap = (int)((idx / O) % taps);
    const int i = (int)(idx / ((long long)O * taps));
    dst[(long long)i * taps * O + (long long)tap * O + o] = to_h16(src[((long long)o * I + i) * taps + (taps - 1 - tap)], f16);
}
// in_conv: [O][C][3][3] -> [O][64], column tap*C + c (matches im2col3x3), zero padded
__global__ void pack_inconv_w_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int C, int f16, int ktot,
                                     int koff, int part) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= O * 64) return;
    const int o = idx / 64, col = idx % 64;
    float v = 0.f;
    if (col < 9 * C) { const int tap = col / C, c = col % C; v = src[((long long)o * C + c) * 9 + tap]; }
    const h16 hi = to_h16(v, f16);
    dst[(long long)o * ktot + koff + col] = part == 0 ? hi : to_h16(v - h16_to_float(hi, f16), f16);
}
// out_conv: [O][C][3][3] -> tap-major rows [tap * O + o][C] (zero rows up to the padded row count): the B operand of the
// pointwise GEMM whose nine column groups the tap-sum kernel gathers (pointwise.cu: tapsum3x3_kernel)
__global__ void pack_outconv_t_kernel(const float* __restrict__ src, h16* __restrict__ dst, int O, int C, int f16, int ktot,
                                      int koff, int part) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 9 * O * C) return;
    const int c = idx % C, row = idx / C;
    const int tap = row / O, o = row % O;
    const float v = src[((long long)o * C + c) * 9 + tap];
    const h16 hi = to_h16(v, f16);
    dst[(long long)row * ktot + koff + c] = part == 0 ? hi : to_h16(v - h16_to_float(hi, f16), f16);
}
__global__ void add_vec_kernel(const float* a, const float* b, float* out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = a[i] + (b ? b[i] : 0.f);
}
// The Python shim rejects labels outside [0, num_classes] (F.one_hot raises in the reference, modules.py:191-196); a
// C caller's out-of-range label is clamped here so that it can never index outside the FiLM table.
__global__ void film_rows_kernel(const int64_t* __restrict__ label, int* __restrict__ film_row, int rows, int rep, int ncls) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    long long r = 0;
    if (label != nullptr && !(rep == 2 && (i & 1))) r = label[i / rep];   // odd rows: y = 0 (diffusion.py:372)
    film_row[i] = (int)(r < 0 ? 0 : r > ncls ? ncls : r);
}
// multitag labels of a chunk -> per-UNet-row multi-hot rows with the CFG interleave (odd rows: all zero, diffusion.py:372)
__global__ void multitag_rows_kernel(const float* __restrict__ label, float* __restrict__ y_rows, int rows, int rep, int ncls) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * ncls) return;
    const int r = i / ncls, k = i % ncls;
    y_rows[i] = (rep == 2 && (r & 1)) ? 0.f : label[(size_t)(r / rep) * ncls + k];
}
// every per-call field is written, the inpainting pointers too (null when the call has none): execs are reused across calls
__global__ void sampler_init_state_kernel(SamplerState* st, int next_step, int start_step, int img0, int t_fp32, const float* noise,
                                          long long noise_stride, unsigned long long seed, vdt_inpaint inp) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        st->next_step = next_step; st->step = next_step; st->start_step = start_step; st->img0 = img0; st->t_fp32 = t_fp32;
        st->noise = noise; st->noise_step_stride = noise_stride; st->seed = seed;
        st->known_a = 0.f; st->known_s = 0.f;
        st->known = inp.known; st->mask = inp.mask; st->known_noise = inp.known_noise;
    }
}
__global__ void set_u64_kernel(unsigned long long* p, unsigned long long v) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *p = v;
}
__global__ void iota_i64_kernel(int64_t* p, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i;
}

// ================================================================================================ plan
struct Weight {
    std::string name;
    std::vector<int64_t> shape;
    int64_t numel = 0;
    float* dev = nullptr;
    bool loaded = false;
};

struct Block {
    int kind;            // 0 res, 1 attn
    std::string name;
    int cin, cout;
    int resample;        // kResNone/Down/Up
    bool concat, push;
    int res_in;          // input resolution
    int film_off = 0;
    // packed
    h16* w1 = nullptr;  // conv1 [cout][9*cin]            | proj_in [3*hid][cin]
    h16* w2 = nullptr;  // conv2 (+skip) [cout][9*cout(+cin)] | proj_out [cin][hid]
    float* bias2 = nullptr;   // conv2.bias (+ skip.bias)
};

enum StepKind { S_CONV, S_GN, S_ATTN, S_IM2COL, S_TEMB, S_LINEAR, S_CLSEMB, S_BEGIN, S_SAMPLE, S_ATTN_F32, S_TAPSUM, S_BEGIN_INV,
                S_INVERT };
struct TapsumArgs { const float* y; const float* bias; float* out; int B, H, W, Cout, ld; };
struct LinearArgs { const float *x, *W, *b; float* out; int rows, K, N, silu; };
struct Im2colArgs { const float* x; h16* out; h16* out_lo; int B, rep, C, H, W, f16; };
struct AttnF32Args { const float* qkv; h16 *hi, *lo; int B, N, heads, d, f16; };
struct TembArgs { const double* t; float* out; int rows, dim; const int* fp32_flag; };
struct ClsArgs { const float* e; const int64_t* y; const float* y_multi; const float *w, *b; int ncls; float* out; int rows, E; };
struct BeginArgs { SamplerState* st; const float* table; double* t_rows; int nrows, T; };

struct Step { StepKind kind; int idx; };

struct Exec {
    int rows = 0;          // UNet batch rows
    int emb_rows = 0;
    bool sampler = false;
    bool has_y = false;
    std::vector<void*> bufs;
    std::vector<size_t> buf_bytes;
    std::vector<char> buf_free;
    std::vector<Step> steps;
    std::vector<std::unique_ptr<ConvParams>> convs;
    std::vector<GroupNormParams> gns;
    std::vector<std::unique_ptr<AttnParams>> attns;
    std::vector<LinearArgs> linears;
    std::vector<Im2colArgs> im2cols;
    std::vector<AttnF32Args> attn32s;
    std::vector<TembArgs> tembs;
    std::vector<ClsArgs> clss;
    std::vector<BeginArgs> begins;
    std::vector<TapsumArgs> tapsums;
    std::vector<SamplerStepParams> samples;
    // fixed I/O staging
    float* xin = nullptr;        // forward: fp32 NCHW [rows, Cin, HW] | sampler: x_t [rows/rep, C, HW]
    float* yout = nullptr;       // fp32 NCHW [rows, Cout, HW]
    double* t_rows = nullptr;    // [emb_rows]
    int64_t* y_rows = nullptr;   // [emb_rows]
    float* y_multi = nullptr;    // multitag labels: fp32 multi-hot [emb_rows, num_classes]
    int* film_row = nullptr;     // [rows] (sampler)
    SamplerState* state = nullptr;
    unsigned long long* drop_seed = nullptr;   // training forward: seed of this call's dropout masks (device word read by the graph)
    float drop_p = 0.f;
    float* pred = nullptr;       // sampler: (guided) x0 prediction of the last executed step [rows/rep, C, HW]
    float* coef_table = nullptr; // [T][kCoefStride] (sampler)
    // sampler signature this exec was built for
    vdt_sampler_config sc{};
    int rep = 1;
    uint64_t last_use = 0;       // LRU stamp of the plan's exec cache
    cudaGraphExec_t graph = nullptr;
    bool graph_failed = false;
    int runs = 0;

    ~Exec() {
        if (graph) cudaGraphExecDestroy(graph);
        for (void* b : bufs) cudaFree(b);
    }
    int acquire(size_t bytes, void** out) {
        bytes = (bytes + 1023) & ~size_t(1023);
        int best = -1;
        for (size_t i = 0; i < bufs.size(); ++i)
            if (buf_free[i] && buf_bytes[i] >= bytes && buf_bytes[i] <= bytes + bytes / 2 &&
                (best < 0 || buf_bytes[i] < buf_bytes[best]))
                best = (int)i;
        if (best < 0) {
            void* p = nullptr;
            CK(cudaMalloc(&p, bytes));
            CK(cudaMemset(p, 0, bytes));
            bufs.push_back(p); buf_bytes.push_back(bytes); buf_free.push_back(0);
            best = (int)bufs.size() - 1;
        }
        buf_free[best] = 0;
        *out = bufs[best];
        return 0;
    }
    void release(void* p) {
        for (size_t i = 0; i < bufs.size(); ++i)
            if (bufs[i] == p) { buf_free[i] = 1; return; }
    }
};

struct vdt_plan {
    vdt_unet_config cfg{};
    int E = 0, hid = 0, levels = 0;
    int num_sms = 148;
    std::vector<Weight> weights;
    std::unordered_map<std::string, int> windex;
    std::vector<Block> blocks;
    int film_total = 0;
    bool finalized = false;
    // packed globals
    h16* w_in = nullptr;                 // in_conv [hid][64]
    h16* w_out = nullptr;                // out_conv.2 tap-major [out_rows][c0]: row tap * Cout + co (pack_outconv_t_kernel)
    int out_rows = 0;                     // 9 * out_channels rounded up to 32
    float* zero_bias = nullptr;           // [out_rows] zeros (the real bias is added by the tap-sum kernel)
    float* w_fc_all = nullptr;            // [film_total][E]
    float* b_fc_all = nullptr;            // [film_total]
    std::vector<void*> owned;
    std::map<std::string, std::unique_ptr<Exec>> execs;
    uint64_t use_clock = 0;
    unsigned long long* sat_count = nullptr;  // device counter: fp16 operand packs that hit +-65504 (saturated)
    int f16 = 1;                          // GEMM operand format: 1 fp16 (default), 0 bf16
    int split = 0;                        // 1: split-precision validation mode (every operand as a hi/lo fp16 pair)
    int stat_cols = 4;                    // columns per GroupNorm statistics entry: 4, or 2 when some group is not a multiple of 4 channels
    // all work runs on an internal stream (the caller's may be the legacy default stream, which
    // cannot be captured); ordering against the caller's stream is kept with two events
    cudaStream_t work = nullptr;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    // The chunks of a sampling batch are independent samples: they alternate between two lanes (streams, each with its
    // own workspace and step graph), so that one chunk's HBM-bound kernels (GroupNorm, small-N attention, 1x1 GEMMs)
    // can run on the SMs' spare warps while the other chunk's tensor-bound conv kernel holds the tensor cores.
    static constexpr int kLanes = 2;
    cudaStream_t lane_stream[kLanes] = {};   // [0] unused: lane 0 is `work`
    cudaEvent_t ev_fork = nullptr, ev_join[kLanes] = {};
    int sync_lanes() {
        for (int l = 1; l < kLanes; ++l)
            if (lane_stream[l] && cudaStreamSynchronize(lane_stream[l]) != cudaSuccess) return 1;
        return 0;
    }

    ~vdt_plan() {
        if (work) cudaStreamSynchronize(work);
        sync_lanes();
        execs.clear();
        if (ev_in) cudaEventDestroy(ev_in);
        if (ev_out) cudaEventDestroy(ev_out);
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (int l = 1; l < kLanes; ++l) {
            if (ev_join[l]) cudaEventDestroy(ev_join[l]);
            if (lane_stream[l]) cudaStreamDestroy(lane_stream[l]);
        }
        if (work) cudaStreamDestroy(work);
        for (auto& w : weights) if (w.dev) cudaFree(w.dev);
        for (void* p : owned) cudaFree(p);
    }
    const float* W(const std::string& k) const { return weights[windex.at(k)].dev; }
    bool has(const std::string& k) const { return windex.count(k) != 0; }
};

static int enter_work(vdt_plan* p, cudaStream_t user) {
    if (!p->work) {
        CK(cudaStreamCreateWithFlags(&p->work, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&p->ev_in, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&p->ev_out, cudaEventDisableTiming));
    }
    CK(cudaEventRecord(p->ev_in, user));
    CK(cudaStreamWaitEvent(p->work, p->ev_in, 0));
    return 0;
}
static int leave_work(vdt_plan* p, cudaStream_t user) {
    CK(cudaEventRecord(p->ev_out, p->work));
    CK(cudaStreamWaitEvent(user, p->ev_out, 0));
    return 0;
}

static void add_weight(vdt_plan* p, const std::string& name, std::vector<int64_t> shape) {
    Weight w;
    w.name = name; w.shape = shape; w.numel = 1;
    for (auto s : shape) w.numel *= s;
    p->windex[name] = (int)p->weights.size();
    p->weights.push_back(w);
}

static void attn_dims(const vdt_unet_config& c, int ch, int* hd, int* nh) {   // unet.py:43-53
    int head_dim = c.head_dim, num_heads = c.num_heads;
    if (head_dim == 0 && num_heads == 0) num_heads = 1;
    if (head_dim == 0) head_dim = ch / num_heads;
    if (num_heads == 0) num_heads = ch / head_dim;
    *hd = head_dim; *nh = num_heads;
}

// Execution order of UNet.forward (unet.py:250-283, 297-321)
static void build_blocks(vdt_plan* p) {
    const vdt_unet_config& c = p->cfg;
    const int L = c.num_levels, nrb = c.num_res_blocks, hid = c.hid_channels;
    std::vector<int> chs(L);
    for (int i = 0; i < L; ++i) chs[i] = hid * c.ch_multipliers[i];
    int res = c.resolution;
    auto add = [&](const std::string& prefix, int cin, int cout, int level, int resample, bool concat, bool push) {
        const bool has_attn = level >= 0 && c.apply_attn[level];
        Block b{};
        b.kind = 0; b.name = prefix + (has_attn ? ".0" : ""); b.cin = cin; b.cout = cout; b.resample = resample;
        b.concat = concat; b.push = push && !has_attn; b.res_in = res;
        p->blocks.push_back(b);
        if (resample == kResDown) res /= 2;
        if (resample == kResUp) res *= 2;
        if (has_attn) {
            Block a{};
            a.kind = 1; a.name = prefix + ".1"; a.cin = cout; a.cout = cout; a.resample = kResNone; a.concat = false;
            a.push = push; a.res_in = res;
            p->blocks.push_back(a);
        }
    };
    auto lvl = [](const char* side, int i, int j) {
        char buf[64];
        snprintf(buf, sizeof(buf), "%s.level_%d.%d", side, i, j);
        return std::string(buf);
    };
    for (int i = 0; i < L; ++i) {
        const int prev = i ? chs[i - 1] : hid;
        add(lvl("downsamples", i, 0), prev, chs[i], i, kResNone, false, true);
        for (int j = 1; j < nrb; ++j) add(lvl("downsamples", i, j), chs[i], chs[i], i, kResNone, false, true);
        if (i != L - 1) add(lvl("downsamples", i, nrb), chs[i], chs[i], i, kResDown, false, true);
    }
    const int mid = chs[L - 1];
    { Block b{}; b.kind = 0; b.name = "middle.0"; b.cin = b.cout = mid; b.res_in = res; p->blocks.push_back(b); }
    { Block b{}; b.kind = 1; b.name = "middle.1"; b.cin = b.cout = mid; b.res_in = res; p->blocks.push_back(b); }
    { Block b{}; b.kind = 0; b.name = "middle.2"; b.cin = b.cout = mid; b.res_in = res; p->blocks.push_back(b); }
    for (int i = L - 1; i >= 0; --i) {
        const int nxt = i == 0 ? hid : chs[i - 1];
        const int prev = i == L - 1 ? chs[L - 1] : chs[i + 1];
        const int cur = chs[i];
        add(lvl("upsamples", i, 0), prev + cur, cur, i, kResNone, true, false);
        for (int j = 1; j < nrb; ++j) add(lvl("upsamples", i, j), 2 * cur, cur, i, kResNone, true, false);
        add(lvl("upsamples", i, nrb), nxt + cur, cur, i, kResNone, true, false);
        if (i != 0) add(lvl("upsamples", i, nrb + 1), cur, cur, i, kResUp, false, false);
    }
}

extern "C" int vdt_plan_create(const vdt_unet_config* cfg, vdt_plan** out) {
    if (!cfg || !out) return fail("null argument");
    const vdt_unet_config& c = *cfg;
    if (c.num_levels < 1 || c.num_levels > VDT_MAX_LEVELS) return fail("num_levels out of range");
    if (c.hid_channels % 64 != 0) return fail("hid_channels must be a multiple of 64 (got %d)", c.hid_channels);
    if (9 * c.in_channels > 64) return fail("in_channels must be <= 7");
    if (c.out_channels > 16) return fail("out_channels must be <= 16");
    if (c.max_rows < 1) return fail("max_rows must be >= 1");
    const int minres = c.resolution >> (c.num_levels - 1);
    if ((minres << (c.num_levels - 1)) != c.resolution) return fail("resolution must be divisible by 2^(levels-1)");
    for (int i = 0, r = c.resolution; i < c.num_levels; ++i, r /= 2)
        if (r < 4 || r > 128) return fail("unsupported feature-map size %d (need 4 <= size <= 128)", r);
    std::unique_ptr<vdt_plan> p(new vdt_plan());
    p->cfg = c;
    p->hid = c.hid_channels;
    p->E = c.embedding_dim ? c.embedding_dim : 4 * c.hid_channels;
    p->levels = c.num_levels;
    if (c.operand_dtype < 0 || c.operand_dtype > 2) return fail("operand_dtype must be 0 (fp16), 1 (bf16) or 2 (fp16 x3 split)");
    p->f16 = c.operand_dtype != 1;
    p->split = c.operand_dtype == 2;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) p->num_sms = n;
    } else {
        cudaGetLastError();
    }
    build_blocks(p.get());
    const int E = p->E, hid = p->hid;
    add_weight(p.get(), "time_embed.0.weight", {E, hid});
    add_weight(p.get(), "time_embed.0.bias", {E});
    add_weight(p.get(), "time_embed.2.weight", {E, E});
    add_weight(p.get(), "time_embed.2.bias", {E});
    if (c.num_classes > 0) {
        // OneHot + Linear (keys class_embed.1.*) or, for multitag data, a stock nn.Linear (keys class_embed.*)
        add_weight(p.get(), c.multitags ? "class_embed.weight" : "class_embed.1.weight", {E, c.num_classes});
        add_weight(p.get(), c.multitags ? "class_embed.bias" : "class_embed.1.bias", {E});
    }
    add_weight(p.get(), "in_conv.weight", {hid, c.in_channels, 3, 3});
    add_weight(p.get(), "in_conv.bias", {hid});
    int film = 0;
    for (auto& b : p->blocks) {
        const std::string& n = b.name;
        if (b.kind == 0) {
            if (b.cin % 64 || b.cout % 64) return fail("channel counts must be multiples of 64 (%s: %d -> %d)", n.c_str(), b.cin, b.cout);
            add_weight(p.get(), n + ".norm1.weight", {b.cin}); add_weight(p.get(), n + ".norm1.bias", {b.cin});
            add_weight(p.get(), n + ".conv1.weight", {b.cout, b.cin, 3, 3}); add_weight(p.get(), n + ".conv1.bias", {b.cout});
            add_weight(p.get(), n + ".fc.weight", {2 * b.cout, E}); add_weight(p.get(), n + ".fc.bias", {2 * b.cout});
            add_weight(p.get(), n + ".norm2.weight", {b.cout}); add_weight(p.get(), n + ".norm2.bias", {b.cout});
            add_weight(p.get(), n + ".conv2.weight", {b.cout, b.cout, 3, 3}); add_weight(p.get(), n + ".conv2.bias", {b.cout});
            if (b.cin != b.cout) {
                add_weight(p.get(), n + ".skip.weight", {b.cout, b.cin, 1, 1}); add_weight(p.get(), n + ".skip.bias", {b.cout});
            }
            b.film_off = film;
            film += 2 * b.cout;
        } else {
            int hd, nh;
            attn_dims(c, b.cin, &hd, &nh);
            if (hd % 64 || hd > 256) return fail("head_dim must be a multiple of 64 and <= 256 (got %d)", hd);
            add_weight(p.get(), n + ".norm.weight", {b.cin}); add_weight(p.get(), n + ".norm.bias", {b.cin});
            add_weight(p.get(), n + ".proj_in.weight", {3 * hd * nh, b.cin, 1, 1}); add_weight(p.get(), n + ".proj_in.bias", {3 * hd * nh});
            add_weight(p.get(), n + ".proj_out.weight", {b.cin, hd * nh, 1, 1}); add_weight(p.get(), n + ".proj_out.bias", {b.cin});
        }
    }
    p->film_total = film;
    for (auto& b : p->blocks)
        if ((b.cin / 32) % 4 != 0 || (b.cout / 32) % 4 != 0) p->stat_cols = 2;
    if (((hid * c.ch_multipliers[0]) / 32) % 4 != 0) p->stat_cols = 2;
    const int c0 = hid * c.ch_multipliers[0];
    add_weight(p.get(), "out_conv.0.weight", {c0}); add_weight(p.get(), "out_conv.0.bias", {c0});
    add_weight(p.get(), "out_conv.2.weight", {c.out_channels, c0, 3, 3}); add_weight(p.get(), "out_conv.2.bias", {c.out_channels});
    *out = p.release();
    return 0;
}

extern "C" void vdt_plan_destroy(vdt_plan* plan) { delete plan; }
extern "C" int vdt_plan_num_weights(const vdt_plan* plan) { return plan ? (int)plan->weights.size() : 0; }
extern "C" const char* vdt_plan_weight_name(const vdt_plan* plan, int i) {
    if (!plan || i < 0 || i >= (int)plan->weights.size()) return nullptr;
    return plan->weights[i].name.c_str();
}
extern "C" int vdt_plan_weight_shape(const vdt_plan* plan, int i, int64_t* shape4, int* ndim) {
    if (!plan || i < 0 || i >= (int)plan->weights.size()) return fail("weight index out of range");
    const Weight& w = plan->weights[i];
    *ndim = (int)w.shape.size();
    for (size_t k = 0; k < w.shape.size(); ++k) shape4[k] = w.shape[k];
    return 0;
}

extern "C" int vdt_plan_load_weight(vdt_plan* plan, const char* key, const float* data, int64_t numel, int on_device) {
    if (!plan || !key || !data) return fail("null argument");
    auto it = plan->windex.find(key);
    if (it == plan->windex.end()) return fail("unexpected key in state_dict: %s", key);
    Weight& w = plan->weights[it->second];
    if (numel != w.numel) return fail("size mismatch for %s: expected %lld elements, got %lld", key, (long long)w.numel, (long long)numel);
    if (!w.dev) CK(cudaMalloc(&w.dev, sizeof(float) * (size_t)w.numel));
    CK(cudaMemcpy(w.dev, data, sizeof(float) * (size_t)w.numel, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    w.loaded = true;
    plan->finalized = false;
    return 0;
}

template <typename T>
static int dev_alloc(vdt_plan* p, T** out, size_t count) {
    void* ptr = nullptr;
    CK(cudaMalloc(&ptr, count * sizeof(T)));
    CK(cudaMemset(ptr, 0, count * sizeof(T)));
    p->owned.push_back(ptr);
    *out = reinterpret_cast<T*>(ptr);
    return 0;
}

static int pack_conv(const float* src, h16* dst, int O, int I, int taps, int ktot, int koff, int f16, int split = 0) {
    const long long n = (long long)O * I * taps;
    const int K = taps * I;
    // split mode: three consecutive K segments W_hi | W_hi | W_lo, multiplied by A_hi | A_lo | A_hi
    for (int part = 0; part < (split ? 3 : 1); ++part) {
        pack_conv_w_kernel<<<(unsigned)((n + 255) / 256), 256>>>(src, dst, O, I, taps, ktot, koff + part * K, f16, part == 2 ? 1 : 0);
        CK(cudaGetLastError());
    }
    return 0;
}

// sub-pixel upsampling conv: columns [parity][segment W_hi | W_hi | W_lo][tap][cin]
static int pack_conv_ups(const float* src, h16* dst, int O, int I, int f16, int split) {
    const long long n = (long long)O * I * 16;
    const int km = split ? 3 : 1, K = 4 * I;
    for (int part = 0; part < km; ++part) {
        pack_conv_ups_kernel<<<(unsigned)((n + 255) / 256), 256>>>(src, dst, O, I, 4 * km * K, km * K, part * K, f16, part == 2 ? 1 : 0);
        CK(cudaGetLastError());
    }
    return 0;
}

// 3x3 conv with an optional fused 1x1 skip conv (w1 != null) as extra K: columns [3x3 segments | skip segments at 9 * I3 * km]
static int pack_conv_skip(const float* w3, const float* w1, h16* dst, int O, int I3, int I1, int f16, int split) {
    const int km = split ? 3 : 1, ktot = (9 * I3 + (w1 ? I1 : 0)) * km;
    CKI(pack_conv(w3, dst, O, I3, 9, ktot, 0, f16, split));
    if (w1) CKI(pack_conv(w1, dst, O, I1, 1, ktot, 9 * I3 * km, f16, split));
    return 0;
}

// in_conv: [O][64 * km], the 64 patch columns of launch_im2col3x3 per segment
static int pack_inconv(const float* src, h16* dst, int O, int C, int f16, int split) {
    const int km = split ? 3 : 1;
    for (int part = 0; part < km; ++part) {
        pack_inconv_w_kernel<<<(O * 64 + 255) / 256, 256>>>(src, dst, O, C, f16, 64 * km, 64 * part, part == 2 ? 1 : 0);
        CK(cudaGetLastError());
    }
    return 0;
}

// out_conv as a pointwise GEMM over tap-major weight rows (9 * Cout, padded with zero rows to a multiple of 32)
static int outconv_rows(int cout) { return (9 * cout + 31) / 32 * 32; }
static int pack_outconv(const float* src, h16* dst, int O, int C, int f16, int split) {
    const int km = split ? 3 : 1;
    for (int part = 0; part < km; ++part) {            // split mode: K segments W_hi | W_hi | W_lo
        pack_outconv_t_kernel<<<(9 * O * C + 255) / 256, 256>>>(src, dst, O, C, f16, C * km, C * part, part == 2 ? 1 : 0);
        CK(cudaGetLastError());
    }
    return 0;
}

extern "C" int vdt_plan_finalize(vdt_plan* p) {
    if (!p) return fail("null plan");
    for (auto& w : p->weights)
        if (!w.loaded) return fail("missing key in state_dict: %s", w.name.c_str());
    if (p->work) CK(cudaStreamSynchronize(p->work));        // re-finalize after re-loading a key: nothing may still run
    if (p->sync_lanes()) return fail("a lane stream failed to synchronise: %s", cudaGetErrorString(cudaGetLastError()));
    p->execs.clear();
    for (void* q : p->owned) cudaFree(q);
    p->owned.clear();
    const vdt_unet_config& c = p->cfg;
    const int E = p->E, hid = p->hid;
    const int sp = p->split, km = sp ? 3 : 1;          // K multiplier of the split mode
    CKI(dev_alloc(p, &p->sat_count, 1));
    CKI(dev_alloc(p, &p->w_in, (size_t)hid * 64 * km));
    CKI(pack_inconv(p->W("in_conv.weight"), p->w_in, hid, c.in_channels, p->f16, sp));
    CKI(dev_alloc(p, &p->w_fc_all, (size_t)p->film_total * E));
    CKI(dev_alloc(p, &p->b_fc_all, (size_t)p->film_total));
    for (auto& b : p->blocks) {
        const std::string& n = b.name;
        if (b.kind == 0) {
            if (b.resample == kResUp) {                  // nearest-upsample folded into conv1 (sub-pixel form, 16 taps in all)
                CKI(dev_alloc(p, &b.w1, (size_t)b.cout * 16 * b.cin * km));
                CKI(pack_conv_ups(p->W(n + ".conv1.weight"), b.w1, b.cout, b.cin, p->f16, sp));
            } else {
                CKI(dev_alloc(p, &b.w1, (size_t)b.cout * 9 * b.cin * km));
                CKI(pack_conv(p->W(n + ".conv1.weight"), b.w1, b.cout, b.cin, 9, 9 * b.cin * km, 0, p->f16, sp));
            }
            const bool skipconv = b.cin != b.cout;
            const int k2 = (9 * b.cout + (skipconv ? b.cin : 0)) * km;
            CKI(dev_alloc(p, &b.w2, (size_t)b.cout * k2));
            CKI(pack_conv_skip(p->W(n + ".conv2.weight"), skipconv ? p->W(n + ".skip.weight") : nullptr, b.w2, b.cout, b.cout, b.cin,
                               p->f16, sp));
            CKI(dev_alloc(p, &b.bias2, (size_t)b.cout));
            add_vec_kernel<<<(b.cout + 255) / 256, 256>>>(p->W(n + ".conv2.bias"), skipconv ? p->W(n + ".skip.bias") : nullptr,
                                                          b.bias2, b.cout);
            CK(cudaGetLastError());
            CK(cudaMemcpy(p->w_fc_all + (size_t)b.film_off * E, p->W(n + ".fc.weight"), sizeof(float) * 2 * b.cout * E,
                          cudaMemcpyDeviceToDevice));
            CK(cudaMemcpy(p->b_fc_all + b.film_off, p->W(n + ".fc.bias"), sizeof(float) * 2 * b.cout, cudaMemcpyDeviceToDevice));
        } else {
            int hd, nh;
            attn_dims(c, b.cin, &hd, &nh);
            const int hidd = hd * nh;
            CKI(dev_alloc(p, &b.w1, (size_t)3 * hidd * b.cin * km));
            CKI(pack_conv(p->W(n + ".proj_in.weight"), b.w1, 3 * hidd, b.cin, 1, b.cin * km, 0, p->f16, sp));
            CKI(dev_alloc(p, &b.w2, (size_t)b.cin * hidd * km));
            CKI(pack_conv(p->W(n + ".proj_out.weight"), b.w2, b.cin, hidd, 1, hidd * km, 0, p->f16, sp));
        }
    }
    const int c0 = hid * c.ch_multipliers[0];
    p->out_rows = outconv_rows(c.out_channels);
    CKI(dev_alloc(p, &p->w_out, (size_t)p->out_rows * c0 * km));
    CKI(dev_alloc(p, &p->zero_bias, (size_t)p->out_rows));
    CKI(pack_outconv(p->W("out_conv.2.weight"), p->w_out, c.out_channels, c0, p->f16, sp));
    CK(cudaDeviceSynchronize());
    p->finalized = true;
    return 0;
}

extern "C" int vdt_stat_slabs_per_image(int32_t h, int32_t w) { return stat_slabs_per_image(h, w); }

extern "C" int vdt_plan_saturations(vdt_plan* p, uint64_t* count, int reset) {
    if (!p || !count) return fail("null argument");
    *count = 0;
    if (!p->sat_count) return 0;                        // not finalized yet: nothing has run
    if (p->work) CK(cudaStreamSynchronize(p->work));
    unsigned long long v = 0;
    CK(cudaMemcpy(&v, p->sat_count, sizeof(v), cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(p->sat_count, 0, sizeof(v)));
    *count = v;
    return 0;
}

extern "C" int vdt_plan_flops(const vdt_plan* p, double* conv, double* attn, double* linear) {
    if (!p) return fail("null plan");
    const vdt_unet_config& c = p->cfg;
    const double E = p->E, hid = p->hid;
    double fc = 0, fa = 0, fl = 0;
    double res = c.resolution;
    fc += 2.0 * res * res * hid * 9 * c.in_channels;                       // in_conv
    fl += 2.0 * (hid * E + E * E) + (c.num_classes > 0 ? 2.0 * c.num_classes * E : 0.0);
    for (const auto& b : p->blocks) {
        const double r = b.res_in, hw = r * r;
        if (b.kind == 0) {
            const double ro = b.resample == kResDown ? r / 2 : b.resample == kResUp ? r * 2 : r;
            fc += 2.0 * ro * ro * b.cout * 9.0 * (b.cin + b.cout);          // conv1 + conv2
            if (b.cin != b.cout) fc += 2.0 * ro * ro * b.cout * b.cin;     // 1x1 skip
            fl += 2.0 * E * 2 * b.cout;                                    // fc
        } else {
            int hd, nh;
            attn_dims(c, b.cin, &hd, &nh);
            const double hidd = (double)hd * nh;
            fc += 2.0 * hw * b.cin * 3 * hidd + 2.0 * hw * hidd * b.cin;   // proj_in + proj_out
            fa += 2.0 * 2.0 * hw * hw * hidd;                              // q^T k and p v
        }
    }
    fc += 2.0 * res * res * c.out_channels * 9.0 * hid * c.ch_multipliers[0];   // out_conv
    if (conv) *conv = fc;
    if (attn) *attn = fa;
    if (linear) *linear = fl;
    return 0;
}

// Can in_conv / norm1 / conv1 of block 0 be shared by the rows of a CFG pair (build_unet_steps: share0)?
static bool cfg_prefix_shareable(const vdt_plan* p) {
    if (p->split || p->blocks.empty() || getenv("VDT_NO_CFG_SHARE") != nullptr) return false;
    const auto& b0 = p->blocks[0];
    const int res = p->cfg.resolution, sc = p->stat_cols;
    const bool stats_ok = stat_slabs_per_image(res, res) > 0 && (p->hid / 32) % sc == 0 && p->hid % sc == 0;
    return b0.kind == 0 && !b0.concat && b0.cin == b0.cout && b0.cin == p->hid && b0.resample == kResNone && stats_ok;
}

// FLOPs the conv kernels actually execute per UNet row (vdt_plan_flops counts the reference's graph): in_conv runs K = 64
// for its 9 * Cin <= 64 patch columns, out_conv 32 output columns for its 9 * Cout, the conv1 of an upsampling block 16 of
// its 36 tap-GEMMs (sub-pixel form), and with cfg_rows != 0 the label-independent prefix runs once per CFG row pair.
extern "C" int vdt_plan_conv_flops_executed(const vdt_plan* p, int32_t cfg_rows, double* out) {
    if (!p || !out) return fail("null argument");
    const vdt_unet_config& c = p->cfg;
    const double hid = p->hid, res = c.resolution;
    const double share = (cfg_rows && cfg_prefix_shareable(p)) ? 0.5 : 1.0;
    double fc = share * 2.0 * res * res * hid * 64.0;
    bool first = true;
    for (const auto& b : p->blocks) {
        const double r = b.res_in, hw = r * r;
        if (b.kind == 0) {
            const double ro = b.resample == kResDown ? r / 2 : b.resample == kResUp ? r * 2 : r;
            const double taps1 = b.resample == kResUp ? 4.0 : 9.0;
            fc += (first ? share : 1.0) * 2.0 * ro * ro * b.cout * taps1 * b.cin + 2.0 * ro * ro * b.cout * 9.0 * b.cout;
            if (b.cin != b.cout) fc += 2.0 * ro * ro * b.cout * b.cin;
        } else {
            int hd, nh;
            attn_dims(c, b.cin, &hd, &nh);
            const double hidd = (double)hd * nh;
            fc += 2.0 * hw * b.cin * 3 * hidd + 2.0 * hw * hidd * b.cin;
        }
        first = false;
    }
    const int ncols = ((9 * c.out_channels + 31) / 32) * 32;
    fc += 2.0 * res * res * ncols * hid * c.ch_multipliers[0];
    *out = fc;
    return 0;
}

// ================================================================================================ conv setup
static int pick_block_n(int cout) {
    if (cout <= 256) return cout;
    for (int bn = 256; bn >= 32; bn -= 32)
        if (cout % bn == 0) return bn;
    return 0;
}

struct ConvGeom { int box_h, box_n, tiles_per_image, rows_per_tile, num_m_tiles; };
static int conv_geom(int n, int h, int w, ConvGeom* g) {
    // One M tile = one TMA box of whole image rows: box_h rows of one image (box_h | h, box_h * w <= 128), or
    // box_n whole images when an image has at most 64 pixels.  Widths that do not divide 128 (28, 14, 7: MNIST)
    // leave the tail of the 128-row tile unused (rows_per_tile < 128; those accumulator rows are never stored).
    if (w < 1 || h < 1 || w > 128) return fail("unsupported feature-map width %d", w);
    if (2 * w * h > 128) {
        int bh = 0;
        for (int d = 1; d <= h; ++d)
            if (h % d == 0 && d * w <= 128) bh = d;
        if (bh == 0) return fail("unsupported feature-map size %dx%d", h, w);
        g->box_h = bh; g->box_n = 1;
        g->tiles_per_image = h / bh; g->rows_per_tile = bh * w; g->num_m_tiles = n * g->tiles_per_image;
    } else {
        g->box_h = h; g->box_n = 128 / (w * h); g->tiles_per_image = 1; g->rows_per_tile = g->box_n * w * h;
        g->num_m_tiles = (n + g->box_n - 1) / g->box_n;
    }
    return 0;
}

// 3x3 conv (optionally with an appended pointwise K-segment) or pure pointwise GEMM
struct ConvSpec {
    const h16* a3 = nullptr; int c3 = 0;       // 3x3 segment: NHWC [n,h,w,c3]
    const h16* a1 = nullptr; int c1 = 0;       // pointwise segment: [n*h*w, c1] with row stride ld1
    const h16* a3_lo = nullptr;                // split-precision mode: lo halves of the operands above
    const h16* a1_lo = nullptr;
    int ld1 = 0;
    int n = 0, h = 0, w = 0;
    const h16* wpacked = nullptr; int cout = 0; int wrows = 0;   // weight rows actually allocated
    const float* bias = nullptr; const float* residual = nullptr;
    int out_mode = kOutF32; float* out_f32 = nullptr; h16* out_bf16 = nullptr;
    int ld = 0, act_silu = 0, f16 = 1;
    float2* stats = nullptr;
    int stat_cols = 4;
    unsigned long long* sat_count = nullptr;
    int ups = 0;          // sub-pixel 2x-upsampling conv: a3 is the LOW-res tensor [n, h, w, c3], the output is [n, 2h, 2w, cout]
    int resid_up = 0;     // residual is the low-res tensor [n, h/2, w/2, ld] of an upsampling block's identity skip
    int resid_rep = 0;    // > 1: residual holds n / resid_rep images, shared by consecutive output images (CFG row pairs)
};

static int setup_conv(const ConvSpec& s, ConvParams* cp) {
    memset(cp, 0, sizeof(*cp));
    const long long M = (long long)s.n * s.h * s.w;
    int seg = 0, ktot = 0;
    // split-precision mode: A_hi*W_hi + A_lo*W_hi + A_hi*W_lo as three K segments over the same geometry
    const h16* a3s[3] = {s.a3, s.a3_lo, s.a3};
    const h16* a1s[3] = {s.a1, s.a1_lo, s.a1};
    const int n3 = s.a3 ? (s.a3_lo ? 3 : 1) : 0, n1 = s.a1 ? (s.a1_lo ? 3 : 1) : 0;
    // GroupNorm statistics slabs (kernels.cuh: stat_slabs_per_image): flat 128-row tiles produce the same slab
    // layout as the image-aligned tiles only when an image is whole tiles (or two / four whole images are one tile)
    const int slabs = stat_slabs_per_image(s.h, s.w);
    const bool flat_ok = ((s.h * s.w) % 128 == 0) || (2 * s.h * s.w <= 128 && slabs > 0);
    const bool geo_pointwise = !s.a3 && s.stats && slabs > 0 && !flat_ok && s.ld1 == s.c1;
    if (s.a3) {
        ConvGeom g;
        CKI(conv_geom(s.n, s.h, s.w, &g));
        for (int k = 0; k < n3; ++k) {
            CKI(make_map_nhwc(&cp->a_map[seg], a3s[k], s.n, s.h, s.w, s.c3, g.box_h, g.box_n));
            cp->seg_taps[seg] = s.ups ? 4 : 9; cp->seg_kblocks[seg] = s.c3 / 64; ktot += (s.ups ? 4 : 9) * s.c3; ++seg;
        }
        if (s.ups) ktot *= 4;                            // one set of weight columns per output parity class
        cp->pointwise = 0; cp->tiles_per_image = g.tiles_per_image; cp->box_h = g.box_h; cp->box_n = g.box_n;
        cp->rows_per_tile = g.rows_per_tile; cp->num_m_tiles = g.num_m_tiles;
        for (int k = 0; k < n1; ++k) {
            // the appended pointwise segment walks the same tiles through the geometric view
            CKI(make_map_nhwc(&cp->a_map[seg], a1s[k], s.n, s.h, s.w, s.c1, g.box_h, g.box_n));
            cp->seg_taps[seg] = 1; cp->seg_kblocks[seg] = s.c1 / 64; ktot += s.c1; ++seg;
        }
    } else if (geo_pointwise) {
        // a pointwise GEMM that must write GroupNorm statistics for images that are not whole 128-row tiles walks
        // the image-aligned tiles of the 3x3 path (one tap) so that no statistics slab mixes two images
        ConvGeom g;
        CKI(conv_geom(s.n, s.h, s.w, &g));
        for (int k = 0; k < n1; ++k) {
            CKI(make_map_nhwc(&cp->a_map[seg], a1s[k], s.n, s.h, s.w, s.c1, g.box_h, g.box_n));
            cp->seg_taps[seg] = 1; cp->seg_kblocks[seg] = s.c1 / 64; ktot += s.c1; ++seg;
        }
        cp->pointwise = 0; cp->tiles_per_image = g.tiles_per_image; cp->box_h = g.box_h; cp->box_n = g.box_n;
        cp->rows_per_tile = g.rows_per_tile; cp->num_m_tiles = g.num_m_tiles;
    } else {
        for (int k = 0; k < n1; ++k) {
            CKI(make_map_rows4d(&cp->a_map[seg], a1s[k], M, s.c1, s.ld1));
            cp->seg_taps[seg] = 1; cp->seg_kblocks[seg] = s.c1 / 64; ktot += s.c1; ++seg;
        }
        cp->pointwise = 1; cp->tiles_per_image = 1; cp->box_h = 1; cp->box_n = 1; cp->rows_per_tile = 128;
        cp->num_m_tiles = (int)((M + 127) / 128);
    }
    cp->num_segs = seg;
    cp->block_n = pick_block_n(s.cout);
    if (cp->block_n == 0) return fail("unsupported output channel count %d", s.cout);
    cp->num_n_tiles = (s.cout + cp->block_n - 1) / cp->block_n;
    CKI(make_map_2d(&cp->b_map, s.wpacked, s.wrows, ktot, ktot, cp->block_n / 2));   // each CTA of a pair fetches half
    cp->M = (int)M; cp->Cout = s.cout; cp->out_mode = s.out_mode; cp->ld = s.ld;
    cp->HW = s.h * s.w; cp->act_silu = s.act_silu; cp->f16 = s.f16;
    cp->bias = s.bias; cp->residual = s.residual; cp->out_f32 = s.out_f32; cp->out_bf16 = s.out_bf16; cp->stat_cols = s.stat_cols;
    cp->stats = (slabs > 0 && (s.a3 || flat_ok || geo_pointwise)) ? s.stats : nullptr;   // statistics slabs never span two images
    cp->ups = s.ups; cp->ups_w = s.w; cp->stat_slabs_img = slabs; cp->resid_up = s.resid_up; cp->out_w = s.w;
    cp->resid_rep = s.residual ? s.resid_rep : 0;
    {
        const char* pt = getenv("VDT_PAIR_TILES");
        if (cp->resid_rep == 2 && !cp->pointwise && cp->box_n == 1 && cp->tiles_per_image >= 1 &&
            cp->num_m_tiles == s.n * cp->tiles_per_image && s.n % 2 == 0 && !(pt && pt[0] == '0'))
            cp->pair_tiles = cp->tiles_per_image;
    }
    if (s.resid_rep > 1 && (s.resid_up || s.ups || s.n % s.resid_rep != 0)) return fail("internal: shared residual on a resampling conv");
    cp->map_shift = -1;                                  // fast row remaps need square power-of-two maps of >= 64 (ups) / 256 pixels
    if ((s.ups || s.resid_up || s.resid_rep > 1) && s.h == s.w && (s.w & (s.w - 1)) == 0)
        for (int k = 3; k < 16; ++k) if ((1 << k) == s.w) cp->map_shift = k;
    if (s.ups && (s.a1 || !s.a3)) return fail("internal: the sub-pixel upsampling conv takes a single 3x3 operand");
    if (s.ups && s.stats && 4 * slabs != stat_slabs_per_image(2 * s.h, 2 * s.w)) cp->stats = nullptr;   // callers check fusability first
    if (s.resid_up && ((s.h | s.w) & 1)) return fail("internal: upsampled residual needs even output sizes");
    cp->sat_count = s.sat_count;
    if (s.cout % 32 != 0) return fail("output channels must be a multiple of 32 (got %d)", s.cout);
    return 0;
}

// ================================================================================================ exec build
static int build_unet_steps(vdt_plan* p, Exec* ex, const float* film, const int* film_row) {
    const vdt_unet_config& c = p->cfg;
    const int R = ex->rows, hid = p->hid;
    int res = c.resolution;
    auto add_conv = [&](const ConvSpec& s) -> int {
        std::unique_ptr<ConvParams> cp(new ConvParams());
        CKI(setup_conv(s, cp.get()));
        ex->convs.push_back(std::move(cp));
        ex->steps.push_back({S_CONV, (int)ex->convs.size() - 1});
        return 0;
    };
    auto add_gn = [&](const GroupNormParams& g) {
        ex->gns.push_back(g);
        ex->steps.push_back({S_GN, (int)ex->gns.size() - 1});
    };
    // ---- in_conv
    // every fp32 stream tensor carries the partial GroupNorm statistics its producing conv wrote
    const int scols = p->stat_cols;
    auto stats_bytes = [&](size_t imgs, int r, int ch) {    // imgs images at r x r
        return ((size_t)imgs * stat_slabs_per_image(r, r) + 4) * (size_t)(ch / scols) * sizeof(float2);
    };
    const bool sp = p->split != 0;
    auto fusable = [scols](int c1, int c2, int r) {   // can a GroupNorm over concat(c1, c2) at r x r use epilogue statistics?
        const int cpg = (c1 + c2) / 32;
        // groups may straddle the concat seam (finalize handles it); no statistics slab may mix two images
        return cpg % scols == 0 && c1 % scols == 0 && stat_slabs_per_image(r, r) > 0;
    };
    // Under CFG the cond / uncond rows of a sample (rows 2i, 2i + 1) see the same x_t and t and differ only in the class
    // embedding, which first enters at the FiLM of block 0's norm2: in_conv, norm1 and conv1 of block 0 are computed once
    // per SAMPLE, norm2 / conv2's identity skip / the last up block's concat read the shared tensors (GroupNormParams::rep1,
    // ConvParams::resid_rep).  Same arithmetic in the same order: results are bit-identical to the row-by-row path.
    const bool share0 = ex->rep == 2 && cfg_prefix_shareable(p);
    const int R0 = share0 ? R / ex->rep : R;                // rows of the tensors computed before the first FiLM
    h16* patches; h16* patches_lo = nullptr; float* h; float2* hst;
    const size_t hw0 = (size_t)res * res;
    CKI(ex->acquire((size_t)R0 * hw0 * 64 * 2, (void**)&patches));
    if (sp) CKI(ex->acquire((size_t)R0 * hw0 * 64 * 2, (void**)&patches_lo));
    ex->im2cols.push_back({ex->xin, patches, patches_lo, R / ex->rep, share0 ? 1 : ex->rep, c.in_channels, res, res, p->f16});
    ex->steps.push_back({S_IM2COL, (int)ex->im2cols.size() - 1});
    CKI(ex->acquire((size_t)R0 * hw0 * hid * 4, (void**)&h));
    CKI(ex->acquire(stats_bytes(R0, res, hid), (void**)&hst));
    {
        ConvSpec s;
        s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
        s.a1 = patches; s.a1_lo = patches_lo; s.c1 = 64; s.ld1 = 64; s.n = R0; s.h = res; s.w = res; s.wpacked = p->w_in; s.cout = hid; s.wrows = hid;
        s.bias = p->W("in_conv.bias"); s.out_mode = kOutF32; s.out_f32 = h; s.ld = hid; s.stats = hst;
        CKI(add_conv(s));
    }
    ex->release(patches);
    float2* meanrstd;                                 // (mean, rstd) scratch shared by all GroupNorms (stream-ordered)
    CKI(ex->acquire((size_t)R * 32 * sizeof(float2), (void**)&meanrstd));
    struct Skip { float* ptr; float2* stats; int ch; int rep; };   // rep 2: R / 2 images shared by the rows of a CFG pair
    std::vector<Skip> stack;
    stack.push_back({h, hst, hid, share0 ? ex->rep : 1});
    bool h_on_stack = true;      // h aliases the top stack entry -> must not be released when replaced
    int hch = hid;
    int h_rep = share0 ? ex->rep : 1;                       // > 1 only between in_conv and block 0's norm2

    for (auto& b : p->blocks) {
        const std::string& n = b.name;
        const int HW = res * res;
        if (b.kind == 0) {
            const float* src2 = nullptr; int c2 = 0; float* src2_buf = nullptr; float2* st2 = nullptr; int rep2 = 1;
            if (b.concat) { Skip sk = stack.back(); stack.pop_back(); src2 = sk.ptr; c2 = sk.ch; src2_buf = sk.ptr; st2 = sk.stats; rep2 = sk.rep; }
            // rows of norm1 / conv1: the shared count while h is still label-independent (block 0 under CFG, see share0)
            const int Rn = R / h_rep;
            if (h_rep > 1 && (b.concat || b.cin != b.cout || b.resample != kResNone))
                return fail("internal: shared rows reach a block that cannot take them (%s)", n.c_str());
            const int cin = hch + c2;
            if (cin != b.cin) return fail("internal: channel bookkeeping mismatch at %s (%d vs %d)", n.c_str(), cin, b.cin);
            const bool skipconv = b.cin != b.cout;
            const int ro = b.resample == kResDown ? res / 2 : b.resample == kResUp ? res * 2 : res;
            const size_t HWo = (size_t)ro * ro;
            // an upsampling block never materialises the upsampled tensors: norm1 runs at the input resolution, conv1 is
            // the sub-pixel form of conv3x3(upsample(.)) and conv2's identity-skip residual reads the low-res stream
            const bool up = b.resample == kResUp;
            if (up && skipconv) return fail("internal: an upsampling block with a skip conv is not part of the reference (%s)", n.c_str());
            const int ra = up ? res : ro;                       // resolution of conv1's A operand
            const size_t HWa = (size_t)ra * ra;
            h16 *a1, *xraw = nullptr, *a1_lo = nullptr, *xraw_lo = nullptr; float* xres = nullptr;
            CKI(ex->acquire((size_t)Rn * HWa * cin * 2, (void**)&a1));
            if (sp) CKI(ex->acquire((size_t)Rn * HWa * cin * 2, (void**)&a1_lo));
            if (skipconv) CKI(ex->acquire((size_t)R * HW * cin * 2, (void**)&xraw));
            if (skipconv && sp) CKI(ex->acquire((size_t)R * HW * cin * 2, (void**)&xraw_lo));
            if (b.resample == kResDown) CKI(ex->acquire((size_t)R * HWo * cin * 4, (void**)&xres));
            GroupNormParams g{};
            g.f16 = p->f16; g.stat_cols = p->stat_cols; g.sat_count = p->sat_count;
            g.src1 = h; g.C1 = hch; g.src2 = src2; g.C2 = c2; g.B = Rn; g.H = res; g.W = res;
            g.rep2 = rep2 > 1 ? rep2 : 0;                   // the in_conv output popped by the last up block may be shared
            if (fusable(hch, c2, res)) { g.stats1 = hst; g.stats2 = st2; g.meanrstd = meanrstd; g.stat_slabs = stat_slabs_per_image(res, res); }
            g.gamma = p->W(n + ".norm1.weight"); g.beta = p->W(n + ".norm1.bias");
            g.silu = 1; g.resample = up ? kResNone : b.resample; g.out_act = a1; g.out_raw = xraw; g.out_res = xres;
            g.out_act_lo = a1_lo; g.out_raw_lo = xraw_lo;
            add_gn(g);
            // conv1: its output only feeds norm2, so it is kept in the 16-bit operand format when norm2 can use
            // the epilogue statistics (otherwise fp32 for the two-pass fallback)
            const bool fuse2 = fusable(b.cout, 0, ro) &&
                               (!up || 4 * stat_slabs_per_image(res, res) == stat_slabs_per_image(ro, ro));
            // (split-precision mode keeps every stream tensor fp32)
            const bool h1_16 = fuse2 && !sp;
            void* h1; float2* h1st = nullptr;
            if (h_rep > 1 && !h1_16) return fail("internal: shared rows need the single-pass norm2 (%s)", n.c_str());
            CKI(ex->acquire((size_t)Rn * HWo * b.cout * (h1_16 ? 2 : 4), &h1));
            if (fuse2) CKI(ex->acquire(stats_bytes(Rn, ro, b.cout), (void**)&h1st));
            {
                ConvSpec s;
                s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
                s.a3 = a1; s.a3_lo = a1_lo; s.c3 = cin; s.n = Rn; s.h = ra; s.w = ra; s.wpacked = b.w1; s.cout = b.cout; s.wrows = b.cout;
                s.ups = up ? 1 : 0;
                s.bias = p->W(n + ".conv1.bias"); s.ld = b.cout; s.stats = h1st;
                if (h1_16) { s.out_mode = kOutBF16; s.out_bf16 = (h16*)h1; } else { s.out_mode = kOutF32; s.out_f32 = (float*)h1; }
                CKI(add_conv(s));
            }
            ex->release(a1);
            if (a1_lo) ex->release(a1_lo);
            // norm2 + FiLM + SiLU
            h16* a2; h16* a2_lo = nullptr;
            CKI(ex->acquire((size_t)R * HWo * b.cout * 2, (void**)&a2));
            if (sp) CKI(ex->acquire((size_t)R * HWo * b.cout * 2, (void**)&a2_lo));
            GroupNormParams g2{};
            g2.f16 = p->f16; g2.stat_cols = p->stat_cols; g2.sat_count = p->sat_count;
            g2.src1 = h1; g2.C1 = b.cout; g2.B = R; g2.H = ro; g2.W = ro; g2.in16 = h1_16 ? 1 : 0;
            g2.stats1 = h1st; g2.meanrstd = meanrstd; g2.stat_slabs = stat_slabs_per_image(ro, ro);
            g2.rep1 = h_rep > 1 ? h_rep : 0;                // every row of a CFG pair normalises the shared conv1 output with its own FiLM
            g2.out_act_lo = a2_lo;
            g2.gamma = p->W(n + ".norm2.weight"); g2.beta = p->W(n + ".norm2.bias");
            g2.film = film; g2.film_row = film_row; g2.film_stride = p->film_total; g2.film_off = b.film_off;
            g2.silu = 1; g2.resample = kResNone; g2.out_act = a2;
            if (ex->drop_p > 0.f) {                      // training mode: nn.Dropout between act2 and conv2 (unet.py:135, 146)
                g2.drop_p = ex->drop_p; g2.drop_seed = ex->drop_seed; g2.drop_layer = (int)ex->gns.size();
            }
            add_gn(g2);
            ex->release(h1);
            if (h1st) ex->release(h1st);
            // conv2 (+ fused 1x1 skip conv as extra K) + residual
            float* hout; float2* houtst;
            CKI(ex->acquire((size_t)R * HWo * b.cout * 4, (void**)&hout));
            CKI(ex->acquire(stats_bytes(R, ro, b.cout), (void**)&houtst));
            {
                ConvSpec s;
                s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
                s.a3 = a2; s.a3_lo = a2_lo; s.c3 = b.cout; s.n = R; s.h = ro; s.w = ro; s.wpacked = b.w2; s.cout = b.cout; s.wrows = b.cout;
                if (skipconv) { s.a1 = xraw; s.a1_lo = xraw_lo; s.c1 = cin; s.ld1 = cin; }
                s.bias = b.bias2;
                s.residual = skipconv ? nullptr : (b.resample == kResDown ? xres : h);
                s.resid_up = (up && !skipconv) ? 1 : 0;
                s.resid_rep = (h_rep > 1 && s.residual == h) ? h_rep : 0;
                s.out_mode = kOutF32; s.out_f32 = hout; s.ld = b.cout; s.stats = houtst;
                CKI(add_conv(s));
            }
            ex->release(a2);
            if (a2_lo) ex->release(a2_lo);
            if (xraw_lo) ex->release(xraw_lo);
            if (xraw) ex->release(xraw);
            if (xres) ex->release(xres);
            if (src2_buf) { ex->release(src2_buf); ex->release(st2); }
            if (!h_on_stack) { ex->release(h); ex->release(hst); }
            h = hout; hst = houtst; hch = b.cout; h_on_stack = false; res = ro; h_rep = 1;
        } else {
            int hd, nh;
            attn_dims(c, b.cin, &hd, &nh);
            const int hidd = hd * nh, N = HW;
            h16 *a, *a_lo = nullptr, *qkv = nullptr, *o, *o_lo = nullptr;
            CKI(ex->acquire((size_t)R * HW * b.cin * 2, (void**)&a));
            if (sp) CKI(ex->acquire((size_t)R * HW * b.cin * 2, (void**)&a_lo));
            GroupNormParams g{};
            g.f16 = p->f16; g.stat_cols = p->stat_cols; g.sat_count = p->sat_count;
            g.src1 = h; g.C1 = hch; g.B = R; g.H = res; g.W = res;
            if (fusable(hch, 0, res)) { g.stats1 = hst; g.meanrstd = meanrstd; g.stat_slabs = stat_slabs_per_image(res, res); }
            g.gamma = p->W(n + ".norm.weight"); g.beta = p->W(n + ".norm.bias");
            g.silu = 0; g.resample = kResNone; g.out_act = a; g.out_act_lo = a_lo;
            add_gn(g);
            CKI(ex->acquire((size_t)R * N * hidd * 2, (void**)&o));
            if (!sp) {
                CKI(ex->acquire((size_t)R * N * 3 * hidd * 2, (void**)&qkv));
                {   // one GEMM for q | k | v, all row-major [R*N, 3*hid]: the attention kernel reads V as an MN-major operand
                    ConvSpec s;
                    s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
                    s.a1 = a; s.c1 = b.cin; s.ld1 = b.cin; s.n = R; s.h = res; s.w = res; s.wpacked = b.w1; s.cout = 3 * hidd;
                    s.wrows = 3 * hidd; s.bias = p->W(n + ".proj_in.bias"); s.out_mode = kOutBF16; s.out_bf16 = qkv;
                    s.ld = 3 * hidd;
                    CKI(add_conv(s));
                }
                ex->release(a);
                std::unique_ptr<AttnParams> ap(new AttnParams());
                memset(ap.get(), 0, sizeof(AttnParams));
                CKI(make_map_2d(&ap->q_map, qkv, (long long)R * N, 3 * hidd, 3 * hidd, 128));
                CKI(make_map_2d(&ap->kv_map, qkv, (long long)R * N, 3 * hidd, 3 * hidd, 64));
                ap->B = R; ap->N = N; ap->heads = nh; ap->d = hd; ap->hid = hidd; ap->f16 = p->f16;
                ap->scale_log2e = (float)(1.4426950408889634 / std::sqrt((double)hd));
                ap->out = o;
                ex->attns.push_back(std::move(ap));
                ex->steps.push_back({S_ATTN, (int)ex->attns.size() - 1});
                ex->release(qkv);
            } else {
                // split-precision validation mode: q | k | v in fp32, attention on CUDA cores in fp32
                float* qkv32;
                CKI(ex->acquire((size_t)R * N * 3 * hidd * 4, (void**)&qkv32));
                CKI(ex->acquire((size_t)R * N * hidd * 2, (void**)&o_lo));
                {
                    ConvSpec s;
                    s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
                    s.a1 = a; s.a1_lo = a_lo; s.c1 = b.cin; s.ld1 = b.cin; s.n = R; s.h = res; s.w = res; s.wpacked = b.w1;
                    s.cout = 3 * hidd; s.wrows = 3 * hidd; s.bias = p->W(n + ".proj_in.bias"); s.out_mode = kOutF32; s.out_f32 = qkv32;
                    s.ld = 3 * hidd;
                    CKI(add_conv(s));
                }
                ex->release(a); ex->release(a_lo);
                ex->attn32s.push_back({qkv32, o, o_lo, R, N, nh, hd, p->f16});
                ex->steps.push_back({S_ATTN_F32, (int)ex->attn32s.size() - 1});
                ex->release(qkv32);
            }
            float* hout; float2* houtst;
            CKI(ex->acquire((size_t)R * HW * b.cin * 4, (void**)&hout));
            CKI(ex->acquire(stats_bytes(R, res, b.cin), (void**)&houtst));
            {
                ConvSpec s;
                s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
                s.a1 = o; s.a1_lo = o_lo; s.c1 = hidd; s.ld1 = hidd; s.n = R; s.h = res; s.w = res; s.wpacked = b.w2; s.cout = b.cin; s.wrows = b.cin;
                s.bias = p->W(n + ".proj_out.bias"); s.residual = h; s.out_mode = kOutF32; s.out_f32 = hout; s.ld = b.cin;
                s.stats = houtst;
                CKI(add_conv(s));
            }
            ex->release(o);
            if (o_lo) ex->release(o_lo);
            if (!h_on_stack) { ex->release(h); ex->release(hst); }
            h = hout; hst = houtst; h_on_stack = false;
        }
        if (b.push) { stack.push_back({h, hst, hch, 1}); h_on_stack = true; }
    }
    if (!stack.empty()) return fail("internal: skip stack not empty (%d)", (int)stack.size());
    // ---- out_conv
    {
        const int HW = res * res;
        h16* a; h16* a_lo = nullptr;
        CKI(ex->acquire((size_t)R * HW * hch * 2, (void**)&a));
        if (sp) CKI(ex->acquire((size_t)R * HW * hch * 2, (void**)&a_lo));
        GroupNormParams g{};
        g.f16 = p->f16; g.stat_cols = p->stat_cols; g.sat_count = p->sat_count;
        g.src1 = h; g.C1 = hch; g.B = R; g.H = res; g.W = res;
        if (fusable(hch, 0, res)) { g.stats1 = hst; g.meanrstd = meanrstd; g.stat_slabs = stat_slabs_per_image(res, res); }
        g.gamma = p->W("out_conv.0.weight"); g.beta = p->W("out_conv.0.bias");
        g.silu = 1; g.resample = kResNone; g.out_act = a; g.out_act_lo = a_lo;
        add_gn(g);
        // 3x3 conv with a handful of output channels: pointwise GEMM Y[pixel, tap * Cout + co] (the activation is read
        // once instead of once per tap) + the tap-sum gather into the NCHW network output (pointwise.cu)
        float* ytap;
        CKI(ex->acquire((size_t)R * HW * p->out_rows * 4, (void**)&ytap));
        ConvSpec s;
        s.f16 = p->f16; s.stat_cols = p->stat_cols; s.sat_count = p->sat_count;
        s.a1 = a; s.a1_lo = a_lo; s.c1 = hch; s.ld1 = hch; s.n = R; s.h = res; s.w = res; s.wpacked = p->w_out;
        s.cout = p->out_rows; s.wrows = p->out_rows; s.bias = p->zero_bias; s.out_mode = kOutF32; s.out_f32 = ytap; s.ld = p->out_rows;
        CKI(add_conv(s));
        ex->tapsums.push_back({ytap, p->W("out_conv.2.bias"), ex->yout, R, res, res, c.out_channels, p->out_rows});
        ex->steps.push_back({S_TAPSUM, (int)ex->tapsums.size() - 1});
        ex->release(ytap);
        if (a_lo) ex->release(a_lo);
        ex->release(a);
        if (!h_on_stack) { ex->release(h); ex->release(hst); }
    }
    return 0;
}

static int add_embedding_steps(vdt_plan* p, Exec* ex, float* film, bool has_y) {
    const int E = p->E, hid = p->hid, ER = ex->emb_rows;
    float *temb, *e1, *e2, *act;
    CKI(ex->acquire((size_t)ER * hid * 4, (void**)&temb));
    CKI(ex->acquire((size_t)ER * E * 4, (void**)&e1));
    CKI(ex->acquire((size_t)ER * E * 4, (void**)&e2));
    CKI(ex->acquire((size_t)ER * E * 4, (void**)&act));
    ex->tembs.push_back({ex->t_rows, temb, ER, hid, ex->state ? &ex->state->t_fp32 : nullptr});
    ex->steps.push_back({S_TEMB, (int)ex->tembs.size() - 1});
    ex->linears.push_back({temb, p->W("time_embed.0.weight"), p->W("time_embed.0.bias"), e1, ER, hid, E, 1});
    ex->steps.push_back({S_LINEAR, (int)ex->linears.size() - 1});
    ex->linears.push_back({e1, p->W("time_embed.2.weight"), p->W("time_embed.2.bias"), e2, ER, E, E, 0});
    ex->steps.push_back({S_LINEAR, (int)ex->linears.size() - 1});
    const bool cls = p->cfg.num_classes > 0 && has_y;
    const bool mt = p->cfg.multitags != 0;
    ex->clss.push_back({e2, (cls && !mt) ? ex->y_rows : nullptr, (cls && mt) ? ex->y_multi : nullptr,
                        cls ? p->W(mt ? "class_embed.weight" : "class_embed.1.weight") : nullptr,
                        cls ? p->W(mt ? "class_embed.bias" : "class_embed.1.bias") : nullptr, p->cfg.num_classes, act, ER, E});
    ex->steps.push_back({S_CLSEMB, (int)ex->clss.size() - 1});
    ex->linears.push_back({act, p->w_fc_all, p->b_fc_all, film, ER, E, p->film_total, 0});
    ex->steps.push_back({S_LINEAR, (int)ex->linears.size() - 1});
    // temb/e1/e2/act stay allocated for the life of the exec (tiny)
    return 0;
}

static int run_steps(vdt_plan* p, Exec* ex, cudaStream_t st, std::vector<cudaEvent_t>* evs = nullptr) {
    size_t ei = 0;
    for (const Step& s : ex->steps) {
        cudaError_t e = cudaSuccess;
        if (evs) cudaEventRecord((*evs)[ei++], st);
        switch (s.kind) {
            case S_CONV: e = launch_conv_gemm(*ex->convs[s.idx], p->num_sms, st); break;
            case S_GN: e = launch_groupnorm(ex->gns[s.idx], st); break;
            case S_ATTN: e = launch_attention(*ex->attns[s.idx], p->num_sms, st); break;
            case S_IM2COL: { auto& a = ex->im2cols[s.idx]; e = launch_im2col3x3(a.x, a.out, a.out_lo, a.B, a.rep, a.C, a.H, a.W, a.f16, st); break; }
            case S_TEMB: { auto& a = ex->tembs[s.idx]; e = launch_timestep_embedding(a.t, a.out, a.rows, a.dim, a.fp32_flag, st); break; }
            case S_LINEAR: { auto& a = ex->linears[s.idx]; e = launch_linear_f32(a.x, a.W, a.b, a.out, a.rows, a.K, a.N, a.silu, st); break; }
            case S_CLSEMB: {
                auto& a = ex->clss[s.idx];
                e = a.y_multi ? launch_class_embed_multitag_silu(a.e, a.y_multi, a.w, a.b, a.ncls, a.out, a.rows, a.E, st)
                              : launch_class_embed_silu(a.e, a.y, a.w, a.b, a.ncls, a.out, a.rows, a.E, st);
                break;
            }
            case S_BEGIN: { auto& a = ex->begins[s.idx]; e = launch_sampler_begin_step(a.st, a.table, a.t_rows, a.nrows, a.T, st); break; }
            case S_SAMPLE: e = launch_sampler_step(ex->samples[s.idx], st); break;
            case S_BEGIN_INV: { auto& a = ex->begins[s.idx]; e = launch_invert_begin_step(a.st, a.table, a.t_rows, a.nrows, a.T, st); break; }
            case S_INVERT: e = launch_invert_step(ex->samples[s.idx], st); break;
            case S_TAPSUM: { auto& a = ex->tapsums[s.idx]; e = launch_tapsum3x3(a.y, a.bias, a.out, a.B, a.H, a.W, a.Cout, a.ld, st); break; }
            case S_ATTN_F32: { auto& a = ex->attn32s[s.idx]; e = launch_attention_f32(a.qkv, a.hi, a.lo, a.B, a.N, a.heads, a.d, a.f16, st); break; }
        }
        if (e != cudaSuccess) return fail("kernel launch failed (step kind %d): %s", (int)s.kind, cudaGetErrorString(e));
    }
    if (evs) cudaEventRecord((*evs)[ei], st);
    return 0;
}

static int run_steps_profiled(vdt_plan* p, Exec* ex, cudaStream_t st) {
    std::vector<cudaEvent_t> evs(ex->steps.size() + 1);
    for (auto& e : evs) CK(cudaEventCreate(&e));
    int rc = run_steps(p, ex, st, &evs);
    if (rc == 0) {
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = fail("profiled step failed: %s", cudaGetErrorString(e));
    }
    if (rc == 0) {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        for (size_t i = 0; i < ex->steps.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, evs[i], evs[i + 1]);
            const StepKind k = ex->steps[i].kind;
            const int fam = k == S_CONV ? VDT_PROF_CONV : k == S_GN ? VDT_PROF_GROUPNORM : (k == S_ATTN || k == S_ATTN_F32) ? VDT_PROF_ATTENTION : VDT_PROF_OTHER;
            g_prof_ms[fam] += ms; g_prof_n[fam] += 1;
        }
    }
    for (auto& e : evs) cudaEventDestroy(e);
    return rc;
}

// Run the exec's step list, through a CUDA graph once it has been captured.
static int run_exec(vdt_plan* p, Exec* ex, cudaStream_t st) {
    if (g_profile.load()) { g_launches += ex->steps.size(); return run_steps_profiled(p, ex, st); }
    // first run is eager (sets function attributes, surfaces launch errors); the second run captures
    if (!ex->graph && !ex->graph_failed && ex->runs++ >= 1) {
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            const int r = run_steps(p, ex, st);
            cudaError_t e2 = cudaStreamEndCapture(st, &g);
            if (r != 0) { if (g) cudaGraphDestroy(g); return r; }
            if (e2 == cudaSuccess && g) {
                if (cudaGraphInstantiate(&ex->graph, g, 0) != cudaSuccess) { ex->graph = nullptr; ex->graph_failed = true; }
                cudaGraphDestroy(g);
            } else {
                ex->graph_failed = true;
            }
        } else {
            ex->graph_failed = true;
        }
        cudaGetLastError();
    }
    g_launches += ex->steps.size();
    if (ex->graph) {
        CK(cudaGraphLaunch(ex->graph, st));
    } else {
        CKI(run_steps(p, ex, st));
    }
    return 0;
}

// The plan keeps a handful of execs (workspace + captured graph per batch size / sampler signature).  A miss on a full
// cache evicts the least recently used entry only; queued work may still use its buffers, hence the stream sync.
// Six entries: a sampling call uses up to three (a full chunk per lane and a ragged tail), which leaves room for plain
// forwards and other batch sizes before an eviction makes a later call rebuild a workspace and re-capture its graph.
constexpr size_t kMaxExecs = 6;
static int exec_cache_lookup(vdt_plan* p, const std::string& key, Exec** out) {
    auto it = p->execs.find(key);
    if (it == p->execs.end()) { *out = nullptr; return 0; }
    it->second->last_use = ++p->use_clock;
    *out = it->second.get();
    return 0;
}
static int exec_cache_make_room(vdt_plan* p) {
    while (p->execs.size() >= kMaxExecs) {
        auto victim = p->execs.begin();
        for (auto it = p->execs.begin(); it != p->execs.end(); ++it)
            if (it->second->last_use < victim->second->last_use) victim = it;
        if (p->work) CK(cudaStreamSynchronize(p->work));
        if (p->sync_lanes()) return fail("a lane stream failed to synchronise: %s", cudaGetErrorString(cudaGetLastError()));
        p->execs.erase(victim);
    }
    return 0;
}

static int get_forward_exec(vdt_plan* p, int rows, bool has_y, float drop_p, Exec** out) {
    char key[96];
    snprintf(key, sizeof(key), "fwd:%d:%d:%.9g", rows, (int)has_y, (double)drop_p);
    CKI(exec_cache_lookup(p, key, out));
    if (*out) return 0;
    CKI(exec_cache_make_room(p));
    std::unique_ptr<Exec> ex(new Exec());
    ex->last_use = ++p->use_clock;
    const vdt_unet_config& c = p->cfg;
    const size_t HW = (size_t)c.resolution * c.resolution;
    ex->rows = rows; ex->emb_rows = rows; ex->sampler = false; ex->has_y = has_y; ex->rep = 1;
    ex->drop_p = drop_p;
    if (drop_p > 0.f) CKI(ex->acquire(sizeof(unsigned long long), (void**)&ex->drop_seed));
    CKI(ex->acquire(rows * HW * c.in_channels * 4, (void**)&ex->xin));
    CKI(ex->acquire(rows * HW * c.out_channels * 4, (void**)&ex->yout));
    CKI(ex->acquire(rows * sizeof(double), (void**)&ex->t_rows));
    CKI(ex->acquire(rows * sizeof(int64_t), (void**)&ex->y_rows));
    if (c.multitags && c.num_classes > 0) CKI(ex->acquire((size_t)rows * c.num_classes * 4, (void**)&ex->y_multi));
    float* film;
    CKI(ex->acquire((size_t)rows * p->film_total * 4, (void**)&film));
    CKI(add_embedding_steps(p, ex.get(), film, has_y));
    CKI(build_unet_steps(p, ex.get(), film, nullptr));
    *out = ex.get();
    p->execs[key] = std::move(ex);
    return 0;
}

static int unet_forward_impl(vdt_plan* p, const float* x, const double* t, const void* y, float* out, int32_t batch,
                             float drop_p, unsigned long long seed, void* stream) {
    if (!p || !x || !t || !out) return fail("null argument");
    if (!p->finalized) return fail("plan not finalized (load every state_dict key, then vdt_plan_finalize)");
    if (!(drop_p >= 0.f && drop_p < 1.f)) return fail("drop_rate must lie in [0, 1) (got %g)", (double)drop_p);
    cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
    CKI(enter_work(p, user));
    cudaStream_t st = p->work;
    const vdt_unet_config& c = p->cfg;
    const size_t HW = (size_t)c.resolution * c.resolution;
    for (int b0 = 0; b0 < batch; b0 += c.max_rows) {
        const int rows = std::min(c.max_rows, batch - b0);
        Exec* ex;
        CKI(get_forward_exec(p, rows, y != nullptr, drop_p, &ex));
        CK(cudaMemcpyAsync(ex->xin, x + (size_t)b0 * c.in_channels * HW, rows * HW * c.in_channels * 4, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(ex->t_rows, t + b0, rows * sizeof(double), cudaMemcpyDeviceToDevice, st));
        if (y && c.multitags)
            CK(cudaMemcpyAsync(ex->y_multi, static_cast<const float*>(y) + (size_t)b0 * c.num_classes,
                               (size_t)rows * c.num_classes * 4, cudaMemcpyDeviceToDevice, st));
        else if (y)
            CK(cudaMemcpyAsync(ex->y_rows, static_cast<const int64_t*>(y) + b0, rows * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        if (ex->drop_seed) {                             // every chunk of the batch draws its own masks
            set_u64_kernel<<<1, 1, 0, st>>>(ex->drop_seed, seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(b0 + 1));
            CK(cudaGetLastError());
        }
        CKI(run_exec(p, ex, st));
        CK(cudaMemcpyAsync(out + (size_t)b0 * c.out_channels * HW, ex->yout, rows * HW * c.out_channels * 4, cudaMemcpyDeviceToDevice, st));
    }
    return leave_work(p, user);
}

extern "C" int vdt_unet_forward(vdt_plan* p, const float* x, const double* t, const void* y, float* out, int32_t batch,
                                void* stream) {
    return unet_forward_impl(p, x, t, y, out, batch, 0.f, 0ull, stream);
}

extern "C" int vdt_unet_forward_train(vdt_plan* p, const float* x, const double* t, const void* y, float* out, int32_t batch,
                                      float drop_rate, uint64_t seed, void* stream) {
    return unet_forward_impl(p, x, t, y, out, batch, drop_rate, (unsigned long long)seed, stream);
}

// ================================================================================================ schedule (host, fp64)
static double logsigmoid_d(double x) { return std::fmin(x, 0.0) - std::log1p(std::exp(-std::fabs(x))); }
static double log1mexp_d(double x) { return x < -9.0 ? std::log1p(-std::exp(x)) : std::log(-std::expm1(x)); }
static double lerp_d(double a, double b, double w) { return w < 0.5 ? a + w * (b - a) : b - (b - a) * (1.0 - w); }

static int logsnr_d(const vdt_sampler_config& sc, double t, double* out) {
    const double PI = 3.14159265358979323846;
    switch (sc.logsnr_schedule) {
        case VDT_SCHED_COSINE: {
            const double t_from = std::atan(std::exp(-0.5 * sc.logsnr_max)) / (0.5 * PI);
            const double t_to = std::atan(std::exp(-0.5 * sc.logsnr_min)) / (0.5 * PI);
            *out = -2.0 * std::log(std::tan(lerp_d(t_from, t_to, t) * PI * 0.5));
            return 0;
        }
        case VDT_SCHED_LINEAR: {
            const double t_from = 1.0 / (1.0 + std::exp(-sc.logsnr_max)), t_to = 1.0 / (1.0 + std::exp(-sc.logsnr_min));
            const double tt = lerp_d(t_from, t_to, t);
            *out = std::log(tt) - std::log1p(-tt);
            return 0;
        }
        case VDT_SCHED_SIGMOID: {
            *out = sc.logsnr_max - lerp_d(0.0, 1.0, t) * (sc.logsnr_max - sc.logsnr_min);
            return 0;
        }
        case VDT_SCHED_LEGACY: {
            const double x_from = 0.9999, x_max = 0.9999, x_min = 0.98, slope = -0.0199;
            const double x_to = lerp_d(x_max, x_min, t);
            const double la = 1000.0 / slope * (x_to * std::log(x_to) - x_to - x_from * std::log(x_from) + x_from);
            *out = la - log1mexp_d(la - 1e-9);
            return 0;
        }
    }
    return fail("unknown logsnr schedule %d", sc.logsnr_schedule);   // NotImplementedError, diffusion.py:96
}

// The prediction converters at one fp32 log-SNR l, fp32 math like the reference's TorchScript converters (diffusion.py:206-245):
// slots 0-5 alpha, sigma, rsqrt(sigmoid l), exp(-l/2), sigmoid l, sigmoid -l and 12-13 rsqrt(sigmoid -l) (pred_eps_from_x0,
// diffusion.py:222-223), exp(l/2) of a vdt_step_coefficients row.
static void converter_slots(float l, float* o) {
    const float sig_pos = 1.0f / (1.0f + std::exp(-l)), sig_neg = 1.0f / (1.0f + std::exp(l));
    o[0] = std::sqrt(sig_pos);
    o[1] = std::sqrt(sig_neg);
    o[2] = 1.0f / std::sqrt(sig_pos);
    o[3] = std::exp(-0.5f * l);
    o[4] = sig_pos;
    o[5] = sig_neg;
    o[12] = 1.0f / std::sqrt(sig_neg);
    o[13] = std::exp(0.5f * l);
}

// DPM-Solver++(2M) is defined here on the data prediction of the DDIM (eta = 0) step only.
static int check_solver(const vdt_sampler_config& sc) {
    if (sc.solver == VDT_SOLVER_FIRST_ORDER) return 0;
    if (sc.solver != VDT_SOLVER_DPMPP_2M) return fail("unknown solver %d", sc.solver);
    if (!sc.use_ddim) return fail("the DPM-Solver++(2M) solver needs use_ddim = 1 (it is not defined for ancestral sampling)");
    if (sc.x0eps_coef)
        return fail("the DPM-Solver++(2M) solver needs x0eps_coef = 0 (under DDIM the reference's (eps, x0) coefficients are "
                    "logarithms, so there is no data-prediction step to extend)");
    return 0;
}

extern "C" int vdt_step_coefficients(const vdt_sampler_config* scp, float* out) {
    if (!scp || !out) return fail("null argument");
    const vdt_sampler_config& sc = *scp;
    const int T = sc.sample_timesteps;
    if (T < 1) return fail("sample_timesteps must be >= 1");
    CKI(check_solver(sc));
    std::vector<double> h(T), c2d(T);                           // lambda_s - lambda_t and the fp64 c2 of every step
    for (int i = 0; i < T; ++i) {
        double ls_d, lt_d;
        // s = step / T, t = (step + 1) / T: fp64 tensors in p_sample (diffusion.py:399), fp32 in p_sample_progressive
        // (diffusion.py:421), where the schedule then sees the fp32-rounded quotients (`_t = t.to(float64)`, :101)
        const double s_in = sc.t_fp32 ? (double)((float)i / (float)T) : (double)i / (double)T;
        const double t_in = sc.t_fp32 ? (double)((float)(i + 1) / (float)T) : (double)(i + 1) / (double)T;
        CKI(logsnr_d(sc, s_in, &ls_d));
        CKI(logsnr_d(sc, t_in, &lt_d));
        const float ls32 = (float)ls_d, lt32 = (float)lt_d;     // broadcast_to casts to x.dtype (diffusion.py:23-26)
        const double ls = ls32, lt = lt32;                      // re-upcast inside the posterior (131, 171)
        const double logr = lt - ls;
        if (!(logr < 0.0)) return fail("log-SNR schedule is not strictly decreasing at step %d", i);   // assert, diffusion.py:119
        double c1, c2, logvar;
        if (sc.use_ddim) {
            if (sc.x0eps_coef) {                     // diffusion.py:180-182: returned un-exponentiated for eta = 0
                c1 = 0.5 * logsigmoid_d(-ls);
                c2 = 0.5 * logsigmoid_d(ls);
            } else {
                c1 = std::exp(0.5 * (logsigmoid_d(-ls) - logsigmoid_d(-lt)));
                c2 = std::exp(log1mexp_d(0.5 * logr) + 0.5 * logsigmoid_d(ls));
            }
            logvar = -INFINITY;
        } else {
            const double l1mr = log1mexp_d(logr);
            if (sc.x0eps_coef) {                     // diffusion.py:137-140
                c1 = std::exp(0.5 * (logsigmoid_d(ls) - lt) + logr);
                c2 = std::sqrt(1.0 / (1.0 + std::exp(-ls)));
            } else {
                c1 = std::exp(logr + 0.5 * (logsigmoid_d(ls) - logsigmoid_d(lt)));
                c2 = std::exp(l1mr + 0.5 * logsigmoid_d(ls));
            }
            const double lo = l1mr + logsigmoid_d(-ls), hi = l1mr + logsigmoid_d(-lt);
            if (sc.model_var_type == VDT_VAR_FIXED_LARGE) logvar = hi;
            else if (sc.model_var_type == VDT_VAR_FIXED_SMALL) logvar = lo;
            else if (sc.model_var_type == VDT_VAR_FIXED_MEDIUM) logvar = lo + sc.intp_frac * (hi - lo);
            else return fail("unknown model_var_type %d", sc.model_var_type);   // NotImplementedError, diffusion.py:161
        }
        float* o = out + (size_t)i * kCoefStride;
        converter_slots(lt32, o);
        o[6] = (float)c1;
        o[7] = (float)c2;
        const float lv32 = (float)logvar;
        o[8] = std::isinf(lv32) ? 0.0f : std::exp(0.5f * lv32);
        o[9] = lv32;
        o[10] = ls32;
        o[11] = lt32;
        o[14] = sc.x0eps_coef ? 1.0f : 0.0f;         // lets vdt_op_sampler_step pick the (eps, x0) form from the row alone
        o[15] = 0.0f;
        h[i] = 0.5 * (ls - lt);
        c2d[i] = c2;
    }
    // DPM-Solver++(2M): with lambda = l / 2 and h_i = lambda_s - lambda_t of step i, D = pred + k (pred - pred_prev) with
    // k = h_i / (2 h_{i+1}) (step i + 1 runs just before step i), written as the DDIM mean plus c2k (pred - pred_prev).
    // The first step (i = T-1) is DDIM; the last (i = 0) returns the guided x0 like DDIM.
    if (sc.solver == VDT_SOLVER_DPMPP_2M)
        for (int i = 1; i < T - 1; ++i) out[(size_t)i * kCoefStride + 15] = (float)(c2d[i] * (h[i] / (2.0 * h[i + 1])));
    return 0;
}

// DDIM inversion runs the deterministic first-order step with the p_sample time grid (fp64 t) and the data-prediction form.
static int check_invert(const vdt_sampler_config& sc) {
    if (sc.sample_timesteps < 1) return fail("sample_timesteps must be >= 1");
    if (!sc.use_ddim) return fail("DDIM inversion needs use_ddim = 1 (the ancestral step is not deterministic)");
    if (sc.x0eps_coef)
        return fail("DDIM inversion needs x0eps_coef = 0 (under DDIM the reference's (eps, x0) coefficients are logarithms)");
    if (sc.solver != VDT_SOLVER_FIRST_ORDER) return fail("DDIM inversion is first-order: solver must be 0 (got %d)", sc.solver);
    if (sc.t_fp32) return fail("DDIM inversion runs the fp64 time grid of p_sample: t_fp32 must be 0");
    return 0;
}

// Row j maps x at s = j/T to x at t = (j+1)/T: converters at lambda_s (the model sees x_s at time s), c1' = sigma_t / sigma_s,
// c2' = alpha_t - alpha_s c1' = -alpha_t expm1((l_s - l_t) / 2), in fp64 from the fp32-rounded log-SNRs and rounded once.
extern "C" int vdt_invert_coefficients(const vdt_sampler_config* scp, float* out) {
    if (!scp || !out) return fail("null argument");
    const vdt_sampler_config& sc = *scp;
    CKI(check_invert(sc));
    const int T = sc.sample_timesteps;
    for (int j = 0; j < T; ++j) {
        double ls_d, lt_d;
        CKI(logsnr_d(sc, (double)j / (double)T, &ls_d));
        CKI(logsnr_d(sc, (double)(j + 1) / (double)T, &lt_d));
        const float ls32 = (float)ls_d, lt32 = (float)lt_d;
        const double ls = ls32, lt = lt32;
        if (!(lt < ls)) return fail("log-SNR schedule is not strictly decreasing at step %d", j);
        float* o = out + (size_t)j * kCoefStride;
        for (int k = 0; k < kCoefStride; ++k) o[k] = 0.0f;
        converter_slots(ls32, o);
        o[6] = (float)std::exp(0.5 * (logsigmoid_d(-lt) - logsigmoid_d(-ls)));
        o[7] = (float)(-std::exp(0.5 * logsigmoid_d(lt)) * std::expm1(0.5 * (ls - lt)));
        o[10] = ls32;
        o[11] = lt32;
    }
    return 0;
}

// ================================================================================================ training step
// Per-sample scalars of GaussianDiffusion.train_loss from the continuous times t (host, fp64): the log-SNR is evaluated in
// fp64 and rounded to fp32 by broadcast_to (diffusion.py:23-26, 293-295); every derived scalar is then fp32 math on that
// fp32 log-SNR, like the reference's TorchScript converters (diffusion.py:206-245).  Row layout = vdt_step_coefficients'
// slots that make sense here: 0 alpha, 1 sigma, 2 rsqrt(sigmoid l), 3 exp(-l/2), 4 sigmoid l, 5 sigmoid -l, 11 l,
// 12 rsqrt(sigmoid -l), 13 exp(l/2).
extern "C" int vdt_train_coefficients(const vdt_sampler_config* scp, const double* t_host, int32_t batch, float* out) {
    if (!scp || !t_host || !out) return fail("null argument");
    for (int i = 0; i < batch; ++i) {
        double l_d;
        CKI(logsnr_d(*scp, t_host[i], &l_d));
        const float l = (float)l_d;
        float* o = out + (size_t)i * kCoefStride;
        for (int k = 0; k < kCoefStride; ++k) o[k] = 0.f;
        converter_slots(l, o);
        o[11] = l;
    }
    return 0;
}

extern "C" int vdt_q_sample(const float* x0, const float* noise, const float* coef_dev, float* x_t, int32_t batch, int32_t chw,
                            void* stream) {
    if (!x0 || !noise || !coef_dev || !x_t) return fail("null argument");
    if (chw % 4) return fail("C*H*W must be a multiple of 4 (got %d)", chw);
    cudaError_t e = launch_q_sample(x0, noise, coef_dev, x_t, batch, chw, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("q_sample launch failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_train_loss(const float* model_out, const float* x0, const float* noise, const float* x_t, const float* coef_dev,
                              float* loss, float* grad_out, int32_t batch, int32_t c, int32_t hw, int32_t model_out_type,
                              int32_t reweight_type, void* stream) {
    if (!model_out || !x0 || !noise || !x_t || !coef_dev || !loss) return fail("null argument");
    if (model_out_type < 0 || model_out_type > 3) return fail("unknown model_out_type %d", model_out_type);
    if (reweight_type < 0 || reweight_type > 3) return fail("unknown reweight_type %d", reweight_type);
    if (reweight_type != 2 && model_out_type == VDT_OUT_BOTH)
        return fail("a single-target reweighting compares the target with the raw model output (diffusion.py:541): "
                    "shapes differ for model_out_type \"both\"");
    cudaError_t e = launch_train_loss(model_out, x0, noise, x_t, coef_dev, loss, grad_out, batch, c, hw, model_out_type, reweight_type,
                                      reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("train_loss launch failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_grad_sq_accumulate(const float* grad, int64_t n, void* scratch, int64_t scratch_bytes, double* sq_accum, void* stream) {
    if (!grad || !sq_accum || !scratch) return fail("null argument");
    if (n < 0 || (size_t)scratch_bytes < grad_sq_scratch_bytes(n)) return fail("scratch too small: %lld bytes needed", (long long)grad_sq_scratch_bytes(n));
    cudaError_t e = launch_grad_sq(grad, n, scratch, sq_accum, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("grad_sq launch failed: %s", cudaGetErrorString(e));
    return 0;
}
extern "C" int64_t vdt_grad_sq_scratch_bytes(int64_t n) { return (int64_t)grad_sq_scratch_bytes(n); }

extern "C" int vdt_adamw_ema_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, float* ema_shadow, int64_t n,
                                  double lr, double beta1, double beta2, double eps, double weight_decay, int32_t step,
                                  const double* grad_sq_total, double max_norm, double ema_decay, void* stream) {
    if (!param || !grad || !exp_avg || !exp_avg_sq) return fail("null argument");
    if (step < 1) return fail("step counts from 1 (torch.optim state['step'] after its increment)");
    cudaError_t e = launch_adamw_ema(param, grad, exp_avg, exp_avg_sq, ema_shadow, n, lr, beta1, beta2, eps, weight_decay, step,
                                     grad_sq_total, (float)max_norm, ema_decay, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("adamw_ema launch failed: %s", cudaGetErrorString(e));
    return 0;
}

// ================================================================================================ sampler
// invert: the DDIM inversion exec (ascending begin-step, invert_step_kernel, vdt_invert_coefficients), cached under its own key
static int get_sampler_exec(vdt_plan* p, const vdt_sampler_config& sc, int imgs, bool has_label, int lane, bool invert, Exec** out) {
    const bool cfg = sc.w_guide > 0.0 && has_label;            // diffusion.py:368
    const int rep = cfg ? 2 : 1;
    // the key holds what shapes the workspace, the coefficient table and the kernel parameters baked into the graph;
    // per-call values (seed, injected-noise tensor, fp32-t mode of p_sample_progressive) live in the device-side
    // SamplerState and are rewritten before every call
    char key[208];
    snprintf(key, sizeof(key), "%s%d:%d:%d:%d:%d:%d:%d:%d:%d:%d:%d:%.17g:%.17g:%.17g:%.17g", invert ? "inv" : "smp", lane, imgs, (int)has_label,
             sc.sample_timesteps, sc.model_out_type, sc.model_var_type, sc.logsnr_schedule, sc.use_ddim, sc.x0eps_coef, sc.t_fp32,
             sc.solver, sc.intp_frac, sc.logsnr_min, sc.logsnr_max, sc.w_guide);
    CKI(exec_cache_lookup(p, key, out));
    if (*out) return 0;
    CKI(exec_cache_make_room(p));
    const vdt_unet_config& c = p->cfg;
    const int Cm = sc.model_out_type == VDT_OUT_BOTH ? 2 * c.in_channels : c.in_channels;
    if (Cm != c.out_channels)
        return fail("model_out_type needs %d output channels but the UNet has %d", Cm, c.out_channels);
    std::unique_ptr<Exec> ex(new Exec());
    ex->last_use = ++p->use_clock;
    const size_t HW = (size_t)c.resolution * c.resolution;
    const int T = sc.sample_timesteps;
    ex->rows = imgs * rep; ex->rep = rep; ex->sampler = true; ex->has_y = has_label; ex->sc = sc;
    const bool cond_model = c.num_classes > 0 && has_label;
    const bool mt = cond_model && c.multitags;           // multi-hot labels: every UNet row has its own embedding row
    ex->emb_rows = mt ? ex->rows : cond_model ? c.num_classes + 1 : 1;
    if (mt) CKI(ex->acquire((size_t)ex->rows * c.num_classes * 4, (void**)&ex->y_multi));
    CKI(ex->acquire(imgs * HW * c.in_channels * 4, (void**)&ex->xin));
    CKI(ex->acquire((size_t)ex->rows * HW * c.out_channels * 4, (void**)&ex->yout));
    CKI(ex->acquire(ex->emb_rows * sizeof(double), (void**)&ex->t_rows));
    CKI(ex->acquire(ex->emb_rows * sizeof(int64_t), (void**)&ex->y_rows));
    CKI(ex->acquire(ex->rows * sizeof(int), (void**)&ex->film_row));
    CKI(ex->acquire(sizeof(SamplerState), (void**)&ex->state));
    CKI(ex->acquire(imgs * HW * c.in_channels * 4, (void**)&ex->pred));
    CKI(ex->acquire((size_t)T * kCoefStride * 4, (void**)&ex->coef_table));
    // on the plan's own stream: the legacy default stream does not order against a non-blocking stream
    iota_i64_kernel<<<(ex->emb_rows + 127) / 128, 128, 0, p->work>>>(ex->y_rows, ex->emb_rows);
    CK(cudaGetLastError());
    std::vector<float> coefs((size_t)T * kCoefStride);
    CKI(invert ? vdt_invert_coefficients(&sc, coefs.data()) : vdt_step_coefficients(&sc, coefs.data()));
    CK(cudaMemcpyAsync(ex->coef_table, coefs.data(), coefs.size() * 4, cudaMemcpyHostToDevice, p->work));
    CK(cudaStreamSynchronize(p->work));              // `coefs` is a host temporary
    float* film;
    CKI(ex->acquire((size_t)ex->emb_rows * p->film_total * 4, (void**)&film));
    ex->begins.push_back({ex->state, ex->coef_table, ex->t_rows, ex->emb_rows, T});
    ex->steps.push_back({invert ? S_BEGIN_INV : S_BEGIN, 0});
    CKI(add_embedding_steps(p, ex.get(), film, cond_model));
    CKI(build_unet_steps(p, ex.get(), film, mt ? nullptr : ex->film_row));
    SamplerStepParams sp{};
    sp.model_out = ex->yout; sp.x_t = ex->xin; sp.x_s = ex->xin; sp.pred_x0 = ex->pred;
    sp.st = ex->state; sp.B = imgs; sp.C = c.in_channels; sp.HW = (int)HW; sp.cfg = cfg ? 1 : 0;
    sp.model_out_type = sc.model_out_type; sp.w = (float)sc.w_guide; sp.x0eps = sc.x0eps_coef ? 1 : 0;
    ex->samples.push_back(sp);
    ex->steps.push_back({invert ? S_INVERT : S_SAMPLE, 0});
    *out = ex.get();
    p->execs[key] = std::move(ex);
    return 0;
}

// known and mask come together; known_noise only with both
static int check_inpaint(const float* known, const float* mask, const float* known_noise) {
    if ((known == nullptr) != (mask == nullptr))
        return fail("inpainting needs both known and mask (got %s without %s)", known ? "known" : "mask", known ? "mask" : "known");
    if (known_noise && !mask) return fail("inpainting known_noise needs known and mask");
    return 0;
}

// The chunk and lane loop shared by sampling and inversion; its callers check every argument first.  Sampling runs steps
// first_step, first_step - 1, ... (num_steps of them) with `start_step` as the first step of the trajectory (see SamplerState);
// inversion (invert) runs first_step, first_step + 1, ...
static int run_sampler_range(vdt_plan* p, const vdt_sampler_config& sc, const vdt_inpaint& inp, float* x, const void* label,
                             const float* step_noise, int32_t batch, int32_t first_step, int32_t num_steps, float* pred_x0,
                             bool carry_pred, int start_step, bool invert, void* stream) {
    cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
    CKI(enter_work(p, user));
    cudaStream_t st = p->work;
    const vdt_unet_config& c = p->cfg;
    const size_t CHW = (size_t)c.in_channels * c.resolution * c.resolution;
    const bool cfg = sc.w_guide > 0.0 && label != nullptr;
    const bool mt = c.multitags && c.num_classes > 0 && label != nullptr;
    const int64_t* row_label = (c.num_classes > 0 && !mt) ? static_cast<const int64_t*>(label) : nullptr;   // an unconditional UNet ignores y (unet.py:289)
    const int rep = cfg ? 2 : 1;
    const int chunk = std::max(1, c.max_rows / rep);
    const int nchunks = (batch + chunk - 1) / chunk;
    // several lanes when there is more than one chunk (per-launch profiling needs a single ordered stream)
    const int lanes = g_profile.load() ? 1 : std::max(1, std::min(vdt_plan::kLanes, nchunks));
    if (lanes > 1) {
        if (!p->ev_fork) CK(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
        CK(cudaEventRecord(p->ev_fork, p->work));
        for (int l = 1; l < lanes; ++l) {
            if (!p->lane_stream[l]) {
                CK(cudaStreamCreateWithFlags(&p->lane_stream[l], cudaStreamNonBlocking));
                CK(cudaEventCreateWithFlags(&p->ev_join[l], cudaEventDisableTiming));
            }
            CK(cudaStreamWaitEvent(p->lane_stream[l], p->ev_fork, 0));
        }
    }
    for (int i0 = 0, ci = 0; i0 < batch; i0 += chunk, ++ci) {
        const int imgs = std::min(chunk, batch - i0);
        const int lane = ci % lanes;
        st = lane ? p->lane_stream[lane] : p->work;
        Exec* ex;
        CKI(get_sampler_exec(p, sc, imgs, label != nullptr, lane, invert, &ex));
        CK(cudaMemcpyAsync(ex->xin, x + (size_t)i0 * CHW, imgs * CHW * 4, cudaMemcpyDeviceToDevice, st));
        if (carry_pred) CK(cudaMemcpyAsync(ex->pred, pred_x0 + (size_t)i0 * CHW, imgs * CHW * 4, cudaMemcpyDeviceToDevice, st));
        if (mt) {
            const int n = ex->rows * c.num_classes;
            multitag_rows_kernel<<<(n + 127) / 128, 128, 0, st>>>(static_cast<const float*>(label) + (size_t)i0 * c.num_classes,
                                                                ex->y_multi, ex->rows, rep, c.num_classes);
        } else {
            film_rows_kernel<<<(ex->rows + 127) / 128, 128, 0, st>>>(row_label ? row_label + i0 : nullptr, ex->film_row, ex->rows, rep,
                                                                     c.num_classes);
        }
        CK(cudaGetLastError());
        sampler_init_state_kernel<<<1, 32, 0, st>>>(ex->state, first_step, start_step, i0, sc.t_fp32 ? 1 : 0, step_noise,
                                                    (long long)batch * (long long)CHW, (unsigned long long)sc.seed, inp);
        CK(cudaGetLastError());
        g_launches += 2;
        for (int step = 0; step < num_steps; ++step) CKI(run_exec(p, ex, st));
        CK(cudaMemcpyAsync(x + (size_t)i0 * CHW, ex->xin, imgs * CHW * 4, cudaMemcpyDeviceToDevice, st));
        if (pred_x0 && num_steps > 0)
            CK(cudaMemcpyAsync(pred_x0 + (size_t)i0 * CHW, ex->pred, imgs * CHW * 4, cudaMemcpyDeviceToDevice, st));
    }
    for (int l = 1; l < lanes; ++l) {
        CK(cudaEventRecord(p->ev_join[l], p->lane_stream[l]));
        CK(cudaStreamWaitEvent(p->work, p->ev_join[l], 0));
    }
    return leave_work(p, user);
}

// checks shared by every fused sampling / inversion entry point, ahead of any CUDA call
static int check_plan_for_sampler(const vdt_plan* p, const vdt_sampler_config& sc) {
    if (!p->finalized) return fail("plan not finalized (load every state_dict key, then vdt_plan_finalize)");
    if (sc.model_out_type < 0 || sc.model_out_type > 3) return fail("unknown model_out_type %d", sc.model_out_type);
    return 0;
}

extern "C" int vdt_p_sample_range_inpaint(vdt_plan* p, const vdt_sampler_config* scp, const vdt_inpaint* inpaint, float* x,
                                          const void* label, const float* step_noise, int32_t batch, int32_t first_step,
                                          int32_t num_steps, float* pred_x0, void* stream) {
    if (!p || !scp || !x) return fail("null argument");
    const vdt_inpaint inp = inpaint ? *inpaint : vdt_inpaint{nullptr, nullptr, nullptr};
    CKI(check_inpaint(inp.known, inp.mask, inp.known_noise));
    const vdt_sampler_config& sc = *scp;
    const int T = sc.sample_timesteps;
    CKI(check_solver(sc));
    // DPM-Solver++(2M) steps after the first read the previous step's guided x0: a range that starts inside the trajectory
    // takes it from pred_x0 (written by the call that ran step first_step + 1), since the exec's pred buffer is shared by
    // every chunk of its lane
    const bool carry_pred = sc.solver == VDT_SOLVER_DPMPP_2M && first_step < T - 1 && num_steps > 0;
    if (carry_pred && !pred_x0)
        return fail("DPM-Solver++(2M) from step %d < T-1 needs pred_x0 holding the guided x0 of step %d", first_step, first_step + 1);
    CKI(check_plan_for_sampler(p, sc));
    if (first_step < 0 || first_step >= T || num_steps < 0 || first_step - num_steps < -1)
        return fail("step range [%d, %d) steps leaves the trajectory of %d steps", first_step, num_steps, T);
    return run_sampler_range(p, sc, inp, x, label, step_noise, batch, first_step, num_steps, pred_x0, carry_pred, T - 1, false,
                             stream);
}

extern "C" int vdt_p_sample_from(vdt_plan* p, const vdt_sampler_config* scp, const vdt_inpaint* inpaint, float* x,
                                 const void* label, const float* step_noise, int32_t batch, int32_t first_step, void* stream) {
    if (!p || !scp || !x) return fail("null argument");
    const vdt_inpaint inp = inpaint ? *inpaint : vdt_inpaint{nullptr, nullptr, nullptr};
    CKI(check_inpaint(inp.known, inp.mask, inp.known_noise));
    const vdt_sampler_config& sc = *scp;
    CKI(check_solver(sc));
    if (first_step < 0 || first_step >= sc.sample_timesteps)
        return fail("first_step %d lies outside [0, %d)", first_step, sc.sample_timesteps);
    CKI(check_plan_for_sampler(p, sc));
    return run_sampler_range(p, sc, inp, x, label, step_noise, batch, first_step, first_step + 1, nullptr, false, first_step,
                             false, stream);
}

extern "C" int vdt_ddim_invert_range(vdt_plan* p, const vdt_sampler_config* scp, float* x, const void* label, int32_t batch,
                                     int32_t first_step, int32_t num_steps, void* stream) {
    if (!p || !scp || !x) return fail("null argument");
    const vdt_sampler_config& sc = *scp;
    CKI(check_invert(sc));
    const int T = sc.sample_timesteps;
    if (first_step < 0 || first_step >= T || num_steps < 0 || num_steps > T - first_step)
        return fail("inversion steps [%d, %d + %d) leave [0, %d)", first_step, first_step, num_steps, T);
    CKI(check_plan_for_sampler(p, sc));
    const vdt_inpaint none{nullptr, nullptr, nullptr};
    return run_sampler_range(p, sc, none, x, label, nullptr, batch, first_step, num_steps, nullptr, false, T - 1, true, stream);
}

extern "C" int vdt_p_sample_range(vdt_plan* p, const vdt_sampler_config* scp, float* x, const void* label,
                                  const float* step_noise, int32_t batch, int32_t first_step, int32_t num_steps,
                                  float* pred_x0, void* stream) {
    return vdt_p_sample_range_inpaint(p, scp, nullptr, x, label, step_noise, batch, first_step, num_steps, pred_x0, stream);
}

extern "C" int vdt_p_sample_inpaint(vdt_plan* p, const vdt_sampler_config* scp, const vdt_inpaint* inpaint, const float* noise,
                                    const void* label, const float* step_noise, float* out, int32_t batch, void* stream) {
    if (!p || !scp || !noise || !out) return fail("null argument");
    if (inpaint) CKI(check_inpaint(inpaint->known, inpaint->mask, inpaint->known_noise));
    const size_t CHW = (size_t)p->cfg.in_channels * p->cfg.resolution * p->cfg.resolution;
    cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
    if (out != noise) CK(cudaMemcpyAsync(out, noise, (size_t)batch * CHW * 4, cudaMemcpyDeviceToDevice, user));
    return vdt_p_sample_range_inpaint(p, scp, inpaint, out, label, step_noise, batch, scp->sample_timesteps - 1,
                                      scp->sample_timesteps, nullptr, stream);
}

extern "C" int vdt_p_sample(vdt_plan* p, const vdt_sampler_config* scp, const float* noise, const void* label,
                            const float* step_noise, float* out, int32_t batch, void* stream) {
    return vdt_p_sample_inpaint(p, scp, nullptr, noise, label, step_noise, out, batch, stream);
}

extern "C" int vdt_p_sample_host(vdt_plan* p, const vdt_sampler_config* scp, const float* noise, const void* label,
                                 const float* step_noise, float* out, int32_t batch) {
    if (!p || !scp || !noise || !out) return fail("null argument");
    const vdt_unet_config& c = p->cfg;
    const size_t CHW = (size_t)c.in_channels * c.resolution * c.resolution;
    const size_t n = (size_t)batch * CHW;
    float *d_noise = nullptr, *d_out = nullptr, *d_sn = nullptr;
    void* d_label = nullptr;
    const size_t label_bytes = (c.multitags && c.num_classes > 0) ? (size_t)batch * c.num_classes * 4 : (size_t)batch * sizeof(int64_t);
    int rc = 0;
    cudaStream_t st = nullptr;
    auto cleanup = [&]() { cudaFree(d_noise); cudaFree(d_out); cudaFree(d_sn); cudaFree(d_label); };
#define CKH(expr)                                                                               \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) { cleanup(); return fail("%s failed: %s", #expr, cudaGetErrorString(_e)); } \
    } while (0)
    CKH(cudaMalloc(&d_noise, n * 4));
    CKH(cudaMalloc(&d_out, n * 4));
    CKH(cudaMemcpyAsync(d_noise, noise, n * 4, cudaMemcpyHostToDevice, st));
    if (label) {
        CKH(cudaMalloc(&d_label, label_bytes));
        CKH(cudaMemcpyAsync(d_label, label, label_bytes, cudaMemcpyHostToDevice, st));
    }
    if (step_noise) {
        CKH(cudaMalloc(&d_sn, n * 4 * scp->sample_timesteps));
        CKH(cudaMemcpyAsync(d_sn, step_noise, n * 4 * scp->sample_timesteps, cudaMemcpyHostToDevice, st));
    }
    rc = vdt_p_sample(p, scp, d_noise, d_label, d_sn, d_out, batch, st);
    if (rc == 0) {
        CKH(cudaMemcpyAsync(out, d_out, n * 4, cudaMemcpyDeviceToHost, st));
        CKH(cudaStreamSynchronize(st));
    }
    cleanup();
#undef CKH
    return rc;
}

// ================================================================================================ kernel-level hooks
extern "C" int vdt_op_conv(const void* x, int32_t batch, int32_t h, int32_t w, int32_t cin, const float* w_oihw, int32_t cout,
                           int32_t ksize, const float* bias, const float* residual, float* out, int32_t f16, void* out16,
                           void* stats_out, int32_t stat_cols, void* stream) {
    if (ksize != 1 && ksize != 3) return fail("ksize must be 1 or 3");
    if (cin % 64) return fail("cin must be a multiple of 64");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int taps = ksize * ksize;
    h16* wp = nullptr;
    const int wrows = std::max(cout, 16);
    CK(cudaMalloc(&wp, (size_t)wrows * taps * cin * 2));
    CK(cudaMemset(wp, 0, (size_t)wrows * taps * cin * 2));
    int rc = pack_conv(w_oihw, wp, cout, cin, taps, taps * cin, 0, f16);
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (rc == 0) {
        ConvSpec s;
        s.f16 = f16;
        if (ksize == 3) { s.a3 = (const h16*)x; s.c3 = cin; } else { s.a1 = (const h16*)x; s.c1 = cin; s.ld1 = cin; }
        s.n = batch; s.h = h; s.w = w; s.wpacked = wp; s.cout = cout; s.wrows = wrows; s.bias = bias; s.residual = residual;
        s.out_mode = kOutF32; s.out_f32 = out; s.ld = cout; s.stats = (float2*)stats_out; s.stat_cols = stat_cols == 2 ? 2 : 4;
        if (out16) { s.out_mode = kOutBF16; s.out_bf16 = (h16*)out16; s.out_f32 = nullptr; }
        std::unique_ptr<ConvParams> cp(new ConvParams());
        rc = setup_conv(s, cp.get());
        if (rc == 0 && stats_out && !cp->stats) rc = fail("no conv-epilogue statistics layout for %dx%d feature maps", h, w);
        if (rc == 0) {
            cudaError_t e = launch_conv_gemm(*cp, nsm, st);
            ++g_launches;
            if (e != cudaSuccess) rc = fail("conv launch failed: %s", cudaGetErrorString(e));
        }
    }
    cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(wp);
    if (rc == 0 && e != cudaSuccess) return fail("conv kernel failed: %s", cudaGetErrorString(e));
    return rc;
}

static int device_sm_count() {
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    return nsm;
}

// One conv in any mode build_unet_steps gives it, with the plan's packers and setup_conv.  Every argument is checked
// before the first CUDA call, so that none of setup_conv's internal refusals can be reached from here.
extern "C" int vdt_op_conv_ex(const vdt_conv_op* op, void* stream) {
    if (!op) return fail("null argument");
    const vdt_conv_op& o = *op;
    if (!o.a3 || !o.w3 || !o.bias) return fail("a3, w3 and bias are required");
    if ((o.out_f32 != nullptr) == (o.out16 != nullptr)) return fail("give exactly one of out_f32 and out16");
    if ((o.a1 != nullptr) != (o.w1 != nullptr)) return fail("a1 and w1 come together");
    if (!o.a1 && o.a1_lo) return fail("a1_lo without a1");
    if (o.a1 && (o.a3_lo != nullptr) != (o.a1_lo != nullptr))
        return fail("split-precision mode packs every weight in three parts: give both a3_lo and a1_lo or neither");
    if (o.f16 != 0 && o.f16 != 1) return fail("f16 must be 0 or 1 (got %d)", o.f16);
    if (o.batch < 1 || o.h < 1 || o.w < 1) return fail("empty input (%d x %d x %d)", o.batch, o.h, o.w);
    if (o.c3 < 64 || o.c3 % 64 || o.cout < 64 || o.cout % 64 || (o.a1 && (o.c1 < 64 || o.c1 % 64)))
        return fail("channel counts must be positive multiples of 64 (c3 %d, c1 %d, cout %d)", o.c3, o.a1 ? o.c1 : 0, o.cout);
    if (o.ups != 0 && o.ups != 1) return fail("ups must be 0 or 1 (got %d)", o.ups);
    if (o.ups && o.a1) return fail("the sub-pixel upsampling conv takes no 1x1 skip operand");
    if (o.ups && o.residual) return fail("the sub-pixel upsampling conv takes no residual");
    if (o.resid_mode < 0 || o.resid_mode > 2) return fail("resid_mode must be 0, 1 or 2 (got %d)", o.resid_mode);
    if (o.resid_mode != 0 && !o.residual) return fail("resid_mode %d needs a residual", o.resid_mode);
    if (o.resid_mode == 1 && ((o.h | o.w) & 1)) return fail("an upsampled residual needs even output sides (got %dx%d)", o.h, o.w);
    if (o.resid_mode == 2 && (o.batch & 1)) return fail("a residual shared by image pairs needs an even batch (got %d)", o.batch);
    ConvGeom geom;
    CKI(conv_geom(o.batch, o.h, o.w, &geom));
    const int H = o.ups ? 2 * o.h : o.h, W = o.ups ? 2 * o.w : o.w;
    if (o.stats) {
        if (o.stat_cols != 2 && o.stat_cols != 4) return fail("stat_cols must be 2 or 4 (got %d)", o.stat_cols);
        const int slabs = stat_slabs_per_image(o.h, o.w);
        if (slabs <= 0 || (o.ups && 4 * slabs != stat_slabs_per_image(H, W)))
            return fail("no conv-epilogue statistics layout for %dx%d feature maps%s", H, W, o.ups ? " from a sub-pixel conv" : "");
    }
    const int split = o.a3_lo ? 1 : 0, km = split ? 3 : 1;
    const int ktot = o.ups ? 16 * o.c3 * km : (9 * o.c3 + (o.a1 ? o.c1 : 0)) * km;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    h16* wp = nullptr;
    CK(cudaMalloc(&wp, (size_t)o.cout * ktot * 2));
    int rc = 0;
    cudaError_t e = cudaMemset(wp, 0, (size_t)o.cout * ktot * 2);
    if (e != cudaSuccess) rc = fail("weight buffer: %s", cudaGetErrorString(e));
    if (rc == 0) rc = o.ups ? pack_conv_ups(o.w3, wp, o.cout, o.c3, o.f16, split)
                            : pack_conv_skip(o.w3, o.w1, wp, o.cout, o.c3, o.c1, o.f16, split);
    if (rc == 0 && (e = cudaStreamSynchronize(nullptr)) != cudaSuccess) rc = fail("weight packing failed: %s", cudaGetErrorString(e));
    if (rc == 0) {
        ConvSpec s;
        s.f16 = o.f16; s.stat_cols = o.stat_cols == 2 ? 2 : 4; s.sat_count = reinterpret_cast<unsigned long long*>(o.sat_count);
        s.a3 = (const h16*)o.a3; s.a3_lo = (const h16*)o.a3_lo; s.c3 = o.c3;
        if (o.a1) { s.a1 = (const h16*)o.a1; s.a1_lo = (const h16*)o.a1_lo; s.c1 = o.c1; s.ld1 = o.c1; }
        s.n = o.batch; s.h = o.h; s.w = o.w; s.wpacked = wp; s.cout = o.cout; s.wrows = o.cout; s.ups = o.ups;
        s.bias = o.bias; s.residual = o.residual; s.resid_up = o.resid_mode == 1; s.resid_rep = o.resid_mode == 2 ? 2 : 0;
        if (o.out16) { s.out_mode = kOutBF16; s.out_bf16 = (h16*)o.out16; } else { s.out_mode = kOutF32; s.out_f32 = o.out_f32; }
        s.ld = o.cout; s.stats = (float2*)o.stats;
        std::unique_ptr<ConvParams> cp(new ConvParams());
        rc = setup_conv(s, cp.get());
        if (rc == 0 && o.stats && !cp->stats) rc = fail("internal: statistics dropped for %dx%d feature maps", H, W);
        if (rc == 0) {
            e = launch_conv_gemm(*cp, device_sm_count(), st);
            ++g_launches;
            if (e != cudaSuccess) rc = fail("conv launch failed: %s", cudaGetErrorString(e));
        }
    }
    e = cudaStreamSynchronize(st);
    cudaFree(wp);
    if (rc == 0 && e != cudaSuccess) return fail("conv kernel failed: %s", cudaGetErrorString(e));
    return rc;
}

// in_conv as the plan runs it: im2col of the fp32 NCHW input into 64 patch columns (image i reads input image i / rep),
// then the pointwise GEMM against pack_inconv's weights, with optional GroupNorm statistics.
extern "C" int vdt_op_in_conv(const float* x_nchw, int32_t batch, int32_t rep, int32_t c, int32_t h, int32_t w, const float* w_oihw,
                              const float* bias, int32_t hid, float* out_nhwc, void* stats_out, int32_t stat_cols, int32_t f16,
                              void* stream) {
    if (!x_nchw || !w_oihw || !bias || !out_nhwc) return fail("null argument");
    if (batch < 1 || h < 1 || w < 1) return fail("empty input (%d x %d x %d)", batch, h, w);
    if (rep != 1 && rep != 2) return fail("rep must be 1 or 2 (got %d)", rep);
    if (c < 1 || 9 * c > 64) return fail("in_conv takes 1 to 7 input channels (got %d)", c);
    if (hid < 64 || hid % 64) return fail("channel counts must be positive multiples of 64 (hid %d)", hid);
    if (f16 != 0 && f16 != 1) return fail("f16 must be 0 or 1 (got %d)", f16);
    if (stats_out) {
        if (stat_cols != 2 && stat_cols != 4) return fail("stat_cols must be 2 or 4 (got %d)", stat_cols);
        if (stat_slabs_per_image(h, w) <= 0) return fail("no conv-epilogue statistics layout for %dx%d feature maps", h, w);
    }
    const int n = batch * rep;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    h16 *wp = nullptr, *patches = nullptr;
    CK(cudaMalloc(&wp, (size_t)hid * 64 * 2));
    int rc = 0;
    cudaError_t e = cudaMalloc(&patches, (size_t)n * h * w * 64 * 2);
    if (e != cudaSuccess) rc = fail("patch buffer: %s", cudaGetErrorString(e));
    if (rc == 0) rc = pack_inconv(w_oihw, wp, hid, c, f16, 0);
    if (rc == 0 && (e = cudaStreamSynchronize(nullptr)) != cudaSuccess) rc = fail("weight packing failed: %s", cudaGetErrorString(e));
    if (rc == 0) {
        e = launch_im2col3x3(x_nchw, patches, nullptr, batch, rep, c, h, w, f16, st);
        ++g_launches;
        if (e != cudaSuccess) rc = fail("im2col launch failed: %s", cudaGetErrorString(e));
    }
    if (rc == 0) {
        ConvSpec s;
        s.f16 = f16; s.stat_cols = stat_cols == 2 ? 2 : 4;
        s.a1 = patches; s.c1 = 64; s.ld1 = 64; s.n = n; s.h = h; s.w = w; s.wpacked = wp; s.cout = hid; s.wrows = hid;
        s.bias = bias; s.out_mode = kOutF32; s.out_f32 = out_nhwc; s.ld = hid; s.stats = (float2*)stats_out;
        std::unique_ptr<ConvParams> cp(new ConvParams());
        rc = setup_conv(s, cp.get());
        if (rc == 0 && stats_out && !cp->stats) rc = fail("internal: statistics dropped for %dx%d feature maps", h, w);
        if (rc == 0) {
            e = launch_conv_gemm(*cp, device_sm_count(), st);
            ++g_launches;
            if (e != cudaSuccess) rc = fail("conv launch failed: %s", cudaGetErrorString(e));
        }
    }
    e = cudaStreamSynchronize(st);
    cudaFree(patches);
    cudaFree(wp);
    if (rc == 0 && e != cudaSuccess) return fail("in_conv kernels failed: %s", cudaGetErrorString(e));
    return rc;
}

// out_conv as the plan runs it: the pointwise GEMM Y[pixel, tap * cout + co] over pack_outconv's tap-major rows (zero bias,
// padded to outconv_rows), then the tap-sum gather + bias into fp32 NCHW.
extern "C" int vdt_op_out_conv(const void* a_16_nhwc, int32_t batch, int32_t h, int32_t w, int32_t c0, const float* w_oihw,
                               int32_t cout, const float* bias, float* out_nchw, int32_t f16, void* stream) {
    if (!a_16_nhwc || !w_oihw || !bias || !out_nchw) return fail("null argument");
    if (batch < 1 || h < 1 || w < 1) return fail("empty input (%d x %d x %d)", batch, h, w);
    if (c0 < 64 || c0 % 64) return fail("channel counts must be positive multiples of 64 (c0 %d)", c0);
    if (cout < 1 || cout > 16) return fail("out_conv takes 1 to 16 output channels (got %d)", cout);
    if (f16 != 0 && f16 != 1) return fail("f16 must be 0 or 1 (got %d)", f16);
    const int rows = outconv_rows(cout);
    const size_t pixels = (size_t)batch * h * w;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    h16* wp = nullptr; float* zero = nullptr; float* ytap = nullptr;
    CK(cudaMalloc(&wp, (size_t)rows * c0 * 2));
    int rc = 0;
    cudaError_t e = cudaMalloc(&zero, (size_t)rows * 4);
    if (e == cudaSuccess) e = cudaMalloc(&ytap, pixels * rows * 4);
    if (e == cudaSuccess) e = cudaMemset(wp, 0, (size_t)rows * c0 * 2);
    if (e == cudaSuccess) e = cudaMemset(zero, 0, (size_t)rows * 4);
    if (e != cudaSuccess) rc = fail("out_conv buffers: %s", cudaGetErrorString(e));
    if (rc == 0) rc = pack_outconv(w_oihw, wp, cout, c0, f16, 0);
    if (rc == 0 && (e = cudaStreamSynchronize(nullptr)) != cudaSuccess) rc = fail("weight packing failed: %s", cudaGetErrorString(e));
    if (rc == 0) {
        ConvSpec s;
        s.f16 = f16;
        s.a1 = (const h16*)a_16_nhwc; s.c1 = c0; s.ld1 = c0; s.n = batch; s.h = h; s.w = w; s.wpacked = wp;
        s.cout = rows; s.wrows = rows; s.bias = zero; s.out_mode = kOutF32; s.out_f32 = ytap; s.ld = rows;
        std::unique_ptr<ConvParams> cp(new ConvParams());
        rc = setup_conv(s, cp.get());
        if (rc == 0) {
            e = launch_conv_gemm(*cp, device_sm_count(), st);
            ++g_launches;
            if (e != cudaSuccess) rc = fail("conv launch failed: %s", cudaGetErrorString(e));
        }
    }
    if (rc == 0) {
        e = launch_tapsum3x3(ytap, bias, out_nchw, batch, h, w, cout, rows, st);
        ++g_launches;
        if (e != cudaSuccess) rc = fail("tapsum launch failed: %s", cudaGetErrorString(e));
    }
    e = cudaStreamSynchronize(st);
    cudaFree(ytap);
    cudaFree(zero);
    cudaFree(wp);
    if (rc == 0 && e != cudaSuccess) return fail("out_conv kernels failed: %s", cudaGetErrorString(e));
    return rc;
}

static int op_groupnorm_impl(const void* src1, int32_t c1, const float* src2, int32_t c2, int32_t batch, int32_t h,
                             int32_t w, const float* gamma, const float* beta, const float* film, int32_t film_stride,
                             int32_t film_off, int32_t silu, int32_t resample, void* out_act, void* out_raw, float* out_res,
                             int32_t f16, const void* stats1, const void* stats2, int32_t stat_cols, int32_t in16, float drop_p,
                             const unsigned long long* drop_seed_dev, int32_t drop_layer, void* stream) {
    GroupNormParams g{};
    g.drop_p = drop_p; g.drop_seed = drop_seed_dev; g.drop_layer = drop_layer;
    g.f16 = f16; g.stats1 = (const float2*)stats1; g.stats2 = (const float2*)stats2; g.in16 = in16; g.stat_cols = stat_cols == 2 ? 2 : 4;
    g.stat_slabs = stat_slabs_per_image(h, w);
    if (stats1 && g.stat_slabs <= 0) return fail("no conv-epilogue statistics layout for %dx%d feature maps", h, w);
    g.src1 = src1; g.C1 = c1; g.src2 = src2; g.C2 = c2; g.B = batch; g.H = h; g.W = w; g.gamma = gamma; g.beta = beta;
    g.film = film; g.film_row = nullptr; g.film_stride = film_stride; g.film_off = film_off; g.silu = silu; g.resample = resample;
    g.out_act = (h16*)out_act; g.out_raw = (h16*)out_raw; g.out_res = out_res;
    float2* scratch = nullptr;
    if (stats1) { CK(cudaMalloc(&scratch, (size_t)batch * 32 * sizeof(float2))); g.meanrstd = scratch; }
    cudaError_t e = launch_groupnorm(g, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (scratch) { cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream)); cudaFree(scratch); }
    if (e != cudaSuccess) return fail("groupnorm launch failed: %s", cudaGetErrorString(e));
    return 0;
}

// ---- backward of a conv layer, first slice of the training step (SURVEY §8 f2) ---------------------------------------
extern "C" int vdt_op_conv_dgrad(const void* dy, int32_t batch, int32_t h, int32_t w, int32_t cin, const float* w_oihw, int32_t cout,
                                 int32_t ksize, float* dx, int32_t f16, void* stream) {
    if (ksize != 1 && ksize != 3) return fail("ksize must be 1 or 3");
    if (cout % 64 || cin % 32) return fail("dgrad needs cout %% 64 == 0 and cin %% 32 == 0 (got %d -> %d)", cin, cout);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int taps = ksize * ksize;
    h16* wp = nullptr;
    CK(cudaMalloc(&wp, (size_t)cin * taps * cout * 2));
    const long long n = (long long)cout * cin * taps;
    pack_conv_dgrad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w_oihw, wp, cout, cin, taps, f16);
    int rc = 0;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = fail("dgrad weight pack failed: %s", cudaGetErrorString(e));
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    if (rc == 0) {
        ConvSpec s;                                    // the conv kernel with the roles of the channel counts swapped
        s.f16 = f16;
        if (ksize == 3) { s.a3 = (const h16*)dy; s.c3 = cout; } else { s.a1 = (const h16*)dy; s.c1 = cout; s.ld1 = cout; }
        s.n = batch; s.h = h; s.w = w; s.wpacked = wp; s.cout = cin; s.wrows = cin;
        float* zero = nullptr;
        CK(cudaMalloc(&zero, (size_t)cin * 4));
        CK(cudaMemsetAsync(zero, 0, (size_t)cin * 4, st));
        s.bias = zero; s.out_mode = kOutF32; s.out_f32 = dx; s.ld = cin;
        std::unique_ptr<ConvParams> cp(new ConvParams());
        rc = setup_conv(s, cp.get());
        if (rc == 0) {
            e = launch_conv_gemm(*cp, nsm, st);
            ++g_launches;
            if (e != cudaSuccess) rc = fail("dgrad launch failed: %s", cudaGetErrorString(e));
        }
        e = cudaStreamSynchronize(st);
        cudaFree(zero);
        if (rc == 0 && e != cudaSuccess) rc = fail("dgrad kernel failed: %s", cudaGetErrorString(e));
    }
    cudaFree(wp);
    return rc;
}

extern "C" int vdt_op_conv_wgrad(const void* x, const void* dy, int32_t batch, int32_t h, int32_t w, int32_t cin, int32_t cout,
                                 int32_t ksize, float* dw_oihw, float* dbias, int32_t f16, void* stream) {
    if (ksize != 1 && ksize != 3) return fail("ksize must be 1 or 3");
    if (cout % 64 || cin % 64) return fail("wgrad needs cout %% 64 == 0 and cin %% 64 == 0 (got %d -> %d)", cin, cout);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    ConvGeom g;
    CKI(conv_geom(batch, h, w, &g));
    std::unique_ptr<WgradParams> wp(new WgradParams());
    memset(wp.get(), 0, sizeof(WgradParams));
    CKI(make_map_nhwc(&wp->dy_map, dy, batch, h, w, cout, g.box_h, g.box_n));
    CKI(make_map_nhwc(&wp->x_map, x, batch, h, w, cin, g.box_h, g.box_n));
    wp->taps = ksize * ksize; wp->Cout = cout; wp->Cin = cin; wp->co_blocks = (cout + 127) / 128;
    wp->ci_block = cin <= 256 ? cin : (cin % 256 == 0 ? 256 : (cin % 192 == 0 ? 192 : (cin % 128 == 0 ? 128 : 64)));
    wp->ci_blocks = cin / wp->ci_block;
    wp->tap_groups = (wp->taps + 1) / 2;
    wp->num_tiles = g.num_m_tiles; wp->tiles_per_image = g.tiles_per_image; wp->box_h = g.box_h; wp->box_n = g.box_n;
    wp->rows_per_tile = g.rows_per_tile; wp->f16 = f16;
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    wp->splits = wgrad_splits(*wp, nsm);
    float* partial = nullptr;
    CK(cudaMalloc(&partial, (size_t)wp->splits * wp->taps * cout * cin * 4));
    wp->partial = partial;
    cudaError_t e = launch_wgrad(*wp, dw_oihw, dbias, (const h16*)dy, (long long)batch * h * w, st);
    g_launches += 2 + (dbias ? 1 : 0);
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaFree(partial);
    if (e != cudaSuccess) return fail("wgrad launch failed: %s", cudaGetErrorString(e));
    if (e2 != cudaSuccess) return fail("wgrad kernel failed: %s", cudaGetErrorString(e2));
    return 0;
}

extern "C" int vdt_op_groupnorm(const void* src1, int32_t c1, const float* src2, int32_t c2, int32_t batch, int32_t h,
                                int32_t w, const float* gamma, const float* beta, const float* film, int32_t film_stride,
                                int32_t film_off, int32_t silu, int32_t resample, void* out_act, void* out_raw, float* out_res,
                                int32_t f16, const void* stats1, const void* stats2, int32_t stat_cols, int32_t in16, void* stream) {
    return op_groupnorm_impl(src1, c1, src2, c2, batch, h, w, gamma, beta, film, film_stride, film_off, silu, resample, out_act,
                             out_raw, out_res, f16, stats1, stats2, stat_cols, in16, 0.f, nullptr, 0, stream);
}

extern "C" int vdt_op_groupnorm_dropout(const void* src1, int32_t c1, int32_t batch, int32_t h, int32_t w, const float* gamma,
                                        const float* beta, int32_t silu, void* out_act, int32_t f16, float drop_p, uint64_t seed,
                                        int32_t layer, void* stream) {
    if (!(drop_p > 0.f && drop_p < 1.f)) return fail("drop_p must lie in (0, 1)");
    unsigned long long* ds = nullptr;
    CK(cudaMalloc(&ds, sizeof(unsigned long long)));
    const unsigned long long sv = seed;
    CK(cudaMemcpy(ds, &sv, sizeof(sv), cudaMemcpyHostToDevice));
    const int rc = op_groupnorm_impl(src1, c1, nullptr, 0, batch, h, w, gamma, beta, nullptr, 0, 0, silu, 0, out_act, nullptr, nullptr,
                                     f16, nullptr, nullptr, 4, 0, drop_p, ds, layer, stream);
    cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream));
    cudaFree(ds);
    return rc;
}

extern "C" int vdt_op_groupnorm_backward(const float* x, const float* grad_out, int32_t c, int32_t batch, int32_t h, int32_t w,
                                         const float* gamma, const float* beta, const float* film, int32_t silu, float drop_p,
                                         uint64_t seed, int32_t layer, float* grad_x, float* grad_gamma, float* grad_beta,
                                         float* grad_film, void* stream) {
    if (!x || !grad_out || !gamma || !beta || !grad_x || !grad_gamma || !grad_beta) return fail("null argument");
    if (batch < 1 || h < 1 || w < 1) return fail("empty input");
    if (c < 64 || c % 64 != 0 || c > 2048)
        return fail("groupnorm backward takes a multiple of 64 channels up to 2048 (got %d)", c);
    if (!(drop_p >= 0.f && drop_p < 1.f)) return fail("drop_p must lie in [0, 1)");
    GroupNormBwdParams q{};
    q.x = x; q.grad_out = grad_out; q.gamma = gamma; q.beta = beta; q.film = film;
    q.B = batch; q.HW = h * w; q.C = c; q.silu = silu;
    q.drop_p = drop_p; q.drop_seed = seed; q.drop_layer = layer;
    q.grad_x = grad_x; q.grad_gamma = grad_gamma; q.grad_beta = grad_beta; q.grad_film = grad_film;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    CK(cudaMalloc(&q.scratch, groupnorm_backward_scratch_bytes(batch, h * w, c)));
    cudaError_t e = launch_groupnorm_backward(q, st);
    g_launches += 5;
    cudaStreamSynchronize(st);
    cudaFree(q.scratch);
    if (e != cudaSuccess) return fail("groupnorm backward: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_op_attention_backward(const float* qkv, const float* grad_out, float* grad_qkv, int32_t batch, int32_t n, int32_t heads,
                                         int32_t d, void* stream) {
    if (!qkv || !grad_out || !grad_qkv) return fail("null argument");
    if (batch < 1 || n < 1 || heads < 1) return fail("empty input");
    if (d != 64 && d != 128 && d != 192 && d != 256) return fail("attention backward takes head dims 64, 128, 192 or 256 (got %d)", d);
    void* stat = nullptr;
    CK(cudaMalloc(&stat, (size_t)batch * n * heads * sizeof(float2)));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = launch_attention_backward_f32(qkv, grad_out, grad_qkv, stat, batch, n, heads, d, st);
    g_launches += 2;
    cudaStreamSynchronize(st);
    cudaFree(stat);
    if (e != cudaSuccess) return fail("attention backward: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_op_attention(const void* qkv, void* out, int32_t batch, int32_t n, int32_t heads, int32_t d,
                                int32_t f16, void* stream) {
    const int hid = heads * d;
    std::unique_ptr<AttnParams> ap(new AttnParams());
    memset(ap.get(), 0, sizeof(AttnParams));
    CKI(make_map_2d(&ap->q_map, qkv, (long long)batch * n, 3 * hid, 3 * hid, 128));
    CKI(make_map_2d(&ap->kv_map, qkv, (long long)batch * n, 3 * hid, 3 * hid, 64));
    ap->B = batch; ap->N = n; ap->heads = heads; ap->d = d; ap->hid = hid; ap->f16 = f16;
    ap->scale_log2e = (float)(1.4426950408889634 / std::sqrt((double)d));
    ap->out = (h16*)out;
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e = launch_attention(*ap, nsm, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("attention launch failed: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" int vdt_images_to_uint8(const float* x, uint8_t* out, int32_t batch, int32_t c, int32_t hw, void* stream) {
    if (!x || !out) return fail("null argument");
    if (batch < 0 || c < 1 || hw < 1) return fail("bad image shape (%d, %d, %d)", batch, c, hw);
    cudaError_t e = launch_images_to_uint8(x, out, batch, c, hw, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("images_to_uint8 launch failed: %s", cudaGetErrorString(e));
    return 0;
}

static int op_sampler_step_impl(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                                int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step,
                                const float* coef_host, float w, float* pred_hist, const float* known, const float* mask,
                                const float* known_noise, uint64_t seed, const float* coef_prev_host, void* stream) {
    if (!coef_host) return fail("null argument");
    if (coef_host[15] != 0.0f && !pred_hist)
        return fail("coefficient row %d is a DPM-Solver++(2M) row (c2k != 0): use vdt_op_sampler_step_hist with the previous "
                    "step's guided x0", step);
    CKI(check_inpaint(known, mask, known_noise));
    if (mask && step > 0 && !coef_prev_host)
        return fail("inpainting at step %d > 0 needs coefficient row %d (alpha_s, sigma_s of this step's s)", step, step - 1);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    SamplerState hs{};
    hs.next_step = step - 1; hs.step = step; hs.img0 = 0; hs.noise = noise; hs.noise_step_stride = 0; hs.seed = seed;
    for (int i = 0; i < kCoefStride; ++i) hs.coef[i] = coef_host[i];
    hs.known = known; hs.mask = mask; hs.known_noise = known_noise;
    if (mask && step > 0) { hs.known_a = coef_prev_host[0]; hs.known_s = coef_prev_host[1]; }
    SamplerState* ds = nullptr;
    CK(cudaMalloc(&ds, sizeof(SamplerState)));
    CK(cudaMemcpy(ds, &hs, sizeof(hs), cudaMemcpyHostToDevice));
    SamplerStepParams sp{};
    sp.model_out = model_out; sp.x_t = x_t; sp.x_s = x_s;
    sp.st = ds; sp.pred_x0 = pred_hist; sp.B = batch; sp.C = c; sp.HW = hw; sp.cfg = cfg;
    sp.model_out_type = model_out_type; sp.w = w; sp.x0eps = coef_host[14] != 0.0f ? 1 : 0;
    cudaError_t e = launch_sampler_step(sp, st);
    ++g_launches;
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaFree(ds);
    if (e != cudaSuccess) return fail("sampler_step launch failed: %s", cudaGetErrorString(e));
    if (e2 != cudaSuccess) return fail("sampler_step failed: %s", cudaGetErrorString(e2));
    return 0;
}

extern "C" int vdt_op_sampler_step(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                                   int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step,
                                   const float* coef_host, float w, void* stream) {
    return op_sampler_step_impl(model_out, x_t, noise, x_s, batch, c, hw, cfg, model_out_type, step, coef_host, w, nullptr,
                                nullptr, nullptr, nullptr, 0, nullptr, stream);
}

extern "C" int vdt_op_sampler_step_hist(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                                        int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step,
                                        const float* coef_host, float w, float* pred_hist, void* stream) {
    if (!pred_hist) return fail("null pred_hist");
    return op_sampler_step_impl(model_out, x_t, noise, x_s, batch, c, hw, cfg, model_out_type, step, coef_host, w, pred_hist,
                                nullptr, nullptr, nullptr, 0, nullptr, stream);
}

extern "C" int vdt_op_sampler_step_known(const float* model_out, const float* x_t, const float* noise, float* x_s, int32_t batch,
                                         int32_t c, int32_t hw, int32_t cfg, int32_t model_out_type, int32_t step,
                                         const float* coef_host, float w, float* pred_hist, const float* known, const float* mask,
                                         const float* known_noise, uint64_t seed, const float* coef_prev_host, void* stream) {
    return op_sampler_step_impl(model_out, x_t, noise, x_s, batch, c, hw, cfg, model_out_type, step, coef_host, w, pred_hist,
                                known, mask, known_noise, seed, coef_prev_host, stream);
}

extern "C" int vdt_op_invert_step(const float* model_out, const float* x, float* x_next, int32_t batch, int32_t c, int32_t hw,
                                  int32_t cfg, int32_t model_out_type, const float* coef_host, float w, void* stream) {
    if (!model_out || !x || !x_next || !coef_host) return fail("null argument");
    if (model_out_type < 0 || model_out_type > 3) return fail("unknown model_out_type %d", model_out_type);
    if (batch < 0 || c < 1 || hw < 1) return fail("bad image shape (%d, %d, %d)", batch, c, hw);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    SamplerState hs{};
    for (int i = 0; i < kCoefStride; ++i) hs.coef[i] = coef_host[i];
    SamplerState* ds = nullptr;
    CK(cudaMalloc(&ds, sizeof(SamplerState)));
    CK(cudaMemcpy(ds, &hs, sizeof(hs), cudaMemcpyHostToDevice));
    SamplerStepParams sp{};
    sp.model_out = model_out; sp.x_t = x; sp.x_s = x_next; sp.st = ds; sp.B = batch; sp.C = c; sp.HW = hw; sp.cfg = cfg ? 1 : 0;
    sp.model_out_type = model_out_type; sp.w = w;
    cudaError_t e = launch_invert_step(sp, st);
    ++g_launches;
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaFree(ds);
    if (e != cudaSuccess) return fail("invert_step launch failed: %s", cudaGetErrorString(e));
    if (e2 != cudaSuccess) return fail("invert_step failed: %s", cudaGetErrorString(e2));
    return 0;
}

// ---- entry points the composed training step (v-diffusion-torch_b200/training.py) adds to the kernel-level hooks ----------
// norm2 -> FiLM -> act2 -> dropout of a ResidualBlock in .train() mode (unet.py:143-146) on a plain fp32 NHWC tensor: the
// same kernel as vdt_op_groupnorm with the FiLM table and the dropout stream both given (drop_p = 0: no dropout).
extern "C" int vdt_op_groupnorm_train(const void* src1, int32_t c1, int32_t batch, int32_t h, int32_t w, const float* gamma,
                                      const float* beta, const float* film, int32_t film_stride, int32_t film_off, int32_t silu,
                                      void* out_act, int32_t f16, float drop_p, uint64_t seed, int32_t layer, void* stream) {
    if (!(drop_p >= 0.f && drop_p < 1.f)) return fail("drop_p must lie in [0, 1)");
    if (drop_p == 0.f)
        return op_groupnorm_impl(src1, c1, nullptr, 0, batch, h, w, gamma, beta, film, film_stride, film_off, silu, 0, out_act, nullptr,
                                 nullptr, f16, nullptr, nullptr, 4, 0, 0.f, nullptr, 0, stream);
    unsigned long long* ds = nullptr;
    CK(cudaMalloc(&ds, sizeof(unsigned long long)));
    const unsigned long long sv = seed;
    cudaError_t e = cudaMemcpy(ds, &sv, sizeof(sv), cudaMemcpyHostToDevice);
    int rc = e == cudaSuccess ? 0 : fail("seed upload failed: %s", cudaGetErrorString(e));
    if (rc == 0)
        rc = op_groupnorm_impl(src1, c1, nullptr, 0, batch, h, w, gamma, beta, film, film_stride, film_off, silu, 0, out_act, nullptr,
                               nullptr, f16, nullptr, nullptr, 4, 0, drop_p, ds, layer, stream);
    cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream));
    cudaFree(ds);
    return rc;
}

// F.linear(x, W, b) [+ SiLU] in fp32 (modules.py:77-78), the kernel the embedding MLP and the FiLM projections run on:
// x [rows, K], W [N, K], b [N] (required) -> out [rows, N].  K <= 1536 (one 8-row slab of x is staged in shared memory).
extern "C" int vdt_op_linear(const float* x, const float* W, const float* b, float* out, int32_t rows, int32_t K, int32_t N,
                             int32_t silu_out, void* stream) {
    if (!x || !W || !b || !out) return fail("null argument");
    if (rows < 0 || K < 1 || N < 1) return fail("bad linear shape (%d, %d, %d)", rows, K, N);
    if ((size_t)K * 8 * sizeof(float) > 48 * 1024) return fail("linear: K = %d exceeds the 1536 columns one slab holds", K);
    cudaError_t e = launch_linear_f32(x, W, b, out, rows, K, N, silu_out, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("linear launch failed: %s", cudaGetErrorString(e));
    return 0;
}

// get_timestep_embedding(t, dim) (functions.py:20-25) for fp64 t: sin | cos halves of 1000 t exp(-k log(1e4) / (dim/2 - 1)).
extern "C" int vdt_op_timestep_embedding(const double* t, float* out, int32_t rows, int32_t dim, void* stream) {
    if (!t || !out) return fail("null argument");
    if (rows < 0 || dim < 4) return fail("bad embedding shape (%d, %d)", rows, dim);
    cudaError_t e = launch_timestep_embedding(t, out, rows, dim, nullptr, reinterpret_cast<cudaStream_t>(stream));
    ++g_launches;
    if (e != cudaSuccess) return fail("timestep embedding launch failed: %s", cudaGetErrorString(e));
    return 0;
}
