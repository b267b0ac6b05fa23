// Host side of the C ABI (include/polmux_ssfm.h): context, tables, plans, the
// SSFM launch loop, layout conversion, amplifier and error counting kernels.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <vector>

#include "../../include/polmux_ssfm.h"
#include "pmx_kernels.cuh"
#include "pmx_launch.h"
#include <cudaTypedefs.h>

// ---------------------------------------------------------------------------
extern const PmxLaunchTable pmx_table_64, pmx_table_128, pmx_table_256, pmx_table_512, pmx_table_1024,
    pmx_table_2048, pmx_table_4096;
extern const PmxLaunchTable pmx_table_f32_64, pmx_table_f32_128, pmx_table_f32_256, pmx_table_f32_512, pmx_table_f32_1024,
    pmx_table_f32_2048, pmx_table_f32_4096;

const PmxLaunchTable* pmx_get_table(int L, int precision) {
    const bool f32 = precision == PMX_F32;
    switch (L) {
        case 64: return f32 ? &pmx_table_f32_64 : &pmx_table_64;
        case 128: return f32 ? &pmx_table_f32_128 : &pmx_table_128;
        case 256: return f32 ? &pmx_table_f32_256 : &pmx_table_256;
        case 512: return f32 ? &pmx_table_f32_512 : &pmx_table_512;
        case 1024: return f32 ? &pmx_table_f32_1024 : &pmx_table_1024;
        case 2048: return f32 ? &pmx_table_f32_2048 : &pmx_table_2048;
        case 4096: return f32 ? &pmx_table_f32_4096 : &pmx_table_4096;
        default: return nullptr;
    }
}

static inline cpx pmx_root(long long m, long long M) {  // exp(-2*pi*i*m/M) in long double
    const long double PI2 = 6.283185307179586476925286766559005768L;
    // reduce to the first octant for accuracy
    m %= M;
    long double a = PI2 * (long double)m / (long double)M;
    return make_double2((double)cosl(a), (double)(-sinl(a)));
}

void pmx_fill_stage_twiddles(int L, cpx* out, int layout) {
    if (layout == 1) {  // L = 1024 as 8 * 16 * 8 (CtaFFT<R, 1024>): [15][8] of W_128^(k*r), then [128] of W_1024^k
        size_t o = 0;
        for (int r = 1; r <= 15; ++r)
            for (int k = 0; k < 8; ++k) out[o++] = pmx_root((long long)k * r, 128);
        for (int k = 0; k < 128; ++k) out[o++] = pmx_root((long long)k, 1024);
        return;
    }
    int ns = 1;
    size_t o = 0;
    while (ns < L) {
        int R = pmx_stage_radix(L, ns);
        if (ns > 1) {  // radix-8 stage: W^k, W^2k, W^4k of W = exp(-2*pi*i/(8*ns))
            for (int r = 1; r <= 4; r *= 2)
                for (int k = 0; k < ns; ++k) out[o++] = pmx_root((long long)k * r, (long long)ns * R);
        }
        ns *= R;
    }
}

// ---------------------------------------------------------------------------
static thread_local std::string g_tls_error;
struct pmx_ctx;
static int set_err(pmx_ctx* ctx, int code, const char* fmt, ...);

struct StageTw {
    cpx* dev = nullptr;
};
struct FourStepTw {  // per-row two-level four-step twiddle table (PmxTw4<L> layout), see pmx_k_fill_tw4
    void* rows = nullptr;
};

struct pmx_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t gstream[3] = {nullptr, nullptr, nullptr};  // streams of the other realization groups (pmx_fiber_exec)
    cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr};
    std::string error;
    std::map<int, StageTw> stage_tw;          // by L
    std::map<long long, FourStepTw> four_tw;  // by N
    struct Occ { int a = 0, b = 0, c = 0, cnl = 0; };
    std::map<int, Occ> setup_done;  // by L: resident CTAs per SM of passes A, B, C and C' (digital backpropagation)
    int sm_count = 148;
    PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
    StepCtl* h_ctl = nullptr;  // pinned readback buffer
    int h_ctl_cap = 0;
    int64_t launches = 0;
    // optional per-pass timing (CUDA events around every pass launch)
    bool profile = false;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<int> ev_kind;  // kind of interval i (events 2i, 2i+1)
    size_t ev_used = 0;
    double prof_ms[4] = {0, 0, 0, 0};
    int64_t prof_n[4] = {0, 0, 0, 0};
};

struct ProfScope {  // records start/stop events around one launch when profiling is on
    pmx_ctx* c;
    bool on;
    ProfScope(pmx_ctx* ctx, int kind) : c(ctx), on(ctx->profile) {
        if (!on) return;
        if (c->ev_used + 2 > c->ev_pool.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            c->ev_pool.push_back(a);
            c->ev_pool.push_back(b);
        }
        c->ev_kind.resize(c->ev_pool.size() / 2);
        c->ev_kind[c->ev_used / 2] = kind;
        cudaEventRecord(c->ev_pool[c->ev_used], c->stream);
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(c->ev_pool[c->ev_used + 1], c->stream);
        c->ev_used += 2;
    }
};

static void prof_collect(pmx_ctx* c) {
    if (!c->ev_used) return;
    cudaStreamSynchronize(c->stream);
    for (size_t i = 0; i < c->ev_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, c->ev_pool[i], c->ev_pool[i + 1]) == cudaSuccess) {
            c->prof_ms[c->ev_kind[i / 2]] += ms;
            c->prof_n[c->ev_kind[i / 2]] += 1;
        }
    }
    c->ev_used = 0;
}

struct pmx_devfield {
    pmx_ctx* ctx;
    int64_t nfft;
    int32_t nfc, batch, precision;
    cpx* data;  // [batch*nfc][nfft][2]; float2 elements behind this pointer when precision == PMX_F32
    size_t cbytes() const { return precision == PMX_F32 ? sizeof(float2) : sizeof(double2); }
    int N1 = 0, N2 = 0;
    int log2N1 = 0, log2N2 = 0;  // time sample n = n1*N2 + n2 is stored at n2*N1 + n1 (0/0: natural order, no SSFM)
    bool has_maps = false;
    CUtensorMap map_cols;  // pass B: box {gB*4 reals, <=256 rows, 1} of the [N2][N1] matrix
    CUtensorMap map_rows;  // passes A, C: 128-byte lines, box {one line, <=256 lines, 1}
};

static int ilog2_exact(int64_t v) {
    int l = 0;
    while ((1ll << l) < v) ++l;
    return ((1ll << l) == v) ? l : -1;
}

// Four-step split N = N1*N2: log2(N1), the balanced split (measured against the unbalanced ones in DESIGN.md §7).
static int split_log2N1(int lg) { return lg / 2; }

// Tensor maps over a resident field for the four-step split N = N1*N2 (see pmx_tma.cuh).
static int build_maps(pmx_ctx* c, pmx_devfield* f) {
    const int lg = ilog2_exact(f->nfft);
    if (lg < 12 || lg > 24) return PMX_OK;  // not a size the SSFM kernels take; other ops still work
    f->N1 = 1 << split_log2N1(lg);
    f->N2 = 1 << (lg - split_log2N1(lg));
    const PmxLaunchTable* tA = pmx_get_table(f->N1, f->precision);
    const PmxLaunchTable* tB = pmx_get_table(f->N2, f->precision);
    if (!tA || !tB) return PMX_OK;
    const cuuint64_t BC = (cuuint64_t)f->batch * f->nfc, N = (cuuint64_t)f->nfft;
    const bool f32 = f->precision == PMX_F32;
    const CUtensorMapDataType dt = f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64;
    const cuuint64_t SAB = f32 ? 16 : 32;  // bytes per Sa (4 reals)
    const cuuint32_t ones[3] = {1, 1, 1};
    // The field is stored transposed in time (sample n1*N2 + n2 at n2*N1 + n1, see pmx_kernels.cuh): an [N2][N1]
    // matrix of Sa per realization-column.
    {   // pass B: gB adjacent columns (k1), all N2 rows
        const int G = tB->gB;
        cuuint64_t dims[3] = {(cuuint64_t)f->N1 * 4, (cuuint64_t)f->N2, BC};
        cuuint64_t strides[2] = {(cuuint64_t)f->N1 * SAB, N * SAB};
        cuuint32_t box[3] = {(cuuint32_t)G * 4, (cuuint32_t)std::min(f->N2, 256), 1};
        const int pitch = G * (int)SAB;  // bytes of one box row = swizzle span (16: none)
        CUtensorMapSwizzle sw = pitch <= 16 ? CU_TENSOR_MAP_SWIZZLE_NONE
                                            : (pitch == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                           : (pitch == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B));
        CUresult r = c->encode(&f->map_cols, dt, 3, f->data, dims, strides, box, ones,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return set_err(c, PMX_ERR_CUDA, "cuTensorMapEncodeTiled(cols) failed: CUresult %d", (int)r);
    }
    {   // passes A and C: gAC adjacent rows (n2) of N1 Sa = contiguous 128-byte lines
        const int sa_per_line = (int)(128 / SAB);  // a 128-byte line holds 4 (FP64) or 8 (FP32) Sa
        const int lines = tA->gAC * f->N1 / sa_per_line;
        cuuint64_t dims[3] = {(cuuint64_t)(f32 ? 32 : 16), N / sa_per_line, BC};
        cuuint64_t strides[2] = {128, N * SAB};
        cuuint32_t box[3] = {(cuuint32_t)(f32 ? 32 : 16), (cuuint32_t)std::min(lines, 256), 1};
        CUresult r = c->encode(&f->map_rows, dt, 3, f->data, dims, strides, box, ones,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return set_err(c, PMX_ERR_CUDA, "cuTensorMapEncodeTiled(rows) failed: CUresult %d", (int)r);
    }
    f->log2N1 = split_log2N1(lg);
    f->log2N2 = lg - f->log2N1;
    f->has_maps = true;
    return PMX_OK;
}

// One step of a PMD-aware DBP plan (pmx_dbp_create), in execution order: what the step control would have left in
// StepCtl, mirrored onto the span's reversed plate table, and the span whose plates the step reads.
struct DbpGeo {
    double dz, leff, scale, dzb_first, dzb_last;
    int ntrunk, n_first, span, bmode;
};

struct pmx_plan {
    pmx_ctx* ctx;
    pmx_fiber_desc d;  // scalar copy (pointers not kept)
    FiberConst fc;
    int N1, N2, log2N1, log2N2;
    const PmxLaunchTable* tA;  // passes A/C (L = N1)
    const PmxLaunchTable* tB;  // pass B   (L = N2)
    double* betat_p = nullptr;
    double* db1_p = nullptr;
    double2* hfilt = nullptr;      // linear-filter plans: H per bin, permuted like betat_p
    long long hfilt_stride = 0;
    PlateConst* plates = nullptr;
    StepCtl* ctl = nullptr;
    StepPkg* pkg = nullptr;  // [batch] step packages written by pmx_k_ctl
    double* trace_dz = nullptr;
    int* trace_ntrunk = nullptr;
    int trace_cap = 0;
    bool single_step;
    bool onchip = false;   // nfft <= 4096: the single-launch kernel of small fields (pmx_onchip.cuh)
    // digital-backpropagation plans (pmx_dbp_create): the constants of passes A (no NL step) and B / C' (gam = -xi*gam), the
    // distinct step packages [npkg][batch] and the package of every step in execution order
    bool dbp = false;
    FiberConst fc_a, fc_c;
    StepPkg* sched = nullptr;
    std::vector<int> sched_idx;
    // PMD-aware DBP: the geometry of every step in execution order (device), each step's span, and whether
    // pmx_dbp_set_plates has filled plates ([nspan][plate_sets][nplates], reversed and negated) and packages
    bool dbp_pmd = false, dbp_plates_set = false;
    int dbp_nspan = 0;
    DbpGeo* geo_d = nullptr;
    std::vector<int> sched_span;
    // DBP of a small field (onchip): sched_idx and sched_span on the device, the on-chip kernel's step table
    int* sched_idx_d = nullptr;
    int* sched_span_d = nullptr;
    // single-channel DBP (pmx_dbp_channel_create): the DBP plan at nfft/decim samples, the band filter at nfft, the
    // work field of the decimated channel, and the channel's shift (mod nfft) and log2(decim)
    pmx_plan* ch_dbp = nullptr;
    pmx_plan* ch_band = nullptr;
    pmx_devfield* ch_work = nullptr;
    long long ch_shift = 0;
    int ch_log2r = 0;
    // filtered DBP (pmx_dbp_set_filter, bw > 0): on-chip, H/N over the transform length; on the three passes, the filter plan
    // of the Gaussian response and its work field (the intensity of two realization-columns per Sa)
    double filt_bw = 0.0;
    double* filt_hn_d = nullptr;
    pmx_plan* filt = nullptr;
    pmx_devfield* filt_work = nullptr;
    // enhanced split-step DBP (pmx_dbp_set_taps, ntaps > 0): the taps, and on the three passes the work field the intensity
    // goes to before its FIR (two realization-columns per Sa)
    int ntaps = 0;
    DbpTaps taps{};
    pmx_devfield* tap_work = nullptr;
};

static int set_err(pmx_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_tls_error = buf;
    if (ctx) ctx->error = buf;
    return code;
}

#define CK(ctx, call)                                                                           \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return set_err(ctx, PMX_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                           __FILE__, __LINE__);                                                 \
    } while (0)

extern "C" int pmx_version(void) { return PMX_VERSION; }

extern "C" int pmx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

extern "C" const char* pmx_last_error(const pmx_ctx* ctx) {
    if (ctx) return ctx->error.c_str();
    return g_tls_error.c_str();
}

extern "C" int pmx_ctx_create(pmx_ctx** out, int device_id) {
    if (!out) return set_err(nullptr, PMX_ERR_INVALID, "pmx_ctx_create: null output pointer");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_err(nullptr, PMX_ERR_CUDA, "no usable CUDA device (%s); this library has no CPU fallback",
                       e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device_id < 0 || device_id >= n)
        return set_err(nullptr, PMX_ERR_INVALID, "device_id %d out of range [0,%d)", device_id, n);
    pmx_ctx* c = new (std::nothrow) pmx_ctx();
    if (!c) return set_err(nullptr, PMX_ERR_INVALID, "out of host memory");
    c->device = device_id;
    CK(nullptr, cudaSetDevice(device_id));
    cudaDeviceProp prop;
    CK(nullptr, cudaGetDeviceProperties(&prop, device_id));
    if (prop.major < 10) {
        delete c;
        return set_err(nullptr, PMX_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                       device_id, prop.major, prop.minor);
    }
    c->sm_count = prop.multiProcessorCount;
    {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t ee = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (ee != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
            delete c;
            return set_err(nullptr, PMX_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
        }
        c->encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    }
    CK(nullptr, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    {  // keep freed blocks cached in the stream-ordered pool: fiber() after fiber() reuses them
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device_id) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    *out = c;
    return PMX_OK;
}

extern "C" void pmx_ctx_destroy(pmx_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (auto& kv : c->stage_tw) cudaFree(kv.second.dev);
    for (auto& kv : c->four_tw) {
        cudaFree(kv.second.rows);
    }
    if (c->h_ctl) cudaFreeHost(c->h_ctl);
    for (int g = 0; g < 3; ++g) {
        if (c->gstream[g]) cudaStreamDestroy(c->gstream[g]);
        if (c->ev_join[g]) cudaEventDestroy(c->ev_join[g]);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int pmx_ctx_sync(pmx_ctx* c) {
    if (!c) return set_err(nullptr, PMX_ERR_INVALID, "null ctx");
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" int pmx_ctx_profile(pmx_ctx* c, int enable) {
    if (!c) return set_err(nullptr, PMX_ERR_INVALID, "null ctx");
    prof_collect(c);
    c->profile = enable != 0;
    if (enable)
        for (int k = 0; k < 4; ++k) {
            c->prof_ms[k] = 0;
            c->prof_n[k] = 0;
        }
    return PMX_OK;
}

extern "C" int pmx_ctx_profile_read(pmx_ctx* c, double* ms, int64_t* n) {
    if (!c || !ms || !n) return set_err(c, PMX_ERR_INVALID, "null argument");
    prof_collect(c);
    for (int k = 0; k < 4; ++k) {
        ms[k] = c->prof_ms[k];
        n[k] = c->prof_n[k];
    }
    return PMX_OK;
}

// debug: per-phase cycle counters of the pass kernels (PMX_TIMING builds); 24 x int64 device buffer
static long long* g_dbg = nullptr;
extern "C" int pmx_debug_timing(pmx_ctx* c, long long* out24, int reset) {
    if (!c) return PMX_ERR_INVALID;
    cudaSetDevice(c->device);
    if (!g_dbg) {
        cudaMalloc(&g_dbg, 24 * sizeof(long long));
        cudaMemset(g_dbg, 0, 24 * sizeof(long long));
    }
    cudaStreamSynchronize(c->stream);
    if (out24) cudaMemcpy(out24, g_dbg, 24 * sizeof(long long), cudaMemcpyDeviceToHost);
    if (reset) cudaMemset(g_dbg, 0, 24 * sizeof(long long));
    return PMX_OK;
}

extern "C" void* pmx_ctx_stream(pmx_ctx* c) { return c ? (void*)c->stream : nullptr; }
extern "C" int64_t pmx_ctx_launch_count(const pmx_ctx* c) { return c ? c->launches : 0; }

// ---------------------------------------------------------------------------
static int get_stage_tw(pmx_ctx* c, const PmxLaunchTable* t, const void** dev) {
    const int L = t->L, precision = t->precision;
    const int key = L + 65536 * precision;
    auto it = c->stage_tw.find(key);
    if (it == c->stage_tw.end()) {
        const int total = t->tw_total;
        std::vector<cpx> h((size_t)(total > 0 ? total : 1));
        pmx_fill_stage_twiddles(L, h.data(), t->tw_layout);
        StageTw s;
        if (precision == PMX_F32) {  // same table, rounded once from the long-double values
            std::vector<float2> hf(h.size());
            for (size_t i = 0; i < h.size(); ++i) hf[i] = make_float2((float)h[i].x, (float)h[i].y);
            CK(c, cudaMalloc(&s.dev, hf.size() * sizeof(float2)));
            CK(c, cudaMemcpyAsync(s.dev, hf.data(), hf.size() * sizeof(float2), cudaMemcpyHostToDevice, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
        } else {
            CK(c, cudaMalloc(&s.dev, h.size() * sizeof(cpx)));
            CK(c, cudaMemcpyAsync(s.dev, h.data(), h.size() * sizeof(cpx), cudaMemcpyHostToDevice, c->stream));
            CK(c, cudaStreamSynchronize(c->stream));
        }
        it = c->stage_tw.emplace(key, s).first;
    }
    *dev = it->second.dev;
    return PMX_OK;
}

// W_N^(r*m) rows for a pass whose in-CTA transform has length L (table of that L gives the row layout) and
// whose tiles are indexed by r in [0, rows): rows * per entries, built on the device once per (N, L).
static int get_four_tw(pmx_ctx* c, long long N, const PmxLaunchTable* t, int rows, const void** out) {
    const long long key = (N * 8192 + t->L) * 2 + t->precision;
    auto it = c->four_tw.find(key);
    if (it == c->four_tw.end()) {
        FourStepTw tw;
        const size_t n = (size_t)rows * t->tw4_per;
        CK(c, cudaMalloc(&tw.rows, n * t->cpx_bytes));
        t->fill_tw4(tw.rows, rows, 2.0 / (double)N, c->stream);
        c->launches++;
        CK(c, cudaGetLastError());
        it = c->four_tw.emplace(key, tw).first;
    }
    *out = it->second.rows;
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// fields

// The pointwise kernels and the step kernels put a field's realization-columns (batch*nfc, or batch) in gridDim.y, which
// CUDA caps at 65535.  Refused up front, so that no kernel on a field or plan fails to launch.
#define PMX_MAX_BATCH_COLS 65535
static int check_batch_cols(pmx_ctx* c, const char* who, int64_t batch, int64_t nfc) {
    if (batch * nfc > PMX_MAX_BATCH_COLS)
        return set_err(c, PMX_ERR_UNSUPPORTED, "%s: batch*nfc = %lld x %lld = %lld realization-columns, at most %d", who,
                       (long long)batch, (long long)nfc, (long long)(batch * nfc), PMX_MAX_BATCH_COLS);
    return PMX_OK;
}

extern "C" int pmx_field_create(pmx_ctx* c, int64_t nfft, int32_t nfc, int32_t batch, int32_t precision,
                                pmx_devfield** out) {
    if (!c || !out) return set_err(c, PMX_ERR_INVALID, "pmx_field_create: null argument");
    *out = nullptr;
    if (precision != PMX_F64 && precision != PMX_F32) return set_err(c, PMX_ERR_INVALID, "unknown precision %d", precision);
    if (nfft <= 0 || nfc <= 0 || batch <= 0) return set_err(c, PMX_ERR_INVALID, "non-positive field size");
    if (int rc = check_batch_cols(c, "pmx_field_create", batch, nfc)) return rc;
    CK(c, cudaSetDevice(c->device));
    pmx_devfield* f = new (std::nothrow) pmx_devfield();
    if (!f) return set_err(c, PMX_ERR_INVALID, "out of host memory");
    f->ctx = c;
    f->nfft = nfft;
    f->nfc = nfc;
    f->batch = batch;
    f->precision = precision;
    size_t bytes = (size_t)batch * nfc * nfft * 2 * f->cbytes();
    cudaError_t e = cudaMallocAsync(&f->data, bytes, c->stream);
    if (e != cudaSuccess) {
        delete f;
        return set_err(c, PMX_ERR_CUDA, "cudaMallocAsync of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    }
    int rc = build_maps(c, f);
    if (rc != PMX_OK) {
        cudaFreeAsync(f->data, c->stream);
        delete f;
        return rc;
    }
    *out = f;
    return PMX_OK;
}

extern "C" void pmx_field_destroy(pmx_devfield* f) {
    if (!f) return;
    cudaSetDevice(f->ctx->device);
    cudaFreeAsync(f->data, f->ctx->stream);
    delete f;
}

extern "C" void* pmx_field_device_ptr(pmx_devfield* f) { return f ? (void*)f->data : nullptr; }

// position of time sample n of a column in the resident field (transposed four-step layout, or natural order)
__host__ __device__ __forceinline__ size_t pmx_mem_index(size_t n, int log2N1, int log2N2) {
    return ((n & (((size_t)1 << log2N2) - 1)) << log2N1) + (n >> log2N2);
}

// planar / complex host layouts (always double) <-> interleaved (xr,xi,yr,yi) in the field's precision;
// i runs over [columns][nfft] in host (time) order, the device side is permuted within each column
template <typename T2>
__device__ __forceinline__ T2 pmx_mk2(double a, double b);
template <>
__device__ __forceinline__ double2 pmx_mk2<double2>(double a, double b) { return make_double2(a, b); }
template <>
__device__ __forceinline__ float2 pmx_mk2<float2>(double a, double b) { return make_float2((float)a, (float)b); }

#define PMX_DEV_INDEX(i) ((((i) >> lg) << lg) + pmx_mem_index((i) & (((size_t)1 << lg) - 1), l1, lg - l1))
template <typename T2>
__global__ void pmx_k_pack_planar(T2* dst, const double* xr, const double* xi, const double* yr,
                                  const double* yi, size_t n, int lg, int l1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t m = PMX_DEV_INDEX(i);
        dst[2 * m] = pmx_mk2<T2>(xr[i], xi ? xi[i] : 0.0);
        dst[2 * m + 1] = pmx_mk2<T2>(yr ? yr[i] : 0.0, yi ? yi[i] : 0.0);
    }
}
template <typename T2>
__global__ void pmx_k_unpack_planar(const T2* src, double* xr, double* xi, double* yr, double* yi, size_t n, int lg, int l1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t m = PMX_DEV_INDEX(i);
        T2 x = src[2 * m], y = src[2 * m + 1];
        xr[i] = x.x;
        xi[i] = x.y;
        yr[i] = y.x;
        yi[i] = y.y;
    }
}
template <typename T2>
__global__ void pmx_k_pack_complex(T2* dst, const double2* x, const double2* y, size_t n, int lg, int l1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t m = PMX_DEV_INDEX(i);
        dst[2 * m] = pmx_mk2<T2>(x[i].x, x[i].y);
        dst[2 * m + 1] = y ? pmx_mk2<T2>(y[i].x, y[i].y) : pmx_mk2<T2>(0.0, 0.0);
    }
}
template <typename T2>
__global__ void pmx_k_unpack_complex(const T2* src, double2* x, double2* y, size_t n, int lg, int l1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t m = PMX_DEV_INDEX(i);
        x[i] = make_double2(src[2 * m].x, src[2 * m].y);
        y[i] = make_double2(src[2 * m + 1].x, src[2 * m + 1].y);
    }
}

static int check_range(pmx_devfield* f, int32_t b0, int32_t nb) {
    if (!f) return set_err(nullptr, PMX_ERR_INVALID, "null field");
    if (b0 < 0 || nb <= 0 || b0 + nb > f->batch)
        return set_err(f->ctx, PMX_ERR_INVALID, "realization range [%d,%d) outside batch %d", b0, b0 + nb, f->batch);
    return PMX_OK;
}

extern "C" int pmx_field_upload(pmx_devfield* f, const pmx_field* h, int32_t b0, int32_t nb) {
    int rc = check_range(f, b0, nb);
    if (rc) return rc;
    pmx_ctx* c = f->ctx;
    if (!h || !h->xr) return set_err(c, PMX_ERR_INVALID, "pmx_field_upload: null host field / xr");
    CK(c, cudaSetDevice(c->device));
    const size_t n = (size_t)nb * f->nfc * f->nfft;
    char* dstb = (char*)f->data + (size_t)b0 * f->nfc * f->nfft * 2 * f->cbytes();
    const bool f32 = f->precision == PMX_F32;
    const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
    if (h->layout == PMX_PLANAR) {
        double* stage = nullptr;
        CK(c, cudaMallocAsync(&stage, 4 * n * sizeof(double), c->stream));
        double* parts[4] = {h->xr, h->xi, h->yr, h->yi};
        double* dparts[4];
        for (int k = 0; k < 4; ++k) {
            dparts[k] = parts[k] ? stage + (size_t)k * n : nullptr;
            if (parts[k])
                CK(c, cudaMemcpyAsync(dparts[k], parts[k], n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        }
        if (f32)
            pmx_k_pack_planar<float2><<<blocks, 256, 0, c->stream>>>((float2*)dstb, dparts[0], dparts[1], dparts[2], dparts[3], n, f->log2N1 + f->log2N2, f->log2N1);
        else
            pmx_k_pack_planar<double2><<<blocks, 256, 0, c->stream>>>((double2*)dstb, dparts[0], dparts[1], dparts[2], dparts[3], n, f->log2N1 + f->log2N2, f->log2N1);
        c->launches++;
        CK(c, cudaGetLastError());
        CK(c, cudaFreeAsync(stage, c->stream));
    } else if (h->layout == PMX_COMPLEX) {
        cpx* stage = nullptr;
        CK(c, cudaMallocAsync(&stage, 2 * n * sizeof(cpx), c->stream));
        CK(c, cudaMemcpyAsync(stage, h->xr, n * sizeof(cpx), cudaMemcpyHostToDevice, c->stream));
        cpx* dy = nullptr;
        if (h->yr) {
            dy = stage + n;
            CK(c, cudaMemcpyAsync(dy, h->yr, n * sizeof(cpx), cudaMemcpyHostToDevice, c->stream));
        }
        if (f32)
            pmx_k_pack_complex<float2><<<blocks, 256, 0, c->stream>>>((float2*)dstb, stage, dy, n, f->log2N1 + f->log2N2, f->log2N1);
        else
            pmx_k_pack_complex<double2><<<blocks, 256, 0, c->stream>>>((double2*)dstb, stage, dy, n, f->log2N1 + f->log2N2, f->log2N1);
        c->launches++;
        CK(c, cudaGetLastError());
        CK(c, cudaFreeAsync(stage, c->stream));
    } else {
        return set_err(c, PMX_ERR_INVALID, "unknown layout %d", h->layout);
    }
    return PMX_OK;
}

extern "C" int pmx_field_download(pmx_devfield* f, pmx_field* h, int32_t b0, int32_t nb) {
    int rc = check_range(f, b0, nb);
    if (rc) return rc;
    pmx_ctx* c = f->ctx;
    if (!h || !h->xr || !h->yr) return set_err(c, PMX_ERR_INVALID, "pmx_field_download: null host arrays");
    CK(c, cudaSetDevice(c->device));
    const size_t n = (size_t)nb * f->nfc * f->nfft;
    const char* srcb = (const char*)f->data + (size_t)b0 * f->nfc * f->nfft * 2 * f->cbytes();
    const bool f32 = f->precision == PMX_F32;
    const int blocks = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
    if (h->layout == PMX_PLANAR) {
        if (!h->xi || !h->yi) return set_err(c, PMX_ERR_INVALID, "planar download needs xr, xi, yr, yi");
        double* stage = nullptr;
        CK(c, cudaMallocAsync(&stage, 4 * n * sizeof(double), c->stream));
        if (f32)
            pmx_k_unpack_planar<float2><<<blocks, 256, 0, c->stream>>>((const float2*)srcb, stage, stage + n, stage + 2 * n, stage + 3 * n, n, f->log2N1 + f->log2N2, f->log2N1);
        else
            pmx_k_unpack_planar<double2><<<blocks, 256, 0, c->stream>>>((const double2*)srcb, stage, stage + n, stage + 2 * n, stage + 3 * n, n, f->log2N1 + f->log2N2, f->log2N1);
        c->launches++;
        CK(c, cudaGetLastError());
        double* parts[4] = {h->xr, h->xi, h->yr, h->yi};
        for (int k = 0; k < 4; ++k)
            CK(c, cudaMemcpyAsync(parts[k], stage + (size_t)k * n, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaFreeAsync(stage, c->stream));
    } else if (h->layout == PMX_COMPLEX) {
        cpx* stage = nullptr;
        CK(c, cudaMallocAsync(&stage, 2 * n * sizeof(cpx), c->stream));
        if (f32)
            pmx_k_unpack_complex<float2><<<blocks, 256, 0, c->stream>>>((const float2*)srcb, stage, stage + n, n, f->log2N1 + f->log2N2, f->log2N1);
        else
            pmx_k_unpack_complex<double2><<<blocks, 256, 0, c->stream>>>((const double2*)srcb, stage, stage + n, n, f->log2N1 + f->log2N2, f->log2N1);
        c->launches++;
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(h->xr, stage, n * sizeof(cpx), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaMemcpyAsync(h->yr, stage + n, n * sizeof(cpx), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaFreeAsync(stage, c->stream));
    } else {
        return set_err(c, PMX_ERR_INVALID, "unknown layout %d", h->layout);
    }
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" int pmx_host_is_pinned(const void* p) {
    if (!p) return 0;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeHost ? 1 : 0;
}

extern "C" int pmx_field_broadcast(pmx_devfield* dst, const pmx_devfield* src) {
    if (!dst || !src) return set_err(nullptr, PMX_ERR_INVALID, "null field");
    pmx_ctx* c = dst->ctx;
    if (dst->nfft != src->nfft || dst->nfc != src->nfc || dst->precision != src->precision)
        return set_err(c, PMX_ERR_INVALID, "pmx_field_broadcast: shape or precision mismatch");
    CK(c, cudaSetDevice(c->device));
    const size_t bytes = (size_t)src->nfc * src->nfft * 2 * src->cbytes();
    for (int b = 0; b < dst->batch; ++b)
        CK(c, cudaMemcpyAsync((char*)dst->data + (size_t)b * bytes, src->data, bytes, cudaMemcpyDeviceToDevice, c->stream));
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// plans
// dst[col][k1*N2 + k2] = src[col][k1 + N1*k2]; *any |= (some element is non-zero)
__global__ void __launch_bounds__(256) pmx_k_permute(const double* __restrict__ src, double* __restrict__ dst,
                                                     int log2N1, int log2N2, int nfc, int* any) {
    const size_t N = (size_t)1 << (log2N1 + log2N2), total = N * nfc;
    int nz = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t col = i >> (log2N1 + log2N2), o = i & (N - 1);
        const size_t k1 = o >> log2N2, k2 = o & (((size_t)1 << log2N2) - 1);
        const double v = src[col * N + k1 + (k2 << log2N1)];
        nz |= (v != 0.0);
        dst[i] = v;
    }
    if (any && __any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0) atomicOr(any, 1);
}

static void fill_plates(const pmx_fiber_desc& d, int sets, const double* db0, const double* theta,
                        const double* epsilon, std::vector<PlateConst>& out) {
    const int np = d.nplates;
    out.resize((size_t)sets * np);
    for (int s = 0; s < sets; ++s) {
        for (int n = 0; n < np; ++n) {
            PlateConst& P = out[(size_t)s * np + n];
            const double th = theta ? theta[(size_t)s * np + n] : 0.0;
            const double ep = epsilon ? epsilon[(size_t)s * np + n] : 0.0;
            const double c = cos(th), sn = sin(th), ce = cos(ep), se = sin(ep);
            // matR = [c -s; s c] * [ce i*se; i*se ce]   (fiber.m:910-912)
            P.r11r = c * ce;  P.r11i = -sn * se;
            P.r12r = -sn * ce; P.r12i = c * se;
            P.r21r = sn * ce; P.r21i = c * se;
            P.r22r = c * ce;  P.r22i = sn * se;
            P.db0 = db0 ? db0[(size_t)s * np + n] : 0.0;
            P.h0r = cos(-0.5 * P.db0);
            P.h0i = sin(-0.5 * P.db0);
        }
        for (int n = 0; n < np; ++n) {
            PlateConst& P = out[(size_t)s * np + n];
            if (n + 1 < np) {
                const PlateConst& Q = out[(size_t)s * np + n + 1];
                // C = Q^H * P  (2x2 complex), computed in long double
                auto cm = [](long double ar, long double ai, long double br, long double bi, long double& rr,
                             long double& ri) {  // conj(a)*b accumulated
                    rr += ar * br + ai * bi;
                    ri += ar * bi - ai * br;
                };
                long double r, i;
                r = i = 0; cm(Q.r11r, Q.r11i, P.r11r, P.r11i, r, i); cm(Q.r21r, Q.r21i, P.r21r, P.r21i, r, i);
                P.c11r = (double)r; P.c11i = (double)i;
                r = i = 0; cm(Q.r11r, Q.r11i, P.r12r, P.r12i, r, i); cm(Q.r21r, Q.r21i, P.r22r, P.r22i, r, i);
                P.c12r = (double)r; P.c12i = (double)i;
                r = i = 0; cm(Q.r12r, Q.r12i, P.r11r, P.r11i, r, i); cm(Q.r22r, Q.r22i, P.r21r, P.r21i, r, i);
                P.c21r = (double)r; P.c21i = (double)i;
                r = i = 0; cm(Q.r12r, Q.r12i, P.r12r, P.r12i, r, i); cm(Q.r22r, Q.r22i, P.r22r, P.r22i, r, i);
                P.c22r = (double)r; P.c22i = (double)i;
            } else {
                P.c11r = 1; P.c11i = 0; P.c12r = 0; P.c12i = 0; P.c21r = 0; P.c21i = 0; P.c22r = 1; P.c22i = 0;
            }
            {   // C = diag(p, p*) * [ka kb; -kb* ka]:  p = c11/|c11|, ka = |c11|, kb = conj(p)*c12
                const long double ar = P.c11r, ai = P.c11i, m = hypotl(ar, ai);
                const long double pr = m > 0 ? ar / m : 1.0L, pi = m > 0 ? ai / m : 0.0L;
                P.ka = (double)m;
                P.pr = (double)pr;
                P.pi = (double)pi;
                P.kbr = (double)(pr * P.c12r + pi * P.c12i);
                P.kbi = (double)(pr * P.c12i - pi * P.c12r);
            }
        }
    }
}

extern "C" int pmx_plan_set_plates(pmx_plan* p, int32_t sets, const double* db0, const double* theta,
                                   const double* epsilon) {
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "null plan");
    pmx_ctx* c = p->ctx;
    if (sets != 1 && sets != p->d.batch)
        return set_err(c, PMX_ERR_INVALID, "plate_sets must be 1 or batch (%d), got %d", p->d.batch, sets);
    CK(c, cudaSetDevice(c->device));
    std::vector<PlateConst> h;
    fill_plates(p->d, sets, db0, theta, epsilon, h);
    if (p->plates == nullptr || sets != p->fc.plate_sets) {
        if (p->plates) CK(c, cudaFreeAsync(p->plates, c->stream));
        p->plates = nullptr;
        CK(c, cudaMallocAsync(&p->plates, h.size() * sizeof(PlateConst), c->stream));
    }
    p->fc.plate_sets = sets;
    CK(c, cudaMemcpyAsync(p->plates, h.data(), h.size() * sizeof(PlateConst), cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" void pmx_plan_destroy(pmx_plan* p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    cudaStream_t st = p->ctx->stream;
    if (p->betat_p) cudaFreeAsync(p->betat_p, st);
    if (p->db1_p) cudaFreeAsync(p->db1_p, st);
    if (p->hfilt) cudaFreeAsync(p->hfilt, st);
    if (p->plates) cudaFreeAsync(p->plates, st);
    if (p->ctl) cudaFreeAsync(p->ctl, st);
    if (p->pkg) cudaFreeAsync(p->pkg, st);
    if (p->trace_dz) cudaFreeAsync(p->trace_dz, st);
    if (p->trace_ntrunk) cudaFreeAsync(p->trace_ntrunk, st);
    if (p->sched) cudaFreeAsync(p->sched, st);
    if (p->geo_d) cudaFreeAsync(p->geo_d, st);
    if (p->sched_idx_d) cudaFreeAsync(p->sched_idx_d, st);
    if (p->sched_span_d) cudaFreeAsync(p->sched_span_d, st);
    pmx_plan_destroy(p->ch_dbp);
    pmx_plan_destroy(p->ch_band);
    pmx_field_destroy(p->ch_work);
    if (p->filt_hn_d) cudaFreeAsync(p->filt_hn_d, st);
    pmx_plan_destroy(p->filt);
    pmx_field_destroy(p->filt_work);
    pmx_field_destroy(p->tap_work);
    delete p;
}

// Which kernels a plan runs.  PLAN_AUTO: the single-launch kernel up to 2^12 samples and 8 columns (PMX_NO_ONCHIP=1 sends
// 2^12 through the three passes), the passes above.  Digital backpropagation fixes the route itself: PLAN_PASSES for
// two-polarization fields of 2^12 samples and more, PLAN_ONCHIP for everything smaller and for the scalar path.
enum PlanRoute { PLAN_AUTO, PLAN_PASSES, PLAN_ONCHIP };
static int plan_create(pmx_ctx* c, const pmx_fiber_desc* d, pmx_plan** out, PlanRoute route) {
    if (!c || !d || !out) return set_err(c, PMX_ERR_INVALID, "pmx_plan_create: null argument");
    *out = nullptr;
    if (d->precision != PMX_F64 && d->precision != PMX_F32)
        return set_err(c, PMX_ERR_INVALID, "unknown precision %d", d->precision);
    const int lg = ilog2_exact(d->nfft);
    if (lg < 6 || lg > 24)
        return set_err(c, PMX_ERR_UNSUPPORTED, "nfft=%lld: this build handles powers of two from 2^6 to 2^24",
                       (long long)d->nfft);
    // Fields of up to 4096 samples run in the single-launch on-chip kernel (one CTA per column, the columns of a
    // realization in one thread-block cluster): at most 8 columns.  PMX_NO_ONCHIP=1 sends 2^12 through the three passes.
    const bool no_onchip = getenv("PMX_NO_ONCHIP") && atoi(getenv("PMX_NO_ONCHIP"));
    const bool onchip = lg <= 12 && d->nfc <= 8 && route != PLAN_PASSES && !(no_onchip && lg == 12 && route == PLAN_AUTO);
    if (lg < 12 && !onchip)
        return set_err(c, PMX_ERR_UNSUPPORTED, "nfft=%lld (< 2^12) with nfc=%d: small fields take at most 8 columns",
                       (long long)d->nfft, d->nfc);
    if (d->nfc < 1 || d->nfc > PMX_MAX_NFC)
        return set_err(c, PMX_ERR_UNSUPPORTED, "nfc=%d outside [1,%d]", d->nfc, PMX_MAX_NFC);
    if (d->batch < 1) return set_err(c, PMX_ERR_INVALID, "batch must be >= 1");
    if (int rc = check_batch_cols(c, "pmx_plan_create", d->batch, d->nfc)) return rc;
    if (d->nplates < 1) return set_err(c, PMX_ERR_INVALID, "nplates must be >= 1");
    if (!(d->length > 0)) return set_err(c, PMX_ERR_INVALID, "length must be > 0");
    const bool scalar = d->disp_mode == PMX_DISP_SCALAR;
    if (!d->gam) return set_err(c, PMX_ERR_INVALID, "gam is required");
    if (!scalar && !d->betat) return set_err(c, PMX_ERR_INVALID, "betat is required in vector dispersion mode");
    if (scalar) {
        if (!d->beta1 || !d->beta2) return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode needs beta1 and beta2");
        if (d->nsymb <= 0 || d->nt <= 0 || (int64_t)d->nsymb * d->nt != d->nfft)
            return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode: nsymb*nt must equal nfft");
        if (!(d->symbolrate > 0)) return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode: symbolrate must be > 0");
    }
    if (d->fls[3] && !d->scalar_field)  // matrix_nl_step raises at fiber.m:853-854
        return set_err(c, PMX_ERR_XPM_VECTOR, "The CNLSE with separate fields is not yet implemented");
    if (d->scalar_field && d->fls[1]) return set_err(c, PMX_ERR_INVALID, "scalar_field excludes the 'p' flag (fiber.m:253-254)");
    if (d->plate_sets != 1 && d->plate_sets != d->batch)
        return set_err(c, PMX_ERR_INVALID, "plate_sets must be 1 or batch");
    if (!(d->dzmaxt > 0)) return set_err(c, PMX_ERR_INVALID, "dzmaxt must be > 0");
    if (d->z_start < 0 || d->dz_first < 0 || d->z_start != d->z_start || d->dz_first != d->dz_first)
        return set_err(c, PMX_ERR_INVALID, "z_start and dz_first must be >= 0");
    if ((d->z_start > 0 || d->dz_first > 0) && d->fls[1])
        return set_err(c, PMX_ERR_UNSUPPORTED, "a resumed propagation (z_start / dz_first) is built for fibers without the 'p' flag");
    CK(c, cudaSetDevice(c->device));

    pmx_plan* p = new (std::nothrow) pmx_plan();
    if (!p) return set_err(c, PMX_ERR_INVALID, "out of host memory");
    p->ctx = c;
    p->d = *d;
    p->d.gam = p->d.db0 = p->d.theta = p->d.epsilon = p->d.betat = p->d.db1 = p->d.beta1 = p->d.beta2 = nullptr;
    p->onchip = onchip;
    p->log2N1 = onchip ? 0 : split_log2N1(lg);   // on-chip: one transform of the full length, bins in natural order
    p->log2N2 = lg - p->log2N1;
    p->N1 = 1 << p->log2N1;
    p->N2 = 1 << p->log2N2;
    p->tA = pmx_get_table(onchip ? p->N2 : p->N1, d->precision);
    p->tB = pmx_get_table(p->N2, d->precision);
    if (!p->tA || !p->tB) {
        delete p;
        return set_err(c, PMX_ERR_UNSUPPORTED, "no kernel built for FFT factors %d x %d", 1 << (lg / 2), 1 << (lg - lg / 2));
    }
    if (onchip) {
        const int key = p->tB->L + 65536 * p->tB->precision + (1 << 20);
        if (!c->setup_done.count(key)) {
            cudaError_t e = p->tB->onchip_setup();
            if (e != cudaSuccess) {
                cudaGetLastError();   // (the failed attribute call is not sticky: clear it, or the next check reports it)
                delete p;
                return set_err(c, PMX_ERR_CUDA, "on-chip kernel setup (L=%d) failed: %s", (int)d->nfft, cudaGetErrorString(e));
            }
            c->setup_done[key] = pmx_ctx::Occ();
        }
    }
    for (const PmxLaunchTable* t : {p->tA, p->tB}) {
        if (onchip) break;
        if (!c->setup_done.count(t->L + 65536 * t->precision)) {
            pmx_ctx::Occ o;
            cudaError_t e = t->setup(&o.a, &o.b, &o.c, &o.cnl);
            if (e != cudaSuccess || o.a < 1 || o.b < 1 || o.c < 1 || o.cnl < 1) {
                cudaGetLastError();   // (as above)
                delete p;
                return set_err(c, PMX_ERR_CUDA, "kernel setup (L=%d) failed: %s (resident CTAs %d/%d/%d/%d)", t->L,
                               cudaGetErrorString(e), o.a, o.b, o.c, o.cnl);
            }
            c->setup_done[t->L + 65536 * t->precision] = o;
            if (getenv("PMX_VERBOSE"))
                fprintf(stderr, "[pmx] L=%d: resident CTAs/SM passA %d passB %d passC %d (smem %zu / %zu B)\n", t->L, o.a, o.b, o.c,
                        t->smemAC, t->smemB);
        }
    }
    FiberConst& f = p->fc;
    memset(&f, 0, sizeof f);
    f.Lf = d->length;
    f.alphalin = d->alphalin;
    f.halfalpha = 0.5 * d->alphalin;  // fiber.m:514
    f.dzmax = d->dzmaxt;
    f.phimax = d->dphimaxt;
    f.lcorr = d->length / d->nplates;  // fiber.m:507
    f.invN = 1.0 / (double)d->nfft;
    for (int k = 0; k < d->nfc; ++k) f.gam[k] = d->manakov ? d->gam[k] * 8 / 9 : d->gam[k];  // fiber.m:500
    f.nplates = d->nplates;
    f.nfc = d->nfc;
    f.spm = d->fls[2] ? 1 : 0;
    f.manakov = d->manakov ? 1 : 0;
    f.plate_sets = d->plate_sets;
    // Without the 'p' flag the front-end passes identity plates and db1 = 0 (fiber.m:290-298):
    // the Jones product is skipped altogether.
    f.pmd = d->fls[1] ? 1 : 0;
    f.keep_basis = (f.pmd && (f.manakov || !f.spm)) ? 1 : 0;
    f.scalar_field = d->scalar_field ? 1 : 0;
    f.xpm = (d->scalar_field && d->fls[3]) ? 1 : 0;
    f.z_start = d->z_start;
    f.dz_first = d->dz_first;
    f.nfc_magic = d->nfc > 1 ? (unsigned)((0x100000000ull + d->nfc - 1) / d->nfc) : 0u;
    const size_t N = (size_t)d->nfft;
    p->single_step = std::isinf(d->dphimaxt) && d->dzmaxt >= d->length;

    if (scalar) {
        f.disp_scalar = 1;
        f.w0 = 2 * M_PI * d->symbolrate;  // fiber.m:352  2*pi*GSTATE.SYMBOLRATE (*FN)
        f.inv_nsymb = 1.0 / (double)d->nsymb;
        f.b30_6 = d->b30 / 6;
        f.dgdrms = f.pmd ? d->dgdrms : 0.0;
        f.domega = f.w0 * ((double)d->nt / 8.0);
        f.g1r = cos(0.5 * f.dgdrms * f.domega);
        f.g1i = -sin(0.5 * f.dgdrms * f.domega);
        f.g2r = cos(f.dgdrms * f.domega);
        f.g2i = -sin(f.dgdrms * f.domega);
        f.g4r = cos(2.0 * f.dgdrms * f.domega);
        f.g4i = -sin(2.0 * f.dgdrms * f.domega);
        bool any = d->b30 != 0.0;
        for (int k = 0; k < d->nfc; ++k) {
            f.beta1[k] = d->beta1[k];
            f.beta2[k] = d->beta2[k];
            any = any || d->beta1[k] != 0.0 || d->beta2[k] != 0.0;
        }
        f.gvd_any = any ? 1 : 0;
        cudaError_t e = cudaMallocAsync(&p->ctl, 2 * (size_t)d->batch * sizeof(StepCtl), c->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(&p->pkg, (size_t)d->batch * sizeof(StepPkg), c->stream);
        if (e != cudaSuccess) {
            pmx_plan_destroy(p);
            return set_err(c, PMX_ERR_CUDA, "plan allocation failed: %s", cudaGetErrorString(e));
        }
    } else
    // dispersion vectors, permuted on the device: bin k1 + N1*k2 -> position k1*N2 + k2
    {
        const size_t bytes = N * d->nfc * sizeof(double);
        double* raw = nullptr;
        int* d_any = nullptr;
        cudaError_t e = cudaMallocAsync(&p->betat_p, bytes, c->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(&raw, bytes, c->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(&d_any, sizeof(int), c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(d_any, 0, sizeof(int), c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(raw, d->betat, bytes, cudaMemcpyHostToDevice, c->stream);
        const int blocks = (int)std::min<size_t>((N * d->nfc + 255) / 256, 148 * 16);
        if (e == cudaSuccess) {
            pmx_k_permute<<<blocks, 256, 0, c->stream>>>(raw, p->betat_p, p->log2N1, p->log2N2, d->nfc, d_any);
            c->launches++;
            e = cudaGetLastError();
        }
        int any = 1;
        if (e == cudaSuccess) e = cudaMemcpyAsync(&any, d_any, sizeof(int), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && f.pmd) {
            e = cudaMallocAsync(&p->db1_p, bytes, c->stream);
            if (e == cudaSuccess) {
                if (d->db1) {
                    // raw is reused: the copy is stream-ordered after the betat permute
                    e = cudaMemcpyAsync(raw, d->db1, bytes, cudaMemcpyHostToDevice, c->stream);
                    if (e == cudaSuccess) {
                        pmx_k_permute<<<blocks, 256, 0, c->stream>>>(raw, p->db1_p, p->log2N1, p->log2N2, d->nfc, nullptr);
                        c->launches++;
                        e = cudaGetLastError();
                    }
                } else {
                    e = cudaMemsetAsync(p->db1_p, 0, bytes, c->stream);
                }
            }
        }
        if (e == cudaSuccess) e = cudaMallocAsync(&p->ctl, 2 * (size_t)d->batch * sizeof(StepCtl), c->stream);
        if (e == cudaSuccess) e = cudaMallocAsync(&p->pkg, (size_t)d->batch * sizeof(StepPkg), c->stream);
        if (raw) cudaFreeAsync(raw, c->stream);
        if (d_any) cudaFreeAsync(d_any, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);  // host vectors may go away; `any` is valid
        if (e != cudaSuccess) {
            pmx_plan_destroy(p);
            return set_err(c, PMX_ERR_CUDA, "plan allocation failed: %s", cudaGetErrorString(e));
        }
        f.gvd_any = any ? 1 : 0;
    }
    int rc = pmx_plan_set_plates(p, d->plate_sets, d->db0, d->theta, d->epsilon);
    if (rc) {
        pmx_plan_destroy(p);
        return rc;
    }
    *out = p;
    return PMX_OK;
}

extern "C" int pmx_plan_create(pmx_ctx* c, const pmx_fiber_desc* d, pmx_plan** out) { return plan_create(c, d, out, PLAN_AUTO); }

// ---------------------------------------------------------------------------
// A linear filter as a plan: one step of a fiber without dispersion, birefringence, nonlinearity or loss whose per-bin
// factor is the caller's H instead of exp(-i*betat*dz).  pmx_fiber_exec on it is u <- ifft(fft(u) .* H).
__global__ void __launch_bounds__(256) pmx_k_permute_c(const double2* __restrict__ src, double2* __restrict__ dst, int log2N1,
                                                       int log2N2, int ncol) {
    const size_t N = (size_t)1 << (log2N1 + log2N2), total = N * ncol;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t col = i >> (log2N1 + log2N2), o = i & (N - 1);
        const size_t k1 = o >> log2N2, k2 = o & (((size_t)1 << log2N2) - 1);
        dst[i] = src[col * N + k1 + (k2 << log2N1)];
    }
}

// The filter plan of pmx_filter_create with H taken from `raw`, a [hcols][nfft] table in FFT order that is already on the
// device (host_raw = 0) or on the host (host_raw = 1).  pmx_pb_table writes its per-node tables on the device and calls
// filter_set_raw again for every chunk of nodes.
static int filter_set_raw(pmx_plan* p, const double2* raw, int32_t hcols) {
    pmx_k_permute_c<<<(unsigned)std::min<size_t>(((size_t)p->d.nfft * hcols + 255) / 256, 148 * 16), 256, 0,
                      p->ctx->stream>>>(raw, p->hfilt, p->log2N1, p->log2N2, hcols);
    p->ctx->launches++;
    return cudaGetLastError() == cudaSuccess ? PMX_OK : PMX_ERR_CUDA;
}

static int filter_create(pmx_ctx* c, int64_t nfft, int32_t nfc, int32_t batch, int32_t precision, const double* H,
                         int host_raw, int32_t hcols, pmx_plan** out) {
    *out = nullptr;
    if (nfc < 1 || (hcols != 1 && hcols != nfc))
        return set_err(c, PMX_ERR_INVALID, "pmx_filter_create: H must have one column, or one per field column");
    if (nfft < 1) return set_err(c, PMX_ERR_INVALID, "pmx_filter_create: nfft");
    const std::vector<double> zeros((size_t)nfft * nfc, 0.0), gam((size_t)nfc, 0.0);
    const double zero1 = 0.0;
    pmx_fiber_desc d;
    memset(&d, 0, sizeof d);
    d.nfft = nfft;
    d.nfc = nfc;
    d.batch = batch;
    d.precision = precision;
    d.length = d.dzmaxt = 1.0;
    d.dphimaxt = INFINITY;
    d.gam = gam.data();
    d.fls[0] = 1;                       // 'g---': exactly one linear step
    d.nplates = d.plate_sets = 1;
    d.db0 = d.theta = d.epsilon = &zero1;
    d.betat = zeros.data();
    d.disp_mode = PMX_DISP_VECTOR;
    d.nsymb = (int32_t)std::min<int64_t>(nfft, INT32_MAX);
    d.nt = 1;
    d.symbolrate = 1.0;
    pmx_plan* p = nullptr;
    int rc = pmx_plan_create(c, &d, &p);
    if (rc) return rc;
    const size_t n = (size_t)nfft * hcols;
    double2* raw = nullptr;
    cudaError_t e = cudaMallocAsync(&p->hfilt, n * sizeof(double2), c->stream);
    if (host_raw) {
        if (e == cudaSuccess) e = cudaMallocAsync(&raw, n * sizeof(double2), c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(raw, H, n * sizeof(double2), cudaMemcpyHostToDevice, c->stream);
    }
    if (e == cudaSuccess) {
        pmx_k_permute_c<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 16), 256, 0, c->stream>>>(
            host_raw ? raw : reinterpret_cast<const double2*>(H), p->hfilt, p->log2N1, p->log2N2, hcols);
        c->launches++;
        e = cudaGetLastError();
    }
    if (raw) cudaFreeAsync(raw, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);   // the caller's H may go away
    if (e != cudaSuccess) {
        pmx_plan_destroy(p);
        return set_err(c, PMX_ERR_CUDA, "pmx_filter_create: %s", cudaGetErrorString(e));
    }
    p->hfilt_stride = hcols > 1 ? (long long)nfft : 0;
    *out = p;
    return PMX_OK;
}

extern "C" int pmx_filter_create(pmx_ctx* c, int64_t nfft, int32_t nfc, int32_t batch, int32_t precision, const double* H,
                                 int32_t hcols, pmx_plan** out) {
    if (!c || !H || !out) return set_err(c, PMX_ERR_INVALID, "pmx_filter_create: null argument");
    return filter_create(c, nfft, nfc, batch, precision, H, 1, hcols, out);
}

// ---------------------------------------------------------------------------
static int ensure_hctl(pmx_ctx* c, int batch) {
    if (c->h_ctl_cap < batch) {
        if (c->h_ctl) cudaFreeHost(c->h_ctl);
        c->h_ctl = nullptr;
        CK(c, cudaMallocHost(&c->h_ctl, (size_t)batch * sizeof(StepCtl)));
        c->h_ctl_cap = batch;
    }
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// Launch scaffold of the three passes, shared by pmx_fiber_exec and pmx_dbp_exec.

// A field runs with a plan of the same device, precision and shape.
static int check_field(pmx_plan* p, const pmx_devfield* fld) {
    pmx_ctx* c = p->ctx;
    // a field may be worked on by a plan of another context of the SAME device (a second stream, e.g. a receive chain running
    // beside the next group's propagation): the caller orders the two streams (every call here returns synchronised)
    if (fld->ctx != c && fld->ctx->device != c->device)
        return set_err(c, PMX_ERR_INVALID, "field and plan belong to contexts on different devices");
    if (fld->precision != p->d.precision)
        return set_err(c, PMX_ERR_INVALID, "field precision %d does not match the plan's %d", fld->precision, p->d.precision);
    if (fld->nfft != p->d.nfft || fld->nfc != p->d.nfc || fld->batch != p->d.batch)
        return set_err(c, PMX_ERR_INVALID, "field shape (%lld,%d,%d) does not match the plan (%lld,%d,%d)",
                       (long long)fld->nfft, fld->nfc, fld->batch, (long long)p->d.nfft, p->d.nfc, p->d.batch);
    if (!p->onchip && !fld->has_maps) return set_err(c, PMX_ERR_INVALID, "field has no tensor maps (unsupported nfft)");
    return PMX_OK;
}

// The launch parameters of plan p on field fld: pa for every kernel, pA and pB for passes A (and C) and B with their
// stage and four-step twiddles (an on-chip plan runs no passes: pA and pB are pa).
static int pass_params(pmx_plan* p, const pmx_devfield* fld, PassParams& pa, PassParams& pA, PassParams& pB) {
    pmx_ctx* c = p->ctx;
    memset(&pa, 0, sizeof pa);
    pa.field = fld->data;
    pa.ctl = p->ctl;
    pa.betat_p = p->betat_p;
    pa.db1_p = p->db1_p;
    pa.hfilt = p->hfilt;
    pa.hfilt_stride = p->hfilt_stride;
    pa.plates = p->plates;
    pa.trace_dz = p->trace_dz;
    pa.trace_ntrunk = p->trace_ntrunk;
    pa.N1 = p->N1;
    pa.N2 = p->N2;
    pa.log2N1 = p->log2N1;
    pa.log2N2 = p->log2N2;
    pa.batch = p->d.batch;
    pa.dbg = g_dbg;
    pa.pkg = p->pkg;
    pA = pB = pa;
    if (p->onchip) return PMX_OK;
    int rc = get_four_tw(c, p->d.nfft, p->tA, p->N2, &pA.tw4);       // pass A: one row per column n2, W_N^(n2*k1), k1 < N1
    if (!rc) rc = get_four_tw(c, p->d.nfft, p->tB, p->N1, &pB.tw4);  // pass B: one row per k1, W_N^(k1*n2), n2 < N2
    if (!rc) rc = get_stage_tw(c, p->tA, &pA.tw_stage);
    if (!rc) rc = get_stage_tw(c, p->tB, &pB.tw_stage);
    return rc;
}

// Realization groups.  The batch is split into groups that run on their own streams with full-size persistent
// grids: while the last CTAs of one group's pass drain (tile-count quantisation, stragglers, the launch gap and
// the one-CTA-per-realization step control), the other group's pass already fills the freed SM slots.
struct PassGroup {
    cudaStream_t st;
    int b0, nb;             // realizations b0 .. b0 + nb - 1
    int gA, gB, gC;         // grids of passes A, B and C
    PassParams pA, pB, pc;  // pass A (and C), pass B, the other kernels: pa, pA, pB of pass_params on the group's realizations
};
struct PassGroups {
    int n;
    int pdl;  // launch with programmatic stream serialization
    PassGroup g[4];
};

// occC: resident CTAs per SM of the pass-C kernel the caller launches; allow_pdl: programmatic dependent launch with a
// single group.
static int plan_groups(pmx_plan* p, const pmx_devfield* fld, const PassParams& pa, const PassParams& pA,
                       const PassParams& pB, int occC, bool allow_pdl, PassGroups& gs) {
    pmx_ctx* c = p->ctx;
    const int batch = p->d.batch, nfc = p->d.nfc;
    const pmx_ctx::Occ oA = c->setup_done[p->N1 + 65536 * p->d.precision], oB = c->setup_done[p->N2 + 65536 * p->d.precision];
    static const int env_groups = getenv("PMX_GROUPS") ? atoi(getenv("PMX_GROUPS")) : 0;
    // two groups pay once a pass has more than about two rounds of tiles; below that a single group with
    // programmatic dependent launches (prologue of the next kernel under the tail of the current one) is faster
    const long tiles_all = (long)(p->N2 / p->tA->gAC) * batch * nfc;
    const int want_groups = env_groups ? env_groups : (tiles_all > 2L * c->sm_count * oA.a ? 2 : 1);
    gs.n = c->profile ? 1 : std::max(1, std::min(std::min(want_groups, 4), batch));
    // programmatic dependent launch pays when nothing else fills the gap between two kernels of a stream, i.e. with a
    // single realization group (a batch of one: the reference-style fiber() call)
    gs.pdl = (gs.n == 1 && allow_pdl) ? 1 : 0;
    for (int g = 1; g < gs.n; ++g)
        if (!c->gstream[g - 1]) {
            CK(c, cudaStreamCreateWithFlags(&c->gstream[g - 1], cudaStreamNonBlocking));
            CK(c, cudaEventCreateWithFlags(&c->ev_join[g - 1], cudaEventDisableTiming));
            if (!c->ev_fork) CK(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        }
    // Persistent grids of one CTA per resident slot -- except when a pass has between one and two rounds of
    // tiles (a batch of one at N = 2^20: 1024 tiles on 592 slots): then one CTA per tile, so that the hardware
    // hands the tiles of the partial second round to whichever slot frees first (measured +8 % at batch 1, N = 2^20;
    // with more rounds the persistent grid is the faster one, grid sizing in DESIGN.md)
    auto grid_of = [&](int tiles, int ctas_per_sm) {
        const int slots = ctas_per_sm * c->sm_count;
        if (tiles > slots && tiles <= 2 * slots) return tiles;
        return std::min(tiles, slots);
    };
    const size_t N = (size_t)p->d.nfft;
    for (int g = 0; g < gs.n; ++g) {
        PassGroup& G = gs.g[g];
        G.b0 = (int)((long long)g * batch / gs.n);
        G.nb = (int)((long long)(g + 1) * batch / gs.n) - G.b0;
        G.st = g == 0 ? c->stream : c->gstream[g - 1];
        for (PassParams* q : {&G.pA, &G.pB, &G.pc}) {
            *q = (q == &G.pA) ? pA : (q == &G.pB ? pB : pa);
            q->field = (char*)pa.field + (size_t)G.b0 * nfc * N * 2 * fld->cbytes();
            q->ctl = pa.ctl + G.b0;
            q->pkg = pa.pkg + G.b0;
            if (p->fc.plate_sets > 1) q->plates = pa.plates + (size_t)G.b0 * p->fc.nplates;
            if (pa.trace_dz) {
                q->trace_dz = pa.trace_dz + (size_t)G.b0 * p->trace_cap;
                q->trace_ntrunk = pa.trace_ntrunk + (size_t)G.b0 * p->trace_cap;
            }
            q->batch = G.nb;
            q->bc0 = G.b0 * nfc;
            q->pdl = gs.pdl;
        }
        const int tilesAC = (p->N2 / p->tA->gAC) * G.nb * nfc, tilesB = (p->N1 / p->tB->gB) * G.nb * nfc;
        G.gA = grid_of(tilesAC, oA.a);
        G.gB = grid_of(tilesB, oB.b);
        G.gC = grid_of(tilesAC, occC);
    }
    return PMX_OK;
}

// The streams of the other groups start after everything queued on the first one so far.
static int fork_groups(pmx_ctx* c, int ngroups) {
    if (ngroups < 2) return PMX_OK;
    CK(c, cudaEventRecord(c->ev_fork, c->stream));
    for (int g = 1; g < ngroups; ++g) CK(c, cudaStreamWaitEvent(c->gstream[g - 1], c->ev_fork, 0));
    return PMX_OK;
}
// The first stream waits for what the other groups have queued.
static int join_groups(pmx_ctx* c, int ngroups) {
    for (int g = 1; g < ngroups; ++g) {
        CK(c, cudaEventRecord(c->ev_join[g - 1], c->gstream[g - 1]));
        CK(c, cudaStreamWaitEvent(c->stream, c->ev_join[g - 1], 0));
    }
    return PMX_OK;
}

extern "C" int pmx_fiber_exec(pmx_plan* p, pmx_devfield* fld, pmx_fiber_result* out) {
    if (!p || !fld) return set_err(nullptr, PMX_ERR_INVALID, "pmx_fiber_exec: null argument");
    pmx_ctx* c = p->ctx;
    int rc = check_field(p, fld);
    if (rc) return rc;
    if (p->dbp) return set_err(c, PMX_ERR_INVALID, "pmx_fiber_exec: a digital-backpropagation plan runs with pmx_dbp_exec");
    CK(c, cudaSetDevice(c->device));
    const int batch = p->d.batch, nfc = p->d.nfc;
    rc = ensure_hctl(c, batch);
    if (rc) return rc;

    // optional schedule trace
    int want_cap = (out && out->trace_dz && out->trace_ntrunk && out->trace_cap > 0) ? out->trace_cap : 0;
    if (want_cap != p->trace_cap) {
        if (p->trace_dz) cudaFreeAsync(p->trace_dz, c->stream);
        if (p->trace_ntrunk) cudaFreeAsync(p->trace_ntrunk, c->stream);
        p->trace_dz = nullptr;
        p->trace_ntrunk = nullptr;
        p->trace_cap = 0;
        if (want_cap) {
            CK(c, cudaMallocAsync(&p->trace_dz, (size_t)batch * want_cap * sizeof(double), c->stream));
            CK(c, cudaMallocAsync(&p->trace_ntrunk, (size_t)batch * want_cap * sizeof(int), c->stream));
            p->trace_cap = want_cap;
        }
    }
    if (p->trace_cap) {
        CK(c, cudaMemsetAsync(p->trace_dz, 0, (size_t)batch * p->trace_cap * sizeof(double), c->stream));
        CK(c, cudaMemsetAsync(p->trace_ntrunk, 0, (size_t)batch * p->trace_cap * sizeof(int), c->stream));
    }
    p->fc.trace_cap = p->trace_cap;

    PassParams pa, pA, pB;
    rc = pass_params(p, fld, pa, pA, pB);
    if (rc) return rc;
    CK(c, cudaMemsetAsync(p->ctl, 0, 2 * (size_t)batch * sizeof(StepCtl), c->stream));   // ([1]: the second block of the fused control)
    CK(c, cudaMemsetAsync(p->pkg, 0, (size_t)batch * sizeof(StepPkg), c->stream));
    // what the caller gets back, from the control blocks read into h_ctl
    auto collect = [&]() -> int {
        int worst = PMX_OK;
        for (int b = 0; b < batch; ++b) {
            const StepCtl& s = c->h_ctl[b];
            int st = (s.state == PMX_ST_ERROR) ? s.err : PMX_OK;
            if (st != PMX_OK && worst == PMX_OK) worst = st;
            if (out) {
                if (out->firstdz) out->firstdz[b] = s.firstdz;
                if (out->ncycle) out->ncycle[b] = s.ncycle;
                if (out->ntot) out->ntot[b] = s.ntot + s.ntrunk - s.nmem;
                if (out->status) out->status[b] = st;
            }
        }
        if (p->trace_cap && out) {
            CK(c, cudaMemcpy(out->trace_dz, p->trace_dz, (size_t)batch * p->trace_cap * sizeof(double), cudaMemcpyDeviceToHost));
            CK(c, cudaMemcpy(out->trace_ntrunk, p->trace_ntrunk, (size_t)batch * p->trace_cap * sizeof(int), cudaMemcpyDeviceToHost));
        }
        if (worst == PMX_ERR_PLATE_INDEX)
            return set_err(c, worst, "trunk counter exceeded nplates=%d (the reference raises an index error at fiber.m:910 "
                                     "for this length/nplates pair)", p->d.nplates);
        if (worst != PMX_OK) return set_err(c, worst, "NaN/Inf met in the step control");
        return PMX_OK;
    };
    if (p->onchip) {   // small field: the whole loop of every realization in one launch
        PassParams q = pa;
        rc = get_stage_tw(c, p->tB, &q.tw_stage);
        if (rc) return rc;
        q.N1 = 1;
        q.N2 = (int)p->d.nfft;
        q.log2N1 = fld->log2N1;   // layout of the resident column (transposed for 2^12, natural below)
        q.log2N2 = fld->log2N2;
        CK(c, p->tB->onchip(nfc, batch, c->stream, q, p->fc));
        c->launches += 1;
        CK(c, cudaMemcpyAsync(c->h_ctl, p->ctl, (size_t)batch * sizeof(StepCtl), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
        return collect();
    }
    // A batch of one (the reference-style fiber() call) has nothing to overlap the step-control kernel with: pass A then
    // runs the control itself (pmx_k_passA<..., FUSED>), three dependent launches per step instead of four.
    // Every CTA of that pass A repeats the (scalar, 2-3 us) control, so it pays while the pass is a single round of CTAs --
    // fields of up to 2^19 samples; measured at 2^16: 31.9 -> 27.9 us per step, at 2^20 (1024 CTAs in two rounds) -3 %.
    const bool fused = batch == 1 && !p->fc.xpm && !c->profile &&
                       (long)(p->N2 / p->tA->gAC) * nfc <= (long)c->sm_count * c->setup_done[p->N1 + 65536 * p->d.precision].a;
    {
        dim3 g(148 * 2, batch * nfc);
        ProfScope ps(c, 3);
        p->tA->init_max(g, c->stream, pa, p->fc);
        c->launches += 1;
        if (!fused) {
            pmx_k_ctl<<<batch, 128, 0, c->stream>>>(pa, p->fc, 1);
            c->launches += 1;
        }
        CK(c, cudaGetLastError());
    }
    int par = 0;          // fused control: the block the next pass A reads
    int fused_first = 1;
    PassGroups gs;
    rc = plan_groups(p, fld, pa, pA, pB, c->setup_done[p->N1 + 65536 * p->d.precision].c, !c->profile && !p->fc.xpm, gs);
    if (rc) return rc;
    const size_t N = (size_t)p->d.nfft;
    int chunk = p->single_step ? 1 : 8;
    int rev[4] = {1, 1, 1, 1};
    long total_steps = 0;
    for (;;) {
        rc = fork_groups(c, gs.n);
        if (rc) return rc;
        for (int s = 0; s < chunk; ++s) {
            for (int gi = 0; gi < gs.n; ++gi) {
                PassGroup& G = gs.g[gi];
                // serpentine tile order: consecutive passes walk the realizations in opposite directions
                G.pA.reverse = (rev[gi] ^= 1);
                if (p->fc.xpm) {  // row sums of |u|^2 over the columns, parked in the (empty) Y slots for pass A
                    p->tA->xpm_sum(dim3((unsigned)std::min<size_t>((N + 255) / 256, 148 * 8), G.nb), G.st, G.pA, p->fc);
                    c->launches++;
                }
                if (fused) {   // pass A reads block `par`, writes block `par ^ 1`; pass C gathers the maxima in the new one
                    G.pA.ctl = p->ctl + par;
                    G.pA.ctl_out = p->ctl + (par ^ 1);
                    G.pA.first = fused_first;
                }
                { ProfScope ps(c, 0); CK(c, p->tA->passA(G.gA, G.st, G.pA, p->fc, fld->map_rows)); }
                G.pB.reverse = (rev[gi] ^= 1);
                { ProfScope ps(c, 1); CK(c, p->tB->passB(G.gB, G.st, G.pB, p->fc, fld->map_cols)); }
                G.pA.reverse = (rev[gi] ^= 1);
                if (fused) {
                    PassParams pC = G.pA;
                    pC.ctl = p->ctl + (par ^ 1);
                    pC.ctl_out = nullptr;
                    CK(c, p->tA->passC(G.gC, G.st, pC, p->fc, fld->map_rows));
                    par ^= 1;
                    fused_first = 0;
                    c->launches += 3;
                    continue;
                }
                { ProfScope ps(c, 2); CK(c, p->tA->passC(G.gC, G.st, G.pA, p->fc, fld->map_rows)); }
                if (gs.pdl) {
                    cudaLaunchConfig_t cfg = {};
                    cfg.gridDim = dim3(G.nb);
                    cfg.blockDim = dim3(128);
                    cfg.stream = G.st;
                    cudaLaunchAttribute at[1];
                    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                    at[0].val.programmaticStreamSerializationAllowed = 1;
                    cfg.attrs = at;
                    cfg.numAttrs = 1;
                    CK(c, cudaLaunchKernelEx(&cfg, pmx_k_ctl, G.pc, p->fc, 0));
                } else {
                    pmx_k_ctl<<<G.nb, 128, 0, G.st>>>(G.pc, p->fc, 0);
                }
                c->launches += 4;
            }
            if (c->profile && c->ev_used > 4096) prof_collect(c);
        }
        total_steps += chunk;
        CK(c, cudaGetLastError());
        rc = join_groups(c, gs.n);
        if (rc) return rc;
        CK(c, cudaMemcpyAsync(c->h_ctl, p->ctl + (fused ? par : 0), (size_t)batch * sizeof(StepCtl), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
        bool all_done = true;
        // (fused control: no kernel follows the last step's passes to turn LAST into DONE; LAST at the end of a chunk --
        // every later launch of the chunk having found the fiber finished -- means the same)
        for (int b = 0; b < batch; ++b)
            if (c->h_ctl[b].state < (fused ? PMX_ST_LAST : PMX_ST_DONE)) all_done = false;
        if (all_done) break;
        if (total_steps > 10000000) return set_err(c, PMX_ERR_NUMERIC, "step loop did not terminate");
        // Size the next chunk from what is left: steps beyond the last one of every realization are launches that
        // exit at once (a few microseconds each), a chunk that ends early costs one more read-back.  With
        // attenuation the step grows like exp(alpha*z) while it is bounded by the nonlinear phase, so
        // (1 - exp(-alpha*r)) / (alpha*dz) steps remain over the length r; r/dz is the bound for constant steps.
        double est = 1.0;
        for (int b = 0; b < batch; ++b) {
            const StepCtl& sc = c->h_ctl[b];
            if (sc.state >= PMX_ST_DONE || !(sc.dz > 0)) continue;
            const double r = std::max(0.0, p->fc.Lf - sc.zprop) + sc.dz;
            const double lin = r / sc.dz;
            const double a = p->fc.alphalin;
            const double ex = (a > 0) ? (1.0 - exp(-a * r)) / (a * sc.dz) : lin;
            est = std::max(est, 0.5 * (lin + ex));
        }
        chunk = (int)std::min(32.0, std::max(1.0, ceil(0.85 * est)));
    }
    return collect();
}

extern "C" int pmx_fiber_run(pmx_ctx* c, const pmx_fiber_desc* d, pmx_field* io, pmx_fiber_result* out) {
    if (!c || !d || !io) return set_err(c, PMX_ERR_INVALID, "pmx_fiber_run: null argument");
    pmx_plan* plan = nullptr;
    pmx_devfield* f = nullptr;
    int rc = pmx_plan_create(c, d, &plan);
    if (rc == PMX_OK) rc = pmx_field_create(c, d->nfft, d->nfc, d->batch, d->precision, &f);
    if (rc == PMX_OK) rc = pmx_field_upload(f, io, 0, d->batch);
    if (rc == PMX_OK) rc = pmx_fiber_exec(plan, f, out);
    if (rc == PMX_OK) rc = pmx_field_download(f, io, 0, d->batch);
    std::string keep = c->error;
    pmx_field_destroy(f);
    pmx_plan_destroy(plan);
    if (rc != PMX_OK) {
        c->error = keep;
        g_tls_error = keep;
    }
    return rc;
}

// ---------------------------------------------------------------------------
// ampliflat: flat gain + ASE (ampliflat.m:78-148)
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// complex standard normal (randn + i*randn): Box-Muller on two 32-bit uniforms
__device__ __forceinline__ cpx pmx_cnormal(uint32_t a, uint32_t b) {
    const double u1 = ((double)a + 0.5) * (1.0 / 4294967296.0);
    const double u2 = ((double)b + 0.5) * (1.0 / 4294967296.0);
    const double r = sqrt(-2.0 * log(u1));
    double s, cs;
    sincospi(2.0 * u2, &s, &cs);
    return make_double2(r * cs, r * s);
}

struct AmpParams {
    void* field;       // double2 or float2 elements (field precision)
    const cpx* noise;  // [batch][2*nfc][N] or null
    double sg;         // sqrt(gain)
    double sigma[PMX_MAX_NFC];
    unsigned long long seed;
    size_t N;
    int nfc, batch;
    int l1, l2;        // field layout: time sample n1*N2 + n2 at n2*N1 + n1 (log2 N1, log2 N2; 0/0 = natural order)
    int asepol;        // bit 0: ASE on X, bit 1: ASE on Y (options.onepol, ampliflat.m:107-118)
    unsigned b0;       // global index of the batch's first realization: the generator is keyed by the realization, so a
                       // Monte-Carlo run draws the same noise however its realizations are grouped or sharded
};

template <typename T2>  // the gain and the noise are evaluated in double in both field precisions
__global__ void __launch_bounds__(256) pmx_k_ampliflat(AmpParams a) {
    const int bc = blockIdx.y, b = bc / a.nfc, col = bc % a.nfc;
    T2* fld = reinterpret_cast<T2*>(a.field) + (size_t)bc * a.N * 2;
    const double sig = a.sigma[col];
    for (size_t m = (size_t)blockIdx.x * blockDim.x + threadIdx.x; m < a.N; m += (size_t)gridDim.x * blockDim.x) {
        const size_t n = ((m & (((size_t)1 << a.l1) - 1)) << a.l2) + (m >> a.l1);  // time index of memory position m
        cpx x = make_double2(fld[2 * m].x * a.sg, fld[2 * m].y * a.sg), y = make_double2(fld[2 * m + 1].x * a.sg, fld[2 * m + 1].y * a.sg);
        if (sig != 0.0) {
            cpx nx, ny;
            if (a.noise) {
                nx = a.noise[((size_t)b * 2 * a.nfc + col) * a.N + n];
                ny = a.noise[((size_t)b * 2 * a.nfc + a.nfc + col) * a.N + n];
            } else {
                uint32_t r[4];
                philox4x32_10((uint32_t)n, (uint32_t)(n >> 32), (uint32_t)col, (uint32_t)b + a.b0, (uint32_t)a.seed,
                              (uint32_t)(a.seed >> 32), r);
                nx = pmx_cnormal(r[0], r[1]);
                ny = pmx_cnormal(r[2], r[3]);
            }
            if (a.asepol & 1) { x.x += sig * nx.x; x.y += sig * nx.y; }
            if (a.asepol & 2) { y.x += sig * ny.x; y.y += sig * ny.y; }
        }
        fld[2 * m] = pmx_mk2<T2>(x.x, x.y);
        fld[2 * m + 1] = pmx_mk2<T2>(y.x, y.y);
    }
}

extern "C" int pmx_ampliflat_exec_pol(pmx_ctx* c, pmx_devfield* f, double gain, const double* sigma,
                                      const double* noise_host, uint64_t seed, int32_t asepol);
extern "C" int pmx_ampliflat_exec(pmx_ctx* c, pmx_devfield* f, double gain, const double* sigma,
                                  const double* noise_host, uint64_t seed) {
    return pmx_ampliflat_exec_pol(c, f, gain, sigma, noise_host, seed, 3);
}
extern "C" int pmx_ampliflat_exec_pol(pmx_ctx* c, pmx_devfield* f, double gain, const double* sigma,
                                      const double* noise_host, uint64_t seed, int32_t asepol) {
    return pmx_ampliflat_exec_at(c, f, gain, sigma, noise_host, seed, asepol, 0);
}
extern "C" int pmx_ampliflat_exec_at(pmx_ctx* c, pmx_devfield* f, double gain, const double* sigma, const double* noise_host,
                                     uint64_t seed, int32_t asepol, uint64_t realization0) {
    if (!c || !f) return set_err(c, PMX_ERR_INVALID, "pmx_ampliflat_exec: null argument");
    if (!(gain > 0)) return set_err(c, PMX_ERR_INVALID, "gain must be > 0");
    CK(c, cudaSetDevice(c->device));
    AmpParams a;
    memset(&a, 0, sizeof a);
    a.field = f->data;
    a.sg = sqrt(gain);  // ampliflat.m:78
    for (int k = 0; k < f->nfc; ++k) a.sigma[k] = sigma ? sigma[k] : 0.0;
    if (asepol < 1 || asepol > 3) return set_err(c, PMX_ERR_INVALID, "asepol must be 1 (X), 2 (Y) or 3 (both)");
    a.asepol = asepol;
    a.seed = seed;
    a.b0 = (unsigned)realization0;
    a.N = (size_t)f->nfft;
    a.nfc = f->nfc;
    a.batch = f->batch;
    a.l1 = f->log2N1;
    a.l2 = f->log2N2;
    cpx* dn = nullptr;
    if (noise_host) {
        const size_t bytes = (size_t)f->batch * 2 * f->nfc * f->nfft * sizeof(cpx);
        CK(c, cudaMallocAsync(&dn, bytes, c->stream));
        CK(c, cudaMemcpyAsync(dn, noise_host, bytes, cudaMemcpyHostToDevice, c->stream));
        a.noise = dn;
    }
    dim3 g((unsigned)std::min<size_t>((a.N + 255) / 256, 148 * 8), f->batch * f->nfc);
    if (f->precision == PMX_F32)
        pmx_k_ampliflat<float2><<<g, 256, 0, c->stream>>>(a);
    else
        pmx_k_ampliflat<double2><<<g, 256, 0, c->stream>>>(a);
    c->launches++;
    CK(c, cudaGetLastError());
    if (dn) CK(c, cudaFreeAsync(dn, c->stream));
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// create_field('unique') (create_field.m:180-199): sum over the channels of the modulated (and delayed, scaled)
// channel fields, written straight into the resident layout
#define PMX_MUX_MAXCH 64
struct MuxParams {
    const double2* sx;  // [nch][N]
    const double2* sy;  // [nch][N] or null
    void* dst;
    long long ndfn[PMX_MUX_MAXCH], dlx[PMX_MUX_MAXCH], dly[PMX_MUX_MAXCH];
    double scale[PMX_MUX_MAXCH];
    size_t N;
    int nch, lg, l1;
};
template <typename T2>
__global__ void __launch_bounds__(256) pmx_k_mux(const __grid_constant__ MuxParams a) {
    const size_t N = a.N, mask = N - 1;
    const double inv = 2.0 / (double)N;
    T2* dst = reinterpret_cast<T2*>(a.dst);
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        double xr = 0.0, xi = 0.0, yr = 0.0, yi = 0.0;
        for (int ch = 0; ch < a.nch; ++ch) {
            // exp(-2*pi*i*ndfn*n/N): (ndfn*n) mod N in integers (N is a power of two), exact argument for sincospi
            const unsigned long long r = ((unsigned long long)a.ndfn[ch] * (unsigned long long)n) & mask;
            double s, c;
            sincospi(-(double)r * inv, &s, &c);
            const double sc = a.scale[ch];
            const double2 vx = a.sx[(size_t)ch * N + ((n - (size_t)a.dlx[ch]) & mask)];
            const double ar = vx.x * sc, ai = vx.y * sc;
            xr += ar * c - ai * s;
            xi += ar * s + ai * c;
            if (a.sy) {
                const double2 vy = a.sy[(size_t)ch * N + ((n - (size_t)a.dly[ch]) & mask)];
                const double br = vy.x * sc, bi = vy.y * sc;
                yr += br * c - bi * s;
                yi += br * s + bi * c;
            }
        }
        const size_t m = pmx_mem_index(n, a.l1, a.lg - a.l1);
        dst[2 * m] = pmx_mk2<T2>(xr, xi);
        dst[2 * m + 1] = pmx_mk2<T2>(yr, yi);
    }
}

extern "C" int pmx_field_mux(pmx_devfield* f, const pmx_field* sig, int32_t nch, const int64_t* ndfn, const double* scale,
                             const int64_t* delayx, const int64_t* delayy) {
    if (!f) return set_err(nullptr, PMX_ERR_INVALID, "pmx_field_mux: null field");
    pmx_ctx* c = f->ctx;
    if (!sig || !sig->xr || !ndfn) return set_err(c, PMX_ERR_INVALID, "pmx_field_mux: null argument");
    if (f->batch != 1 || f->nfc != 1) return set_err(c, PMX_ERR_INVALID, "pmx_field_mux: the multiplexed field has one column, batch 1");
    if (nch < 1 || nch > PMX_MUX_MAXCH) return set_err(c, PMX_ERR_INVALID, "pmx_field_mux: 1..%d channels, got %d", PMX_MUX_MAXCH, nch);
    const int lg = ilog2_exact(f->nfft);
    if (lg < 0) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_field_mux: nfft must be a power of two");
    CK(c, cudaSetDevice(c->device));
    const size_t N = (size_t)f->nfft, n = (size_t)nch * N;
    MuxParams a;
    memset(&a, 0, sizeof a);
    const bool has_y = sig->layout == PMX_PLANAR ? (sig->yr != nullptr) : (sig->yr != nullptr);
    double2* stage = nullptr;
    CK(c, cudaMallocAsync(&stage, (has_y ? 2 : 1) * n * sizeof(double2), c->stream));
    if (sig->layout == PMX_COMPLEX) {
        CK(c, cudaMemcpyAsync(stage, sig->xr, n * sizeof(double2), cudaMemcpyHostToDevice, c->stream));
        if (has_y) CK(c, cudaMemcpyAsync(stage + n, sig->yr, n * sizeof(double2), cudaMemcpyHostToDevice, c->stream));
    } else if (sig->layout == PMX_PLANAR) {  // interleave on the way: strided 2-D copies of the two planes
        const double* planes[4] = {sig->xr, sig->xi, sig->yr, sig->yi};
        CK(c, cudaMemsetAsync(stage, 0, (has_y ? 2 : 1) * n * sizeof(double2), c->stream));
        for (int k = 0; k < (has_y ? 4 : 2); ++k)
            if (planes[k])
                CK(c, cudaMemcpy2DAsync((double*)(stage + (k / 2) * n) + (k & 1), sizeof(double2), planes[k], sizeof(double),
                                        sizeof(double), n, cudaMemcpyHostToDevice, c->stream));
    } else {
        cudaFreeAsync(stage, c->stream);
        return set_err(c, PMX_ERR_INVALID, "unknown layout %d", sig->layout);
    }
    a.sx = stage;
    a.sy = has_y ? stage + n : nullptr;
    a.dst = f->data;
    a.N = N;
    a.nch = nch;
    a.lg = lg;
    a.l1 = f->log2N1 + f->log2N2 == lg ? f->log2N1 : 0;
    if (f->log2N1 + f->log2N2 != lg) a.lg = 0, a.l1 = 0;  // natural order (sizes without tensor maps)
    for (int k = 0; k < nch; ++k) {
        a.ndfn[k] = (long long)(((ndfn[k] % (int64_t)N) + (int64_t)N) % (int64_t)N);
        a.scale[k] = scale ? scale[k] : 1.0;
        a.dlx[k] = delayx ? (long long)(((delayx[k] % (int64_t)N) + (int64_t)N) % (int64_t)N) : 0;
        a.dly[k] = delayy ? (long long)(((delayy[k] % (int64_t)N) + (int64_t)N) % (int64_t)N) : 0;
    }
    const int blocks = (int)std::min<size_t>((N + 255) / 256, 148 * 16);
    if (f->precision == PMX_F32)
        pmx_k_mux<float2><<<blocks, 256, 0, c->stream>>>(a);
    else
        pmx_k_mux<double2><<<blocks, 256, 0, c->stream>>>(a);
    c->launches++;
    CK(c, cudaGetLastError());
    CK(c, cudaFreeAsync(stage, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));  // the host arrays belong to the caller
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// span loop (ex06_ber.m:110-115): nspan x [ fiber ; ampliflat ] on a resident field
extern "C" int pmx_link_exec(pmx_plan* p, pmx_devfield* f, const pmx_link_desc* l, pmx_fiber_result* out) {
    if (!p || !f || !l) return set_err(p ? p->ctx : nullptr, PMX_ERR_INVALID, "pmx_link_exec: null argument");
    pmx_ctx* c = p->ctx;
    if (l->nspan < 1) return set_err(c, PMX_ERR_INVALID, "pmx_link_exec: nspan must be >= 1");
    const bool redraw = l->db0 || l->theta || l->epsilon;
    if (redraw && !(l->db0 && l->theta && l->epsilon))
        return set_err(c, PMX_ERR_INVALID, "pmx_link_exec: db0, theta and epsilon come together");
    if (redraw && l->plate_sets != 1 && l->plate_sets != p->d.batch)
        return set_err(c, PMX_ERR_INVALID, "pmx_link_exec: plate_sets must be 1 or batch (%d), got %d", p->d.batch, l->plate_sets);
    if (l->gain < 0 || l->gain != l->gain) return set_err(c, PMX_ERR_INVALID, "pmx_link_exec: negative gain");
    const int batch = p->d.batch;
    const size_t per_span = redraw ? (size_t)l->plate_sets * p->d.nplates : 0;
    const size_t noise_span = (size_t)batch * 2 * p->d.nfc * (size_t)p->d.nfft * 2;  // doubles
    std::vector<double> zeros((size_t)p->d.nfc, 0.0);
    for (int k = 0; k < l->nspan; ++k) {
        int rc = PMX_OK;
        if (redraw)
            rc = pmx_plan_set_plates(p, l->plate_sets, l->db0 + k * per_span, l->theta + k * per_span, l->epsilon + k * per_span);
        if (rc != PMX_OK) return rc;
        pmx_fiber_result r = {};
        if (out) {
            r.firstdz = out->firstdz ? out->firstdz + (size_t)k * batch : nullptr;
            r.ncycle = out->ncycle ? out->ncycle + (size_t)k * batch : nullptr;
            r.ntot = out->ntot ? out->ntot + (size_t)k * batch : nullptr;
            r.status = out->status ? out->status + (size_t)k * batch : nullptr;
        }
        rc = pmx_fiber_exec(p, f, &r);
        if (rc != PMX_OK) return rc;
        if (l->gain > 0) {
            rc = pmx_ampliflat_exec_at(c, f, l->gain, l->sigma ? l->sigma : zeros.data(),
                                       l->noise ? l->noise + (size_t)k * noise_span : nullptr,
                                       l->seeds ? l->seeds[k] : (uint64_t)k, l->asepol ? l->asepol : 3, l->realization0);
            if (rc != PMX_OK) return rc;
        }
    }
    return PMX_OK;
}

extern "C" int pmx_link_run(pmx_ctx* c, const pmx_fiber_desc* d, const pmx_link_desc* l, pmx_field* io,
                            pmx_fiber_result* out) {
    if (!c || !d || !l || !io) return set_err(c, PMX_ERR_INVALID, "pmx_link_run: null argument");
    pmx_plan* plan = nullptr;
    pmx_devfield* f = nullptr;
    int rc = pmx_plan_create(c, d, &plan);
    if (rc == PMX_OK) rc = pmx_field_create(c, d->nfft, d->nfc, d->batch, d->precision, &f);
    if (rc == PMX_OK) rc = pmx_field_upload(f, io, 0, d->batch);
    if (rc == PMX_OK) rc = pmx_link_exec(plan, f, l, out);
    if (rc == PMX_OK) rc = pmx_field_download(f, io, 0, d->batch);
    std::string keep = c->error;
    pmx_field_destroy(f);
    pmx_plan_destroy(plan);
    if (rc != PMX_OK) {
        c->error = keep;
        g_tls_error = keep;
    }
    return rc;
}

// ---------------------------------------------------------------------------
// integer error count (ber_estimate.m:118)
__global__ void __launch_bounds__(256) pmx_k_count(const uint8_t* hat, const uint8_t* pat, size_t n,
                                                   unsigned long long* counts) {
    const int b = blockIdx.y;
    const uint8_t* h = hat + (size_t)b * n;
    unsigned int local = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        local += (h[i] != pat[i]);
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(&counts[b], (unsigned long long)local);
}

extern "C" int pmx_count_errors(pmx_ctx* c, const uint8_t* hat, const uint8_t* pat, int64_t n, int32_t batch,
                                int64_t* counts_dev) {
    if (!c || !hat || !pat || !counts_dev || n <= 0 || batch <= 0)
        return set_err(c, PMX_ERR_INVALID, "pmx_count_errors: bad argument");
    if (int rc = check_batch_cols(c, "pmx_count_errors", batch, 1)) return rc;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaMemsetAsync(counts_dev, 0, (size_t)batch * sizeof(int64_t), c->stream));
    dim3 g((unsigned)std::min<size_t>(((size_t)n + 255) / 256, 148 * 4), batch);
    pmx_k_count<<<g, 256, 0, c->stream>>>(hat, pat, (size_t)n, (unsigned long long*)counts_dev);
    c->launches++;
    CK(c, cudaGetLastError());
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// data-aided QPSK decision + bit-error count (see the header)
__global__ void __launch_bounds__(256) pmx_k_qpsk_phase(const cpx* field, const uint8_t* sym, int nsymb, int nt, size_t N,
                                                        int l1, int l2, double* acc /*[batch][2][2]*/) {
    const int b = blockIdx.y;
    const cpx* fld = field + (size_t)b * N * 2;
    double ax = 0, ay = 0, bx = 0, by = 0;  // sum r conj(s) for X (ax,ay) and Y (bx,by)
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < nsymb; k += gridDim.x * blockDim.x) {
        cpx rx, ry;
        ld_sa(fld + pmx_mem_index((size_t)k * nt, l1, l2) * 2, rx, ry);
        const int sx = sym[k], sy = sym[nsymb + k];
        const double sxr = (sx & 1) ? 1.0 : -1.0, sxi = (sx & 2) ? 1.0 : -1.0;
        const double syr = (sy & 1) ? 1.0 : -1.0, syi = (sy & 2) ? 1.0 : -1.0;
        ax += rx.x * sxr + rx.y * sxi;
        ay += rx.y * sxr - rx.x * sxi;
        bx += ry.x * syr + ry.y * syi;
        by += ry.y * syr - ry.x * syi;
    }
    for (int o = 16; o > 0; o >>= 1) {
        ax += __shfl_xor_sync(0xffffffffu, ax, o);
        ay += __shfl_xor_sync(0xffffffffu, ay, o);
        bx += __shfl_xor_sync(0xffffffffu, bx, o);
        by += __shfl_xor_sync(0xffffffffu, by, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&acc[b * 4 + 0], ax);
        atomicAdd(&acc[b * 4 + 1], ay);
        atomicAdd(&acc[b * 4 + 2], bx);
        atomicAdd(&acc[b * 4 + 3], by);
    }
}

__global__ void __launch_bounds__(256) pmx_k_qpsk_count(const cpx* field, const uint8_t* sym, int nsymb, int nt, size_t N,
                                                        int l1, int l2, const double* acc, unsigned long long* counts) {
    const int b = blockIdx.y;
    const cpx* fld = field + (size_t)b * N * 2;
    // e^{-i phi} up to a positive factor: conj of the accumulated correlation
    const double cxr = acc[b * 4 + 0], cxi = -acc[b * 4 + 1], cyr = acc[b * 4 + 2], cyi = -acc[b * 4 + 3];
    unsigned int errs = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < nsymb; k += gridDim.x * blockDim.x) {
        cpx rx, ry;
        ld_sa(fld + pmx_mem_index((size_t)k * nt, l1, l2) * 2, rx, ry);
        const double xr = rx.x * cxr - rx.y * cxi, xi = rx.x * cxi + rx.y * cxr;
        const double yr = ry.x * cyr - ry.y * cyi, yi = ry.x * cyi + ry.y * cyr;
        const int dx = (xr > 0 ? 1 : 0) | (xi > 0 ? 2 : 0), dy = (yr > 0 ? 1 : 0) | (yi > 0 ? 2 : 0);
        errs += __popc((dx ^ sym[k]) & 3) + __popc((dy ^ sym[nsymb + k]) & 3);
    }
    for (int o = 16; o > 0; o >>= 1) errs += __shfl_xor_sync(0xffffffffu, errs, o);
    if ((threadIdx.x & 31) == 0 && errs) atomicAdd(&counts[b], (unsigned long long)errs);
}

extern "C" int pmx_qpsk_count(pmx_ctx* c, pmx_devfield* f, const uint8_t* sym, int32_t nsymb, int32_t nt,
                              int64_t* counts_dev) {
    if (!c || !f || !sym || !counts_dev) return set_err(c, PMX_ERR_INVALID, "pmx_qpsk_count: null argument");
    if (f->nfc != 1) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_qpsk_count: single-column ('unique') fields only");
    if (f->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_qpsk_count: FP64 fields only");
    if ((int64_t)nsymb * nt != f->nfft) return set_err(c, PMX_ERR_INVALID, "pmx_qpsk_count: nsymb*nt must equal nfft");
    CK(c, cudaSetDevice(c->device));
    uint8_t* dsym = nullptr;
    double* acc = nullptr;
    CK(c, cudaMallocAsync(&dsym, 2 * (size_t)nsymb, c->stream));
    CK(c, cudaMallocAsync(&acc, (size_t)f->batch * 4 * sizeof(double), c->stream));
    CK(c, cudaMemcpyAsync(dsym, sym, 2 * (size_t)nsymb, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemsetAsync(acc, 0, (size_t)f->batch * 4 * sizeof(double), c->stream));
    CK(c, cudaMemsetAsync(counts_dev, 0, (size_t)f->batch * sizeof(int64_t), c->stream));
    dim3 g((unsigned)std::min((nsymb + 255) / 256, 148), f->batch);
    pmx_k_qpsk_phase<<<g, 256, 0, c->stream>>>(f->data, dsym, nsymb, nt, (size_t)f->nfft, f->log2N1, f->log2N2, acc);
    pmx_k_qpsk_count<<<g, 256, 0, c->stream>>>(f->data, dsym, nsymb, nt, (size_t)f->nfft, f->log2N1, f->log2N2, acc,
                                                (unsigned long long*)counts_dev);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaFreeAsync(dsym, c->stream));
    CK(c, cudaFreeAsync(acc, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));  // `sym` is a host buffer of the caller
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// Blind DSP core of the reference's coherent receiver on the device (pmx_dsp_count): one complex sample per symbol and
// polarization -> constant-modulus 2x2 FIR polarization demultiplexer (cmaadaptivefilter.m:33-55 inside the
// convergence loop of cmapolardemux, dsp4cohdec.m:353-427) -> carrier frequency and phase by Viterbi & Viterbi
// (vitvit, dsp4cohdec.m:320-345, 241-283) -> decision (samp2pat.m:60-67) -> differential decoding
// (pat_decoder.m:68-82) -> X/Y swap test and error count (ex20_coherent_polmux.m:168-176, ber_estimate.m:118).
// Nothing here knows the waveplates or the transmitted symbols; the caller hands in the decoded reference pattern to
// count against.  The adaptive filter and the scans are sequential in the symbol index by definition: they run as a few
// threads per realization, all realizations of the batch in parallel.  FP64.
#define PMX_DSP_MAX_TAPS 15

// sig[(b*2 + pol)*L + k] = field sample at time index k*nt + shift (circular): the centre of symbol k for a field, the
// centre delayed by the receiver's filters for its currents (fastshift(Irx, round(-delay*NT)), dsp4cohdec.m:167-169);
// divided by `peak` (dsp4cohdec.m:226-227) or, with peak = 0, by sqrt(mean |s|^2 over both polarizations)
#define PMX_DECIM_MAX_TAPS 65
struct DecimTaps {   // the decimator's low-pass FIR (decimate(...,'fir'), dsp4cohdec.m:176-184); n <= 1: none
    int n;
    double h[PMX_DECIM_MAX_TAPS];
};
__global__ void __launch_bounds__(256) pmx_k_dsp_sample(const cpx* field, size_t N, int l1, int l2, int nsymb, int nt,
                                                        long long shift, double peak, double nlr_alpha, int raw, DecimTaps fir,
                                                        cpx* sig) {
    __shared__ double red[256];
    const int b = blockIdx.x;
    const cpx* fld = field + (size_t)b * N * 2;
    cpx* sx = sig + ((size_t)b * 2 + 0) * nsymb;
    cpx* sy = sig + ((size_t)b * 2 + 1) * nsymb;
    auto at = [&](int k) { return pmx_mem_index((size_t)(((long long)k * nt + shift) & (long long)(N - 1)), l1, l2); };
    PMX_ASSERT(shift >= 0 && (size_t)shift < N && (size_t)nsymb * nt == N && at(nsymb - 1) < N);
    auto block_sum = [&](double v) {   // fixed tree: the same result on every run
        __syncthreads();
        red[threadIdx.x] = v;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        return red[0];
    };
    double acc = 0.0;
    for (int k = threadIdx.x; k < nsymb; k += blockDim.x) {
        cpx x, y;
        if (fir.n > 1) {
            // filter(b,1,I) read at the sampling instant plus the filter's group delay (n-1)/2, as decimate compensates
            // it: sum_j b(j) * I(c + (n-1)/2 - j), circular
            const long long c0 = (long long)k * nt + shift + (fir.n - 1) / 2;
            double xr = 0.0, xi = 0.0, yr = 0.0, yi = 0.0;
            for (int j = 0; j < fir.n; ++j) {
                const size_t m = pmx_mem_index((size_t)((c0 - j) & (long long)(N - 1)), l1, l2);
                const cpx u = fld[2 * m], v = fld[2 * m + 1];
                xr += fir.h[j] * u.x;
                xi += fir.h[j] * u.y;
                yr += fir.h[j] * v.x;
                yi += fir.h[j] * v.y;
            }
            x = make_double2(xr, xi);
            y = make_double2(yr, yi);
        } else {
            const size_t m = at(k);
            x = fld[2 * m];
            y = fld[2 * m + 1];
        }
        sx[k] = x;
        sy[k] = y;
        acc += x.x * x.x + x.y * x.y + y.x * y.x + y.y * y.y;
    }
    if (raw) return;   // the samples as they are: a dispersion-compensating filter comes first (dsp4cohdec.m:198-210)
    if (nlr_alpha != 0.0) {
        // NLRotation (dsp4cohdec.m:308-315), before the normalisation as in the reference: Phases + alpha*(Asquare - mean(Asquare)),
        // Asquare = |s_x|^2 + |s_y|^2 of the symbol
        double asq = 0.0;
        for (int k = threadIdx.x; k < nsymb; k += blockDim.x) {
            const double ax = hypot(sx[k].x, sx[k].y), ay = hypot(sy[k].x, sy[k].y);
            asq += ax * ax + ay * ay;
        }
        const double mean = block_sum(asq) / (double)nsymb;
        for (int k = threadIdx.x; k < nsymb; k += blockDim.x) {
            const double ax = hypot(sx[k].x, sx[k].y), ay = hypot(sy[k].x, sy[k].y);
            const double dp = nlr_alpha * ((ax * ax + ay * ay) - mean);
            double sn, cs;
            sincos(atan2(sx[k].y, sx[k].x) + dp, &sn, &cs);
            sx[k] = make_double2(ax * cs, ax * sn);
            sincos(atan2(sy[k].y, sy[k].x) + dp, &sn, &cs);
            sy[k] = make_double2(ay * cs, ay * sn);
        }
    }
    if (peak > 0.0) {   // Signals/peak: a division in the reference (dsp4cohdec.m:226-227)
        for (int k = threadIdx.x; k < nsymb; k += blockDim.x) {
            sx[k] = make_double2(sx[k].x / peak, sx[k].y / peak);
            sy[k] = make_double2(sy[k].x / peak, sy[k].y / peak);
        }
    } else {
        const double inv = 1.0 / sqrt(block_sum(acc) / (2.0 * nsymb));
        for (int k = threadIdx.x; k < nsymb; k += blockDim.x) {
            sx[k] = make_double2(sx[k].x * inv, sx[k].y * inv);
            sy[k] = make_double2(sy[k].x * inv, sy[k].y * inv);
        }
    }
}

// cmapolardemux: four threads per realization, one per (filter, input column): thread (f, p) keeps the taps h_f(:, p),
// forms the column sum sum_j xx(k+j, p) * h_f(j, p) in the interpreter's order (products and sums rounded separately,
// j ascending), the two column sums of a filter are added through a shuffle (column 0 + column 1, as sum(sum(.)) does),
// and each thread updates its own taps.  The same arithmetic as one thread per filter, half the dependent chain.
// (TAPS is a template parameter so that the taps and the input window live in registers)
template <int TAPS>
__global__ void __launch_bounds__(32) pmx_k_dsp_cma(const cpx* sig, cpx* out, int L, double mu, double r1, double r2,
                                                    double phizero, int repetitions, int* passes) {
    constexpr int taps = TAPS;
    const int b = blockIdx.x, lane = threadIdx.x;
    if (lane >= 4) return;
    const int f = lane >> 1, p = lane & 1;          // filter, input column
    const cpx* xin = sig + ((size_t)b * 2 + p) * L;
    cpx* y = out + ((size_t)b * 2 + f) * L;
    const int half = taps / 2;
    const double R = f == 0 ? r1 : r2;
    cpx h[TAPS], ho[TAPS];
#pragma unroll
    for (int j = 0; j < taps; ++j) h[j] = make_double2(0.0, 0.0);
    // hzero(halftaps+1,:,:) = M = [cos sin; -sin cos]; filter f takes row f, this thread its entry p
    h[half] = make_double2(f == 0 ? (p == 0 ? cos(phizero) : sin(phizero)) : (p == 0 ? -sin(phizero) : cos(phizero)), 0.0);
    int c = 1;
    bool conv = false;
    while (!conv && c < repetitions) {
#pragma unroll
        for (int j = 0; j < taps; ++j) ho[j] = h[j];
        cpx w[TAPS];   // sliding window extendedx(k .. k+taps-1) = x(k - half .. k + half) circularly
#pragma unroll
        for (int j = 1; j < taps; ++j) {
            int i = j - 1 - half;
            i = i < 0 ? i + L : i;
            w[j] = xin[i % L];
        }
        for (int k = 0; k < L; ++k) {
            cpx s = make_double2(0.0, 0.0);
#pragma unroll
            for (int j = 0; j + 1 < taps; ++j) w[j] = w[j + 1];
            {
                int i = k + half;
                w[taps - 1] = xin[i >= L ? i - L : i];
            }
#pragma unroll
            for (int j = 0; j < taps; ++j) {
                const cpx q = make_double2(__dadd_rn(__dmul_rn(w[j].x, h[j].x), -__dmul_rn(w[j].y, h[j].y)),
                                           __dadd_rn(__dmul_rn(w[j].x, h[j].y), __dmul_rn(w[j].y, h[j].x)));
                s = make_double2(__dadd_rn(s.x, q.x), __dadd_rn(s.y, q.y));
            }
            const double ox = __shfl_xor_sync(0xfu, s.x, 1), oy = __shfl_xor_sync(0xfu, s.y, 1);
            const cpx yk = p == 0 ? make_double2(__dadd_rn(s.x, ox), __dadd_rn(s.y, oy))     // column 0 + column 1
                                  : make_double2(__dadd_rn(ox, s.x), __dadd_rn(oy, s.y));
            if (p == 0) y[k] = yk;
            // incr = mu .* errorfuncma(Y, R) .* conj(xx):  E = Y .* (R - abs(Y).^2)
            const double a = hypot(yk.x, yk.y), g = __dadd_rn(R, -__dmul_rn(a, a));
            const cpx e = make_double2(__dmul_rn(mu, __dmul_rn(yk.x, g)), __dmul_rn(mu, __dmul_rn(yk.y, g)));
#pragma unroll
            for (int j = 0; j < taps; ++j)
                h[j] = make_double2(__dadd_rn(h[j].x, __dadd_rn(__dmul_rn(e.x, w[j].x), __dmul_rn(e.y, w[j].y))),
                                    __dadd_rn(h[j].y, __dadd_rn(__dmul_rn(e.y, w[j].x), -__dmul_rn(e.x, w[j].y))));
        }
        // (the reference keeps the old taps when the new ones are all zero: any(any(h_new)), dsp4cohdec.m:404-407)
        double moved = 0.0, nz = 0.0;
#pragma unroll
        for (int j = 0; j < taps; ++j) {
            moved = fmax(moved, hypot(ho[j].x - h[j].x, ho[j].y - h[j].y));
            nz = fmax(nz, fmax(fabs(h[j].x), fabs(h[j].y)));
        }
        for (int o = 1; o < 4; o <<= 1) {   // over both filters and both columns
            moved = fmax(moved, __shfl_xor_sync(0xfu, moved, o));
            nz = fmax(nz, __shfl_xor_sync(0xfu, nz, o));
        }
        if (nz == 0.0) {
#pragma unroll
            for (int j = 0; j < taps; ++j) h[j] = ho[j];
            moved = 0.0;
        }
        if (moved < 5e-5) conv = true;
        ++c;
    }
    if (lane == 0 && passes) passes[b] = c - 1;
}

// The same filter with one lane per (filter, input column, tap) -- 4*TAPS <= 32 lanes of one warp: every lane forms ONE
// product and updates ONE tap, the products of a (filter, column) group are fetched by shuffles and added in the
// interpreter's order (tap index ascending, then column 0 + column 1) by all its lanes alike.  A quarter of the issued
// FP64 instructions of the four-lane form (every warp instruction costs the same whether 4 or 28 lanes are active).
// |Y|^2 is taken as re^2 + im^2 (the reference squares abs(Y): the two differ in the last bits only).
template <int TAPS>
__global__ void __launch_bounds__(32) pmx_k_dsp_cma_w(const cpx* sig, cpx* out, int L, double mu, double r1, double r2,
                                                      double phizero, int repetitions, int* passes) {
    static_assert(4 * TAPS <= 32, "one warp");
    constexpr int taps = TAPS, NL = 4 * TAPS;
    const int b = blockIdx.x, lane = threadIdx.x;
    const bool act = lane < NL;
    const int l = act ? lane : 0;                      // (idle lanes shadow lane 0 and never store)
    const int f = l / (2 * taps), p = (l / taps) & 1, j = l % taps;
    const unsigned full = 0xffffffffu;
    const cpx* xin = sig + ((size_t)b * 2 + p) * L;
    cpx* y = out + ((size_t)b * 2 + f) * L;
    const int half = taps / 2, base = l - j, other = base + (p ? -taps : taps);
    const double R = f == 0 ? r1 : r2;
    // hzero(halftaps+1,:,:) = M = [cos sin; -sin cos]; filter f takes row f, column p its entry
    cpx h = make_double2(j == half ? (f == 0 ? (p == 0 ? cos(phizero) : sin(phizero)) : (p == 0 ? -sin(phizero) : cos(phizero))) : 0.0, 0.0);
    int c = 1;
    bool conv = false;
    auto at = [&](int i) { i %= L; return xin[i < 0 ? i + L : i]; };
    while (!conv && c < repetitions) {
        const cpx ho = h;
        // window of symbol k: w_j = x(k - half + j), circular; lane j holds w_j of symbol k - 1 before the shift
        cpx w = at(-1 - half + j);
        cpx nxt = at(half);                            // the sample entering at k = 0 (lane taps-1 uses it)
        for (int k = 0; k < L; ++k) {
            PMX_ASSERT(base >= 0 && base + taps <= NL && other >= 0 && other + taps <= NL && (base % taps) == 0);
            const double wx = __shfl_down_sync(full, w.x, 1), wy = __shfl_down_sync(full, w.y, 1);
            w = (j == taps - 1) ? nxt : make_double2(wx, wy);
            {
                const int i = k + 1 + half;
                nxt = xin[i >= L ? i - L : i];         // for the next symbol: its latency hides behind this one
            }
            const cpx q = make_double2(__dadd_rn(__dmul_rn(w.x, h.x), -__dmul_rn(w.y, h.y)),
                                       __dadd_rn(__dmul_rn(w.x, h.y), __dmul_rn(w.y, h.x)));
            cpx sacc = make_double2(0.0, 0.0);
#pragma unroll
            for (int jj = 0; jj < taps; ++jj)
                sacc = make_double2(__dadd_rn(sacc.x, __shfl_sync(full, q.x, base + jj)), __dadd_rn(sacc.y, __shfl_sync(full, q.y, base + jj)));
            const double ox = __shfl_sync(full, sacc.x, other), oy = __shfl_sync(full, sacc.y, other);
            const cpx yk = p == 0 ? make_double2(__dadd_rn(sacc.x, ox), __dadd_rn(sacc.y, oy))     // column 0 + column 1
                                  : make_double2(__dadd_rn(ox, sacc.x), __dadd_rn(oy, sacc.y));
            if (act && p == 0 && j == 0) y[k] = yk;
            // incr = mu .* errorfuncma(Y, R) .* conj(xx):  E = Y .* (R - abs(Y).^2)
            const double g = __dadd_rn(R, -__dadd_rn(__dmul_rn(yk.x, yk.x), __dmul_rn(yk.y, yk.y)));
            const cpx e = make_double2(__dmul_rn(mu, __dmul_rn(yk.x, g)), __dmul_rn(mu, __dmul_rn(yk.y, g)));
            h = make_double2(__dadd_rn(h.x, __dadd_rn(__dmul_rn(e.x, w.x), __dmul_rn(e.y, w.y))),
                             __dadd_rn(h.y, __dadd_rn(__dmul_rn(e.y, w.x), -__dmul_rn(e.x, w.y))));
        }
        // (the reference keeps the old taps when the new ones are all zero: any(any(h_new)), dsp4cohdec.m:404-407)
        double moved = act ? hypot(ho.x - h.x, ho.y - h.y) : 0.0, nz = act ? fmax(fabs(h.x), fabs(h.y)) : 0.0;
        for (int o = 16; o > 0; o >>= 1) {   // over both filters, both columns and all taps
            moved = fmax(moved, __shfl_xor_sync(full, moved, o));
            nz = fmax(nz, __shfl_xor_sync(full, nz, o));
        }
        if (nz == 0.0) {
            h = ho;
            moved = 0.0;
        }
        if (moved < 5e-5) conv = true;
        ++c;
    }
    if (lane == 0 && passes) passes[b] = c - 1;
}

// easipolardemux (dsp4cohdec.m:428-482) around easiadaptivefilter.m:28-61 for its single 2x2 tap: Y = H*x, then
// H <- (I - mu*E(Y))*H with errorfun's E (:55-61; its products are a*b as written there).  Sequential in the symbol index;
// one thread per realization, products and sums rounded separately as the interpreter does.
struct dc2 { double x, y; };
__device__ __forceinline__ double2 pmx_cm(double2 a, double2 b) {   // a*b, no contraction
    return make_double2(__dadd_rn(__dmul_rn(a.x, b.x), -__dmul_rn(a.y, b.y)), __dadd_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x)));
}
__device__ __forceinline__ double2 pmx_cdiv(double2 a, double2 b) {   // a/b
    const double d = __dadd_rn(__dmul_rn(b.x, b.x), __dmul_rn(b.y, b.y));
    return make_double2(__ddiv_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), d),
                        __ddiv_rn(__dadd_rn(__dmul_rn(a.y, b.x), -__dmul_rn(a.x, b.y)), d));
}
__global__ void __launch_bounds__(32) pmx_k_dsp_easi(const cpx* sig, cpx* out, int L, double mu, double phizero, int repetitions,
                                                     int* passes) {
    const int b = blockIdx.x;
    if (threadIdx.x != 0) return;
    const cpx* x1 = sig + ((size_t)b * 2 + 0) * L;
    const cpx* x2 = sig + ((size_t)b * 2 + 1) * L;
    cpx* y1o = out + ((size_t)b * 2 + 0) * L;
    cpx* y2o = out + ((size_t)b * 2 + 1) * L;
    // hzero(1,:,:) = M = [cos sin; -sin cos]; h1 = its first row, h2 its second
    double2 h11 = make_double2(cos(phizero), 0.0), h12 = make_double2(sin(phizero), 0.0);
    double2 h21 = make_double2(-sin(phizero), 0.0), h22 = make_double2(cos(phizero), 0.0);
    int c = 1;
    bool conv = false;
    while (!conv && c < repetitions) {
        const double2 o11 = h11, o12 = h12, o21 = h21, o22 = h22;
        double2 nx1 = x1[0], nx2 = x2[0];
        for (int k = 0; k < L; ++k) {
            const double2 a1 = nx1, a2 = nx2;
            if (k + 1 < L) {
                nx1 = x1[k + 1];
                nx2 = x2[k + 1];
            }
            const double2 p1 = pmx_cm(a1, h11), p2 = pmx_cm(a2, h12), q1 = pmx_cm(a1, h21), q2 = pmx_cm(a2, h22);
            const double2 ya = make_double2(__dadd_rn(p1.x, p2.x), __dadd_rn(p1.y, p2.y));
            const double2 yb = make_double2(__dadd_rn(q1.x, q2.x), __dadd_rn(q1.y, q2.y));
            y1o[k] = ya;
            y2o[k] = yb;
            const double aa = sqrt(__dadd_rn(__dmul_rn(ya.x, ya.x), __dmul_rn(ya.y, ya.y)));
            const double ab = sqrt(__dadd_rn(__dmul_rn(yb.x, yb.x), __dmul_rn(yb.y, yb.y)));
            const double na = __dmul_rn(aa, aa), nb = __dmul_rn(ab, ab);
            const double d1 = __dadd_rn(1.0, __dmul_rn(mu, __dadd_rn(na, nb)));
            const double2 d2 = make_double2(__dadd_rn(1.0, __dmul_rn(mu, __dadd_rn(__dmul_rn(ya.x, aa), __dmul_rn(yb.x, ab)))),
                                            __dmul_rn(mu, __dadd_rn(__dmul_rn(ya.y, aa), __dmul_rn(yb.y, ab))));
            const double2 pab = pmx_cm(ya, yb);
            const double2 t = make_double2(__ddiv_rn(pab.x, d1), __ddiv_rn(pab.y, d1));
            const double dn = __dadd_rn(na, -nb);
            const double2 u = pmx_cdiv(make_double2(__dmul_rn(pab.x, dn), __dmul_rn(pab.y, dn)), d2);
            const double e11 = __ddiv_rn(__dadd_rn(na, -1.0), d1), e22 = __ddiv_rn(__dadd_rn(nb, -1.0), d1);
            const double2 e12 = make_double2(__dadd_rn(t.x, u.x), __dadd_rn(t.y, u.y));
            const double2 e21 = make_double2(__dadd_rn(t.x, -u.x), __dadd_rn(t.y, -u.y));
            // h11 = (1-mu*E11)*h1(1) + (-mu*E12)*h2(1), ... (easiadaptivefilter.m:40-43)
            const double g1 = __dadd_rn(1.0, -__dmul_rn(mu, e11)), g2 = __dadd_rn(1.0, -__dmul_rn(mu, e22));
            const double2 m12 = make_double2(-__dmul_rn(mu, e12.x), -__dmul_rn(mu, e12.y));
            const double2 m21 = make_double2(-__dmul_rn(mu, e21.x), -__dmul_rn(mu, e21.y));
            const double2 r1 = pmx_cm(m12, h21), r2 = pmx_cm(m12, h22), r3 = pmx_cm(m21, h11), r4 = pmx_cm(m21, h12);
            const double2 n11 = make_double2(__dadd_rn(__dmul_rn(g1, h11.x), r1.x), __dadd_rn(__dmul_rn(g1, h11.y), r1.y));
            const double2 n12 = make_double2(__dadd_rn(__dmul_rn(g1, h12.x), r2.x), __dadd_rn(__dmul_rn(g1, h12.y), r2.y));
            const double2 n21 = make_double2(__dadd_rn(r3.x, __dmul_rn(g2, h21.x)), __dadd_rn(r3.y, __dmul_rn(g2, h21.y)));
            const double2 n22 = make_double2(__dadd_rn(r4.x, __dmul_rn(g2, h22.x)), __dadd_rn(r4.y, __dmul_rn(g2, h22.y)));
            h11 = n11;
            h12 = n12;
            h21 = n21;
            h22 = n22;
        }
        const double nz = fmax(fmax(fmax(fabs(h11.x), fabs(h11.y)), fmax(fabs(h12.x), fabs(h12.y))),
                               fmax(fmax(fabs(h21.x), fabs(h21.y)), fmax(fabs(h22.x), fabs(h22.y))));
        if (nz == 0.0) {   // any(any(h_new)): all-zero taps are not taken over (dsp4cohdec.m:470-473)
            h11 = o11;
            h12 = o12;
            h21 = o21;
            h22 = o22;
        }
        const double moved = fmax(fmax(hypot(o11.x - h11.x, o11.y - h11.y), hypot(o12.x - h12.x, o12.y - h12.y)),
                                  fmax(hypot(o21.x - h21.x, o21.y - h21.y), hypot(o22.x - h22.x, o22.y - h22.y)));
        if (moved < 5e-5) conv = true;
        ++c;
    }
    if (passes) passes[b] = c - 1;
}

// Carrier recovery of one (realization, polarization) stream by one CTA: frequency estimate (navg = freqavg) ->
// cumulated phase omega, cleaned to match the circularity -> demodulation -> Viterbi & Viterbi phase (navg = phasavg,
// unwrapped) -> phases = angle(s .* fastexp(-omega - theta + pi/4)).  w1, w2: complex scratch of L entries, om: real.
// Every thread owns a contiguous chunk of the symbols; the two running quantities (cumsum of the frequency estimate,
// unwrap of the phase) are block-wide scans: the unwrap as an exact integer count of 2*pi jumps.
__device__ __forceinline__ cpx pmx_cpow_int(cpx a, int n) {   // a^n, n >= 1, by repeated multiplication
    cpx r = a;
    for (int i = 1; i < n; ++i) r = make_double2(r.x * a.x - r.y * a.y, r.x * a.y + r.y * a.x);
    return r;
}
// out(n) = mean(in(n-N+1 .. n)), N = 2k+1, circular, for n in [n0, n1): a running sum seeded from its own N terms
__device__ __forceinline__ void pmx_circ_avg_chunk(const cpx* in, cpx* out, int L, int k, int n0, int n1) {
    if (n0 >= n1) return;
    const int N = 2 * k + 1;
    const double invN = 1.0 / N;
    cpx run = make_double2(0.0, 0.0);
    for (int j = 0; j < N; ++j) {
        int i = (n0 - j) % L;
        i = i < 0 ? i + L : i;
        run.x += in[i].x;
        run.y += in[i].y;
    }
    out[n0] = make_double2(run.x * invN, run.y * invN);
    for (int n = n0 + 1; n < n1; ++n) {
        int i0 = (n - N) % L;
        i0 = i0 < 0 ? i0 + L : i0;
        run.x += in[n].x - in[i0].x;
        run.y += in[n].y - in[i0].y;
        out[n] = make_double2(run.x * invN, run.y * invN);
    }
}
// exclusive scan of one value per thread over the CTA (blockDim.x <= 1024); every thread gets its offset and the total
template <typename T>
__device__ __forceinline__ T pmx_block_exscan(T v, T* sh /*[32]*/, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T u = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += u;
    }
    __syncthreads();   // sh may still be read from a previous scan
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    T woff = 0, tot = 0;
    for (int w = 0; w < nwarp; ++w) {
        if (w < warp) woff += sh[w];
        tot += sh[w];
    }
    *total = tot;
    return woff + inc - v;
}
#define PMX_CARRIER_THREADS 1024
__global__ void __launch_bounds__(PMX_CARRIER_THREADS) pmx_k_dsp_carrier(const cpx* sig, cpx* w1, cpx* w2, double* om,
                                                                         double* phases, int L, int M, int freqavg, int phasavg,
                                                                         int P, double offset) {
    __shared__ double shd[32];
    __shared__ long long shl[32];
    __shared__ double s_o0, s_oe;
    const int s_id = blockIdx.x;   // one (realization, polarization) stream per CTA
    const cpx* s = sig + (size_t)s_id * L;
    cpx* a = w1 + (size_t)s_id * L;
    cpx* bq = w2 + (size_t)s_id * L;
    double* omg = om + (size_t)s_id * L;
    double* ph = phases + (size_t)s_id * L;
    const double TWO_PI = 6.283185307179586476925286766559, PI = 3.14159265358979323846;
    const int chunk = (L + blockDim.x - 1) / blockDim.x;
    const int n0 = min(L, (int)threadIdx.x * chunk), n1 = min(L, n0 + chunk);
    PMX_ASSERT(n0 <= n1 && n1 <= L && (threadIdx.x + 1 < blockDim.x || n1 == L));
    if (freqavg > 0) {
        for (int n = threadIdx.x; n < L; n += blockDim.x) {   // (s .* conj(fastshift(s,1))).^M
            const cpx p = s[n], q = s[n == 0 ? L - 1 : n - 1];
            a[n] = pmx_cpow_int(make_double2(p.x * q.x + p.y * q.y, p.y * q.x - p.x * q.y), M);
        }
        __syncthreads();
        pmx_circ_avg_chunk(a, bq, L, freqavg, n0, n1);
        double acc = 0.0;
        for (int n = n0; n < n1; ++n) {   // omega = cumsum(angle(.)/M): local sums, then the offsets of the chunks
            acc += atan2(bq[n].y, bq[n].x) / M;
            omg[n] = acc;
        }
        double total;
        const double off = pmx_block_exscan<double>(acc, shd, &total);
        for (int n = n0; n < n1; ++n) omg[n] += off;
        __syncthreads();
        if (threadIdx.x == 0) {
            s_o0 = omg[0];
            s_oe = omg[L - 1];
        }
        __syncthreads();
        const double o0 = s_o0, oe = s_oe;
        const double closest = o0 + rint((oe - o0) / 2 / PI) * 2 * PI;
        const double ratio = closest / oe;
        for (int n = threadIdx.x; n < L; n += blockDim.x) omg[n] = (omg[n] - o0) * ratio + o0;
    } else {
        for (int n = threadIdx.x; n < L; n += blockDim.x) omg[n] = 0.0;
    }
    __syncthreads();
    for (int n = threadIdx.x; n < L; n += blockDim.x) {   // demodulate, then abs(s).^P .* fastexp(angle(s.^M))  (or s.^P when P == M)
        double sn, cs;
        sincos(-omg[n], &sn, &cs);
        const cpx d = make_double2(s[n].x * cs - s[n].y * sn, s[n].x * sn + s[n].y * cs);
        const cpx dm = pmx_cpow_int(d, M);
        if (P == M) {
            a[n] = dm;
        } else {
            const double mag = pow(hypot(d.x, d.y), (double)P), ang = atan2(dm.y, dm.x);
            sincos(ang, &sn, &cs);
            a[n] = make_double2(mag * cs, mag * sn);
        }
    }
    __syncthreads();
    const cpx* sm = a;
    if (phasavg > 0) {
        pmx_circ_avg_chunk(a, bq, L, phasavg, n0, n1);
        sm = bq;
        __syncthreads();
    }
    // theta = unwrap(angle(.))/M: unwrap(n) = angle(n) - 2*pi*(number of upward minus downward jumps up to n), jumps where
    // the step between neighbours exceeds pi (numpy.unwrap / the interpreter's unwrap)
    long long local = 0;
    for (int n = n0; n < n1; ++n) {
        if (n == 0) continue;
        const double dd = atan2(sm[n].y, sm[n].x) - atan2(sm[n - 1].y, sm[n - 1].x);
        if (fabs(dd) > PI) local += (long long)rint(dd / TWO_PI);
    }
    long long totl;
    long long jumps = pmx_block_exscan<long long>(local, shl, &totl);
    for (int n = n0; n < n1; ++n) {   // phases = angle(s .* fastexp(-omega - theta + offset))
        const double ang = atan2(sm[n].y, sm[n].x);
        if (n > 0) {
            const double dd = ang - atan2(sm[n - 1].y, sm[n - 1].x);
            if (fabs(dd) > PI) jumps += (long long)rint(dd / TWO_PI);
        }
        const double unw = ang - TWO_PI * (double)jumps;
        const double arg = -omg[n] - unw / M + offset;
        double sn, cs;
        sincos(arg, &sn, &cs);
        ph[n] = atan2(s[n].x * sn + s[n].y * cs, s[n].x * cs - s[n].y * sn);
    }
}

// decision + differential decoding + the four error sums of the swap test: acc[b*4 + {xx, xy, yy, yx}]
__device__ __forceinline__ int pmx_star_of(double phase) {   // samp2pat 'coherent' bits -> pat2stars (binary) quadrant
    const int first = fabs(phase) <= 1.57079632679489661923 ? 1 : 0, second = phase > 0 ? 1 : 0;
    // [0 0] -> 1 (0), [0 1] -> i (1), [1 1] -> -1 (2), [1 0] -> -i (3): index = multiples of pi/2
    return first == 0 ? (second == 0 ? 0 : 1) : (second == 1 ? 2 : 3);
}
__global__ void __launch_bounds__(256) pmx_k_dsp_decide(const double* phases, const uint8_t* ref, int L, unsigned long long* acc) {
    const int b = blockIdx.y;
    const double* px = phases + (size_t)b * 2 * L;
    const double* py = px + L;
    unsigned long long e[4] = {0, 0, 0, 0};
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < L; k += gridDim.x * blockDim.x) {
        const int km = k == 0 ? L - 1 : k - 1;
        int bits[2][2];
        for (int p = 0; p < 2; ++p) {
            const double* q = p ? py : px;
            // stars_r = conj(stars_t(k)) .* stars_t(k-1): quadrant difference; stars2pat then inverts both bits
            const int d = (pmx_star_of(q[km]) - pmx_star_of(q[k])) & 3;
            const int m0 = (d == 2 || d == 3) ? 1 : 0, m1 = (d == 1 || d == 2) ? 1 : 0;
            bits[p][0] = 1 - m0;
            bits[p][1] = 1 - m1;
        }
        const uint8_t* r = ref + (size_t)k * 4;   // decoded reference pattern [x1 x2 y1 y2]
        e[0] += (r[0] != bits[0][0]) + (r[1] != bits[0][1]);
        e[1] += (r[0] != bits[1][0]) + (r[1] != bits[1][1]);
        e[2] += (r[2] != bits[1][0]) + (r[3] != bits[1][1]);
        e[3] += (r[2] != bits[0][0]) + (r[3] != bits[0][1]);
    }
    for (int i = 0; i < 4; ++i) {
        for (int o = 16; o > 0; o >>= 1) e[i] += __shfl_xor_sync(0xffffffffu, e[i], o);
        if ((threadIdx.x & 31) == 0 && e[i]) atomicAdd(&acc[(size_t)b * 4 + i], e[i]);
    }
}
__global__ void pmx_k_dsp_final(const unsigned long long* acc, int batch, unsigned long long* counts) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    const unsigned long long xx = acc[b * 4], xy = acc[b * 4 + 1], yy = acc[b * 4 + 2], yx = acc[b * 4 + 3];
    counts[b] = (xy < xx) ? xy + yx : xx + yy;   // ex20_coherent_polmux.m:168-173: swap when Y decodes the X pattern better
}

// |s| of every sample (Amplitudes = abs(Signals), dsp4cohdec.m:286)
__global__ void __launch_bounds__(256) pmx_k_dsp_abs(const cpx* s, size_t n, double* out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = hypot(s[i].x, s[i].y);
}

// the two sampled streams of a realization as the two polarizations of a field of L samples (field layout)
__global__ void __launch_bounds__(256) pmx_k_dsp_pack(const cpx* sig, int L, int l1, int l2, cpx* field) {
    const int b = blockIdx.y;
    const cpx* sx = sig + ((size_t)b * 2 + 0) * L;
    const cpx* sy = sig + ((size_t)b * 2 + 1) * L;
    cpx* fld = field + (size_t)b * L * 2;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < L; k += gridDim.x * blockDim.x) {
        const size_t m = pmx_mem_index((size_t)k, l1, l2);
        fld[2 * m] = sx[k];
        fld[2 * m + 1] = sy[k];
    }
}

// sampler, polarization demultiplexer, carrier recovery; then either the decision + count (ref_patmat, counts_dev) or the
// phases / amplitudes handed back to the host (phases, amps: [batch][2][nsymb])
static int dsp_core(pmx_ctx* c, pmx_devfield* f, const pmx_dsp_desc* d, const uint8_t* ref_patmat, int64_t* counts_dev,
                    double* phases, double* amps, int32_t* passes_host, const char* who) {
    if (f->nfc != 1) return set_err(c, PMX_ERR_UNSUPPORTED, "%s: single-column ('unique') fields only", who);
    if (f->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "%s: FP64 fields only", who);
    if ((int64_t)d->nsymb * d->nt != f->nfft) return set_err(c, PMX_ERR_INVALID, "%s: nsymb*nt must equal nfft", who);
    if (d->taps < 1 || d->taps > PMX_DSP_MAX_TAPS || !(d->taps & 1))
        return set_err(c, PMX_ERR_INVALID, "%s: taps must be odd, 1..%d", who, PMX_DSP_MAX_TAPS);
    if (d->modorder != 2) return set_err(c, PMX_ERR_UNSUPPORTED, "%s: QPSK (modorder 2) only", who);
    if (!(d->mu > 0)) return set_err(c, PMX_ERR_INVALID, "%s: mu must be > 0", who);
    CK(c, cudaSetDevice(c->device));
    const int L = d->nsymb, B = f->batch;
    const size_t n = (size_t)B * 2 * L;
    cpx *sig = nullptr, *y = nullptr, *w1 = nullptr, *w2 = nullptr;
    double *om = nullptr, *ph = nullptr;
    uint8_t* dref = nullptr;
    unsigned long long* acc = nullptr;
    int* dpass = nullptr;
    CK(c, cudaMallocAsync(&sig, n * sizeof(cpx), c->stream));
    CK(c, cudaMallocAsync(&y, n * sizeof(cpx), c->stream));
    CK(c, cudaMallocAsync(&w1, n * sizeof(cpx), c->stream));
    CK(c, cudaMallocAsync(&w2, n * sizeof(cpx), c->stream));
    CK(c, cudaMallocAsync(&om, n * sizeof(double), c->stream));
    CK(c, cudaMallocAsync(&ph, n * sizeof(double), c->stream));
    CK(c, cudaMallocAsync(&dref, (size_t)L * 4, c->stream));
    CK(c, cudaMallocAsync(&acc, (size_t)B * 4 * sizeof(unsigned long long), c->stream));
    CK(c, cudaMallocAsync(&dpass, (size_t)B * sizeof(int), c->stream));
    if (ref_patmat) CK(c, cudaMemcpyAsync(dref, ref_patmat, (size_t)L * 4, cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemsetAsync(acc, 0, (size_t)B * 4 * sizeof(unsigned long long), c->stream));
    CK(c, cudaMemsetAsync(dpass, 0, (size_t)B * sizeof(int), c->stream));
    {
        const long long N = (long long)f->nfft;
        const long long sh = (((long long)d->sample_shift % N) + N) % N;
        DecimTaps fir;
        fir.n = 0;
        if (d->decim_ntaps > 1 && d->decim_taps) {
            if (d->decim_ntaps > PMX_DECIM_MAX_TAPS || !(d->decim_ntaps & 1)) {
                for (void* q : {(void*)sig, (void*)y, (void*)w1, (void*)w2, (void*)om, (void*)ph, (void*)dref, (void*)acc, (void*)dpass})
                    cudaFreeAsync(q, c->stream);
                return set_err(c, PMX_ERR_INVALID, "%s: decim_ntaps must be odd, <= %d", who, PMX_DECIM_MAX_TAPS);
            }
            fir.n = d->decim_ntaps;
            for (int j = 0; j < fir.n; ++j) fir.h[j] = d->decim_taps[j];
        }
        pmx_k_dsp_sample<<<B, 256, 0, c->stream>>>(f->data, (size_t)f->nfft, f->log2N1, f->log2N2, L, d->nt, sh, d->peak, d->nlr_alpha,
                                                  d->dcf_h ? 1 : 0, fir, sig);
    }
    if (d->dcf_h) {
        // p.applydcf: Signals = ifft(fft(Signals) .* Hfilt) on the sampled signals (dsp4cohdec.m:198-210), before the
        // non-linear rotation and the normalisation.  The two streams of a realization become the polarizations of a field
        // of nsymb samples, a filter plan does the rest; the sampler then runs again over that field (one sample per symbol).
        pmx_devfield* tf = nullptr;
        pmx_plan* fp = nullptr;
        int rc = pmx_field_create(c, L, 1, B, PMX_F64, &tf);
        if (rc == PMX_OK) rc = pmx_filter_create(c, L, 1, B, PMX_F64, d->dcf_h, 1, &fp);
        if (rc == PMX_OK) {
            pmx_k_dsp_pack<<<dim3((unsigned)std::min((L + 255) / 256, 64), B), 256, 0, c->stream>>>(sig, L, tf->log2N1, tf->log2N2, tf->data);
            c->launches++;
            rc = pmx_fiber_exec(fp, tf, nullptr);
        }
        if (rc == PMX_OK) {
            DecimTaps none;
            none.n = 0;
            pmx_k_dsp_sample<<<B, 256, 0, c->stream>>>(tf->data, (size_t)L, tf->log2N1, tf->log2N2, L, 1, 0, d->peak, d->nlr_alpha, 0, none, sig);
            c->launches++;
            if (cudaGetLastError() != cudaSuccess) rc = set_err(c, PMX_ERR_CUDA, "%s: dispersion-compensation kernels failed", who);
        }
        std::string keep = c->error;
        pmx_plan_destroy(fp);
        pmx_field_destroy(tf);
        if (rc != PMX_OK) {
            c->error = keep;
            for (void* q : {(void*)sig, (void*)y, (void*)w1, (void*)w2, (void*)om, (void*)ph, (void*)dref, (void*)acc, (void*)dpass})
                cudaFreeAsync(q, c->stream);
            return rc;
        }
    }
    const cpx* stream_in = sig;
    cpx* stage_out = y;
    int* dpass_easi = nullptr;
    if (d->apply_easi) {   // 'easi' / first half of 'combo' (dsp4cohdec.m:234-241)
        if (!(d->easi_mu > 0)) {
            for (void* q : {(void*)sig, (void*)y, (void*)w1, (void*)w2, (void*)om, (void*)ph, (void*)dref, (void*)acc, (void*)dpass})
                cudaFreeAsync(q, c->stream);
            return set_err(c, PMX_ERR_INVALID, "%s: easi_mu must be > 0", who);
        }
        CK(c, cudaMallocAsync(&dpass_easi, (size_t)B * sizeof(int), c->stream));
        CK(c, cudaMemsetAsync(dpass_easi, 0, (size_t)B * sizeof(int), c->stream));
        const int rep = d->easi_max_passes > 0 ? d->easi_max_passes + 1 : 20 * (int)ceil(1.0 / ((double)L * d->easi_mu));
        pmx_k_dsp_easi<<<B, 32, 0, c->stream>>>(sig, y, L, d->easi_mu, d->easi_phizero, rep, dpass_easi);
        c->launches++;
        stream_in = y;
        stage_out = sig;
    }
    if (d->apply_cma) {
        const int rep = d->max_passes > 0 ? d->max_passes + 1 : 50 * (int)ceil(1.0 / ((double)L * d->mu));
        const cpx* cin = stream_in;
        cpx* cout_ = stage_out;
        switch (d->taps) {
#define PMX_CMA_CASE(T) case T: pmx_k_dsp_cma<T><<<B, 32, 0, c->stream>>>(cin, cout_, L, d->mu, d->R[0], d->R[1], d->phizero, rep, dpass); break;
#define PMX_CMA_WARP(T) case T: pmx_k_dsp_cma_w<T><<<B, 32, 0, c->stream>>>(cin, cout_, L, d->mu, d->R[0], d->R[1], d->phizero, rep, dpass); break;
            PMX_CMA_WARP(1) PMX_CMA_WARP(3) PMX_CMA_WARP(5) PMX_CMA_WARP(7) PMX_CMA_CASE(9) PMX_CMA_CASE(11) PMX_CMA_CASE(13)
            PMX_CMA_CASE(15)
#undef PMX_CMA_CASE
#undef PMX_CMA_WARP
        }
        stream_in = stage_out;
        c->launches++;
    }
    pmx_k_dsp_carrier<<<2 * B, PMX_CARRIER_THREADS, 0, c->stream>>>(stream_in, w1, w2, om, ph, L, 1 << d->modorder, d->freqavg, d->phasavg,
                                                   d->poworder, d->modorder > 1 ? 0.78539816339744830962 : 0.0);
    c->launches += 2;
    if (counts_dev) {
        dim3 g((unsigned)std::min((L + 255) / 256, 64), B);
        pmx_k_dsp_decide<<<g, 256, 0, c->stream>>>(ph, dref, L, acc);
        pmx_k_dsp_final<<<(B + 127) / 128, 128, 0, c->stream>>>(acc, B, (unsigned long long*)counts_dev);
        c->launches += 2;
    }
    CK(c, cudaGetLastError());
    if (phases) CK(c, cudaMemcpyAsync(phases, ph, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (amps) {   // the carrier is a pure phase: abs(Signals .* Carrier) = abs(Signals)
        pmx_k_dsp_abs<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 8), 256, 0, c->stream>>>(stream_in, n, om);
        c->launches++;
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(amps, om, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    if (passes_host) CK(c, cudaMemcpyAsync(passes_host, dpass, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (dpass_easi && d->easi_passes)
        CK(c, cudaMemcpyAsync(d->easi_passes, dpass_easi, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    for (void* q : {(void*)sig, (void*)y, (void*)w1, (void*)w2, (void*)om, (void*)ph, (void*)dref, (void*)acc, (void*)dpass,
                    (void*)dpass_easi})
        if (q) CK(c, cudaFreeAsync(q, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));   // ref_patmat / phases / passes_host are host buffers of the caller
    return PMX_OK;
}

extern "C" int pmx_dsp_count(pmx_ctx* c, pmx_devfield* f, const pmx_dsp_desc* d, const uint8_t* ref_patmat, int64_t* counts_dev,
                             int32_t* passes_host) {
    if (!c || !f || !d || !ref_patmat || !counts_dev) return set_err(c, PMX_ERR_INVALID, "pmx_dsp_count: null argument");
    return dsp_core(c, f, d, ref_patmat, counts_dev, nullptr, nullptr, passes_host, "pmx_dsp_count");
}

extern "C" int pmx_dsp_phases(pmx_ctx* c, pmx_devfield* f, const pmx_dsp_desc* d, double* phases, double* amps,
                              int32_t* passes_host) {
    if (!c || !f || !d || !phases) return set_err(c, PMX_ERR_INVALID, "pmx_dsp_phases: null argument");
    return dsp_core(c, f, d, nullptr, nullptr, phases, amps, passes_host, "pmx_dsp_phases");
}

// ---------------------------------------------------------------------------
// building blocks of the local-error adaptive step (scalar path, fiber.m:639-679,938-1010); FP64
__global__ void __launch_bounds__(256) pmx_k_scalar_nl(cpx* field, size_t N, int nfc, const double* gam /*[nfc], device*/,
                                                       double leff, double atten, int spm, int xpm) {
    const int b = blockIdx.y;
    cpx* fld = field + (size_t)b * nfc * N * 2;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        double sum = 0.0;
        if (xpm)
            for (int k = 0; k < nfc; ++k) {  // sum(pow,2)
                const cpx x = fld[((size_t)k * N + n) * 2];
                sum = __dadd_rn(sum, __dadd_rn(__dmul_rn(x.x, x.x), __dmul_rn(x.y, x.y)));
            }
        for (int k = 0; k < nfc; ++k) {
            cpx x = fld[((size_t)k * N + n) * 2];
            if (spm || xpm) {
                double pw = __dadd_rn(__dmul_rn(x.x, x.x), __dmul_rn(x.y, x.y));
                if (xpm) pw = spm ? __dadd_rn(__dmul_rn(2.0, sum), -pw) : __dmul_rn(2.0, __dadd_rn(sum, -pw));
                double sn, cs;
                pmx_sincos_fast(__dmul_rn(__dmul_rn(-gam[k], pw), leff), &sn, &cs);
                x = cmul(x, make_double2(cs, sn));
            }
            fld[((size_t)k * N + n) * 2] = make_double2(__dmul_rn(x.x, atten), __dmul_rn(x.y, atten));
        }
    }
}

static int need_f64(pmx_ctx* c, const pmx_devfield* f, const char* who) {
    if (!c || !f) return set_err(c, PMX_ERR_INVALID, "%s: null argument", who);
    if (f->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "%s: FP64 fields only", who);
    return PMX_OK;
}

extern "C" int pmx_scalar_nl_exec(pmx_ctx* c, pmx_devfield* f, const double* gam, double leff, double atten, int32_t spm,
                                  int32_t xpm) {
    int rc = need_f64(c, f, "pmx_scalar_nl_exec");
    if (rc) return rc;
    if (!gam) return set_err(c, PMX_ERR_INVALID, "pmx_scalar_nl_exec: gam is required");
    CK(c, cudaSetDevice(c->device));
    double* dg = nullptr;
    CK(c, cudaMallocAsync(&dg, f->nfc * sizeof(double), c->stream));
    CK(c, cudaMemcpyAsync(dg, gam, f->nfc * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    dim3 g((unsigned)std::min<size_t>(((size_t)f->nfft + 255) / 256, 148 * 8), f->batch);
    pmx_k_scalar_nl<<<g, 256, 0, c->stream>>>(f->data, (size_t)f->nfft, f->nfc, dg, leff, atten, spm, xpm);
    c->launches++;
    CK(c, cudaGetLastError());
    CK(c, cudaFreeAsync(dg, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));  // gam is a host buffer of the caller
    return PMX_OK;
}

extern "C" int pmx_plan_set_length(pmx_plan* p, double length) {
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "null plan");
    if (!(length > 0)) return set_err(p->ctx, PMX_ERR_INVALID, "length must be > 0");
    if (!p->single_step) return set_err(p->ctx, PMX_ERR_INVALID, "pmx_plan_set_length: only for plans of a one-step (linear) flag");
    p->d.length = length;
    p->d.dzmaxt = length;
    p->fc.Lf = length;
    p->fc.dzmax = length;
    p->fc.lcorr = length / p->d.nplates;
    return PMX_OK;
}

__global__ void __launch_bounds__(256) pmx_k_max_power(const cpx* field, size_t N, unsigned long long* out) {
    const int bc = blockIdx.y;
    const cpx* fld = field + (size_t)bc * N * 2;
    unsigned long long vmax = 0ull;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (size_t)gridDim.x * blockDim.x) {
        cpx x, y;
        ld_sa(fld + 2 * n, x, y);
        const unsigned long long key = pmx_pow_key(power_ref(x, y));
        vmax = key > vmax ? key : vmax;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, vmax, o);
        vmax = other > vmax ? other : vmax;
    }
    if ((threadIdx.x & 31) == 0) atomicMax(&out[bc], vmax);
}

extern "C" int pmx_field_max_power(pmx_ctx* c, pmx_devfield* f, double* umax) {
    int rc = need_f64(c, f, "pmx_field_max_power");
    if (rc) return rc;
    if (!umax) return set_err(c, PMX_ERR_INVALID, "pmx_field_max_power: null output");
    CK(c, cudaSetDevice(c->device));
    const int nbc = f->batch * f->nfc;
    unsigned long long* d = nullptr;
    CK(c, cudaMallocAsync(&d, nbc * sizeof(unsigned long long), c->stream));
    CK(c, cudaMemsetAsync(d, 0, nbc * sizeof(unsigned long long), c->stream));
    dim3 g((unsigned)std::min<size_t>(((size_t)f->nfft + 255) / 256, 148 * 8), nbc);
    pmx_k_max_power<<<g, 256, 0, c->stream>>>(f->data, (size_t)f->nfft, d);
    c->launches++;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(umax, d, nbc * sizeof(double), cudaMemcpyDeviceToHost, c->stream));  // key == bit pattern
    CK(c, cudaFreeAsync(d, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

// mean over the samples of |x|^2 + |y|^2 per realization-column (avg_power.m:63-76 for a separate-channel field: the
// spectral sum over all bins divided by Nfft^2 is the time average, by Parseval).  Two stages with fixed summation
// trees -- CTA (chunk, column) writes one partial, thread 0 of a second launch adds the partials left to right -- so the
// result is the same on every run.  E = double2 or float2 elements; the sum is taken in double either way.
template <typename E>
__global__ void __launch_bounds__(256) pmx_k_mean_power(const E* field, size_t N, double* part) {
    __shared__ double redx[256], redy[256];
    const E* fld = field + (size_t)blockIdx.y * N * 2;
    const size_t per = (N + gridDim.x - 1) / gridDim.x;
    const size_t n0 = blockIdx.x * per, n1 = n0 + per < N ? n0 + per : N;
    double ax = 0.0, ay = 0.0;
    for (size_t n = n0 + threadIdx.x; n < n1; n += blockDim.x) {
        const E x = fld[2 * n], y = fld[2 * n + 1];
        ax += (double)x.x * x.x + (double)x.y * x.y;
        ay += (double)y.x * y.x + (double)y.y * y.y;
    }
    redx[threadIdx.x] = ax;
    redy[threadIdx.x] = ay;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) {
            redx[threadIdx.x] += redx[threadIdx.x + o];
            redy[threadIdx.x] += redy[threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        part[2 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x)] = redx[0];
        part[2 * ((size_t)blockIdx.y * gridDim.x + blockIdx.x) + 1] = redy[0];
    }
}

// out[0..nbc) = mean |x|^2, out[nbc..2nbc) = mean |y|^2
__global__ void pmx_k_mean_power_fin(const double* part, int nchunk, size_t N, int nbc, double* out) {
    const int bc = blockIdx.x * blockDim.x + threadIdx.x;
    if (bc >= nbc) return;
    double ax = 0.0, ay = 0.0;
    for (int i = 0; i < nchunk; ++i) {
        ax += part[2 * ((size_t)bc * nchunk + i)];
        ay += part[2 * ((size_t)bc * nchunk + i) + 1];
    }
    out[bc] = ax / (double)N;
    out[nbc + bc] = ay / (double)N;
}

extern "C" int pmx_field_mean_power_xy(pmx_ctx* c, pmx_devfield* f, double* px, double* py) {
    if (!c || !f || !px || !py) return set_err(c, PMX_ERR_INVALID, "pmx_field_mean_power: null argument");
    CK(c, cudaSetDevice(c->device));
    const int nbc = f->batch * f->nfc;
    const int nchunk = (int)std::max<size_t>(1, std::min<size_t>(((size_t)f->nfft + 4095) / 4096, (148 * 8 + nbc - 1) / nbc));
    double* d = nullptr;
    CK(c, cudaMallocAsync(&d, (2 * (size_t)nbc * nchunk + 2 * nbc) * sizeof(double), c->stream));
    double* dout = d + 2 * (size_t)nbc * nchunk;
    dim3 g(nchunk, nbc);
    if (f->precision == PMX_F32)
        pmx_k_mean_power<float2><<<g, 256, 0, c->stream>>>(reinterpret_cast<const float2*>(f->data), (size_t)f->nfft, d);
    else
        pmx_k_mean_power<double2><<<g, 256, 0, c->stream>>>(reinterpret_cast<const double2*>(f->data), (size_t)f->nfft, d);
    pmx_k_mean_power_fin<<<(nbc + 127) / 128, 128, 0, c->stream>>>(d, nchunk, (size_t)f->nfft, nbc, dout);
    c->launches += 2;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(px, dout, nbc * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(py, dout + nbc, nbc * sizeof(double), cudaMemcpyDeviceToHost, c->stream);
    cudaFreeAsync(d, c->stream);
    CK(c, e);
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" int pmx_field_mean_power(pmx_ctx* c, pmx_devfield* f, double* pavg) {
    if (!c || !f || !pavg) return set_err(c, PMX_ERR_INVALID, "pmx_field_mean_power: null argument");
    const int nbc = f->batch * f->nfc;
    std::vector<double> px(nbc), py(nbc);
    int rc = pmx_field_mean_power_xy(c, f, px.data(), py.data());
    if (rc) return rc;
    for (int i = 0; i < nbc; ++i) pavg[i] = px[i] + py[i];   // E = Ex + Ey (avg_power.m:131)
    return PMX_OK;
}

__global__ void __launch_bounds__(256) pmx_k_maxdiff2(const cpx* a, const cpx* b, size_t n_sa, unsigned long long* out) {
    unsigned long long vmax = 0ull;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < n_sa; n += (size_t)gridDim.x * blockDim.x) {
        const cpx x = a[2 * n], z = b[2 * n];
        const double dr = __dadd_rn(x.x, -z.x), di = __dadd_rn(x.y, -z.y);
        const unsigned long long key = pmx_pow_key(__dadd_rn(__dmul_rn(dr, dr), __dmul_rn(di, di)));
        vmax = key > vmax ? key : vmax;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, vmax, o);
        vmax = other > vmax ? other : vmax;
    }
    if ((threadIdx.x & 31) == 0) atomicMax(out, vmax);
}

static int same_shape(pmx_ctx* c, const pmx_devfield* a, const pmx_devfield* b, const char* who) {
    if (a->nfft != b->nfft || a->nfc != b->nfc || a->batch != b->batch || a->precision != b->precision)
        return set_err(c, PMX_ERR_INVALID, "%s: fields differ in shape or precision", who);
    return PMX_OK;
}

extern "C" int pmx_field_maxdiff2(pmx_ctx* c, pmx_devfield* a, pmx_devfield* b, double* out) {
    int rc = need_f64(c, a, "pmx_field_maxdiff2");
    if (rc == PMX_OK) rc = need_f64(c, b, "pmx_field_maxdiff2");
    if (rc == PMX_OK) rc = same_shape(c, a, b, "pmx_field_maxdiff2");
    if (rc) return rc;
    if (!out) return set_err(c, PMX_ERR_INVALID, "pmx_field_maxdiff2: null output");
    CK(c, cudaSetDevice(c->device));
    unsigned long long* d = nullptr;
    CK(c, cudaMallocAsync(&d, sizeof(unsigned long long), c->stream));
    CK(c, cudaMemsetAsync(d, 0, sizeof(unsigned long long), c->stream));
    const size_t n_sa = (size_t)a->batch * a->nfc * a->nfft;
    pmx_k_maxdiff2<<<(unsigned)std::min<size_t>((n_sa + 255) / 256, 148 * 8), 256, 0, c->stream>>>(a->data, b->data, n_sa, d);
    c->launches++;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(out, d, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaFreeAsync(d, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

__global__ void __launch_bounds__(256) pmx_k_lincomb(cpx* dst, double ca, const cpx* a, double cb, const cpx* b, size_t n_cpx) {
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < n_cpx; n += (size_t)gridDim.x * blockDim.x) {
        const cpx x = a[n], z = b[n];
        dst[n] = make_double2(__dadd_rn(__dmul_rn(ca, x.x), -__dmul_rn(cb, z.x)), __dadd_rn(__dmul_rn(ca, x.y), -__dmul_rn(cb, z.y)));
    }
}

extern "C" int pmx_field_lincomb(pmx_ctx* c, pmx_devfield* dst, double ca, pmx_devfield* a, double cb, pmx_devfield* b) {
    int rc = need_f64(c, dst, "pmx_field_lincomb");
    if (rc == PMX_OK) rc = need_f64(c, a, "pmx_field_lincomb");
    if (rc == PMX_OK) rc = need_f64(c, b, "pmx_field_lincomb");
    if (rc == PMX_OK) rc = same_shape(c, dst, a, "pmx_field_lincomb");
    if (rc == PMX_OK) rc = same_shape(c, dst, b, "pmx_field_lincomb");
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    const size_t n_cpx = (size_t)dst->batch * dst->nfc * dst->nfft * 2;
    pmx_k_lincomb<<<(unsigned)std::min<size_t>((n_cpx + 255) / 256, 148 * 8), 256, 0, c->stream>>>(dst->data, ca, a->data, cb, b->data, n_cpx);
    c->launches++;
    CK(c, cudaGetLastError());
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// inverse_pmd.m:73-131 on the device.  update_U (:152-161) only ever propagates the first row (a, b) of U -- the second
// is rebuilt as (-b*, a*) after every update -- so the state is two complex numbers per frequency.
struct cplx {
    double re, im;
};
static inline cplx cmulh(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
static inline cplx cconjh(cplx a) { return {a.re, -a.im}; }
static inline cplx caddh(cplx a, cplx b) { return {a.re + b.re, a.im + b.im}; }
// getmatR (inverse_pmd.m:164-168): (cos(theta)*sig0 - sin(theta)*sig3i) * complex(cos(eps)*sig0, sin(eps)*sig2)
static void get_mat_r(double theta, double eps, cplx m[4]) {
    const double c = std::cos(theta), s = std::sin(theta), ce = std::cos(eps), se = std::sin(eps);
    const cplx rt[4] = {{c, 0}, {-s, 0}, {s, 0}, {c, 0}};
    const cplx re[4] = {{ce, 0}, {0, se}, {0, se}, {ce, 0}};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) m[2 * i + j] = caddh(cmulh(rt[2 * i], re[j]), cmulh(rt[2 * i + 1], re[2 + j]));
}

// one fiber: ab <- first row of (R_last * prod_k D_k R_k' R_(k-1) * D_1 R_1') * [a b; -b* a*]; allgvd += betat*lcorr*ntrunk
__global__ void __launch_bounds__(128) pmx_k_pmd_update(double2* ab, double* allgvd, const double* db1, const double* betat,
                                                         const double2* rows, const double* db0, int ntrunk, double lcorr,
                                                         size_t nfft) {
    const size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nfft) return;
    double2 a = ab[2 * n], b = ab[2 * n + 1];
    const double d1 = db1[n];
    for (int k = 0; k <= ntrunk; ++k) {
        double2 t11 = rows[2 * k], t12 = rows[2 * k + 1];
        if (k < ntrunk) {   // l1 = fastexp(-deltabeta), deltabeta = 0.5*(db1 + db0(k)) (:95-97,115-118); the last update has l1 = 1
            double sn, cs;
            sincos(-(0.5 * (d1 + db0[k])), &sn, &cs);
            const double2 l1 = make_double2(cs, sn);
            t11 = make_double2(l1.x * t11.x - l1.y * t11.y, l1.x * t11.y + l1.y * t11.x);
            t12 = make_double2(l1.x * t12.x - l1.y * t12.y, l1.x * t12.y + l1.y * t12.x);
        }
        const double2 u21 = make_double2(-b.x, b.y), u22 = make_double2(a.x, -a.y);
        const double2 na = make_double2((t11.x * a.x - t11.y * a.y) + (t12.x * u21.x - t12.y * u21.y),
                                        (t11.x * a.y + t11.y * a.x) + (t12.x * u21.y + t12.y * u21.x));
        const double2 nb = make_double2((t11.x * b.x - t11.y * b.y) + (t12.x * u22.x - t12.y * u22.y),
                                        (t11.x * b.y + t11.y * b.x) + (t12.x * u22.y + t12.y * u22.x));
        a = na;
        b = nb;
    }
    ab[2 * n] = a;
    ab[2 * n + 1] = b;
    allgvd[n] += betat[n] * lcorr * (double)ntrunk;
}

// U = Hgvd .* [a b; -b* a*], Uinv = U' (inverse_pmd.m:123-131), written in the interpreter's column-major [2][2][nfft]
__global__ void __launch_bounds__(128) pmx_k_pmd_finish(const double2* ab, const double* allgvd, int gvd, size_t nfft,
                                                         double2* U, double2* Uinv) {
    const size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= nfft) return;
    const double2 a = ab[2 * n], b = ab[2 * n + 1];
    double2 u[4] = {a, make_double2(-b.x, b.y), b, make_double2(a.x, -a.y)};   // (1,1) (2,1) (1,2) (2,2)
    if (gvd) {
        double sn, cs;
        sincos(-allgvd[n], &sn, &cs);
        for (int i = 0; i < 4; ++i) u[i] = make_double2(cs * u[i].x - sn * u[i].y, cs * u[i].y + sn * u[i].x);
    }
    if (U)
        for (int i = 0; i < 4; ++i) U[4 * n + i] = u[i];
    if (Uinv) {
        Uinv[4 * n + 0] = make_double2(u[0].x, -u[0].y);   // Uinv(1,1) = conj(U(1,1))
        Uinv[4 * n + 1] = make_double2(u[2].x, -u[2].y);   // Uinv(2,1) = conj(U(1,2))
        Uinv[4 * n + 2] = make_double2(u[1].x, -u[1].y);   // Uinv(1,2) = conj(U(2,1))
        Uinv[4 * n + 3] = make_double2(u[3].x, -u[3].y);
    }
}

extern "C" int pmx_pmd_matrix(pmx_ctx* c, int64_t nfft, int32_t nfiber, const pmx_brf* brf, const double* mat, int32_t gvd,
                              double* U, double* Uinv) {
    if (!c || !brf || nfiber < 1 || nfft < 1) return set_err(c, PMX_ERR_INVALID, "pmx_pmd_matrix: bad arguments");
    for (int f = 0; f < nfiber; ++f)
        if (brf[f].ntrunk < 1 || !brf[f].db0 || !brf[f].theta || !brf[f].epsilon || !brf[f].betat || !brf[f].db1)
            return set_err(c, PMX_ERR_INVALID, "pmx_pmd_matrix: fiber %d of the chain is incomplete", f);
    CK(c, cudaSetDevice(c->device));
    const size_t N = (size_t)nfft;
    int maxtr = 0;
    for (int f = 0; f < nfiber; ++f) maxtr = std::max(maxtr, brf[f].ntrunk);
    // one allocation: ab [2N] double2, allgvd [N], db1 [N], betat [N], rows [2(maxtr+1)] double2, db0 [maxtr], U, Uinv [4N] double2
    const size_t bytes = 2 * N * 16 + 3 * N * 8 + 2 * (size_t)(maxtr + 1) * 16 + (size_t)maxtr * 8 + 8 * N * 16;
    unsigned char* d = nullptr;
    CK(c, cudaMallocAsync(&d, bytes, c->stream));
    double2* ab = reinterpret_cast<double2*>(d);
    double2* dU = ab + 2 * N;
    double2* dUinv = dU + 4 * N;
    double2* drows = dUinv + 4 * N;
    double* dgvd = reinterpret_cast<double*>(drows + 2 * (size_t)(maxtr + 1));
    double* ddb1 = dgvd + N;
    double* dbetat = ddb1 + N;
    double* ddb0 = dbetat + N;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t r) {
        if (e == cudaSuccess) e = r;
    };
    // U = eye, or the first row of options.mat (update_U with l1 = l2 = 1, inverse_pmd.m:87-89)
    std::vector<cplx> init(2 * N);
    const cplx a0 = mat ? cplx{mat[0], mat[1]} : cplx{1.0, 0.0}, b0 = mat ? cplx{mat[2], mat[3]} : cplx{0.0, 0.0};
    for (size_t n = 0; n < N; ++n) {
        init[2 * n] = a0;
        init[2 * n + 1] = b0;
    }
    step(cudaMemcpyAsync(ab, init.data(), 2 * N * 16, cudaMemcpyHostToDevice, c->stream));
    step(cudaMemsetAsync(dgvd, 0, N * 8, c->stream));
    std::vector<cplx> rows;
    const unsigned grid = (unsigned)((N + 127) / 128);
    for (int f = 0; f < nfiber && e == cudaSuccess; ++f) {
        const pmx_brf& b = brf[f];
        rows.assign(2 * (size_t)(b.ntrunk + 1), cplx{0, 0});
        cplx m1[4], m2[4];
        get_mat_r(b.theta[0], b.epsilon[0], m1);
        rows[0] = cconjh(m1[0]);                         // matR' : first row = conj of the first column
        rows[1] = cconjh(m1[2]);
        for (int k = 1; k < b.ntrunk; ++k) {             // matR2' * matR1 (:100-102)
            get_mat_r(b.theta[k - 1], b.epsilon[k - 1], m1);
            get_mat_r(b.theta[k], b.epsilon[k], m2);
            for (int j = 0; j < 2; ++j) rows[2 * k + j] = caddh(cmulh(cconjh(m2[0]), m1[j]), cmulh(cconjh(m2[2]), m1[2 + j]));
        }
        get_mat_r(b.theta[b.ntrunk - 1], b.epsilon[b.ntrunk - 1], m1);
        rows[2 * b.ntrunk] = m1[0];
        rows[2 * b.ntrunk + 1] = m1[1];
        step(cudaMemcpyAsync(drows, rows.data(), rows.size() * 16, cudaMemcpyHostToDevice, c->stream));
        step(cudaMemcpyAsync(ddb0, b.db0, (size_t)b.ntrunk * 8, cudaMemcpyHostToDevice, c->stream));
        step(cudaMemcpyAsync(ddb1, b.db1, N * 8, cudaMemcpyHostToDevice, c->stream));
        step(cudaMemcpyAsync(dbetat, b.betat, N * 8, cudaMemcpyHostToDevice, c->stream));
        pmx_k_pmd_update<<<grid, 128, 0, c->stream>>>(ab, dgvd, ddb1, dbetat, drows, ddb0, b.ntrunk, b.lcorr, N);
        c->launches++;
        step(cudaGetLastError());
        step(cudaStreamSynchronize(c->stream));          // rows / the caller's arrays are pageable host memory reused next turn
    }
    if (e == cudaSuccess) {
        pmx_k_pmd_finish<<<grid, 128, 0, c->stream>>>(ab, dgvd, gvd ? 1 : 0, N, U ? dU : nullptr, Uinv ? dUinv : nullptr);
        c->launches++;
        step(cudaGetLastError());
        if (U) step(cudaMemcpyAsync(U, dU, 4 * N * 16, cudaMemcpyDeviceToHost, c->stream));
        if (Uinv) step(cudaMemcpyAsync(Uinv, dUinv, 4 * N * 16, cudaMemcpyDeviceToHost, c->stream));
    }
    cudaFreeAsync(d, c->stream);
    cudaError_t es = cudaStreamSynchronize(c->stream);
    CK(c, e);
    CK(c, es);
    return PMX_OK;
}

template <typename E>
__global__ void __launch_bounds__(256) pmx_k_jones(E* field, size_t n_sa, double j0, double j1, double j2, double j3, double j4,
                                                    double j5, double j6, double j7) {
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < n_sa; n += (size_t)gridDim.x * blockDim.x) {
        const E x = field[2 * n], y = field[2 * n + 1];
        const double xr = x.x, xi = x.y, yr = y.x, yi = y.y;
        E ox, oy;
        ox.x = (j0 * xr - j1 * xi) + (j2 * yr - j3 * yi);
        ox.y = (j0 * xi + j1 * xr) + (j2 * yi + j3 * yr);
        oy.x = (j4 * xr - j5 * xi) + (j6 * yr - j7 * yi);
        oy.y = (j4 * xi + j5 * xr) + (j6 * yi + j7 * yr);
        field[2 * n] = ox;
        field[2 * n + 1] = oy;
    }
}

extern "C" int pmx_field_jones(pmx_ctx* c, pmx_devfield* f, const double* j) {
    if (!c || !f || !j) return set_err(c, PMX_ERR_INVALID, "pmx_field_jones: null argument");
    CK(c, cudaSetDevice(c->device));
    const size_t n_sa = (size_t)f->batch * f->nfc * f->nfft;
    const unsigned grid = (unsigned)std::min<size_t>((n_sa + 255) / 256, 148 * 8);
    if (f->precision == PMX_F32)
        pmx_k_jones<float2><<<grid, 256, 0, c->stream>>>(reinterpret_cast<float2*>(f->data), n_sa, j[0], j[1], j[2], j[3], j[4],
                                                         j[5], j[6], j[7]);
    else
        pmx_k_jones<double2><<<grid, 256, 0, c->stream>>>(reinterpret_cast<double2*>(f->data), n_sa, j[0], j[1], j[2], j[3],
                                                          j[4], j[5], j[6], j[7]);
    c->launches++;
    CK(c, cudaGetLastError());
    return PMX_OK;
}

// inverse_pmd(brf, options) on host buffers (what the MEX gateway binds for matlab/inverse_pmd.m): inv(U) of a chain is the
// linear step of every fiber taken backwards -- plates in reverse order, db0, db1 and betat negated, no loss -- one
// single-step run of the SSFM passes per fiber on the resident field, then the constant Jones matrix of options.mat;
// U / Uinv from pmx_pmd_matrix.  apply = 0: the field is left alone (io may be NULL).
extern "C" int pmx_inverse_pmd_run(pmx_ctx* c, int64_t nfft, int32_t nfiber, const pmx_brf* brf, const double* mat, int32_t gvd,
                                   int32_t apply, pmx_field* io, double* U, double* Uinv) {
    if (!c || !brf || nfiber < 1) return set_err(c, PMX_ERR_INVALID, "pmx_inverse_pmd_run: bad arguments");
    if (apply && !io) return set_err(c, PMX_ERR_INVALID, "pmx_inverse_pmd_run: a field is required when it is to be transformed");
    int rc = PMX_OK;
    if (U || Uinv) rc = pmx_pmd_matrix(c, nfft, nfiber, brf, mat, gvd, U, Uinv);
    if (rc != PMX_OK || !apply) return rc;
    const size_t N = (size_t)nfft;
    pmx_devfield* f = nullptr;
    rc = pmx_field_create(c, nfft, 1, 1, PMX_F64, &f);
    if (rc == PMX_OK) rc = pmx_field_upload(f, io, 0, 1);
    std::vector<double> nbt(N), ndb1(N), rdb0, rth, rep;
    const double gam0 = 0.0;
    for (int k = nfiber - 1; k >= 0 && rc == PMX_OK; --k) {
        const pmx_brf& b = brf[k];
        if (b.ntrunk < 1 || !b.db0 || !b.theta || !b.epsilon || !b.betat || !b.db1) {
            rc = set_err(c, PMX_ERR_INVALID, "pmx_inverse_pmd_run: fiber %d of the chain is incomplete", k);
            break;
        }
        const int nt = b.ntrunk;
        rdb0.resize(nt);
        rth.resize(nt);
        rep.resize(nt);
        for (int n = 0; n < nt; ++n) {
            rdb0[n] = -b.db0[nt - 1 - n];
            rth[n] = b.theta[nt - 1 - n];
            rep[n] = b.epsilon[nt - 1 - n];
        }
        for (size_t n = 0; n < N; ++n) {
            nbt[n] = gvd ? -b.betat[n] : 0.0;
            ndb1[n] = -b.db1[n];
        }
        pmx_fiber_desc d;
        memset(&d, 0, sizeof d);
        d.nfft = nfft;
        d.nfc = 1;
        d.batch = 1;
        d.precision = PMX_F64;
        d.length = d.dzmaxt = b.lcorr * nt;
        d.dphimaxt = INFINITY;
        d.gam = &gam0;
        d.fls[0] = 1;
        d.fls[1] = 1;
        d.nplates = nt;
        d.plate_sets = 1;
        d.db0 = rdb0.data();
        d.theta = rth.data();
        d.epsilon = rep.data();
        d.betat = nbt.data();
        d.db1 = ndb1.data();
        d.disp_mode = PMX_DISP_VECTOR;
        d.nsymb = (int32_t)std::min<int64_t>(nfft, INT32_MAX);
        d.nt = 1;
        d.symbolrate = 1.0;
        pmx_plan* p = nullptr;
        rc = pmx_plan_create(c, &d, &p);
        if (rc == PMX_OK) rc = pmx_fiber_exec(p, f, nullptr);
        std::string keep = c->error;
        pmx_plan_destroy(p);
        if (rc != PMX_OK) c->error = keep;
    }
    if (rc == PMX_OK && mat) {   // U = chain * [m11 m12; -m12* m11*]  ->  Uinv = [m11* -m12; m12* m11] * chain'
        const double j[8] = {mat[0], -mat[1], -mat[2], -mat[3], mat[2], -mat[3], mat[0], mat[1]};
        rc = pmx_field_jones(c, f, j);
    }
    if (rc == PMX_OK) rc = pmx_field_download(f, io, 0, 1);
    std::string keep = c->error;
    pmx_field_destroy(f);
    if (rc != PMX_OK) c->error = keep;
    return rc;
}

// ---------------------------------------------------------------------------
// Front-end of the coherent receiver (receiver_cohmix.m): copies of field columns, the channel's frequency shift, LO
// mixing + photodetection.  The two filters in between are filter plans (pmx_filter_create).
extern "C" int pmx_field_copy_cols(pmx_devfield* dst, int32_t dst_bc, const pmx_devfield* src, int32_t src_bc, int32_t count) {
    if (!dst || !src) return set_err(nullptr, PMX_ERR_INVALID, "null field");
    pmx_ctx* c = dst->ctx;
    if (dst->nfft != src->nfft || dst->precision != src->precision)
        return set_err(c, PMX_ERR_INVALID, "pmx_field_copy_cols: length or precision mismatch");
    if (count < 0 || dst_bc < 0 || src_bc < 0 || dst_bc + count > dst->batch * dst->nfc || src_bc + count > src->batch * src->nfc)
        return set_err(c, PMX_ERR_INVALID, "pmx_field_copy_cols: column range outside the field");
    CK(c, cudaSetDevice(c->device));
    const size_t col = (size_t)src->nfft * 2 * src->cbytes();
    CK(c, cudaMemcpyAsync((char*)dst->data + (size_t)dst_bc * col, (const char*)src->data + (size_t)src_bc * col, (size_t)count * col,
                          cudaMemcpyDeviceToDevice, c->stream));
    return PMX_OK;
}

// time index of the sample stored at position pos of a column
__device__ __forceinline__ size_t pmx_time_index(size_t pos, int l1, int l2) {
    return ((pos & (((size_t)1 << l1) - 1)) << l2) + (pos >> l1);
}

// u(n) <- u(n) * exp(+i*2*pi*m*n/N): the spectrum moves up by m bins (x.sigx(nind), receiver_cohmix.m:93,172)
template <typename E>
__global__ void __launch_bounds__(256) pmx_k_modulate(E* field, size_t N, int l1, int l2, long long m) {
    E* fld = field + (size_t)blockIdx.y * N * 2;
    for (size_t pos = (size_t)blockIdx.x * blockDim.x + threadIdx.x; pos < N; pos += (size_t)gridDim.x * blockDim.x) {
        PMX_ASSERT(pmx_time_index(pos, l1, l2) < N && m >= 0 && (unsigned long long)m < N && ((size_t)1 << (l1 + l2)) == N);
        const unsigned long long r = ((unsigned long long)m * (unsigned long long)pmx_time_index(pos, l1, l2)) & (N - 1);  // m*n mod N
        double sn, cs;
        sincospi(2.0 * (double)r / (double)N, &sn, &cs);
        const E x = fld[2 * pos], y = fld[2 * pos + 1];
        E ox, oy;
        ox.x = (double)x.x * cs - (double)x.y * sn;
        ox.y = (double)x.x * sn + (double)x.y * cs;
        oy.x = (double)y.x * cs - (double)y.y * sn;
        oy.y = (double)y.x * sn + (double)y.y * cs;
        fld[2 * pos] = ox;
        fld[2 * pos + 1] = oy;
    }
}

extern "C" int pmx_field_modulate(pmx_ctx* c, pmx_devfield* f, int64_t m) {
    if (!c || !f) return set_err(c, PMX_ERR_INVALID, "pmx_field_modulate: null argument");
    CK(c, cudaSetDevice(c->device));
    const size_t N = (size_t)f->nfft;
    const long long mm = ((m % (long long)N) + (long long)N) % (long long)N;
    dim3 g((unsigned)std::min<size_t>((N + 255) / 256, 148 * 8), f->batch * f->nfc);
    if (f->precision == PMX_F32)
        pmx_k_modulate<float2><<<g, 256, 0, c->stream>>>(reinterpret_cast<float2*>(f->data), N, f->log2N1, f->log2N2, mm);
    else
        pmx_k_modulate<double2><<<g, 256, 0, c->stream>>>(reinterpret_cast<double2*>(f->data), N, f->log2N1, f->log2N2, mm);
    c->launches++;
    CK(c, cudaGetLastError());
    return PMX_OK;
}

// Resampling of single-channel DBP (pmx_dbp_channel_create) between a one-column field of N samples (layout l1/l2) and
// the M = N/r = N >> lr samples of the channel (layout m1/m2); one realization per blockIdx.y.  The phase index is
// reduced modulo N in integers and the argument of sincospi is exact, as in pmx_k_modulate.
// Gather: v[n] = u[n*r] * exp(+i*2*pi*m*n*r/N) -- the band-passed channel at baseband, decimated.
template <typename E>
__global__ void __launch_bounds__(256) pmx_k_band_gather(const E* __restrict__ field, int l1, int l2, E* __restrict__ chan,
                                                         int m1, int m2, size_t N, int lr, long long m) {
    const size_t M = N >> lr;
    const E* src = field + (size_t)blockIdx.y * N * 2;
    E* dst = chan + (size_t)blockIdx.y * M * 2;
    for (size_t pos = (size_t)blockIdx.x * blockDim.x + threadIdx.x; pos < M; pos += (size_t)gridDim.x * blockDim.x) {
        const size_t t = pmx_time_index(pos, m1, m2) << lr;
        const size_t sp = pmx_mem_index(t, l1, l2);
        PMX_ASSERT(t < N && sp < N && m >= 0 && (unsigned long long)m < N);
        const unsigned long long r = ((unsigned long long)m * (unsigned long long)t) & (N - 1);   // m*n*r mod N
        double sn, cs;
        sincospi(2.0 * (double)r / (double)N, &sn, &cs);
        const E x = src[2 * sp], y = src[2 * sp + 1];
        E ox, oy;
        ox.x = (double)x.x * cs - (double)x.y * sn;
        ox.y = (double)x.x * sn + (double)x.y * cs;
        oy.x = (double)y.x * cs - (double)y.y * sn;
        oy.y = (double)y.x * sn + (double)y.y * cs;
        dst[2 * pos] = ox;
        dst[2 * pos + 1] = oy;
    }
}

// Stuff: u[n] = r * v[n/r] * exp(-i*2*pi*m*n/N) where r divides n, 0 elsewhere; the band filter that follows interpolates.
template <typename E>
__global__ void __launch_bounds__(256) pmx_k_band_stuff(const E* __restrict__ chan, int m1, int m2, E* __restrict__ field,
                                                        int l1, int l2, size_t N, int lr, long long m) {
    const size_t M = N >> lr;
    const E* src = chan + (size_t)blockIdx.y * M * 2;
    E* dst = field + (size_t)blockIdx.y * N * 2;
    const double rr = (double)(1 << lr);
    for (size_t pos = (size_t)blockIdx.x * blockDim.x + threadIdx.x; pos < N; pos += (size_t)gridDim.x * blockDim.x) {
        const size_t n = pmx_time_index(pos, l1, l2);
        E ox, oy;
        ox.x = ox.y = oy.x = oy.y = 0;
        if ((n & (((size_t)1 << lr) - 1)) == 0) {
            const size_t sp = pmx_mem_index(n >> lr, m1, m2);
            PMX_ASSERT(n < N && sp < M && m >= 0 && (unsigned long long)m < N);
            const unsigned long long r = ((unsigned long long)m * (unsigned long long)n) & (N - 1);   // m*n mod N
            double sn, cs;
            sincospi(2.0 * (double)r / (double)N, &sn, &cs);
            const E x = src[2 * sp], y = src[2 * sp + 1];
            ox.x = rr * ((double)x.x * cs + (double)x.y * sn);
            ox.y = rr * ((double)x.y * cs - (double)x.x * sn);
            oy.x = rr * ((double)y.x * cs + (double)y.y * sn);
            oy.y = rr * ((double)y.y * cs - (double)y.x * sn);
        }
        dst[2 * pos] = ox;
        dst[2 * pos + 1] = oy;
    }
}

// The four mixer outputs and the photocurrents of one polarization (receiver_cohmix.m:253-277), as the interpreter forms
// them: E1 = j*s + j*lo, E2 = s - lo, E3 = j*s - lo, E4 = -s + j*lo, I_k = real(E_k .* conj(E_k)); balanced detection
// returns (I1 - I2, I3 - I4), single photodiodes (I1, I3).  The pair is stored as one complex sample.
__device__ __forceinline__ double2 pmx_mix_pd(double sr, double si, double lr, double li, int balanced) {
    const double e1r = -si - li, e1i = sr + lr;
    const double e3r = -si - lr, e3i = sr - li;
    const double i1 = e1r * e1r + e1i * e1i, i3 = e3r * e3r + e3i * e3i;
    if (!balanced) return make_double2(i1, i3);
    const double e2r = sr - lr, e2i = si - li;
    const double e4r = -sr - li, e4i = -si + lr;
    const double i2 = e2r * e2r + e2i * e2i, i4 = e4r * e4r + e4i * e4i;
    return make_double2(i1 - i2, i3 - i4);
}

template <typename E>
__global__ void __launch_bounds__(256) pmx_k_cohmix(E* field, size_t N, int l1, int l2, double ecw, double detune,
                                                     const double* lophase, int balanced) {
    E* fld = field + (size_t)blockIdx.y * N * 2;
    for (size_t pos = (size_t)blockIdx.x * blockDim.x + threadIdx.x; pos < N; pos += (size_t)gridDim.x * blockDim.x) {
        const size_t n = pmx_time_index(pos, l1, l2);
        PMX_ASSERT(n < N && pmx_mem_index(n, l1, l2) == pos);
        // Elo = LO_Ecw * fastexp(LO_Detuning + LO_PhaseNoise), LO_Detuning = 2*pi*kdet/Nfft*(1:Nfft)' (:200,219)
        const double ph = (detune != 0.0 ? detune * (double)(n + 1) : 0.0) + (lophase ? lophase[n] : 0.0);
        double sn, cs;
        sincos(ph, &sn, &cs);
        const double lr = ecw * cs, li = ecw * sn;
        const E x = fld[2 * pos], y = fld[2 * pos + 1];
        const double2 zx = pmx_mix_pd(x.x, x.y, lr, li, balanced), zy = pmx_mix_pd(y.x, y.y, lr, li, balanced);
        E ox, oy;
        ox.x = zx.x; ox.y = zx.y; oy.x = zy.x; oy.y = zy.y;
        fld[2 * pos] = ox;
        fld[2 * pos + 1] = oy;
    }
}

extern "C" int pmx_cohmix_exec(pmx_ctx* c, pmx_devfield* f, double lo_ecw, double lo_detune, const double* lo_phase,
                               int32_t balanced) {
    if (!c || !f) return set_err(c, PMX_ERR_INVALID, "pmx_cohmix_exec: null argument");
    CK(c, cudaSetDevice(c->device));
    const size_t N = (size_t)f->nfft;
    double* dph = nullptr;
    if (lo_phase) {
        CK(c, cudaMallocAsync(&dph, N * sizeof(double), c->stream));
        cudaError_t e = cudaMemcpyAsync(dph, lo_phase, N * sizeof(double), cudaMemcpyHostToDevice, c->stream);
        if (e != cudaSuccess) {
            cudaFreeAsync(dph, c->stream);
            CK(c, e);
        }
    }
    dim3 g((unsigned)std::min<size_t>((N + 255) / 256, 148 * 8), f->batch * f->nfc);
    if (f->precision == PMX_F32)
        pmx_k_cohmix<float2><<<g, 256, 0, c->stream>>>(reinterpret_cast<float2*>(f->data), N, f->log2N1, f->log2N2, lo_ecw,
                                                         lo_detune, dph, balanced ? 1 : 0);
    else
        pmx_k_cohmix<double2><<<g, 256, 0, c->stream>>>(reinterpret_cast<double2*>(f->data), N, f->log2N1, f->log2N2, lo_ecw,
                                                          lo_detune, dph, balanced ? 1 : 0);
    c->launches++;
    cudaError_t e = cudaGetLastError();
    if (dph) {
        cudaFreeAsync(dph, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);   // lo_phase is the caller's pageable memory
    }
    CK(c, e);
    return PMX_OK;
}

// ADC with a finite number of bits (dsp4cohdec.m:157-162) on the currents of a realization: M = max over its samples and
// currents of |I|, then I <- round((I + M)/2/M*2^bits)*2*M/2^bits - M, the interpreter's order of operations
__global__ void __launch_bounds__(256) pmx_k_adc_max(const cpx* field, size_t n_cpx, unsigned long long* out) {
    const cpx* fld = field + (size_t)blockIdx.y * n_cpx;
    unsigned long long vmax = 0ull;
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < n_cpx; n += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long k = pmx_pow_key(fmax(fabs(fld[n].x), fabs(fld[n].y)));
        vmax = k > vmax ? k : vmax;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, vmax, o);
        vmax = other > vmax ? other : vmax;
    }
    if ((threadIdx.x & 31) == 0) atomicMax(&out[blockIdx.y], vmax);
}
__global__ void __launch_bounds__(256) pmx_k_adc_quant(cpx* field, size_t n_cpx, const double* maxv, double levels) {
    cpx* fld = field + (size_t)blockIdx.y * n_cpx;
    const double M = maxv[blockIdx.y];
    auto q = [&](double v) { return round((v + M) / 2 / M * levels) * 2 * M / levels - M; };
    for (size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x; n < n_cpx; n += (size_t)gridDim.x * blockDim.x)
        fld[n] = make_double2(q(fld[n].x), q(fld[n].y));
}

extern "C" int pmx_field_quantize(pmx_ctx* c, pmx_devfield* f, int32_t bits) {
    int rc = need_f64(c, f, "pmx_field_quantize");
    if (rc) return rc;
    if (bits < 1 || bits > 52) return set_err(c, PMX_ERR_INVALID, "pmx_field_quantize: bits must be 1..52");
    CK(c, cudaSetDevice(c->device));
    const size_t n_cpx = (size_t)f->nfc * f->nfft * 2;
    unsigned long long* d = nullptr;
    CK(c, cudaMallocAsync(&d, f->batch * sizeof(unsigned long long), c->stream));
    CK(c, cudaMemsetAsync(d, 0, f->batch * sizeof(unsigned long long), c->stream));
    dim3 g((unsigned)std::min<size_t>((n_cpx + 255) / 256, 148 * 4), f->batch);
    pmx_k_adc_max<<<g, 256, 0, c->stream>>>(f->data, n_cpx, d);
    pmx_k_adc_quant<<<g, 256, 0, c->stream>>>(f->data, n_cpx, reinterpret_cast<const double*>(d), ldexp(1.0, bits));   // key == bit pattern
    c->launches += 2;
    cudaError_t e = cudaGetLastError();
    cudaFreeAsync(d, c->stream);
    CK(c, e);
    return PMX_OK;
}

// The whole sample work of receiver_cohmix.m on host buffers, for callers that are not the Python mirror (the MEX gateway)
extern "C" int pmx_cohmix_run(pmx_ctx* c, const pmx_cohmix_desc* d, const pmx_field* sig, double* iric, double* avgeb) {
    if (!c || !d || !sig || !iric) return set_err(c, PMX_ERR_INVALID, "pmx_cohmix_run: null argument");
    if (!d->hf_opt || !d->hf_el) return set_err(c, PMX_ERR_INVALID, "pmx_cohmix_run: both filter responses are required");
    const size_t N = (size_t)d->nfft;
    pmx_devfield *f = nullptr, *tmp = nullptr;
    pmx_plan *fo = nullptr, *fe = nullptr, *fb = nullptr;
    int rc = pmx_field_create(c, d->nfft, 1, 1, d->precision, &f);
    if (rc == PMX_OK) rc = pmx_field_upload(f, sig, 0, 1);
    if (rc == PMX_OK && d->ndfn) rc = pmx_field_modulate(c, f, d->ndfn);
    if (rc == PMX_OK && avgeb) {   // energy of the channel's band before the optical filter (receiver_cohmix.m:174-175,233-234)
        const bool all = d->ndfnl + d->ndfnr >= d->nfft;
        pmx_devfield* src = f;
        if (!all) {
            std::vector<double> band(2 * N, 0.0);
            for (size_t k = 0; k < N; ++k)
                if ((int64_t)k < d->ndfnl || (int64_t)k >= d->nfft - d->ndfnr) band[2 * k] = 1.0;
            rc = pmx_field_create(c, d->nfft, 1, 1, d->precision, &tmp);
            if (rc == PMX_OK) rc = pmx_field_copy_cols(tmp, 0, f, 0, 1);
            if (rc == PMX_OK) rc = pmx_filter_create(c, d->nfft, 1, 1, d->precision, band.data(), 1, &fb);
            if (rc == PMX_OK) rc = pmx_fiber_exec(fb, tmp, nullptr);
            src = tmp;
        }
        if (rc == PMX_OK) rc = pmx_field_mean_power_xy(c, src, &avgeb[0], &avgeb[1]);
    }
    if (rc == PMX_OK) rc = pmx_filter_create(c, d->nfft, 1, 1, d->precision, d->hf_opt, 1, &fo);
    if (rc == PMX_OK) rc = pmx_fiber_exec(fo, f, nullptr);
    if (rc == PMX_OK) rc = pmx_cohmix_exec(c, f, d->lo_ecw, d->lo_detune, d->lo_phase, d->balanced);
    if (rc == PMX_OK) {
        // real(ifft(fft(I) .* H)) of a real I is ifft(fft(I) .* Hh), Hh(k) = (H(k) + conj(H(-k)))/2: the two currents of a
        // polarization ride one complex transform
        std::vector<double> hh(2 * N);
        for (size_t k = 0; k < N; ++k) {
            const size_t m = (N - k) & (N - 1);
            hh[2 * k] = 0.5 * (d->hf_el[2 * k] + d->hf_el[2 * m]);
            hh[2 * k + 1] = 0.5 * (d->hf_el[2 * k + 1] - d->hf_el[2 * m + 1]);
        }
        rc = pmx_filter_create(c, d->nfft, 1, 1, d->precision, hh.data(), 1, &fe);
    }
    if (rc == PMX_OK) rc = pmx_fiber_exec(fe, f, nullptr);
    if (rc == PMX_OK) {   // Iric = [I_x Q_x I_y Q_y], column-major: the planar download
        pmx_field out;
        memset(&out, 0, sizeof out);
        out.layout = PMX_PLANAR;
        out.xr = iric;
        out.xi = iric + N;
        std::vector<double> scratch;
        if (d->two_pol) {
            out.yr = iric + 2 * N;
            out.yi = iric + 3 * N;
        } else {
            scratch.resize(2 * N);
            out.yr = scratch.data();
            out.yi = scratch.data() + N;
        }
        rc = pmx_field_download(f, &out, 0, 1);
    }
    std::string keep = c->error;
    pmx_plan_destroy(fo);
    pmx_plan_destroy(fe);
    pmx_plan_destroy(fb);
    pmx_field_destroy(f);
    pmx_field_destroy(tmp);
    if (rc != PMX_OK) c->error = keep;
    return rc;
}

// ---------------------------------------------------------------------------
// Local-error adaptive step on the scalar path: scalar_a_ssfm / adaptssfm (fiber.m:639-679, 938-1010) and the
// x.dphiadapt variant of scalar_ssfm (fiber.m:588-611).  The accept/reject logic is host code as in the reference;
// nl_step + attenuation, lin_step, the error norm and the Richardson combination run on the resident field.
namespace {
double nextstep_host(double dzmax, double phimax, const double* gam, int nfc, double alphalin, const double* umax) {
    double pmax = 0.0;
    for (int k = 0; k < nfc; ++k) {                        // nextstep, fiber.m:693-715
        const double gp = gam[k] * umax[k];
        pmax = (k == 0) ? gp : std::max(pmax, gp);
    }
    const double leff = phimax / pmax, dl = alphalin * leff;
    if (dl >= 1.0) return dzmax;
    const double step = (alphalin == 0.0) ? leff : (-1.0 / alphalin) * log(1.0 - dl);
    return step > dzmax ? dzmax : step;
}

struct LocalErrorStepper {
    pmx_ctx* c;
    const pmx_fiber_desc* d;
    pmx_devfield *u = nullptr, *uh = nullptr, *ust = nullptr;
    pmx_plan* lin = nullptr;
    double err_tol, safety;
    int nrej = 0;
    ~LocalErrorStepper() {
        pmx_plan_destroy(lin);
        pmx_field_destroy(uh);
        pmx_field_destroy(ust);
        pmx_field_destroy(u);
    }
    int init(pmx_ctx* ctx, const pmx_fiber_desc* desc, const pmx_field* io, double tol, double sf) {
        c = ctx;
        d = desc;
        err_tol = tol;
        safety = sf;
        int rc = pmx_field_create(c, d->nfft, d->nfc, 1, PMX_F64, &u);
        if (rc == PMX_OK) rc = pmx_field_create(c, d->nfft, d->nfc, 1, PMX_F64, &uh);
        if (rc == PMX_OK) rc = pmx_field_create(c, d->nfft, d->nfc, 1, PMX_F64, &ust);
        if (rc != PMX_OK) return rc;
        pmx_field h = *io;
        h.yr = h.yi = nullptr;                             // the scalar path has no Y polarization
        rc = pmx_field_upload(u, &h, 0, 1);
        if (rc != PMX_OK) return rc;
        // lin_step(betat*dz, u) = ifft(fft(u).*fastexp(-betat*dz)): a one-step plan of the same dispersion, no loss
        pmx_fiber_desc l = *d;
        l.batch = 1;
        l.precision = PMX_F64;
        l.fls[1] = l.fls[2] = l.fls[3] = 0;
        l.dphimaxt = INFINITY;
        l.dzmaxt = l.length;
        l.alphalin = 0.0;
        l.manakov = 0;
        l.nplates = 1;
        l.plate_sets = 1;
        l.db0 = l.theta = l.epsilon = nullptr;
        l.db1 = nullptr;
        l.dgdrms = 0.0;
        l.scalar_field = 1;
        l.z_start = l.dz_first = 0.0;
        return pmx_plan_create(c, &l, &lin);
    }
    int nl(pmx_devfield* f, double dz) {                   // nl_step + u*exp(-halfalpha*dz)
        const double a = d->alphalin;
        const double leff = (a == 0.0) ? dz : (1.0 - exp(-a * dz)) / a;
        return pmx_scalar_nl_exec(c, f, d->gam, leff, exp(-0.5 * a * dz), d->fls[2], d->fls[3]);
    }
    int lstep(pmx_devfield* f, double dz) {
        int rc = pmx_plan_set_length(lin, dz);
        return rc != PMX_OK ? rc : pmx_fiber_exec(lin, f, nullptr);
    }
    int first_step(double* dz, double* umax) {
        int rc = pmx_field_max_power(c, u, umax);
        if (rc == PMX_OK) *dz = nextstep_host(d->dzmaxt, d->dphimaxt, d->gam, d->nfc, d->alphalin, umax);
        return rc;
    }
    // adaptssfm (:966-1009): one step of length dz against two half steps.  The field advances only when accepted.
    int try_step(double dz, bool* accepted, double* prop) {
        const double dz2 = 0.5 * dz, dz4 = 0.25 * dz;
        int rc = pmx_field_broadcast(ust, u);
        if (rc == PMX_OK) rc = pmx_field_broadcast(uh, u);
        if (rc == PMX_OK) rc = nl(u, dz2);
        if (rc == PMX_OK) rc = lstep(u, dz);
        if (rc == PMX_OK) rc = nl(u, dz2);
        if (rc == PMX_OK) rc = nl(uh, dz4);
        if (rc == PMX_OK) rc = lstep(uh, dz2);
        if (rc == PMX_OK) rc = nl(uh, dz2);
        if (rc == PMX_OK) rc = lstep(uh, dz2);
        if (rc == PMX_OK) rc = nl(uh, dz4);
        double md2 = 0.0;
        if (rc == PMX_OK) rc = pmx_field_maxdiff2(c, u, uh, &md2);
        if (rc != PMX_OK) return rc;
        const double est_err = sqrt(md2) / dz;
        *prop = safety * sqrt(err_tol / est_err) * dz;
        if (est_err > err_tol) {                           // reject the step
            ++nrej;
            *accepted = false;
            return pmx_field_broadcast(u, ust);
        }
        *accepted = true;
        return pmx_field_lincomb(c, u, 4.0 / 3.0, uh, 1.0 / 3.0, u);   // Richardson extrapolation
    }
};
}  // namespace

extern "C" int pmx_scalar_adaptive_run(pmx_ctx* c, const pmx_fiber_desc* d, double ltol, double safety, int32_t first_only,
                                       pmx_field* io, pmx_fiber_result* out) {
    if (!c || !d || !io) return set_err(c, PMX_ERR_INVALID, "pmx_scalar_adaptive_run: null argument");
    if (!d->scalar_field || d->fls[1])
        return set_err(c, PMX_ERR_INVALID, "adaptive step available in absence of polarization effects");   // fiber.m:372-374
    if (d->batch != 1) return set_err(c, PMX_ERR_UNSUPPORTED, "the local-error adaptive step takes one realization per call");
    if (d->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "the local-error adaptive step runs in FP64 only");
    if (!(ltol > 0) || !(safety > 0)) return set_err(c, PMX_ERR_INVALID, "ltol and the safety factor must be > 0");
    if (d->nfc > PMX_MAX_NFC) return set_err(c, PMX_ERR_UNSUPPORTED, "nfc=%d outside [1,%d]", d->nfc, PMX_MAX_NFC);
    LocalErrorStepper st;
    int rc = st.init(c, d, io, ltol, safety);
    if (rc != PMX_OK) return rc;
    double dz = 0.0, umax[PMX_MAX_NFC];
    rc = st.first_step(&dz, umax);
    if (rc != PMX_OK) return rc;
    double firstdz = dz;
    int ncycle = 1;
    if (!first_only) {                                     // scalar_a_ssfm, fiber.m:664-678
        double zdone = 0.0;
        while (zdone < d->length) {
            if (zdone + dz > d->length) dz = d->length - zdone;
            bool ok = false;
            double prop = 0.0;
            rc = st.try_step(dz, &ok, &prop);
            if (rc != PMX_OK) return rc;
            if (ok) {
                zdone = zdone + dz;
                ++ncycle;
            }
            dz = prop;
            if (dz > d->dzmaxt) dz = d->dzmaxt;
            if (ncycle + st.nrej > 10000000) return set_err(c, PMX_ERR_NUMERIC, "adaptive step loop did not terminate");
        }
    } else {                                               // scalar_ssfm with tolflag == 1, fiber.m:588-611
        if (d->alphalin == 0.0)
            return set_err(c, PMX_ERR_INVALID, "x.dphiadapt needs attenuation: fiber.m:607 divides (1-exp(-alpha*zdone)) by "
                                               "(1-exp(-alpha*dzini))");
        double dphimaxt = d->dphimaxt;
        if (dz >= d->dzmaxt) {                             // :589-597
            double maxpow = 0.0;
            for (int k = 0; k < d->nfc; ++k) maxpow = (k == 0) ? d->gam[k] * umax[k] : std::max(maxpow, d->gam[k] * umax[k]);
            dphimaxt = maxpow * (1.0 - exp(-d->alphalin * dz)) / d->alphalin;
        }
        const double dzini = dz;
        double zdone = 0.0;
        while (zdone == 0.0) {                             // :600-603
            bool ok = false;
            double prop = 0.0;
            rc = st.try_step(dz, &ok, &prop);
            if (rc != PMX_OK) return rc;
            if (ok) zdone = zdone + dz;
            dz = prop;
            if (st.nrej > 100000) return set_err(c, PMX_ERR_NUMERIC, "adaptive first step did not converge");
        }
        if (dz > d->dzmaxt) dz = d->dzmaxt;                // :604
        dphimaxt = dphimaxt * (1.0 - exp(-d->alphalin * zdone)) / (1.0 - exp(-d->alphalin * dzini));   // :607
        pmx_fiber_desc rest = *d;
        rest.dphimaxt = dphimaxt;
        rest.z_start = zdone;
        rest.dz_first = dz;
        pmx_plan* plan = nullptr;
        rc = pmx_plan_create(c, &rest, &plan);
        double fdz = 0.0;
        int32_t ncyc = 0, ntot = 0, status = 0;
        pmx_fiber_result r = {&fdz, &ncyc, &ntot, &status, nullptr, nullptr, 0};
        if (rc == PMX_OK) rc = pmx_fiber_exec(plan, st.u, &r);
        std::string keep = c->error;
        pmx_plan_destroy(plan);
        if (rc != PMX_OK) {
            c->error = keep;
            g_tls_error = keep;
            return rc;
        }
        firstdz = zdone;                                   // :609-611: the adaptive step counts as one
        ncycle = ncyc + 1;
    }
    pmx_field h = *io;
    std::vector<double> ybuf;
    if (h.layout == PMX_PLANAR) {                          // the download wants all four planes; Y is discarded
        ybuf.resize((size_t)2 * d->nfc * d->nfft);
        if (!h.xi) return set_err(c, PMX_ERR_INVALID, "planar output needs xr and xi");
        h.yr = ybuf.data();
        h.yi = ybuf.data() + (size_t)d->nfc * d->nfft;
    } else {
        ybuf.resize((size_t)2 * d->nfc * d->nfft);
        h.yr = ybuf.data();
    }
    rc = pmx_field_download(st.u, &h, 0, 1);
    if (rc != PMX_OK) return rc;
    if (out) {
        if (out->firstdz) out->firstdz[0] = firstdz;
        if (out->ncycle) out->ncycle[0] = ncycle;
        if (out->ntot) out->ntot[0] = 0;
        if (out->status) out->status[0] = PMX_OK;
    }
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// Digital backpropagation (polmux_ssfm.h, pmx_dbp_desc): a step of length h is the three passes of a forward step --
// pass A without the nonlinear step, pass B with the dispersion negated, pass C' (pmx_k_passC<..., NL = true>) with the scale
// exp(+alpha*h/2)/N and the nonlinear step with gam -> -xi*gam -- in the order N(-xi*gam) L(-h) A(-h), the inverse of the
// forward A(h) L(h) N(h).  The schedule is known when the plan is made: every step's package is built here and the host
// enqueues the whole link without reading anything back.
//
// PMD-aware DBP (pmd = 1): pass B of step j applies the inverse of the forward step's trunk product.  The forward step
// covers plates n_first .. n_first+ntrunk-1 with pieces dzb_first, lcorr, ..., dzb_last (checkstep); its inverse is the
// same product on the table with the plates reversed (n' = nplates-1-n) and db0, db1, betat negated, over the pieces in
// reverse order -- a forward matrix_step of the reversed fiber with n_first' = nplates - n_first - ntrunk and the first
// and last piece swapped.  The partition is the forward run's own, replayed here from the forward steps: a fresh
// checkstep on the reversed coordinate would round differently at the plate boundaries.

// pmx_ctl_next's checkstep on each span's forward steps, same operation order (zprop accumulated step by step, the last
// step ending at the fiber length; the host compiles this without FMA contraction), mirrored; execution order.
static int dbp_geometry(pmx_ctx* c, const pmx_fiber_desc& fd, const pmx_dbp_desc* g, const std::vector<double>& h,
                        const std::vector<int>& nstep, std::vector<DbpGeo>& geo) {
    const int np = fd.nplates;
    const double Lf = fd.length, lcorr = fd.length / np, alpha = fd.alphalin, halfalpha = 0.5 * fd.alphalin;
    const double invN = 1.0 / (double)fd.nfft, ig = g->gain > 0 ? 1.0 / std::sqrt(g->gain) : 1.0;
    size_t total = 0;
    for (int k = 0; k < g->nspan; ++k) total += (size_t)nstep[k];
    if (fd.batch < 1 || fd.batch > 65535)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: PMD-aware DBP takes batches of 1 to 65535, got %d", fd.batch);
    const double bytes = (double)total * fd.batch * sizeof(StepPkg);
    if (bytes > (double)(1u << 30))
        return set_err(c, PMX_ERR_INVALID,
                       "pmx_dbp_create: the step package table of PMD-aware DBP (%zu steps x batch %d x %zu B) exceeds 1 GiB", total,
                       fd.batch, sizeof(StepPkg));
    std::vector<size_t> span0(g->nspan, 0);
    for (int k = 1; k < g->nspan; ++k) span0[k] = span0[k - 1] + nstep[k - 1];
    geo.clear();
    geo.reserve(total);
    std::vector<DbpGeo> fw;
    for (int k = g->nspan - 1; k >= 0; --k) {
        fw.assign(nstep[k], DbpGeo());
        double zprop = 0.0, dz_miss = 0.0;
        int ntot = 0;
        for (int j = 0; j < nstep[k]; ++j) {
            const double dz = h[span0[k] + j];
            zprop = zprop + dz;
            const double zend = (j == nstep[k] - 1) ? Lf : zprop;
            const int nzc = (int)std::ceil(zend / lcorr);
            int ntrunk, nmem;
            double dzb_first, dzb_last;
            if (dz_miss == 0.0) {
                nmem = 0;
                ntrunk = nzc - ntot;
                const double dzlast = dz - lcorr * (double)(ntrunk - 1);
                dzb_first = (ntrunk > 1) ? lcorr : dzlast;
                dzb_last = dzlast;
                dz_miss = lcorr - dzlast;
            } else {
                nmem = 1;
                ntrunk = nzc - ntot + 1;
                if (ntrunk == 1) {
                    dzb_first = dzb_last = dz;
                    dz_miss = dz_miss - dz;
                } else {
                    const double dzlast = (dz - dz_miss) - lcorr * (double)(ntrunk - 2);
                    dzb_first = dz_miss;
                    dzb_last = dzlast;
                    dz_miss = lcorr - dzlast;
                }
            }
            const int n_first = ntot - nmem;
            if (ntrunk > 0 && (ntot + ntrunk - nmem > np || n_first < 0))   // brf.theta(n) index error (fiber.m:910)
                return set_err(c, PMX_ERR_PLATE_INDEX, "pmx_dbp_create: step %d of span %d reaches plate %d of %d", j, k,
                               ntot + ntrunk - nmem, np);
            DbpGeo& G = fw[j];
            G.dz = dz;
            G.leff = (alpha == 0.0) ? dz : (1.0 - std::exp(-alpha * dz)) / alpha;   // fiber.m:827-831
            G.scale = std::exp(halfalpha * dz) * invN * (j == nstep[k] - 1 ? ig : 1.0);
            G.ntrunk = std::max(ntrunk, 0);
            G.n_first = np - n_first - ntrunk;   // mirrored
            G.dzb_first = dzb_last;
            G.dzb_last = dzb_first;
            G.span = k;
            G.bmode = ntrunk > 0 ? (PMX_BM_ENTRY_R | PMX_BM_EXIT_R) : 0;   // laboratory basis between the steps
            ntot += ntrunk - nmem;
        }
        for (int j = nstep[k] - 1; j >= 0; --j) geo.push_back(fw[j]);
    }
    return PMX_OK;
}

// The step packages of a PMD-aware DBP plan, one CTA per (step, realization): the geometry goes into a step control
// block in shared memory and pmx_pkg_fill builds the package from it as the step control does for a forward step.
__global__ void __launch_bounds__(128) pmx_k_dbp_pkg(const DbpGeo* __restrict__ geo, const PlateConst* plates, StepPkg* out,
                                                     FiberConst f, int batch) {
    const int s = blockIdx.x, b = blockIdx.y;
    __shared__ StepCtl c;
    const DbpGeo& G = geo[s];
    StepPkg* g = out + (size_t)s * batch + b;
    if (threadIdx.x == 0) {
        c.dz_cur = G.dz;
        c.leff = G.leff;
        c.scale = G.scale;
        c.dzb_first = G.dzb_first;
        c.dzb_last = G.dzb_last;
        c.ntrunk = G.ntrunk;
        c.n_first = G.n_first;
        c.bmode = G.bmode;
        g->state = PMX_ST_RUN;
    }
    __syncthreads();
    pmx_pkg_fill(&c, g, f, plates + ((size_t)G.span * f.plate_sets + (f.plate_sets > 1 ? b : 0)) * f.nplates);
}

static int dbp_channel_exec(pmx_plan* p, pmx_devfield* fld);

// Filtered DBP (polmux_ssfm.h): the Gaussian H[k] = exp(-(ln 2/2) (k_s/bw)^2) at the signed bin k_s of the plan's grid.
extern "C" int pmx_dbp_set_filter(pmx_plan* p, double bw) {
    if (!(bw >= 0) || !std::isfinite(bw))
        return set_err(p ? p->ctx : nullptr, PMX_ERR_INVALID, "pmx_dbp_set_filter: bw must be finite and >= 0 (0: no filter), got %g", bw);
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "pmx_dbp_set_filter: null plan");
    pmx_ctx* c = p->ctx;
    if (!p->dbp) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_filter: not a digital-backpropagation plan");
    if (p->ch_dbp) return pmx_dbp_set_filter(p->ch_dbp, bw);   // single-channel DBP: the same bins on the M-sample grid
    if (bw > 0 && p->ntaps > 0)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_filter: the plan has FIR taps (pmx_dbp_set_taps); a plan takes one or the other");
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));   // no queued work still reads the old response
    if (p->filt_hn_d) CK(c, cudaFreeAsync(p->filt_hn_d, c->stream));
    p->filt_hn_d = nullptr;
    pmx_plan_destroy(p->filt);
    p->filt = nullptr;
    pmx_field_destroy(p->filt_work);
    p->filt_work = nullptr;
    p->filt_bw = 0.0;
    if (bw == 0.0) return PMX_OK;
    const int64_t N = p->d.nfft;
    const double a = 0.5 * std::log(2.0);
    std::vector<double> H((size_t)N);
    for (int64_t k = 0; k < N; ++k) {
        const double ks = (double)(k < N / 2 ? k : k - N) / bw;
        H[k] = std::exp(-a * (ks * ks));
    }
    int rc = PMX_OK;
    if (p->onchip) {   // H/N: the kernel's inverse transform is unscaled
        for (auto& v : H) v *= p->fc.invN;
        CK(c, cudaMallocAsync(&p->filt_hn_d, H.size() * sizeof(double), c->stream));
        CK(c, cudaMemcpyAsync(p->filt_hn_d, H.data(), H.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    } else {
        std::vector<double> Hc(2 * (size_t)N, 0.0);
        for (int64_t k = 0; k < N; ++k) Hc[2 * k] = H[k];
        const int nw = (p->d.batch * p->d.nfc + 1) / 2;   // two realization-columns per Sa
        rc = pmx_filter_create(c, N, 1, nw, p->d.precision, Hc.data(), 1, &p->filt);
        if (!rc) rc = pmx_field_create(c, N, 1, nw, p->d.precision, &p->filt_work);
        if (rc) {
            pmx_plan_destroy(p->filt);
            p->filt = nullptr;
            return rc;
        }
    }
    p->filt_bw = bw;
    return PMX_OK;
}

// Enhanced split-step DBP (polmux_ssfm.h): the taps c[0..2k] of the FIR on the intensity of every nonlinear step.
extern "C" int pmx_dbp_set_taps(pmx_plan* p, int32_t ntaps, const double* taps) {
    pmx_ctx* c = p ? p->ctx : nullptr;
    if (ntaps < 0 || ntaps > PMX_MAX_TAPS || (ntaps > 0 && ntaps % 2 == 0))
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: ntaps must be odd and at most %d (0: no taps), got %d", PMX_MAX_TAPS, ntaps);
    if (ntaps > 0 && !taps) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: null taps");
    for (int j = 0; j < ntaps; ++j)
        if (!std::isfinite(taps[j])) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: tap %d is not finite", j);
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "pmx_dbp_set_taps: null plan");
    if (!p->dbp) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: not a digital-backpropagation plan");
    if (p->ch_dbp) return pmx_dbp_set_taps(p->ch_dbp, ntaps, taps);   // single-channel DBP: the taps act on the M-sample grid
    if (ntaps > 0 && p->filt_bw > 0)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: the plan has a filter bandwidth (pmx_dbp_set_filter); a plan takes one or the other");
    if (ntaps > p->d.nfft)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_taps: %d taps on a grid of %lld samples", ntaps, (long long)p->d.nfft);
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));   // no queued work still reads the old work field
    pmx_field_destroy(p->tap_work);
    p->tap_work = nullptr;
    p->ntaps = 0;
    p->taps = DbpTaps{};
    if (ntaps == 0) return PMX_OK;
    if (!p->onchip) {
        const int nw = (p->d.batch * p->d.nfc + 1) / 2;   // two realization-columns per Sa
        const int rc = pmx_field_create(c, p->d.nfft, 1, nw, p->d.precision, &p->tap_work);
        if (rc) return rc;
    }
    p->taps.k = ntaps / 2;
    for (int j = 0; j < ntaps; ++j) p->taps.c[j] = taps[j];
    p->ntaps = ntaps;
    return PMX_OK;
}

extern "C" int pmx_dbp_set_plates(pmx_plan* p, int32_t sets, const double* db0, const double* theta, const double* epsilon) {
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "pmx_dbp_set_plates: null plan");
    if (p->ch_dbp) return pmx_dbp_set_plates(p->ch_dbp, sets, db0, theta, epsilon);   // single-channel DBP: its M-sample plan
    pmx_ctx* c = p->ctx;
    if (!p->dbp_pmd) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_plates: not a PMD-aware DBP plan (pmx_dbp_create with pmd = 1)");
    if (sets != 1 && sets != p->d.batch)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_plates: plate_sets must be 1 or batch (%d), got %d", p->d.batch, sets);
    if (!db0 || !theta || !epsilon) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_set_plates: db0, theta and epsilon are required");
    const int np = p->d.nplates;
    const size_t per = (size_t)sets * np;
    std::vector<double> r[3];
    for (auto& v : r) v.resize(per);
    std::vector<PlateConst> all, one;
    all.reserve((size_t)p->dbp_nspan * per);
    for (int k = 0; k < p->dbp_nspan; ++k) {   // reversed plate order, db0 negated (inverse_pmd)
        for (int s = 0; s < sets; ++s)
            for (int n = 0; n < np; ++n) {
                const size_t src = (size_t)k * per + (size_t)s * np + (np - 1 - n), dst = (size_t)s * np + n;
                r[0][dst] = -db0[src];
                r[1][dst] = theta[src];
                r[2][dst] = epsilon[src];
            }
        fill_plates(p->d, sets, r[0].data(), r[1].data(), r[2].data(), one);
        all.insert(all.end(), one.begin(), one.end());
    }
    CK(c, cudaSetDevice(c->device));
    if (p->plates) CK(c, cudaFreeAsync(p->plates, c->stream));
    p->plates = nullptr;
    p->dbp_plates_set = false;
    CK(c, cudaMallocAsync(&p->plates, all.size() * sizeof(PlateConst), c->stream));
    CK(c, cudaMemcpyAsync(p->plates, all.data(), all.size() * sizeof(PlateConst), cudaMemcpyHostToDevice, c->stream));
    p->fc.plate_sets = p->fc_a.plate_sets = p->fc_c.plate_sets = sets;
    pmx_k_dbp_pkg<<<dim3((unsigned)p->sched_idx.size(), (unsigned)p->d.batch), 128, 0, c->stream>>>(p->geo_d, p->plates, p->sched,
                                                                                                     p->fc, p->d.batch);
    c->launches++;
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(c->stream));   // the host vectors go away
    p->dbp_plates_set = true;
    return PMX_OK;
}

// An on-chip DBP plan walks its step table on the device: the package index of every step and, PMD-aware, its span.
static int dbp_upload_steps(pmx_plan* p) {
    if (!p->onchip) return PMX_OK;
    pmx_ctx* c = p->ctx;
    const size_t n = p->sched_idx.size();
    cudaError_t err = cudaMallocAsync(&p->sched_idx_d, n * sizeof(int), c->stream);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(p->sched_idx_d, p->sched_idx.data(), n * sizeof(int), cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess && p->dbp_pmd) {
        err = cudaMallocAsync(&p->sched_span_d, n * sizeof(int), c->stream);
        if (err == cudaSuccess)
            err = cudaMemcpyAsync(p->sched_span_d, p->sched_span.data(), n * sizeof(int), cudaMemcpyHostToDevice, c->stream);
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
    if (err != cudaSuccess) return set_err(c, PMX_ERR_CUDA, "pmx_dbp_create: step index table: %s", cudaGetErrorString(err));
    return PMX_OK;
}

extern "C" int pmx_dbp_create(pmx_ctx* c, const pmx_fiber_desc* fd, const pmx_dbp_desc* g, pmx_plan** out) {
    // (the descriptors are checked before the context, so that the checks run without a device)
    if (!fd || !g || !out) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: null argument");
    *out = nullptr;
    // The route follows from the field: the scalar path and fields below 2^12 samples run the whole link in one launch of
    // the on-chip kernel (one CTA per column, the columns of a realization in one cluster: at most 8), two-polarization
    // fields of 2^12 samples and more the three passes of every step.
    const bool scalar = fd->scalar_field != 0;
    if (fd->fls[3] && !scalar) return set_err(c, PMX_ERR_XPM_VECTOR, "The CNLSE with separate fields is not yet implemented");
    const int lg = ilog2_exact(fd->nfft);
    if (scalar && (lg < 6 || lg > 12))
        return set_err(c, PMX_ERR_UNSUPPORTED,
                       "digital backpropagation on the scalar path: nfft=%lld, built for powers of two from 2^6 to 2^12",
                       (long long)fd->nfft);
    if (lg < 6 || lg > 24)
        return set_err(c, PMX_ERR_UNSUPPORTED, "digital backpropagation: nfft=%lld, built for powers of two from 2^6 to 2^24",
                       (long long)fd->nfft);
    const bool onchip = scalar || lg < 12;
    if (onchip && (fd->nfc < 1 || fd->nfc > 8))
        return set_err(c, PMX_ERR_UNSUPPORTED,
                       "digital backpropagation %s: nfc=%d, built for 1 to 8 columns (the columns of a realization form one "
                       "thread-block cluster)", scalar ? "on the scalar path" : "below 2^12 samples", fd->nfc);
    if (g->nspan < 1) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: nspan must be >= 1");
    if (!std::isfinite(g->xi)) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: xi must be finite");
    if (!(g->gain >= 0) || !std::isfinite(g->gain)) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: gain must be >= 0 (0: none)");
    if (!(fd->length > 0) || !std::isfinite(fd->length)) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: length must be > 0");
    if (g->pmd != 0 && g->pmd != 1) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: pmd must be 0 or 1");
    const bool pmd = g->pmd != 0;
    if (pmd && !fd->fls[1])
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: PMD-aware DBP (pmd = 1) needs the fiber's 'p' flag");
    if (pmd && fd->nplates < 1)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: PMD-aware DBP (pmd = 1) needs nplates >= 1");
    // the steps of every span, forward order
    std::vector<double> h;
    std::vector<int> nstep(g->nspan);
    if (g->steps_per_span > 0) {
        if ((long long)g->steps_per_span * g->nspan > 10000000)
            return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: more than 10^7 steps in all");
        for (int k = 0; k < g->nspan; ++k) {
            nstep[k] = g->steps_per_span;
            for (int j = 0; j < g->steps_per_span; ++j) h.push_back(fd->length / g->steps_per_span);
        }
    } else if (g->steps_per_span < 0) {
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: steps_per_span must be >= 0");
    } else {
        if (!g->span_steps || !g->step_len)
            return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: an explicit schedule needs span_steps and step_len");
        size_t o = 0;
        for (int k = 0; k < g->nspan; ++k) {
            const int n = g->span_steps[k];
            if (n < 1 || (long long)o + n > 10000000)
                return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: span %d has %d steps (at least one, at most 10^7 in all)", k, n);
            double sum = 0;
            for (int j = 0; j < n; ++j, ++o) {
                const double v = g->step_len[o];
                if (!(v >= 0) || !std::isfinite(v))
                    return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: step %d of span %d is negative or not finite (%g)", j, k, v);
                sum += v;
                h.push_back(v);
            }
            if (std::fabs(sum - fd->length) > 1e-9 * fd->length)
                return set_err(c, PMX_ERR_INVALID, "pmx_dbp_create: the steps of span %d sum to %.17g, not the fiber length %.17g", k,
                               sum, fd->length);
            nstep[k] = n;
        }
    }
    std::vector<DbpGeo> geo;
    if (pmd) {
        const int rc = dbp_geometry(c, *fd, g, h, nstep, geo);
        if (rc) return rc;
    }
    if (!c) return set_err(nullptr, PMX_ERR_INVALID, "pmx_dbp_create: null context");
    // the virtual fiber: no XPM, dispersion negated, one step at a time; without pmd no PMD either, with pmd the plates
    // come from pmx_dbp_set_plates and db1 (dgdrms) is negated
    const double zero1 = 0.0;
    std::vector<double> nb1, nb2, nbt, ndb1;
    pmx_fiber_desc e = *fd;
    e.fls[1] = pmd ? 1 : 0;
    e.nplates = pmd ? fd->nplates : 1;
    e.plate_sets = 1;
    e.db0 = e.theta = e.epsilon = pmd ? nullptr : &zero1;
    e.db1 = nullptr;
    e.dgdrms = pmd ? -fd->dgdrms : 0.0;
    if (pmd && fd->disp_mode != PMX_DISP_SCALAR && fd->db1 && fd->nfc >= 1 && fd->nfc <= PMX_MAX_NFC) {
        ndb1.assign(fd->db1, fd->db1 + (size_t)fd->nfc * fd->nfft);
        for (auto& v : ndb1) v = -v;
        e.db1 = ndb1.data();
    }
    e.dphimaxt = INFINITY;
    e.dzmaxt = fd->length;
    e.z_start = e.dz_first = 0.0;
    if (fd->disp_mode == PMX_DISP_SCALAR) {
        if (!fd->beta1 || !fd->beta2) return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode needs beta1 and beta2");
        for (int k = 0; k < std::max(fd->nfc, 0) && k < PMX_MAX_NFC; ++k) {
            nb1.push_back(-fd->beta1[k]);
            nb2.push_back(-fd->beta2[k]);
        }
        e.beta1 = nb1.data();
        e.beta2 = nb2.data();
        e.b30 = -fd->b30;
    } else if (fd->betat && fd->nfc >= 1 && fd->nfc <= PMX_MAX_NFC) {
        nbt.assign(fd->betat, fd->betat + (size_t)fd->nfc * fd->nfft);
        for (auto& v : nbt) v = -v;
        e.betat = nbt.data();
    }
    pmx_plan* p = nullptr;
    int rc = plan_create(c, &e, &p, onchip ? PLAN_ONCHIP : PLAN_PASSES);
    if (rc) return rc;
    p->dbp = true;
    p->fc_a = p->fc;
    p->fc_a.spm = 0;                            // pass A: the transform only
    p->fc_c = p->fc;
    for (int k = 0; k < p->fc.nfc; ++k) p->fc_c.gam[k] = -g->xi * p->fc.gam[k];   // (gam carries the Manakov 8/9)
    if (pmd) {   // one package per step and realization, built by pmx_dbp_set_plates from the geometry table
        const size_t bytes = geo.size() * (size_t)p->d.batch * sizeof(StepPkg);
        cudaError_t err = cudaMallocAsync(&p->sched, bytes, c->stream);
        if (err == cudaSuccess) err = cudaMemsetAsync(p->sched, 0, bytes, c->stream);
        if (err == cudaSuccess) err = cudaMallocAsync(&p->geo_d, geo.size() * sizeof(DbpGeo), c->stream);
        if (err == cudaSuccess)
            err = cudaMemcpyAsync(p->geo_d, geo.data(), geo.size() * sizeof(DbpGeo), cudaMemcpyHostToDevice, c->stream);
        if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
        if (err != cudaSuccess) {
            pmx_plan_destroy(p);
            return set_err(c, PMX_ERR_CUDA, "pmx_dbp_create: step table: %s", cudaGetErrorString(err));
        }
        p->dbp_pmd = true;
        p->dbp_nspan = g->nspan;
        for (size_t s = 0; s < geo.size(); ++s) {
            p->sched_idx.push_back((int)s);
            p->sched_span.push_back(geo[s].span);
        }
        rc = dbp_upload_steps(p);
        if (rc) {
            pmx_plan_destroy(p);
            return rc;
        }
        *out = p;
        return PMX_OK;
    }
    // step packages in execution order: spans last first, each span's steps reversed; the amplifier's 1/sqrt(G) joins the
    // scale of a span's first step.  Equal packages are stored once.
    const FiberConst& f = p->fc;
    const double ig = g->gain > 0 ? 1.0 / std::sqrt(g->gain) : 1.0;
    std::vector<StepPkg> uniq;
    std::map<std::pair<double, double>, int> seen;
    std::vector<size_t> span0(g->nspan, 0);
    for (int k = 1; k < g->nspan; ++k) span0[k] = span0[k - 1] + nstep[k - 1];
    for (int k = g->nspan - 1; k >= 0; --k)
        for (int j = nstep[k] - 1; j >= 0; --j) {
            const double hh = h[span0[k] + j];
            const double scale = std::exp(f.halfalpha * hh) * f.invN * (j == nstep[k] - 1 ? ig : 1.0);
            auto it = seen.find({hh, scale});
            if (it == seen.end()) {
                StepPkg s;
                memset(&s, 0, sizeof s);
                s.dz_cur = s.dzb_first = s.dzb_last = hh;
                s.leff = (f.alphalin == 0.0) ? hh : (1.0 - std::exp(-f.alphalin * hh)) / f.alphalin;   // fiber.m:827-831
                s.scale = scale;
                s.ntrunk = 1;
                s.state = PMX_ST_RUN;
                if (f.disp_scalar && f.gvd_any) {   // third difference of the common phase (pmx_ctl_step)
                    const double a3 = -(hh * (6.0 * f.b30_6) * f.domega * f.domega * f.domega);
                    s.gd3_r = std::cos(a3);
                    s.gd3_i = std::sin(a3);
                }
                it = seen.emplace(std::make_pair(hh, scale), (int)uniq.size()).first;
                uniq.push_back(s);
            }
            p->sched_idx.push_back(it->second);
        }
    const int batch = p->d.batch;
    std::vector<StepPkg> tab(uniq.size() * (size_t)batch);
    for (size_t u = 0; u < uniq.size(); ++u)
        for (int b = 0; b < batch; ++b) tab[u * batch + b] = uniq[u];
    cudaError_t err = cudaMallocAsync(&p->sched, tab.size() * sizeof(StepPkg), c->stream);
    if (err == cudaSuccess) err = cudaMemcpyAsync(p->sched, tab.data(), tab.size() * sizeof(StepPkg), cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
    if (err != cudaSuccess) {
        pmx_plan_destroy(p);
        return set_err(c, PMX_ERR_CUDA, "pmx_dbp_create: step table: %s", cudaGetErrorString(err));
    }
    rc = dbp_upload_steps(p);
    if (rc) {
        pmx_plan_destroy(p);
        return rc;
    }
    *out = p;
    return PMX_OK;
}

// Filtered and enhanced split-step DBP on the three passes, per step: passes A and B, pass C' without its nonlinear
// epilogue (spm = 0 makes pmx_nl_step a no-op), the intensity into the work field, then either the filter plan on it and
// the nonlinear step from the filtered intensity, or the nonlinear step from the FIR of the taps (pmx_k_dbp_nl_fir).  The
// filter plan runs on the context's stream, so the realization groups join before it.
static int dbp_filtered_passes(pmx_plan* p, pmx_devfield* fld, const PassParams& pa, PassGroups& gs) {
    pmx_ctx* c = p->ctx;
    const int batch = p->d.batch;
    FiberConst fc_lin = p->fc_c;
    fc_lin.spm = 0;
    const dim3 grid((unsigned)std::min<int64_t>((p->d.nfft + 255) / 256, 148 * 4), (unsigned)(batch * p->d.nfc));
    int rev[4] = {1, 1, 1, 1};
    for (size_t s = 0; s < p->sched_idx.size(); ++s) {
        StepPkg* pk = p->sched + (size_t)p->sched_idx[s] * batch;
        int rc = fork_groups(c, gs.n);
        if (rc) return rc;
        for (int gi = 0; gi < gs.n; ++gi) {
            PassGroup& G = gs.g[gi];
            G.pA.pkg = G.pB.pkg = pk + G.b0;
            if (p->dbp_pmd)
                G.pB.plates = p->plates + ((size_t)p->sched_span[s] * p->fc.plate_sets + (p->fc.plate_sets > 1 ? G.b0 : 0)) *
                                              p->fc.nplates;
            G.pA.reverse = (rev[gi] ^= 1);
            CK(c, p->tA->passA(G.gA, G.st, G.pA, p->fc_a, fld->map_rows));
            G.pB.reverse = (rev[gi] ^= 1);
            CK(c, p->tB->passB(G.gB, G.st, G.pB, p->fc_c, fld->map_cols));
            G.pA.reverse = (rev[gi] ^= 1);
            CK(c, p->tA->passC_nl(G.gC, G.st, G.pA, fc_lin, fld->map_rows));
            c->launches += 3;
        }
        CK(c, cudaGetLastError());
        rc = join_groups(c, gs.n);
        if (rc) return rc;
        if (p->ntaps > 0) {
            p->tA->dbp_intensity(grid, c->stream, pa, p->fc_c, p->tap_work->data);
            CK(c, p->tA->dbp_nl_fir(c->stream, pa, p->fc_c, p->tap_work->data, pk, p->taps));
            c->launches += 2;
            continue;
        }
        p->tA->dbp_intensity(grid, c->stream, pa, p->fc_c, p->filt_work->data);
        c->launches++;
        CK(c, cudaGetLastError());
        rc = pmx_fiber_exec(p->filt, p->filt_work, nullptr);
        if (rc) return rc;
        p->tA->dbp_nl_filt(grid, c->stream, pa, p->fc_c, p->filt_work->data, pk);
        c->launches++;
        CK(c, cudaGetLastError());
    }
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" int pmx_dbp_exec(pmx_plan* p, pmx_devfield* fld) {
    if (!p || !fld) return set_err(nullptr, PMX_ERR_INVALID, "pmx_dbp_exec: null argument");
    pmx_ctx* c = p->ctx;
    if (!p->dbp) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_exec: the plan was not made by pmx_dbp_create");
    if (p->ch_dbp) return dbp_channel_exec(p, fld);
    if (p->dbp_pmd && !p->dbp_plates_set)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_exec: a PMD-aware plan needs its plates (pmx_dbp_set_plates) first");
    int rc = check_field(p, fld);
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    const int batch = p->d.batch;
    PassParams pa, pA, pB;
    rc = pass_params(p, fld, pa, pA, pB);
    if (rc) return rc;
    if (p->onchip) {   // small field or scalar path: the whole link of every realization in one launch
        PassParams q = pa;
        rc = get_stage_tw(c, p->tB, &q.tw_stage);
        if (rc) return rc;
        q.N1 = 1;
        q.N2 = (int)p->d.nfft;
        q.log2N1 = fld->log2N1;   // layout of the resident column (transposed for 2^12, natural below)
        q.log2N2 = fld->log2N2;
        DbpSteps ds;
        ds.pkg = p->sched;
        ds.idx = p->sched_idx_d;
        ds.span = p->dbp_pmd ? p->sched_span_d : nullptr;
        ds.nstep = (int)p->sched_idx.size();
        ds.pkg_bytes = p->dbp_pmd ? (int)sizeof(StepPkg) : PMX_PKG_HEAD;   // without PMD no step reads past the header
        ds.plate_stride = (long long)p->fc.plate_sets * p->fc.nplates;
        if (p->ntaps > 0)
            CK(c, p->tB->onchip_dbp_taps(p->d.nfc, batch, c->stream, q, p->fc_c, DbpTapSteps{ds, p->taps}));
        else if (p->filt_bw > 0)
            CK(c, p->tB->onchip_dbp_filt(p->d.nfc, batch, c->stream, q, p->fc_c, DbpFiltSteps{ds, p->filt_hn_d}));
        else
            CK(c, p->tB->onchip_dbp(p->d.nfc, batch, c->stream, q, p->fc_c, ds));
        c->launches += 1;
        CK(c, cudaStreamSynchronize(c->stream));
        return PMX_OK;
    }
    // realization groups and dependent launches as in pmx_fiber_exec; pass C' has an occupancy of its own
    PassGroups gs;
    rc = plan_groups(p, fld, pa, pA, pB, c->setup_done[p->N1 + 65536 * p->d.precision].cnl, true, gs);
    if (rc) return rc;
    if (p->filt_bw > 0 || p->ntaps > 0) return dbp_filtered_passes(p, fld, pa, gs);
    rc = fork_groups(c, gs.n);
    if (rc) return rc;
    int rev[4] = {1, 1, 1, 1};
    for (size_t s = 0; s < p->sched_idx.size(); ++s) {
        StepPkg* pk = p->sched + (size_t)p->sched_idx[s] * batch;
        for (int gi = 0; gi < gs.n; ++gi) {
            PassGroup& G = gs.g[gi];
            G.pA.pkg = G.pB.pkg = pk + G.b0;
            if (p->dbp_pmd)   // the step's span: trunks beyond the package's PMX_PKG_PLATES are read from its table
                G.pB.plates = p->plates + ((size_t)p->sched_span[s] * p->fc.plate_sets + (p->fc.plate_sets > 1 ? G.b0 : 0)) *
                                              p->fc.nplates;
            G.pA.reverse = (rev[gi] ^= 1);   // serpentine tile order, as in pmx_fiber_exec
            CK(c, p->tA->passA(G.gA, G.st, G.pA, p->fc_a, fld->map_rows));
            G.pB.reverse = (rev[gi] ^= 1);
            CK(c, p->tB->passB(G.gB, G.st, G.pB, p->fc_c, fld->map_cols));
            G.pA.reverse = (rev[gi] ^= 1);
            CK(c, p->tA->passC_nl(G.gC, G.st, G.pA, p->fc_c, fld->map_rows));
            c->launches += 3;
        }
    }
    CK(c, cudaGetLastError());
    rc = join_groups(c, gs.n);
    if (rc) return rc;
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// One channel of a one-column multiplex at M = N/r samples (pmx_dbp_band), shared by single-channel DBP and single-channel
// PB-NLC: down = band filter at N, gather to M; up = stuff back to N, band filter.

// The N-grid bin of M-grid bin j: (k - m) mod N for the signed k of j (m the channel's shift mod N)
static size_t band_bin(int64_t j, int64_t M, int64_t N, long long m) {
    return (size_t)((((j < M / 2 ? j : j - M) - m) % N + N) % N);
}

// The band filter at N samples: H = 1 on the channel's M bins
static int band_filter_create(pmx_ctx* c, int64_t N, int64_t M, long long m, int batch, int precision, pmx_plan** out) {
    std::vector<double> H(2 * (size_t)N, 0.0);
    for (int64_t j = 0; j < M; ++j) H[2 * band_bin(j, M, N, m)] = 1.0;
    return pmx_filter_create(c, N, 1, batch, precision, H.data(), 1, out);
}

// fld (N samples) -> w (M samples): the band filter in place on fld, then the channel at baseband, decimated, into w
static int band_down(pmx_plan* band, pmx_devfield* fld, pmx_devfield* w, int lr, long long m) {
    pmx_ctx* c = band->ctx;
    int rc = check_field(band, fld);   // device, precision, nfft, one column, batch
    if (!rc) rc = pmx_fiber_exec(band, fld, nullptr);
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    const size_t N = (size_t)fld->nfft, M = (size_t)w->nfft;
    const dim3 gm((unsigned)std::min<size_t>((M + 255) / 256, 148 * 8), fld->batch);
    if (fld->precision == PMX_F32)
        pmx_k_band_gather<float2><<<gm, 256, 0, c->stream>>>(reinterpret_cast<const float2*>(fld->data), fld->log2N1, fld->log2N2,
                                                              reinterpret_cast<float2*>(w->data), w->log2N1, w->log2N2, N, lr, m);
    else
        pmx_k_band_gather<double2><<<gm, 256, 0, c->stream>>>(reinterpret_cast<const double2*>(fld->data), fld->log2N1,
                                                               fld->log2N2, reinterpret_cast<double2*>(w->data), w->log2N1,
                                                               w->log2N2, N, lr, m);
    c->launches++;
    CK(c, cudaGetLastError());
    return PMX_OK;
}

// w (M samples) -> fld (N samples): stuffed back onto the channel's bins, then the band filter in place on fld
static int band_up(pmx_plan* band, pmx_devfield* w, pmx_devfield* fld, int lr, long long m) {
    pmx_ctx* c = band->ctx;
    const size_t N = (size_t)fld->nfft;
    const dim3 gn((unsigned)std::min<size_t>((N + 255) / 256, 148 * 8), fld->batch);
    if (fld->precision == PMX_F32)
        pmx_k_band_stuff<float2><<<gn, 256, 0, c->stream>>>(reinterpret_cast<const float2*>(w->data), w->log2N1, w->log2N2,
                                                             reinterpret_cast<float2*>(fld->data), fld->log2N1, fld->log2N2, N,
                                                             lr, m);
    else
        pmx_k_band_stuff<double2><<<gn, 256, 0, c->stream>>>(reinterpret_cast<const double2*>(w->data), w->log2N1, w->log2N2,
                                                              reinterpret_cast<double2*>(fld->data), fld->log2N1, fld->log2N2, N,
                                                              lr, m);
    c->launches++;
    CK(c, cudaGetLastError());
    return pmx_fiber_exec(band, fld, nullptr);
}

// Single-channel DBP (polmux_ssfm.h, pmx_dbp_band): down, the DBP plan of M samples, up.  The M-sample plan is an ordinary
// pmx_dbp_create plan on vector tables: the channel's own dispersion, so that nothing in the step kernels knows about the
// channel's offset.
extern "C" int pmx_dbp_channel_create(pmx_ctx* c, const pmx_fiber_desc* fd, const pmx_dbp_desc* g, const pmx_dbp_band* band,
                                      pmx_plan** out) {
    // (checked before the context, like pmx_dbp_create)
    if (!fd || !g || !band || !out) return set_err(c, PMX_ERR_INVALID, "pmx_dbp_channel_create: null argument");
    *out = nullptr;
    const int lg = ilog2_exact(fd->nfft), lr = ilog2_exact(band->decim);
    if (band->decim < 2 || lr < 1)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_channel_create: decim=%d, must be a power of two >= 2", band->decim);
    if (lg < 6 || lg > 24)
        return set_err(c, PMX_ERR_UNSUPPORTED, "single-channel digital backpropagation: nfft=%lld, built for powers of two from "
                       "2^6 to 2^24", (long long)fd->nfft);
    if (lg - lr < 6)
        return set_err(c, PMX_ERR_INVALID, "pmx_dbp_channel_create: nfft/decim = %lld/%d samples, at least 2^6 are needed",
                       (long long)fd->nfft, band->decim);
    if (fd->nfc != 1)
        return set_err(c, PMX_ERR_UNSUPPORTED, "single-channel digital backpropagation: nfc=%d, built for one column holding "
                       "every channel (a 'unique' multiplex)", fd->nfc);
    const int64_t N = fd->nfft, M = N >> lr;
    if (fd->scalar_field && lg - lr > 12)
        return set_err(c, PMX_ERR_UNSUPPORTED, "single-channel digital backpropagation on the scalar path: nfft/decim=%lld, "
                       "built for at most 2^12 samples", (long long)M);
    const long long m = ((band->shift % N) + N) % N;
    auto bin = [&](int64_t j) { return band_bin(j, M, N, m); };
    const bool pmd = g->pmd == 1 && fd->fls[1];
    std::vector<double> bt((size_t)M), d1;
    if (fd->disp_mode == PMX_DISP_SCALAR) {
        if (!fd->beta1 || !fd->beta2) return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode needs beta1 and beta2");
        if (fd->nsymb <= 0 || fd->nt <= 0 || (int64_t)fd->nsymb * fd->nt != N)
            return set_err(c, PMX_ERR_INVALID, "scalar dispersion mode: nsymb*nt must equal nfft");
        // fiber.m:350-358 at the channel's bins, in the host's operation order: FN = fftshift(-NT/2 + (0:N-1)/NSYMB)
        // (reset_all.m:153), omega = 2*pi*symbolrate*FN
        if (pmd) d1.resize((size_t)M);
        for (int64_t j = 0; j < M; ++j) {
            const int64_t i = (int64_t)((bin(j) + (size_t)(N / 2)) & (size_t)(N - 1));   // index before the fftshift
            const double fn = -fd->nt / 2.0 + (double)i * (1.0 / fd->nsymb);
            const double om = 2 * M_PI * fd->symbolrate * fn;
            bt[j] = om * fd->beta1[0] + 0.5 * (om * om) * fd->beta2[0] + std::pow(om, 3) * fd->b30 / 6;
            if (pmd) d1[j] = fd->dgdrms * om;
        }
    } else {
        if (!fd->betat) return set_err(c, PMX_ERR_INVALID, "betat is required in vector dispersion mode");
        for (int64_t j = 0; j < M; ++j) bt[j] = fd->betat[bin(j)];
        if (pmd && fd->db1) {
            d1.resize((size_t)M);
            for (int64_t j = 0; j < M; ++j) d1[j] = fd->db1[bin(j)];
        }
    }
    pmx_fiber_desc e = *fd;
    e.nfft = M;
    e.disp_mode = PMX_DISP_VECTOR;
    e.betat = bt.data();
    e.db1 = d1.empty() ? nullptr : d1.data();
    pmx_plan* inner = nullptr;
    int rc = pmx_dbp_create(c, &e, g, &inner);   // validates the rest before it needs the context
    if (rc) return rc;
    pmx_plan* p = new (std::nothrow) pmx_plan();
    if (!p) {
        pmx_plan_destroy(inner);
        return set_err(c, PMX_ERR_INVALID, "out of host memory");
    }
    p->ctx = c;
    p->d = *fd;
    p->d.gam = p->d.db0 = p->d.theta = p->d.epsilon = p->d.betat = p->d.db1 = p->d.beta1 = p->d.beta2 = nullptr;
    p->dbp = true;
    p->ch_dbp = inner;
    p->ch_shift = m;
    p->ch_log2r = lr;
    rc = band_filter_create(c, N, M, m, fd->batch, fd->precision, &p->ch_band);
    if (!rc) rc = pmx_field_create(c, M, 1, fd->batch, fd->precision, &p->ch_work);
    if (rc) {
        pmx_plan_destroy(p);
        return rc;
    }
    *out = p;
    return PMX_OK;
}

static int dbp_channel_exec(pmx_plan* p, pmx_devfield* fld) {
    int rc = band_down(p->ch_band, fld, p->ch_work, p->ch_log2r, p->ch_shift);
    if (!rc) rc = pmx_dbp_exec(p->ch_dbp, p->ch_work);
    if (!rc) rc = band_up(p->ch_band, p->ch_work, fld, p->ch_log2r, p->ch_shift);
    return rc;
}

// ---------------------------------------------------------------------------
// Perturbation-based nonlinearity compensation (pmx_pb_create / pmx_pb_exec, see the header): projection onto the pulses,
// the first-order triplet sum at the symbol rate, reconstruction.  FP64, one-column fields, either resident layout.
struct PbCoef {   // one entry of the list, C' = -j*gamma*s^2*C folded on the host
    double cr, ci;
    int m, n;
};
struct pmx_pb_plan {
    pmx_ctx* ctx;
    int64_t nfft;
    int nsymb, nt, batch, npulse, ncoef, K;
    double wa, wb, wc, xi, inorm;
    double* pulse = nullptr;  // [npulse]
    PbCoef* coef = nullptr;   // [ncoef]
    cpx* A = nullptr;         // [batch][2][nsymb] projected symbols
    cpx* D = nullptr;         // [batch][2][nsymb] perturbation
    // single-channel PB-NLC (pmx_pb_channel_create): the stage at nfft/decim samples, the band filter at nfft, the work field
    // of the decimated channel, and the channel's shift (mod nfft) and log2(decim)
    pmx_pb_plan* ch_pb = nullptr;
    pmx_plan* ch_band = nullptr;
    pmx_devfield* ch_work = nullptr;
    long long ch_shift = 0;
    int ch_log2r = 0;
    // XPM-aware single-channel PB-NLC (pmx_pb_xpm_create), on the channel plan: the interferers' shifts (mod nfft) and band
    // filters, the copy of the field each is cut from, their symbols B [nint][batch][2][nsymb], their folded tables
    // concatenated with offsets [nint+1], the halos of the XPM kernel (max |m|; max of |n| and |m+n|) and the weights
    int xpm_n = 0, xpm_ha = 0, xpm_hb = 0;
    long long xpm_shift[PMX_PB_XPM_MAX_INT] = {};
    pmx_plan* xpm_band[PMX_PB_XPM_MAX_INT] = {};
    pmx_devfield* xpm_copy = nullptr;
    cpx* xpm_B = nullptr;
    PbCoef* xpm_coef = nullptr;
    int* xpm_off = nullptr;
    double xpm_w[4] = {};
};

// A^{x,y}_k = sum_j p[j] u[(k*nt - np/2 + j) mod N] * inorm (j ascending); thread per symbol, grid.y the realization
__global__ void __launch_bounds__(256) pmx_k_pb_project(const cpx* __restrict__ field, size_t N, int l1, int l2, int nsymb,
                                                        int nt, const double* __restrict__ pulse, int np, double inorm,
                                                        cpx* __restrict__ A) {
    const int b = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nsymb) return;
    const cpx* fld = field + (size_t)b * N * 2;
    const size_t t0 = ((size_t)k * nt + N - (size_t)(np / 2)) & (N - 1);
    double axr = 0, axi = 0, ayr = 0, ayi = 0;
    for (int j = 0; j < np; ++j) {
        cpx x, y;
        ld_sa(fld + 2 * pmx_mem_index((t0 + j) & (N - 1), l1, l2), x, y);
        const double p = pulse[j];
        axr = fma(p, x.x, axr);
        axi = fma(p, x.y, axi);
        ayr = fma(p, y.x, ayr);
        ayi = fma(p, y.y, ayi);
    }
    A[(size_t)(2 * b) * nsymb + k] = make_double2(axr * inorm, axi * inorm);
    A[(size_t)(2 * b + 1) * nsymb + k] = make_double2(ayr * inorm, ayi * inorm);
}

// The triplet sum.  A CTA takes PMX_PB_TILE symbols of one realization and lands them with a 2K-symbol halo on either side
// (indices k+m, k+n, k+m+n with |m|, |n| <= K), both polarizations, in shared memory.  A thread owns PMX_PB_RB symbols, so
// every coefficient it reads (the same entry for all threads: a broadcast) feeds PMX_PB_RB independent sums.  Its symbols are
// PMX_PB_THREADS apart rather than adjacent: the loads of one coefficient share nothing between neighbouring symbols, and
// a warp then reads 32 consecutive 16-byte samples per load, without bank conflicts.  Per entry and symbol the loop runs
// 4 complex products xx, yy, xy, yx (8 FMA + 8 MUL), the weighted sums a*xx + c*yy, a*yy + c*xx (4 FMA + 4 MUL), b*xy,
// b*yx (4 MUL), T^x = q^x conj(A^x_{k+m+n}) + b*xy conj(A^y_{k+m+n}) and T^y likewise (12 FMA + 4 MUL) and the two
// accumulations C'*T (8 FMA): 52 FP64 instructions, 32 FMA and 20 MUL, 84 flops per entry and symbol (an FMA counted as
// two), from 6 shared-memory loads of 16 bytes.  Fixed order, no atomics.
#define PMX_PB_THREADS 128
#define PMX_PB_RB 4
#define PMX_PB_TILE (PMX_PB_THREADS * PMX_PB_RB)
__device__ __forceinline__ double2 pb_mul(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
// a*conj(b), and acc + a*conj(b)
__device__ __forceinline__ double2 pb_mul_conj(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, a.y * b.y), fma(a.y, b.x, -a.x * b.y));
}
__device__ __forceinline__ double2 pb_mac_conj(double2 acc, double2 a, double2 b) {
    return make_double2(fma(a.y, b.y, fma(a.x, b.x, acc.x)), fma(-a.x, b.y, fma(a.y, b.x, acc.y)));
}
__global__ void __launch_bounds__(PMX_PB_THREADS) pmx_k_pb_triplet(const cpx* __restrict__ A, int nsymb,
                                                                   const PbCoef* __restrict__ coef, int ncoef, int K,
                                                                   double wa, double wb, double wc, cpx* __restrict__ D) {
    extern __shared__ __align__(16) unsigned char smp[];
    const int H = 2 * K, span = PMX_PB_TILE + 2 * H;
    cpx* sx = reinterpret_cast<cpx*>(smp);   // [span]: symbol k0 - H + i at i
    cpx* sy = sx + span;
    const int b = blockIdx.y, k0 = blockIdx.x * PMX_PB_TILE;
    const cpx* ax = A + (size_t)(2 * b) * nsymb;
    const cpx* ay = ax + nsymb;
    for (int i = threadIdx.x; i < span; i += PMX_PB_THREADS) {
        int k = (k0 - H + i) % nsymb;
        if (k < 0) k += nsymb;
        sx[i] = ax[k];
        sy[i] = ay[k];
    }
    __syncthreads();
    double2 dx[PMX_PB_RB], dy[PMX_PB_RB];
#pragma unroll
    for (int r = 0; r < PMX_PB_RB; ++r) dx[r] = dy[r] = make_double2(0.0, 0.0);
    const int base = H + threadIdx.x;
    for (int i = 0; i < ncoef; ++i) {
        const double cr = __ldg(&coef[i].cr), ci = __ldg(&coef[i].ci);
        const int m = __ldg(&coef[i].m), n = __ldg(&coef[i].n);
#pragma unroll
        for (int r = 0; r < PMX_PB_RB; ++r) {
            const int o = base + r * PMX_PB_THREADS;
            const double2 xm = sx[o + m], ym = sy[o + m], xn = sx[o + n], yn = sy[o + n];
            const double2 xs = sx[o + m + n], ys = sy[o + m + n];
            const double2 xx = pb_mul(xm, xn), yy = pb_mul(ym, yn), xy = pb_mul(xm, yn), yx = pb_mul(ym, xn);
            const double2 qx = make_double2(fma(wa, xx.x, wc * yy.x), fma(wa, xx.y, wc * yy.y));
            const double2 qy = make_double2(fma(wa, yy.x, wc * xx.x), fma(wa, yy.y, wc * xx.y));
            const double2 bxy = make_double2(wb * xy.x, wb * xy.y), byx = make_double2(wb * yx.x, wb * yx.y);
            const double2 tx = pb_mac_conj(pb_mul_conj(qx, xs), bxy, ys);
            const double2 ty = pb_mac_conj(pb_mul_conj(qy, ys), byx, xs);
            dx[r] = make_double2(fma(cr, tx.x, fma(-ci, tx.y, dx[r].x)), fma(cr, tx.y, fma(ci, tx.x, dx[r].y)));
            dy[r] = make_double2(fma(cr, ty.x, fma(-ci, ty.y, dy[r].x)), fma(cr, ty.y, fma(ci, ty.x, dy[r].y)));
        }
    }
#pragma unroll
    for (int r = 0; r < PMX_PB_RB; ++r) {
        const int k = k0 + threadIdx.x + r * PMX_PB_THREADS;
        if (k < nsymb) {
            D[(size_t)(2 * b) * nsymb + k] = dx[r];
            D[(size_t)(2 * b + 1) * nsymb + k] = dy[r];
        }
    }
}

// u[t] -= xi * sum_k p[t - k*nt + np/2] * Delta_k, k descending from the last symbol whose pulse covers t
__global__ void __launch_bounds__(256) pmx_k_pb_apply(cpx* __restrict__ field, size_t N, int l1, int l2, int nsymb, int nt,
                                                      const double* __restrict__ pulse, int np, const cpx* __restrict__ D,
                                                      double xi) {
    const int b = blockIdx.y;
    cpx* fld = field + (size_t)b * N * 2;
    const cpx* dx = D + (size_t)(2 * b) * nsymb;
    const cpx* dy = dx + nsymb;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < N; t += (size_t)gridDim.x * blockDim.x) {
        const long long h = (long long)t + np / 2;
        long long k = h / nt;
        int j = (int)(h - k * nt);
        double axr = 0, axi = 0, ayr = 0, ayi = 0;
        for (; j < np; j += nt, --k) {
            int kk = (int)(k % nsymb);
            if (kk < 0) kk += nsymb;
            const double p = pulse[j];
            const cpx ex = dx[kk], ey = dy[kk];
            axr = fma(p, ex.x, axr);
            axi = fma(p, ex.y, axi);
            ayr = fma(p, ey.x, ayr);
            ayi = fma(p, ey.y, ayi);
        }
        const size_t pos = 2 * pmx_mem_index(t, l1, l2);
        cpx x, y;
        ld_sa(fld + pos, x, y);
        x = make_double2(fma(-xi, axr, x.x), fma(-xi, axi, x.y));
        y = make_double2(fma(-xi, ayr, y.x), fma(-xi, ayi, y.y));
        st_sa(fld + pos, x, y);
    }
}

// The XPM triplet sum (pmx_pb_xpm_create): Delta += the inter-channel triplets of every interferer, on the COI's symbols A
// and the interferer's B.  Shaped like pmx_k_pb_triplet: a CTA takes PMX_PB_TILE symbols of one realization, lands A with
// a halo of ha = max |m| and, per interferer in turn, B with a halo of hb = max(|n|, |m+n|), both polarizations, in shared
// memory; a thread owns PMX_PB_RB symbols PMX_PB_THREADS apart and reads each coefficient as a broadcast.  The sums start
// from the SPM Delta and take the interferers in list order, each table in list order: a fixed order, no atomics.  Per entry
// and symbol the loop runs the 4 products B*conj(B) P = Bx_n conj(Bx_s), Q = By_n conj(By_s), R = Bx_n conj(By_s),
// S = By_n conj(Bx_s) (8 FMA + 8 MUL), the 4 weighted sums w1*P + w2*Q, w3*R + w4*S, w1*Q + w2*P, w3*S + w4*R (8 FMA +
// 8 MUL), T^x = A^x_m u + A^y_m v and T^y likewise (8 FMA + 4 MUL + 8 FMA) and the two accumulations C'*T (8 FMA): 56 FP64
// instructions, 36 FMA and 20 MUL, 92 flops per entry and symbol (an FMA counted as two), from 6 shared-memory loads of 16
// bytes.
__device__ __forceinline__ double2 pb_mac(double2 acc, double2 a, double2 b) {   // acc + a*b
    return make_double2(fma(-a.y, b.y, fma(a.x, b.x, acc.x)), fma(a.y, b.x, fma(a.x, b.y, acc.y)));
}
__global__ void __launch_bounds__(PMX_PB_THREADS) pmx_k_pb_xpm(const cpx* __restrict__ A, const cpx* __restrict__ B,
                                                               int nsymb, int batch, int nint, const PbCoef* __restrict__ coef,
                                                               const int* __restrict__ off, int ha, int hb, double w1,
                                                               double w2, double w3, double w4, cpx* __restrict__ D) {
    extern __shared__ __align__(16) unsigned char smp[];
    const int sa = PMX_PB_TILE + 2 * ha, sb = PMX_PB_TILE + 2 * hb;
    cpx* ax = reinterpret_cast<cpx*>(smp);   // [sa]: symbol k0 - ha + i at i
    cpx* ay = ax + sa;
    cpx* bx = ay + sa;                        // [sb]: symbol k0 - hb + i at i
    cpx* by = bx + sb;
    const int b = blockIdx.y, k0 = blockIdx.x * PMX_PB_TILE;
    const cpx* gax = A + (size_t)(2 * b) * nsymb;
    for (int i = threadIdx.x; i < sa; i += PMX_PB_THREADS) {
        int k = (k0 - ha + i) % nsymb;
        if (k < 0) k += nsymb;
        ax[i] = gax[k];
        ay[i] = gax[nsymb + k];
    }
    double2 dx[PMX_PB_RB], dy[PMX_PB_RB];
#pragma unroll
    for (int r = 0; r < PMX_PB_RB; ++r) {
        const int k = k0 + threadIdx.x + r * PMX_PB_THREADS;
        dx[r] = k < nsymb ? D[(size_t)(2 * b) * nsymb + k] : make_double2(0.0, 0.0);
        dy[r] = k < nsymb ? D[(size_t)(2 * b + 1) * nsymb + k] : make_double2(0.0, 0.0);
    }
    for (int c = 0; c < nint; ++c) {
        __syncthreads();   // the previous interferer's tile is read
        const cpx* gbx = B + ((size_t)c * batch + b) * 2 * nsymb;
        for (int i = threadIdx.x; i < sb; i += PMX_PB_THREADS) {
            int k = (k0 - hb + i) % nsymb;
            if (k < 0) k += nsymb;
            bx[i] = gbx[k];
            by[i] = gbx[nsymb + k];
        }
        __syncthreads();
        const int e = __ldg(&off[c + 1]);
        for (int i = __ldg(&off[c]); i < e; ++i) {
            const double cr = __ldg(&coef[i].cr), ci = __ldg(&coef[i].ci);
            const int m = __ldg(&coef[i].m), n = __ldg(&coef[i].n);
#pragma unroll
            for (int r = 0; r < PMX_PB_RB; ++r) {
                const int o = threadIdx.x + r * PMX_PB_THREADS;
                const double2 xm = ax[ha + o + m], ym = ay[ha + o + m];
                const double2 xn = bx[hb + o + n], yn = by[hb + o + n], xs = bx[hb + o + m + n], ys = by[hb + o + m + n];
                const double2 P = pb_mul_conj(xn, xs), Q = pb_mul_conj(yn, ys), R = pb_mul_conj(xn, ys), S = pb_mul_conj(yn, xs);
                const double2 u = make_double2(fma(w1, P.x, w2 * Q.x), fma(w1, P.y, w2 * Q.y));
                const double2 v = make_double2(fma(w3, R.x, w4 * S.x), fma(w3, R.y, w4 * S.y));
                const double2 u2 = make_double2(fma(w1, Q.x, w2 * P.x), fma(w1, Q.y, w2 * P.y));
                const double2 v2 = make_double2(fma(w3, S.x, w4 * R.x), fma(w3, S.y, w4 * R.y));
                const double2 tx = pb_mac(pb_mul(xm, u), ym, v);
                const double2 ty = pb_mac(pb_mul(ym, u2), xm, v2);
                dx[r] = make_double2(fma(cr, tx.x, fma(-ci, tx.y, dx[r].x)), fma(cr, tx.y, fma(ci, tx.x, dx[r].y)));
                dy[r] = make_double2(fma(cr, ty.x, fma(-ci, ty.y, dy[r].x)), fma(cr, ty.y, fma(ci, ty.x, dy[r].y)));
            }
        }
    }
#pragma unroll
    for (int r = 0; r < PMX_PB_RB; ++r) {
        const int k = k0 + threadIdx.x + r * PMX_PB_THREADS;
        if (k < nsymb) {
            D[(size_t)(2 * b) * nsymb + k] = dx[r];
            D[(size_t)(2 * b + 1) * nsymb + k] = dy[r];
        }
    }
}

// The three launches of the stage on a field of the plan's nfft and batch (checked by the caller)
static void pb_project(pmx_pb_plan* p, const pmx_devfield* f, cpx* out) {
    pmx_ctx* c = p->ctx;
    pmx_k_pb_project<<<dim3((unsigned)((p->nsymb + 255) / 256), p->batch), 256, 0, c->stream>>>(
        f->data, (size_t)p->nfft, f->log2N1, f->log2N2, p->nsymb, p->nt, p->pulse, p->npulse, p->inorm, out);
    c->launches++;
}
static int pb_triplet(pmx_pb_plan* p) {
    pmx_ctx* c = p->ctx;
    const int smem = (PMX_PB_TILE + 4 * p->K) * 2 * (int)sizeof(cpx);
    if (smem > 48 * 1024) CK(c, cudaFuncSetAttribute(pmx_k_pb_triplet, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    pmx_k_pb_triplet<<<dim3((unsigned)((p->nsymb + PMX_PB_TILE - 1) / PMX_PB_TILE), p->batch), PMX_PB_THREADS, smem,
                       c->stream>>>(p->A, p->nsymb, p->coef, p->ncoef, p->K, p->wa, p->wb, p->wc, p->D);
    c->launches++;
    return PMX_OK;
}
static void pb_apply(pmx_pb_plan* p, pmx_devfield* f) {
    pmx_ctx* c = p->ctx;
    const size_t N = (size_t)p->nfft;
    pmx_k_pb_apply<<<dim3((unsigned)std::min<size_t>((N + 255) / 256, 148 * 8), p->batch), 256, 0, c->stream>>>(
        f->data, N, f->log2N1, f->log2N2, p->nsymb, p->nt, p->pulse, p->npulse, p->D, p->xi);
    c->launches++;
}

// XPM-aware single channel (xi != 0): every interferer cut from a copy of the field and projected, then the COI's down,
// projection and SPM triplets, the XPM triplets added to Delta, apply and up
static int pb_xpm_exec(pmx_pb_plan* p, pmx_devfield* f) {
    pmx_ctx* c = p->ctx;
    pmx_pb_plan* s = p->ch_pb;
    const size_t per = (size_t)p->batch * 2 * s->nsymb;
    int rc = PMX_OK;
    for (int i = 0; i < p->xpm_n && !rc; ++i) {
        rc = pmx_field_copy_cols(p->xpm_copy, 0, f, 0, p->batch);
        if (!rc) rc = band_down(p->xpm_band[i], p->xpm_copy, p->ch_work, p->ch_log2r, p->xpm_shift[i]);
        if (!rc) pb_project(s, p->ch_work, p->xpm_B + i * per);
    }
    if (!rc) rc = band_down(p->ch_band, f, p->ch_work, p->ch_log2r, p->ch_shift);
    if (rc) return rc;
    CK(c, cudaSetDevice(c->device));
    pb_project(s, p->ch_work, s->A);
    if (int e = pb_triplet(s)) return e;
    const int smem = (2 * (PMX_PB_TILE + 2 * p->xpm_ha) + 2 * (PMX_PB_TILE + 2 * p->xpm_hb)) * (int)sizeof(cpx);
    if (smem > 48 * 1024) CK(c, cudaFuncSetAttribute(pmx_k_pb_xpm, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    pmx_k_pb_xpm<<<dim3((unsigned)((s->nsymb + PMX_PB_TILE - 1) / PMX_PB_TILE), p->batch), PMX_PB_THREADS, smem, c->stream>>>(
        s->A, p->xpm_B, s->nsymb, p->batch, p->xpm_n, p->xpm_coef, p->xpm_off, p->xpm_ha, p->xpm_hb, p->xpm_w[0], p->xpm_w[1],
        p->xpm_w[2], p->xpm_w[3], s->D);
    c->launches++;
    pb_apply(s, p->ch_work);
    CK(c, cudaGetLastError());
    return band_up(p->ch_band, p->ch_work, f, p->ch_log2r, p->ch_shift);
}

extern "C" int pmx_pb_create(pmx_ctx* c, const pmx_pb_desc* d, pmx_pb_plan** out) {
    // (the descriptor is checked before the context, so that the checks run without a device)
    if (!d || !out) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: null argument");
    *out = nullptr;
    if (d->nfc != 1)
        return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_create: nfc=%d, PB-NLC takes one-column fields holding one channel",
                       d->nfc);
    if (d->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_create: FP64 fields only");
    const int lg = ilog2_exact(d->nfft);
    if (lg < 6 || lg > 24)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: nfft=%lld, built for powers of two from 2^6 to 2^24",
                       (long long)d->nfft);
    if (d->nsymb < 1 || d->nt < 1 || (int64_t)d->nsymb * d->nt != d->nfft)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: nsymb*nt = %d x %d must equal nfft = %lld", d->nsymb, d->nt,
                       (long long)d->nfft);
    if (d->batch < 1) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: batch must be >= 1");
    if (int rc = check_batch_cols(c, "pmx_pb_create", d->batch, 1)) return rc;
    if (!d->pulse || d->npulse < 2 || d->npulse % 2 || d->npulse > 16 * d->nt || d->npulse > d->nfft)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: npulse=%d, the pulse must have an even count of 2 to min(16*nt, "
                       "nfft) = %lld samples", d->npulse, (long long)std::min<int64_t>(16 * (int64_t)d->nt, d->nfft));
    double e = 0;
    for (int j = 0; j < d->npulse; ++j) {
        if (!std::isfinite(d->pulse[j])) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: pulse sample %d is not finite", j);
        e += d->pulse[j] * d->pulse[j];
    }
    if (!(e > 0) || !std::isfinite(e)) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: the pulse has no energy");
    for (int i = 0; i < 3; ++i)
        if (!std::isfinite(d->weights[i])) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: weight %d is not finite", i);
    if (!std::isfinite(d->gamma) || !std::isfinite(d->xi) || !std::isfinite(d->scale))
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: gamma, xi and scale must be finite");
    if (d->ncoef < 1 || d->ncoef > PMX_PB_MAX_COEF)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: ncoef=%d, 1 to %d entries", d->ncoef, PMX_PB_MAX_COEF);
    if (!d->m || !d->n || !d->coef) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: null coefficient list");
    std::vector<PbCoef> list(d->ncoef);
    const double g = d->gamma * d->scale * d->scale;
    int K = 0;
    for (int i = 0; i < d->ncoef; ++i) {
        const int m = d->m[i], n = d->n[i];
        if (std::abs(m) > PMX_PB_MAX_K || std::abs(n) > PMX_PB_MAX_K)
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: entry %d has (m, n) = (%d, %d), |m| and |n| at most %d", i, m,
                           n, PMX_PB_MAX_K);
        const double cr = d->coef[2 * i], ci = d->coef[2 * i + 1];
        if (!std::isfinite(cr) || !std::isfinite(ci))
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: coefficient %d is not finite", i);
        list[i] = PbCoef{g * ci, -(g * cr), m, n};   // -j*gamma*s^2*C
        K = std::max(K, std::max(std::abs(m), std::abs(n)));
    }
    if (!c) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: null ctx");
    CK(c, cudaSetDevice(c->device));
    pmx_pb_plan* p = new (std::nothrow) pmx_pb_plan();
    if (!p) return set_err(c, PMX_ERR_INVALID, "pmx_pb_create: out of host memory");
    p->ctx = c;
    p->nfft = d->nfft;
    p->nsymb = d->nsymb;
    p->nt = d->nt;
    p->batch = d->batch;
    p->npulse = d->npulse;
    p->ncoef = d->ncoef;
    p->K = K;
    p->wa = d->weights[0];
    p->wb = d->weights[1];
    p->wc = d->weights[2];
    p->xi = d->xi;
    p->inorm = 1.0 / e;
    const size_t sym_bytes = (size_t)d->batch * 2 * d->nsymb * sizeof(cpx);
    cudaError_t err = cudaMallocAsync(&p->pulse, sizeof(double) * d->npulse, c->stream);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->coef, sizeof(PbCoef) * d->ncoef, c->stream);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->A, sym_bytes, c->stream);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->D, sym_bytes, c->stream);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(p->pulse, d->pulse, sizeof(double) * d->npulse, cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(p->coef, list.data(), sizeof(PbCoef) * d->ncoef, cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(p->A, 0, sym_bytes, c->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(p->D, 0, sym_bytes, c->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);   // the host tables are the caller's and this frame's
    if (err != cudaSuccess) {
        pmx_pb_destroy(p);
        return set_err(c, PMX_ERR_CUDA, "pmx_pb_create: %s", cudaGetErrorString(err));
    }
    *out = p;
    return PMX_OK;
}

extern "C" int pmx_pb_exec(pmx_pb_plan* p, pmx_devfield* f) {
    if (!p || !f) return set_err(p ? p->ctx : nullptr, PMX_ERR_INVALID, "pmx_pb_exec: null argument");
    pmx_ctx* c = p->ctx;
    if (f->nfc != 1)
        return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_exec: nfc=%d, PB-NLC takes one-column fields holding one channel",
                       f->nfc);
    if (f->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_exec: FP64 fields only");
    if (f->nfft != p->nfft)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_exec: the field has nfft=%lld, the plan %lld", (long long)f->nfft,
                       (long long)p->nfft);
    if (f->batch != p->batch)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_exec: the field has batch %d, the plan %d", f->batch, p->batch);
    if (p->ch_pb) {   // single channel: down, the stage at nfft/decim samples, up
        if (p->xpm_n && p->xi != 0) return pb_xpm_exec(p, f);
        int rc = band_down(p->ch_band, f, p->ch_work, p->ch_log2r, p->ch_shift);
        if (!rc) rc = pmx_pb_exec(p->ch_pb, p->ch_work);
        if (!rc) rc = band_up(p->ch_band, p->ch_work, f, p->ch_log2r, p->ch_shift);
        return rc;
    }
    if (p->xi == 0) return PMX_OK;   // nothing to subtract: the field is left as it is
    CK(c, cudaSetDevice(c->device));
    pb_project(p, f, p->A);
    if (int rc = pb_triplet(p)) return rc;
    pb_apply(p, f);
    CK(c, cudaGetLastError());
    return PMX_OK;
}

extern "C" int pmx_pb_symbols(pmx_pb_plan* p, double* A, double* delta) {
    if (!p) return set_err(nullptr, PMX_ERR_INVALID, "pmx_pb_symbols: null plan");
    if (p->ch_pb) return pmx_pb_symbols(p->ch_pb, A, delta);
    pmx_ctx* c = p->ctx;
    const size_t bytes = (size_t)p->batch * 2 * p->nsymb * sizeof(cpx);
    CK(c, cudaSetDevice(c->device));
    if (A) CK(c, cudaMemcpyAsync(A, p->A, bytes, cudaMemcpyDeviceToHost, c->stream));
    if (delta) CK(c, cudaMemcpyAsync(delta, p->D, bytes, cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

extern "C" void pmx_pb_destroy(pmx_pb_plan* p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    for (void* q : {(void*)p->pulse, (void*)p->coef, (void*)p->A, (void*)p->D, (void*)p->xpm_B, (void*)p->xpm_coef,
                    (void*)p->xpm_off})
        if (q) cudaFreeAsync(q, p->ctx->stream);
    pmx_pb_destroy(p->ch_pb);
    pmx_plan_destroy(p->ch_band);
    pmx_field_destroy(p->ch_work);
    for (pmx_plan* q : p->xpm_band) pmx_plan_destroy(q);
    pmx_field_destroy(p->xpm_copy);
    delete p;
}

// Single-channel PB-NLC (polmux_ssfm.h): down, the stage of pmx_pb_create at M = nfft/decim samples, up, as single-channel
// DBP does it.  The descriptor is the stage's at M samples; the plan runs on fields of N = M*decim samples.
extern "C" int pmx_pb_channel_create(pmx_ctx* c, const pmx_pb_desc* d, const pmx_dbp_band* band, pmx_pb_plan** out) {
    // (checked before the context, like pmx_pb_create)
    if (!d || !band || !out) return set_err(c, PMX_ERR_INVALID, "pmx_pb_channel_create: null argument");
    *out = nullptr;
    const int lm = ilog2_exact(d->nfft), lr = ilog2_exact(band->decim);
    if (band->decim < 2 || lr < 1)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_channel_create: decim=%d, must be a power of two >= 2", band->decim);
    if (d->nfft < 64)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_channel_create: nfft/decim = %lld/%d samples, at least 2^6 are needed",
                       (long long)d->nfft * band->decim, band->decim);
    if (lm >= 0 && lm + lr > 24)
        return set_err(c, PMX_ERR_UNSUPPORTED, "single-channel PB-NLC: nfft=%lld, built for powers of two from 2^6 to 2^24",
                       (long long)d->nfft * band->decim);
    if (d->nfc != 1)
        return set_err(c, PMX_ERR_UNSUPPORTED, "single-channel PB-NLC: nfc=%d, built for one column holding every channel "
                       "(a 'unique' multiplex)", d->nfc);
    if (d->precision != PMX_F64) return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_channel_create: FP64 fields only");
    pmx_pb_plan* inner = nullptr;
    int rc = pmx_pb_create(c, d, &inner);   // validates the rest before it needs the context
    if (rc) return rc;
    const int64_t M = d->nfft, N = M << lr;
    pmx_pb_plan* p = new (std::nothrow) pmx_pb_plan();
    if (!p) {
        pmx_pb_destroy(inner);
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_channel_create: out of host memory");
    }
    p->ctx = c;
    p->nfft = N;
    p->nsymb = d->nsymb;
    p->nt = d->nt << lr;
    p->batch = d->batch;
    p->xi = d->xi;
    p->ch_pb = inner;
    p->ch_shift = ((band->shift % N) + N) % N;
    p->ch_log2r = lr;
    rc = band_filter_create(c, N, M, p->ch_shift, d->batch, PMX_F64, &p->ch_band);
    if (!rc) rc = pmx_field_create(c, M, 1, d->batch, PMX_F64, &p->ch_work);
    if (rc) {
        pmx_pb_destroy(p);
        return rc;
    }
    *out = p;
    return PMX_OK;
}

// XPM-aware single-channel PB-NLC (polmux_ssfm.h): the channel plan, plus per interferer a band filter at N, and the
// interferers' symbols and tables for pmx_k_pb_xpm
extern "C" int pmx_pb_xpm_create(pmx_ctx* c, const pmx_pb_desc* d, const pmx_dbp_band* band, const pmx_pb_xpm_desc* x,
                                 pmx_pb_plan** out) {
    // (checked before the context, like pmx_pb_channel_create)
    if (!d || !band || !x || !out) return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: null argument");
    *out = nullptr;
    if (x->nint < 1 || x->nint > PMX_PB_XPM_MAX_INT)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: nint=%d, 1 to %d interferers", x->nint, PMX_PB_XPM_MAX_INT);
    if (!x->shift || !x->ncoef || !x->m || !x->n || !x->coef)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: null interferer list");
    for (int i = 0; i < 4; ++i)
        if (!std::isfinite(x->weights[i])) return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: weight %d is not finite", i);
    int64_t total = 0;
    std::vector<int> off(x->nint + 1, 0);   // [nint+1] where each interferer's table starts
    for (int i = 0; i < x->nint; ++i) {
        if (x->ncoef[i] < 1)
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: interferer %d has ncoef=%d, at least 1", i, x->ncoef[i]);
        total += x->ncoef[i];
        off[i + 1] = (int)std::min<int64_t>(total, INT32_MAX);
    }
    if (total > PMX_PB_MAX_COEF)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: %lld entries in all, at most %d", (long long)total,
                       PMX_PB_MAX_COEF);
    // the shifts mod N, when the band and the descriptor give N (otherwise pmx_pb_channel_create refuses them below)
    const int lr = ilog2_exact(band->decim);
    if (band->decim >= 2 && lr >= 1 && d->nfft >= 1 && d->nfft <= ((int64_t)1 << 30)) {
        const int64_t N = d->nfft << lr;
        auto mod = [N](int64_t v) { return ((v % N) + N) % N; };
        for (int i = 0; i < x->nint; ++i) {
            if (mod(x->shift[i]) == mod(band->shift))
                return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: interferer %d has the channel's own shift %lld", i,
                               (long long)x->shift[i]);
            for (int j = 0; j < i; ++j)
                if (mod(x->shift[i]) == mod(x->shift[j]))
                    return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: interferers %d and %d have the same shift %lld", j,
                                   i, (long long)x->shift[i]);
        }
    }
    const double g = d->gamma * d->scale * d->scale;
    std::vector<PbCoef> list((size_t)total);
    int ha = 0, hb = 0;
    for (int64_t i = 0; i < total; ++i) {
        const int m = x->m[i], n = x->n[i];
        if (std::abs(m) > PMX_PB_MAX_K || std::abs(n) > PMX_PB_XPM_MAX_N)
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: entry %lld has (m, n) = (%d, %d), |m| at most %d and |n| "
                           "at most %d", (long long)i, m, n, PMX_PB_MAX_K, PMX_PB_XPM_MAX_N);
        const double cr = x->coef[2 * i], ci = x->coef[2 * i + 1];
        if (!std::isfinite(cr) || !std::isfinite(ci))
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_create: coefficient %lld is not finite", (long long)i);
        list[i] = PbCoef{g * ci, -(g * cr), m, n};   // -j*gamma*s^2*C
        ha = std::max(ha, std::abs(m));
        hb = std::max(hb, std::max(std::abs(n), std::abs(m + n)));
    }
    pmx_pb_plan* p = nullptr;
    int rc = pmx_pb_channel_create(c, d, band, &p);   // validates the rest before it needs the context
    if (rc) return rc;
    const int64_t N = p->nfft;
    p->xpm_n = x->nint;
    p->xpm_ha = ha;
    p->xpm_hb = hb;
    for (int i = 0; i < 4; ++i) p->xpm_w[i] = x->weights[i];
    for (int i = 0; i < x->nint && !rc; ++i) {
        p->xpm_shift[i] = ((x->shift[i] % N) + N) % N;
        rc = band_filter_create(c, N, d->nfft, p->xpm_shift[i], d->batch, PMX_F64, &p->xpm_band[i]);
    }
    if (!rc) rc = pmx_field_create(c, N, 1, d->batch, PMX_F64, &p->xpm_copy);
    if (rc) {
        pmx_pb_destroy(p);
        return rc;
    }
    const size_t bbytes = (size_t)x->nint * d->batch * 2 * d->nsymb * sizeof(cpx);
    cudaError_t err = cudaSetDevice(c->device);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->xpm_B, bbytes, c->stream);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->xpm_coef, sizeof(PbCoef) * total, c->stream);
    if (err == cudaSuccess) err = cudaMallocAsync(&p->xpm_off, sizeof(int) * off.size(), c->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(p->xpm_B, 0, bbytes, c->stream);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(p->xpm_coef, list.data(), sizeof(PbCoef) * total, cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess)
        err = cudaMemcpyAsync(p->xpm_off, off.data(), sizeof(int) * off.size(), cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);   // the host tables are this frame's
    if (err != cudaSuccess) {
        pmx_pb_destroy(p);
        return set_err(c, PMX_ERR_CUDA, "pmx_pb_xpm_create: %s", cudaGetErrorString(err));
    }
    *out = p;
    return PMX_OK;
}

extern "C" int pmx_pb_xpm_symbols(pmx_pb_plan* p, int32_t i, double* B) {
    if (!p || !B) return set_err(p ? p->ctx : nullptr, PMX_ERR_INVALID, "pmx_pb_xpm_symbols: null argument");
    pmx_ctx* c = p->ctx;
    if (i < 0 || i >= p->xpm_n)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_xpm_symbols: interferer %d, the plan has %d", i, p->xpm_n);
    const size_t per = (size_t)p->batch * 2 * p->ch_pb->nsymb;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaMemcpyAsync(B, p->xpm_B + i * per, per * sizeof(cpx), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return PMX_OK;
}

// ---------------------------------------------------------------------------
// The PB-NLC triplet table on the device (pmx_pb_table, see the header).  The dispersed pulses g_q of a chunk of nodes are
// one filter plan of Ws samples with a column per node (H = exp(-i*bt*zeta_q), written on the device); the lag sums
// R[m][n] = sum_q w_q sum_t b(t) conj(b(t - n*nt)), b(t) = conj(g_q(t)) g_q(t - m*nt), are taken directly.  A CTA of
// pmx_k_pb_lagsum owns one (node, m) and a group of tiles of the window: per step it lands b for RC phases r and TJ + K
// symbols j (t = j*nt + r, K symbols of halo before the tile) in shared memory, phase-major, so that the threads of the lags
// n, n+1, ... of one phase read consecutive samples b_r[j - n] and share b_r[j] as a broadcast.  A thread owns up to
// PMX_PBT_IT (phase, lag) items; the phases are summed in shared memory and the tile groups and nodes by
// pmx_k_pb_lagreduce, every sum in a fixed order without atomics.  The rows n < 0 are conj(R[m][-n]) (the correlation of a
// circular sequence), so only 0 <= n <= K are summed.
#define PMX_PBT_THREADS 256
#define PMX_PBT_IT 4          // (phase, lag) items per thread: RC*(K+1) <= PMX_PBT_THREADS*PMX_PBT_IT
#define PMX_PBT_SAMPLES 1024  // samples of b per step: RC phases x TJ symbols
#define PMX_PBT_GROUPS 4      // tile groups of a window, each a CTA of its own

// the real pulse p0 (time order) into the x polarization of every column of a resident field; y = 0
__global__ void __launch_bounds__(256) pmx_k_pb_fill(cpx* __restrict__ field, int lg, int l1, int l2, int ncol,
                                                     const double* __restrict__ p0) {
    const size_t N = (size_t)1 << lg, total = N * ncol;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t col = i >> lg, t = i & (N - 1);
        st_sa(field + 2 * (col * N + pmx_mem_index(t, l1, l2)), make_double2(p0[t], 0.0), make_double2(0.0, 0.0));
    }
}

// raw[col][k] = exp(-i*bt[k]*zeta[col]) = (cos, -sin) of the product, FFT order, as pbnlc._lin_step forms it
__global__ void __launch_bounds__(256) pmx_k_pb_disp(double2* __restrict__ raw, const double* __restrict__ bt, int lg,
                                                     const double* __restrict__ zeta, int ncol) {
    const size_t N = (size_t)1 << lg, total = N * ncol;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        double s, c;
        sincos(bt[i & (N - 1)] * zeta[i >> lg], &s, &c);
        raw[i] = make_double2(c, -s);
    }
}

// e[i] = |x[(i + N/2) mod N]|^2 of column 0: the energy of the pulse in fftshift order (the default window's rule)
__global__ void __launch_bounds__(256) pmx_k_pb_energy(const cpx* __restrict__ field, int lg, int l1, int l2,
                                                       double* __restrict__ e) {
    const size_t N = (size_t)1 << lg;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (size_t)gridDim.x * blockDim.x) {
        const cpx x = field[2 * pmx_mem_index((i + N / 2) & (N - 1), l1, l2)];
        e[i] = x.x * x.x + x.y * x.y;
    }
}

// part[q][m][group][n] = sum over the group's tiles and every phase of b(t) conj(b(t - n*nt)) for node q (the column q of
// field), 0 <= n <= K; grid (groups, K+1, nodes)
__global__ void __launch_bounds__(PMX_PBT_THREADS) pmx_k_pb_lagsum(const cpx* __restrict__ field, int lg, int l1, int l2,
                                                                   int nt, int K, int RC, int TJ, int tiles_per_group,
                                                                   cpx* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char smp[];
    cpx* sb = reinterpret_cast<cpx*>(smp);   // [RC][TJ + K]: b at symbol J0 - K + jj, phase r0 + rr
    const size_t N = (size_t)1 << lg;
    const int q = blockIdx.z, m = blockIdx.y, grp = blockIdx.x;
    const int K1 = K + 1, row = TJ + K, items = RC * K1, nu = (items + PMX_PBT_THREADS - 1) / PMX_PBT_THREADS;
    const cpx* g = field + (size_t)q * N * 2;
    const long long shift = (long long)m * nt;
    int off[PMX_PBT_IT], lag[PMX_PBT_IT];
    double2 acc[PMX_PBT_IT];
#pragma unroll
    for (int u = 0; u < PMX_PBT_IT; ++u) {
        const int it = threadIdx.x + u * PMX_PBT_THREADS;
        const int rr = it < items ? it / K1 : 0;
        lag[u] = it < items ? it - rr * K1 : 0;
        off[u] = rr * row;
        acc[u] = make_double2(0.0, 0.0);
    }
    for (int tile = 0; tile < tiles_per_group; ++tile) {
        const long long J0 = (long long)(grp * tiles_per_group + tile) * TJ;
        for (int r0 = 0; r0 < nt; r0 += RC) {
            __syncthreads();   // the previous step's reads are done
            for (int i = threadIdx.x; i < RC * row; i += PMX_PBT_THREADS) {
                const int jj = i / RC, rr = i - jj * RC;
                const long long t = (J0 - K + jj) * nt + r0 + rr;
                const cpx a = g[2 * pmx_mem_index((size_t)t & (N - 1), l1, l2)];
                const cpx b = g[2 * pmx_mem_index((size_t)(t - shift) & (N - 1), l1, l2)];
                sb[rr * row + jj] = pb_mul_conj(b, a);   // conj(g(t)) g(t - m*nt)
            }
            __syncthreads();
            for (int jj = K; jj < row; ++jj) {
#pragma unroll
                for (int u = 0; u < PMX_PBT_IT; ++u)
                    if (u < nu) acc[u] = pb_mac_conj(acc[u], sb[off[u] + jj], sb[off[u] + jj - lag[u]]);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PMX_PBT_IT; ++u) {
        const int it = threadIdx.x + u * PMX_PBT_THREADS;
        if (it < items) sb[it] = acc[u];   // [rr][n]: items <= RC*row
    }
    __syncthreads();
    for (int n = threadIdx.x; n < K1; n += PMX_PBT_THREADS) {
        double2 s = make_double2(0.0, 0.0);
        for (int rr = 0; rr < RC; ++rr) s = make_double2(s.x + sb[rr * K1 + n].x, s.y + sb[rr * K1 + n].y);
        part[(((size_t)q * K1 + m) * gridDim.x + grp) * K1 + n] = s;
    }
}

// R[m][n] (+)= sum_q w[q] * sum_group part[q][m][group][n], nodes ascending; first = 1 starts from zero
__global__ void __launch_bounds__(256) pmx_k_pb_lagreduce(const cpx* __restrict__ part, int nq, int K1, int ngrp,
                                                          const double* __restrict__ w, cpx* __restrict__ R, int first) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= K1 * K1) return;
    const int m = idx / K1, n = idx - m * K1;
    double2 acc = first ? make_double2(0.0, 0.0) : R[idx];
    for (int q = 0; q < nq; ++q) {
        double2 s = make_double2(0.0, 0.0);
        for (int gi = 0; gi < ngrp; ++gi) {
            const cpx v = part[(((size_t)q * K1 + m) * ngrp + gi) * K1 + n];
            s = make_double2(s.x + v.x, s.y + v.y);
        }
        acc = make_double2(fma(w[q], s.x, acc.x), fma(w[q], s.y, acc.y));
    }
    R[idx] = acc;
}

// Gauss-Legendre nodes and weights on [-1, 1], ascending (Newton on P_n from the usual first guesses; the odd order's
// middle node exactly 0)
static void gauss_legendre(int nq, std::vector<double>& x, std::vector<double>& w) {
    x.assign(nq, 0.0);
    w.assign(nq, 0.0);
    auto legendre = [nq](double z, double& pp) {   // P_n(z), and P_n'(z) into pp
        double p1 = 1.0, p2 = 0.0;
        for (int j = 1; j <= nq; ++j) {
            const double p3 = p2;
            p2 = p1;
            p1 = ((2.0 * j - 1.0) * z * p2 - (j - 1.0) * p3) / j;
        }
        pp = nq * (z * p1 - p2) / (z * z - 1.0);
        return p1;
    };
    for (int i = 0; i < (nq + 1) / 2; ++i) {
        double z = std::cos(M_PI * (i + 0.75) / (nq + 0.5)), pp = 0.0;
        if (2 * i + 1 == nq) z = 0.0;
        for (int it = 0; it < 100; ++it) {
            const double dz = legendre(z, pp) / pp;
            z -= dz;
            if (std::fabs(dz) <= 1e-16) break;
        }
        legendre(z, pp);
        const double wi = 2.0 / ((1.0 - z * z) * pp * pp);
        x[i] = -z;
        x[nq - 1 - i] = z;
        w[i] = w[nq - 1 - i] = wi;
    }
}

static int pb_table_check(pmx_ctx* c, const pmx_pb_table_desc* d) {
    const int lg = ilog2_exact(d->nfft);
    if (lg < 6 || lg > 24)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: nfft=%lld, built for powers of two from 2^6 to 2^24",
                       (long long)d->nfft);
    if (d->nt < 1 || d->nfft % d->nt)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: nt=%d must divide nfft = %lld (nsymb*nt = nfft)", d->nt,
                       (long long)d->nfft);
    if (!d->pulse || d->npulse < 2 || d->npulse % 2 || d->npulse > 16 * d->nt || d->npulse > d->nfft)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: npulse=%d, the pulse must have an even count of 2 to min(16*nt, "
                       "nfft) = %lld samples", d->npulse, (long long)std::min<int64_t>(16 * (int64_t)d->nt, d->nfft));
    double e = 0;
    for (int j = 0; j < d->npulse; ++j) {
        if (!std::isfinite(d->pulse[j])) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: pulse sample %d is not finite", j);
        e += d->pulse[j] * d->pulse[j];
    }
    if (!(e > 0) || !std::isfinite(e)) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: the pulse has no energy");
    if (d->K < 0 || d->K > PMX_PB_MAX_K)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: K=%d, |m| and |n| at most %d", d->K, PMX_PB_MAX_K);
    if (d->nquad < 1) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: nquad=%d, at least one node per span", d->nquad);
    if (d->nspan < 1) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: nspan=%d, at least one span", d->nspan);
    if ((int64_t)d->nspan * d->nquad > (1 << 20))
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: nspan*nquad = %d x %d nodes, at most 2^20", d->nspan, d->nquad);
    if (!std::isfinite(d->length) || !(d->length > 0))
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: the span length must be finite and positive");
    if (!std::isfinite(d->alphalin) || d->alphalin < 0)
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: alphalin must be finite and non-negative");
    if (!std::isfinite(d->prune)) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: prune must be finite");
    if (!d->betat) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: null betat");
    for (int64_t k = 0; k < d->nfft; ++k)
        if (!std::isfinite(d->betat[k]))
            return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: betat[%lld] is not finite", (long long)k);
    const int64_t nsymb = d->nfft / d->nt;
    if (d->window < 0 || (d->window > 0 && nsymb % d->window))
        return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: the window (%d symbols) must divide the block (%lld symbols)",
                       d->window, (long long)nsymb);
    if (d->window > 0 && (int64_t)d->window * d->nt < 64)
        return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_table: a window of %lld samples, at least 2^6 are needed",
                       (long long)d->window * d->nt);
    return PMX_OK;
}

// Disperses p0 (time order, Ws = 2^lg samples) by exp(-i*bt*zeta) for each of the ncol zeta into the columns of f with the
// filter plan fp (created on the first call: *fp == nullptr); raw: [ncol][Ws] device scratch.
static int pb_disperse(pmx_ctx* c, int lg, int ncol, const double* d_bt, const double* d_zeta, const double* d_p0,
                       double2* raw, pmx_devfield* f, pmx_plan** fp) {
    const size_t total = ((size_t)1 << lg) * ncol;
    const unsigned grid = (unsigned)std::min<size_t>((total + 255) / 256, 148 * 16);
    pmx_k_pb_disp<<<grid, 256, 0, c->stream>>>(raw, d_bt, lg, d_zeta, ncol);
    pmx_k_pb_fill<<<grid, 256, 0, c->stream>>>(f->data, lg, f->log2N1, f->log2N2, ncol, d_p0);
    c->launches += 2;
    CK(c, cudaGetLastError());
    int rc = PMX_OK;
    if (!*fp) rc = filter_create(c, (int64_t)1 << lg, ncol, 1, PMX_F64, reinterpret_cast<const double*>(raw), 0, ncol, fp);
    else if (filter_set_raw(*fp, raw, ncol)) rc = set_err(c, PMX_ERR_CUDA, "pmx_pb_table: the filter table launch failed");
    if (!rc) rc = pmx_fiber_exec(*fp, f, nullptr);
    return rc;
}

// device buffers of one pmx_pb_table call, released whatever happens
struct PbTableScratch {
    pmx_ctx* c;
    std::vector<void*> bufs;
    pmx_devfield* f = nullptr;
    pmx_plan* fp = nullptr;
    explicit PbTableScratch(pmx_ctx* ctx) : c(ctx) {}
    template <typename T>
    cudaError_t alloc(T** p, size_t count) {
        *p = nullptr;
        cudaError_t e = cudaMallocAsync(p, std::max<size_t>(count, 1) * sizeof(T), c->stream);
        if (e == cudaSuccess) bufs.push_back(*p);
        return e;
    }
    void release_field() {
        pmx_plan_destroy(fp);
        pmx_field_destroy(f);
        fp = nullptr;
        f = nullptr;
    }
    ~PbTableScratch() {
        release_field();
        for (void* p : bufs) cudaFreeAsync(p, c->stream);
        cudaStreamSynchronize(c->stream);
    }
};

#define PBT_CK(call)                                                                                     \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) return set_err(c, PMX_ERR_CUDA, "pmx_pb_table: %s", cudaGetErrorString(e__)); \
    } while (0)

// the default window (pbnlc.default_window): the pulse on nfft samples dispersed over nspan*length on the device, its
// energy in fftshift order on the host
static int pb_default_window(pmx_ctx* c, const pmx_pb_table_desc* d, int* W) {
    const int lg = ilog2_exact(d->nfft);
    const size_t N = (size_t)d->nfft;
    const int64_t nsymb = d->nfft / d->nt;
    std::vector<double> p0(N, 0.0);
    for (int j = 0; j < d->npulse; ++j) p0[(size_t)((j - d->npulse / 2) % (int64_t)N + (int64_t)N) % N] = d->pulse[j];
    const double zeta = d->length * d->nspan;
    PbTableScratch s(c);
    double *d_bt = nullptr, *d_zeta = nullptr, *d_p0 = nullptr, *d_e = nullptr;
    double2* raw = nullptr;
    PBT_CK(s.alloc(&d_bt, N));
    PBT_CK(s.alloc(&d_zeta, 1));
    PBT_CK(s.alloc(&d_p0, N));
    PBT_CK(s.alloc(&d_e, N));
    PBT_CK(s.alloc(&raw, N));
    PBT_CK(cudaMemcpyAsync(d_bt, d->betat, N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    PBT_CK(cudaMemcpyAsync(d_zeta, &zeta, sizeof(double), cudaMemcpyHostToDevice, c->stream));
    PBT_CK(cudaMemcpyAsync(d_p0, p0.data(), N * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    int rc = pmx_field_create(c, d->nfft, 1, 1, PMX_F64, &s.f);
    if (!rc) rc = pb_disperse(c, lg, 1, d_bt, d_zeta, d_p0, raw, s.f, &s.fp);
    if (rc) return rc;
    pmx_k_pb_energy<<<(unsigned)std::min<size_t>((N + 255) / 256, 148 * 16), 256, 0, c->stream>>>(s.f->data, lg, s.f->log2N1,
                                                                                                s.f->log2N2, d_e);
    c->launches++;
    PBT_CK(cudaGetLastError());
    std::vector<double> e(N);
    PBT_CK(cudaMemcpyAsync(e.data(), d_e, N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    PBT_CK(cudaStreamSynchronize(c->stream));
    double tot = 0;
    for (double v : e) tot += v;
    const double tol = 1e-9, vlo = 0.5 * tol, vhi = 1 - 0.5 * tol;
    size_t lo = N, hi = N;
    double cum = 0;
    for (size_t i = 0; i < N; ++i) {   // searchsorted(c, v): the first i with c[i] >= v
        cum += e[i];
        const double ci = cum / tot;
        if (lo == N && ci >= vlo) lo = i;
        if (hi == N && ci >= vhi) {
            hi = i;
            break;
        }
    }
    const double need = (double)(hi - lo + 1) / d->nt + 2 * d->K + 8;
    int64_t w = 1;
    while (w < need) w *= 2;
    *W = (int)std::min<int64_t>(w, nsymb);
    return PMX_OK;
}

extern "C" int pmx_pb_table(pmx_ctx* c, const pmx_pb_table_desc* d, int32_t* m_out, int32_t* n_out, double* coef_out,
                            int32_t* ncoef, int32_t* window_used) {
    // (the descriptor is checked before the context, so that the checks run without a device)
    if (!d || !m_out || !n_out || !coef_out || !ncoef) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: null argument");
    if (int rc = pb_table_check(c, d)) return rc;
    if (!c) return set_err(c, PMX_ERR_INVALID, "pmx_pb_table: null ctx");
    CK(c, cudaSetDevice(c->device));
    const int K = d->K, K1 = K + 1, nt = d->nt;
    int W = d->window;
    if (W == 0) {
        if (int rc = pb_default_window(c, d, &W)) return rc;
        if ((int64_t)W * nt < 64)
            return set_err(c, PMX_ERR_UNSUPPORTED, "pmx_pb_table: a window of %lld samples, at least 2^6 are needed",
                           (long long)W * nt);
    }
    const int64_t Ws = (int64_t)W * nt;
    const int lg = ilog2_exact(Ws);
    // the nodes, the window's bins and pulse
    std::vector<double> gx, gw;
    gauss_legendre(d->nquad, gx, gw);
    const int nq = d->nspan * d->nquad;
    const int chunk = std::min(nq, Ws >= 4096 ? 64 : 8);   // columns per filter plan (on-chip kernels below 2^12: 8)
    const int nchunk = (nq + chunk - 1) / chunk;
    std::vector<double> zeta((size_t)nchunk * chunk), wq(nq), bt(Ws), p0(Ws, 0.0);
    for (int s = 0; s < d->nspan; ++s)
        for (int i = 0; i < d->nquad; ++i) {
            const double z = 0.5 * d->length * (gx[i] + 1.0);
            zeta[(size_t)s * d->nquad + i] = s * d->length + z;
            wq[(size_t)s * d->nquad + i] = 0.5 * d->length * gw[i] * std::exp(-d->alphalin * z);
        }
    for (size_t i = nq; i < zeta.size(); ++i) zeta[i] = zeta[nq - 1];   // the last chunk's spare columns (not summed)
    const int64_t stride = d->nfft / Ws;
    for (int64_t k = 0; k < Ws; ++k) bt[k] = d->betat[k * stride];
    for (int j = 0; j < d->npulse; ++j) p0[(size_t)(((j - d->npulse / 2) % Ws + Ws) % Ws)] = d->pulse[j];
    double norm = 0;
    for (int j = 0; j < d->npulse; ++j) norm += d->pulse[j] * d->pulse[j];
    // the lag-sum geometry: RC phases x TJ symbols per step, groups of tiles
    int RC = 1;
    while (RC * 2 <= nt && RC * 2 * K1 <= PMX_PBT_THREADS * PMX_PBT_IT) RC *= 2;
    const int TJ = (int)std::min<int64_t>(W, std::max(1, PMX_PBT_SAMPLES / RC));
    const int tiles = W / TJ, ngrp = std::min(tiles, PMX_PBT_GROUPS), tpg = tiles / ngrp;
    const int smem = RC * (TJ + K) * (int)sizeof(cpx);
    if (smem > 48 * 1024) CK(c, cudaFuncSetAttribute(pmx_k_pb_lagsum, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    std::vector<double2> R((size_t)K1 * K1);
    {
        PbTableScratch s(c);
        double *d_bt = nullptr, *d_zeta = nullptr, *d_w = nullptr, *d_p0 = nullptr;
        double2 *raw = nullptr, *part = nullptr, *d_R = nullptr;
        PBT_CK(s.alloc(&d_bt, Ws));
        PBT_CK(s.alloc(&d_zeta, zeta.size()));
        PBT_CK(s.alloc(&d_w, nq));
        PBT_CK(s.alloc(&d_p0, Ws));
        PBT_CK(s.alloc(&raw, (size_t)Ws * chunk));
        PBT_CK(s.alloc(&part, (size_t)chunk * K1 * ngrp * K1));
        PBT_CK(s.alloc(&d_R, (size_t)K1 * K1));
        PBT_CK(cudaMemcpyAsync(d_bt, bt.data(), Ws * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        PBT_CK(cudaMemcpyAsync(d_zeta, zeta.data(), zeta.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        PBT_CK(cudaMemcpyAsync(d_w, wq.data(), nq * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        PBT_CK(cudaMemcpyAsync(d_p0, p0.data(), Ws * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        int rc = pmx_field_create(c, Ws, chunk, 1, PMX_F64, &s.f);
        if (rc) return rc;
        for (int ch = 0; ch < nchunk; ++ch) {
            const int q0 = ch * chunk, nc = std::min(chunk, nq - q0);
            rc = pb_disperse(c, lg, chunk, d_bt, d_zeta + q0, d_p0, raw, s.f, &s.fp);
            if (rc) return rc;
            pmx_k_pb_lagsum<<<dim3((unsigned)ngrp, (unsigned)K1, (unsigned)nc), PMX_PBT_THREADS, smem, c->stream>>>(
                s.f->data, lg, s.f->log2N1, s.f->log2N2, nt, K, RC, TJ, tpg, part);
            pmx_k_pb_lagreduce<<<(unsigned)((K1 * K1 + 255) / 256), 256, 0, c->stream>>>(part, nc, K1, ngrp, d_w + q0, d_R,
                                                                                       ch == 0);
            c->launches += 2;
            PBT_CK(cudaGetLastError());
        }
        PBT_CK(cudaMemcpyAsync(R.data(), d_R, R.size() * sizeof(double2), cudaMemcpyDeviceToHost, c->stream));
        PBT_CK(cudaStreamSynchronize(c->stream));
    }
    // the table: rows m >= 0 from R (lags n < 0 conjugate), rows m < 0 conjugate, then exactly symmetric, pruned
    const int D = 2 * K + 1;
    std::vector<double2> C((size_t)D * D);
    auto row = [&](int m, int n) {   // R[m][n] / sum p^2 for m >= 0, any |n| <= K
        const double2 v = R[(size_t)m * K1 + std::abs(n)];
        return make_double2(v.x / norm, n < 0 ? -v.y / norm : v.y / norm);
    };
    for (int m = -K; m <= K; ++m)
        for (int n = -K; n <= K; ++n) {
            const double2 v = row(std::abs(m), n);
            C[(size_t)(m + K) * D + (n + K)] = m < 0 ? make_double2(v.x, -v.y) : v;
        }
    std::vector<double2> S(C.size());
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            const double2 a = C[(size_t)i * D + j], b = C[(size_t)j * D + i];
            S[(size_t)i * D + j] = make_double2(0.5 * (a.x + b.x), 0.5 * (a.y + b.y));
        }
    const double thr = d->prune * std::hypot(S[(size_t)K * D + K].x, S[(size_t)K * D + K].y);
    int cnt = 0;
    for (int i = 0; i < D; ++i)
        for (int j = 0; j < D; ++j) {
            const double2 v = S[(size_t)i * D + j];
            if (d->prune != 0 && !(std::hypot(v.x, v.y) >= thr)) continue;
            m_out[cnt] = i - K;
            n_out[cnt] = j - K;
            coef_out[2 * cnt] = v.x;
            coef_out[2 * cnt + 1] = v.y;
            ++cnt;
        }
    *ncoef = cnt;
    if (window_used) *window_used = W;
    return PMX_OK;
}
