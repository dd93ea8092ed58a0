// b200bo.cu - C ABI (include/b200bo.h) over the sm_100a kernels.  No CPU fallback: every
// compute entry point needs a CUDA device and reports B200BO_ERR_CUDA without one.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <dlfcn.h>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>

#include "fit_kernels.cuh"
#include "predict_kernels.cuh"
#include "predict16.cuh"
#include "predict_tc3.cuh"

using namespace b200bo;

constexpr int kDefaultTcVariant = 4;  // fp32 mode: 4 = N = 256 per MMA + row-block pairs (measured 115.7 ms; 3 = un-paired 124.7; 2 = 128-wide pairs 120.6, same box)
constexpr int kDefaultPredictWarps = 16;  // measured A/B (DESIGN.md 6): 550.1 ms vs 561.7 ms per 2^20 candidates at C3

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

static int set_err(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return set_err(B200BO_ERR_CUDA, "%s failed: %s (%s:%d)", #call,                  \
                           cudaGetErrorString(e__), __FILE__, __LINE__);                      \
    } while (0)

#define LAUNCHED() (g_launches.fetch_add(1, std::memory_order_relaxed))

// NVTX ranges around the phases of the path (fit / lml / predict_acq / select / exchange): visible in any
// NVTX-aware profiler, free otherwise (header-only NVTX3 resolves its injection library lazily).
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return B200BO_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess)
            return set_err(B200BO_ERR_CUDA, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        cap = bytes;
        return B200BO_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

struct b200bo_gp {
    int device = 0;
    int sm_count = 0;
    long long n = 0;
    int np = 0, d = 0;
    bool has_data = false, fitted = false;
    // kernel of the last fit
    int family = 0, nu = B200BO_NU_25;
    double constv = 1.0, jitter = 0.0;  // jitter = alpha + WhiteKernel noise_level (diagonal of K)
    double noise = 0.0;
    double y_mean = 0.0, y_std = 1.0;
    std::vector<double> y_norm;  // host copy of normalised targets (n)
    std::vector<double> y_raw;   // host copy of the raw targets (n)
    bool normalize = false;
    std::vector<int> xform;      // host copy (d) or empty
    DevBuf X, Xs, y, K, L, W, WT, T, alphav, v1, v2, ls, xf, info, part;
    // predict-side scratch (used when this handle is gps[0] of a call)
    DevBuf pscratch, xc, out_acq, out_mu, out_sd, sel, clamp;
    // small-batch path scratch (per GP) + work-unit tables (rebuilt when np changes)
    DevBuf s_ksm, s_partial, s_mupart, s_unit, s_rb, s_colsq;
    int s_np = 0, s_nunits = 0;
    // fp32 mode: L^-1 as tf32 (hi,lo) UMMA operand images (built on first use after a fit)
    DevBuf tc_linv;
    bool tc_valid = false;
    DevBuf cov_xc, cov_kst, cov_v, cov_c, cov_out, cov_mu;  // predict(return_cov=True) scratch
    DevBuf sel_cta;         // per-CTA running selection lists of the fused kernels
    // pruned selection: screen keys [m], survivors / pilot (coordinates + global index), counters
    // ([0] survivors, [1] pilot candidates, [2] tau); work of the last call for b200bo_last_select_stats
    DevBuf prune_key, surv, pilot, prune_cnt;
    long long st_screened = 0, st_full = 0;
    bool st_pruned = false;
    DevBuf pbounds, prow;   // throughput mode: Philox bounds (lo, span) / regenerated winner rows
    bool replica = false;   // predict-only copy made by b200bo_gp_replicate
    // look-ahead Cholesky: bulk stream, chain/bulk events, copy of the next diagonal step's panel block
    cudaStream_t bulk_stream = nullptr;
    cudaEvent_t ev_chain = nullptr, ev_bulk = nullptr;
    DevBuf pside;
    // CUDA graph of the theta-independent part of a factorisation (run_factor)
    cudaStream_t cap_stream = nullptr;
    cudaGraphExec_t fgraph_exec = nullptr;
    unsigned long long fgraph_key[16] = {0};
    long long fgraph_nodes = 0;
    // streamed host batches: copy / execute streams and the double-buffer events
    cudaStream_t copy_stream = nullptr, exec_stream = nullptr;
    cudaEvent_t chunk_up[2] = {nullptr, nullptr}, chunk_done[2] = {nullptr, nullptr};
    int precision = B200BO_PRECISION_FP64;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // fit-side work (set_data / fit / lml) of this handle is issued on this stream: the legacy default
    // stream (nullptr) unless b200bo_gp_set_private_stream gave the handle its own, so that several
    // handles driven from different host threads factorise concurrently
    cudaStream_t stream = nullptr;
};

// stream of the fit-side entry point in flight on this thread
static thread_local cudaStream_t g_st = nullptr;
struct StreamScope {
    cudaStream_t prev;
    explicit StreamScope(const b200bo_gp* gp) : prev(g_st) { g_st = gp ? gp->stream : nullptr; }
    ~StreamScope() { g_st = prev; }
};

static thread_local b200bo_gp* g_last_timed = nullptr;

// wait for the fit-side stream (the whole device when it is the legacy default stream)
static int sync_fit_stream() {
    if (g_st)
        CU(cudaStreamSynchronize(g_st));
    else
        CU(cudaDeviceSynchronize());
    return B200BO_OK;
}
// host <-> device copies ordered in the fit-side stream; d2h returns with the data on the host
static int h2d(void* dst, const void* src, size_t bytes) {
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_st));
    return B200BO_OK;
}
static int d2h(void* dst, const void* src, size_t bytes) {
    CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_st));
    CU(cudaStreamSynchronize(g_st));
    return B200BO_OK;
}

static inline int round_up(long long v, int m) { return (int)(((v + m - 1) / m) * m); }

extern "C" int b200bo_version(void) { return B200BO_VERSION; }
extern "C" const char* b200bo_last_error(void) { return g_err; }
extern "C" int64_t b200bo_launch_count(void) { return g_launches.load(); }

extern "C" int b200bo_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// device properties, timing events and the opt-in shared-memory sizes of the big kernels
static int init_handle(b200bo_gp* gp) {
    CU(cudaDeviceGetAttribute(&gp->sm_count, cudaDevAttrMultiProcessorCount, gp->device));
    CU(cudaEventCreate(&gp->ev0));
    CU(cudaEventCreate(&gp->ev1));
    CU(cudaFuncSetAttribute(predict_acq_kernel<PREDICT_IMPL_DFMA, false>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDfma));
    CU(cudaFuncSetAttribute(predict_acq_kernel<PREDICT_IMPL_DFMA, true>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDfma));
    CU(cudaFuncSetAttribute(predict_acq_kernel<PREDICT_IMPL_DMMA, false>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq_kernel<PREDICT_IMPL_DMMA, true>,
                            cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(potrf_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            kPotrfSmemBytes));
    CU(cudaFuncSetAttribute(potrf_diag_legacy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            kPotrfLegacySmemBytes));
    CU(cudaFuncSetAttribute(predict_acq_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            kPredictSmemBytesTc));
    CU(cudaFuncSetAttribute(predict_acq_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            kPredictSmemBytesTc));
    CU(cudaFuncSetAttribute(predict_acq_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            kPredictSmemBytesTc2));
    CU(cudaFuncSetAttribute(predict_acq_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesTc3));
    CU(cudaFuncSetAttribute(predict_acq_tc4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesTc4));
    CU(cudaFuncSetAttribute(small_trsv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmallTrsvSmemBytes));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<true, P16_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<false, P16_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<true, P16_SCREEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<false, P16_SCREEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<true, P16_GATHER>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(predict_acq16_kernel<false, P16_GATHER>, cudaFuncAttributeMaxDynamicSharedMemorySize, kPredictSmemBytesDmma));
    CU(cudaFuncSetAttribute(trailing_update64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTrailSmemBytes));
    CU(cudaFuncSetAttribute(dgemm128_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemm128SmemBytes));
    CU(cudaFuncSetAttribute(dgemm128_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemm128SmemBytes));
    CU(cudaFuncSetAttribute(dgemm128_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemm128SmemBytes));
    return B200BO_OK;
}

extern "C" int b200bo_gp_create(b200bo_gp** out, int device) {
    if (!out) return set_err(B200BO_ERR_ARG, "out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_err(B200BO_ERR_CUDA,
                       "no CUDA device available (%s); this engine has no CPU fallback",
                       e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= ndev) return set_err(B200BO_ERR_ARG, "device %d out of range", device);
    CU(cudaSetDevice(device));
    b200bo_gp* gp = new b200bo_gp();
    gp->device = device;
    const int rc = init_handle(gp);
    if (rc != B200BO_OK) {
        b200bo_gp_destroy(gp);
        return rc;
    }
    *out = gp;
    return B200BO_OK;
}

extern "C" void b200bo_gp_destroy(b200bo_gp* gp) {
    if (!gp) return;
    cudaSetDevice(gp->device);
    DevBuf* bufs[] = {&gp->X, &gp->Xs, &gp->y, &gp->K, &gp->L, &gp->W, &gp->WT, &gp->T,
                      &gp->alphav, &gp->v1, &gp->v2, &gp->ls, &gp->xf, &gp->info, &gp->part,
                      &gp->pscratch, &gp->xc, &gp->out_acq, &gp->out_mu, &gp->out_sd, &gp->sel,
                      &gp->clamp, &gp->s_ksm, &gp->s_partial, &gp->s_mupart, &gp->s_unit, &gp->s_rb, &gp->s_colsq,
                      &gp->tc_linv, &gp->cov_xc, &gp->cov_kst, &gp->cov_v, &gp->cov_c, &gp->cov_out, &gp->cov_mu,
                      &gp->sel_cta, &gp->pbounds, &gp->prow, &gp->pside, &gp->prune_key, &gp->surv, &gp->pilot,
                      &gp->prune_cnt};
    for (DevBuf* b : bufs) b->release();
    if (gp->stream) cudaStreamDestroy(gp->stream);
    if (gp->fgraph_exec) cudaGraphExecDestroy(gp->fgraph_exec);
    if (gp->cap_stream) cudaStreamDestroy(gp->cap_stream);
    if (gp->bulk_stream) cudaStreamDestroy(gp->bulk_stream);
    if (gp->ev_chain) cudaEventDestroy(gp->ev_chain);
    if (gp->ev_bulk) cudaEventDestroy(gp->ev_bulk);
    if (gp->copy_stream) cudaStreamDestroy(gp->copy_stream);
    if (gp->exec_stream) cudaStreamDestroy(gp->exec_stream);
    for (int i = 0; i < 2; ++i) {
        if (gp->chunk_up[i]) cudaEventDestroy(gp->chunk_up[i]);
        if (gp->chunk_done[i]) cudaEventDestroy(gp->chunk_done[i]);
    }
    if (gp->ev0) cudaEventDestroy(gp->ev0);
    if (gp->ev1) cudaEventDestroy(gp->ev1);
    if (g_last_timed == gp) g_last_timed = nullptr;
    delete gp;
}

extern "C" int64_t b200bo_gp_n(const b200bo_gp* gp) { return gp ? gp->n : 0; }
extern "C" int b200bo_gp_dim(const b200bo_gp* gp) { return gp ? gp->d : 0; }

extern "C" int b200bo_gp_set_precision(b200bo_gp* gp, int precision) {
    if (!gp) return set_err(B200BO_ERR_ARG, "gp is NULL");
    if (precision != B200BO_PRECISION_FP64 && precision != B200BO_PRECISION_FP32)
        return set_err(B200BO_ERR_ARG, "unknown precision %d", precision);
    gp->precision = precision;
    return B200BO_OK;
}

extern "C" int b200bo_gp_set_private_stream(b200bo_gp* gp, int enable) {
    if (!gp) return set_err(B200BO_ERR_ARG, "gp is NULL");
    CU(cudaSetDevice(gp->device));
    if (enable && !gp->stream) {
        CU(cudaStreamCreate(&gp->stream));  // a blocking stream: still ordered against legacy-stream work
    } else if (!enable && gp->stream) {
        CU(cudaStreamSynchronize(gp->stream));
        CU(cudaStreamDestroy(gp->stream));
        gp->stream = nullptr;
    }
    return B200BO_OK;
}

extern "C" int b200bo_gp_set_transform(b200bo_gp* gp, const int32_t* xform, int d) {
    if (!gp) return set_err(B200BO_ERR_ARG, "gp is NULL");
    gp->xform.clear();
    if (xform) {
        if (d <= 0 || d > B200BO_MAX_DIM) return set_err(B200BO_ERR_ARG, "bad d=%d", d);
        for (int j = 0; j < d; ++j) {
            if (xform[j] != B200BO_XFORM_IDENTITY && xform[j] != B200BO_XFORM_ROUND)
                return set_err(B200BO_ERR_UNSUPPORTED, "transform code %d unsupported", xform[j]);
            gp->xform.push_back(xform[j]);
        }
    }
    gp->fitted = false;
    return B200BO_OK;
}

// ---------------------------------------------------------------------------------------
// data upload + y normalisation (SK/gaussian_process/_gpr.py:275-285)
// ---------------------------------------------------------------------------------------
extern "C" int b200bo_gp_set_data(b200bo_gp* gp, const double* X, const double* y, int64_t n, int d,
                                  int normalize_y) {
    if (!gp || !X || !y) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (n <= 0 || d <= 0 || d > B200BO_MAX_DIM)
        return set_err(B200BO_ERR_ARG, "bad shape n=%lld d=%d (d <= %d)", (long long)n, d, B200BO_MAX_DIM);
    if (n > 46000) return set_err(B200BO_ERR_ARG, "n=%lld too large", (long long)n);
    if (!gp->xform.empty() && (int)gp->xform.size() != d)
        return set_err(B200BO_ERR_ARG, "transform has %zu entries, d=%d", gp->xform.size(), d);
    CU(cudaSetDevice(gp->device));
    StreamScope scope(gp);
    gp->fitted = false;
    gp->replica = false;
    gp->tc_valid = false;
    gp->n = n;
    gp->d = d;
    gp->np = round_up(n, kPad);
    const size_t np = gp->np;
    // y statistics in the order numpy uses for small arrays is irrelevant at 1e-16; use
    // a compensated sum so the result is the correctly rounded mean / population std.
    double mean = 0.0, sd = 1.0;
    gp->y_norm.assign(y, y + n);
    gp->y_raw.assign(y, y + n);
    gp->normalize = normalize_y != 0;
    if (normalize_y) {
        long double s = 0.0L;
        for (int64_t i = 0; i < n; ++i) s += y[i];
        mean = (double)(s / (long double)n);
        long double q = 0.0L;
        for (int64_t i = 0; i < n; ++i) {
            const long double t = (long double)y[i] - (long double)mean;
            q += t * t;
        }
        sd = (double)sqrtl(q / (long double)n);
        if (sd == 0.0) sd = 1.0;
        for (int64_t i = 0; i < n; ++i) gp->y_norm[i] = (y[i] - mean) / sd;
    }
    gp->y_mean = mean;
    gp->y_std = sd;
    int rc;
    if ((rc = gp->X.reserve(sizeof(double) * np * d))) return rc;
    if ((rc = gp->Xs.reserve(sizeof(double) * np * d))) return rc;
    if ((rc = gp->y.reserve(sizeof(double) * np))) return rc;
    if ((rc = gp->alphav.reserve(sizeof(double) * np))) return rc;
    if ((rc = gp->v1.reserve(sizeof(double) * np))) return rc;
    if ((rc = gp->v2.reserve(sizeof(double) * np))) return rc;
    if ((rc = gp->ls.reserve(sizeof(double) * B200BO_MAX_DIM))) return rc;
    if ((rc = gp->xf.reserve(sizeof(int) * B200BO_MAX_DIM))) return rc;
    if ((rc = gp->info.reserve(sizeof(int)))) return rc;
    if ((rc = gp->part.reserve(sizeof(double) * 64))) return rc;
    if ((rc = gp->K.reserve(sizeof(double) * np * np))) return rc;
    if ((rc = gp->L.reserve(sizeof(double) * np * np))) return rc;
    if ((rc = gp->W.reserve(sizeof(double) * np * np))) return rc;
    if ((rc = gp->WT.reserve(sizeof(double) * np * np))) return rc;
    if ((rc = gp->T.reserve(sizeof(double) * np * np))) return rc;
    if ((rc = h2d(gp->X.p, X, sizeof(double) * n * d))) return rc;
    CU(cudaMemsetAsync(gp->y.p, 0, sizeof(double) * np, g_st));
    if ((rc = h2d(gp->y.p, gp->y_norm.data(), sizeof(double) * n))) return rc;
    if (!gp->xform.empty() && (rc = h2d(gp->xf.p, gp->xform.data(), sizeof(int) * d))) return rc;
    if ((rc = sync_fit_stream())) return rc;  // the caller may release X / y on return
    gp->has_data = true;
    return B200BO_OK;
}

static int check_kernel(const b200bo_gp* gp, const b200bo_kernel* k) {
    if (!k || !k->length_scale) return set_err(B200BO_ERR_ARG, "kernel/length_scale is NULL");
    if (k->family != B200BO_KERNEL_MATERN && k->family != B200BO_KERNEL_RBF)
        return set_err(B200BO_ERR_UNSUPPORTED, "kernel family %d unsupported", k->family);
    if (k->family == B200BO_KERNEL_MATERN && (k->nu < B200BO_NU_05 || k->nu > B200BO_NU_INF))
        return set_err(B200BO_ERR_UNSUPPORTED, "Matern nu code %d unsupported", k->nu);
    if (k->n_length_scale != 1 && k->n_length_scale != gp->d)
        return set_err(B200BO_ERR_ARG, "n_length_scale=%d must be 1 or d=%d", k->n_length_scale, gp->d);
    for (int j = 0; j < k->n_length_scale; ++j)
        if (!(k->length_scale[j] > 0.0)) return set_err(B200BO_ERR_ARG, "length_scale must be > 0");
    if (!(k->const_value > 0.0)) return set_err(B200BO_ERR_ARG, "const_value must be > 0");
    if (!(k->noise_level >= 0.0)) return set_err(B200BO_ERR_ARG, "noise_level must be >= 0");
    return B200BO_OK;
}

static int potrf_mode() {  // 0 look-ahead (default), 1 serial blocked, 2 legacy unblocked
    const char* pv = getenv("B200BO_POTRF");
    if (pv && (pv[0] == 'l' || pv[0] == 'L')) return 2;
    if (pv && (pv[0] == 's' || pv[0] == 'S')) return 1;
    return 0;
}
static int trail_kernel() {  // 1: 64x128 tiles, 2 CTAs/SM (default); 0: the generic 128x128 GEMM (B200BO_TRAIL=gemm)
    const char* e = getenv("B200BO_TRAIL");
    return (e && e[0] == 'g') ? 0 : 1;
}
static bool gemm_force64() {
    const char* e = getenv("B200BO_GEMM");
    return e && e[0] == '6';
}

static int ensure_bulk_stream(b200bo_gp* gp) {
    if (!gp->bulk_stream) {
        CU(cudaStreamCreateWithFlags(&gp->bulk_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&gp->ev_chain, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&gp->ev_bulk, cudaEventDisableTiming));
    }
    return B200BO_OK;
}

template <bool TA, bool TB>
static int gemm(int M, int N, int K, double alpha, const double* A, int lda, long long sA,
                const double* B, int ldb, long long sB, double beta, double* C, int ldc,
                long long sC, int batch, int lower_only, int kmode, int skip = 0, const cudaStream_t* stp = nullptr,
                double* side = nullptr) {
    if (M <= 0 || N <= 0 || K <= 0 || batch <= 0) return B200BO_OK;
    const cudaStream_t st = stp ? *stp : g_st;
    // 128x128 pipelined tiles wherever a tile can be filled; the 64x64 kernel for narrow panels / small blocks
    if (M >= 128 && N >= 128 && !gemm_force64()) {
        dim3 grid((N + 127) / 128, (M + 127) / 128, batch);
        dgemm128_kernel<TA, TB><<<grid, 256, kGemm128SmemBytes, st>>>(M, N, K, alpha, A, lda, sA, B, ldb, sB, beta,
                                                                      C, ldc, sC, lower_only, kmode, skip, side);
    } else {
        dim3 grid(N / 64, M / 64, batch);
        dgemm64_kernel<TA, TB><<<grid, 256, 0, st>>>(M, N, K, alpha, A, lda, sA, B, ldb, sB, beta, C, ldc, sC,
                                                     lower_only, kmode, skip);
    }
    LAUNCHED();
    CU(cudaGetLastError());
    return B200BO_OK;
}

// K build + Cholesky + explicit triangular inverse.  On return L holds the clean lower factor,
// W = L^-1 (lower).  *info_out = 0 or the failing pivot (1-based).
static int transpose_W(b200bo_gp* gp);
static int solve_alpha(b200bo_gp* gp);

// Everything of a factorisation whose kernel ARGUMENTS do not depend on the hyper-parameters: K -> L, blocked
// Cholesky, zeroing of the upper triangle, L^-1 by recursive doubling, its transpose, alpha_ = K^-1 y.  Issued on g_st
// (+ the bulk stream of the look-ahead); no host synchronisation, no allocation: the sequence is CUDA-graph capturable.
// A non-positive pivot is replaced by 1 inside the diagonal kernel (arithmetic stays finite) and reported through
// gp->info, which the caller reads afterwards.
static int factor_body(b200bo_gp* gp) {
    const int np = gp->np;
    int rc;
    double* L = gp->L.as<double>();
    double* W = gp->W.as<double>();
    double* T = gp->T.as<double>();
    CU(cudaMemcpyAsync(L, gp->K.p, sizeof(double) * (size_t)np * np, cudaMemcpyDeviceToDevice, g_st));
    CU(cudaMemsetAsync(W, 0, sizeof(double) * (size_t)np * np, g_st));
    CU(cudaMemsetAsync(gp->info.p, 0, sizeof(int), g_st));
    // right-looking blocked Cholesky, panel width 64.  B200BO_POTRF=legacy selects the first
    // (unblocked) diagonal-block kernel, B200BO_POTRF=serial the blocked kernel without look-ahead, for A/B
    // measurements.
    const bool legacy_potrf = potrf_mode() == 2, serial_potrf = potrf_mode() == 1;
    if (legacy_potrf || serial_potrf || np <= 128) {
        for (int j0 = 0; j0 < np; j0 += 64) {
            if (legacy_potrf)
                potrf_diag_legacy_kernel<<<1, 256, kPotrfLegacySmemBytes, g_st>>>(L, np, j0, W + (size_t)j0 * np + j0, np,
                                                                            gp->info.as<int>());
            else
                potrf_diag_kernel<<<1, 256, kPotrfSmemBytes, g_st>>>(L, np, j0, W + (size_t)j0 * np + j0, np,
                                                               gp->info.as<int>(), nullptr, nullptr, 0);
            LAUNCHED();
            const int below = np - j0 - 64;
            if (below > 0) {
                double* panel = L + (size_t)(j0 + 64) * np + j0;
                // L_ij = A_ij * inv(L_jj)^T
                if ((rc = gemm<false, true>(below, 64, 64, 1.0, panel, np, 0, W + (size_t)j0 * np + j0, np, 0,
                                            0.0, panel, np, 0, 1, 0, 0)))
                    return rc;
                // trailing update (lower tiles only): A_ik -= L_ij L_kj^T
                if ((rc = gemm<false, true>(below, below, 64, -1.0, panel, np, 0, panel, np, 0, 1.0,
                                            L + (size_t)(j0 + 64) * np + j0 + 64, np, 0, 1, 1, 0)))
                    return rc;
            }
        }
    } else {
        // Look-ahead: the 64 diagonal blocks are a dependent chain of single-CTA kernels; everything else of a
        // step (panel solve, trailing update) is bulk work for the whole GPU.  The chain runs on the handle's
        // stream, the bulk on a second stream; the diagonal kernel of step j+1 resolves its dependence on
        // panel j itself (potrf_diag_kernel, look-ahead form) from a copy of A[j+1, j] taken before the bulk
        // panel solve, and the bulk trailing update leaves block (j+1, j+1) alone.  Every value is produced by
        // exactly one kernel: the result does not depend on how the two streams interleave.
        const cudaStream_t sb = gp->bulk_stream;
        // A[j+1, j] as it is BEFORE the bulk panel solve of panel j overwrites it in place: produced by the trailing
        // update of panel j-1 (its epilogue stores that block a second time, densely), double-buffered by step parity
        double* Pside[2] = {gp->pside.as<double>(), gp->pside.as<double>() + 64 * 64};
        CU(cudaEventRecord(gp->ev_chain, g_st));
        CU(cudaStreamWaitEvent(sb, gp->ev_chain, 0));  // K build / copies issued so far
        copy_block64_kernel<<<1, 256, 0, sb>>>(L + (size_t)64 * np, np, Pside[1]);  // A[1, 0]: no earlier panel touches it
        LAUNCHED();
        CU(cudaEventRecord(gp->ev_bulk, sb));
        potrf_diag_kernel<<<1, 256, kPotrfSmemBytes, g_st>>>(L, np, 0, W, np, gp->info.as<int>(), nullptr, nullptr, 0);
        LAUNCHED();
        CU(cudaEventRecord(gp->ev_chain, g_st));
        for (int j0 = 0, j = 0; j0 + 64 < np; j0 += 64, ++j) {
            const int below = np - j0 - 64;
            double* panel = L + (size_t)(j0 + 64) * np + j0;  // rows below the diagonal block, columns of panel j
            const double* Dj = W + (size_t)j0 * np + j0;
            // chain: diagonal block j+1.  Its inputs: Pside[(j+1)&1] (written by the trailing update of panel j-1, or the
            // initial copy) and A[j+1, j+1] with the updates of panels < j - both complete when ev_bulk (recorded after
            // that trailing update) has fired; inv(L_jj) comes from the previous kernel of this stream.
            CU(cudaStreamWaitEvent(g_st, gp->ev_bulk, 0));
            potrf_diag_kernel<<<1, 256, kPotrfSmemBytes, g_st>>>(L, np, j0 + 64, W + (size_t)(j0 + 64) * np + j0 + 64, np,
                                                           gp->info.as<int>(), Pside[(j + 1) & 1], Dj, np);
            LAUNCHED();
            // bulk: panel solve (needs inv(L_jj): ev_chain of the PREVIOUS chain kernel), then the trailing update of
            // panel j on everything but block (j+1, j+1); it also leaves A[j+2, j+1] in Pside[j&1] for the next step
            CU(cudaStreamWaitEvent(sb, gp->ev_chain, 0));
            CU(cudaEventRecord(gp->ev_chain, g_st));  // re-recorded AFTER the wait above was enqueued: now marks step j+1
            if ((rc = gemm<false, true>(below, 64, 64, 1.0, panel, np, 0, Dj, np, 0, 0.0, panel, np, 0, 1, 0, 0, 0, &sb)))
                return rc;
            if (below >= 1024 && !gemm_force64() && trail_kernel() == 1) {  // large updates only: measured no gain below
                dim3 grid((below + 127) / 128, below / 64);
                trailing_update64_kernel<<<grid, 256, kTrailSmemBytes, sb>>>(below, panel, np, L + (size_t)(j0 + 64) * np + j0 + 64,
                                                                            np, 64, Pside[j & 1]);
                LAUNCHED();
                CU(cudaGetLastError());
            } else if ((rc = gemm<false, true>(below, below, 64, -1.0, panel, np, 0, panel, np, 0, 1.0,
                                               L + (size_t)(j0 + 64) * np + j0 + 64, np, 0, 1, 1, 0, 64, &sb, Pside[j & 1])))
                return rc;
            CU(cudaEventRecord(gp->ev_bulk, sb));
        }
        CU(cudaEventRecord(gp->ev_bulk, sb));
        CU(cudaStreamWaitEvent(g_st, gp->ev_bulk, 0));
    }
    {
        dim3 blk(32, 8), grd((np + 31) / 32, (np + 7) / 8);
        zero_upper_kernel<<<grd, blk, 0, g_st>>>(L, np);
        LAUNCHED();
    }
    // W = L^-1 by recursive doubling over diagonal blocks:
    //   inv([[A,0],[C,B]]) = [[A^-1,0],[-B^-1 C A^-1, B^-1]]
    for (int s = 64; s < np; s *= 2) {
        const int full = np / (2 * s);
        const int rem = np % (2 * s);
        const long long stride = (long long)2 * s * ((long long)np + 1);
        if (full > 0) {
            // T = C * A^-1      (A^-1 lower-triangular: k >= n0)
            if ((rc = gemm<false, false>(s, s, s, 1.0, L + (size_t)s * np, np, stride, W, np, stride, 0.0,
                                         T + (size_t)s * np, np, stride, full, 0, 2)))
                return rc;
            // W21 = -B^-1 * T   (B^-1 lower-triangular: k < m0 + 64)
            if ((rc = gemm<false, false>(s, s, s, -1.0, W + (size_t)s * np + s, np, stride,
                                         T + (size_t)s * np, np, stride, 0.0, W + (size_t)s * np, np,
                                         stride, full, 0, 1)))
                return rc;
        }
        if (rem > s) {
            const int m2 = rem - s;
            const size_t o = (size_t)full * 2 * s;
            const double* C = L + (o + s) * np + o;
            double* Tt = T + (o + s) * np + o;
            if ((rc = gemm<false, false>(m2, s, s, 1.0, C, np, 0, W + o * np + o, np, 0, 0.0, Tt, np, 0, 1,
                                         0, 2)))
                return rc;
            if ((rc = gemm<false, false>(m2, s, m2, -1.0, W + (o + s) * np + o + s, np, 0, Tt, np, 0, 0.0,
                                         W + (o + s) * np + o, np, 0, 1, 0, 1)))
                return rc;
        }
    }
    CU(cudaGetLastError());
    if ((rc = transpose_W(gp))) return rc;
    return solve_alpha(gp);
}


// One LML evaluation is ~350 dependent launches and ~250 event operations: issued one by one the HOST is the
// bottleneck (2-3 us per call, the kernels of a 64-wide step are shorter than that).  The sequence has the same
// arguments whatever theta is, so it is captured ONCE per handle and training-set size into a CUDA graph (both
// streams of the look-ahead join the capture) and replayed with one call.  B200BO_GRAPH=0 issues it directly.
static int run_factor(b200bo_gp* gp) {
    int rc;
    if ((rc = ensure_bulk_stream(gp))) return rc;
    if ((rc = gp->pside.reserve(sizeof(double) * 2 * 64 * 64))) return rc;
    // graphs pay off where the launch-by-launch host cost matters (measured: N=4096 5.70 vs 5.92 ms; N=1024 no gain) and
    // cost a capture + instantiation per handle and size: used from np >= 2048 (B200BO_GRAPH=0 never, =1 always)
    const char* ge = getenv("B200BO_GRAPH");
    if ((ge && ge[0] == '0') || (!(ge && ge[0] == '1') && gp->np < 2048)) return factor_body(gp);
    const unsigned long long key[] = {(unsigned long long)gp->np, (unsigned long long)gp->K.p, (unsigned long long)gp->L.p,
                                      (unsigned long long)gp->W.p, (unsigned long long)gp->WT.p, (unsigned long long)gp->T.p,
                                      (unsigned long long)gp->alphav.p, (unsigned long long)gp->y.p, (unsigned long long)gp->v1.p,
                                      (unsigned long long)gp->v2.p, (unsigned long long)gp->info.p, (unsigned long long)gp->pside.p,
                                      (unsigned long long)(potrf_mode() * 4 + trail_kernel() * 2 + (gemm_force64() ? 1 : 0))};
    constexpr int NKEY = sizeof(key) / sizeof(key[0]);
    if (!gp->fgraph_exec || memcmp(key, gp->fgraph_key, sizeof(key)) != 0) {
        if (gp->fgraph_exec) {
            cudaGraphExecDestroy(gp->fgraph_exec);
            gp->fgraph_exec = nullptr;
        }
        if (!gp->cap_stream) CU(cudaStreamCreateWithFlags(&gp->cap_stream, cudaStreamNonBlocking));
        const long long before = g_launches.load();
        cudaStream_t saved = g_st;
        g_st = gp->cap_stream;
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(gp->cap_stream, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            rc = factor_body(gp);
            e = cudaStreamEndCapture(gp->cap_stream, &graph);
            if (rc == B200BO_OK && e == cudaSuccess) e = cudaGraphInstantiate(&gp->fgraph_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
        }
        g_st = saved;
        gp->fgraph_nodes = g_launches.load() - before;
        g_launches.store(before);  // nothing ran during the capture
        if (rc != B200BO_OK || e != cudaSuccess || !gp->fgraph_exec) {
            cudaGetLastError();
            gp->fgraph_exec = nullptr;
            static bool warned = false;
            if (!warned) {
                warned = true;
                fprintf(stderr, "b200bo: CUDA-graph capture of the factorisation failed (%s); issuing the launches directly\n",
                        e != cudaSuccess ? cudaGetErrorString(e) : g_err);
            }
            return factor_body(gp);
        }
        static_assert(NKEY <= 16, "key");
        memcpy(gp->fgraph_key, key, sizeof(key));
    }
    CU(cudaGraphLaunch(gp->fgraph_exec, g_st));
    g_launches.fetch_add(gp->fgraph_nodes, std::memory_order_relaxed);
    return B200BO_OK;
}

// K build + Cholesky + explicit triangular inverse + alpha_.  On return L holds the clean lower factor,
// W = L^-1 (lower), WT its transpose.  *info_out = 0 or the failing pivot (1-based).
static int factorize(b200bo_gp* gp, const b200bo_kernel* kern, double jitter, int* info_out) {
    const int n = (int)gp->n, np = gp->np, d = gp->d;
    double ls[B200BO_MAX_DIM];
    for (int j = 0; j < d; ++j) ls[j] = kern->length_scale[kern->n_length_scale == 1 ? 0 : j];
    int rc;
    if ((rc = h2d(gp->ls.p, ls, sizeof(double) * d))) return rc;
    const int* xf = gp->xform.empty() ? nullptr : gp->xf.as<int>();
    {
        const long long tot = (long long)np * d;
        scale_x_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, g_st>>>(gp->X.as<double>(), gp->ls.as<double>(), xf,
                                                               gp->Xs.as<double>(), n, np, d);
        LAUNCHED();
    }
    {
        dim3 blk(32, 8), grd(np / 32, np / 32);
        double* Kp = gp->K.as<double>();
        const double* Xsp = gp->Xs.as<double>();
        switch (cov_code(kern->family, kern->nu)) {
            case 0: kbuild_kernel<0><<<grd, blk, 0, g_st>>>(Xsp, Kp, n, np, d, kern->const_value, jitter); break;
            case 1: kbuild_kernel<1><<<grd, blk, 0, g_st>>>(Xsp, Kp, n, np, d, kern->const_value, jitter); break;
            case 2: kbuild_kernel<2><<<grd, blk, 0, g_st>>>(Xsp, Kp, n, np, d, kern->const_value, jitter); break;
            default: kbuild_kernel<3><<<grd, blk, 0, g_st>>>(Xsp, Kp, n, np, d, kern->const_value, jitter); break;
        }
        LAUNCHED();
    }
    CU(cudaGetLastError());
    if ((rc = run_factor(gp))) return rc;
    int info = 0;
    if ((rc = d2h(&info, gp->info.p, sizeof(int)))) return rc;
    *info_out = info;
    return B200BO_OK;
}

static int transpose_W(b200bo_gp* gp) {
    const int np = gp->np;
    dim3 blk(32, 8), grd(np / 32, np / 32);
    transpose_kernel<<<grd, blk, 0, g_st>>>(gp->W.as<double>(), gp->WT.as<double>(), np);
    LAUNCHED();
    CU(cudaGetLastError());
    return B200BO_OK;
}

// alpha_ = K^-1 y via the explicit inverse factors + one step of iterative refinement
static int solve_alpha(b200bo_gp* gp) {
    const int np = gp->np;
    const int wpb = 8;  // warps per block
    dim3 blk(32 * wpb), grd((np + wpb - 1) / wpb);
    double* a = gp->alphav.as<double>();
    double* v1 = gp->v1.as<double>();
    double* v2 = gp->v2.as<double>();
    const double* y = gp->y.as<double>();
    // z = W y ; a = W^T z
    gemv_rows_kernel<<<grd, blk, 0, g_st>>>(gp->W.as<double>(), np, y, v1, np, np, 1);
    gemv_rows_kernel<<<grd, blk, 0, g_st>>>(gp->WT.as<double>(), np, v1, a, np, np, 2);
    // r = y - K a ; a += W^T W r
    gemv_rows_kernel<<<grd, blk, 0, g_st>>>(gp->K.as<double>(), np, a, v1, np, np, 0);
    residual_kernel<<<(np + 255) / 256, 256, 0, g_st>>>(y, v1, np);
    gemv_rows_kernel<<<grd, blk, 0, g_st>>>(gp->W.as<double>(), np, v1, v2, np, np, 1);
    gemv_rows_kernel<<<grd, blk, 0, g_st>>>(gp->WT.as<double>(), np, v2, v1, np, np, 2);
    axpy1_kernel<<<(np + 255) / 256, 256, 0, g_st>>>(a, v1, np);
    for (int i = 0; i < 7; ++i) LAUNCHED();
    CU(cudaGetLastError());
    return B200BO_OK;
}

extern "C" int b200bo_gp_fit(b200bo_gp* gp, const double* X, const double* y, int64_t n, int d,
                             const b200bo_kernel* kern, double alpha, int normalize_y, int64_t* info) {
    int rc;
    if ((rc = b200bo_gp_set_data(gp, X, y, n, d, normalize_y))) return rc;
    if ((rc = check_kernel(gp, kern))) return rc;
    StreamScope scope(gp);
    NvtxRange nvtx_range("b200bo:fit");
    if (info) *info = 0;
    int finfo = 0;
    if ((rc = factorize(gp, kern, alpha + kern->noise_level, &finfo))) return rc;
    if (finfo != 0) {
        if (info) *info = finfo;
        return set_err(B200BO_ERR_NOT_PD, "%d-th leading minor of the array is not positive definite", finfo);
    }
    if ((rc = sync_fit_stream())) return rc;
    gp->family = kern->family;
    gp->nu = kern->family == B200BO_KERNEL_RBF ? B200BO_NU_INF : kern->nu;
    gp->constv = kern->const_value;
    gp->jitter = alpha + kern->noise_level;
    gp->noise = kern->noise_level;
    gp->fitted = true;
    return B200BO_OK;
}

// Append one training point at the hyper-parameters of the last fit, O(N^2) (SURVEY.md 8f rank 3).
// Falls outside the padded capacity (n == np) -> B200BO_ERR_STATE: the caller refits from scratch.
extern "C" int b200bo_gp_append(b200bo_gp* gp, const double* x_new, double y_new, int64_t* info) {
    if (!gp || !x_new) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!gp->fitted) return set_err(B200BO_ERR_STATE, "GP handle is not fitted");
    if (gp->replica) return set_err(B200BO_ERR_STATE, "handle is a predict-only replica: append to the source and replicate again");
    if (gp->n >= gp->np) return set_err(B200BO_ERR_STATE, "no padding slack left (n == np): refit");
    CU(cudaSetDevice(gp->device));
    const int n = (int)gp->n, np = gp->np, d = gp->d;
    if (info) *info = 0;
    int rc;
    if ((rc = gp->xc.reserve(sizeof(double) * B200BO_MAX_DIM))) return rc;
    CU(cudaMemcpy(gp->xc.p, x_new, sizeof(double) * d, cudaMemcpyHostToDevice));
    CU(cudaMemset(gp->info.p, 0, sizeof(int)));
    const int* xf = gp->xform.empty() ? nullptr : gp->xf.as<int>();
    double* kvec = gp->v1.as<double>();
    double* lvec = gp->v2.as<double>();
    double* tvec = gp->alphav.as<double>();  // alpha_ is recomputed below; reuse as scratch
    if (n > 0) {
        append_krow_kernel<<<(n + 127) / 128, 128>>>(gp->xc.as<double>(), gp->ls.as<double>(), xf, gp->Xs.as<double>(),
                                                     gp->X.as<double>(), kvec, n, d, gp->family, gp->nu, gp->constv);
        const int wpb = 8;
        dim3 blk(32 * wpb), grd((n + wpb - 1) / wpb);
        gemv_rows_kernel<<<grd, blk>>>(gp->W.as<double>(), np, kvec, lvec, n, n, 1);   // l = W k
        append_rows_kernel<<<1, 256>>>(gp->K.as<double>(), gp->L.as<double>(), kvec, lvec, n, np,
                                       gp->constv + gp->jitter, gp->info.as<int>(), gp->part.as<double>());
        gemv_rows_kernel<<<grd, blk>>>(gp->WT.as<double>(), np, lvec, tvec, n, n, 2);  // t = W^T l
        for (int i = 0; i < 4; ++i) LAUNCHED();
    }
    int finfo = 0;
    CU(cudaMemcpy(&finfo, gp->info.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (finfo != 0) {
        gp->fitted = false;  // row n of K/L is garbage now
        if (info) *info = finfo;
        return set_err(B200BO_ERR_NOT_PD, "%d-th leading minor of the array is not positive definite", finfo);
    }
    append_winv_kernel<<<(n + 1 + 127) / 128, 128>>>(gp->W.as<double>(), gp->WT.as<double>(), tvec,
                                                     gp->part.as<double>(), n, np);
    LAUNCHED();
    // targets: new normalisation statistics, alpha_ = K^-1 y
    gp->y_raw.push_back(y_new);
    const int64_t nn = n + 1;
    gp->y_norm = gp->y_raw;
    double mean = 0.0, sd = 1.0;
    if (gp->normalize) {
        long double s = 0.0L;
        for (int64_t i = 0; i < nn; ++i) s += gp->y_raw[i];
        mean = (double)(s / (long double)nn);
        long double q = 0.0L;
        for (int64_t i = 0; i < nn; ++i) {
            const long double t = (long double)gp->y_raw[i] - (long double)mean;
            q += t * t;
        }
        sd = (double)sqrtl(q / (long double)nn);
        if (sd == 0.0) sd = 1.0;
        for (int64_t i = 0; i < nn; ++i) gp->y_norm[i] = (gp->y_raw[i] - mean) / sd;
    }
    gp->y_mean = mean;
    gp->y_std = sd;
    CU(cudaMemcpy(gp->y.p, gp->y_norm.data(), sizeof(double) * nn, cudaMemcpyHostToDevice));
    gp->n = nn;
    gp->tc_valid = false;
    if ((rc = solve_alpha(gp))) return rc;
    CU(cudaDeviceSynchronize());
    return B200BO_OK;
}

extern "C" int b200bo_gp_lml(b200bo_gp* gp, const b200bo_kernel* kern, double alpha, int has_const,
                             double* lml, double* grad) {
    if (!gp || !lml) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!gp->has_data) return set_err(B200BO_ERR_STATE, "no training data: call b200bo_gp_set_data");
    int rc;
    if ((rc = check_kernel(gp, kern))) return rc;
    CU(cudaSetDevice(gp->device));
    StreamScope scope(gp);
    NvtxRange nvtx_range("b200bo:lml");
    gp->fitted = false;  // buffers are being overwritten
    gp->tc_valid = false;
    const int n = (int)gp->n, np = gp->np, d = gp->d;
    const int aniso = kern->n_length_scale > 1;
    const int want_noise = (has_const & 2) ? 1 : 0;
    has_const &= 1;
    const int ntheta_k = (has_const ? 1 : 0) + kern->n_length_scale;  // produced by the pair kernel
    const int ntheta = ntheta_k + want_noise;
    int finfo = 0;
    if ((rc = factorize(gp, kern, alpha + kern->noise_level, &finfo))) return rc;
    if (finfo != 0) {  // SK/_gpr.py:590-593
        *lml = -std::numeric_limits<double>::infinity();
        if (grad)
            for (int p = 0; p < ntheta; ++p) grad[p] = 0.0;
        return B200BO_OK;
    }
    diag_kernel<<<(n + 255) / 256, 256, 0, g_st>>>(gp->L.as<double>(), np, gp->v1.as<double>(), n);
    LAUNCHED();
    std::vector<double> a(n), dg(n);
    if ((rc = d2h(a.data(), gp->alphav.p, sizeof(double) * n))) return rc;
    if ((rc = d2h(dg.data(), gp->v1.p, sizeof(double) * n))) return rc;
    long double ya = 0.0L, ld = 0.0L;
    for (int i = 0; i < n; ++i) {
        ya += (long double)gp->y_norm[i] * a[i];
        ld += logl((long double)dg[i]);
    }
    *lml = (double)(-0.5L * ya - ld - (long double)n / 2.0L * logl(2.0L * 3.14159265358979323846264338327950288L));
    if (grad) {
        // Kinv = W^T W  (W lower: k >= max(m0, n0)); lower tiles only - the gradient kernel uses symmetry
        if ((rc = gemm<true, false>(np, np, np, 1.0, gp->W.as<double>(), np, 0, gp->W.as<double>(), np, 0,
                                    0.0, gp->T.as<double>(), np, 0, 1, 1, 3)))
            return rc;
        size_t nblk;
        const int cov = cov_code(kern->family, kern->nu);
        if (d <= LG_DMAX) {
            // 64x64 patches on or below the diagonal, covariance and iso/aniso as template parameters
            const int nb64 = (n + 63) / 64;
            dim3 grd(nb64, nb64);
            nblk = (size_t)nb64 * (nb64 + 1) / 2;
            if ((rc = gp->part.reserve(sizeof(double) * nblk * ntheta_k))) return rc;
            const double* Xsp = gp->Xs.as<double>();
            const double* Ki = gp->T.as<double>();
            const double* al = gp->alphav.as<double>();
            double* pt = gp->part.as<double>();
#define B200BO_LG(COV)                                                                                              \
    if (aniso)                                                                                                      \
        lml_grad_tile_kernel<COV, true><<<grd, 256, 0, g_st>>>(Xsp, Ki, np, al, n, d, kern->const_value, has_const, pt, ntheta_k); \
    else                                                                                                            \
        lml_grad_tile_kernel<COV, false><<<grd, 256, 0, g_st>>>(Xsp, Ki, np, al, n, d, kern->const_value, has_const, pt, ntheta_k);
            switch (cov) {
                case 0: B200BO_LG(0) break;
                case 1: B200BO_LG(1) break;
                case 2: B200BO_LG(2) break;
                default: B200BO_LG(3) break;
            }
#undef B200BO_LG
        } else {
            dim3 grd((n + 15) / 16, (n + 15) / 16);
            nblk = (size_t)grd.x * grd.y;
            if ((rc = gp->part.reserve(sizeof(double) * nblk * ntheta_k))) return rc;
            lml_grad_kernel<<<grd, 256, 0, g_st>>>(gp->Xs.as<double>(), gp->T.as<double>(), np, gp->alphav.as<double>(),
                                                   n, d, kern->family,
                                                   kern->family == B200BO_KERNEL_RBF ? B200BO_NU_INF : kern->nu,
                                                   kern->const_value, has_const, aniso, gp->part.as<double>(), ntheta_k);
        }
        LAUNCHED();
        CU(cudaGetLastError());
        std::vector<double> part(nblk * ntheta_k);
        if ((rc = d2h(part.data(), gp->part.p, sizeof(double) * nblk * ntheta_k))) return rc;
        for (int p = 0; p < ntheta_k; ++p) {
            long double s = 0.0L;
            for (size_t b = 0; b < nblk; ++b) s += part[b * ntheta_k + p];
            grad[p] = (double)s;
        }
        if (want_noise) {
            // dK/dlog(noise_level) = noise_level * I (SK/gaussian_process/kernels.py:1311-1322):
            // grad = 0.5 * noise_level * sum_i (alpha_i^2 - (K^-1)_ii)
            diag_kernel<<<(n + 255) / 256, 256, 0, g_st>>>(gp->T.as<double>(), np, gp->v2.as<double>(), n);
            LAUNCHED();
            std::vector<double> kd(n);
            if ((rc = d2h(kd.data(), gp->v2.p, sizeof(double) * n))) return rc;
            long double sn = 0.0L;
            for (int i = 0; i < n; ++i) sn += (long double)a[i] * a[i] - (long double)kd[i];
            grad[ntheta_k] = (double)(0.5L * (long double)kern->noise_level * sn);
        }
    }
    return B200BO_OK;
}

extern "C" int b200bo_gp_get(b200bo_gp* gp, int what, double* out, int64_t len) {
    if (!gp || !out) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!gp->fitted) return set_err(B200BO_ERR_STATE, "GP handle is not fitted");
    CU(cudaSetDevice(gp->device));
    const size_t n = gp->n, np = gp->np;
    const void* src = nullptr;
    if (gp->replica && (what == B200BO_GET_L || what == B200BO_GET_K))
        return set_err(B200BO_ERR_STATE, "a predict-only replica holds no K / L: read them from the source handle");
    switch (what) {
        case B200BO_GET_L: src = gp->L.p; break;
        case B200BO_GET_K: src = gp->K.p; break;
        case B200BO_GET_LINV: src = gp->W.p; break;
        case B200BO_GET_ALPHA:
            if (len != (int64_t)n) return set_err(B200BO_ERR_ARG, "len must be n");
            CU(cudaMemcpy(out, gp->alphav.p, sizeof(double) * n, cudaMemcpyDeviceToHost));
            return B200BO_OK;
        case B200BO_GET_YSTATS:
            if (len != 2) return set_err(B200BO_ERR_ARG, "len must be 2");
            out[0] = gp->y_mean;
            out[1] = gp->y_std;
            return B200BO_OK;
        default: return set_err(B200BO_ERR_ARG, "unknown selector %d", what);
    }
    if (len != (int64_t)(n * n)) return set_err(B200BO_ERR_ARG, "len must be n*n");
    CU(cudaMemcpy2D(out, sizeof(double) * n, src, sizeof(double) * np, sizeof(double) * n, n,
                    cudaMemcpyDeviceToHost));
    return B200BO_OK;
}

// ---------------------------------------------------------------------------------------
// predict / acquisition
// ---------------------------------------------------------------------------------------
// small-batch path: work-unit tables + scratch for one GP
static int ensure_small(b200bo_gp* gp) {
    const int np = gp->np;
    if (gp->s_np == np) return B200BO_OK;
    std::vector<int2> units, rbs;
    const int nrb = np / SROWS;
    for (int i = 0; i < nrb; ++i) {
        const int K = (i + 1) * SROWS;
        const int nj = (K + SKCH - 1) / SKCH;
        rbs.push_back(make_int2((int)units.size(), nj));
        for (int j = 0; j < nj; ++j) units.push_back(make_int2(i, j));
    }
    int rc;
    if ((rc = gp->s_unit.reserve(sizeof(int2) * units.size()))) return rc;
    if ((rc = gp->s_rb.reserve(sizeof(int2) * rbs.size()))) return rc;
    if ((rc = gp->s_ksm.reserve(sizeof(double) * (size_t)SMAXP * np * SMC))) return rc;
    if ((rc = gp->s_partial.reserve(sizeof(double) * (size_t)SMAXP * units.size() * SROWS * SMC))) return rc;
    if ((rc = gp->s_mupart.reserve(sizeof(double) * (size_t)SMAXP * (np / 128) * SMC))) return rc;
    if ((rc = gp->s_colsq.reserve(sizeof(double) * (size_t)SMAXP * (np / SROWS) * SMC))) return rc;
    CU(cudaMemcpy(gp->s_unit.p, units.data(), sizeof(int2) * units.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(gp->s_rb.p, rbs.data(), sizeof(int2) * rbs.size(), cudaMemcpyHostToDevice));
    gp->s_np = np;
    gp->s_nunits = (int)units.size();
    return B200BO_OK;
}

// Cost model (microseconds, measured orders of magnitude on B200) choosing between the tiled
// persistent kernel and the small-batch path.  B200BO_SMALL_PATH=0/1 forces one of them.
// B200BO_PATH_STABLE: the decision is taken for a nominal batch of one pass (SMC rows) whatever m is,
// so an optimiser's f(x) and its finite-difference stencil always run through the same kernels.
static bool use_small_path(long long m, int np_max, int n_gps, int sm_count, int path) {
    const char* e = getenv("B200BO_SMALL_PATH");
    if (e && (e[0] == '0' || e[0] == '1')) return e[0] == '1';
    if (m <= 0) return false;
    if (path == B200BO_PATH_STABLE) m = SMC;
    const double x = (np_max / 4096.0) * (np_max / 4096.0);
    const double passes = (double)((m + SMC - 1) / SMC);
    const double tiles = (double)((m + PBN - 1) / PBN);
    const double t_small = passes * (15.0 + 60.0 * x) * n_gps;
    const double t_big = std::ceil(tiles / sm_count) * (10.0 + 9000.0 * x) * n_gps;
    return t_small < t_big;
}

// GEMM inner-loop variant of the fused predict kernel: "dmma" (mma.sync m8n8k4 f64, default) or
// "dfma" (8x8 register tiles).  Both are exact fp64 with fixed-order reductions; the environment
// variable B200BO_PREDICT_IMPL selects one for A/B measurements.
static int predict_impl(int precision) {
    const char* e = getenv("B200BO_PREDICT_IMPL");
    if (e && (e[0] == 'd' || e[0] == 'D') && (e[1] == 'f' || e[1] == 'F')) return PREDICT_IMPL_DFMA;
    if (e && (e[0] == 't' || e[0] == 'T')) return PREDICT_IMPL_TF32;  // "tf32": fp32 mode on tcgen05
    if (e && (e[0] == 'd' || e[0] == 'D')) return PREDICT_IMPL_DMMA;
    return precision == B200BO_PRECISION_FP32 ? PREDICT_IMPL_TF32 : PREDICT_IMPL_DMMA;
}

// 8-warp (predict_acq_kernel) or 16-warp (predict_acq16_kernel) version of the fp64 kernel;
// B200BO_PREDICT_WARPS=8|16 overrides the default for A/B measurements
static int predict_warps() {
    const char* e = getenv("B200BO_PREDICT_WARPS");
    if (e && e[0] == '1' && e[1] == '6') return 16;
    if (e && e[0] == '8') return 8;
    return kDefaultPredictWarps;
}

// fp32 mode operand images of L^-1 (once per fit)
static int ensure_tc(b200bo_gp* gp, cudaStream_t stream) {
    if (gp->tc_valid) return B200BO_OK;
    const int np = gp->np;
    int rc;
    if ((rc = gp->tc_linv.reserve((size_t)(np / PBM) * (np / tc::kTcK) * 2 * tc::kTcImgBytes))) return rc;
    dim3 grid(np / tc::kTcK, np / PBM);
    pretile_linv_tc_kernel<<<grid, 256, 0, stream>>>(gp->W.as<double>(), np, gp->tc_linv.as<uint8_t>());
    LAUNCHED();
    CU(cudaGetLastError());
    gp->tc_valid = true;
    return B200BO_OK;
}

static int check_spec(const b200bo_acq* spec) {
    if (!spec) return set_err(B200BO_ERR_ARG, "spec is NULL");
    if (spec->n_gps < 1 || spec->n_gps > B200BO_MAX_GPS)
        return set_err(B200BO_ERR_ARG, "n_gps=%d out of range [1,%d]", spec->n_gps, B200BO_MAX_GPS);
    if (spec->kind < B200BO_ACQ_UCB || spec->kind > B200BO_ACQ_NONE)
        return set_err(B200BO_ERR_ARG, "unknown acquisition kind %d", spec->kind);
    if (spec->path != B200BO_PATH_AUTO && spec->path != B200BO_PATH_STABLE)
        return set_err(B200BO_ERR_ARG, "unknown path policy %d", spec->path);
    for (int g = 0; g < spec->n_gps; ++g) {
        const b200bo_gp* gp = spec->gps[g];
        if (!gp) return set_err(B200BO_ERR_ARG, "gps[%d] is NULL", g);
        if (!gp->fitted) return set_err(B200BO_ERR_STATE, "gps[%d] is not fitted", g);
        if (gp->d != spec->gps[0]->d) return set_err(B200BO_ERR_ARG, "gps[%d] has a different dimension", g);
        if (gp->device != spec->gps[0]->device)
            return set_err(B200BO_ERR_ARG, "gps[%d] lives on a different device", g);
        if (g >= 1 && !(spec->lb[g] < spec->ub[g]))
            return set_err(B200BO_ERR_ARG, "constraint %d: lb must be < ub", g);
    }
    return B200BO_OK;
}

// Where a launch's candidates come from: a device matrix (parity mode: the reference's host MT19937 stream,
// uploaded) or the in-kernel Philox generator (throughput mode).
struct CandSrc {
    const double* d_Xc = nullptr;
    bool philox = false;
    uint64_t seed = 0;
    const double* lo = nullptr;  // host, d entries
    const double* hi = nullptr;
};

// resume != 0: the per-CTA selection lists of the previous launch on this handle are continued instead of
// re-initialised (chunked batches: one merge after the last chunk); finish == 0 skips the merge.
// m_call: candidates of the whole chunked call (0: this launch's m).
struct SelMode {
    int resume = 0;
    int finish = 1;
    long long m_call = 0;
};

template <int MODE>
static void launch16(bool dreg, int grid, const PredictParams& P, cudaStream_t stream) {
    if (dreg)
        predict_acq16_kernel<true, MODE><<<grid, P16_NT, kPredictSmemBytesDmma, stream>>>(P);
    else
        predict_acq16_kernel<false, MODE><<<grid, P16_NT, kPredictSmemBytesDmma, stream>>>(P);
    LAUNCHED();
}

// Pruned selection (DESIGN.md 4.1): whether a fused-selection call takes it.  The acquisition must grow with
// sigma; the records alone are asked for; the screen (phase A + kScreenBlocks row blocks per candidate) must be
// a small part of the full product (np >= 8 row blocks); and the batch must span enough waves of tiles to repay
// the two full-tile latencies of the pilot and the survivor launch (measured, DESIGN.md 6).
constexpr int kPruneMinBlocks = 8;
constexpr long long kPruneMinWaves = 4;

static bool prune_eligible(const b200bo_acq* spec, long long m_call, int np_max, int sm_count) {
    const bool monotone = spec->kind == B200BO_ACQ_EI || spec->kind == B200BO_ACQ_POI ||
                          (spec->kind == B200BO_ACQ_UCB && spec->kappa >= 0.0);
    return monotone && spec->n_gps == 1 && np_max >= kPruneMinBlocks * PBM &&
           (m_call + PBN - 1) / PBN >= kPruneMinWaves * sm_count;
}

// screen -> pilot (first launch of a call only: tau = k-th exact key of the candidates with the k smallest bounds
// of each screen CTA; chunks after the first keep it) -> compaction of the survivors' coordinates (so chunk
// buffers can be reused), and on the finishing launch one gather launch over all survivors into the per-CTA lists
// P.sel_cta (grid sm_count) that the caller merges.  No host synchronisation; the counters stay on the device.
static int launch_pruned(b200bo_gp* g0, const PredictParams& P, int grid, bool dreg, const SelMode& sm,
                         long long m_call, void* d_sel, cudaStream_t stream) {
    int rc;
    const int d = P.d, k = P.sel_k, nsm = g0->sm_count;
    const size_t pilot_cap = (size_t)nsm * k;
    if ((rc = g0->prune_key.reserve(sizeof(unsigned long long) * (size_t)P.m))) return rc;
    if ((rc = g0->prune_cnt.reserve(3 * sizeof(unsigned long long)))) return rc;
    if ((rc = g0->pilot.reserve(sizeof(double) * pilot_cap * (d + 1)))) return rc;
    if ((rc = g0->surv.reserve(sizeof(double) * (size_t)m_call * (d + 1)))) return rc;
    unsigned long long* cnt = g0->prune_cnt.as<unsigned long long>();
    const GatherBuf pilot{g0->pilot.as<double>(), reinterpret_cast<long long*>(g0->pilot.as<double>() + pilot_cap * d),
                          cnt + 1};
    const GatherBuf surv{g0->surv.as<double>(), reinterpret_cast<long long*>(g0->surv.as<double>() + (size_t)m_call * d),
                         cnt};
    if (!sm.resume) CU(cudaMemsetAsync(cnt, 0, 2 * sizeof(unsigned long long), stream));
    PredictParams S = P;
    S.screen_key = g0->prune_key.as<unsigned long long>();
    S.sel_resume = 0;
    launch16<P16_SCREEN>(dreg, grid, S, stream);
    PredictParams G = P;
    G.m = 0;
    G.sel_resume = 0;
    if (!sm.resume) {
        prune_pilot_kernel<<<grid, SEL_MAXK, 0, stream>>>(P, P.sel_cta, k, pilot);
        G.gather_x = pilot.x;
        G.gather_idx = pilot.idx;
        G.gather_count = pilot.count;
        launch16<P16_GATHER>(dreg, nsm, G, stream);
        // the pilot's records go to d_sel only to derive tau: the final merge overwrites them
        merge_sel_kernel<<<1, 256, 0, stream>>>(P.sel_cta, nsm, k, reinterpret_cast<SelRecord*>(d_sel));
        prune_tau_kernel<<<1, 32, 0, stream>>>(reinterpret_cast<const SelRecord*>(d_sel), k, cnt + 2);
        LAUNCHED();
        LAUNCHED();
        LAUNCHED();
    }
    prune_compact_kernel<<<(unsigned)((P.m + 255) / 256), 256, 0, stream>>>(S, cnt + 2, surv);
    LAUNCHED();
    if (sm.finish) {
        G.gather_x = surv.x;
        G.gather_idx = surv.idx;
        G.gather_count = surv.count;
        launch16<P16_GATHER>(dreg, nsm, G, stream);
    }
    return B200BO_OK;
}

static int eval_core(const b200bo_acq* spec, const CandSrc& src, int64_t m, double* d_acq_neg, double* d_mu,
                     double* d_sd, int k, void* d_sel, int64_t index_base, cudaStream_t stream,
                     SelMode sm = SelMode()) {
    int rc;
    if ((rc = check_spec(spec))) return rc;
    if (m < 0 || (m > 0 && !src.philox && !src.d_Xc)) return set_err(B200BO_ERR_ARG, "bad candidates");
    if (src.philox && (!src.lo || !src.hi)) return set_err(B200BO_ERR_ARG, "Philox mode needs lo/hi");
    if (k < 0 || k > B200BO_MAX_TOPK) return set_err(B200BO_ERR_ARG, "k=%d out of range", k);
    if (k > 0 && !d_sel) return set_err(B200BO_ERR_ARG, "d_sel is NULL");
    b200bo_gp* g0 = spec->gps[0];
    CU(cudaSetDevice(g0->device));
    NvtxRange nvtx_range("b200bo:predict_acq");
    PredictParams P;
    memset(&P, 0, sizeof(P));
    int np_max = 0;
    for (int g = 0; g < spec->n_gps; ++g) {
        b200bo_gp* gp = spec->gps[g];
        GpDev& G = P.gp[g];
        G.Xs = gp->Xs.as<double>();
        G.linvT = gp->WT.as<double>();
        G.alphav = gp->alphav.as<double>();
        G.ls = gp->ls.as<double>();
        G.xform = gp->xform.empty() ? nullptr : gp->xf.as<int>();
        G.linv_tc = nullptr;
        G.n = (int)gp->n;
        G.np = gp->np;
        G.family = gp->family;
        G.nu = gp->nu;
        G.constv = gp->constv;
        G.prior = gp->constv + gp->noise;
        G.y_mean = gp->y_mean;
        G.y_std = gp->y_std;
        G.lb = spec->lb[g];
        G.ub = spec->ub[g];
        np_max = gp->np > np_max ? gp->np : np_max;
    }
    P.n_gps = spec->n_gps;
    P.d = g0->d;
    P.acq_kind = spec->kind;
    P.kappa = spec->kappa;
    P.xi = spec->xi;
    P.y_max = spec->y_max;
    P.Xc = src.philox ? nullptr : src.d_Xc;
    P.index_base = index_base;
    if (src.philox) {
        double pb[2 * B200BO_MAX_DIM];
        for (int j = 0; j < P.d; ++j) {
            if (!(src.lo[j] <= src.hi[j])) return set_err(B200BO_ERR_ARG, "Philox bounds: lo > hi in column %d", j);
            pb[j] = src.lo[j];
            pb[P.d + j] = src.hi[j] - src.lo[j];
        }
        if ((rc = g0->pbounds.reserve(sizeof(double) * 2 * B200BO_MAX_DIM))) return rc;
        CU(cudaMemcpyAsync(g0->pbounds.p, pb, sizeof(double) * 2 * P.d, cudaMemcpyHostToDevice, stream));
        P.pbounds = g0->pbounds.as<double>();
        P.seed = src.seed;
    }
    P.m = m;
    P.acq_out = d_acq_neg;
    P.mu_out = d_mu;
    P.sd_out = d_sd;
    if ((rc = g0->clamp.reserve(2 * sizeof(unsigned long long)))) return rc;
    P.clamp_count = g0->clamp.as<unsigned long long>();
    if (!sm.resume) CU(cudaMemsetAsync(g0->clamp.p, 0, 2 * sizeof(unsigned long long), stream));
    const long long ntiles = (m + PBN - 1) / PBN;
    int grid = (int)(ntiles < g0->sm_count ? ntiles : g0->sm_count);
    if (sm.resume || !sm.finish) grid = g0->sm_count;  // chunked batches keep one list per SM across launches
    const bool small = grid > 0 && !sm.resume && sm.finish &&
                       use_small_path(m, np_max, spec->n_gps, g0->sm_count, spec->path);
    const bool p16 = predict_impl(g0->precision) == PREDICT_IMPL_DMMA && predict_warps() == 16;
    const long long m_call = sm.m_call ? sm.m_call : m;
    const bool prune = !small && grid > 0 && k > 0 && p16 && !P.acq_out && !P.mu_out && !P.sd_out &&
                       prune_eligible(spec, m_call, np_max, g0->sm_count);
    if (!sm.resume) {
        g0->st_screened = g0->st_full = 0;
        g0->st_pruned = prune;
    }
    (prune ? g0->st_screened : g0->st_full) += m;
    bool fused_sel = false;
    if (small) {
        if (k > 0 && !P.acq_out) {  // the small path selects from the materialised values
            if ((rc = g0->out_acq.reserve(sizeof(double) * (size_t)(m > 0 ? m : 1)))) return rc;
            P.acq_out = g0->out_acq.as<double>();
        }
        SmallParams S;
        memset(&S, 0, sizeof(S));
        S.P = P;
        for (int g = 0; g < spec->n_gps; ++g) {
            b200bo_gp* gp = spec->gps[g];
            if ((rc = ensure_small(gp))) return rc;
            S.sg[g].W = gp->W.as<double>();
            S.sg[g].ksm = gp->s_ksm.as<double>();
            S.sg[g].partial = gp->s_partial.as<double>();
            S.sg[g].mu_part = gp->s_mupart.as<double>();
            S.sg[g].colsq_rb = gp->s_colsq.as<double>();
            S.sg[g].unit_tab = gp->s_unit.as<int2>();
            S.sg[g].rb_tab = gp->s_rb.as<int2>();
            S.nunits[g] = gp->s_nunits;
        }
        S.m_end = m;
        CU(cudaEventRecord(g0->ev0, stream));
        for (long long c0 = 0; c0 < m; c0 += (long long)SMAXP * SMC) {
            S.c0 = c0;
            const long long left = m - c0;
            const int npass = (int)((left + SMC - 1) / SMC < SMAXP ? (left + SMC - 1) / SMC : SMAXP);
            for (int g = 0; g < spec->n_gps; ++g) {
                small_kstar_kernel<<<dim3(spec->gps[g]->np / 128, npass), 256, 0, stream>>>(S, g);
                small_trsv_kernel<<<dim3(spec->gps[g]->s_nunits, (npass + STPG - 1) / STPG), 256, kSmallTrsvSmemBytes, stream>>>(S, g, npass);
                small_reduce_kernel<<<dim3(spec->gps[g]->np / SROWS, npass), 256, 0, stream>>>(S, g);
                LAUNCHED();
                LAUNCHED();
                LAUNCHED();
            }
            small_finish_kernel<<<npass, 256, 0, stream>>>(S);
            LAUNCHED();
        }
        CU(cudaGetLastError());
        CU(cudaEventRecord(g0->ev1, stream));
        g_last_timed = g0;
    } else if (grid > 0) {
        if (k > 0) {  // selection fused into the epilogue: no acq[M] needed
            if ((rc = g0->sel_cta.reserve(sizeof(SelList) * (size_t)g0->sm_count))) return rc;
            P.sel_cta = g0->sel_cta.as<SelList>();
            P.sel_k = k;
            P.sel_resume = sm.resume;
            fused_sel = true;
        }
        P.scratch_stride = (long long)np_max * PBN;
        if ((rc = g0->pscratch.reserve(sizeof(double) * (size_t)P.scratch_stride * g0->sm_count))) return rc;
        P.scratch = g0->pscratch.as<double>();
        CU(cudaEventRecord(g0->ev0, stream));
        const bool dreg = P.d <= kPredictMaxDimRegs;
        if (predict_impl(g0->precision) == PREDICT_IMPL_TF32) {
            for (int g = 0; g < spec->n_gps; ++g) {
                if ((rc = ensure_tc(spec->gps[g], stream))) return rc;
                P.gp[g].linv_tc = spec->gps[g]->tc_linv.as<uint8_t>();
            }
            CU(cudaEventRecord(g0->ev0, stream));  // exclude the one-off tiling from the kernel time
            const char* tv = getenv("B200BO_TC_VARIANT");  // "1": non-overlapped version, "2"/"3": see kDefaultTcVariant
            const int variant = (tv && tv[0] >= '1' && tv[0] <= '4') ? tv[0] - '0' : kDefaultTcVariant;
            if (dreg && (variant == 3 || variant == 4)) {
                // N = 256 per MMA: candidate tiles of 256, two K* image buffers of np x 2 KiB per CTA
                const long long nt3 = (m + T3N - 1) / T3N;
                if (!(sm.resume || !sm.finish)) grid = (int)(nt3 < g0->sm_count ? nt3 : g0->sm_count);
                P.scratch_stride = (long long)np_max * 512;
                if ((rc = g0->pscratch.reserve(sizeof(double) * (size_t)P.scratch_stride * g0->sm_count))) return rc;
                P.scratch = g0->pscratch.as<double>();
                if (variant == 4)
                    predict_acq_tc4_kernel<<<grid, TC2_NT, kPredictSmemBytesTc4, stream>>>(P);
                else
                    predict_acq_tc3_kernel<<<grid, TC2_NT, kPredictSmemBytesTc3, stream>>>(P);
            } else if (dreg && variant != 1) {
                // overlapped version: two K* image buffers per CTA
                P.scratch_stride *= 2;
                if (const char* dbg = getenv("B200BO_TC_DEBUG")) P.pad0 = atoi(dbg);
                if ((rc = g0->pscratch.reserve(sizeof(double) * (size_t)P.scratch_stride * g0->sm_count))) return rc;
                P.scratch = g0->pscratch.as<double>();
                predict_acq_tc2_kernel<<<grid, TC2_NT, kPredictSmemBytesTc2, stream>>>(P);
            } else if (dreg) {
                predict_acq_tc_kernel<true><<<grid, PNT, kPredictSmemBytesTc, stream>>>(P);
            } else {
                predict_acq_tc_kernel<false><<<grid, PNT, kPredictSmemBytesTc, stream>>>(P);
            }
        } else if (prune) {
            if ((rc = launch_pruned(g0, P, grid, dreg, sm, m_call, d_sel, stream))) return rc;
            grid = g0->sm_count;  // the survivors' gather launch produced the lists merged below
        } else if (p16) {
            launch16<P16_FULL>(dreg, grid, P, stream);
        } else if (predict_impl(g0->precision) == PREDICT_IMPL_DMMA) {
            if (dreg)
                predict_acq_kernel<PREDICT_IMPL_DMMA, true><<<grid, PNT, kPredictSmemBytesDmma, stream>>>(P);
            else
                predict_acq_kernel<PREDICT_IMPL_DMMA, false><<<grid, PNT, kPredictSmemBytesDmma, stream>>>(P);
        } else {
            if (dreg)
                predict_acq_kernel<PREDICT_IMPL_DFMA, true><<<grid, PNT, kPredictSmemBytesDfma, stream>>>(P);
            else
                predict_acq_kernel<PREDICT_IMPL_DFMA, false><<<grid, PNT, kPredictSmemBytesDfma, stream>>>(P);
        }
        if (!p16) LAUNCHED();  // launch16 counts its own
        CU(cudaGetLastError());
        CU(cudaEventRecord(g0->ev1, stream));
        g_last_timed = g0;
    }
    if (k > 0 && sm.finish) {
        NvtxRange nvtx_sel("b200bo:select");
        if (fused_sel) {
            merge_sel_kernel<<<1, 256, 0, stream>>>(g0->sel_cta.as<SelList>(), grid, k,
                                                    reinterpret_cast<SelRecord*>(d_sel));
        } else if (m > 0) {
            select_kernel<<<1, 1024, 0, stream>>>(P.acq_out, m, k, reinterpret_cast<SelRecord*>(d_sel), index_base);
        } else {
            CU(cudaMemsetAsync(d_sel, 0xFF, sizeof(SelRecord) * (k + 1), stream));  // empty: index -1, value NaN
        }
        LAUNCHED();
        CU(cudaGetLastError());
    }
    return B200BO_OK;
}

extern "C" int b200bo_acq_eval_dev(const b200bo_acq* spec, const double* d_Xc, int64_t m,
                                   double* d_acq_neg, double* d_mu, double* d_sd, int k, void* d_sel,
                                   int64_t index_base, void* stream_) {
    CandSrc src;
    src.d_Xc = d_Xc;
    return eval_core(spec, src, m, d_acq_neg, d_mu, d_sd, k, d_sel, index_base, (cudaStream_t)stream_);
}

extern "C" int b200bo_acq_select_philox_dev(const b200bo_acq* spec, uint64_t seed, const double* lo,
                                            const double* hi, int64_t m, int64_t index_base, int k, void* d_sel,
                                            void* stream_) {
    if (k <= 0) return set_err(B200BO_ERR_ARG, "k must be > 0");
    if (m <= 0) return set_err(B200BO_ERR_ARG, "m must be > 0");
    CandSrc src;
    src.philox = true;
    src.seed = seed;
    src.lo = lo;
    src.hi = hi;
    return eval_core(spec, src, m, nullptr, nullptr, nullptr, k, d_sel, index_base, (cudaStream_t)stream_);
}

extern "C" int b200bo_last_select_stats(int64_t* screened, int64_t* evaluated) {
    if (!screened || !evaluated) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!g_last_timed) return set_err(B200BO_ERR_STATE, "no timed kernel on this thread");
    const b200bo_gp* g = g_last_timed;
    CU(cudaSetDevice(g->device));
    CU(cudaEventSynchronize(g->ev1));
    *screened = g->st_screened;
    *evaluated = g->st_full;
    if (g->st_pruned) {
        unsigned long long c[2];
        CU(cudaMemcpy(c, g->prune_cnt.p, sizeof(c), cudaMemcpyDeviceToHost));
        *evaluated = (int64_t)(c[0] + c[1]);
    }
    return B200BO_OK;
}

extern "C" int b200bo_last_kernel_ms(float* ms) {
    if (!ms) return set_err(B200BO_ERR_ARG, "ms is NULL");
    if (!g_last_timed) return set_err(B200BO_ERR_STATE, "no timed kernel on this thread");
    CU(cudaSetDevice(g_last_timed->device));
    CU(cudaEventSynchronize(g_last_timed->ev1));
    CU(cudaEventElapsedTime(ms, g_last_timed->ev0, g_last_timed->ev1));
    return B200BO_OK;
}

// Host-buffer front end shared by predict / acq_eval / argmin_topk.  Large selection-only batches are
// streamed: the candidate matrix goes up in chunks of a whole number of tiles per SM on a copy stream while
// the previous chunk is evaluated (double-buffered device chunks), the per-CTA selection lists carry over
// from launch to launch and are merged once - the H2D copy disappears behind the kernel.
constexpr long long kChunkTilesPerSm = 8;

static int ensure_copy_stream(b200bo_gp* g0) {
    if (!g0->copy_stream) {
        CU(cudaStreamCreateWithFlags(&g0->copy_stream, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&g0->exec_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CU(cudaEventCreateWithFlags(&g0->chunk_up[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&g0->chunk_done[i], cudaEventDisableTiming));
        }
    }
    return B200BO_OK;
}

// sklearn's validate_data rejects NaN / inf in X; the kernels count them while loading the candidates
static int check_nonfinite(b200bo_gp* g0) {
    unsigned long long c[2] = {0, 0};
    CU(cudaMemcpy(c, g0->clamp.p, sizeof(c), cudaMemcpyDeviceToHost));
    if (c[1] != 0) return set_err(B200BO_ERR_ARG, "Input X contains NaN or infinity.");
    return B200BO_OK;
}

static int run_host_chunked(const b200bo_acq* spec, const double* Xc, int64_t m, int k, SelRecord* sel_host) {
    b200bo_gp* g0 = spec->gps[0];
    int rc;
    if ((rc = ensure_copy_stream(g0))) return rc;
    const int d = g0->d;
    const long long chunk = kChunkTilesPerSm * PBN * g0->sm_count;
    if ((rc = g0->xc.reserve(sizeof(double) * (size_t)2 * chunk * d))) return rc;
    if ((rc = g0->sel.reserve(sizeof(SelRecord) * (B200BO_MAX_TOPK + 1)))) return rc;
    double* buf[2] = {g0->xc.as<double>(), g0->xc.as<double>() + (size_t)chunk * d};
    int i = 0;
    for (long long c0 = 0; c0 < m; c0 += chunk, ++i) {
        const long long mc = (m - c0) < chunk ? (m - c0) : chunk;
        const int b = i & 1;
        if (i >= 2) CU(cudaStreamWaitEvent(g0->copy_stream, g0->chunk_done[b], 0));  // buffer b consumed
        CU(cudaMemcpyAsync(buf[b], Xc + (size_t)c0 * d, sizeof(double) * (size_t)mc * d, cudaMemcpyHostToDevice,
                           g0->copy_stream));
        CU(cudaEventRecord(g0->chunk_up[b], g0->copy_stream));
        CU(cudaStreamWaitEvent(g0->exec_stream, g0->chunk_up[b], 0));
        CandSrc src;
        src.d_Xc = buf[b];
        SelMode sm;
        sm.resume = i > 0;
        sm.finish = (c0 + chunk >= m);
        sm.m_call = m;
        if ((rc = eval_core(spec, src, mc, nullptr, nullptr, nullptr, k, g0->sel.p, c0, g0->exec_stream, sm)))
            return rc;
        CU(cudaEventRecord(g0->chunk_done[b], g0->exec_stream));
    }
    CU(cudaStreamSynchronize(g0->exec_stream));
    CU(cudaMemcpy(sel_host, g0->sel.p, sizeof(SelRecord) * (k + 1), cudaMemcpyDeviceToHost));
    return check_nonfinite(g0);
}

static int run_host(const b200bo_acq* spec, const double* Xc, int64_t m, double* acq_neg, double* mu,
                    double* sd, int k, SelRecord* sel_host, int64_t* n_clamped, int64_t index_base = 0) {
    int rc;
    if ((rc = check_spec(spec))) return rc;
    if (m < 0 || (m > 0 && !Xc)) return set_err(B200BO_ERR_ARG, "bad candidates");
    b200bo_gp* g0 = spec->gps[0];
    CU(cudaSetDevice(g0->device));
    {
        int np_max = 0;
        for (int g = 0; g < spec->n_gps; ++g) np_max = spec->gps[g]->np > np_max ? spec->gps[g]->np : np_max;
        const long long chunk = kChunkTilesPerSm * PBN * g0->sm_count;
        const char* e = getenv("B200BO_CHUNKED");
        const bool allow = !(e && e[0] == '0');
        if (allow && k > 0 && sel_host && !acq_neg && !mu && !sd && !n_clamped && index_base == 0 && m >= 2 * chunk &&
            !use_small_path(m, np_max, spec->n_gps, g0->sm_count, spec->path))
            return run_host_chunked(spec, Xc, m, k, sel_host);
    }
    const size_t mm = (size_t)(m > 0 ? m : 1);
    if ((rc = g0->xc.reserve(sizeof(double) * mm * g0->d))) return rc;
    if (acq_neg && (rc = g0->out_acq.reserve(sizeof(double) * mm))) return rc;
    if (mu && (rc = g0->out_mu.reserve(sizeof(double) * mm))) return rc;
    if (sd && (rc = g0->out_sd.reserve(sizeof(double) * mm))) return rc;
    if ((rc = g0->sel.reserve(sizeof(SelRecord) * (B200BO_MAX_TOPK + 1)))) return rc;
    if (m > 0) CU(cudaMemcpy(g0->xc.p, Xc, sizeof(double) * (size_t)m * g0->d, cudaMemcpyHostToDevice));
    CandSrc src;
    src.d_Xc = g0->xc.as<double>();
    if ((rc = eval_core(spec, src, m, acq_neg ? g0->out_acq.as<double>() : nullptr,
                        mu ? g0->out_mu.as<double>() : nullptr, sd ? g0->out_sd.as<double>() : nullptr, k,
                        g0->sel.p, index_base, nullptr)))
        return rc;
    CU(cudaDeviceSynchronize());
    if (m > 0) {
        if (acq_neg) CU(cudaMemcpy(acq_neg, g0->out_acq.p, sizeof(double) * m, cudaMemcpyDeviceToHost));
        if (mu) CU(cudaMemcpy(mu, g0->out_mu.p, sizeof(double) * m, cudaMemcpyDeviceToHost));
        if (sd) CU(cudaMemcpy(sd, g0->out_sd.p, sizeof(double) * m, cudaMemcpyDeviceToHost));
    }
    if (k > 0 && sel_host)
        CU(cudaMemcpy(sel_host, g0->sel.p, sizeof(SelRecord) * (k + 1), cudaMemcpyDeviceToHost));
    if (n_clamped) {
        unsigned long long c = 0;
        CU(cudaMemcpy(&c, g0->clamp.p, sizeof(c), cudaMemcpyDeviceToHost));
        *n_clamped = (int64_t)c;
    }
    return m > 0 ? check_nonfinite(g0) : B200BO_OK;
}

extern "C" int b200bo_gp_predict(b200bo_gp* gp, const double* Xc, int64_t m, double* mu, double* sd,
                                 int64_t* n_clamped) {
    if (!gp || !mu) return set_err(B200BO_ERR_ARG, "NULL argument");
    b200bo_acq spec;
    memset(&spec, 0, sizeof(spec));
    spec.kind = B200BO_ACQ_NONE;
    spec.n_gps = 1;
    spec.gps[0] = gp;
    return run_host(&spec, Xc, m, nullptr, mu, sd, 0, nullptr, n_clamped);
}

extern "C" int b200bo_gp_predict_cov(b200bo_gp* gp, const double* Xc, int64_t m, double* mu, double* cov) {
    if (!gp || !Xc || !mu || !cov) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!gp->fitted) return set_err(B200BO_ERR_STATE, "GP handle is not fitted");
    if (m <= 0 || m > 16384) return set_err(B200BO_ERR_ARG, "return_cov supports 1 <= m <= 16384 (m=%lld)", (long long)m);
    CU(cudaSetDevice(gp->device));
    StreamScope scope(nullptr);  // legacy default stream
    const int n = (int)gp->n, np = gp->np, d = gp->d, mi = (int)m, mp = round_up(m, 128);
    int rc;
    if ((rc = gp->cov_xc.reserve(sizeof(double) * (size_t)mp * d))) return rc;
    if ((rc = gp->cov_kst.reserve(sizeof(double) * (size_t)np * mp))) return rc;
    if ((rc = gp->cov_v.reserve(sizeof(double) * (size_t)np * mp))) return rc;
    if ((rc = gp->cov_c.reserve(sizeof(double) * (size_t)mp * mp))) return rc;
    if ((rc = gp->cov_out.reserve(sizeof(double) * (size_t)mi * mi))) return rc;
    if ((rc = gp->cov_mu.reserve(sizeof(double) * (size_t)mp))) return rc;
    if ((rc = gp->xc.reserve(sizeof(double) * (size_t)mi * d))) return rc;
    CU(cudaMemcpy(gp->xc.p, Xc, sizeof(double) * (size_t)mi * d, cudaMemcpyHostToDevice));
    const int* xf = gp->xform.empty() ? nullptr : gp->xf.as<int>();
    {
        const long long tot = (long long)mp * d;
        scale_xc_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(gp->xc.as<double>(), gp->ls.as<double>(), xf,
                                                                gp->cov_xc.as<double>(), mi, mp, d);
        dim3 blk(32, 8), grd((mp + 31) / 32, (np + 7) / 8);
        kcross_kernel<<<grd, blk>>>(gp->Xs.as<double>(), gp->cov_xc.as<double>(), gp->cov_kst.as<double>(), n, np,
                                    mi, mp, d, gp->family, gp->nu, gp->constv);
        cross_mean_kernel<<<(mi + 127) / 128, 128>>>(gp->cov_kst.as<double>(), gp->alphav.as<double>(),
                                                     gp->cov_mu.as<double>(), np, mi, mp, gp->y_mean, gp->y_std);
        LAUNCHED();
        LAUNCHED();
        LAUNCHED();
    }
    // V = L^-1 K*^T  (np x mp) ; VtV = V^T V (mp x mp)
    if ((rc = gemm<false, false>(np, mp, np, 1.0, gp->W.as<double>(), np, 0, gp->cov_kst.as<double>(), mp, 0, 0.0,
                                 gp->cov_v.as<double>(), mp, 0, 1, 0, 1)))
        return rc;
    if ((rc = gemm<true, false>(mp, mp, np, 1.0, gp->cov_v.as<double>(), mp, 0, gp->cov_v.as<double>(), mp, 0, 0.0,
                                gp->cov_c.as<double>(), mp, 0, 1, 0, 0)))
        return rc;
    {
        dim3 blk(32, 8), grd((mi + 31) / 32, (mi + 7) / 8);
        cov_finish_kernel<<<grd, blk>>>(gp->cov_xc.as<double>(), gp->cov_c.as<double>(), mp, gp->cov_out.as<double>(),
                                        mi, d, gp->family, gp->nu, gp->constv, gp->y_std, gp->noise);
        LAUNCHED();
    }
    CU(cudaGetLastError());
    CU(cudaMemcpy(mu, gp->cov_mu.p, sizeof(double) * (size_t)mi, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(cov, gp->cov_out.p, sizeof(double) * (size_t)mi * mi, cudaMemcpyDeviceToHost));
    return B200BO_OK;
}

extern "C" int b200bo_acq_eval(const b200bo_acq* spec, const double* Xc, int64_t m, double* acq_neg) {
    if (!acq_neg && m > 0) return set_err(B200BO_ERR_ARG, "acq_neg is NULL");
    if (spec && spec->kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    return run_host(spec, Xc, m, acq_neg, nullptr, nullptr, 0, nullptr, nullptr);
}

static void unpack_records(const SelRecord* sel, int k, double* best_val, int64_t* best_idx, double* topk_val,
                           int64_t* topk_idx) {
    if (best_val) *best_val = sel[0].value;
    if (best_idx) *best_idx = sel[0].index;
    for (int i = 0; i < k; ++i) {
        if (topk_val) topk_val[i] = sel[1 + i].value;
        if (topk_idx) topk_idx[i] = sel[1 + i].index;
    }
}

extern "C" int b200bo_acq_argmin_topk(const b200bo_acq* spec, const double* Xc, int64_t m, int k,
                                      double* best_val, int64_t* best_idx, double* topk_val,
                                      int64_t* topk_idx, double* acq_neg) {
    if (k < 0 || k > B200BO_MAX_TOPK) return set_err(B200BO_ERR_ARG, "k=%d out of range", k);
    if (m <= 0) return set_err(B200BO_ERR_ARG, "m must be > 0");
    if (spec && spec->kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    SelRecord sel[B200BO_MAX_TOPK + 1];
    // k = 0 still needs the argmin record: run the selection with one round
    int rc = run_host(spec, Xc, m, acq_neg, nullptr, nullptr, k > 0 ? k : 1, sel, nullptr);
    if (rc) return rc;
    unpack_records(sel, k, best_val, best_idx, topk_val, topk_idx);
    return B200BO_OK;
}

// ---------------------------------------------------------------------------------------
// throughput mode (device Philox candidates)
// ---------------------------------------------------------------------------------------
// coordinates of the records' rows, regenerated on the device of g0 into host memory (k+1 rows)
static int philox_rows_of_records(b200bo_gp* g0, uint64_t seed, const SelRecord* d_rec, int nrec, int d,
                                  double* rows_host, cudaStream_t stream) {
    int rc;
    if ((rc = g0->prow.reserve(sizeof(double) * (size_t)(B200BO_MAX_TOPK + 1) * B200BO_MAX_DIM))) return rc;
    philox_rows_kernel<<<nrec, 64, 0, stream>>>(seed, g0->pbounds.as<double>(), d, d_rec, nrec, g0->prow.as<double>());
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(rows_host, g0->prow.p, sizeof(double) * (size_t)nrec * d, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    return B200BO_OK;
}

extern "C" int b200bo_acq_argmin_topk_philox(const b200bo_acq* spec, uint64_t seed, const double* lo,
                                             const double* hi, int64_t m, int64_t index_base, int k,
                                             double* best_val, int64_t* best_idx, double* best_x, double* topk_val,
                                             int64_t* topk_idx, double* topk_x) {
    if (k < 0 || k > B200BO_MAX_TOPK) return set_err(B200BO_ERR_ARG, "k=%d out of range", k);
    if (m <= 0) return set_err(B200BO_ERR_ARG, "m must be > 0");
    int rc;
    if ((rc = check_spec(spec))) return rc;
    if (spec->kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    b200bo_gp* g0 = spec->gps[0];
    CU(cudaSetDevice(g0->device));
    if ((rc = g0->sel.reserve(sizeof(SelRecord) * (B200BO_MAX_TOPK + 1)))) return rc;
    const int kk = k > 0 ? k : 1;
    if ((rc = b200bo_acq_select_philox_dev(spec, seed, lo, hi, m, index_base, kk, g0->sel.p, nullptr))) return rc;
    SelRecord sel[B200BO_MAX_TOPK + 1];
    CU(cudaMemcpy(sel, g0->sel.p, sizeof(SelRecord) * (kk + 1), cudaMemcpyDeviceToHost));
    unpack_records(sel, k, best_val, best_idx, topk_val, topk_idx);
    if (best_x || (topk_x && k > 0)) {
        std::vector<double> rows((size_t)(kk + 1) * g0->d);
        if ((rc = philox_rows_of_records(g0, seed, g0->sel.as<SelRecord>(), kk + 1, g0->d, rows.data(), nullptr)))
            return rc;
        if (best_x) memcpy(best_x, rows.data(), sizeof(double) * g0->d);
        if (topk_x && k > 0) memcpy(topk_x, rows.data() + g0->d, sizeof(double) * (size_t)k * g0->d);
    }
    return B200BO_OK;
}

extern "C" int b200bo_philox_rows(int device, uint64_t seed, const double* lo, const double* hi, int d,
                                  const int64_t* idx, int64_t n_idx, double* out) {
    if (!lo || !hi || !idx || !out) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (d <= 0 || d > B200BO_MAX_DIM || n_idx < 0) return set_err(B200BO_ERR_ARG, "bad shape");
    if (n_idx == 0) return B200BO_OK;
    CU(cudaSetDevice(device));
    std::vector<SelRecord> rec((size_t)n_idx);
    std::vector<double> pb(2 * d);
    for (int j = 0; j < d; ++j) {
        pb[j] = lo[j];
        pb[d + j] = hi[j] - lo[j];
    }
    for (int64_t i = 0; i < n_idx; ++i) {
        rec[i].value = 0.0;
        rec[i].index = idx[i];
    }
    SelRecord* d_rec = nullptr;
    double *d_pb = nullptr, *d_out = nullptr;
    CU(cudaMalloc(&d_rec, sizeof(SelRecord) * n_idx));
    CU(cudaMalloc(&d_pb, sizeof(double) * 2 * d));
    CU(cudaMalloc(&d_out, sizeof(double) * n_idx * d));
    CU(cudaMemcpy(d_rec, rec.data(), sizeof(SelRecord) * n_idx, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_pb, pb.data(), sizeof(double) * 2 * d, cudaMemcpyHostToDevice));
    philox_rows_kernel<<<(unsigned)n_idx, 64>>>(seed, d_pb, d, d_rec, (int)n_idx, d_out);
    LAUNCHED();
    cudaError_t e = cudaMemcpy(out, d_out, sizeof(double) * n_idx * d, cudaMemcpyDeviceToHost);
    cudaFree(d_rec);
    cudaFree(d_pb);
    cudaFree(d_out);
    if (e != cudaSuccess) return set_err(B200BO_ERR_CUDA, "philox_rows: %s", cudaGetErrorString(e));
    return B200BO_OK;
}

// ---------------------------------------------------------------------------------------
// multi-GPU (one process, G devices of one box): SURVEY.md 8e
// ---------------------------------------------------------------------------------------
extern "C" int b200bo_gp_replicate(const b200bo_gp* src, int device, b200bo_gp** out) {
    if (!src || !out) return set_err(B200BO_ERR_ARG, "NULL argument");
    if (!src->fitted) return set_err(B200BO_ERR_STATE, "source GP handle is not fitted");
    b200bo_gp* dst = nullptr;
    int rc;
    if ((rc = b200bo_gp_create(&dst, device))) return rc;
    NvtxRange nvtx_range("b200bo:replicate");
    dst->n = src->n;
    dst->np = src->np;
    dst->d = src->d;
    dst->family = src->family;
    dst->nu = src->nu;
    dst->constv = src->constv;
    dst->jitter = src->jitter;
    dst->noise = src->noise;
    dst->y_mean = src->y_mean;
    dst->y_std = src->y_std;
    dst->normalize = src->normalize;
    dst->xform = src->xform;
    dst->precision = src->precision;
    dst->replica = true;
    const size_t np = src->np, d = src->d;
    struct Item {
        DevBuf* to;
        const DevBuf* from;
        size_t bytes;
    } items[] = {
        {&dst->Xs, &src->Xs, sizeof(double) * np * d},        {&dst->WT, &src->WT, sizeof(double) * np * np},
        {&dst->W, &src->W, sizeof(double) * np * np},          {&dst->alphav, &src->alphav, sizeof(double) * np},
        {&dst->ls, &src->ls, sizeof(double) * B200BO_MAX_DIM}, {&dst->xf, &src->xf, sizeof(int) * B200BO_MAX_DIM},
    };
    for (const Item& it : items) {
        if ((rc = it.to->reserve(it.bytes))) {
            b200bo_gp_destroy(dst);
            return rc;
        }
        cudaError_t e = cudaMemcpyPeer(it.to->p, device, it.from->p, src->device, it.bytes);
        if (e != cudaSuccess) {
            b200bo_gp_destroy(dst);
            return set_err(B200BO_ERR_CUDA, "cudaMemcpyPeer %d -> %d failed: %s", src->device, device,
                           cudaGetErrorString(e));
        }
    }
    CU(cudaSetDevice(src->device));
    CU(cudaDeviceSynchronize());
    CU(cudaSetDevice(device));
    CU(cudaDeviceSynchronize());
    dst->fitted = true;
    *out = dst;
    return B200BO_OK;
}

// NCCL is reached through dlopen so that the library has no link-time dependency on it: inside a Python
// process that already imported torch this binds to torch's bundled libnccl.so.2, otherwise to the system one.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static std::mutex g_multi_mu;

static int load_nccl() {
    if (g_nccl.handle) return B200BO_OK;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return set_err(B200BO_ERR_CUDA, "cannot load libnccl.so.2: %s", dlerror());
    g_nccl.CommInitAll = (decltype(g_nccl.CommInitAll))dlsym(h, "ncclCommInitAll");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(h, "ncclAllGather");
    g_nccl.GroupStart = (decltype(g_nccl.GroupStart))dlsym(h, "ncclGroupStart");
    g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))dlsym(h, "ncclGroupEnd");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
    if (!g_nccl.CommInitAll || !g_nccl.AllGather || !g_nccl.GroupStart || !g_nccl.GroupEnd || !g_nccl.GetErrorString)
        return set_err(B200BO_ERR_CUDA, "libnccl.so.2 lacks a required symbol");
    g_nccl.handle = h;
    return B200BO_OK;
}

#define NC(call)                                                                                    \
    do {                                                                                            \
        ncclResult_t r__ = (call);                                                                  \
        if (r__ != ncclSuccess)                                                                     \
            return set_err(B200BO_ERR_CUDA, "%s failed: %s", #call, g_nccl.GetErrorString(r__));    \
    } while (0)

constexpr int kMaxDev = 16;
struct MultiCtx {
    int n = 0;
    int dev[kMaxDev];
    ncclComm_t comm[kMaxDev];
    cudaStream_t stream[kMaxDev];
    SelRecord* sel[kMaxDev];     // (MAX_TOPK+1) local records on device g
    SelRecord* gather[kMaxDev];  // n * (MAX_TOPK+1) records on device g
    SelRecord* merged = nullptr; // (MAX_TOPK+1) on device 0
};
static std::map<std::vector<int>, MultiCtx*> g_multi;

// communicators + exchange buffers for a device list (created on first use, kept for the process lifetime)
static int multi_ctx(const b200bo_acq* specs, int n_dev, MultiCtx** out) {
    if (!specs || n_dev < 1 || n_dev > kMaxDev) return set_err(B200BO_ERR_ARG, "n_dev=%d out of range [1,%d]", n_dev, kMaxDev);
    std::vector<int> devs;
    int rc;
    for (int g = 0; g < n_dev; ++g) {
        if ((rc = check_spec(&specs[g]))) return rc;
        if (specs[g].n_gps != specs[0].n_gps || specs[g].kind != specs[0].kind)
            return set_err(B200BO_ERR_ARG, "specs[%d] describes a different acquisition", g);
        const int dv = specs[g].gps[0]->device;
        for (int q : devs)
            if (q == dv) return set_err(B200BO_ERR_ARG, "device %d appears twice", dv);
        devs.push_back(dv);
    }
    auto it = g_multi.find(devs);
    if (it != g_multi.end()) {
        *out = it->second;
        return B200BO_OK;
    }
    if ((rc = load_nccl())) return rc;
    MultiCtx* c = new MultiCtx();
    c->n = n_dev;
    for (int g = 0; g < n_dev; ++g) c->dev[g] = devs[g];
    NC(g_nccl.CommInitAll(c->comm, n_dev, c->dev));
    for (int g = 0; g < n_dev; ++g) {
        CU(cudaSetDevice(c->dev[g]));
        CU(cudaStreamCreateWithFlags(&c->stream[g], cudaStreamNonBlocking));
        CU(cudaMalloc(&c->sel[g], sizeof(SelRecord) * (B200BO_MAX_TOPK + 1)));
        CU(cudaMalloc(&c->gather[g], sizeof(SelRecord) * (B200BO_MAX_TOPK + 1) * n_dev));
    }
    CU(cudaSetDevice(c->dev[0]));
    CU(cudaMalloc(&c->merged, sizeof(SelRecord) * (B200BO_MAX_TOPK + 1)));
    g_multi[devs] = c;
    *out = c;
    return B200BO_OK;
}

static void shard_range(int64_t m, int g, int n, int64_t* s, int64_t* e) {
    const int64_t base = m / n, rem = m % n;
    *s = g * base + (g < rem ? g : rem);
    *e = *s + base + (g < rem ? 1 : 0);
}

// run fn(g) on one host thread per device; the first failing rc and its message come back to the caller
template <typename F>
static int per_device(int n_dev, F fn) {
    std::vector<int> rcs(n_dev, 0);
    std::vector<std::string> msgs(n_dev);
    std::vector<std::thread> th;
    for (int g = 0; g < n_dev; ++g)
        th.emplace_back([&, g]() {
            rcs[g] = fn(g);
            if (rcs[g]) msgs[g] = g_err;
        });
    for (auto& t : th) t.join();
    for (int g = 0; g < n_dev; ++g)
        if (rcs[g]) return set_err(rcs[g], "device slot %d: %s", g, msgs[g].c_str());
    return B200BO_OK;
}

// the ONE exchange step + merge; the (k+1) merged records land in sel_host
static int multi_exchange(MultiCtx* c, int k, SelRecord* sel_host) {
    NvtxRange nvtx_range("b200bo:exchange");
    const size_t bytes = sizeof(SelRecord) * (k + 1);
    NC(g_nccl.GroupStart());
    for (int g = 0; g < c->n; ++g)
        NC(g_nccl.AllGather(c->sel[g], c->gather[g], bytes, ncclInt8, c->comm[g], c->stream[g]));
    NC(g_nccl.GroupEnd());
    CU(cudaSetDevice(c->dev[0]));
    merge_records_kernel<<<1, 32, 0, c->stream[0]>>>(c->gather[0], c->n, k, c->merged);
    LAUNCHED();
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(sel_host, c->merged, bytes, cudaMemcpyDeviceToHost, c->stream[0]));
    for (int g = 0; g < c->n; ++g) {
        CU(cudaSetDevice(c->dev[g]));
        CU(cudaStreamSynchronize(c->stream[g]));
    }
    return B200BO_OK;
}

extern "C" int b200bo_multi_gpu_acq_argmin_topk(const b200bo_acq* specs, int n_dev, const double* Xc, int64_t m,
                                                int k, double* best_val, int64_t* best_idx, double* topk_val,
                                                int64_t* topk_idx) {
    if (k < 0 || k > B200BO_MAX_TOPK) return set_err(B200BO_ERR_ARG, "k=%d out of range", k);
    if (m <= 0 || !Xc) return set_err(B200BO_ERR_ARG, "bad candidates");
    std::lock_guard<std::mutex> lock(g_multi_mu);
    MultiCtx* c = nullptr;
    int rc;
    if ((rc = multi_ctx(specs, n_dev, &c))) return rc;
    if (specs[0].kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    const int kk = k > 0 ? k : 1;
    const int d = specs[0].gps[0]->d;
    rc = per_device(n_dev, [&](int g) -> int {
        int64_t s, e;
        shard_range(m, g, n_dev, &s, &e);
        b200bo_gp* g0 = specs[g].gps[0];
        CU(cudaSetDevice(g0->device));
        int r;
        const int64_t mg = e - s;
        if ((r = g0->xc.reserve(sizeof(double) * (size_t)(mg > 0 ? mg : 1) * d))) return r;
        if (mg > 0)
            CU(cudaMemcpyAsync(g0->xc.p, Xc + (size_t)s * d, sizeof(double) * (size_t)mg * d, cudaMemcpyHostToDevice,
                               c->stream[g]));
        CandSrc src;
        src.d_Xc = g0->xc.as<double>();
        return eval_core(&specs[g], src, mg, nullptr, nullptr, nullptr, kk, c->sel[g], s, c->stream[g]);
    });
    if (rc) return rc;
    SelRecord sel[B200BO_MAX_TOPK + 1];
    if ((rc = multi_exchange(c, kk, sel))) return rc;
    for (int g = 0; g < n_dev; ++g) {
        CU(cudaSetDevice(specs[g].gps[0]->device));
        if (specs[g].gps[0]->clamp.p && (rc = check_nonfinite(specs[g].gps[0]))) return rc;
    }
    unpack_records(sel, k, best_val, best_idx, topk_val, topk_idx);
    return B200BO_OK;
}

extern "C" int b200bo_multi_gpu_acq_argmin_topk_philox(const b200bo_acq* specs, int n_dev, uint64_t seed,
                                                       const double* lo, const double* hi, int64_t m,
                                                       int64_t index_base, int k, double* best_val,
                                                       int64_t* best_idx, double* best_x, double* topk_val,
                                                       int64_t* topk_idx, double* topk_x) {
    if (k < 0 || k > B200BO_MAX_TOPK) return set_err(B200BO_ERR_ARG, "k=%d out of range", k);
    if (m <= 0) return set_err(B200BO_ERR_ARG, "m must be > 0");
    std::lock_guard<std::mutex> lock(g_multi_mu);
    MultiCtx* c = nullptr;
    int rc;
    if ((rc = multi_ctx(specs, n_dev, &c))) return rc;
    if (specs[0].kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    const int kk = k > 0 ? k : 1;
    rc = per_device(n_dev, [&](int g) -> int {
        int64_t s, e;
        shard_range(m, g, n_dev, &s, &e);
        CU(cudaSetDevice(specs[g].gps[0]->device));
        if (e == s) {
            CU(cudaMemsetAsync(c->sel[g], 0xFF, sizeof(SelRecord) * (kk + 1), c->stream[g]));
            return B200BO_OK;
        }
        CandSrc src;
        src.philox = true;
        src.seed = seed;
        src.lo = lo;
        src.hi = hi;
        return eval_core(&specs[g], src, e - s, nullptr, nullptr, nullptr, kk, c->sel[g], index_base + s, c->stream[g]);
    });
    if (rc) return rc;
    SelRecord sel[B200BO_MAX_TOPK + 1];
    if ((rc = multi_exchange(c, kk, sel))) return rc;
    unpack_records(sel, k, best_val, best_idx, topk_val, topk_idx);
    if (best_x || (topk_x && k > 0)) {
        b200bo_gp* g0 = specs[0].gps[0];
        CU(cudaSetDevice(g0->device));
        std::vector<double> rows((size_t)(kk + 1) * g0->d);
        if ((rc = philox_rows_of_records(g0, seed, c->merged, kk + 1, g0->d, rows.data(), c->stream[0]))) return rc;
        if (best_x) memcpy(best_x, rows.data(), sizeof(double) * g0->d);
        if (topk_x && k > 0) memcpy(topk_x, rows.data() + g0->d, sizeof(double) * (size_t)k * g0->d);
    }
    return B200BO_OK;
}

extern "C" int b200bo_multi_gpu_acq_eval(const b200bo_acq* specs, int n_dev, const double* Xc, int64_t m,
                                         const int64_t* offsets, double* acq_neg) {
    if (m < 0 || (m > 0 && (!Xc || !acq_neg))) return set_err(B200BO_ERR_ARG, "bad candidates");
    if (!specs || n_dev < 1 || n_dev > kMaxDev) return set_err(B200BO_ERR_ARG, "n_dev=%d out of range", n_dev);
    int rc;
    for (int g = 0; g < n_dev; ++g) {
        if ((rc = check_spec(&specs[g]))) return rc;
        if (specs[g].kind == B200BO_ACQ_NONE) return set_err(B200BO_ERR_ARG, "kind NONE has no acquisition");
    }
    if (offsets) {
        if (offsets[0] != 0 || offsets[n_dev] != m) return set_err(B200BO_ERR_ARG, "offsets must span [0, m]");
        for (int g = 0; g < n_dev; ++g)
            if (offsets[g + 1] < offsets[g]) return set_err(B200BO_ERR_ARG, "offsets must be non-decreasing");
    }
    const int d = specs[0].gps[0]->d;
    return per_device(n_dev, [&](int g) -> int {
        int64_t s, e;
        if (offsets) {
            s = offsets[g];
            e = offsets[g + 1];
        } else {
            shard_range(m, g, n_dev, &s, &e);
        }
        if (e == s) return B200BO_OK;
        return run_host(&specs[g], Xc + (size_t)s * d, e - s, acq_neg + s, nullptr, nullptr, 0, nullptr, nullptr);
    });
}
