// C-ABI glue of libbgmm: argument checks, error reporting, layout queries, data preparation, dispatch.
#include "bgmm_common.cuh"
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

namespace bgmm {

static thread_local char g_err[512] = "";
thread_local int64_t g_launches = 0;
static double g_robust_threshold = 2.0e4;

double robust_threshold() { return g_robust_threshold; }

bool pdl_enabled() {
    static const int on = [] { const char* e = getenv("BGMM_PDL"); return (e == nullptr || atoi(e) != 0) ? 1 : 0; }();
    return on != 0;
}

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return BGMM_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return BGMM_ECUDA;
}

int launch_pass_simple(const PassArgs& a, int K, int D, int dtype, int direct, cudaStream_t stream);
int simple_grid_cap(int K, int D);
bool dmma_supported(int K, int D, int dtype);
int launch_pass_dmma(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream);
int64_t dmma_workspace_doubles(int K, int D);
bool f32_supported(int K, int D, int dtype);
int launch_pass_f32(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream);
int64_t f32_workspace_doubles(int K, int D);
bool large_supported(int K, int D, int dtype);
int launch_pass_large(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream);
int64_t large_workspace_doubles(int K, int D);
bool tf32_pass_supported(int K, int D, int dtype);
int launch_pass_tf32(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream);
int64_t tf32_workspace_doubles(int K, int D, int64_t n);
int launch_pass_batched(const void* x, int64_t n, int K, int D, const BatchDesc& bd, double* sup, double* workspace,
                        double* r_scratch, cudaStream_t stream);

// ---- data preparation ----
constexpr int PREP_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(PREP_THREADS) colsum_partial_kernel(const T* __restrict__ x, int64_t total,
                                                                     int64_t stride, double* __restrict__ ws) {
    // `stride` is a multiple of D, so a thread always visits the same column: acc is a per-column partial.
    const int64_t t = (int64_t)blockIdx.x * PREP_THREADS + threadIdx.x;
    if (t >= stride) return;
    double acc = 0.0;
    for (int64_t e = t; e < total; e += stride) acc += (double)x[e];
    ws[t] = acc;
}

__global__ void colsum_final_kernel(const double* __restrict__ ws, int64_t stride, int D, double* __restrict__ out) {
    // one warp per column, fixed order -> deterministic
    const int d = blockIdx.x, lane = threadIdx.x;
    double acc = 0.0;
    for (int64_t t = d + (int64_t)lane * D; t < stride; t += (int64_t)32 * D) acc += ws[t];
    acc = warp_sum(acc);
    if (lane == 0) out[d] = acc;
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(PREP_THREADS) center_kernel(const TI* __restrict__ x, TO* __restrict__ y, int64_t total,
                                                             int D, const double* __restrict__ c) {
    const int64_t stride = (int64_t)gridDim.x * PREP_THREADS;
    for (int64_t e = (int64_t)blockIdx.x * PREP_THREADS + threadIdx.x; e < total; e += stride)
        y[e] = (TO)((double)x[e] - c[e % D]);
}

static int64_t colsum_stride(int D) {
    int64_t threads = (int64_t)148 * 8 * PREP_THREADS;
    if (threads < D) threads = D;
    return threads / D * D;
}

}  // namespace bgmm

using namespace bgmm;

extern "C" int bgmm_abi_version(void) { return BGMM_ABI_VERSION; }
extern "C" double bgmm_robust_threshold(void) { return g_robust_threshold; }
extern "C" double bgmm_set_robust_threshold(double t) {
    const double old = g_robust_threshold;
    g_robust_threshold = t;
    return old;
}
extern "C" const char* bgmm_last_error(void) { return g_err; }
extern "C" int64_t bgmm_launch_count(void) { return g_launches; }

extern "C" int bgmm_layout(int K, int D, int hist_len, int64_t* off, int64_t* poff) {
    if (K <= 0 || D <= 0 || hist_len < 1 || off == nullptr || poff == nullptr) {
        set_error("bgmm_layout: bad argument");
        return BGMM_EINVAL;
    }
    const Layout L = make_layout(K, D, hist_len);
    off[BGMM_OFF_CENTER] = L.center; off[BGMM_OFF_ALPHA0] = L.alpha0; off[BGMM_OFF_KAPPA0] = L.kappa0;
    off[BGMM_OFF_NU0] = L.nu0; off[BGMM_OFF_M0] = L.m0; off[BGMM_OFF_W0INV] = L.w0inv; off[BGMM_OFF_LNB0] = L.lnb0;
    off[BGMM_OFF_LNC0] = L.lnc0; off[BGMM_OFF_PARAMS0] = L.params[0]; off[BGMM_OFF_PARAMS1] = L.params[1];
    off[BGMM_OFF_STATS] = L.stats; off[BGMM_OFF_NS] = L.ns; off[BGMM_OFF_XBAR] = L.xbar; off[BGMM_OFF_SMATS] = L.smats;
    off[BGMM_OFF_VLK] = L.vlk; off[BGMM_OFF_VLTERMS] = L.vlterms; off[BGMM_OFF_VLHIST] = L.vlhist;
    off[BGMM_OFF_CTRL] = L.ctrl; off[BGMM_OFF_TOTAL] = L.total; off[BGMM_OFF_STATS_LEN] = L.stats_len;
    off[BGMM_OFF_PARAMS_LEN] = L.params_len; off[BGMM_OFF_PITCH] = L.pitch; off[BGMM_OFF_SHIFT] = L.shift;
    poff[BGMM_P_ALPHA] = L.p_alpha; poff[BGMM_P_KAPPA] = L.p_kappa; poff[BGMM_P_NU] = L.p_nu; poff[BGMM_P_M] = L.p_m;
    poff[BGMM_P_WINV] = L.p_winv; poff[BGMM_P_W] = L.p_w; poff[BGMM_P_ELNPI] = L.p_elnpi;
    poff[BGMM_P_ELNDET] = L.p_elndet; poff[BGMM_P_LNB] = L.p_lnb; poff[BGMM_P_COEF] = L.p_coef;
    poff[BGMM_P_ACST] = L.p_acst; poff[BGMM_P_LINV] = L.p_linv;
    return BGMM_OK;
}

extern "C" int64_t bgmm_workspace_doubles(int K, int D) {
    if (K <= 0 || D <= 0) return 0;
    const int64_t len = (int64_t)K * feat_pitch(D) + 8;
    int64_t w = (int64_t)simple_grid_cap(K, D) * len;
    const int64_t wd = dmma_workspace_doubles(K, D);
    if (wd > w) w = wd;
    const int64_t wf = f32_workspace_doubles(K, D);
    if (wf > w) w = wf;
    const int64_t wl = large_workspace_doubles(K, D);
    if (wl > w) w = wl;
    const int64_t wc = colsum_stride(D);
    if (wc > w) w = wc;
    return w;
}

extern "C" int bgmm_colsum(const void* x, int64_t n, int D, int dtype, double* out, double* ws, void* stream) {
    if (x == nullptr && n > 0) { set_error("bgmm_colsum: x is NULL"); return BGMM_EINVAL; }
    if (n < 0 || D <= 0 || out == nullptr || ws == nullptr || (dtype != BGMM_F64 && dtype != BGMM_F32)) {
        set_error("bgmm_colsum: bad argument (n=%lld D=%d dtype=%d)", (long long)n, D, dtype);
        return BGMM_EINVAL;
    }
    const int64_t stride = colsum_stride(D), total = n * D;
    const int grid = (int)((stride + PREP_THREADS - 1) / PREP_THREADS);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == BGMM_F64) launch(colsum_partial_kernel<double>, grid, PREP_THREADS, 0, s, (const double*)x, total, stride, ws);
    else launch(colsum_partial_kernel<float>, grid, PREP_THREADS, 0, s, (const float*)x, total, stride, ws);
    launch(colsum_final_kernel, D, 32, 0, s, ws, stride, D, out);
    return check_cuda(cudaGetLastError(), "bgmm_colsum launch");
}

extern "C" int bgmm_center(const void* x, int dtype_in, void* y, int dtype_out, int64_t n, int D, const double* c,
                           void* stream) {
    if (n < 0 || D <= 0 || c == nullptr || ((x == nullptr || y == nullptr) && n > 0)) {
        set_error("bgmm_center: bad argument");
        return BGMM_EINVAL;
    }
    if (n == 0) return BGMM_OK;
    const int64_t total = n * D;
    int64_t grid64 = (total + PREP_THREADS - 1) / PREP_THREADS;
    const int grid = (int)(grid64 < 148 * 16 ? grid64 : 148 * 16);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype_in == BGMM_F64 && dtype_out == BGMM_F64)
        launch(center_kernel<double, double>, grid, PREP_THREADS, 0, s, (const double*)x, (double*)y, total, D, c);
    else if (dtype_in == BGMM_F64 && dtype_out == BGMM_F32)
        launch(center_kernel<double, float>, grid, PREP_THREADS, 0, s, (const double*)x, (float*)y, total, D, c);
    else if (dtype_in == BGMM_F32 && dtype_out == BGMM_F32)
        launch(center_kernel<float, float>, grid, PREP_THREADS, 0, s, (const float*)x, (float*)y, total, D, c);
    else if (dtype_in == BGMM_F32 && dtype_out == BGMM_F64)
        launch(center_kernel<float, double>, grid, PREP_THREADS, 0, s, (const float*)x, (double*)y, total, D, c);
    else { set_error("bgmm_center: bad dtype"); return BGMM_EINVAL; }
    return check_cuda(cudaGetLastError(), "bgmm_center launch");
}

extern "C" int bgmm_batch_capacity(int K, int D) {
    if (K <= 0 || D <= 0 || !large_supported(K, D, BGMM_F64)) return 1;
    const int Kp = (K + 7) & ~7;
    int r = 64 / Kp;
    if (r > BGMM_MAX_BATCH) r = BGMM_MAX_BATCH;
    return r < 1 ? 1 : r;
}

extern "C" int bgmm_pass_batched(const void* x, int64_t n, int K, int D, int R, double* const* states, double* sup,
                                 double* workspace, double* r_scratch, void* stream) {
    if (K <= 0 || D <= 0 || n < 0 || R < 2 || R > BGMM_MAX_BATCH || states == nullptr || sup == nullptr ||
        workspace == nullptr || r_scratch == nullptr || (x == nullptr && n > 0)) {
        set_error("bgmm_pass_batched: bad argument (n=%lld K=%d D=%d R=%d)", (long long)n, K, D, R);
        return BGMM_EINVAL;
    }
    if (R > bgmm_batch_capacity(K, D)) {
        set_error("bgmm_pass_batched: R=%d exceeds the capacity %d of K=%d D=%d", R, bgmm_batch_capacity(K, D), K, D);
        return BGMM_ENOSUP;
    }
    BatchDesc bd;
    bd.R = R;
    for (int i = 0; i < BGMM_MAX_BATCH; ++i) bd.st[i] = i < R ? states[i] : nullptr;
    for (int i = 0; i < R; ++i)
        if (bd.st[i] == nullptr) { set_error("bgmm_pass_batched: member state %d is NULL", i); return BGMM_EINVAL; }
    cudaStream_t s = (cudaStream_t)stream;
    int rc = launch_pass_batched(x, n, K, D, bd, sup, workspace, r_scratch, s);
    if (rc) return rc;
    if (g_robust_threshold < INFINITY) {
        // conditioning guard, per member: returns at once unless that member's ctrl.robust is set
        for (int i = 0; i < R && rc == 0; ++i) {
            PassArgs a{x, n, bd.st[i], workspace, nullptr, nullptr, nullptr, nullptr, 0};
            rc = launch_pass_simple(a, K, D, BGMM_F64, 1, s);
        }
    }
    return rc;
}

extern "C" int64_t bgmm_tf32_workspace_doubles(int K, int D, int64_t n) {
    if (K <= 0 || D <= 0 || n < 0) return 0;
    return tf32_workspace_doubles(K, D, n);
}

extern "C" int bgmm_pass_supported(int K, int D, int dtype, int variant) {
    if (K <= 0 || D <= 0 || (dtype != BGMM_F64 && dtype != BGMM_F32)) return 0;
    if (variant == BGMM_PASS_DMMA) return dmma_supported(K, D, dtype) ? 1 : 0;
    if (variant == BGMM_PASS_F32) return f32_supported(K, D, dtype) ? 1 : 0;
    if (variant == BGMM_PASS_LARGE) return large_supported(K, D, dtype) ? 1 : 0;
    if (variant == BGMM_PASS_TF32) return tf32_pass_supported(K, D, dtype) ? 1 : 0;
    return variant == BGMM_PASS_SIMPLE || variant == BGMM_PASS_AUTO || variant == BGMM_PASS_DIRECT;
}

extern "C" int bgmm_pass_resolve(int K, int D, int dtype, int variant, int has_r_in) {
    if (has_r_in) return variant == BGMM_PASS_DIRECT ? BGMM_PASS_DIRECT : BGMM_PASS_SIMPLE;
    if (variant != BGMM_PASS_AUTO) return variant;
    if (dmma_supported(K, D, dtype)) return BGMM_PASS_DMMA;
    if (large_supported(K, D, dtype)) return BGMM_PASS_LARGE;
    if (f32_supported(K, D, dtype)) return BGMM_PASS_F32;
    if (tf32_pass_supported(K, D, dtype)) return BGMM_PASS_TF32;
    return BGMM_PASS_SIMPLE;
}

extern "C" int bgmm_pass(const void* x, int64_t n, int K, int D, int dtype, double* state, double* workspace,
                         double* r_out, double* lnrho_out, int32_t* argmax_out, const double* r_in, int variant,
                         int force, void* stream) {
    if (K <= 0 || D <= 0 || n < 0 || state == nullptr || workspace == nullptr || (x == nullptr && n > 0) ||
        (dtype != BGMM_F64 && dtype != BGMM_F32)) {
        set_error("bgmm_pass: bad argument (n=%lld K=%d D=%d dtype=%d)", (long long)n, K, D, dtype);
        return BGMM_EINVAL;
    }
    PassArgs a{x, n, state, workspace, r_out, lnrho_out, argmax_out, r_in, force & BGMM_FORCE};
    a.no_publish = (force & BGMM_FORCE_NO_PUBLISH) ? 1 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    variant = bgmm_pass_resolve(K, D, dtype, variant, r_in != nullptr);
    if (r_in != nullptr) {                                     // statistics of given responsibilities: no E-step; moments
        if (variant != BGMM_PASS_SIMPLE && variant != BGMM_PASS_DIRECT) {   // about the centre (SIMPLE) or state.SHIFT (DIRECT)
            set_error("bgmm_pass: variant %d does not take r_in", variant);
            return BGMM_ENOSUP;
        }
        a.ignore_robust = 1;
        return launch_pass_simple(a, K, D, dtype, variant == BGMM_PASS_DIRECT ? 1 : 0, s);
    }
    if (variant == BGMM_PASS_DIRECT) {                         // forced: whatever ctrl.robust says
        a.ignore_robust = 1;
        return launch_pass_simple(a, K, D, dtype, 1, s);
    }
    int rc;
    if (variant == BGMM_PASS_LARGE) {
        rc = launch_pass_large(a, K, D, dtype, s);
    } else if (variant == BGMM_PASS_F32) {
        if (!f32_supported(K, D, dtype)) {
            set_error("bgmm_pass: F32 variant does not support K=%d D=%d dtype=%d", K, D, dtype);
            return BGMM_ENOSUP;
        }
        rc = launch_pass_f32(a, K, D, dtype, s);
    } else if (variant == BGMM_PASS_DMMA) {
        if (!dmma_supported(K, D, dtype)) {
            set_error("bgmm_pass: DMMA variant does not support K=%d D=%d dtype=%d", K, D, dtype);
            return BGMM_ENOSUP;
        }
        rc = launch_pass_dmma(a, K, D, dtype, s);
    } else if (variant == BGMM_PASS_TF32) {
        a.crit_limit = 4096;
        rc = launch_pass_tf32(a, K, D, dtype, s);
    } else if (variant == BGMM_PASS_SIMPLE) {
        rc = launch_pass_simple(a, K, D, dtype, 0, s);
    } else {
        set_error("bgmm_pass: unknown variant %d", variant);
        return BGMM_EINVAL;
    }
    if (rc) return rc;
    // conditioning guard: the kernels above returned at once if ctrl.robust is set; this one returns at once if it is not
    if (g_robust_threshold < INFINITY) rc = launch_pass_simple(a, K, D, dtype, 1, s);
    return rc;
}
