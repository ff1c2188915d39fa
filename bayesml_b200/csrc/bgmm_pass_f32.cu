// bgmm_pass, fp32 streaming variant (BGMM_PASS_F32) for small D (<= 3) and K (<= 8): BASELINE config C3
// (N = 200M, D = 2, K = 8, "fp32 mode").
//
// One thread owns one sample at a time; everything per sample lives in registers:
//   E-step   ln rho_nk in base 2, whitened form  a2_k - |L'_k^T (x' - m'_k)|^2   (L' = chol(nu W) * sqrt(log2(e)/2)),
//            softmax with MUFU.EX2 / MUFU.RCP, entropy term with MUFU.LG2;
//   M-stats  raw_k += r_nk * phi(x'_n) in per-thread fp32 accumulators, flushed every F32_FLUSH samples through a
//            warp shuffle reduction into per-warp fp64 accumulators in shared memory (fp32 error stays ~1e-7 relative).
// X is streamed once with coalesced vector loads (D*4 bytes per sample); r never touches HBM.  The whitened form keeps
// (x' - m'_k) explicit, so fp32 cancellation does not grow with the distance of a component from the centre.
// The kernel is FP32-issue bound, not HBM bound (SURVEY.md §8d: 8 components per 8-byte sample).
// Two E-step forms, chosen per launch from the conditioning criterion bgmm_small leaves in ctrl.CRIT (§2 of DESIGN.md):
//   crit <= 128 (BASELINE C3: 107): the feature-map form  c_k + b_k.x' + x'^T Q_k x'  — 5 FMAs per (sample, component) at
//                D = 2 on the phi values the statistics need anyway; fp32 error ~ 6e-8 * crit * sqrt(P) <= 2e-5 in ln rho;
//   otherwise:   the whitened form, 9 operations, which keeps (x' - m'_k) explicit and does not degrade with crit.
// OUT = false is the loop instantiation (no r / ln rho / argmax stores, no argmax tracking).
// Replaces `_update_q_z` :772-784, `_calc_n_x_bar_s` :725-732, `xlogy` :704 (reference GMM file) in fp32 mode; parity
// bar 1e-4 relative against the fp64 oracle fed the same fp32-rounded X.
#include "bgmm_common.cuh"
#include <math.h>
#include <stdlib.h>

namespace bgmm {

constexpr int F32_THREADS = 128;
constexpr int F32_KMAX = 8;
constexpr int F32_FLUSH = 128;       // samples per thread between flushes of the fp32 accumulators

__device__ __forceinline__ float ex2_approx(float x) {       // MUFU.EX2, flush-to-zero: 2^x for x <= 0 (2 ulp)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// per-CTA partial from the per-warp float64 accumulators, then the finish of the pass (last CTA: sum in CTA order, publish)
template <int P>
__device__ __forceinline__ void f32_epilogue(const PassArgs& a, const Layout& L, volatile int* ctrl,
                                             double (&wsum)[F32_THREADS / 32][F32_KMAX * P + 1]) {
    constexpr int NW = F32_THREADS / 32;
    const int K = L.K, tid = threadIdx.x;
    // ---- per-CTA partial (fp64, logical layout [K][pitch]) ----
    const int64_t len = L.stats_len;
    double* part = a.workspace + (int64_t)blockIdx.x * len;
    for (int64_t o = tid; o < len; o += F32_THREADS) part[o] = 0.0;
    __syncthreads();
    for (int i = tid; i < K * P; i += F32_THREADS) {
        const int k = i / P, p = i - k * P;
        double v = 0.0;
        for (int w = 0; w < NW; ++w) v += wsum[w][k * P + p];
        part[(int64_t)k * L.pitch + p] = v;
    }
    if (tid == 0) {
        double v = 0.0;
        for (int w = 0; w < NW; ++w) v += wsum[w][F32_KMAX * P];
        part[(int64_t)K * L.pitch + BGMM_STATS_ENTROPY] = v;
    }
    finish_pass(a, L, ctrl, 0.0);                 // moments about the centre
}

template <int D>
struct F32Params {                   // per component, fp32, in shared memory
    float m[D];
    float lt[D * (D + 1) / 2];       // packed lower triangle of L' (row-major: (i, j<=i) at i(i+1)/2 + j)
    float a2;                        // ln rho constant in base 2
};

constexpr int F32_FEAT_CRIT = 128;   // feature-map E-step up to this value of ctrl.CRIT

template <int D, bool OUT>
__global__ void __launch_bounds__(F32_THREADS) pass_f32_kernel(const PassArgs a, const Layout L, const int skip_if_feat) {
    constexpr int P = 1 + D + D * (D + 1) / 2;
    constexpr int NW = F32_THREADS / 32;
    __shared__ F32Params<D> prm[F32_KMAX];
    __shared__ double wsum[NW][F32_KMAX * P + 1];
    __shared__ double red[40];
    const int K = L.K, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust)) return;
    const double* Pc = a.state + L.params[ctrl[BGMM_CTRL_CUR]];
    const float* __restrict__ x = static_cast<const float*>(a.x);
    const bool feat = ctrl[BGMM_CTRL_CRIT] <= F32_FEAT_CRIT;   // uniform: which E-step form this launch uses
    if (skip_if_feat && feat) return;                           // pass_f32x2_kernel (launched just before) did this pass

    // ---- prologue: whitening factors of Lambda_k = nu_k W_k (fp64 Cholesky of a D x D matrix per component) ----
    if (tid < F32_KMAX) {
        const int k = tid;
        F32Params<D>& q = prm[k];
        if (k < K) {
            const double nu = Pc[L.p_nu + k], kappa = Pc[L.p_kappa + k];
            const double* W = Pc + L.p_w + (int64_t)k * D * D;
            double lo[D][D];
            bool ok = true;
            for (int i = 0; i < D; ++i)
                for (int j = 0; j <= i; ++j) {
                    double s = nu * W[i * D + j];
                    for (int l = 0; l < j; ++l) s -= lo[i][l] * lo[j][l];
                    if (i == j) { ok = ok && (s > 0.0); lo[i][i] = sqrt(s); }
                    else lo[i][j] = s / lo[j][j];
                }
            const double sc = sqrt(0.5 * 1.4426950408889634074);
            for (int i = 0; i < D; ++i) {
                q.m[i] = (float)Pc[L.p_m + (int64_t)k * D + i];
                for (int j = 0; j <= i; ++j) q.lt[i * (i + 1) / 2 + j] = (float)(lo[i][j] * sc);
            }
            const double ak = Pc[L.p_elnpi + k] + 0.5 * (Pc[L.p_elndet + k] - D * 1.837877066409345483560659472811 - D / kappa);
            q.a2 = (float)(ak * 1.4426950408889634074);
            if (!ok) ctrl[BGMM_CTRL_ERROR] = 1;
            if (feat) {
                // the same slots hold the feature-map coefficients in base 2: a2 <- constant, m[i] <- linear, lt[(i,j)] <- quadratic
                const double* cf = Pc + L.p_coef + (int64_t)k * L.pitch;
                const double l2e = 1.4426950408889634074;
                q.a2 = (float)(cf[0] * l2e);
                for (int i = 0; i < D; ++i) q.m[i] = (float)(cf[1 + i] * l2e);
                for (int i = 0; i < D * (D + 1) / 2; ++i) q.lt[i] = (float)(cf[1 + D + i] * l2e);
            }
        } else {
            for (int i = 0; i < D; ++i) q.m[i] = 0.f;
            for (int i = 0; i < D * (D + 1) / 2; ++i) q.lt[i] = 0.f;
            q.a2 = -1.0e30f;                                  // padded components: r == 0 exactly
        }
    }
    for (int i = lane; i < F32_KMAX * P + 1; i += 32) wsum[warp][i] = 0.0;
    __syncthreads();

    // D <= 2: the component parameters live in registers (48 floats at D=2, K=8); per-(n,k) shared-memory broadcasts
    // would make the kernel LSU bound.  D = 3 keeps them in shared memory (register budget).
    constexpr bool kRegParams = (D <= 2);
    constexpr int NLT = D * (D + 1) / 2;
    float pm[kRegParams ? F32_KMAX : 1][D], plt[kRegParams ? F32_KMAX : 1][NLT], pa2[kRegParams ? F32_KMAX : 1];
    if constexpr (kRegParams) {
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
#pragma unroll
            for (int i = 0; i < D; ++i) pm[k][i] = prm[k].m[i];
#pragma unroll
            for (int i = 0; i < NLT; ++i) plt[k][i] = prm[k].lt[i];
            pa2[k] = prm[k].a2;
        }
    }
    float acc[F32_KMAX][P];
#pragma unroll
    for (int k = 0; k < F32_KMAX; ++k)
#pragma unroll
        for (int p = 0; p < P; ++p) acc[k][p] = 0.f;
    float ent = 0.f;
    int pending = 0;

    auto flush = [&]() {
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k)
#pragma unroll
            for (int p = 0; p < P; ++p) {
                float v = acc[k][p];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) wsum[warp][k * P + p] += (double)v;
                acc[k][p] = 0.f;
            }
        float v = ent;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) wsum[warp][F32_KMAX * P] += (double)v;
        ent = 0.f;
        pending = 0;
    };

    // warp-uniform loop (every lane runs the same number of iterations; rows past the end are masked) so that the
    // full-warp shuffles of flush() are always executed by all 32 lanes
    const int64_t stride = (int64_t)gridDim.x * F32_THREADS;
    auto load_row = [&](int64_t row, float (&dst)[D]) {
        if (row < a.n) {
            if constexpr (D == 2) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(x) + row);
                dst[0] = v.x; dst[1] = v.y;
            } else {
#pragma unroll
                for (int i = 0; i < D; ++i) dst[i] = __ldg(x + row * D + i);
            }
        } else {
#pragma unroll
            for (int i = 0; i < D; ++i) dst[i] = 0.f;
        }
    };
    // software pipeline: the loads of the next two grid-stride rows are in flight while this row is processed
    float xn1[D], xn2[D];
    {
        const int64_t b0 = (int64_t)blockIdx.x * F32_THREADS + warp * 32 + lane;
        load_row(b0, xn1);
        load_row(b0 + stride, xn2);
    }
    for (int64_t base = (int64_t)blockIdx.x * F32_THREADS + warp * 32; base < a.n; base += stride) {
        const int64_t n = base + lane;
        const bool valid = n < a.n;
        float xv[D];
#pragma unroll
        for (int i = 0; i < D; ++i) { xv[i] = xn1[i]; xn1[i] = xn2[i]; }
        load_row(n + 2 * stride, xn2);
        // the register rotation above touches the row loaded ONE iteration ago (22 % of the stall samples in the round-2 C3
        // profile when it came from HBM): pull the rows of six iterations ahead into L2 so that load is a ~300-cycle hit
        if (n + 6 * stride < a.n) asm volatile("prefetch.global.L2 [%0];" ::"l"(x + (n + 6 * stride) * D));
        // statistics features about the global centre: phi = [1, x, x_i x_j (i >= j)] (also the E-step's in the feature form)
        float phi[P];
        phi[0] = 1.f;
#pragma unroll
        for (int i = 0; i < D; ++i) phi[1 + i] = xv[i];
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) phi[1 + D + i * (i + 1) / 2 + j] = xv[i] * xv[j];
        // E-step
        float l2[F32_KMAX];
        float mx = -3.0e38f;
        if (feat) {
#pragma unroll
            for (int k = 0; k < F32_KMAX; ++k) {
                float v = kRegParams ? pa2[kRegParams ? k : 0] : prm[k].a2;
#pragma unroll
                for (int i = 0; i < D; ++i) v = fmaf(kRegParams ? pm[kRegParams ? k : 0][i] : prm[k].m[i], phi[1 + i], v);
#pragma unroll
                for (int i = 0; i < NLT; ++i) v = fmaf(kRegParams ? plt[kRegParams ? k : 0][i] : prm[k].lt[i], phi[1 + D + i], v);
                l2[k] = v;
                mx = fmaxf(mx, v);
            }
        } else {
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            float d[D];
#pragma unroll
            for (int i = 0; i < D; ++i) d[i] = xv[i] - (kRegParams ? pm[kRegParams ? k : 0][i] : prm[k].m[i]);
            float qf = 0.f;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                float y = 0.f;
#pragma unroll
                for (int i = j; i < D; ++i)
                    y = fmaf(kRegParams ? plt[kRegParams ? k : 0][i * (i + 1) / 2 + j] : prm[k].lt[i * (i + 1) / 2 + j], d[i], y);
                qf = fmaf(y, y, qf);
            }
            l2[k] = (kRegParams ? pa2[kRegParams ? k : 0] : prm[k].a2) - qf;
            mx = fmaxf(mx, l2[k]);
        }
        }
        if (OUT && a.lnrho_out != nullptr && valid) {
#pragma unroll
            for (int k = 0; k < F32_KMAX; ++k)          // unrolled + guarded: keeps l2[] in registers
                if (k < K) a.lnrho_out[n * K + k] = (double)l2[k] * 0.693147180559945309417232121458;
        }
        float s = 0.f, dot = 0.f, e[F32_KMAX];
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            const float z = l2[k] - mx;                 // finite: padded components sit at -1e30
            e[k] = ex2_approx(z);
            s += e[k];
            dot = fmaf(e[k], z, dot);
        }
        const float inv = valid ? rcp_approx(s) : 0.f;  // 1 <= s <= K
        if (valid) ent += 0.693147180559945309f * (dot * inv - lg2_approx(s));
        int best = 0;
        float bestv = -1.f;
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            const float r = e[k] * inv;
            e[k] = r;
            if (OUT) { if (r > bestv) { bestv = r; best = k; } }
            acc[k][0] += r;
#pragma unroll
            for (int p = 1; p < P; ++p) acc[k][p] = fmaf(r, phi[p], acc[k][p]);
        }
        if (OUT && a.r_out != nullptr && valid) {
#pragma unroll
            for (int k = 0; k < F32_KMAX; ++k)
                if (k < K) a.r_out[n * K + k] = (double)e[k];
        }
        if (OUT && a.argmax_out != nullptr && valid) a.argmax_out[n] = best;
        if (++pending == F32_FLUSH) flush();
    }
    flush();
    __syncthreads();

    f32_epilogue<P>(a, L, ctrl, wsum);
    (void)red;
}

// ---- D = 2, feature-map form, loop instantiation: two samples per thread in packed f32x2 arithmetic ----
// BASELINE C3's shape.  The scalar kernel above issues ~155 instructions per sample; here everything except the E-step dot
// products (whose coefficients are per-component scalars held in registers) works on PAIRS of consecutive samples in
// 64-bit registers: phi, the softmax subtraction / sum / entropy dot product, r and the 48 statistics accumulators (FFMA2 /
// FADD2 / FMUL2: ~107 instructions per sample).  Launched before pass_f32_kernel<2, false>, which returns at once when this
// kernel took the pass (and does the pass itself when the conditioning criterion asks for the whitened form).
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

__global__ void __launch_bounds__(F32_THREADS, 2) pass_f32x2_kernel(const PassArgs a, const Layout L) {
    constexpr int D = 2, P = 6, NW = F32_THREADS / 32;
    __shared__ float cf[F32_KMAX][P];
    __shared__ double wsum[NW][F32_KMAX * P + 1];
    const int K = L.K, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust)) return;
    if (!(ctrl[BGMM_CTRL_CRIT] <= F32_FEAT_CRIT)) return;       // whitened form: the scalar kernel does this pass
    const double* Pc = a.state + L.params[ctrl[BGMM_CTRL_CUR]];
    const float* __restrict__ x = static_cast<const float*>(a.x);
    if (tid < F32_KMAX * P) {
        const int k = tid / P, p = tid - k * P;
        // base-2 feature-map coefficients [const, x, y, xx, xy, yy]; padded components sit at -1e30 (r == 0 exactly)
        cf[k][p] = k < K ? (float)(Pc[L.p_coef + (int64_t)k * L.pitch + p] * 1.4426950408889634074) : (p == 0 ? -1.0e30f : 0.f);
    }
    for (int i = lane; i < F32_KMAX * P + 1; i += 32) wsum[warp][i] = 0.0;
    __syncthreads();
    // the E-step stays scalar: (coefficient, coefficient) pairs for a packed E-step would need 96 more registers; measured
    // with them the compiler rebuilds the pairs per use and the kernel is 11 % slower
    float c[F32_KMAX][P];
#pragma unroll
    for (int k = 0; k < F32_KMAX; ++k)
#pragma unroll
        for (int p = 0; p < P; ++p) c[k][p] = cf[k][p];
    f32x2 acc[F32_KMAX][P];
#pragma unroll
    for (int k = 0; k < F32_KMAX; ++k)
#pragma unroll
        for (int p = 0; p < P; ++p) acc[k][p] = 0ull;
    float ent = 0.f;
    int pending = 0;
    auto flush = [&]() {
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k)
#pragma unroll
            for (int p = 0; p < P; ++p) {
                float lo, hi;
                upk(acc[k][p], lo, hi);
                float v = lo + hi;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) wsum[warp][k * P + p] += (double)v;
                acc[k][p] = 0ull;
            }
        float v = ent;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) wsum[warp][F32_KMAX * P] += (double)v;
        ent = 0.f;
        pending = 0;
    };
    // a thread owns the samples 2 q and 2 q + 1 of pair q: one 16-byte load, a warp reads 512 contiguous bytes
    const int64_t npairs = (a.n + 1) >> 1, stride = (int64_t)gridDim.x * F32_THREADS;
    auto load_pair = [&](int64_t q) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (2 * q + 1 < a.n) v = __ldg(reinterpret_cast<const float4*>(x) + q);
        else if (2 * q < a.n) { const float2 h = __ldg(reinterpret_cast<const float2*>(x) + 2 * q); v.x = h.x; v.y = h.y; }
        return v;
    };
    const int64_t q0 = (int64_t)blockIdx.x * F32_THREADS + warp * 32 + lane;
    float4 xn1 = load_pair(q0), xn2 = load_pair(q0 + stride);
    for (int64_t base = (int64_t)blockIdx.x * F32_THREADS + warp * 32; base < npairs; base += stride) {
        const int64_t q = base + lane;
        const bool va = 2 * q < a.n, vb = 2 * q + 1 < a.n;
        const float4 xv = xn1;
        xn1 = xn2;
        xn2 = load_pair(q + 2 * stride);
        if (q + 6 * stride < npairs) asm volatile("prefetch.global.L2 [%0];" ::"l"(x + (q + 6 * stride) * 4));
        const f32x2 X = pk(xv.x, xv.z), Y = pk(xv.y, xv.w);
        const f32x2 XX = mul2(X, X), XY = mul2(X, Y), YY = mul2(Y, Y);
        float xxa, xxb, xya, xyb, yya, yyb;
        upk(XX, xxa, xxb); upk(XY, xya, xyb); upk(YY, yya, yyb);
        float la[F32_KMAX], lb[F32_KMAX];
        float mxa = -3.0e38f, mxb = -3.0e38f;
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            float u = fmaf(c[k][1], xv.x, c[k][0]), w = fmaf(c[k][1], xv.z, c[k][0]);
            u = fmaf(c[k][2], xv.y, u);  w = fmaf(c[k][2], xv.w, w);
            u = fmaf(c[k][3], xxa, u);   w = fmaf(c[k][3], xxb, w);
            u = fmaf(c[k][4], xya, u);   w = fmaf(c[k][4], xyb, w);
            u = fmaf(c[k][5], yya, u);   w = fmaf(c[k][5], yyb, w);
            la[k] = u; lb[k] = w;
            mxa = fmaxf(mxa, u); mxb = fmaxf(mxb, w);
        }
        const f32x2 NMX = pk(-mxa, -mxb);
        f32x2 E[F32_KMAX], S = 0ull, DOT = 0ull;
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            const f32x2 Z = add2(pk(la[k], lb[k]), NMX);        // finite: padded components sit at -1e30
            float za, zb;
            upk(Z, za, zb);
            E[k] = pk(ex2_approx(za), ex2_approx(zb));
            S = add2(S, E[k]);
            DOT = fma2(E[k], Z, DOT);
        }
        float sa, sb, da, db;
        upk(S, sa, sb); upk(DOT, da, db);
        const float inva = va ? rcp_approx(sa) : 0.f, invb = vb ? rcp_approx(sb) : 0.f;       // 1 <= s <= K
        if (va) ent += 0.693147180559945309f * (da * inva - lg2_approx(sa));
        if (vb) ent += 0.693147180559945309f * (db * invb - lg2_approx(sb));
        const f32x2 INV = pk(inva, invb);
#pragma unroll
        for (int k = 0; k < F32_KMAX; ++k) {
            const f32x2 R = mul2(E[k], INV);
            acc[k][0] = add2(acc[k][0], R);
            acc[k][1] = fma2(R, X, acc[k][1]);
            acc[k][2] = fma2(R, Y, acc[k][2]);
            acc[k][3] = fma2(R, XX, acc[k][3]);
            acc[k][4] = fma2(R, XY, acc[k][4]);
            acc[k][5] = fma2(R, YY, acc[k][5]);
        }
        if (++pending == F32_FLUSH / 2) flush();
    }
    flush();
    __syncthreads();
    f32_epilogue<P>(a, L, ctrl, wsum);
    (void)D;
}

bool f32_supported(int K, int D, int dtype) { return dtype == BGMM_F32 && D >= 1 && D <= 3 && K <= F32_KMAX; }

template <int D, bool OUT>
static int f32_grid(int64_t n) {
    int dev = 0, sms = 148, occ = 1;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pass_f32_kernel<D, OUT>, F32_THREADS, 0);
    if (occ < 1) occ = 1;
    const int64_t want = (n + F32_THREADS - 1) / F32_THREADS;
    int64_t cap = (int64_t)sms * occ;                          // one resident wave: persistent grid-stride CTAs
    if (cap > 1024) cap = 1024;
    return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

int64_t f32_workspace_doubles(int K, int D) {
    if (!(D >= 1 && D <= 3 && K <= F32_KMAX)) return 0;
    return (int64_t)1024 * ((int64_t)K * feat_pitch(D) + 8);
}

int launch_pass_f32(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream) {
    if (!f32_supported(K, D, dtype)) {
        set_error("bgmm_pass(f32): unsupported shape K=%d D=%d dtype=%d", K, D, dtype);
        return BGMM_ENOSUP;
    }
    const Layout L = make_layout(K, D, 1);
    const bool out = a.r_out != nullptr || a.lnrho_out != nullptr || a.argmax_out != nullptr;
    // C3's shape in the loop: the packed two-samples-per-thread kernel first; the scalar kernel then returns at once unless the
    // conditioning criterion asked for the whitened form (BGMM_F32_PACKED=0 keeps the scalar kernel alone)
    const char* env_packed = getenv("BGMM_F32_PACKED");         // read per launch: tests compare the two kernels
    const int packed_on = (env_packed == nullptr || atoi(env_packed) != 0) ? 1 : 0;
    const int packed = (D == 2 && !out && packed_on) ? 1 : 0;
    if (packed) {
        int dev = 0, sms = 148, occ = 1;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pass_f32x2_kernel, F32_THREADS, 0);
        if (occ < 1) occ = 1;
        const int64_t want = ((a.n + 1) / 2 + F32_THREADS - 1) / F32_THREADS;
        int64_t cap = (int64_t)sms * occ;
        if (cap > 1024) cap = 1024;
        launch(pass_f32x2_kernel, (int)(want < 1 ? 1 : (want < cap ? want : cap)), F32_THREADS, 0, stream, a, L);
    }
#define BGMM_F32_CASE(d, o) if (D == d && out == o) launch(pass_f32_kernel<d, o>, f32_grid<d, o>(a.n), F32_THREADS, 0, stream, a, L, packed);
    BGMM_F32_CASE(1, false) BGMM_F32_CASE(1, true) BGMM_F32_CASE(2, false) BGMM_F32_CASE(2, true)
    BGMM_F32_CASE(3, false) BGMM_F32_CASE(3, true)
#undef BGMM_F32_CASE
    return check_cuda(cudaGetLastError(), "pass_f32_kernel launch");
}

}  // namespace bgmm
