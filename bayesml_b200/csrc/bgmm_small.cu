// bgmm_small: the O(K D^3) part of one VB iteration, one CTA per mixture component.
//
// Replaces, in /root/reference/bayesml/gaussianmixture/_gaussianmixture.py:
//   _update_q_mu_lambda :758-770   kappa, m, nu, W^-1 from (N_k, x_bar_k, S_k); W = inv(W^-1)
//   _update_q_pi        :741-743   alpha = alpha0 + N
//   _calc_q_pi_features :738-739   E[ln pi_k] = psi(alpha_k) - psi(sum alpha)
//   _calc_q_lambda_features :745-756   E[ln|Lambda|], ln B(W, nu)   (E[Lambda] = nu W is folded into coef)
//   _calc_vl            :671-723   all K-sized ELBO terms (the O(N K) term sum r ln r comes from bgmm_pass)
//   update_posterior    :869       the convergence test, on the device (no host sync in the loop)
// The reference inverts with LAPACK LU (`np.linalg.inv`, `slogdet`); W^-1 is SPD so this kernel uses one
// Cholesky factorisation for the inverse and the log-determinant (agrees to cond*eps, tested vs the oracle).
#include "bgmm_common.cuh"
#include <math.h>

namespace bgmm {

// The kernel below is straight-line code executed once per launch, so its running time is dominated by instruction
// fetch (cold I-cache after the big pass kernel) unless the code stays small: the libm calls are kept out of line.
__device__ __noinline__ double lgamma_ni(double x) { return lgamma(x); }
__device__ __noinline__ double log_ni(double x) { return log(x); }

// psi(x), x > 0: upward recurrence to x >= 10 then the asymptotic series (error < 1e-16 relative there).
__device__ __noinline__ double digamma_pos(double x) {
    double r = 0.0;
    while (x < 10.0) { r -= 1.0 / x; x += 1.0; }
    const double inv = 1.0 / x, inv2 = inv * inv;
    double s = 691.0 / 32760.0 - inv2 * (1.0 / 12.0);
    s = 1.0 / 132.0 - inv2 * s;
    s = 1.0 / 240.0 - inv2 * s;
    s = 1.0 / 252.0 - inv2 * s;
    s = 1.0 / 120.0 - inv2 * s;
    s = 1.0 / 12.0 - inv2 * s;
    return r + log_ni(x) - 0.5 * inv - inv2 * s;
}

constexpr double LN2 = 0.693147180559945309417232121458;
constexpr double LNPI = 1.144729885849400174143427351353;
constexpr double LN2PI = 1.837877066409345483560659472811;

__device__ __forceinline__ double ld_peer(const double* p) {     // peer / exchange memory: never from a stale L1 line
    double v;
    asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}

// ---- the stages both kernels share ----------------------------------------------------------------------------------
// small_kernel (D > 32) runs component k with a CTA, small_warp_kernel (D <= 32) with one warp.  They differ in the dense
// algebra (Cholesky, L^-1, W, the quadratic part of the coefficient row), in where the D x D operands live and in how the
// special functions are evaluated.  Everything else is written once below, templated on the team that runs it.

struct BlockTeam {                        // small_kernel: the CTA, block barriers
    const int rank, size;
    double* scratch;                      // >= 33 doubles of shared memory for the reductions
    __device__ explicit BlockTeam(double* s) : rank(threadIdx.x), size(blockDim.x), scratch(s) {}
    __device__ void sync() const { __syncthreads(); }
    __device__ double sum(double v) const { return block_sum(v, scratch); }
    __device__ void sum4(double& a, double& b, double& c, double& d) const { block_sum4(a, b, c, d, scratch); }
    template <class F> __device__ void rows(int D, F f) const { for (int i = rank; i < D; i += size) f(i); }
    // true in every thread of the CTA that increments *ticket last of n; it then sees the stores of every other CTA
    __device__ bool last(int* ticket, int n) const {
        __shared__ int is_last;
        __threadfence();
        __syncthreads();
        if (rank == 0) is_last = (atomicAdd(ticket, 1) == n - 1);
        __syncthreads();
        return is_last;
    }
};

struct WarpTeam {                         // small_warp_kernel: one warp, warp-synchronous
    static constexpr int size = 32;
    const int rank;
    __device__ WarpTeam() : rank(threadIdx.x) {}
    __device__ void sync() const { __syncwarp(); }
    __device__ double sum(double v) const { return warp_sum(v); }
    __device__ void sum4(double& a, double& b, double& c, double& d) const {
        a = warp_sum(a); b = warp_sum(b); c = warp_sum(c); d = warp_sum(d);
    }
    template <class F> __device__ void rows(int D, F f) const { if (rank < D) f(rank); }   // D <= 32: lane i owns row i
    __device__ bool last(int* ticket, int n) const {
        __threadfence();
        __syncwarp();
        int is_last = 0;
        if (rank == 0) is_last = (atomicAdd(ticket, 1) == n - 1);
        return __shfl_sync(0xffffffffu, is_last, 0);
    }
};

// Where a kernel keeps the D x D operands of the shared stages: S_k as the ELBO traces and the M-step read it (s, kept by
// keep_s), and the new W^-1 that the M-step leaves for the kernel's Cholesky (a).  e = i * D + j.
struct BlockMats {                        // S_k is read back from state.SMATS; W^-1 goes to the dynamic [D][D] block
    const double* S;
    double* A;
    __device__ double s(int e, int, int) const { return S[e]; }
    __device__ void keep_s(int, int, int, double) const {}
    __device__ double& a(int e, int, int) const { return A[e]; }
};

constexpr int SW_LP = 33;                 // pitch of small_warp_kernel's shared matrices: conflict-free rows and columns

struct WarpMats {                         // S_k and W^-1 in shared memory at pitch SW_LP
    double* Am;
    double* Bm;
    __device__ double s(int, int i, int j) const { return Bm[i * SW_LP + j]; }
    __device__ void keep_s(int, int i, int j, double v) const { Bm[i * SW_LP + j] = v; }
    __device__ double& a(int, int i, int j) const { return Am[i * SW_LP + j]; }
};

// Parameters of component k in the current set (those the pass used): the ELBO terms are evaluated under them.
struct CurParams { double kappa = 1.0, nu = 0.0, alpha = 1.0, elnpi = 0.0, elndet = 0.0, lnb = 0.0; };
struct Traces { double trs = 0.0, q1 = 0.0, q2 = 0.0, tr0 = 0.0; };

// What the stages of component k (= blockIdx.x) read: the mode, the parameter sets, the prior of k and, in a fused call,
// the ranks' exchange blocks xb (an array of the kernel's own: indexed by rank, it lives in local memory).
struct SmallCtx {
    double* st;
    const Layout& L;
    const int K, D, DD, k;
    volatile int* ctrl;
    const bool iterate, stats_only, fused;
    const double** xb;
    int cur, world = 1;
    double *Pc, *Pn;
    const double *m0, *w0inv;
    double alpha0, kappa0, nu0;

    __device__ SmallCtx(double* st_, const Layout& L_, int D_, int mode, const CommDesc* cd, const double** xb_)
        : st(st_), L(L_), K(L_.K), D(D_), DD(D_ * D_), k(blockIdx.x), ctrl(reinterpret_cast<volatile int*>(st_ + L_.ctrl)),
          iterate(mode == BGMM_SMALL_ITERATE), stats_only(mode == BGMM_SMALL_STATS),
          fused(cd != nullptr && (mode == BGMM_SMALL_ITERATE || mode == BGMM_SMALL_STATS)), xb(xb_) {}

    // false: the loop is done (every CTA reads ctrl.DONE before any CTA can take the last ticket)
    __device__ bool begin() {
        if (iterate && ctrl[BGMM_CTRL_DONE]) return false;
        cur = ctrl[BGMM_CTRL_CUR];
        Pc = st + L.params[cur];
        Pn = iterate ? st + L.params[cur ^ 1] : Pc;
        m0 = st + L.m0 + (int64_t)k * D;
        w0inv = st + L.w0inv + (int64_t)k * DD;
        alpha0 = st[L.alpha0 + k]; kappa0 = st[L.kappa0 + k]; nu0 = st[L.nu0 + k];
        return true;
    }
    // offset o of the ranks' published statistics, summed in rank order
    __device__ double peer_sum(int64_t o) const {
        double acc = 0.0;
#pragma unroll 8                          // the ranks of one 8-GPU node in one round of loads
        for (int r = 0; r < world; ++r) acc += ld_peer(xb[r] + o);
        return acc;
    }
    // statistic at offset o of state.STATS: in a fused call summed over the ranks (rows other CTAs own, and the tail CTA 0
    // owns, may not be received yet), otherwise the local value
    __device__ double stat(int64_t o) const { return fused ? peer_sum(o) : st[L.stats + o]; }
    __device__ CurParams current() const {
        CurParams p;
        p.kappa = Pc[L.p_kappa + k]; p.nu = Pc[L.p_nu + k]; p.alpha = Pc[L.p_alpha + k];
        p.elnpi = Pc[L.p_elnpi + k]; p.elndet = Pc[L.p_elndet + k]; p.lnb = Pc[L.p_lnb + k];
        return p;
    }
};

// ---- fused all-reduce over peer memory: wait for every rank's stamp, sum row k (and, in CTA 0, the tail) in rank order ----
template <class T>
__device__ __forceinline__ void receive(const T& t, SmallCtx& c, const CommDesc* cd) {
    const Layout& L = c.L;
    c.world = cd->world;
    const int seq = c.ctrl[BGMM_CTRL_SEQ] - 1;                  // the exchange published by the preceding bgmm_pass
    const int64_t len = L.stats_len;
    if (t.rank < c.world) {
        const unsigned long long* flag = reinterpret_cast<const unsigned long long*>(cd->xchg[cd->rank] + 2 * len) +
                                         (seq & 1) * BGMM_MAX_RANKS + t.rank;
        unsigned long long v;
        do {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
        } while (v < (unsigned long long)(seq + 1));
    }
    t.sync();
    for (int r = 0; r < c.world; ++r) c.xb[r] = cd->xchg[r] + (int64_t)(seq & 1) * len;
    double* row = c.st + L.stats + (int64_t)c.k * L.pitch;      // this CTA owns row k of the reduced statistics
    for (int p = t.rank; p < L.pitch; p += t.size) row[p] = c.peer_sum((int64_t)c.k * L.pitch + p);
    if (c.k == 0 && t.rank < 8) c.st[L.stats + (int64_t)c.K * L.pitch + t.rank] = c.peer_sum((int64_t)c.K * L.pitch + t.rank);
    t.sync();
}

// ---- statistics of component k from the moments about the centre (feature-map kernels) or about shift_k (DIRECT kernel;
//      format slot > 0):  x_bar = shift + d_bar,  S = M2 / N - d_bar d_bar^T.  Returns N_k. ----
template <class T, class M>
__device__ __forceinline__ double component_stats(const T& t, const M& m, const SmallCtx& c, double* xbar, double* dbar) {
    const Layout& L = c.L;
    const int D = c.D, DD = c.DD, k = c.k;
    double* st = c.st;
    const double* raw = st + L.stats + (int64_t)k * L.pitch;
    const double N = raw[0];
    const bool shifted = c.stat((int64_t)c.K * L.pitch + BGMM_STATS_FORMAT) > 0.5;
    const double* sh = st + L.shift + (int64_t)k * D;
    double* S = st + L.smats + (int64_t)k * DD;
    if (N > 0.0) {
        const double invN = 1.0 / N;
        t.rows(D, [&](int i) {
            const double db = raw[1 + i] * invN;
            dbar[i] = db;
            xbar[i] = shifted ? sh[i] + db : db;
        });
        t.sync();
        for (int e = t.rank; e < DD; e += t.size) {
            const int i = e / D, j = e - i * D, hi = max(i, j), lo = min(i, j);
            const double v = raw[1 + D + hi * (hi + 1) / 2 + lo] * invN - dbar[i] * dbar[j];
            S[e] = v;
            m.keep_s(e, i, j, v);
        }
    } else {
        // reference :729 — x_bar_vecs[k] keeps the un-normalised sum (0 in the original frame), s_mats[k] stale
        t.rows(D, [&](int i) { xbar[i] = -st[L.center + i]; });
        for (int e = t.rank; e < DD; e += t.size) m.keep_s(e, e / D, e % D, S[e]);
    }
    t.sync();
    t.rows(D, [&](int i) { st[L.xbar + (int64_t)k * D + i] = xbar[i]; });
    if (t.rank == 0) st[L.ns + k] = N;
    // STATS: x_bar_k becomes the shift of a following centred-statistics sweep (engine.refine_smats: the reference's
    // two-pass s_mats, :730-732, from the materialised responsibilities)
    if (c.stats_only && N > 0.0) t.rows(D, [&](int i) { st[L.shift + (int64_t)k * D + i] = xbar[i]; });
    return N;
}

// ---- the traces of the ELBO terms of component k under the current parameters p ----
template <class T, class M>
__device__ __forceinline__ Traces elbo_traces(const T& t, const M& m, const SmallCtx& c, const CurParams& p,
                                              const double* xbar, double* dev, double* lin) {
    const int D = c.D, DD = c.DD;
    const double* W = c.Pc + c.L.p_w + (int64_t)c.k * DD;
    const double* mc = c.Pc + c.L.p_m + (int64_t)c.k * D;
    // the deviations (x_bar - m), (m - m0) go to shared memory first so the D x D loop only streams W and W0^-1
    t.rows(D, [&](int i) { dev[i] = xbar[i] - mc[i]; lin[i] = mc[i] - c.m0[i]; });
    t.sync();
    Traces tr;
#pragma unroll 4                          // four loads of W and of W0^-1 in flight per thread
    for (int e = t.rank; e < DD; e += t.size) {
        const int i = e / D, j = e - i * D;
        const double w = W[e];
        tr.trs += m.s(e, i, j) * w;
        tr.q1 += dev[i] * w * dev[j];
        tr.q2 += lin[i] * w * lin[j];
        tr.tr0 += c.w0inv[e] * w;
    }
    t.sum4(tr.trs, tr.q1, tr.q2, tr.tr0);
    t.sync();       // dev / lin are reused by the M-step
    return tr;
}

// The K-sized ELBO terms of component k (the O(N K) term sum r ln r comes from bgmm_pass), from the traces and
// ln kappa0, ln kappa, lnGamma(alpha), psi(alpha) of the current parameters.
__device__ __forceinline__ void elbo_terms(const SmallCtx& c, double N, const CurParams& p, const Traces& tr,
                                           double ln_kappa0, double ln_kappa, double lg_alpha, double psi_alpha) {
    const int D = c.D;
    const double kappa0 = c.kappa0, nu0 = c.nu0, kappa = p.kappa, nu = p.nu, elndet = p.elndet, elnpi = p.elnpi;
    double* vk = c.st + c.L.vlk + (int64_t)c.k * 8;
    const double lnb0 = c.st[c.L.lnb0 + c.k];
    vk[0] = N * (elndet - D / kappa - nu * tr.trs - nu * tr.q1 - D * LN2PI) / 2.0;                   // :673-683
    vk[1] = N * elnpi;                                                                             // :686
    vk[2] = (c.alpha0 - 1.0) * elnpi;                                                              // :689
    vk[3] = (D * (ln_kappa0 - LN2PI - kappa0 / kappa) - kappa0 * nu * tr.q2 + 2.0 * lnb0
             + (nu0 - D) * elndet - nu * tr.tr0) / 2.0;                                            // :692-701
    vk[4] = lg_alpha - (p.alpha - 1.0) * psi_alpha;                                                // :707 (per-k part)
    vk[5] = (D * (1.0 + LN2PI - ln_kappa) - 2.0 * p.lnb - (nu - D) * elndet + nu * D) / 2.0;       // :710-715
    vk[6] = p.alpha;
}

// ---- M-step (:758-768, :742) into the other parameter set; W^-1 also to m.a.  Returns sum_j alpha_j of the new set. ----
template <class T, class M>
__device__ __forceinline__ double m_step(const T& t, const M& m, const SmallCtx& c, double N, const double* xbar,
                                         double* mnew, double* dev, double& kn, double& nun, double& an) {
    const Layout& L = c.L;
    const int D = c.D, DD = c.DD, k = c.k;
    const double kappa0 = c.kappa0;
    double* Pn = c.Pn;
    kn = kappa0 + N; nun = c.nu0 + N; an = c.alpha0 + N;
    t.rows(D, [&](int i) {
        mnew[i] = (kappa0 * c.m0[i] + N * xbar[i]) / kn;
        dev[i] = xbar[i] - c.m0[i];
    });
    t.sync();
    const double c2 = kappa0 * N / kn;
    double* winv_out = Pn + L.p_winv + (int64_t)k * DD;
    for (int e = t.rank; e < DD; e += t.size) {
        const int i = e / D, j = e - i * D;
        const double v = c.w0inv[e] + N * m.s(e, i, j) + c2 * (dev[i] * dev[j]);
        m.a(e, i, j) = v;
        winv_out[e] = v;
    }
    double asum = 0.0;
    for (int j = t.rank; j < c.K; j += t.size) asum += c.st[L.alpha0 + j] + c.stat((int64_t)j * L.pitch);
    const double alpha_sum_new = t.sum(asum);
    if (t.rank == 0) { Pn[L.p_kappa + k] = kn; Pn[L.p_nu + k] = nun; Pn[L.p_alpha + k] = an; }
    t.rows(D, [&](int i) { Pn[L.p_m + (int64_t)k * D + i] = mnew[i]; });
    return alpha_sum_new;
}

// FEATURES: no M-step; the features and the coefficient row are those of the current set.  Returns sum_j alpha_j.
template <class T, class M>
__device__ __forceinline__ double current_set(const T& t, const M& m, const SmallCtx& c, double* mnew, double& kn,
                                              double& nun, double& an) {
    const Layout& L = c.L;
    const int D = c.D, DD = c.DD, k = c.k;
    const double* Pc = c.Pc;
    kn = Pc[L.p_kappa + k]; nun = Pc[L.p_nu + k]; an = Pc[L.p_alpha + k];
    t.rows(D, [&](int i) { mnew[i] = Pc[L.p_m + (int64_t)k * D + i]; });
    for (int e = t.rank; e < DD; e += t.size) m.a(e, e / D, e % D) = Pc[L.p_winv + (int64_t)k * DD + e];
    double asum = 0.0;
    for (int j = t.rank; j < c.K; j += t.size) asum += Pc[L.p_alpha + j];
    return t.sum(asum);
}

// ---- features of the new set (:738-739, :745-756) from ln|W^-1| and E[ln pi]; returns E[ln|Lambda|] ----
template <class T>
__device__ __forceinline__ void nu_sums(const T& t, int D, double nun, double& ps, double& gs) {
    ps = 0.0; gs = 0.0;
    for (int i = t.rank; i < D; i += t.size) {
        const double a = (nun - i) / 2.0;
        ps += digamma_pos(a);
        gs += lgamma_ni(a);
    }
    ps = t.sum(ps);
    gs = t.sum(gs);
}
template <class T>
__device__ __forceinline__ double store_features(const T& t, const SmallCtx& c, double nun, double ps, double gs,
                                                 double logdet, double elnpi_n) {
    const int D = c.D;
    const double elndet_n = ps + D * LN2 - logdet;
    const double lnb_n = (nun * logdet - nun * D * LN2 - D * (D - 1) / 2.0 * LNPI - gs * 2.0) / 2.0;
    if (t.rank == 0) {
        c.Pn[c.L.p_elndet + c.k] = elndet_n;
        c.Pn[c.L.p_lnb + c.k] = lnb_n;
        c.Pn[c.L.p_elnpi + c.k] = elnpi_n;
    }
    return elndet_n;
}

// ---- the scalar part of the E-step coefficient row (ln rho = coef . phi(x'), Lambda = nu W) with mq = m^T Lambda m,
//      its zero padding, the conditioning criterion and the DIRECT kernel's shift ----
template <class T>
__device__ __forceinline__ void store_row(const T& t, const SmallCtx& c, const double* hmm_vlx, double elnpi_n,
                                          double elndet_n, double kn, double mq, double crit_n, const double* xbar,
                                          const double* mnew) {
    const Layout& L = c.L;
    const int D = c.D, k = c.k;
    double* coef = c.Pn + L.p_coef + (int64_t)k * L.pitch;
    for (int q = L.P + t.rank; q < L.pitch; q += t.size) coef[q] = 0.0;
    if (t.rank == 0) {
        // hidden-Markov emission density (_hiddenmarkovnormal.py:988-992): no E[ln pi] term in ln rho
        const double acst = (hmm_vlx != nullptr ? 0.0 : elnpi_n) + (elndet_n - D * LN2PI - D / kn) / 2.0;
        coef[0] = acst - 0.5 * mq;
        c.Pn[L.p_acst + k] = acst;                              // ln rho constant of the DIRECT form (no m^T Lambda m term)
        // conditioning of the feature-map form for this component: the terms of coef . phi(x') are of size
        // mq = m'^T Lambda m' for the samples the component is responsible for, the result is O(D)
        // (K = 1: r == 1 exactly whatever ln rho is, and the moments about the global centre ARE the centred ones)
        c.st[L.vlk + (int64_t)k * 8 + 7] = (c.K == 1) ? 0.0 : crit_n * mq;
    }
    // the point the DIRECT kernel takes the next moments about: this pass's x_bar_k (the next one will be close), or the
    // new m_k while the component has no statistics yet
    double* sh = c.st + L.shift + (int64_t)k * D;
    const bool have_xbar = c.iterate && crit_n > 0.0;
    t.rows(D, [&](int i) { sh[i] = have_xbar ? xbar[i] : mnew[i]; });
}

// ---- last CTA: conditioning flag of the new parameter set; sum the ELBO, convergence test (:869), flip the sets ----
// The first W threads of the team sum the per-component terms: W = 1 in component order, W = 32 lane-strided, then
// across the warp.
template <int W, class T>
__device__ __forceinline__ void finish_iteration(const T& t, const SmallCtx& c, int max_itr, double tol,
                                                 const double* hmm_vlx, double robust_thresh) {
    const Layout& L = c.L;
    const int K = c.K, lane = t.rank;
    volatile int* ctrl = c.ctrl;
    if (!t.last(const_cast<int*>(&ctrl[BGMM_CTRL_TICKET]), K) || lane >= W) return;
    __threadfence();
    double* st = c.st;
    const double* vkg = st + L.vlk;
    double px = 0, pz = 0, ppi = 0, pml = 0, qpi = 0, qml = 0, asum = 0, crit = 0;
    for (int j = lane; j < K; j += W) {
        px += __ldcg(vkg + j * 8 + 0); pz += __ldcg(vkg + j * 8 + 1); ppi += __ldcg(vkg + j * 8 + 2);
        pml += __ldcg(vkg + j * 8 + 3); qpi += __ldcg(vkg + j * 8 + 4); qml += __ldcg(vkg + j * 8 + 5);
        asum += __ldcg(vkg + j * 8 + 6);
        crit = fmax(crit, __ldcg(vkg + j * 8 + 7));
    }
    if (W > 1) {
        px = warp_sum(px); pz = warp_sum(pz); ppi = warp_sum(ppi); pml = warp_sum(pml); qpi = warp_sum(qpi);
        qml = warp_sum(qml); asum = warp_sum(asum);
        for (int o = 16; o > 0; o >>= 1) crit = fmax(crit, __shfl_xor_sync(0xffffffffu, crit, o));
    }
    const int robust = crit > robust_thresh ? 1 : 0;
    const int critq = crit < 1073741824.0 ? (int)ceil(crit) : 1073741824;     // NaN -> the large value
    if (!c.iterate) {
        if (lane == 0) { ctrl[BGMM_CTRL_ROBUST] = robust; ctrl[BGMM_CTRL_CRIT] = critq; ctrl[BGMM_CTRL_TICKET] = 0; }
        return;
    }
    double lg_asum, psi_as;
    if (W > 1) {    // lane 0: lgamma(sum alpha), lane 1: digamma(sum alpha) — one divergent pair instead of two serial calls
        double sf = 0.0;
        if (lane == 0) sf = lgamma_ni(asum);
        if (lane == 1) sf = digamma_pos(asum);
        lg_asum = __shfl_sync(0xffffffffu, sf, 0);
        psi_as = __shfl_sync(0xffffffffu, sf, 1);
        if (lane != 0) return;
    } else {
        lg_asum = lgamma_ni(asum);
        psi_as = digamma_pos(asum);
    }
    ppi += st[L.lnc0];
    double qz = -st[L.stats + (int64_t)K * L.pitch + BGMM_STATS_ENTROPY];     // -sum r ln r (:704)
    qpi += -lg_asum + (asum - K) * psi_as;                                       // dirichlet entropy (:707)
    double extra = 0.0;
    if (hmm_vlx != nullptr) {      // hidden-Markov ELBO (_hiddenmarkovnormal.py:869-932): terms from hmm_trans_kernel
        pz = hmm_vlx[0];
        qz = hmm_vlx[2];
        extra = hmm_vlx[1] + hmm_vlx[3];
    }
    const double vl = px + pz + ppi + pml + qz + qpi + qml + extra;           // :717-723
    double* vt = st + L.vlterms;
    vt[0] = px; vt[1] = pz; vt[2] = ppi; vt[3] = pml; vt[4] = qz; vt[5] = qpi; vt[6] = qml; vt[7] = vl;
    const int iter = ctrl[BGMM_CTRL_ITER];
    double* hist = st + L.vlhist;
    if (iter < L.hist_len) hist[iter] = vl;
    bool conv = false;
    if (iter >= 1 && iter - 1 < L.hist_len) {
        const double vb = hist[iter - 1];
        conv = fabs((vl - vb) / vb) < tol;
    }
    if (conv) { ctrl[BGMM_CTRL_CONVERGED] = 1; ctrl[BGMM_CTRL_DONE] = 1; }
    else if (iter >= max_itr || ctrl[BGMM_CTRL_ERROR]) { ctrl[BGMM_CTRL_DONE] = 1; }   // error: queued launches become no-ops
    else { ctrl[BGMM_CTRL_CUR] = c.cur ^ 1; ctrl[BGMM_CTRL_ROBUST] = robust; ctrl[BGMM_CTRL_CRIT] = critq; }
    ctrl[BGMM_CTRL_ITER] = iter + 1;
    ctrl[BGMM_CTRL_TICKET] = 0;
}

__global__ void __launch_bounds__(256) small_kernel(double* __restrict__ st, const Layout L, const int mode,
                                                    const int max_itr, const double tol,
                                                    const CommDesc* __restrict__ cd,
                                                    const double* __restrict__ hmm_vlx, const double robust_thresh) {
    extern __shared__ double sm[];
    pdl_trigger();
    pdl_wait();
    const double* xb[BGMM_MAX_RANKS];
    SmallCtx c(st, L, L.D, mode, cd, xb);
    if (!c.begin()) return;
    const int D = L.D, DD = D * D, k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    double* A = sm;             // [D][D]  W^-1 -> L -> L^-1
    double* xbar = A + DD;      // [D]
    double* dev = xbar + D;     // [D]
    double* mnew = dev + D;     // [D]
    double* lin = mnew + D;     // [D]
    double* rdiag = lin + D;    // [D]  1 / L_jj
    double* ldiag = rdiag + D;  // [D]  L_jj
    double* scratch = ldiag + D;  // [48]: [0..33] block reductions, [34..37] special-function values
    const BlockTeam t(scratch);
    const BlockMats mats{st + L.smats + (int64_t)k * DD, A};
    if (c.fused) receive(t, c, cd);

    double N = 0.0, crit_n = 1.0;        // crit_n: weight of this component in the conditioning criterion, min(N_k, 1)
    double kn, nun, an, alpha_sum_new;
    if (c.iterate || c.stats_only) {
        N = component_stats(t, mats, c, xbar, lin);
        crit_n = fmin(N, 1.0);
        if (c.stats_only) return;
        const CurParams p = c.current();
        // the four special-function values of the ELBO terms, one per thread, while the loads of the traces are in flight
        double sf = 0.0;
        if (tid == 0) sf = log_ni(c.kappa0);
        else if (tid == 1) sf = log_ni(p.kappa);
        else if (tid == 2) sf = lgamma_ni(p.alpha);
        else if (tid == 3) sf = digamma_pos(p.alpha);
        if (tid < 4) scratch[34 + tid] = sf;
        const Traces tr = elbo_traces(t, mats, c, p, xbar, dev, lin);
        if (tid == 0) elbo_terms(c, N, p, tr, scratch[34], scratch[35], scratch[36], scratch[37]);
        alpha_sum_new = m_step(t, mats, c, N, xbar, mnew, dev, kn, nun, an);
    } else {
        alpha_sum_new = current_set(t, mats, c, mnew, kn, nun, an);
    }
    __syncthreads();

    // ---- Cholesky A = L L^T (lower, in place, right-looking).  Latency-bound: every thread forms 1/sqrt(a_jj) itself
    //      (no divide, no single-thread step), two barriers per column; rdiag keeps 1/L_jj for the inversion ----
    bool spd = true;
    for (int j = 0; j < D; ++j) {
        const double ajj = A[j * D + j];
        if (!(ajj > 0.0)) spd = false;
        const double rs = rsqrt(ajj);
        for (int i = j + 1 + tid; i < D; i += nt) A[i * D + j] *= rs;
        if (tid == 0) { rdiag[j] = rs; ldiag[j] = ajj * rs; }
        __syncthreads();
        const int rem = D - j - 1;
        for (int e = tid; e < rem * rem; e += nt) {
            const int i = j + 1 + e / rem, l = j + 1 + e % rem;
            if (l <= i) A[i * D + l] -= A[i * D + j] * A[l * D + j];
        }
        __syncthreads();
    }
    double ld = 0.0;
    for (int i = tid; i < D; i += nt) ld += log_ni(ldiag[i]);
    const double logdet = 2.0 * block_sum(ld, scratch);  // ln|W^-1|
    if (!spd && tid == 0) c.ctrl[BGMM_CTRL_ERROR] = 1;     // the finaliser below stops the loop

    // ---- L <- L^-1 in place (column sweep from the last column; lower triangular; 1/L_jj from rdiag) ----
    for (int j = D - 1; j >= 0; --j) {
        const double inv_jj = rdiag[j];
        // x = L[j+1:, j]; new x_i = -inv_jj * sum_{l=j+1..i} Linv[i][l] * x_l
        for (int i = j + 1 + tid; i < D; i += nt) lin[i] = A[i * D + j];
        __syncthreads();
        for (int i = j + 1 + tid; i < D; i += nt) {
            double acc = 0.0;
            for (int l = j + 1; l <= i; ++l) acc += A[i * D + l] * lin[l];
            A[i * D + j] = -inv_jj * acc;
        }
        if (tid == 0) A[j * D + j] = inv_jj;
        __syncthreads();
    }

    {   // L^-1 itself: the whitening operand of the fp32-mode tensor-core E-step (zero above the diagonal)
        double* Lo = c.Pn + L.p_linv + (int64_t)k * DD;
        for (int e = tid; e < DD; e += nt) Lo[e] = (e % D <= e / D) ? A[e] : 0.0;
    }
    // ---- W = L^-T L^-1 ----
    double* Wout = c.Pn + L.p_w + (int64_t)k * DD;
    for (int e = tid; e < DD; e += nt) {
        const int i = e / D, j = e - i * D;
        double acc = 0.0;
        for (int l = max(i, j); l < D; ++l) acc += A[l * D + i] * A[l * D + j];
        Wout[e] = acc;
    }

    double ps, gs;
    nu_sums(t, D, nun, ps, gs);
    const double elnpi_n = digamma_pos(an) - digamma_pos(alpha_sum_new);
    const double elndet_n = store_features(t, c, nun, ps, gs, logdet, elnpi_n);
    __syncthreads();  // Wout visible to the whole CTA

    // ---- the linear and quadratic parts of the coefficient row ----
    for (int i = tid; i < D; i += nt) {
        double acc = 0.0;
        for (int j = 0; j < D; ++j) acc += Wout[i * D + j] * mnew[j];
        lin[i] = nun * acc;
    }
    __syncthreads();
    double mq = 0.0;
    for (int i = tid; i < D; i += nt) mq += mnew[i] * lin[i];
    mq = block_sum(mq, scratch);
    store_row(t, c, hmm_vlx, elnpi_n, elndet_n, kn, mq, crit_n, xbar, mnew);
    double* coef = c.Pn + L.p_coef + (int64_t)k * L.pitch;
    for (int i = tid; i < D; i += nt) coef[1 + i] = lin[i];
    const int nq = D * (D + 1) / 2;
    for (int q = tid; q < nq; q += nt) {
        int i = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
        while (i * (i + 1) / 2 > q) --i;
        while ((i + 1) * (i + 2) / 2 <= q) ++i;
        const int j = q - i * (i + 1) / 2;
        coef[1 + D + q] = (i == j) ? -0.5 * nun * Wout[i * D + i] : -nun * Wout[i * D + j];
    }
    finish_iteration<1>(t, c, max_itr, tol, hmm_vlx, robust_thresh);
}

// ---- D <= 32: component k by ONE WARP, warp-synchronous throughout -------------------------------------------------------
// small_kernel's running time (~45 us at K = 32, D = 16) is a chain of block barriers and single-thread steps around a
// 16 x 16 factorisation; at 8 GPUs it is half of the per-iteration time that does not shrink with the shard (VERDICT r1,
// weak #5).  Here lane i owns row i (Cholesky, left-looking), then column i (L^-1 by forward substitution) and row i again
// (W = L^-T L^-1), everything in shared memory with conflict-free pitch 33 and __syncwarp only; the special functions are
// evaluated in merged SIMT calls (one digamma / lgamma / log call serves all lanes' different arguments) and the last CTA
// sums the ELBO with all 32 lanes.  The other stages are the shared ones above, run by a WarpTeam.
// DT > 0: D is the compile-time constant DT (the loops of the D x D algebra unroll completely: the warp is latency bound,
// ~9 cycles per instruction, and loop control was two thirds of its instruction stream — profiles/r02_small_warp_*);
// DT == 0: any D <= 32 at run time.
template <int DT>
__global__ void __launch_bounds__(32) small_warp_kernel(double* __restrict__ st, const Layout L, const int mode,
                                                        const int max_itr, const double tol,
                                                        const CommDesc* __restrict__ cd,
                                                        const double* __restrict__ hmm_vlx, const double robust_thresh) {
    __shared__ double Am[32 * SW_LP];        // W^-1 (lower triangle used) -> L -> W
    __shared__ double Bm[32 * SW_LP];        // S -> L^-1
    __shared__ double xbar[32], dev[32], lin[32], mnew[32], rd[32];
    pdl_trigger();
    pdl_wait();
    const double* xb[BGMM_MAX_RANKS];
    SmallCtx c(st, L, DT > 0 ? DT : L.D, mode, cd, xb);
    if (!c.begin()) return;
    const int D = c.D, DD = D * D, k = blockIdx.x, lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    const WarpTeam t;
    const WarpMats mats{Am, Bm};
    if (c.fused) receive(t, c, cd);

    double kn, nun, an, alpha_sum_new, N = 0.0, crit_n = 1.0;
    CurParams p;
    Traces tr;
    if (c.iterate || c.stats_only) {
        N = component_stats(t, mats, c, xbar, lin);
        crit_n = fmin(N, 1.0);
        if (c.stats_only) return;
        p = c.current();
        tr = elbo_traces(t, mats, c, p, xbar, dev, lin);
        alpha_sum_new = m_step(t, mats, c, N, xbar, mnew, dev, kn, nun, an);
    } else {
        alpha_sum_new = current_set(t, mats, c, mnew, kn, nun, an);
    }
    __syncwarp();
    // ---- Cholesky A = L L^T, left-looking: lane i owns row i; L[j][l] (l < j) is final when column j starts ----
    bool spd = true;
    double mydiag = 1.0;
#pragma unroll
    for (int j = 0; j < D; ++j) {
        double s0 = Am[lane * SW_LP + j], s1 = 0.0;
        int l = 0;
#pragma unroll
        for (; l + 1 < j; l += 2) {
            s0 = fma(-Am[lane * SW_LP + l], Am[j * SW_LP + l], s0);
            s1 = fma(-Am[lane * SW_LP + l + 1], Am[j * SW_LP + l + 1], s1);
        }
        if (l < j) s0 = fma(-Am[lane * SW_LP + l], Am[j * SW_LP + l], s0);
        const double s = s0 + s1;
        const double sjj = __shfl_sync(full, s, j);
        spd = spd && (sjj > 0.0);
        const double rs = rsqrt(sjj);
        const double v = (lane == j) ? sjj * rs : (lane > j ? s * rs : 0.0);
        __syncwarp();                          // every lane has read row j's entries before lane j overwrites A[j][j]
        Am[lane * SW_LP + j] = v;
        if (lane == j) { mydiag = v; rd[j] = rs; }
        __syncwarp();
    }
    const double ld = (lane < D) ? log_ni(mydiag) : 0.0;
    const double logdet = 2.0 * warp_sum(ld);  // ln|W^-1|
    if (!spd && lane == 0) c.ctrl[BGMM_CTRL_ERROR] = 1;

    // ---- L^-1 by forward substitution: lane j owns COLUMN j (B[i][j], i = 0..D-1); no cross-lane dependence ----
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double a0 = (i == lane) ? 1.0 : 0.0, a1 = 0.0;
        int l = 0;
#pragma unroll
        for (; l + 1 < i; l += 2) {
            a0 = fma(-Am[i * SW_LP + l], Bm[l * SW_LP + lane], a0);
            a1 = fma(-Am[i * SW_LP + l + 1], Bm[(l + 1) * SW_LP + lane], a1);
        }
        if (l < i) a0 = fma(-Am[i * SW_LP + l], Bm[l * SW_LP + lane], a0);
        Bm[i * SW_LP + lane] = (i >= lane && lane < D) ? (a0 + a1) * rd[i] : 0.0;
    }
    __syncwarp();
    {   // L^-1 itself: the whitening operand of the fp32-mode tensor-core E-step
        double* Lo = c.Pn + L.p_linv + (int64_t)k * DD;
        for (int e = lane; e < DD; e += 32) Lo[e] = Bm[(e / D) * SW_LP + (e % D)];
    }

    // ---- W = L^-T L^-1: lane a owns row a; W[a][b] = sum_{l >= max(a,b)} Linv[l][a] Linv[l][b] ----
#pragma unroll
    for (int b = 0; b < D; ++b) {
        double a0 = 0.0, a1 = 0.0;
        int l = b;
#pragma unroll
        for (; l + 1 < D; l += 2) {
            a0 = fma(Bm[l * SW_LP + lane], Bm[l * SW_LP + b], a0);
            a1 = fma(Bm[(l + 1) * SW_LP + lane], Bm[(l + 1) * SW_LP + b], a1);
        }
        if (l < D) a0 = fma(Bm[l * SW_LP + lane], Bm[l * SW_LP + b], a0);
        Am[lane * SW_LP + b] = a0 + a1;        // L is no longer needed
    }
    __syncwarp();
    double* Wout = c.Pn + L.p_w + (int64_t)k * DD;
    for (int e = lane; e < DD; e += 32) Wout[e] = Am[(e / D) * SW_LP + (e % D)];

    // ---- special functions, merged SIMT calls: lanes i < D take (nu - i)/2, three more lanes the scalar arguments ----
    double ps, gs, psi_x = 0.0, lg_x = 0.0, ln_x = 0.0;
    nu_sums(t, D, nun, ps, gs);
    {
        // lane 0: alpha_cur, lane 1: alpha_new, lane 2: sum alpha_new  (digamma);  lane 0: alpha_cur (lgamma);
        // lane 0: kappa0, lane 1: kappa_cur (log)
        const double pa = lane == 0 ? p.alpha : (lane == 1 ? an : alpha_sum_new);
        if (lane < 3) psi_x = digamma_pos(pa);
        if (lane == 0) lg_x = lgamma_ni(p.alpha);
        if (lane < 2) ln_x = log_ni(lane == 0 ? c.kappa0 : p.kappa);
    }
    const double psi_alpha = __shfl_sync(full, psi_x, 0), psi_an = __shfl_sync(full, psi_x, 1),
                 psi_asum = __shfl_sync(full, psi_x, 2), lg_alpha = __shfl_sync(full, lg_x, 0),
                 ln_kappa0 = __shfl_sync(full, ln_x, 0), ln_kappa = __shfl_sync(full, ln_x, 1);
    const double elnpi_n = psi_an - psi_asum;
    const double elndet_n = store_features(t, c, nun, ps, gs, logdet, elnpi_n);

    // ---- the linear and quadratic parts of the coefficient row ----
    double li = 0.0;
    if (lane < D) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < D; ++j) acc = fma(Am[lane * SW_LP + j], mnew[j], acc);
        li = nun * acc;
    }
    const double mq = warp_sum(lane < D ? mnew[lane] * li : 0.0);
    double* coef = c.Pn + L.p_coef + (int64_t)k * L.pitch;
    if (lane < D) {
        coef[1 + lane] = li;
        const int base = 1 + D + lane * (lane + 1) / 2;
        for (int j = 0; j < lane; ++j) coef[base + j] = -nun * Am[lane * SW_LP + j];
        coef[base + lane] = -0.5 * nun * Am[lane * SW_LP + lane];
    }
    if (c.iterate && lane == 0) elbo_terms(c, N, p, tr, ln_kappa0, ln_kappa, lg_alpha, psi_alpha);
    store_row(t, c, hmm_vlx, elnpi_n, elndet_n, kn, mq, crit_n, xbar, mnew);
    finish_iteration<32>(t, c, max_itr, tol, hmm_vlx, robust_thresh);
}

// Transition-matrix part of the hidden-Markov VB step, one CTA.  Replaces, in
// /root/reference/bayesml/hiddenmarkovnormal/_hiddenmarkovnormal.py:
//   _update_q_a :984-986 (zeta = zeta0 + M), _calc_q_a_features :851-854 (ln a~, a~ = exp(ln a~ - max), ln C(zeta)),
//   and the ELBO terms that involve A, xi, gamma_0 and the scaling constants: _vl_p_z :886, _vl_p_a :892,
//   _vl_q_z :906-909, _vl_q_a :915.
// It runs BEFORE small_kernel in every iteration: it reads ctrl.cur (small_kernel's finaliser flips it afterwards),
// evaluates the ELBO terms under the CURRENT set and writes the new set into the other slot.
__global__ void __launch_bounds__(256) hmm_trans_kernel(double* __restrict__ st, const Layout L, double* __restrict__ hst,
                                                        const HmmLayout H, const int mode) {
    __shared__ double red[40];
    __shared__ double rowsum[64];
    const int K = H.K, KK = K * K, tid = threadIdx.x, nt = blockDim.x;
    volatile int* ctrl = reinterpret_cast<volatile int*>(st + L.ctrl);
    const bool iterate = (mode == BGMM_SMALL_ITERATE);
    if (iterate && ctrl[BGMM_CTRL_DONE]) return;
    const int cur = ctrl[BGMM_CTRL_CUR];
    double* Sc = hst + H.set[cur];
    double* Sn = iterate ? hst + H.set[cur ^ 1] : Sc;
    if (iterate) {
        const double* Pc = st + L.params[cur];
        const double* ms = hst + H.ms;
        const double* zeta0 = hst + H.zeta0;
        const double amax = Sc[H.s_misc + 0], lncz = Sc[H.s_misc + 1];
        double pmax = -INFINITY;
        for (int k = 0; k < K; ++k) pmax = fmax(pmax, Pc[L.p_elnpi + k]);
        double t_pz = 0.0, t_pa = 0.0, t_qz = 0.0, t_qa = 0.0;
        for (int e = tid; e < KK; e += nt) {
            const double la = Sc[H.s_lna + e], m = ms[e];
            t_pz += m * la;
            t_pa += (zeta0[e] - 1.0) * la;
            t_qz += m * (la - amax);
            t_qa += (Sc[H.s_zeta + e] - 1.0) * la;
        }
        for (int k = tid; k < K; k += nt) {
            const double g0 = hst[H.g0 + k], lp = Pc[L.p_elnpi + k];
            t_pz += g0 * lp;
            t_qz += g0 * (lp - pmax);
        }
        block_sum4(t_pz, t_pa, t_qz, t_qa, red);
        if (tid == 0) {
            double* vlx = hst + H.vlx;
            vlx[0] = t_pz;
            vlx[1] = hst[H.lncz0] + t_pa;
            vlx[2] = -hst[H.sc + 1] - t_qz + hst[H.sc + 0];
            vlx[3] = -lncz - t_qa;
        }
        __syncthreads();
        for (int e = tid; e < KK; e += nt) Sn[H.s_zeta + e] = zeta0[e] + ms[e];
        __syncthreads();
    }
    // features of the (new) set
    for (int r = tid; r < K; r += nt) {
        double s = 0.0;
        for (int k = 0; k < K; ++k) s += Sn[H.s_zeta + r * K + k];
        rowsum[r] = s;
    }
    __syncthreads();
    double mx = -INFINITY, lc = 0.0;
    for (int e = tid; e < KK; e += nt) {
        const int r = e / K;
        const double z = Sn[H.s_zeta + e];
        const double la = digamma_pos(z) - digamma_pos(rowsum[r]);
        Sn[H.s_lna + e] = la;
        mx = fmax(mx, la);
        lc -= lgamma_ni(z);
    }
    for (int r = tid; r < K; r += nt) lc += lgamma_ni(rowsum[r]);
    mx = block_max(mx, red);
    lc = block_sum(lc, red);
    for (int e = tid; e < KK; e += nt) Sn[H.s_at + e] = exp(Sn[H.s_lna + e] - mx);
    // Projective (Hilbert-metric) diameter of A~: Delta = max_{j,j'} [max_k d_k - min_k d_k], d_k = ln a~_jk - ln a~_j'k.
    // Every forward / backward step contracts the Hilbert distance between two message vectors by tau = tanh(Delta / 4)
    // (Birkhoff), whatever the emission values (diagonal scalings leave the metric unchanged); the scan kernels use
    // ln tau and ln Delta to decide whether a chunk is long enough to forget its boundary vector (bgmm_hmm.cu).
    double dl = 0.0;
    for (int pr = tid; pr < KK; pr += nt) {
        const int j = pr / K, j2 = pr - j * K;
        if (j2 <= j) continue;
        double hi = -INFINITY, lo = INFINITY;
        for (int k = 0; k < K; ++k) {
            const double d = Sn[H.s_lna + j * K + k] - Sn[H.s_lna + j2 * K + k];
            hi = fmax(hi, d);
            lo = fmin(lo, d);
        }
        dl = fmax(dl, hi - lo);
    }
    dl = block_max(dl, red);
    if (tid == 0) {
        Sn[H.s_misc + 0] = mx;
        Sn[H.s_misc + 1] = lc;
        Sn[H.s_misc + 2] = log1p(-2.0 / (exp(0.5 * dl) + 1.0));      // ln tanh(Delta / 4)
        Sn[H.s_misc + 3] = log_ni(dl);                                // ln Delta (-inf when A~ is exactly uniform)
    }
}

// small_kernel's shared memory: the [D][D] matrix, six D-vectors and 48 doubles of scratch
static size_t small_smem_bytes(int D) { return sizeof(double) * ((size_t)D * D + 6 * (size_t)D + 48); }

static int check_small_smem(const char* who, int D) {
    if (small_smem_bytes(D) <= 227 * 1024) return BGMM_OK;
    set_error("%s: D=%d needs %zu B of shared memory (> 227 KiB)", who, D, small_smem_bytes(D));
    return BGMM_ENOSUP;
}

// One bgmm_small step for entry point `who`: small_warp_kernel<DT> for D <= 32, else small_kernel with 128 threads up to
// D = 64 and 256 above.
static int launch_small(const char* who, int K, int D, double* state, const Layout& L, int mode, int max_itr, double tol,
                        const CommDesc* cd, const double* hmm_vlx, cudaStream_t stream) {
    if (int rc = check_small_smem(who, D)) return rc;
    const size_t smem = small_smem_bytes(D);
    const double thr = robust_threshold();
    const char* what = "cudaFuncSetAttribute(small_kernel)";
    cudaError_t e = cudaSuccess;
    if (smem > 48 * 1024)     // per launch: the attribute is per device
        e = cudaFuncSetAttribute(small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && D <= 32) {
        what = "small_warp_kernel launch";
        auto kern = D == 2 ? small_warp_kernel<2> : D == 4 ? small_warp_kernel<4> : D == 8 ? small_warp_kernel<8>
                  : D == 16 ? small_warp_kernel<16> : small_warp_kernel<0>;
        e = launch_pdl(kern, dim3(K), dim3(32), 0, stream, state, L, mode, max_itr, tol, cd, hmm_vlx, thr);
    } else if (e == cudaSuccess) {
        what = "small_kernel launch";
        e = launch_pdl(small_kernel, dim3(K), dim3(D <= 64 ? 128 : 256), smem, stream, state, L, mode, max_itr, tol, cd,
                       hmm_vlx, thr);
    }
    if (e == cudaSuccess) return BGMM_OK;
    set_error("%s: %s: %s", who, what, cudaGetErrorString(e));
    return BGMM_ECUDA;
}

}  // namespace bgmm

extern "C" int bgmm_hmm_layout(int K, int64_t* off) {
    using namespace bgmm;
    if (K <= 0 || off == nullptr) { set_error("bgmm_hmm_layout: bad argument"); return BGMM_EINVAL; }
    const HmmLayout H = make_hmm_layout(K);
    const int64_t v[BGMM_HMM_OFF_COUNT] = {H.zeta0, H.lncz0, H.set[0], H.set[1], H.s_zeta, H.s_lna, H.s_at, H.s_misc,
                                           H.ms, H.g0, H.sc, H.vlx, H.total};
    for (int i = 0; i < BGMM_HMM_OFF_COUNT; ++i) off[i] = v[i];
    return BGMM_OK;
}

extern "C" int bgmm_hmm_small(int K, int D, double* state, double* hst, int mode, int max_itr, double tol, int hist_len,
                              void* stream) {
    using namespace bgmm;
    if (K <= 0 || K > 64 || D <= 0 || state == nullptr || hst == nullptr || hist_len < 1) {
        set_error("bgmm_hmm_small: bad argument (K=%d D=%d state=%p hst=%p hist_len=%d)", K, D, (void*)state, (void*)hst,
                  hist_len);
        return BGMM_EINVAL;
    }
    if (mode != BGMM_SMALL_FEATURES && mode != BGMM_SMALL_ITERATE && mode != BGMM_SMALL_STATS) {
        set_error("bgmm_hmm_small: unknown mode %d", mode);
        return BGMM_EINVAL;
    }
    // launch_small checks this again; here it has to come before hmm_trans_kernel changes the state
    if (int rc = check_small_smem("bgmm_hmm_small", D)) return rc;
    const Layout L = make_layout(K, D, hist_len);
    const HmmLayout H = make_hmm_layout(K);
    if (mode != BGMM_SMALL_STATS) {
        int rc = check_cuda(launch(hmm_trans_kernel, 1, 256, 0, (cudaStream_t)stream, state, L, hst, H, mode),
                            "bgmm_hmm_small: hmm_trans_kernel launch");
        if (rc) return rc;
    }
    return launch_small("bgmm_hmm_small", K, D, state, L, mode, max_itr, tol, nullptr, hst + H.vlx, (cudaStream_t)stream);
}

extern "C" int bgmm_small(int K, int D, double* state, int mode, int max_itr, double tol, int hist_len,
                          const void* comm_desc, void* stream) {
    using namespace bgmm;
    if (K <= 0 || D <= 0 || state == nullptr || hist_len < 1) {
        set_error("bgmm_small: bad argument (K=%d D=%d state=%p hist_len=%d)", K, D, (void*)state, hist_len);
        return BGMM_EINVAL;
    }
    if (mode != BGMM_SMALL_FEATURES && mode != BGMM_SMALL_ITERATE && mode != BGMM_SMALL_STATS) {
        set_error("bgmm_small: unknown mode %d", mode);
        return BGMM_EINVAL;
    }
    return launch_small("bgmm_small", K, D, state, make_layout(K, D, hist_len), mode, max_itr, tol,
                        static_cast<const CommDesc*>(comm_desc), nullptr, (cudaStream_t)stream);
}
