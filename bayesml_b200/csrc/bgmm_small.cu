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

__global__ void __launch_bounds__(256) small_kernel(double* __restrict__ st, const Layout L, const int mode,
                                                    const int max_itr, const double tol,
                                                    const CommDesc* __restrict__ cd,
                                                    const double* __restrict__ hmm_vlx, const double robust_thresh) {
    extern __shared__ double sm[];
    pdl_trigger();
    pdl_wait();
    const int K = L.K, D = L.D, DD = D * D, k = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    volatile int* ctrl = reinterpret_cast<volatile int*>(st + L.ctrl);
    const bool iterate = (mode == BGMM_SMALL_ITERATE), stats_only = (mode == BGMM_SMALL_STATS);
    if (iterate && ctrl[BGMM_CTRL_DONE]) return;  // every CTA reads this before any CTA can take the last ticket
    const int cur = ctrl[BGMM_CTRL_CUR];
    double* Pc = st + L.params[cur];
    double* Pn = iterate ? st + L.params[cur ^ 1] : Pc;

    double* A = sm;             // [D][D]  W^-1 -> L -> L^-1
    double* xbar = A + DD;      // [D]
    double* dev = xbar + D;     // [D]
    double* mnew = dev + D;     // [D]
    double* lin = mnew + D;     // [D]
    double* rdiag = lin + D;    // [D]  1 / L_jj
    double* ldiag = rdiag + D;  // [D]  L_jj
    double* scratch = ldiag + D;  // [48]: [0..33] block reductions, [34..37] special-function values

    const double* center = st + L.center;
    const double* m0 = st + L.m0 + (int64_t)k * D;
    const double* w0inv = st + L.w0inv + (int64_t)k * DD;
    const double alpha0 = st[L.alpha0 + k], kappa0 = st[L.kappa0 + k], nu0 = st[L.nu0 + k];

    double kn, nun, an, alpha_sum_new;

    // ---- fused all-reduce over peer memory: wait for every rank's stamp, sum the published blocks in rank order ----
    const bool fused = (cd != nullptr) && (iterate || stats_only);
    const double* xb[BGMM_MAX_RANKS];
    int world = 1;
    if (fused) {
        world = cd->world;
        const int seq = ctrl[BGMM_CTRL_SEQ] - 1;                // the exchange published by the preceding bgmm_pass
        const int64_t len = L.stats_len;
        if (tid < world) {
            const unsigned long long* flag = reinterpret_cast<const unsigned long long*>(cd->xchg[cd->rank] + 2 * len) +
                                             (seq & 1) * BGMM_MAX_RANKS + tid;
            unsigned long long v;
            do {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
            } while (v < (unsigned long long)(seq + 1));
        }
        __syncthreads();
        for (int r = 0; r < world; ++r) xb[r] = cd->xchg[r] + (int64_t)(seq & 1) * len;
        double* row = st + L.stats + (int64_t)k * L.pitch;      // this CTA owns row k of the reduced statistics
        for (int p = tid; p < L.pitch; p += nt) {
            double acc = 0.0;
            for (int r = 0; r < world; ++r) acc += ld_peer(xb[r] + (int64_t)k * L.pitch + p);
            row[p] = acc;
        }
        if (k == 0 && tid < 8) {
            double acc = 0.0;
            for (int r = 0; r < world; ++r) acc += ld_peer(xb[r] + (int64_t)K * L.pitch + tid);
            st[L.stats + (int64_t)K * L.pitch + tid] = acc;
        }
        __syncthreads();
    }

    double crit_n = 1.0;                 // weight of this component in the conditioning criterion: min(N_k, 1)
    if (iterate || stats_only) {
        // ---- statistics of component k from the moments about the centre (feature-map kernels) or about
        //      shift_k (DIRECT kernel; format slot > 0):  x_bar = shift + d_bar,  S = M2 / N - d_bar d_bar^T ----
        const double* raw = st + L.stats + (int64_t)k * L.pitch;
        const double N = raw[0];
        crit_n = fmin(N, 1.0);
        double fmt;
        if (fused) {                                            // CTA 0 owns the tail: sum the format marker from the peers
            fmt = 0.0;
            for (int r = 0; r < world; ++r) fmt += ld_peer(xb[r] + (int64_t)K * L.pitch + BGMM_STATS_FORMAT);
        } else {
            fmt = st[L.stats + (int64_t)K * L.pitch + BGMM_STATS_FORMAT];
        }
        const bool shifted = fmt > 0.5;
        const double* sh = st + L.shift + (int64_t)k * D;
        double* S = st + L.smats + (int64_t)k * DD;
        if (N > 0.0) {
            const double invN = 1.0 / N;
            for (int i = tid; i < D; i += nt) {
                const double db = raw[1 + i] * invN;
                lin[i] = db;
                xbar[i] = shifted ? sh[i] + db : db;
            }
            __syncthreads();
            for (int e = tid; e < DD; e += nt) {
                const int i = e / D, j = e - i * D, hi = max(i, j), lo = min(i, j);
                S[e] = raw[1 + D + hi * (hi + 1) / 2 + lo] * invN - lin[i] * lin[j];
            }
        } else {
            // reference :729 — x_bar_vecs[k] keeps the un-normalised sum (0 in the original frame), s_mats[k] stale
            for (int i = tid; i < D; i += nt) xbar[i] = -center[i];
        }
        __syncthreads();
        for (int i = tid; i < D; i += nt) st[L.xbar + (int64_t)k * D + i] = xbar[i];
        if (tid == 0) st[L.ns + k] = N;
        if (stats_only) {
            // x_bar_k becomes the shift of a following centred-statistics sweep (engine.refine_smats: the reference's
            // two-pass s_mats, :730-732, from the materialised responsibilities)
            if (N > 0.0)
                for (int i = tid; i < D; i += nt) st[L.shift + (int64_t)k * D + i] = xbar[i];
            return;
        }

        // ---- ELBO terms of component k under the CURRENT parameters (those the pass used) ----
        const double kappa = Pc[L.p_kappa + k], nu = Pc[L.p_nu + k], alpha = Pc[L.p_alpha + k];
        const double elnpi = Pc[L.p_elnpi + k], elndet = Pc[L.p_elndet + k], lnb = Pc[L.p_lnb + k];
        const double* W = Pc + L.p_w + (int64_t)k * DD;
        const double* m = Pc + L.p_m + (int64_t)k * D;
        // the deviations (x_bar - m), (m - m0) go to shared memory first so the D x D loop only streams W and W0^-1
        for (int i = tid; i < D; i += nt) { dev[i] = xbar[i] - m[i]; lin[i] = m[i] - m0[i]; }
        // the four special-function values of the ELBO terms, one per lane, while the loads of the loop are in flight
        double sf = 0.0;
        if (tid == 0) sf = log_ni(kappa0);
        else if (tid == 1) sf = log_ni(kappa);
        else if (tid == 2) sf = lgamma_ni(alpha);
        else if (tid == 3) sf = digamma_pos(alpha);
        if (tid < 4) scratch[34 + tid] = sf;
        __syncthreads();
        double t_trs = 0.0, t_q1 = 0.0, t_q2 = 0.0, t_tr0 = 0.0;
#pragma unroll 4
        for (int e = tid; e < DD; e += nt) {
            const int i = e / D, j = e - i * D;
            const double w = W[e];
            t_trs += S[e] * w;
            t_q1 += dev[i] * w * dev[j];
            t_q2 += lin[i] * w * lin[j];
            t_tr0 += w0inv[e] * w;
        }
        block_sum4(t_trs, t_q1, t_q2, t_tr0, scratch);
        if (tid == 0) {
            double* vk = st + L.vlk + (int64_t)k * 8;
            const double lnb0 = st[L.lnb0 + k];
            const double ln_kappa0 = scratch[34], ln_kappa = scratch[35], lg_alpha = scratch[36], psi_alpha = scratch[37];
            vk[0] = N * (elndet - D / kappa - nu * t_trs - nu * t_q1 - D * LN2PI) / 2.0;          // :673-683
            vk[1] = N * elnpi;                                                                     // :686
            vk[2] = (alpha0 - 1.0) * elnpi;                                                        // :689
            vk[3] = (D * (ln_kappa0 - LN2PI - kappa0 / kappa) - kappa0 * nu * t_q2 + 2.0 * lnb0
                     + (nu0 - D) * elndet - nu * t_tr0) / 2.0;                                     // :692-701
            vk[4] = lg_alpha - (alpha - 1.0) * psi_alpha;                                          // :707 (per-k part)
            vk[5] = (D * (1.0 + LN2PI - ln_kappa) - 2.0 * lnb - (nu - D) * elndet + nu * D) / 2.0;  // :710-715
            vk[6] = alpha;
            vk[7] = 0.0;
        }
        __syncthreads();       // dev / lin are reused by the M-step below

        // ---- M-step (:758-768, :742) into the other parameter set ----
        kn = kappa0 + N; nun = nu0 + N; an = alpha0 + N;
        for (int i = tid; i < D; i += nt) {
            mnew[i] = (kappa0 * m0[i] + N * xbar[i]) / kn;
            dev[i] = xbar[i] - m0[i];
        }
        __syncthreads();
        const double c2 = kappa0 * N / kn;
        double* winv_out = Pn + L.p_winv + (int64_t)k * DD;
        for (int e = tid; e < DD; e += nt) {
            const int i = e / D, j = e - i * D;
            const double v = w0inv[e] + N * S[e] + c2 * (dev[i] * dev[j]);
            A[e] = v;
            winv_out[e] = v;
        }
        double asum = 0.0;
        for (int j = tid; j < K; j += nt) {
            double nj;
            if (fused) {                                        // other CTAs own the other rows: sum N_j from the peers
                nj = 0.0;
                for (int r = 0; r < world; ++r) nj += ld_peer(xb[r] + (int64_t)j * L.pitch);
            } else {
                nj = st[L.stats + (int64_t)j * L.pitch];
            }
            asum += st[L.alpha0 + j] + nj;
        }
        alpha_sum_new = block_sum(asum, scratch);
        if (tid == 0) { Pn[L.p_kappa + k] = kn; Pn[L.p_nu + k] = nun; Pn[L.p_alpha + k] = an; }
        for (int i = tid; i < D; i += nt) Pn[L.p_m + (int64_t)k * D + i] = mnew[i];
    } else {
        kn = Pc[L.p_kappa + k]; nun = Pc[L.p_nu + k]; an = Pc[L.p_alpha + k];
        for (int i = tid; i < D; i += nt) mnew[i] = Pc[L.p_m + (int64_t)k * D + i];
        for (int e = tid; e < DD; e += nt) A[e] = Pc[L.p_winv + (int64_t)k * DD + e];
        double asum = 0.0;
        for (int j = tid; j < K; j += nt) asum += Pc[L.p_alpha + j];
        alpha_sum_new = block_sum(asum, scratch);
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
    if (!spd && tid == 0) ctrl[BGMM_CTRL_ERROR] = 1;       // the finaliser below stops the loop

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
        double* Lo = Pn + L.p_linv + (int64_t)k * DD;
        for (int e = tid; e < DD; e += nt) Lo[e] = (e % D <= e / D) ? A[e] : 0.0;
    }
    // ---- W = L^-T L^-1 ----
    double* Wout = Pn + L.p_w + (int64_t)k * DD;
    for (int e = tid; e < DD; e += nt) {
        const int i = e / D, j = e - i * D;
        double acc = 0.0;
        for (int l = max(i, j); l < D; ++l) acc += A[l * D + i] * A[l * D + j];
        Wout[e] = acc;
    }

    // ---- features (:738-739, :745-756) ----
    double ps = 0.0, gs = 0.0;
    for (int i = tid; i < D; i += nt) {
        const double a = (nun - i) / 2.0;
        ps += digamma_pos(a);
        gs += lgamma_ni(a);
    }
    ps = block_sum(ps, scratch);
    gs = block_sum(gs, scratch);
    const double elndet_n = ps + D * LN2 - logdet;
    const double lnb_n = (nun * logdet - nun * D * LN2 - D * (D - 1) / 2.0 * LNPI - gs * 2.0) / 2.0;
    const double elnpi_n = digamma_pos(an) - digamma_pos(alpha_sum_new);
    if (tid == 0) {
        Pn[L.p_elndet + k] = elndet_n;
        Pn[L.p_lnb + k] = lnb_n;
        Pn[L.p_elnpi + k] = elnpi_n;
    }
    __syncthreads();  // Wout visible to the whole CTA

    // ---- E-step coefficient row: ln rho = coef . phi(x'), Lambda = nu W ----
    for (int i = tid; i < D; i += nt) {
        double acc = 0.0;
        for (int j = 0; j < D; ++j) acc += Wout[i * D + j] * mnew[j];
        lin[i] = nun * acc;
    }
    __syncthreads();
    double mq = 0.0;
    for (int i = tid; i < D; i += nt) mq += mnew[i] * lin[i];
    mq = block_sum(mq, scratch);
    double* coef = Pn + L.p_coef + (int64_t)k * L.pitch;
    // hidden-Markov emission density (_hiddenmarkovnormal.py:988-992): no E[ln pi] term in ln rho
    if (tid == 0) {
        const double acst = (hmm_vlx != nullptr ? 0.0 : elnpi_n) + (elndet_n - D * LN2PI - D / kn) / 2.0;
        coef[0] = acst - 0.5 * mq;
        Pn[L.p_acst + k] = acst;                                // ln rho constant of the DIRECT form (no m^T Lambda m term)
        // conditioning of the feature-map form for this component: the terms of coef . phi(x') are of size
        // mq = m'^T Lambda m' for the samples the component is responsible for, the result is O(D)
        // (K = 1: r == 1 exactly whatever ln rho is, and the moments about the global centre ARE the centred ones)
        st[L.vlk + (int64_t)k * 8 + 7] = (K == 1) ? 0.0 : crit_n * mq;
    }
    // the point the DIRECT kernel takes the next moments about: this pass's x_bar_k (the next one will be close), or the
    // new m_k while the component has no statistics yet
    if (!stats_only) {
        double* sh = st + L.shift + (int64_t)k * D;
        const bool have_xbar = iterate && crit_n > 0.0;
        for (int i = tid; i < D; i += nt) sh[i] = have_xbar ? xbar[i] : mnew[i];
    }
    for (int i = tid; i < D; i += nt) coef[1 + i] = lin[i];
    const int nq = D * (D + 1) / 2;
    for (int q = tid; q < nq; q += nt) {
        int i = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
        while (i * (i + 1) / 2 > q) --i;
        while ((i + 1) * (i + 2) / 2 <= q) ++i;
        const int j = q - i * (i + 1) / 2;
        coef[1 + D + q] = (i == j) ? -0.5 * nun * Wout[i * D + i] : -nun * Wout[i * D + j];
    }
    for (int q = L.P + tid; q < L.pitch; q += nt) coef[q] = 0.0;

    // ---- last CTA: conditioning flag of the new parameter set; sum the ELBO, convergence test (:869), flip the sets ----
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const int t = atomicAdd(const_cast<int*>(&ctrl[BGMM_CTRL_TICKET]), 1);
        is_last = (t == K - 1);
    }
    __syncthreads();
    if (!is_last || tid != 0) return;
    __threadfence();
    volatile const double* vk = st + L.vlk;
    double crit = 0.0;
    for (int j = 0; j < K; ++j) crit = fmax(crit, vk[j * 8 + 7]);
    const int robust = crit > robust_thresh ? 1 : 0;
    const int critq = crit < 1073741824.0 ? (int)ceil(crit) : 1073741824;     // NaN -> the large value
    if (!iterate) {
        ctrl[BGMM_CTRL_ROBUST] = robust;
        ctrl[BGMM_CTRL_CRIT] = critq;
        ctrl[BGMM_CTRL_TICKET] = 0;
        return;
    }
    double px = 0, pz = 0, ppi = 0, pml = 0, qpi = 0, qml = 0, asum = 0;
    for (int j = 0; j < K; ++j) {
        px += vk[j * 8 + 0]; pz += vk[j * 8 + 1]; ppi += vk[j * 8 + 2]; pml += vk[j * 8 + 3];
        qpi += vk[j * 8 + 4]; qml += vk[j * 8 + 5]; asum += vk[j * 8 + 6];
    }
    ppi += st[L.lnc0];
    double qz = -st[L.stats + (int64_t)K * L.pitch + BGMM_STATS_ENTROPY];     // -sum r ln r (:704)
    qpi += -lgamma_ni(asum) + (asum - K) * digamma_pos(asum);                    // dirichlet entropy (:707)
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
    else { ctrl[BGMM_CTRL_CUR] = cur ^ 1; ctrl[BGMM_CTRL_ROBUST] = robust; ctrl[BGMM_CTRL_CRIT] = critq; }
    ctrl[BGMM_CTRL_ITER] = iter + 1;
    ctrl[BGMM_CTRL_TICKET] = 0;
}

// ---- D <= 32: the same computation as small_kernel by ONE WARP per component, warp-synchronous throughout -------------
// small_kernel's running time (~45 us at K = 32, D = 16) is a chain of block barriers and single-thread steps around a
// 16 x 16 factorisation; at 8 GPUs it is half of the per-iteration time that does not shrink with the shard (VERDICT r1,
// weak #5).  Here lane i owns row i (Cholesky, left-looking), then column i (L^-1 by forward substitution) and row i again
// (W = L^-T L^-1), everything in shared memory with conflict-free pitch 33 and __syncwarp only; the special functions are
// evaluated in merged SIMT calls (one digamma / lgamma / log call serves all lanes' different arguments) and the last CTA
// sums the ELBO with all 32 lanes.  Same formulas, same outputs and control flow as small_kernel (which stays for D > 32).
// DT > 0: D is the compile-time constant DT (the loops of the D x D algebra unroll completely: the warp is latency bound,
// ~9 cycles per instruction, and loop control was two thirds of its instruction stream — profiles/r02_small_warp_*);
// DT == 0: any D <= 32 at run time.
constexpr int SW_LP = 33;

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
    const int K = L.K, D = DT > 0 ? DT : L.D, DD = D * D, k = blockIdx.x, lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    volatile int* ctrl = reinterpret_cast<volatile int*>(st + L.ctrl);
    const bool iterate = (mode == BGMM_SMALL_ITERATE), stats_only = (mode == BGMM_SMALL_STATS);
    if (iterate && ctrl[BGMM_CTRL_DONE]) return;
    const int cur = ctrl[BGMM_CTRL_CUR];
    double* Pc = st + L.params[cur];
    double* Pn = iterate ? st + L.params[cur ^ 1] : Pc;
    const double* center = st + L.center;
    const double* m0 = st + L.m0 + (int64_t)k * D;
    const double* w0inv = st + L.w0inv + (int64_t)k * DD;
    const double alpha0 = st[L.alpha0 + k], kappa0 = st[L.kappa0 + k], nu0 = st[L.nu0 + k];

    // ---- fused all-reduce over peer memory (as in small_kernel) ----
    const bool fused = (cd != nullptr) && (iterate || stats_only);
    const double* xb[BGMM_MAX_RANKS];
    int world = 1;
    if (fused) {
        world = cd->world;
        const int seq = ctrl[BGMM_CTRL_SEQ] - 1;
        const int64_t len = L.stats_len;
        if (lane < world) {
            const unsigned long long* flag = reinterpret_cast<const unsigned long long*>(cd->xchg[cd->rank] + 2 * len) +
                                             (seq & 1) * BGMM_MAX_RANKS + lane;
            unsigned long long v;
            do {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
            } while (v < (unsigned long long)(seq + 1));
        }
        __syncwarp();
        for (int r = 0; r < world; ++r) xb[r] = cd->xchg[r] + (int64_t)(seq & 1) * len;
        double* row = st + L.stats + (int64_t)k * L.pitch;
        for (int p = lane; p < L.pitch; p += 32) {
            double acc = 0.0;
            for (int r = 0; r < world; ++r) acc += ld_peer(xb[r] + (int64_t)k * L.pitch + p);
            row[p] = acc;
        }
        if (k == 0 && lane < 8) {
            double acc = 0.0;
            for (int r = 0; r < world; ++r) acc += ld_peer(xb[r] + (int64_t)K * L.pitch + lane);
            st[L.stats + (int64_t)K * L.pitch + lane] = acc;
        }
        __syncwarp();
    }

    double kn, nun, an, alpha_sum_new, N = 0.0, crit_n = 1.0;
    double t_trs = 0.0, t_q1 = 0.0, t_q2 = 0.0, t_tr0 = 0.0;
    double kappa_c = 1.0, nu_c = 0.0, alpha_c = 1.0, elnpi_c = 0.0, elndet_c = 0.0, lnb_c = 0.0;
    if (iterate || stats_only) {
        // ---- statistics of component k (moments about the centre, or about shift_k when the format slot is > 0) ----
        const double* raw = st + L.stats + (int64_t)k * L.pitch;
        N = raw[0];
        crit_n = fmin(N, 1.0);
        double fmt;
        if (fused) {
            fmt = 0.0;
            for (int r = 0; r < world; ++r) fmt += ld_peer(xb[r] + (int64_t)K * L.pitch + BGMM_STATS_FORMAT);
        } else {
            fmt = st[L.stats + (int64_t)K * L.pitch + BGMM_STATS_FORMAT];
        }
        const bool shifted = fmt > 0.5;
        const double* sh = st + L.shift + (int64_t)k * D;
        double* S = st + L.smats + (int64_t)k * DD;
        if (N > 0.0) {
            const double invN = 1.0 / N;
            if (lane < D) {
                const double db = raw[1 + lane] * invN;
                lin[lane] = db;
                xbar[lane] = shifted ? sh[lane] + db : db;
            }
            __syncwarp();
            for (int e = lane; e < DD; e += 32) {
                const int i = e / D, j = e - i * D, hi = max(i, j), lo = min(i, j);
                const double v = raw[1 + D + hi * (hi + 1) / 2 + lo] * invN - lin[i] * lin[j];
                S[e] = v;
                Bm[i * SW_LP + j] = v;
            }
        } else {
            // reference :729 — x_bar_vecs[k] keeps the un-normalised sum (0 in the original frame), s_mats[k] stale
            if (lane < D) xbar[lane] = -center[lane];
            for (int e = lane; e < DD; e += 32) Bm[(e / D) * SW_LP + (e % D)] = S[e];
        }
        __syncwarp();
        if (lane < D) st[L.xbar + (int64_t)k * D + lane] = xbar[lane];
        if (lane == 0) st[L.ns + k] = N;
        if (stats_only) {
            if (N > 0.0 && lane < D) st[L.shift + (int64_t)k * D + lane] = xbar[lane];
            return;
        }
        // ---- ELBO sums of component k under the CURRENT parameters (those the pass used) ----
        kappa_c = Pc[L.p_kappa + k]; nu_c = Pc[L.p_nu + k]; alpha_c = Pc[L.p_alpha + k];
        elnpi_c = Pc[L.p_elnpi + k]; elndet_c = Pc[L.p_elndet + k]; lnb_c = Pc[L.p_lnb + k];
        const double* W = Pc + L.p_w + (int64_t)k * DD;
        const double* m = Pc + L.p_m + (int64_t)k * D;
        if (lane < D) { dev[lane] = xbar[lane] - m[lane]; lin[lane] = m[lane] - m0[lane]; }
        __syncwarp();
        for (int e = lane; e < DD; e += 32) {
            const int i = e / D, j = e - i * D;
            const double w = W[e];
            t_trs += Bm[i * SW_LP + j] * w;
            t_q1 += dev[i] * w * dev[j];
            t_q2 += lin[i] * w * lin[j];
            t_tr0 += w0inv[e] * w;
        }
        t_trs = warp_sum(t_trs); t_q1 = warp_sum(t_q1); t_q2 = warp_sum(t_q2); t_tr0 = warp_sum(t_tr0);
        __syncwarp();       // dev / lin are reused below

        // ---- M-step (:758-768, :742) into the other parameter set ----
        kn = kappa0 + N; nun = nu0 + N; an = alpha0 + N;
        if (lane < D) {
            mnew[lane] = (kappa0 * m0[lane] + N * xbar[lane]) / kn;
            dev[lane] = xbar[lane] - m0[lane];
        }
        __syncwarp();
        const double c2 = kappa0 * N / kn;
        double* winv_out = Pn + L.p_winv + (int64_t)k * DD;
        for (int e = lane; e < DD; e += 32) {
            const int i = e / D, j = e - i * D;
            const double v = w0inv[e] + N * Bm[i * SW_LP + j] + c2 * (dev[i] * dev[j]);
            Am[i * SW_LP + j] = v;
            winv_out[e] = v;
        }
        double asum = 0.0;
        for (int j = lane; j < K; j += 32) {
            double nj;
            if (fused) {
                nj = 0.0;
                for (int r = 0; r < world; ++r) nj += ld_peer(xb[r] + (int64_t)j * L.pitch);
            } else {
                nj = st[L.stats + (int64_t)j * L.pitch];
            }
            asum += st[L.alpha0 + j] + nj;
        }
        alpha_sum_new = warp_sum(asum);
        if (lane == 0) { Pn[L.p_kappa + k] = kn; Pn[L.p_nu + k] = nun; Pn[L.p_alpha + k] = an; }
        if (lane < D) Pn[L.p_m + (int64_t)k * D + lane] = mnew[lane];
    } else {
        kn = Pc[L.p_kappa + k]; nun = Pc[L.p_nu + k]; an = Pc[L.p_alpha + k];
        if (lane < D) mnew[lane] = Pc[L.p_m + (int64_t)k * D + lane];
        for (int e = lane; e < DD; e += 32) Am[(e / D) * SW_LP + (e % D)] = Pc[L.p_winv + (int64_t)k * DD + e];
        double asum = 0.0;
        for (int j = lane; j < K; j += 32) asum += Pc[L.p_alpha + j];
        alpha_sum_new = warp_sum(asum);
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
    if (!spd && lane == 0) ctrl[BGMM_CTRL_ERROR] = 1;

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
        double* Lo = Pn + L.p_linv + (int64_t)k * DD;
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
    double* Wout = Pn + L.p_w + (int64_t)k * DD;
    for (int e = lane; e < DD; e += 32) Wout[e] = Am[(e / D) * SW_LP + (e % D)];

    // ---- special functions, merged SIMT calls: lanes i < D take (nu - i)/2, three more lanes the scalar arguments ----
    double ps = 0.0, gs = 0.0, psi_x = 0.0, lg_x = 0.0, ln_x = 0.0;
    for (int i = lane; i < D; i += 32) {
        const double a = (nun - i) / 2.0;
        ps += digamma_pos(a);
        gs += lgamma_ni(a);
    }
    ps = warp_sum(ps);
    gs = warp_sum(gs);
    {
        // lane 0: alpha_cur, lane 1: alpha_new, lane 2: sum alpha_new  (digamma);  lane 0: alpha_cur (lgamma);
        // lane 0: kappa0, lane 1: kappa_cur (log)
        const double pa = lane == 0 ? alpha_c : (lane == 1 ? an : alpha_sum_new);
        if (lane < 3) psi_x = digamma_pos(pa);
        if (lane == 0) lg_x = lgamma_ni(alpha_c);
        if (lane < 2) ln_x = log_ni(lane == 0 ? kappa0 : kappa_c);
    }
    const double psi_alpha = __shfl_sync(full, psi_x, 0), psi_an = __shfl_sync(full, psi_x, 1),
                 psi_asum = __shfl_sync(full, psi_x, 2), lg_alpha = __shfl_sync(full, lg_x, 0),
                 ln_kappa0 = __shfl_sync(full, ln_x, 0), ln_kappa = __shfl_sync(full, ln_x, 1);
    const double elndet_n = ps + D * LN2 - logdet;
    const double lnb_n = (nun * logdet - nun * D * LN2 - D * (D - 1) / 2.0 * LNPI - gs * 2.0) / 2.0;
    const double elnpi_n = psi_an - psi_asum;
    if (lane == 0) {
        Pn[L.p_elndet + k] = elndet_n;
        Pn[L.p_lnb + k] = lnb_n;
        Pn[L.p_elnpi + k] = elnpi_n;
    }

    // ---- E-step coefficient row: ln rho = coef . phi(x'), Lambda = nu W ----
    double li = 0.0;
    if (lane < D) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < D; ++j) acc = fma(Am[lane * SW_LP + j], mnew[j], acc);
        li = nun * acc;
    }
    const double mq = warp_sum(lane < D ? mnew[lane] * li : 0.0);
    double* coef = Pn + L.p_coef + (int64_t)k * L.pitch;
    if (lane < D) {
        coef[1 + lane] = li;
        const int base = 1 + D + lane * (lane + 1) / 2;
        for (int j = 0; j < lane; ++j) coef[base + j] = -nun * Am[lane * SW_LP + j];
        coef[base + lane] = -0.5 * nun * Am[lane * SW_LP + lane];
    }
    for (int q = L.P + lane; q < L.pitch; q += 32) coef[q] = 0.0;
    if (lane == 0) {
        const double acst = (hmm_vlx != nullptr ? 0.0 : elnpi_n) + (elndet_n - D * LN2PI - D / kn) / 2.0;
        coef[0] = acst - 0.5 * mq;
        Pn[L.p_acst + k] = acst;
        double* vk = st + L.vlk + (int64_t)k * 8;
        if (iterate) {
            const double lnb0 = st[L.lnb0 + k];
            vk[0] = N * (elndet_c - D / kappa_c - nu_c * t_trs - nu_c * t_q1 - D * LN2PI) / 2.0;           // :673-683
            vk[1] = N * elnpi_c;                                                                          // :686
            vk[2] = (alpha0 - 1.0) * elnpi_c;                                                             // :689
            vk[3] = (D * (ln_kappa0 - LN2PI - kappa0 / kappa_c) - kappa0 * nu_c * t_q2 + 2.0 * lnb0
                     + (nu0 - D) * elndet_c - nu_c * t_tr0) / 2.0;                                        // :692-701
            vk[4] = lg_alpha - (alpha_c - 1.0) * psi_alpha;                                               // :707 (per-k part)
            vk[5] = (D * (1.0 + LN2PI - ln_kappa) - 2.0 * lnb_c - (nu_c - D) * elndet_c + nu_c * D) / 2.0;  // :710-715
            vk[6] = alpha_c;
        }
        vk[7] = (K == 1) ? 0.0 : crit_n * mq;             // conditioning of the feature-map form (see small_kernel)
    }
    {
        double* sh = st + L.shift + (int64_t)k * D;
        const bool have_xbar = iterate && crit_n > 0.0;
        if (lane < D) sh[lane] = have_xbar ? xbar[lane] : mnew[lane];
    }

    // ---- last CTA: conditioning flag of the new set; ELBO sum (all lanes), convergence test (:869), flip ----
    __threadfence();
    __syncwarp();
    int is_last = 0;
    if (lane == 0) is_last = (atomicAdd(const_cast<int*>(&ctrl[BGMM_CTRL_TICKET]), 1) == K - 1);
    is_last = __shfl_sync(full, is_last, 0);
    if (!is_last) return;
    __threadfence();
    const double* vkg = st + L.vlk;
    double px = 0, pz = 0, ppi = 0, pml = 0, qpi = 0, qml = 0, asum = 0, crit = 0;
    for (int j = lane; j < K; j += 32) {
        px += __ldcg(vkg + j * 8 + 0); pz += __ldcg(vkg + j * 8 + 1); ppi += __ldcg(vkg + j * 8 + 2);
        pml += __ldcg(vkg + j * 8 + 3); qpi += __ldcg(vkg + j * 8 + 4); qml += __ldcg(vkg + j * 8 + 5);
        asum += __ldcg(vkg + j * 8 + 6);
        crit = fmax(crit, __ldcg(vkg + j * 8 + 7));
    }
    px = warp_sum(px); pz = warp_sum(pz); ppi = warp_sum(ppi); pml = warp_sum(pml); qpi = warp_sum(qpi);
    qml = warp_sum(qml); asum = warp_sum(asum);
    for (int o = 16; o > 0; o >>= 1) crit = fmax(crit, __shfl_xor_sync(full, crit, o));
    const int robust = crit > robust_thresh ? 1 : 0;
    const int critq = crit < 1073741824.0 ? (int)ceil(crit) : 1073741824;     // NaN -> the large value
    if (!iterate) {
        if (lane == 0) { ctrl[BGMM_CTRL_ROBUST] = robust; ctrl[BGMM_CTRL_CRIT] = critq; ctrl[BGMM_CTRL_TICKET] = 0; }
        return;
    }
    // lane 0: lgamma(sum alpha), lane 1: digamma(sum alpha) — one divergent pair instead of two serial calls
    double sf = 0.0;
    if (lane == 0) sf = lgamma_ni(asum);
    if (lane == 1) sf = digamma_pos(asum);
    const double lg_asum = __shfl_sync(full, sf, 0), psi_as = __shfl_sync(full, sf, 1);
    if (lane != 0) return;
    ppi += st[L.lnc0];
    double qz = -st[L.stats + (int64_t)K * L.pitch + BGMM_STATS_ENTROPY];     // -sum r ln r (:704)
    qpi += -lg_asum + (asum - K) * psi_as;                                       // dirichlet entropy (:707)
    double extra = 0.0;
    if (hmm_vlx != nullptr) {
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
    else if (iter >= max_itr || ctrl[BGMM_CTRL_ERROR]) { ctrl[BGMM_CTRL_DONE] = 1; }
    else { ctrl[BGMM_CTRL_CUR] = cur ^ 1; ctrl[BGMM_CTRL_ROBUST] = robust; ctrl[BGMM_CTRL_CRIT] = critq; }
    ctrl[BGMM_CTRL_ITER] = iter + 1;
    ctrl[BGMM_CTRL_TICKET] = 0;
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
    // block max, then block sum
    for (int o = 16; o; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = red[0];
    for (int w = 1; w < (nt >> 5); ++w) mx = fmax(mx, red[w]);
    __syncthreads();
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
    for (int o = 16; o; o >>= 1) dl = fmax(dl, __shfl_xor_sync(0xffffffffu, dl, o));
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = dl;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < (nt >> 5); ++w) dl = fmax(dl, red[w]);
        Sn[H.s_misc + 0] = mx;
        Sn[H.s_misc + 1] = lc;
        Sn[H.s_misc + 2] = log1p(-2.0 / (exp(0.5 * dl) + 1.0));      // ln tanh(Delta / 4)
        Sn[H.s_misc + 3] = log_ni(dl);                                // ln Delta (-inf when A~ is exactly uniform)
    }
}

// D <= 32 runs the warp-synchronous kernel; the block kernel is the path for larger D
static bool use_warp_kernel(int D) { return D <= 32; }

static cudaError_t launch_small_warp(int K, int D, cudaStream_t stream, double* state, const Layout& L, int mode, int max_itr,
                                     double tol, const CommDesc* cd, const double* hmm_vlx) {
    const double thr = robust_threshold();
#define BGMM_SW_CASE(d) if (D == d) return launch_pdl(small_warp_kernel<d>, dim3(K), dim3(32), 0, stream, state, L, mode, \
                                                      max_itr, tol, cd, hmm_vlx, thr);
    BGMM_SW_CASE(2) BGMM_SW_CASE(4) BGMM_SW_CASE(8) BGMM_SW_CASE(16)
#undef BGMM_SW_CASE
    return launch_pdl(small_warp_kernel<0>, dim3(K), dim3(32), 0, stream, state, L, mode, max_itr, tol, cd, hmm_vlx, thr);
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
    const Layout L = make_layout(K, D, hist_len);
    const HmmLayout H = make_hmm_layout(K);
    const size_t smem = sizeof(double) * ((size_t)D * D + 6 * (size_t)D + 48);
    if (smem > 227 * 1024) {
        set_error("bgmm_hmm_small: D=%d needs %zu B of shared memory (> 227 KiB)", D, smem);
        return BGMM_ENOSUP;
    }
    if (smem > 48 * 1024) {
        int rc = check_cuda(cudaFuncSetAttribute(small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(small_kernel)");
        if (rc) return rc;
    }
    if (mode != BGMM_SMALL_STATS) launch(hmm_trans_kernel, 1, 256, 0, (cudaStream_t)stream, state, L, hst, H, mode);
    if (use_warp_kernel(D))
        return check_cuda(launch_small_warp(K, D, (cudaStream_t)stream, state, L, mode, max_itr, tol, nullptr,
                                            (const double*)(hst + H.vlx)), "hmm small (warp) launch");
    const int nt = D <= 16 ? 32 : (D <= 32 ? 64 : (D <= 64 ? 128 : 256));
    launch(small_kernel, K, nt, smem, (cudaStream_t)stream, state, L, mode, max_itr, tol, nullptr, hst + H.vlx,
           robust_threshold());
    return check_cuda(cudaGetLastError(), "hmm small launch");
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
    const Layout L = make_layout(K, D, hist_len);
    const size_t smem = sizeof(double) * ((size_t)D * D + 6 * (size_t)D + 48);
    if (smem > 227 * 1024) {
        set_error("bgmm_small: D=%d needs %zu B of shared memory (> 227 KiB)", D, smem);
        return BGMM_ENOSUP;
    }
    if (smem > 48 * 1024) {   // per launch: the attribute is per device
        int rc = check_cuda(cudaFuncSetAttribute(small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(small_kernel)");
        if (rc) return rc;
    }
    if (use_warp_kernel(D))
        return check_cuda(launch_small_warp(K, D, (cudaStream_t)stream, state, L, mode, max_itr, tol,
                                            static_cast<const CommDesc*>(comm_desc), (const double*)nullptr),
                          "small_warp_kernel launch");
    // latency-bound kernel full of block barriers: one warp per component while the D x D work is tiny
    const int nt = D <= 16 ? 32 : (D <= 32 ? 64 : (D <= 64 ? 128 : 256));
    return check_cuda(launch_pdl(small_kernel, dim3(K), dim3(nt), smem, (cudaStream_t)stream, state, L, mode, max_itr, tol,
                                 static_cast<const CommDesc*>(comm_desc), (const double*)nullptr, robust_threshold()),
                      "small_kernel launch");
}
