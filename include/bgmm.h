/*
 * bgmm.h — C ABI of the B200-native variational-Bayes Gaussian-mixture hot path.
 *
 * The reference (bayesml/BayesML, pure Python/numpy) has NO FFI / plugin interface: the boundary it exposes
 * is the Python class `bayesml.gaussianmixture.LearnModel`.  This header declares the device entry points
 * that the drop-in Python class (`bayesml_b200.gaussianmixture.LearnModel`) binds with ctypes; each entry
 * point cites the reference method it replaces (all paths: bayesml/gaussianmixture/_gaussianmixture.py).
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.  All pointers are DEVICE pointers unless
 *     the name ends in `_host`.  The library allocates nothing and frees nothing: the caller owns every
 *     buffer (sizes from bgmm_layout / bgmm_workspace_doubles) and passes the cudaStream_t to launch on.
 *   - every call is asynchronous on `stream` and returns 0 on success, a negative BGMM_E* code otherwise;
 *     bgmm_last_error() returns a thread-local message.
 *   - numbers: the model state is float64.  X is float64 (dtype BGMM_F64) or float32 (BGMM_F32, "fp32 mode").
 *   - coordinates: X is CENTRED once on upload (x' = x - c, c = global column mean) and every m-vector in the
 *     device state is expressed in the centred frame; the model is shift-covariant, the host adds c back.
 *
 * Feature-map formulation (DESIGN.md §3).  With P = 1 + D + D(D+1)/2 and
 *     phi(x') = [ 1, x'_0..x'_{D-1}, x'_i x'_j (i >= j, packed lower-triangular: idx = i(i+1)/2 + j) ]
 *   E-step   ln rho_nk = coef_k . phi(x'_n)                      (replaces _update_q_z :772-783)
 *   M-stats  raw_k     = sum_n r_nk phi(x'_n)                    (replaces _calc_n_x_bar_s :725-732)
 * so both are GEMMs against the same phi tile.  Rows of coef / raw have pitch PITCH = round_up(P, 8).
 */
#ifndef BGMM_H_
#define BGMM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BGMM_ABI_VERSION 6

/* dtype of X */
#define BGMM_F64 0
#define BGMM_F32 1

/* error codes */
#define BGMM_OK 0
#define BGMM_EINVAL (-1)   /* bad argument (shape, NULL pointer, unsupported size) */
#define BGMM_ECUDA (-2)    /* CUDA runtime error; see bgmm_last_error() */
#define BGMM_ENOSUP (-3)   /* shape not supported by the requested kernel variant */

/* pass variants (bgmm_pass `variant`) */
#define BGMM_PASS_AUTO 0   /* pick the fastest kernel that supports (K, D, dtype) */
#define BGMM_PASS_SIMPLE 1 /* generic scalar-FMA kernel: any K, D */
#define BGMM_PASS_DMMA 2   /* fp64 tensor-pipe kernel (mma.sync.m8n8k4.f64): K*PITCH accumulators on chip */
#define BGMM_PASS_F32 3    /* fp32-mode streaming kernel: X float32, D <= 3, K <= 8 (fp64 accumulation of partials) */
#define BGMM_PASS_LARGE 4  /* fp64 large K*P regime (D <= 128, K <= 64): E kernel (r -> HBM) + output-stationary M kernel;
                              needs r_out != NULL */
#define BGMM_PASS_TF32 6   /* fp32 mode on the 5th-generation tensor cores (tcgen05.mma kind::tf32, 3xTF32 operands, TMEM
                              accumulators): X float32, 2 <= K <= 64, D <= 31, K * P within 128 TMEM columns.  Whitened E-step
                              GEMM + feature-map statistics GEMM; `workspace` must hold bgmm_tf32_workspace_doubles(K, D, n).
                              Hands over to the DIRECT kernel above ctrl.CRIT = 4096. */
#define BGMM_PASS_DIRECT 5 /* conditioning-safe form, any K, D: ln rho from the explicit differences (x - m_k) and
                              statistics about a per-component shift (state.SHIFT) instead of the global centre.
                              Every other variant is a feature-map kernel whose cancellation error grows like
                              eps * (m_k - c)^T Lambda_k (m_k - c); bgmm_small evaluates that quantity for every new
                              parameter set and raises ctrl.ROBUST when it exceeds bgmm_robust_threshold(); bgmm_pass then
                              runs THIS kernel instead of the requested one (decided on the device, no host sync). */

/* bgmm_small `mode` */
#define BGMM_SMALL_FEATURES 0 /* features + coef of params[cur] from (alpha, m, kappa, nu, W^-1); no statistics used */
#define BGMM_SMALL_ITERATE 1  /* ELBO of (params[cur], stats); convergence test; M-step into params[1-cur]; flip */
#define BGMM_SMALL_STATS 2    /* only ns / x_bar / s_mats from STATS (after the final pass, :895)                 */

/* indices into the offsets table written by bgmm_layout (units: doubles from the start of the state block,
 * except BGMM_OFF_CTRL which is also in doubles but addresses an int32[16] region) */
enum {
    BGMM_OFF_CENTER = 0,     /* c[D]                    global centre subtracted from X                      */
    BGMM_OFF_ALPHA0,         /* h0_alpha_vec[K]                                                              */
    BGMM_OFF_KAPPA0,         /* h0_kappas[K]                                                                 */
    BGMM_OFF_NU0,            /* h0_nus[K]                                                                    */
    BGMM_OFF_M0,             /* h0_m_vecs[K][D]  (centred)                                                   */
    BGMM_OFF_W0INV,          /* h0_w_mats_inv[K][D][D]                                                       */
    BGMM_OFF_LNB0,           /* _ln_b_h0_w_nus[K]                                                            */
    BGMM_OFF_LNC0,           /* _ln_c_h0_alpha[1] (+pad)                                                     */
    BGMM_OFF_PARAMS0,        /* parameter set 0 (see BGMM_P_* below)                                         */
    BGMM_OFF_PARAMS1,        /* parameter set 1 (ping-pong)                                                  */
    BGMM_OFF_STATS,          /* raw[K][PITCH] then tail[8] (slots BGMM_STATS_* below)                        */
    BGMM_OFF_NS,             /* ns[K]                                                                        */
    BGMM_OFF_XBAR,           /* x_bar_vecs[K][D] (centred)                                                   */
    BGMM_OFF_SMATS,          /* s_mats[K][D][D]                                                              */
    BGMM_OFF_VLK,            /* per-component ELBO partials [K][8]                                           */
    BGMM_OFF_VLTERMS,        /* [8]: p_x, p_z, p_pi, p_mu_lambda, q_z, q_pi, q_mu_lambda, vl                 */
    BGMM_OFF_VLHIST,         /* vl history [hist_len]                                                        */
    BGMM_OFF_CTRL,           /* int32[16]: see BGMM_CTRL_*                                                   */
    BGMM_OFF_TOTAL,          /* total size of the state block in doubles                                     */
    BGMM_OFF_STATS_LEN,      /* K*PITCH + 8: length (doubles) of the all-reduced statistics buffer           */
    BGMM_OFF_PARAMS_LEN,     /* length of one parameter set                                                  */
    BGMM_OFF_PITCH,          /* PITCH                                                                        */
    BGMM_OFF_SHIFT,          /* shift[K][D] (centred frame): the point the DIRECT kernel takes its moments about
                                (previous x_bar_k, or m_k before the first pass); maintained by bgmm_small        */
    BGMM_N_OFFSETS
};

/* slots of the statistics tail: state.STATS[K*PITCH + slot], written by every bgmm_pass, read by bgmm_small */
enum {
    BGMM_STATS_ENTROPY = 0,  /* sum_n sum_k r ln r                                                              */
    BGMM_STATS_ROWS = 1,     /* rows the statistics were taken over                                             */
    BGMM_STATS_FORMAT = 2    /* > 0: the moments are taken about state.SHIFT (DIRECT kernel), else about 0      */
};

/* sub-offsets inside one parameter set (written by bgmm_layout into `param_offsets`) */
enum {
    BGMM_P_ALPHA = 0,  /* hn_alpha_vec[K]        */
    BGMM_P_KAPPA,      /* hn_kappas[K]           */
    BGMM_P_NU,         /* hn_nus[K]              */
    BGMM_P_M,          /* hn_m_vecs[K][D] (centred) */
    BGMM_P_WINV,       /* hn_w_mats_inv[K][D][D] */
    BGMM_P_W,          /* hn_w_mats[K][D][D]     */
    BGMM_P_ELNPI,      /* _e_ln_pi_vec[K]        */
    BGMM_P_ELNDET,     /* _e_ln_lambda_dets[K]   */
    BGMM_P_LNB,        /* _ln_b_hn_w_nus[K]      */
    BGMM_P_COEF,       /* coef[K][PITCH]  E-step coefficient rows */
    BGMM_P_ACST,       /* a_k[K] = E[ln pi_k] + (E[ln|Lambda_k|] - D ln 2pi - D/kappa_k)/2: ln rho constant of the DIRECT form */
    BGMM_P_LINV,       /* Linv[K][D][D]: inverse of the lower Cholesky factor of W^-1 (W = Linv^T Linv), i.e. the whitening
                          y = sqrt(nu) Linv (x - m) with |y|^2 = (x-m)^T (nu W) (x-m); operand of the fp32-mode tensor-core E-step */
    BGMM_N_PARAM_OFFSETS
};

/* control words (int32) */
enum {
    BGMM_CTRL_CUR = 0,    /* which parameter set is current (0/1)                                   */
    BGMM_CTRL_ITER,       /* number of ELBO evaluations so far (0 = none; 1 = post-init value done) */
    BGMM_CTRL_DONE,       /* 1 -> bgmm_pass / bgmm_small(ITERATE) return immediately (no-ops)       */
    BGMM_CTRL_CONVERGED,  /* 1 -> the tolerance test fired (:869)                                   */
    BGMM_CTRL_TICKET,     /* internal: last-CTA election for bgmm_small                             */
    BGMM_CTRL_PASS_TICKET,/* internal: last-CTA election for bgmm_pass                              */
    BGMM_CTRL_ERROR,      /* 1 -> a W^-1 was not positive definite (Cholesky failed)                */
    BGMM_CTRL_SEQ,        /* number of peer-memory exchanges published so far                       */
    BGMM_CTRL_ROBUST,     /* 1 -> the current parameter set is ill-conditioned for the feature-map kernels:
                             bgmm_pass runs the DIRECT kernel (set by bgmm_small for every new parameter set)  */
    BGMM_CTRL_CRIT,       /* the conditioning criterion itself, ceil(min(crit, 2^30)), for kernels with their own limit
                             (the fp32 kernel takes the feature-map E-step up to 128)                                 */
    BGMM_CTRL_COMM_LO = 10, /* low / high 32 bits of the DEVICE address of the peer-exchange descriptor (see below), or 0.  */
    BGMM_CTRL_COMM_HI,    /* When set (by the caller, once), every bgmm_pass PUBLISHES the statistics it has just reduced
                             (copy into the own exchange block + stamps) from the reduction's last CTA: no separate
                             launch.  Suppressed per call with BGMM_FORCE_NO_PUBLISH.                                    */
    BGMM_N_CTRL = 16
};

int bgmm_abi_version(void);
const char* bgmm_last_error(void);
/* Number of CUDA kernels libbgmm has launched from the calling host thread since the library was loaded (launches the
 * runtime accepted; copies and memsets are not kernels).  The difference around a call is what that call launched,
 * including kernels the device turns into no-ops (passes queued after convergence, the idle side of the conditioning
 * guard).  A call rejected by its argument checks launches nothing. */
int64_t bgmm_launch_count(void);

/* Sizes.  offsets[BGMM_N_OFFSETS], param_offsets[BGMM_N_PARAM_OFFSETS] are HOST arrays. */
int bgmm_layout(int K, int D, int hist_len, int64_t* offsets_host, int64_t* param_offsets_host);
/* doubles of scratch needed by bgmm_pass for per-CTA partial statistics */
int64_t bgmm_workspace_doubles(int K, int D);

/* ---- data preparation (no reference counterpart: the reference keeps x on the host) ----
 * column sums of the local rows (fp64 accumulation, deterministic), to build the global centre c */
int bgmm_colsum(const void* x_raw, int64_t n, int D, int dtype_in, double* colsum_out /*[D]*/,
                double* workspace, void* stream);
/* x'[n][d] = x_raw[n][d] - c[d], written as dtype_out (may alias x_raw when dtypes match) */
int bgmm_center(const void* x_raw, int dtype_in, void* x_out, int dtype_out, int64_t n, int D,
                const double* center /*[D]*/, void* stream);

/* ---- the hot path ----
 * bgmm_pass: one E-step + sufficient-statistics sweep over the local rows of centred X.
 *   replaces `_update_q_z` (:772-784) incl. `_calc_n_x_bar_s` (:725-732) and the O(N K) term of `_calc_vl` (:704).
 *   Reads coef from params[ctrl.cur]; writes state.STATS (raw moments about the centre, sum r ln r, rows).
 *   r_out / lnrho_out ([n][K] float64) and argmax_out ([n] int32, first index on ties — np.argmax, :1191) are
 *   optional (NULL inside the VB loop: r never touches HBM).
 *   r_in (optional, [n][K] float64): statistics of GIVEN responsibilities instead of the E-step
 *   (`_init_random_responsibility` :734-736); variant SIMPLE/AUTO: moments about the centre, DIRECT: about state.SHIFT
 *   (the reference's two-pass centred `s_mats`, :730-732, when SHIFT holds x_bar).  No-op when ctrl.done != 0 unless `force`. */
#define BGMM_FORCE 1            /* `force` bit 0: run although ctrl.done is set                                          */
#define BGMM_FORCE_NO_PUBLISH 2 /* `force` bit 1: do not publish to the peer-exchange block (a pass that is not followed by
                                   a consuming bgmm_small, e.g. predictive densities of the local rows)                 */
int bgmm_pass(const void* x, int64_t n, int K, int D, int dtype, double* state, double* workspace,
              double* r_out, double* lnrho_out, int32_t* argmax_out, const double* r_in,
              int variant, int force, void* stream);

/* Conditioning guard of the feature-map kernels.  bgmm_small computes, for every new parameter set,
 *   crit = max_k min(N_k, 1) * (m_k - c)^T (nu_k W_k) (m_k - c)     (N_k = 1 before the first statistics exist)
 * and sets ctrl.ROBUST = (crit > threshold).  Default 2e4 (calibrated on the B200, tests/cond_sweep.py: below it every hyperparameter stays within 1e-9 of its own
 * value or 1e-13 of its array's scale, whichever is larger);
 * +inf disables the guard, 0 forces the DIRECT kernel.  Process-wide; returns the previous value. */
double bgmm_set_robust_threshold(double threshold);
double bgmm_robust_threshold(void);

/* ---- batched restarts (north_star (4); the restart loop `update_posterior` :847-883) ----
 * One sweep over X for R independent mixtures of K components each (R restarts of the same fit, each with its own state
 * block): their coefficient rows are stacked into ONE E-GEMM / M-GEMM of R * Kp components (Kp = K rounded up to 8;
 * R * Kp <= 64) with one softmax per group, so X is read once and the feature fragments are generated once for all R.
 * `states_host`: HOST array of R device pointers (member state blocks, bgmm_layout(K, D, .)); `super_state`: a zeroed
 * block of bgmm_layout(R * Kp, D, 1) doubles owned by the caller; `workspace`: bgmm_workspace_doubles(R * Kp, D);
 * `r_scratch`: [n][R * Kp] float64.  Per member the effect equals bgmm_pass(variant LARGE): STATS of every member that is
 * not done is overwritten; members whose ctrl.robust is set are redone by their own DIRECT pass; a no-op when every member
 * is done.  fp64 only. */
#define BGMM_MAX_BATCH 8
int bgmm_pass_batched(const void* x, int64_t n, int K, int D, int R, double* const* states_host, double* super_state,
                      double* workspace, double* r_scratch, void* stream);
/* largest R (>= 1) that bgmm_pass_batched accepts for this shape (1: batching not available) */
int bgmm_batch_capacity(int K, int D);

/* doubles of workspace the TF32 variant needs for n local rows (it includes r as float32 [n][K rounded up to 4]); 0 when
 * the shape is not supported by that variant */
int64_t bgmm_tf32_workspace_doubles(int K, int D, int64_t n);

/* 1 when `variant` (BGMM_PASS_SIMPLE / _DMMA / _F32 / _LARGE / _DIRECT / _TF32) can run this shape, else 0 */
int bgmm_pass_supported(int K, int D, int dtype, int variant);
/* the concrete variant BGMM_PASS_AUTO resolves to (has_r_in: statistics of given responsibilities) */
int bgmm_pass_resolve(int K, int D, int dtype, int variant, int has_r_in);

/* bgmm_small: everything that is O(K D^3): replaces `_update_q_mu_lambda` (:758-770), `_update_q_pi` (:741-743),
 *   `_calc_q_pi_features` (:738-739), `_calc_q_lambda_features` (:745-756), the K-sized terms of `_calc_vl`
 *   (:671-723) and the convergence test (:869).  One CTA per component; Cholesky-based inverse / log-det.
 *   mode FEATURES: params[cur] holds (alpha, m, kappa, nu, W^-1) from the host; fills W, features, coef.
 *   mode ITERATE : vl of (params[cur], STATS) -> vlhist[iter]; if iter >= 1 and |(vl - vl_prev)/vl_prev| < tol
 *                  -> converged, done; else if iter == max_itr -> done; else M-step into params[1-cur], flip cur.
 *                  Also refreshes ns / x_bar / s_mats (s_mats[k] untouched when N_k == 0, as at :729).
 *   mode STATS   : ns / x_bar / s_mats only; parameters and control words untouched. */
int bgmm_small(int K, int D, double* state, int mode, int max_itr, double tol, int hist_len, const void* comm_desc,
               void* stream);

/* ---- either side of the loop (SURVEY.md §8 f2 / f3) ----
 * bgmm_pred_logdensity: out[n] = ln sum_k exp(ck[k] - hk[k] * log1p(Delta2_nk / nuk[k])), the log predictive density of the
 *   mixture of Student-t distributions (/root/reference/bayesml/gaussianmixture/__init__.py:86-97; the reference evaluates
 *   it one point at a time through scipy.stats.multivariate_t, _gaussianmixture.py:1086-1099).  Delta2_nk is recovered from
 *   lnrho[n][K] (bgmm_pass output for a parameter set with Lambda_k = p_lambda_mats[k]) and that set's constants acst[K]
 *   (state: params[cur] + BGMM_P_ACST): lnrho = acst - Delta2 / 2.  Caller supplies (device pointers)
 *   ck = ln p_pi + lnGamma((nu+D)/2) - lnGamma(nu/2) + ln|Lambda|/2 - D/2 ln(nu pi),  hk = (nu + D)/2,  nuk = p_nus.  K <= 64. */
int bgmm_pred_logdensity(const double* lnrho, int64_t n, int K, const double* acst, const double* ck, const double* hk,
                         const double* nuk, double* out, void* stream);
/* bgmm_dirichlet1: r_out[n][K] ~ Dirichlet(1_K) per row (`_init_random_responsibility` :734-735 on the device).
 *   Philox4x32-10 keyed by `seed`, counter = (row_offset + local row, pair index): independent of the sharding.  This is
 *   NOT numpy's PCG64 / ziggurat stream: same distribution, different numbers (opt-in, `device_init=True`). */
int bgmm_dirichlet1(double* r_out, int64_t n, int K, uint64_t seed, int64_t row_offset, void* stream);
/* bgmm_gen_sample: `GenModel.gen_sample` (:241-264, a per-sample Python loop in the reference) on the device:
 *   z_out[n] (int32 class index) ~ Cat(pi) from the cumulative sums cdf[K], x_out[n][D] = mu[z] + chol[z] eps with
 *   chol[k] = lower Cholesky factor of Lambda_k^-1 ([K][D][D]) and eps ~ N(0, I) (Philox + Box-Muller, keyed by `seed` and
 *   the global row index row_offset + i).  Same distribution as the reference, NOT numpy's random stream.  D <= 256. */
int bgmm_gen_sample(double* x_out, int32_t* z_out, int64_t n, int K, int D, const double* cdf, const double* mu,
                    const double* chol, uint64_t seed, int64_t row_offset, void* stream);
/* bgmm_hmm_gen_sample: `hiddenmarkovnormal.GenModel.gen_sample` on the device: z_out[n] (int32 state indices) is a Markov
 *   chain, z_0 ~ pi and z_i ~ A[z_{i-1}], restarting from pi at every sequence start; x_out[n][D] = mu[z] + chol[z] eps as in
 *   bgmm_gen_sample.  Same distribution as the host loop, NOT numpy's random stream.  K <= 32, D <= 256.
 *   cdf[(K+1)][K] (device): row 0 the inverse-CDF table of pi, row 1 + s that of row s of A.  Each row is the cumulative
 *   sum of its probabilities with the entry of its LAST positive-probability state set to 2.0; state k is drawn for
 *   uniform u in (0, 1) as the first k with u <= cdf[row][k].  A zero-probability state is then never drawn, even when the
 *   rounded cumulative sum ends below 1 and u falls above it.
 *   seq_starts[n_seqs] (HOST, int64): first rows of the sequences, starting with 0, strictly increasing, below n; NULL or
 *   n_seqs = 1 for one sequence.  It is copied into the workspace with cudaMemcpyAsync (a pinned array must stay valid
 *   until the stream reaches the copy).
 *   Philox4x32-10 keyed by `seed`, counter = (global element index, word, own tag): word 0 gives the state's uniform, words
 *   1.. the normals, so the sample does not depend on the chunking or on how the rows are split into sequences.
 *   The chain is sampled exactly by composing the per-element transition maps over chunks of chunk_len elements (0 = the
 *   default, at most 4096 chunks; a chunk_len giving more than 4096 chunks is BGMM_EINVAL); the result does not depend on
 *   chunk_len.  workspace: bgmm_hmm_gen_workspace_bytes(K, n, n_seqs, chunk_len) bytes of device memory (0 for a bad
 *   argument). */
int64_t bgmm_hmm_gen_workspace_bytes(int K, int64_t n, int64_t n_seqs, int64_t chunk_len);
int bgmm_hmm_gen_sample(double* x_out, int32_t* z_out, int64_t n, int K, int D, const double* cdf, const double* mu,
                        const double* chol, const int64_t* seq_starts, int64_t n_seqs, uint64_t seed, int64_t chunk_len,
                        void* workspace, void* stream);
/* bgmm_hmm_init_random: the 'random_responsibility' initial state of `hiddenmarkovnormal.LearnModel` (`_init_random_
 *   responsibility`) drawn on the device, ready for bgmm_hmm_pass(_seqs) in mode BGMM_HMM_STATS_FROM_GAMMA: gamma[n][K],
 *   hst.MS = sum of xi_i over the elements that are not sequence starts, hst.G0 = gamma summed over the sequence starts,
 *   hst.SC = 0 (hst: the bgmm_hmm_layout block).  Same distribution as the host rule, NOT numpy's random stream.
 *   Element i draws xt_i[j][k] (j, k < K) as K^2 standard exponentials -ln u, and xi_i = xt_i / (sum of its K^2 entries),
 *   i.e. Dirichlet(1_{K^2}).  u comes from Philox4x32-10 keyed by `seed` (key = seed low, high 32 bits) at counter
 *   (i low, i high, p, 0x484d4d49): pair p = r * K + k (r < ceil(K/2)) gives entry (2r, k) from words 0, 1 and entry
 *   (2r + 1, k) from words 2, 3 (unused when 2r + 1 = K), u = ((w_hi << 32 | w_lo) >> 11) + 0.5) / 2^53 as in
 *   bgmm_dirichlet1.  An element's draw does not depend on how the rows are split into sequences.
 *   Rules: gamma_i = column sums sum_j xi_i[j][.], except at every sequence start s: gamma_s = row sums sum_k xi_{s+1}[.][k]
 *   when its sequence is longer than 1, else the row sums of xi_s.  One sequence of n = 1: gamma_0 = row 0 of xt_0 divided
 *   by its sum (Dirichlet(1_K)), MS = 0.
 *   seq_starts[n_seqs] (device) and seq_starts_host[n_seqs] (the same values on the host; the checks read it): first rows
 *   of the sequences, starting with 0, strictly increasing, below n; n_seqs = 1 (pointers ignored, may be NULL) for one
 *   sequence.  K <= 32.  MS and G0 are summed in an order fixed by (n, K): a re-run gives the same bits.
 *   workspace: bgmm_hmm_init_random_workspace_doubles(K, n) doubles (0 for a bad argument). */
int64_t bgmm_hmm_init_random_workspace_doubles(int K, int64_t n);
int bgmm_hmm_init_random(int64_t n, int K, uint64_t seed, const int64_t* seq_starts_host, const int64_t* seq_starts,
                         int64_t n_seqs, double* gamma, double* hst, double* workspace, void* stream);

/* ---- 5th-generation tensor cores (fp32 mode) ----
 * bgmm_tc_selftest: D[128][N] = A[128][Kd] . B[N][Kd]^T with tcgen05.mma kind::tf32 (operands staged in shared memory in the
 * no-swizzle canonical layout, K-major or MN-major; accumulator in tensor memory, read back with tcgen05.ld) — the unit test
 * of the descriptor conventions the fp32-mode kernels use.  A, B, D: device float32 arrays, row-major as written. */
int bgmm_tc_selftest(const float* A, const float* B, float* D, int N, int Kd, int a_mn_major, int b_mn_major, void* stream);

/* ---- multi-GPU exchange over NVLink peer memory (no reference counterpart: the reference is single-process) ----
 * Row-sharded fit: the per-iteration all-reduce of state.STATS is fused into bgmm_small.  Every rank owns an exchange
 * block  [2][stats_len] doubles | [2][BGMM_MAX_RANKS] uint64 stamps  allocated by bgmm_comm_alloc (cudaMalloc, zeroed)
 * and mapped by its peers through CUDA IPC (bgmm_comm_open on the 64-byte handle).  `comm_desc` is a DEVICE struct
 *   { int32 world; int32 rank; int64 reserved; double* xchg[BGMM_MAX_RANKS]; }   (xchg[rank] = own block)
 * built by the caller.  With its address in ctrl.COMM, the last CTA of every bgmm_pass's reduction copies state.STATS into
 * the own block, fences at system scope and stamps every peer; bgmm_small with comm_desc != NULL (modes ITERATE, STATS)
 * waits for all stamps, sums the peers' blocks in rank order (bit-identical result on every rank) and stores the sums back
 * into state.STATS.  comm_desc == NULL: state.STATS is used as is (single GPU, or all-reduced by the caller, e.g.
 * ncclAllReduce). */
#define BGMM_MAX_RANKS 16
int64_t bgmm_comm_block_doubles(int K, int D);
int bgmm_comm_alloc(int64_t doubles, void** base_out, void* ipc_handle_out /* 64 bytes, host */);
int bgmm_comm_open(const void* ipc_handle /* 64 bytes, host */, void** peer_ptr_out);
int bgmm_comm_close(void* peer_ptr);
int bgmm_comm_free(void* base);

/* ---- hidden-Markov model with Gaussian emissions (SURVEY.md §8 f1) -----------------------------------------------
 * Replaces the VB loop body of /root/reference/bayesml/hiddenmarkovnormal/_hiddenmarkovnormal.py
 * `LearnModel.update_posterior` (:1028-1134).  The Gauss-Wishart / Dirichlet(eta) part of the model is the mixture's,
 * so it lives in the SAME state block (bgmm_layout; alpha plays eta, :981).  The transition-matrix part lives in a
 * second block "hst" (doubles; offsets from bgmm_hmm_layout):
 *   ZETA0 [K][K] prior h0_zeta_vecs | LNCZ0 ln C(zeta0) sum (:828) |
 *   SET0 / SET1 (ping-pong with ctrl.cur): +SET_ZETA [K][K] hn_zeta_vecs, +SET_LNA ln a~ (:852), +SET_AT a~ = exp(ln a~
 *   - max) (:853), +SET_MISC {max ln a~, ln C(zeta) sum (:854)} |
 *   MS [K][K] sum_i xi_i (:839) | G0 [K] gamma_0 | SC {sum_i ln c_i, sum gamma.ln rho, warm-up window of the last pass} |
 *   VLX {E ln p(z) :886, E ln p(A) :892, -E ln q(z) :906-909, -E ln q(A) :915}. */
enum {
    BGMM_HMM_OFF_ZETA0 = 0, BGMM_HMM_OFF_LNCZ0, BGMM_HMM_OFF_SET0, BGMM_HMM_OFF_SET1, BGMM_HMM_OFF_SET_ZETA,
    BGMM_HMM_OFF_SET_LNA, BGMM_HMM_OFF_SET_AT, BGMM_HMM_OFF_SET_MISC, BGMM_HMM_OFF_MS, BGMM_HMM_OFF_G0,
    BGMM_HMM_OFF_SC, BGMM_HMM_OFF_VLX, BGMM_HMM_OFF_TOTAL, BGMM_HMM_OFF_COUNT
};
int bgmm_hmm_layout(int K, int64_t* off /* [BGMM_HMM_OFF_COUNT] */);
/* 1 when the device path covers this shape (float64, K <= 32, D <= 128), else 0 */
int bgmm_hmm_supported(int K, int D);
/* doubles of scratch the scan needs for a sequence of n elements */
int64_t bgmm_hmm_scan_workspace_doubles(int K, int64_t n);

/* bgmm_hmm_pass `mode` */
#define BGMM_HMM_FULL 0             /* `_update_q_z` :1020-1026: emission density, forward, backward, gamma, xi, statistics */
#define BGMM_HMM_STATS_FROM_GAMMA 1 /* `_calc_n_m_x_bar_s` :837-845 of a given gamma (random_responsibility init :944-952);
                                       the caller has written MS, G0 and SC into hst                                      */
#define BGMM_HMM_EMISSION_ONLY 2    /* `_calc_rho` :988-996 only: lnrho[n][K] (the other per-element buffers may be NULL)    */
/* One E-step over the whole (centred, float64) sequence x[n][D] with the CURRENT parameter set:
 *   lnrho[n][K] (:988-996), alpha[n][K] and cs[n] (:999-1006), gamma[n][K] (:1014), optionally beta_out[n][K]
 *   (:1008-1011; NULL inside the loop), hst.MS / G0 / SC, and the gamma-weighted raw moments into state.STATS.
 * The two recursions run as chunked three-phase scans (csrc/bgmm_hmm.cu).  `workspace`: bgmm_workspace_doubles(K, D);
 * `scan_ws`: bgmm_hmm_scan_workspace_doubles(K, n).  No-op when ctrl.done != 0 unless `force`. */
int bgmm_hmm_pass(const void* x, int64_t n, int K, int D, double* state, double* hst, double* workspace, double* scan_ws,
                  double* lnrho, double* alpha, double* gamma, double* cs, double* beta_out, int mode, int force,
                  void* stream);
/* bgmm_small for the hidden-Markov model: hmm_trans_kernel (`_update_q_a` :984-986, `_calc_q_a_features` :851-854, the
 * ELBO terms with A / xi / gamma_0 / c) followed by the mixture's small kernel with ln rho free of E[ln pi] (:989-992)
 * and the 9-term ELBO (:869-932).  Modes as bgmm_small. */
int bgmm_hmm_small(int K, int D, double* state, double* hst, int mode, int max_itr, double tol, int hist_len, void* stream);

/* Viterbi path (`estimate_latent_vars(viterbi=True)`, :1466-1480) from lnrho[n][K], ln pi~ [K] and ln a~ [K][K] (device
 * pointers): omega[n][K] (:1469-1471), phi[n][K] (int32, row 0 is not written — the reference leaves it zero, :1472) and
 * path[n] (int32 state indices, :1474-1479).  The recursion keeps the reference's operation order, so the outputs are
 * bit-identical to numpy's for identical inputs.  K <= 32. */
int bgmm_hmm_viterbi(int64_t n, int K, const double* lnrho, const double* lnpi, const double* lna, double* omega,
                     int32_t* phi, int32_t* path, void* stream);

/* ---- several independent sequences sharing one posterior (`lengths=`) ---------------------------------------------
 * x[n][D] holds the sequences concatenated in order; seq_starts[n_seqs] (int64, seq_starts[0] == 0, strictly increasing,
 * < n) are their first rows.  The recursions restart at every sequence start (forward from pi~, backward from ones), xi
 * is zero there (MS counts transitions inside sequences only) and G0 = sum over sequence starts of gamma there.
 *
 * bgmm_hmm_seq_plan (host): the chunk table bgmm_hmm_pass_seqs runs on (every sequence is cut into chunks of the
 * single-sequence chunk length; no chunk crosses a sequence start).  Returns the table's length in int64 (and fills
 * `plan` when cap is at least that), or BGMM_EINVAL for a bad argument.  The caller copies it to the device once. */
int64_t bgmm_hmm_seq_plan(int64_t n, int64_t n_seqs, const int64_t* seq_starts, int64_t* plan, int64_t cap);
/* doubles of scratch bgmm_hmm_pass_seqs needs (0 for a bad argument) */
int64_t bgmm_hmm_seq_workspace_doubles(int K, int64_t n, int64_t n_seqs);
/* bgmm_hmm_pass over several sequences: `plan` the host table from bgmm_hmm_seq_plan, `plan_dev` the same on the device;
 * `scan_ws`: bgmm_hmm_seq_workspace_doubles(K, n, n_seqs). */
int bgmm_hmm_pass_seqs(const void* x, int64_t n, int K, int D, double* state, double* hst, double* workspace,
                       double* scan_ws, double* lnrho, double* alpha, double* gamma, double* cs, double* beta_out, int mode,
                       int force, const int64_t* plan, const int64_t* plan_dev, void* stream);
/* bgmm_hmm_viterbi per sequence (seq_starts: device), the sequences decoded in parallel; phi is 0 at every sequence start.
 * Bit-identical to the numpy recursion run sequence by sequence. */
int bgmm_hmm_viterbi_seqs(int64_t n, int K, const double* lnrho, const double* lnpi, const double* lna, double* omega,
                          int32_t* phi, int32_t* path, const int64_t* seq_starts, int64_t n_seqs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BGMM_H_ */
