// bgmm_hmm_pass: the E-step of the variational-Bayes hidden-Markov model with Gaussian emissions on one B200.
//
// Replaces, in /root/reference/bayesml/hiddenmarkovnormal/_hiddenmarkovnormal.py, `_update_q_z` :1020-1026 =
//   _calc_rho :988-997          ln rho[n][k] (emission log density under q)        -> e_large_kernel, ln-rho-only mode
//   _forward :999-1006          alpha_i = rho_i o (alpha_{i-1} A~) / c_i            -> hmm_basis_mma / hmm_seq / hmm_fwd
//   _backward :1008-1011        beta_i = A~ (rho_{i+1} o beta_{i+1}) / c_{i+1}       -> hmm_basis_mma / hmm_seq / hmm_bwd
//   _update_gamma :1013-1014    gamma = alpha o beta                                 -> hmm_bwd
//   _update_xi :1016-1018       xi_i = alpha_{i-1} rho_i A~ beta_i / c_i; only sum_i xi_i (= ms, :839) is formed
//   _calc_n_m_x_bar_s :837-845  N_k, x_bar_k, S_k with gamma as weights              -> m_large_kernel + reduction
//
// The reference runs both recursions sequentially over the sequence (a Python loop).  Here the sequence is cut into
// chunks and each recursion becomes three phases (numpy model + test: tools/hmm_scan_model.py):
//   A  (parallel over chunk x start state): the recursion from each unit vector -> chunk transfer matrix, every row
//      normalised with its log scale kept;
//   B  (one warp, sequential over chunks): propagate the boundary vector through the transfer matrices;
//   C  (parallel over chunks): the reference's exact recursion from the chunk's boundary vector, writing alpha, c
//      (forward) or gamma, sum xi, sum gamma ln rho (backward).
// Phase A costs K times phase C (N K^3 flops) and runs on the FP64 tensor pipe (hmm_basis_mma_kernel: the K runs of a
// chunk as one matrix recursion).  Phases B and C are FP64 CUDA-core work on small per-state vectors; in phase C a group
// of KP = 2^ceil(log2 K) lanes owns one chunk (32 / KP chunks per warp), state vectors are exchanged through a per-warp
// shared-memory line (one STS + K/2 broadcast LDS.128 per step).  All sums are in a fixed order (deterministic).
// Several independent sequences (bgmm_hmm_pass_seqs): every sequence is cut into its own chunks (ScanPlan.coff), so no
// recursion meets a restart inside a chunk; phase B is segmented per sequence and the windows are clamped to it.
#include "bgmm_common.cuh"
#include "bgmm_mma.cuh"
#include <math.h>
#include <stdlib.h>
#include <type_traits>

namespace bgmm {

int launch_pass_large_part(const PassArgs& a, int K, int D, int dtype, int which, cudaStream_t stream, int group_blocks = 0);
bool large_supported(int K, int D, int dtype);

constexpr int HW = 4;            // warps per CTA in the scan kernels
constexpr int HT = 32 * HW;

struct ScanPlan {
    int64_t n;
    int K, L, nch;
    int window_cap;      // longest warm-up window the mixing mode may use (0 disables it); env BGMM_HMM_WINDOW_CAP
};


template <int KP>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = KP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// every lane publishes `v`; returns nothing — the caller then reads the KP values of its group from `line`
template <int KP>
__device__ __forceinline__ void publish(double* line, int lane, double v) {
    line[lane] = v;
    __syncwarp();
}

// dot of the group's published vector with this lane's K-vector `m`, four independent partial sums
template <int KP>
__device__ __forceinline__ double group_dot(const double* line, int gbase, const double (&m)[KP]) {
    double s0 = 0.0, s1 = 0.0;
    if (KP >= 2) {
        const double2* p = reinterpret_cast<const double2*>(line + gbase);
#pragma unroll
        for (int j = 0; j < KP / 2; ++j) {
            const double2 v = p[j];
            s0 = fma(v.x, m[2 * j], s0);
            s1 = fma(v.y, m[2 * j + 1], s1);
        }
    }
    return s0 + s1;
}

// ---------------------------------------------------------------------------------------------------------------
struct ScanBufs {
    const double* lnrho;   // [n][K]
    const double* rhohat;  // [n][K] exp(ln rho - row max): what the recursions multiply by (rho_i / c_i = rhohat_i / chat_i)
    const double* rowmax;  // [n]    max_k ln rho
    double* chat;          // [n]    c_i exp(-row max): the normaliser in rhohat units
    double* ichat;         // [n]    1 / chat_i (hmm_cs_kernel), what the backward kernels multiply by
    double* alpha;         // [n][K]
    double* gamma;         // [n][K]
    double* cs;            // [n]
    double* beta_out;      // [n][K] or NULL
    double* tf;            // [nch][K][K] transfer matrices (forward, then reused backward)
    double* ls;            // [nch][K]    their log scales
    double* vb;            // [nch][K]    chunk boundary vectors (forward, then reused backward)
    double* ps;            // [nch][K][K] xi-sum partials
    double* plc;           // [nch]       sum ln c partials
    double* pgl;           // [nch]       sum gamma ln rho partials
    double* seq2;          // two-level sweep: group matrices [72][K][K], log scales [72][K], boundary vectors [72][K]
};

// Several sequences (bgmm_hmm_pass_seqs): chunk c covers elements [coff[c], coff[c+1]) of the sequence [sst[c], sen[c]);
// chunks never cross a sequence start.  The scan kernels take it as a trailing argument of type SeqArg<SEQS>, empty for
// one sequence (chunk c = [cL, min(cL + L, n))), so the one-sequence instantiations keep the single-sequence arguments.
struct SeqTable {
    const int64_t* coff;
    const int64_t* sst;
    const int64_t* sen;
    double* pg0;           // [nch][K] gamma at the first element of chunks that start a sequence
};
struct NoSeqTable {};
template <bool SEQS> using SeqArg = typename std::conditional<SEQS, SeqTable, NoSeqTable>::type;

struct ChunkInfo {
    int64_t i0, i1;      // the chunk's elements [i0, i1)
    int64_t s0, s1;      // its sequence's elements [s0, s1)
};
// The scan kernels are instantiated twice: SEQS = false is the one-sequence code (chunk c = [cL, min(cL + L, n)), the
// expressions of the single-sequence path), SEQS = true reads the chunk table through chunk_info.
__device__ __forceinline__ ChunkInfo chunk_info(const ScanPlan& sp, const SeqTable& T, int c) {
    ChunkInfo ci;
    if (c >= sp.nch) c = sp.nch - 1;                 // idle lane groups past the last chunk: the table ends there
    ci.i0 = T.coff[c];
    ci.i1 = T.coff[c + 1];
    ci.s0 = T.sst[c];
    ci.s1 = T.sen[c];
    return ci;
}
// steps a warp's recursion loop runs: the chunk length, or (several sequences) the longest live chunk of the warp
__device__ __forceinline__ int warp_steps(bool live, const ChunkInfo& ci) {
    return (int)__reduce_max_sync(0xffffffffu, live ? (unsigned)(ci.i1 - ci.i0) : 0u);
}
// pi~ = exp(ln pi~ - max) (:849), component kk
__device__ __forceinline__ double pi_tilde(const double* st, const Layout& L, int K, int kk) {
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    const double* Pc = st + L.params[ctrl[BGMM_CTRL_CUR]];
    double pmax = -INFINITY;
    for (int k = 0; k < K; ++k) pmax = fmax(pmax, Pc[L.p_elnpi + k]);
    return kk < K ? exp(Pc[L.p_elnpi + kk] - pmax) : 0.0;
}

__device__ __forceinline__ const double* current_at(const double* st, const Layout& L, const double* hst, const HmmLayout& H) {
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    return hst + H.set[ctrl[BGMM_CTRL_CUR]] + H.s_at;
}

// Mixing mode.  Two message vectors at Hilbert distance <= Delta are at distance <= tau^(W-1) Delta after W steps of
// either recursion (Birkhoff contraction, tau = tanh(Delta(A~) / 4); the emission values are diagonal scalings and do not
// change the metric).  Below 1e-18 the W-step transfer matrix is rank one in fp64, so the boundary vector of a chunk is
//   forward : the normalised end vector of ONE run over the W elements before the chunk, from any start;
//   backward: ONE un-normalised run over the W elements after the chunk from the all-ones vector, true scale included:
//             U w = (U 1)(alpha_end . w) / (alpha_end . 1) = U 1, because alpha_end . w = sum_k gamma_k = 1.
// hmm_window returns the smallest such W for the current A~ (hmm_trans_kernel stores ln tau and ln Delta), or 0 when the
// window would cost more than the exact alternative — the K basis runs per chunk (phase A) + the sequential sweep (B).
// Windows that reach the end of the sequence start from the true vector there (pi~ / ones) and are exact.
__device__ __forceinline__ int hmm_window(const double* st, const Layout& L, const double* hst, const HmmLayout& H,
                                          const ScanPlan& sp) {
    const int chunk_len = sp.L, K = sp.K;
    if (sp.window_cap <= 0) return 0;
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    const double* misc = hst + H.set[ctrl[BGMM_CTRL_CUR]] + H.s_misc;
    const double lntau = misc[2], lndelta = misc[3];
    if (!(lndelta > -INFINITY)) return 8;                     // A~ exactly uniform: rank one after a single step
    if (!(lntau < 0.0)) return 0;
    const double w = ceil((-41.5 - lndelta) / lntau) + 1.0;     // tau^(W-1) Delta < 1e-18
    const double cap = fmin((double)sp.window_cap, 0.5 * (double)chunk_len * (double)K);
    if (!(w <= cap)) return 0;
    return w < 8.0 ? 8 : (int)w;
}

// Phase C, forward: the exact recursion over one chunk from its boundary vector v[c] (pi~ where a sequence starts);
// writes alpha and chat.  Lane kk of a group owns state kk and column kk of A~.
template <int KP, bool SEQS>
__global__ void __launch_bounds__(HT) hmm_fwd_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                     const double* __restrict__ hst, const HmmLayout H, const int force,
                                                     const ScanBufs B, const SeqArg<SEQS> T) {
    __shared__ __align__(16) double lines[HW][2][32];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    constexpr int G = 32 / KP;
    const int K = sp.K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, kk = lane % KP, grp = lane / KP;
    const double* at = current_at(st, L, hst, H);
    const double* __restrict__ rhohat = B.rhohat;
    const int64_t item = ((int64_t)blockIdx.x * HW + warp) * G + grp;
    const int c = (int)item;
    ChunkInfo ci{};
    if constexpr (SEQS) ci = chunk_info(sp, T, c);
    const bool live = item < sp.nch, mine = live && kk < K;
    if (SEQS && !__any_sync(0xffffffffu, live)) return;
    double acol[KP];
#pragma unroll
    for (int j = 0; j < KP; ++j) acol[j] = (mine && j < K) ? at[j * K + kk] : 0.0;
    double a = 0.0;
    if (SEQS && ci.i0 == ci.s0) a = mine ? pi_tilde(st, L, K, kk) : 0.0;   // a sequence starts
    else if (mine) a = B.vb[(int64_t)c * K + kk];
    const int64_t i0 = SEQS ? ci.i0 : (int64_t)c * sp.L;
    const int nst = SEQS ? warp_steps(live, ci) : sp.L;
    // emission values are fetched two steps ahead of the dependent chain (which runs through `a` only)
    auto RH = [&](int64_t i, int s) {
        return (mine && (SEQS ? i < ci.i1 : (s < sp.L && i < sp.n))) ? rhohat[i * K + kk] : 0.0;
    };
    double rho_c = RH(i0, 0), rho_n = RH(i0 + 1, 1);
    for (int s = 0; s < nst; ++s) {
        const int64_t i = i0 + s;
        const double rho = rho_c;
        rho_c = rho_n;
        rho_n = RH(i + 2, s + 2);
        double* line = lines[warp][s & 1];
        publish<KP>(line, lane, a);
        const double dot = group_dot<KP>(line, grp * KP, acol);
        const double u = rho * ((SEQS ? i == ci.s0 : i == 0) ? a : dot);   // :1000 — the first element has no transition
        const double sum = group_sum<KP>(u);                       // chat_i; c_i, 1 / chat_i and sum ln c_i: hmm_cs_kernel
        if (live && i < (SEQS ? ci.i1 : sp.n)) {
            a = u / sum;
            if (mine) B.alpha[i * K + kk] = a;
            if (kk == 0) B.chat[i] = sum;
        }
    }
}

// c_i = chat_i e^{max_i} (:1001-1004), 1 / chat_i and the chunk's sum of ln c_i (for -E ln q(z), :909): element-wise, kept
// out of the sequential recursions.  One CTA per chunk, fixed-order block sum.
template <bool SEQS>
__global__ void __launch_bounds__(128) hmm_cs_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                     const int force, const ScanBufs B, const SeqArg<SEQS> T) {
    __shared__ double red[40];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    const int c = blockIdx.x;
    ChunkInfo ci{};
    if constexpr (SEQS) ci = chunk_info(sp, T, c);
    const int64_t i0 = SEQS ? ci.i0 : (int64_t)c * sp.L;
    const int64_t i1 = SEQS ? ci.i1 : (i0 + sp.L < sp.n ? i0 + sp.L : sp.n);
    double acc = 0.0;
    for (int64_t i = i0 + threadIdx.x; i < i1; i += 128) {
        const double ch = B.chat[i], mx = B.rowmax[i];
        B.cs[i] = ch * exp(mx);
        B.ichat[i] = 1.0 / ch;
        acc += log(ch) + mx;
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) B.plc[c] = acc;
}

// Phase B (both directions): the sequential sweep over the chunk transfer matrices, one CTA.
//   forward : v[0] = pi~ = exp(ln pi~ - max) (:849, :1000); v[c+1] = normalise(sum_j v[c][j] e^{ls_j} T_c[j][:])
//   backward: w[nch-1] = 1 (:939);  w[c-1][k] = sum_j w[c][j] e^{ls_j} U_c[j][k]          (true scale kept)
// Warps 1..3 stage batches of chunk matrices into shared memory (double buffered) and turn the log scales into
// e_j = exp(ls_j - max_j ls) (+ exp(max) for the backward sweep) — everything that does not depend on the running
// vector; warp 0 runs the recurrence from shared memory: multiply, one shared-memory exchange, K FMAs, one division.
// The normaliser of the forward sweep is sum_j w_j (the rows of T sum to one), formed redundantly by every lane in a
// fixed order instead of a shuffle reduction after the matrix-vector product.
constexpr int SEQ_T = 128;
// Two-level sweep (r02).  The recurrence over nch - 1 chunk matrices is sequential (~0.3 us per step: one shared-memory
// exchange, K dependent FMAs, a reciprocal), 1.2 ms per direction at 4096 chunks.  It is a product of matrices, so it is cut
// into groups of SEQ_GLEN steps:
//   mode 1 (grid = groups x start-state blocks): the recurrence over ONE group's steps from every unit vector -> the
//           group's transfer matrix (rows normalised, log scale kept: forward; true scale: backward) — the chunk-level
//           phase A one level up;
//   mode 2 (one CTA): the same sequential sweep, over the <= 64 group matrices -> the vector at every group boundary;
//   mode 3 (grid = groups): the recurrence over one group's steps from its boundary vector, writing every chunk's vector.
// mode 0 is the single-CTA sweep over everything (few chunks).  Same arithmetic per step in all modes; the association
// of the matrix products differs (1e-16 relative), the order of every sum is fixed.
constexpr int SEQ_GLEN = 64;
struct SeqLevel {
    int mode, nsteps, ngroups;
    const double* tf;      // [.][K][K] matrices the steps read (chunk transfer matrices, or group matrices in mode 2)
    const double* ls;      // [.][K]    their log scales
    double* vb;            // [.][K]    vectors the steps write (chunk boundary vectors, or group boundary vectors in mode 2)
    double* tg;            // [ngroups][K][K] mode 1 output
    double* lsg;           // [ngroups][K]    mode 1 output
    const double* vbg;     // [ngroups][K]    mode 3 input: the vector at the start of every group
};
// several sequences: the swept chunk range (a trailing kernel argument, empty for one sequence)
struct SeqRange {
    int cbase;             // modes 0, 1, 3: chunk index of the first chunk of the swept range
    const int64_t* segs;   // mode 0: CTA b sweeps chunks [segs[2b], segs[2b] + segs[2b+1]) (cbase, nsteps unused); or NULL
};
template <bool SEQS> using SeqRangeArg = typename std::conditional<SEQS, SeqRange, NoSeqTable>::type;
__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__host__ __device__ inline int seq_batch(int K) {
    const int per = (K * K + K + 8) * 8;
    int b = (200 * 1024) / (2 * per);
    return b > 64 ? 64 : (b < 1 ? 1 : b);
}

template <int KP, bool FWD, bool SEQS>
__global__ void __launch_bounds__(SEQ_T) hmm_seq_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                        const double* __restrict__ hst, const HmmLayout H,
                                                        const int force, const SeqLevel lv, const SeqRangeArg<SEQS> R) {
    extern __shared__ __align__(16) double sq[];
    __shared__ __align__(16) double lines[2][32];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    if (hmm_window(st, L, hst, H, sp) > 0) return;   // mixing mode: the window kernel wrote the boundary vectors
    const int K = sp.K, KK = K * K, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb_chunk = seq_batch(K);
    const int stride = KK + K + 8;                       // per chunk: matrix [K][K] | e [K] | {exp(max), ...}
    int cb = 0, nsteps_all = lv.nsteps;                  // the swept chunk range: [cb, cb + nsteps_all]
    if constexpr (SEQS) {
        cb = R.cbase;
        if (R.segs != nullptr) {                         // segmented sweep: one sequence per CTA
            cb = (int)R.segs[2 * blockIdx.x];
            nsteps_all = (int)R.segs[2 * blockIdx.x + 1] - 1;
        }
    }
    // this CTA's range of sequential positions [s_lo, s_lo + nsteps): everything (modes 0, 2) or one group (modes 1, 3)
    const int grp = (lv.mode == 1 || lv.mode == 3) ? (int)blockIdx.x : 0;
    const int s_lo = grp * SEQ_GLEN;
    const int nsteps = (lv.mode == 1 || lv.mode == 3) ? min(SEQ_GLEN, (SEQS ? nsteps_all : lv.nsteps) - s_lo)
                                                      : (SEQS ? nsteps_all : lv.nsteps);
    const int nbatch = (nsteps + nb_chunk - 1) / nb_chunk;
    const int n_items = (SEQS ? nsteps_all : lv.nsteps) + 1;   // chunks (modes 0, 1, 3) or groups + 1 (mode 2) along the sweep
    const bool mine = lane < K;
    // item (chunk / group) handled at sequential position s, and the item whose vector that step produces
    auto chunk_of = [&](int s) {
        const int q = (FWD || lv.mode == 2) ? s : n_items - 1 - s;
        return SEQS ? cb + q : q;
    };
    auto out_of = [&](int s) {
        const int q = (FWD || lv.mode == 2) ? s + 1 : n_items - 2 - s;
        return SEQS ? cb + q : q;
    };
    double a = 0.0, lsacc = 0.0;
    if (warp == 0) {
        if (lv.mode == 1) {
            a = (lane == (int)blockIdx.y) ? 1.0 : 0.0;   // unit vector of start state blockIdx.y
        } else if (lv.mode == 3) {
            a = mine ? lv.vbg[(int64_t)grp * K + lane] : 0.0;
            if (grp == 0 && mine) lv.vb[(int64_t)chunk_of(0) * K + lane] = a;
        } else {
            if (FWD) {
                const double* Pc = st + L.params[ctrl[BGMM_CTRL_CUR]];
                double pmax = -INFINITY;
                for (int k = 0; k < K; ++k) pmax = fmax(pmax, Pc[L.p_elnpi + k]);
                a = mine ? exp(Pc[L.p_elnpi + lane] - pmax) : 0.0;
            } else {
                a = mine ? 1.0 : 0.0;
            }
            if (mine) lv.vb[(int64_t)chunk_of(0) * K + lane] = a;
        }
    }
    auto load_batch = [&](int b, int t0, int nt) {       // threads t0 .. t0+nt-1 of the CTA
        double* dst = sq + (size_t)(b & 1) * nb_chunk * stride;
        const int s0 = b * nb_chunk, cnt = min(nb_chunk, nsteps - s0);
        for (int q = 0; q < cnt; ++q) {
            const int c = chunk_of(s_lo + s0 + q);
            const double* src = lv.tf + (int64_t)c * KK;
            // asynchronous copies: a whole batch is in flight at once (a load -> store loop would serialise on latency)
            if ((K & 1) == 0) {             // K even: every row pair is 16-byte aligned on both sides (stride is even too)
                for (int e = 2 * (tid - t0); e < KK; e += 2 * nt) cp_async16(dst + q * stride + e, src + e);
                for (int e = 2 * (tid - t0); e < K; e += 2 * nt) cp_async16(dst + q * stride + KK + e, lv.ls + (int64_t)c * K + e);
            } else {
                for (int e = tid - t0; e < KK; e += nt) cp_async8(dst + q * stride + e, src + e);
                for (int e = tid - t0; e < K; e += nt) cp_async8(dst + q * stride + KK + e, lv.ls + (int64_t)c * K + e);
            }
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
    };
    auto scale_batch = [&](int b, int t0, int nt) {      // ls -> e = exp(ls - max), exp(max)
        double* dst = sq + (size_t)(b & 1) * nb_chunk * stride;
        const int s0 = b * nb_chunk, cnt = min(nb_chunk, nsteps - s0);
        if (K <= 8) {                                    // many small chunks per batch: one thread per chunk
            for (int q = tid - t0; q < cnt; q += nt) {
                double* e = dst + q * stride + KK;
                double mx = -INFINITY;
                for (int j = 0; j < K; ++j) mx = fmax(mx, e[j]);
                for (int j = 0; j < K; ++j) e[j] = (mx > -INFINITY) ? exp(e[j] - mx) : 0.0;
                e[K] = (mx > -INFINITY) ? exp(mx) : 0.0;
            }
            return;
        }
        for (int q = (tid - t0) >> 5; q < cnt; q += nt >> 5) {      // few large chunks: one warp per chunk, lane = j
            double* e = dst + q * stride + KK;
            const double v = lane < K ? e[lane] : -INFINITY;
            double mx = v;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            if (lane < K) e[lane] = (mx > -INFINITY) ? exp(v - mx) : 0.0;
            if (lane == 0) e[K] = (mx > -INFINITY) ? exp(mx) : 0.0;
        }
    };
    if (nbatch > 0) {
        load_batch(0, 0, SEQ_T);
        __syncthreads();
        scale_batch(0, 0, SEQ_T);
        __syncthreads();
    }
    for (int b = 0; b < nbatch; ++b) {
        if (warp > 0) {
            if (b + 1 < nbatch) {
                load_batch(b + 1, 32, SEQ_T - 32);
                asm volatile("bar.sync 1, 96;" ::: "memory");
                scale_batch(b + 1, 32, SEQ_T - 32);
            }
        } else {
            const double* src = sq + (size_t)(b & 1) * nb_chunk * stride;
            const int s0 = b * nb_chunk, cnt = min(nb_chunk, nsteps - s0);
            // column `lane` of the chunk matrix, the scale factors: fetched one step ahead of the dependent chain
            double m[KP], mn[KP], e_c, e_n, sc_c = 0.0, sc_n = 0.0;
            auto fetch = [&](int q, double (&dst)[KP], double& e, double& sc) {
                const double* M = src + q * stride;
#pragma unroll
                for (int j = 0; j < KP; ++j) dst[j] = (mine && j < K) ? M[j * K + lane] : 0.0;
                e = mine ? M[KK + lane] : 0.0;
                if (!FWD) sc = M[KK + K];
            };
            fetch(0, mn, e_n, sc_n);
            for (int q = 0; q < cnt; ++q) {
#pragma unroll
                for (int j = 0; j < KP; ++j) m[j] = mn[j];
                e_c = e_n; sc_c = sc_n;
                double* line = lines[q & 1];
                line[lane] = a * e_c;
                __syncwarp();
                if (q + 1 < cnt) fetch(q + 1, mn, e_n, sc_n);
                double n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0, w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
                const double2* lp = reinterpret_cast<const double2*>(line);
                if (KP >= 4) {
#pragma unroll
                    for (int j = 0; j < KP / 4; ++j) {
                        const double2 u = lp[2 * j], v = lp[2 * j + 1];
                        n0 = fma(u.x, m[4 * j], n0);     w0 += u.x;
                        n1 = fma(u.y, m[4 * j + 1], n1); w1 += u.y;
                        n2 = fma(v.x, m[4 * j + 2], n2); w2 += v.x;
                        n3 = fma(v.y, m[4 * j + 3], n3); w3 += v.y;
                    }
                } else {
                    const double2 u = lp[0];
                    n0 = fma(u.x, m[0], n0); w0 += u.x;
                    n1 = fma(u.y, m[1], n1); w1 += u.y;
                }
                const double nv = (n0 + n1) + (n2 + n3);
                const int64_t o = out_of(s_lo + s0 + q);
                if (FWD) {
                    const double wsum = (w0 + w1) + (w2 + w3);
                    // the reciprocal runs beside the dot product.  wsum == 0 only in mode 1: a unit start state that the
                    // first chunk makes impossible — its row is exactly zero with log scale -inf, as in phase A
                    a = nv * (wsum > 0.0 ? 1.0 / wsum : 0.0);
                    if (lv.mode == 1) lsacc += log(wsum);              // off the dependent chain (a does not wait for it)
                } else {
                    a = nv * sc_c;
                }
                if (lv.mode != 1 && mine) lv.vb[o * K + lane] = a;
            }
        }
        __syncthreads();
    }
    if (lv.mode == 1 && warp == 0) {
        // row blockIdx.y of this group's transfer matrix: the end vector of the run from that unit vector (+ its log scale)
        const int64_t row = (int64_t)grp * K + blockIdx.y;
        if (mine) lv.tg[row * K + lane] = a;
        if (lane == 0) lv.lsg[row] = FWD ? lsacc : 0.0;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Phase C', backward: the recursion over one chunk (descending i) from its boundary vector w[c] (ones where a sequence
// ends); gamma, the xi sum S[j][k] = sum_i alpha_{i-1}[j] rho_i[k] beta_i[k] / c_i (A~ is applied once at the end),
// sum gamma ln rho, gamma_0, optionally beta.  Lane kk owns state kk and ROW kk of A~.
template <int KP, bool SEQS>
__global__ void __launch_bounds__(HT) hmm_bwd_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                     double* __restrict__ hst, const HmmLayout H, const int force,
                                                     const ScanBufs B, const SeqArg<SEQS> T) {
    __shared__ __align__(16) double lines[HW][2][32];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    constexpr int G = 32 / KP;
    const int K = sp.K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, kk = lane % KP, grp = lane / KP;
    const double* at = current_at(st, L, hst, H);
    const double* __restrict__ lnrho = B.lnrho;
    const double* __restrict__ rhohat = B.rhohat;
    const double* __restrict__ alpha = B.alpha;
    const double* __restrict__ cs = B.ichat;                 // rho_i / c_i = rhohat_i * (1 / chat_i)
    const int64_t item = ((int64_t)blockIdx.x * HW + warp) * G + grp;
    const int c = (int)item;
    ChunkInfo ci{};
    if constexpr (SEQS) ci = chunk_info(sp, T, c);
    const bool live = item < sp.nch, mine = live && kk < K;
    if (SEQS && !__any_sync(0xffffffffu, live)) return;
    double arow[KP], srow[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) arow[k] = (mine && k < K) ? at[kk * K + k] : 0.0;
#pragma unroll
    for (int k = 0; k < KP; ++k) srow[k] = 0.0;
    const int64_t i0 = SEQS ? ci.i0 : (int64_t)c * sp.L;
    const int64_t i1 = (SEQS ? ci.i1 : (i0 + sp.L < sp.n ? i0 + sp.L : sp.n)) - 1;   // last element of the chunk
    const int nst = SEQS ? warp_steps(live, ci) : sp.L;
    double b = 0.0;
    if (SEQS && ci.i1 == ci.s1) b = mine ? 1.0 : 0.0;                   // a sequence ends (:939)
    else if (mine) b = B.vb[(int64_t)c * K + kk];
    double gl = 0.0;
    // loads run two steps ahead, exp / reciprocal one step ahead of the dependent chain (which runs through b only)
    auto LR = [&](int64_t i) { return (mine && i >= i0) ? lnrho[i * K + kk] : 0.0; };
    auto RH = [&](int64_t i) { return (mine && i >= i0) ? rhohat[i * K + kk] : 0.0; };
    auto CI = [&](int64_t i) { return (live && i >= i0) ? cs[i] : 1.0; };
    auto AL = [&](int64_t i) { return (mine && i >= 0) ? alpha[i * K + kk] : 0.0; };
    double lr_c = LR(i1), rho_c = RH(i1), inv_c = CI(i1);
    double lr_n = LR(i1 - 1), rho_n = RH(i1 - 1), ci_n = CI(i1 - 1);
    double al_c = AL(i1), al_p = AL(i1 - 1), al_pp = AL(i1 - 2);
    for (int s = 0; s < nst; ++s) {
        const int64_t i = i1 - s;
        const bool in = live && i >= i0, on = mine && i >= i0;
        const double lr = lr_c, rho = rho_c, inv = inv_c, al = al_c, aprev = al_p;
        lr_c = lr_n; rho_c = rho_n; inv_c = ci_n;
        lr_n = LR(i - 2); rho_n = RH(i - 2); ci_n = CI(i - 2);
        al_c = al_p; al_p = al_pp; al_pp = AL(i - 3);
        const double rb = on ? rho * b : 0.0;                          // rho_i[k] beta_i[k]
        if (on) {
            const double g = al * b;                                   // :1014
            B.gamma[i * K + kk] = g;
            if (B.beta_out != nullptr) B.beta_out[i * K + kk] = b;
            gl = fma(g, lr, gl);
            if constexpr (!SEQS) {
                if (i == 0) hst[H.g0 + kk] = g;
            } else {
                if (i == ci.s0) T.pg0[(int64_t)c * K + kk] = g;        // summed over sequence starts: hmm_reduce_kernel
            }
        }
        double* line = lines[warp][s & 1];
        publish<KP>(line, lane, rb);
        const double dot = group_dot<KP>(line, grp * KP, arow);        // (A~ (rho o beta))[kk]
        // alpha_{i-1}[kk] / c_i (:1017-1018); xi = 0 at a (sequence) start
        const double f = (on && (SEQS ? i > ci.s0 : i >= 1)) ? aprev * inv : 0.0;
        const double2* p = reinterpret_cast<const double2*>(line + grp * KP);
#pragma unroll
        for (int k2 = 0; k2 < KP / 2; ++k2) {
            const double2 vv = p[k2];
            srow[2 * k2] = fma(f, vv.x, srow[2 * k2]);
            srow[2 * k2 + 1] = fma(f, vv.y, srow[2 * k2 + 1]);
        }
        if (in) b = dot * inv;                                         // :1010-1011
    }
    if (mine) {
#pragma unroll
        for (int k = 0; k < KP; ++k)
            if (k < K) B.ps[((int64_t)c * K + kk) * K + k] = srow[k];
    }
    const double t = group_sum<KP>(gl);
    if (live && kk == 0) B.pgl[c] = t;
}

// Phase A / A' on the FP64 tensor pipe, for every K (K <= 8 runs as KP = 8, zero-padded).  The K basis runs of a chunk
// are ONE matrix recursion: with row j0 of S the message vector started from unit vector j0,
//     forward :  S <- (S . A~) o rho_i          (column scaling; `_hiddenmarkovnormal.py` :999-1004 applied to K vectors)
//     backward:  S <- ((S o rho_i) . A~^T) / chat_i                                              (:1010-1011)
// i.e. a right-multiplication by a CONSTANT matrix per step.  One warp owns one chunk and keeps S in DMMA accumulator
// fragments (m8n8k4: lane (r, q) holds S[8 mb + r][8 nb + 2 q + e], e = 0, 1).  The same registers are the A operand of
// the next step: for fixed (kb, e) they form an 8 x 4 tile over the columns k = 8 kb + 2 q + e, a permuted k-block, and the
// sum over k does not care about the order as long as the constant B fragments use the same rows — so there is no
// layout conversion, no shuffle and no shared memory in the step: (KP/8)^3 * 2 DMMAs (128 at K = 32) + KP scalings.
// As K separate vector recursions the same 2 K^3 flops per element would be K dependent mat-vec chains through shared
// memory; this form is bound by the DMMA pipe.  Rows are renormalised every 8 steps (and at the end of a forward chunk:
// phase B relies on rows summing to one); a row whose sum is exactly zero (its start state is impossible) stays exactly
// zero with log scale -inf, so it weighs nothing in phase B.
template <int KP, bool FWD, bool SEQS>
__global__ void __launch_bounds__(HT, KP >= 32 ? 1 : 4) hmm_basis_mma_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                              const double* __restrict__ hst, const HmmLayout H,
                                                              const int force, const ScanBufs B, const SeqArg<SEQS> T) {
    constexpr int NB = KP / 8;
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    if (hmm_window(st, L, hst, H, sp) > 0) return;
    const int K = sp.K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, r = lane >> 2, q = lane & 3;
    const int64_t item = (int64_t)blockIdx.x * HW + warp;
    if (item >= sp.nch - 1) return;                               // whole warps only: no block barrier below
    const int c = FWD ? (int)item : 1 + (int)item;                // forward: chunks 0 .. nch-2, backward: 1 .. nch-1
    ChunkInfo ci{};
    if constexpr (SEQS) ci = chunk_info(sp, T, c);
    if (SEQS && (FWD ? ci.i1 == ci.s1 : ci.i0 == ci.s0)) return;           // the sequence ends / starts here: no neighbour to feed
    const double* at = current_at(st, L, hst, H);
    const double* __restrict__ rhohat = B.rhohat;
    const double* __restrict__ ichat = B.ichat;
    // constant B fragments: R[k][n] with k = 8 kb + 2 q + e, n = 8 nb + r;  R = A~ (forward) or A~^T (backward)
    double bc[NB][2][NB];
#pragma unroll
    for (int kb = 0; kb < NB; ++kb)
#pragma unroll
        for (int e = 0; e < 2; ++e)
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
                const int k = 8 * kb + 2 * q + e, n = 8 * nb + r;
                bc[kb][e][nb] = (k < K && n < K) ? (FWD ? at[k * K + n] : at[n * K + k]) : 0.0;
            }
    double sm[NB][NB][2], slog[NB];
#pragma unroll
    for (int mb = 0; mb < NB; ++mb) {
        slog[mb] = 0.0;
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int row = 8 * mb + r, col = 8 * nb + 2 * q + e;
                sm[mb][nb][e] = (row == col && row < K) ? 1.0 : 0.0;
            }
    }
    const int64_t i0 = SEQS ? ci.i0 : (int64_t)c * sp.L;
    const int64_t i1 = (SEQS ? ci.i1 : (i0 + sp.L < sp.n ? i0 + sp.L : sp.n)) - 1;
    const int nsteps = (int)(i1 - i0 + 1);
    // emission values (this lane's 2 NB columns) two steps ahead of the dependent chain
    auto load_rho = [&](int s, double (&dst)[NB][2]) {
        const int64_t i = FWD ? i0 + s : i1 - s;
        const bool ok = s < nsteps;
        const double sc = FWD ? 1.0 : (ok ? ichat[i] : 0.0);
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int col = 8 * nb + 2 * q + e;
                dst[nb][e] = (ok && col < K) ? rhohat[i * K + col] * sc : 0.0;
            }
    };
    double rc[NB][2], rn[NB][2];
    load_rho(0, rc);
    load_rho(1, rn);
    for (int s = 0; s < nsteps; ++s) {
        double rho[NB][2];
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 2; ++e) { rho[nb][e] = rc[nb][e]; rc[nb][e] = rn[nb][e]; }
        load_rho(s + 2, rn);
        const bool no_transition = FWD && i0 + s == (SEQS ? ci.s0 : 0);   // :1000 — the first element has no transition
#pragma unroll
        for (int mb = 0; mb < NB; ++mb) {
            if (!FWD) {
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) { sm[mb][nb][0] *= rho[nb][0]; sm[mb][nb][1] *= rho[nb][1]; }
            }
            if (!no_transition) {
                double o[NB][2];
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) { o[nb][0] = 0.0; o[nb][1] = 0.0; }
#pragma unroll
                for (int kb = 0; kb < NB; ++kb)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb) dmma(o[nb][0], o[nb][1], sm[mb][kb][e], bc[kb][e][nb]);
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) { sm[mb][nb][0] = o[nb][0]; sm[mb][nb][1] = o[nb][1]; }
            }
            if (FWD) {
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) { sm[mb][nb][0] *= rho[nb][0]; sm[mb][nb][1] *= rho[nb][1]; }
            }
        }
        if ((s & 7) == 7 || (FWD && s == nsteps - 1)) {
#pragma unroll
            for (int mb = 0; mb < NB; ++mb) {
                double sum = 0.0;
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) sum += sm[mb][nb][0] + sm[mb][nb][1];
                sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                if (sum > 0.0) {
                    const double inv = 1.0 / sum;
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) { sm[mb][nb][0] *= inv; sm[mb][nb][1] *= inv; }
                    slog[mb] += log(sum);
                } else {
                    // impossible start (forward) / end (backward) state: exactly zero response, log scale -inf
#pragma unroll
                    for (int nb = 0; nb < NB; ++nb) { sm[mb][nb][0] = 0.0; sm[mb][nb][1] = 0.0; }
                    slog[mb] = -INFINITY;
                }
            }
        }
    }
#pragma unroll
    for (int mb = 0; mb < NB; ++mb) {
        const int j0 = 8 * mb + r;
        if (j0 < K) {
#pragma unroll
            for (int nb = 0; nb < NB; ++nb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int col = 8 * nb + 2 * q + e;
                    if (col < K) B.tf[((int64_t)c * K + j0) * K + col] = sm[mb][nb][e];
                }
            if (q == 0) B.ls[(int64_t)c * K + j0] = slog[mb];
        }
    }
}

// Mixing mode: the boundary vector of every chunk from a warm-up window of W elements (see hmm_window).
//   FWD : v[c] = normalised alpha at element cL-1, run over [cL-W, cL-1] from a flat vector (from pi~ when the window
//         reaches element 0, where the first element has no transition: then it is the exact recursion);
//   !FWD: w[c] = beta at the last element e of chunk c, un-normalised run from ones over [e+1, e+W] (exact when the
//         window reaches element N-1, where beta = 1, :939).
template <int KP, bool FWD, bool SEQS>
__global__ void __launch_bounds__(HT) hmm_window_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                        double* hst, const HmmLayout H,
                                                        const int force, const ScanBufs B, const SeqArg<SEQS> T) {
    __shared__ __align__(16) double lines[HW][2][32];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    const int W = hmm_window(st, L, hst, H, sp);
    if (FWD && blockIdx.x == 0 && threadIdx.x == 0) hst[H.sc + 2] = (double)W;   // diagnostics: the path taken
    if (W <= 0) return;
    constexpr int G = 32 / KP;
    const int K = sp.K, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, kk = lane % KP, grp = lane / KP;
    const double* at = current_at(st, L, hst, H);
    const double* __restrict__ rhohat = B.rhohat;
    const double* __restrict__ chat = B.ichat;             // 1 / chat_i
    const int c = (int)(((int64_t)blockIdx.x * HW + warp) * G + grp);
    const bool live = c < sp.nch, mine = live && kk < K;
    ChunkInfo ci{};
    if constexpr (SEQS) ci = chunk_info(sp, T, c);
    // a chunk that starts (FWD) / ends (!FWD) its sequence takes the exact vector there, pi~ / ones: no window to run
    const bool edge = SEQS ? (FWD ? ci.i0 == ci.s0 : ci.i1 == ci.s1) : (FWD && c == 0);
    if (SEQS && !__any_sync(0xffffffffu, live && !edge)) {
        if (mine) B.vb[(int64_t)c * K + kk] = FWD ? pi_tilde(st, L, K, kk) : 1.0;
        return;
    }
    double av[KP];                                          // FWD: column kk of A~;  !FWD: row kk
#pragma unroll
    for (int j = 0; j < KP; ++j) av[j] = (mine && j < K) ? (FWD ? at[j * K + kk] : at[kk * K + j]) : 0.0;
    // The window is walked in blocks of 8 steps: the 8 emission values (and normalisers) of the NEXT block are in flight
    // while this block runs, so the global-load latency is spread over 8 steps of the dependent chain.
    const int WB = (W + 7) >> 3;
    if (FWD) {
        const double* Pc = st + L.params[ctrl[BGMM_CTRL_CUR]];
        double pmax = -INFINITY;
        for (int k = 0; k < K; ++k) pmax = fmax(pmax, Pc[L.p_elnpi + k]);
        const double pt = (kk < K) ? exp(Pc[L.p_elnpi + kk] - pmax) : 0.0;      // pi~ (:849)
        const int64_t S = SEQS ? ci.s0 : 0;                 // the window is clamped to the chunk's sequence
        const int64_t end = (SEQS ? ci.i0 : (int64_t)c * sp.L) - 1;   // last element before chunk c
        const int64_t first = end - 8 * (int64_t)WB + 1;    // first element of the window (may be < S)
        double a = mine ? (first <= S ? pt : 1.0) : 0.0;
        auto RH = [&](int64_t i) { return (mine && i >= S && i <= end) ? rhohat[i * K + kk] : 0.0; };
        double rc[8], rn[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) rn[t] = RH(first + t);
        for (int blk = 0; blk < WB; ++blk) {
            const int64_t ib = first + 8 * (int64_t)blk;
#pragma unroll
            for (int t = 0; t < 8; ++t) rc[t] = rn[t];
            if (blk + 1 < WB) {
#pragma unroll
                for (int t = 0; t < 8; ++t) rn[t] = RH(ib + 8 + t);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int64_t i = ib + t;
                double* line = lines[warp][t & 1];
                publish<KP>(line, lane, a);
                const double dot = group_dot<KP>(line, grp * KP, av);
                const double u = rc[t] * (i == S ? a : dot);
                const bool on = live && i >= S;
                if (t == 7) {
                    const double sum = group_sum<KP>(u);
                    if (on) a = u / sum;
                } else if (on) {
                    a = u;
                }
            }
        }
        if (mine) B.vb[(int64_t)c * K + kk] = edge ? pt : a;
    } else {
        const int64_t e = (SEQS ? ci.i1 : ((int64_t)(c + 1) * sp.L < sp.n ? (int64_t)(c + 1) * sp.L : sp.n)) - 1;   // last element of chunk c
        const int64_t S1 = SEQS ? ci.s1 : sp.n;             // end of its sequence: the window is clamped there
        const int64_t top = e + 8 * (int64_t)WB;            // first element visited (may be > S1-1)
        double b = mine ? 1.0 : 0.0;
        auto RH = [&](int64_t i) { return (mine && i > e && i < S1) ? rhohat[i * K + kk] : 0.0; };
        auto CI = [&](int64_t i) { return (live && i > e && i < S1) ? chat[i] : 1.0; };
        double rc[8], rn[8], ic[8], cn[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) { rn[t] = RH(top - t); cn[t] = CI(top - t); }
        for (int blk = 0; blk < WB; ++blk) {
            const int64_t ib = top - 8 * (int64_t)blk;
#pragma unroll
            for (int t = 0; t < 8; ++t) { rc[t] = rn[t]; ic[t] = cn[t]; }
            if (blk + 1 < WB) {
#pragma unroll
                for (int t = 0; t < 8; ++t) { rn[t] = RH(ib - 8 - t); cn[t] = CI(ib - 8 - t); }
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int64_t i = ib - t;
                const bool on = live && i > e && i < S1;
                double* line = lines[warp][t & 1];
                publish<KP>(line, lane, on ? rc[t] * b : 0.0);
                const double dot = group_dot<KP>(line, grp * KP, av);
                if (on) b = dot * ic[t];                    // :1010-1011
            }
        }
        if (mine) B.vb[(int64_t)c * K + kk] = b;
    }
}

// ms[j][k] = A~[j][k] * sum_c S_c[j][k] (:839 with :1017), sc[0] = sum_i ln c_i, sc[1] = sum gamma ln rho; fixed order.
// SEQS: also G0 = sum over the sequence starts of gamma there.
template <bool SEQS>
__global__ void __launch_bounds__(256) hmm_reduce_kernel(const ScanPlan sp, const double* __restrict__ st, const Layout L,
                                                         double* __restrict__ hst, const HmmLayout H, const int force,
                                                         const ScanBufs B, const SeqArg<SEQS> T) {
    __shared__ double part[8][32];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    const double* at = current_at(st, L, hst, H);
    const int KK = sp.K * sp.K, e = blockIdx.x * 32 + (threadIdx.x & 31), sl = threadIdx.x >> 5;
    double acc = 0.0;
    if (e < KK) {
        for (int c = sl; c < sp.nch; c += 8) acc += B.ps[(int64_t)c * KK + e];
    } else if (e == KK) {
        for (int c = sl; c < sp.nch; c += 8) acc += B.plc[c];
    } else if (e == KK + 1) {
        for (int c = sl; c < sp.nch; c += 8) acc += B.pgl[c];
    } else if (SEQS && e < KK + 2 + sp.K) {
        if constexpr (SEQS) {
            for (int c = sl; c < sp.nch; c += 8)
                if (T.coff[c] == T.sst[c]) acc += T.pg0[(int64_t)c * sp.K + (e - KK - 2)];
        }
    }
    part[sl][threadIdx.x & 31] = acc;
    __syncthreads();
    if (sl == 0) {
        double t = 0.0;
        for (int s = 0; s < 8; ++s) t += part[s][threadIdx.x];
        if (e < KK) hst[H.ms + e] = at[e] * t;
        else if (e == KK) hst[H.sc + 0] = t;
        else if (e == KK + 1) hst[H.sc + 1] = t;
        else if (SEQS && e < KK + 2 + sp.K) hst[H.g0 + (e - KK - 2)] = t;
    }
}

static int64_t scan_ws_doubles(int K, int64_t n, int64_t nch) {
    const int64_t KK = (int64_t)K * K;
    // transfer matrices + log scales + boundary vectors + S partials + the two scalar partial arrays
    // + rhohat [n][K], row max [n], chat [n]
    // + the two-level sweep's group matrices, log scales and boundary vectors (<= 64 + 1 groups)
    return nch * KK + nch * K + nch * K + nch * KK + 2 * nch + 64 + n * K + 3 * n + 72 * (KK + 2 * K) + 2;
}

// Phase B of one direction over nsteps chunk matrices: the single-CTA sweep, or (>= 4 groups of SEQ_GLEN steps) group
// matrices -> group sweep -> expansion
static bool two_level_sweep(int64_t nsteps) { return (nsteps + SEQ_GLEN - 1) / SEQ_GLEN >= 4; }

// the sweep over chunks [cbase, cbase + nsteps] (cbase = 0 unless SEQS)
template <int KP, bool FWD, bool SEQS>
static void launch_seq(const ScanPlan& sp, double* st, const Layout& L, double* hst, const HmmLayout& H, int force,
                       const ScanBufs& B, size_t smem_seq, cudaStream_t stream, int cbase, int nsteps) {
    const int K = sp.K;
    const int ngroups = (nsteps + SEQ_GLEN - 1) / SEQ_GLEN;
    SeqLevel lv{0, nsteps, ngroups, B.tf, B.ls, B.vb, nullptr, nullptr, nullptr};
    SeqRangeArg<SEQS> R{};
    if constexpr (SEQS) R = SeqRange{cbase, nullptr};
    if (!two_level_sweep(nsteps)) {
        launch(hmm_seq_kernel<KP, FWD, SEQS>, 1, SEQ_T, smem_seq, stream, sp, st, L, hst, H, force, lv, R);
        return;
    }
    double* tg = B.seq2;                                   // [ngroups][K][K]
    double* lsg = tg + (int64_t)72 * K * K;                // [ngroups][K]
    double* vbg = lsg + (int64_t)72 * K;                   // [ngroups + 1][K]
    lv.mode = 1; lv.tg = tg; lv.lsg = lsg;
    launch(hmm_seq_kernel<KP, FWD, SEQS>, dim3(ngroups, K), SEQ_T, smem_seq, stream, sp, st, L, hst, H, force, lv, R);
    SeqLevel l2{2, ngroups - 1, ngroups, tg, lsg, vbg, nullptr, nullptr, nullptr};   // the last group's matrix is not needed
    launch(hmm_seq_kernel<KP, FWD, SEQS>, 1, SEQ_T, smem_seq, stream, sp, st, L, hst, H, force, l2, SeqRangeArg<SEQS>{});   // group level: cbase 0
    lv.mode = 3; lv.tg = nullptr; lv.lsg = nullptr; lv.vbg = vbg;
    launch(hmm_seq_kernel<KP, FWD, SEQS>, ngroups, SEQ_T, smem_seq, stream, sp, st, L, hst, H, force, lv, R);
}

// Phase B of one direction over several sequences: sequences of one chunk need none; the others are swept in parallel
// (one CTA each, segmented), except those long enough for the two-level sweep, which get it one after another.
// plan: see bgmm_hmm_seq_plan.
template <int KP, bool FWD>
static void launch_seq_segs(const ScanPlan& sp, double* st, const Layout& L, double* hst, const HmmLayout& H, int force,
                            const ScanBufs& B, size_t smem_seq, cudaStream_t stream, const int64_t* plan,
                            const int64_t* segs_dev) {
    const int64_t nshort = plan[4], nlong = plan[5];
    const int64_t* segs = plan + 8 + 3 * plan[3] + 1;
    if (nshort > 0) {
        SeqLevel lv{0, 0, 0, B.tf, B.ls, B.vb, nullptr, nullptr, nullptr};
        launch(hmm_seq_kernel<KP, FWD, true>, (unsigned)nshort, SEQ_T, smem_seq, stream, sp, st, L, hst, H, force, lv,
               SeqRange{0, segs_dev});
    }
    for (int64_t q = nshort; q < nshort + nlong; ++q)
        launch_seq<KP, FWD, true>(sp, st, L, hst, H, force, B, smem_seq, stream, (int)segs[2 * q], (int)segs[2 * q + 1] - 1);
}

// plan: NULL for one sequence, else the host copy of bgmm_hmm_seq_plan's table (segs_dev: its segment list on the device)
template <int KP, bool SEQS>
static int launch_scan(const ScanPlan& sp, double* st, const Layout& L, double* hst, const HmmLayout& H, int force,
                       const ScanBufs& B, const SeqArg<SEQS>& T, cudaStream_t stream, const int64_t* plan,
                       const int64_t* segs_dev) {
    constexpr int G = 32 / KP;
    const int per_cta = HW * G;
    const unsigned gc = (unsigned)((sp.nch + per_cta - 1) / per_cta);
    const size_t smem_seq = (size_t)2 * seq_batch(sp.K) * (sp.K * sp.K + sp.K + 8) * sizeof(double);
    {   // per launch: the attribute is per device
        cudaError_t e = cudaFuncSetAttribute(hmm_seq_kernel<KP, true, SEQS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(hmm_seq_kernel<KP, false, SEQS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(hmm_seq)");
    }
    // boundary vectors: either {basis runs, sequential sweep} or {one warm-up window per chunk}; the device decides
    // (hmm_window) from the current A~, the kernels of the other branch return at once
    const unsigned gm = (unsigned)((sp.nch - 1 + HW - 1) / HW);          // basis runs: one warp per chunk
    // basis runs and sweeps only where a sequence has more than one chunk
    const bool multi = plan == nullptr ? sp.nch > 1 : plan[4] + plan[5] > 0;
    if (multi) launch(hmm_basis_mma_kernel<(KP >= 8 ? KP : 8), true, SEQS>, gm, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    if (plan == nullptr) launch_seq<KP, true, false>(sp, st, L, hst, H, force, B, smem_seq, stream, 0, sp.nch - 1);
    else launch_seq_segs<KP, true>(sp, st, L, hst, H, force, B, smem_seq, stream, plan, segs_dev);
    launch(hmm_window_kernel<KP, true, SEQS>, gc, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    launch(hmm_fwd_kernel<KP, SEQS>, gc, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    launch(hmm_cs_kernel<SEQS>, sp.nch, 128, 0, stream, sp, st, L, force, B, T);
    if (multi) launch(hmm_basis_mma_kernel<(KP >= 8 ? KP : 8), false, SEQS>, gm, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    if (plan == nullptr) launch_seq<KP, false, false>(sp, st, L, hst, H, force, B, smem_seq, stream, 0, sp.nch - 1);
    else launch_seq_segs<KP, false>(sp, st, L, hst, H, force, B, smem_seq, stream, plan, segs_dev);
    launch(hmm_window_kernel<KP, false, SEQS>, gc, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    launch(hmm_bwd_kernel<KP, SEQS>, gc, HT, 0, stream, sp, st, L, hst, H, force, B, T);
    const int nred = sp.K * sp.K + 2 + (SEQS ? sp.K : 0);
    launch(hmm_reduce_kernel<SEQS>, (nred + 31) / 32, 256, 0, stream, sp, st, L, hst, H, force, B, T);
    return check_cuda(cudaGetLastError(), "hmm scan launch");
}

// ---------------------------------------------------------------------------------------------------------------
// Emission pass for small D (<= 8): `_calc_rho` :988-996 as ln rho[n][k] = coef_k . phi(x'_n), one thread per element.
// The tiled large-regime kernel is tile-latency bound at these sizes (a 64-row tile is a few KB); here the coefficient
// rows are broadcast from shared memory, phi(x) (P = 1 + D + D(D+1)/2 <= 45 values) lives in registers and the kernel
// streams x once and writes ln rho, rhohat = exp(ln rho - row max) and the row max: HBM bound.
template <int D>
__global__ void __launch_bounds__(256, 2) hmm_emit_small_kernel(const double* __restrict__ x, const int64_t n, const int K,
                                                                const double* __restrict__ st, const Layout L,
                                                                const int force, double* __restrict__ lnrho,
                                                                double* __restrict__ rhohat, double* __restrict__ rowmax) {
    constexpr int P = 1 + D + D * (D + 1) / 2;
    constexpr int PP = (P + 1) & ~1;                        // even pitch: rows of cf stay 16-byte aligned
    __shared__ __align__(16) double cf[32 * PP];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (!force && ctrl[BGMM_CTRL_DONE]) return;
    const double* __restrict__ coef = st + L.params[ctrl[BGMM_CTRL_CUR]] + L.p_coef;
    for (int e = threadIdx.x; e < K * PP; e += 256) {
        const int k = e / PP, p = e - k * PP;
        cf[e] = p < P ? coef[(int64_t)k * L.pitch + p] : 0.0;
    }
    __syncthreads();
    // a warp owns 32 consecutive elements: its [32][K] block of ln rho / rhohat is contiguous in memory, so the values are
    // staged in shared memory (odd pitch) and written out with consecutive lanes on consecutive addresses
    extern __shared__ __align__(16) double stage_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, KS = K | 1;
    double* stg = stage_raw + (size_t)warp * (32 * KS + 32);
    double* mxs = stg + 32 * KS;
    for (int64_t base = (int64_t)blockIdx.x * 256 + warp * 32; base < n; base += (int64_t)gridDim.x * 256) {
        const int64_t row = base + lane;
        const bool valid = row < n;
        double phi[PP];
        phi[0] = 1.0;
        if (PP > P) phi[PP - 1] = 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i) phi[1 + i] = valid ? x[row * D + i] : 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) phi[1 + D + i * (i + 1) / 2 + j] = phi[1 + i] * phi[1 + j];
        double mx = -INFINITY;
#pragma unroll 1
        for (int k = 0; k < K; ++k) {                       // the component loop stays rolled: phi is the register budget
            const double2* c2 = reinterpret_cast<const double2*>(cf + k * PP);
            double a0 = 0.0, a1 = 0.0;
#pragma unroll
            for (int p = 0; p < PP / 2; ++p) {
                const double2 c = c2[p];
                a0 = fma(c.x, phi[2 * p], a0);
                a1 = fma(c.y, phi[2 * p + 1], a1);
            }
            const double lr = a0 + a1;
            stg[lane * KS + k] = lr;
            mx = fmax(mx, lr);
        }
        mxs[lane] = mx;
        if (rowmax != nullptr && valid) rowmax[row] = mx;
        __syncwarp();
        const int64_t lim = (n - base < 32 ? n - base : 32) * K;
        for (int e = lane; e < lim; e += 32) {
            const int r = e / K, k = e - r * K;
            const double lr = stg[r * KS + k];
            lnrho[base * K + e] = lr;
            if (rhohat != nullptr) rhohat[base * K + e] = exp_nonpos(lr - mxs[r]);
        }
        __syncwarp();
    }
}

template <int D>
static int launch_emit_small_d(const void* x, int64_t n, int K, const double* st, const Layout& L, int force, double* lnrho,
                               double* rhohat, double* rowmax, cudaStream_t s) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int64_t g = (n + 255) / 256;
    if (g > (int64_t)sms * 8) g = (int64_t)sms * 8;
    const size_t smem = (size_t)8 * (32 * (K | 1) + 32) * sizeof(double);
    cudaError_t e = cudaFuncSetAttribute(hmm_emit_small_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(hmm_emit_small)");
    launch(hmm_emit_small_kernel<D>, (unsigned)g, 256, smem, s, static_cast<const double*>(x), n, K, st, L, force, lnrho, rhohat,
           rowmax);
    return check_cuda(cudaGetLastError(), "hmm_emit_small launch");
}

// D <= 8 and K <= 32: the thread-per-element kernel; otherwise -1 (the caller uses the large-regime E kernel)
static int launch_emit_small(const void* x, int64_t n, int K, int D, const double* st, const Layout& L, int force,
                             double* lnrho, double* rhohat, double* rowmax, cudaStream_t s) {
    if (K > 32) return -1;
    switch (D) {
        case 1: return launch_emit_small_d<1>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 2: return launch_emit_small_d<2>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 3: return launch_emit_small_d<3>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 4: return launch_emit_small_d<4>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 5: return launch_emit_small_d<5>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 6: return launch_emit_small_d<6>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 7: return launch_emit_small_d<7>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        case 8: return launch_emit_small_d<8>(x, n, K, st, L, force, lnrho, rhohat, rowmax, s);
        default: return -1;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Viterbi (_hiddenmarkovnormal.py:1466-1480): omega_0 = ln rho_0 + ln pi~;  omega_i[k] = ln rho_i[k] + max_j (ln a~_jk +
// omega_{i-1}[j]), phi_i[k] = argmax_j (first maximum, as np.argmax); then the path is traced back from argmax omega_{N-1}.
// The recursion is sequential in i and is kept in the reference's operation order (same additions, same comparison order),
// so omega / phi / the path are bit-identical to numpy's for identical ln rho.  One CTA: warps 1..3 stage ln rho tiles
// into shared memory (cp.async, double buffered), warp 0 runs the recursion (lane k owns state k and column k of ln a~).
constexpr int VT_TILE = 256;       // steps per staged tile
template <int KP>
__global__ void __launch_bounds__(SEQ_T) hmm_viterbi_fwd_kernel(const int64_t n, const int K, const double* __restrict__ lnrho,
                                                                const double* __restrict__ lnpi,
                                                                const double* __restrict__ lna, double* __restrict__ omega,
                                                                int32_t* __restrict__ phi) {
    extern __shared__ __align__(16) double vt[];            // [2][VT_TILE][K]
    __shared__ __align__(16) double lines[2][32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool mine = lane < K;
    const int64_t ntile = (n + VT_TILE - 1) / VT_TILE;
    auto load_tile = [&](int64_t t, int t0, int nt) {
        double* dst = vt + (size_t)(t & 1) * VT_TILE * K;
        const int64_t base = t * VT_TILE * K;
        const int64_t cnt = (t * VT_TILE + VT_TILE <= n ? (int64_t)VT_TILE : n - t * VT_TILE) * K;
        for (int64_t e = tid - t0; e < cnt; e += nt) cp_async8(dst + e, lnrho + base + e);
        asm volatile("cp.async.wait_all;" ::: "memory");
    };
    double acol[KP];
#pragma unroll
    for (int j = 0; j < KP; ++j) acol[j] = (mine && j < K) ? lna[j * K + lane] : -INFINITY;
    double om = 0.0;
    load_tile(0, 0, SEQ_T);
    __syncthreads();
    for (int64_t t = 0; t < ntile; ++t) {
        if (warp > 0) {
            if (t + 1 < ntile) load_tile(t + 1, 32, SEQ_T - 32);
        } else {
            const double* src = vt + (size_t)(t & 1) * VT_TILE * K;
            const int cnt = (int)(t * VT_TILE + VT_TILE <= n ? (int64_t)VT_TILE : n - t * VT_TILE);
            for (int q = 0; q < cnt; ++q) {
                const int64_t i = t * VT_TILE + q;
                const double lr = mine ? src[q * K + lane] : 0.0;
                int arg = 0;
                if (i == 0) {
                    om = mine ? lr + lnpi[lane] : -INFINITY;                 // :1469
                } else {
                    double* line = lines[q & 1];
                    line[lane] = om;
                    __syncwarp();
                    double best = -INFINITY;
#pragma unroll
                    for (int j = 0; j < KP; ++j) {
                        if (j < K) {
                            const double cand = acol[j] + line[j];           // ln a~[j][k] + omega_{i-1}[j]   (:1471-1472)
                            if (j == 0 || cand > best) { best = cand; arg = j; }
                        }
                    }
                    om = lr + best;
                }
                if (mine) { omega[i * K + lane] = om; phi[i * K + lane] = arg; }
            }
        }
        __syncthreads();
    }
}

// back-tracking (:1474-1479): z_{N-1} = argmax omega_{N-1}; z_i = phi_{i+1}[z_{i+1}].  phi tiles are staged backwards.
__global__ void __launch_bounds__(SEQ_T) hmm_viterbi_back_kernel(const int64_t n, const int K, const double* __restrict__ omega,
                                                                 const int32_t* __restrict__ phi, int32_t* __restrict__ path) {
    extern __shared__ __align__(16) int32_t pt[];           // [TB][K]
    constexpr int TB = 1024;
    __shared__ int32_t zs[TB];
    const int tid = threadIdx.x;
    __shared__ int cur;
    if (tid == 0) {
        int best = 0;
        double bv = omega[(n - 1) * K];
        for (int k = 1; k < K; ++k) {
            const double v = omega[(n - 1) * K + k];
            if (v > bv) { bv = v; best = k; }
        }
        cur = best;
        path[n - 1] = best;
    }
    __syncthreads();
    // elements n-2 .. 0 in tiles of TB, highest tile first; element i needs phi[i+1]
    for (int64_t hi = n - 2; hi >= 0; hi -= TB) {
        const int64_t lo = hi - TB + 1 > 0 ? hi - TB + 1 : 0;
        const int cnt = (int)(hi - lo + 1);
        for (int64_t e = tid; e < (int64_t)cnt * K; e += SEQ_T) pt[e] = phi[(lo + 1) * K + e];       // rows lo+1 .. hi+1
        __syncthreads();
        if (tid == 0) {
            int z = cur;
            for (int q = cnt - 1; q >= 0; --q) {
                z = pt[q * K + z];
                zs[q] = z;
            }
            cur = z;
        }
        __syncthreads();
        for (int q = tid; q < cnt; q += SEQ_T) path[lo + q] = zs[q];
        __syncthreads();
    }
}

// Viterbi over several sequences: one warp per sequence (lane k owns state k and column k of ln a~), the recursion in the
// same operation order as hmm_viterbi_fwd_kernel, restarted at every sequence start (omega = ln rho + ln pi~, phi = 0),
// then lane 0 traces the path back from argmax omega at the sequence's last element.  Sequences run in parallel.
template <int KP>
__global__ void __launch_bounds__(128) hmm_viterbi_seqs_kernel(const int64_t n, const int K, const int64_t n_seqs,
                                                               const int64_t* __restrict__ starts,
                                                               const double* __restrict__ lnrho,
                                                               const double* __restrict__ lnpi,
                                                               const double* __restrict__ lna, double* __restrict__ omega,
                                                               int32_t* __restrict__ phi, int32_t* __restrict__ path) {
    __shared__ __align__(16) double lines[4][2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t q = (int64_t)blockIdx.x * 4 + warp;
    if (q >= n_seqs) return;
    const int64_t s0 = starts[q], s1 = q + 1 < n_seqs ? starts[q + 1] : n;
    const bool mine = lane < K;
    double acol[KP];
#pragma unroll
    for (int j = 0; j < KP; ++j) acol[j] = (mine && j < K) ? lna[j * K + lane] : -INFINITY;
    // ln rho two steps ahead of the dependent chain
    auto LR = [&](int64_t i) { return (mine && i < s1) ? lnrho[i * K + lane] : 0.0; };
    double lr_c = LR(s0), lr_n = LR(s0 + 1);
    double om = mine ? lr_c + lnpi[lane] : -INFINITY;                   // :1469
    if (mine) { omega[s0 * K + lane] = om; phi[s0 * K + lane] = 0; }
    for (int64_t i = s0 + 1; i < s1; ++i) {
        lr_c = lr_n;
        lr_n = LR(i + 1);
        double* line = lines[warp][i & 1];
        line[lane] = om;
        __syncwarp();
        double best = -INFINITY;
        int arg = 0;
#pragma unroll
        for (int j = 0; j < KP; ++j) {
            if (j < K) {
                const double cand = acol[j] + line[j];                   // ln a~[j][k] + omega_{i-1}[j]   (:1471-1472)
                if (j == 0 || cand > best) { best = cand; arg = j; }
            }
        }
        om = lr_c + best;
        if (mine) { omega[i * K + lane] = om; phi[i * K + lane] = arg; }
    }
    __syncwarp();                                                       // phi of the whole sequence is visible to lane 0
    if (lane == 0) {                                                    // :1474-1479
        const double* o = omega + (s1 - 1) * K;
        int z = 0;
        double bv = o[0];
        for (int k = 1; k < K; ++k)
            if (o[k] > bv) { bv = o[k]; z = k; }
        path[s1 - 1] = z;
        for (int64_t i = s1 - 2; i >= s0; --i) {
            z = phi[(i + 1) * K + z];
            path[i] = z;
        }
    }
}

}  // namespace bgmm

extern "C" int bgmm_hmm_viterbi_seqs(int64_t n, int K, const double* lnrho, const double* lnpi, const double* lna,
                                     double* omega, int32_t* phi, int32_t* path, const int64_t* seq_starts, int64_t n_seqs,
                                     void* stream) {
    using namespace bgmm;
    if (n <= 0 || K < 1 || K > 32 || n_seqs < 1 || n_seqs > n || lnrho == nullptr || lnpi == nullptr || lna == nullptr ||
        omega == nullptr || phi == nullptr || path == nullptr || seq_starts == nullptr) {
        set_error("bgmm_hmm_viterbi_seqs: bad argument (n=%lld K=%d n_seqs=%lld, K <= 32, 1 <= n_seqs <= n)", (long long)n,
                  K, (long long)n_seqs);
        return BGMM_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned g = (unsigned)((n_seqs + 3) / 4);
    if (K <= 2) launch(hmm_viterbi_seqs_kernel<2>, g, 128, 0, s, n, K, n_seqs, seq_starts, lnrho, lnpi, lna, omega, phi, path);
    else if (K <= 4) launch(hmm_viterbi_seqs_kernel<4>, g, 128, 0, s, n, K, n_seqs, seq_starts, lnrho, lnpi, lna, omega, phi, path);
    else if (K <= 8) launch(hmm_viterbi_seqs_kernel<8>, g, 128, 0, s, n, K, n_seqs, seq_starts, lnrho, lnpi, lna, omega, phi, path);
    else if (K <= 16) launch(hmm_viterbi_seqs_kernel<16>, g, 128, 0, s, n, K, n_seqs, seq_starts, lnrho, lnpi, lna, omega, phi, path);
    else launch(hmm_viterbi_seqs_kernel<32>, g, 128, 0, s, n, K, n_seqs, seq_starts, lnrho, lnpi, lna, omega, phi, path);
    return check_cuda(cudaGetLastError(), "viterbi_seqs launch");
}

extern "C" int bgmm_hmm_viterbi(int64_t n, int K, const double* lnrho, const double* lnpi, const double* lna, double* omega,
                                int32_t* phi, int32_t* path, void* stream) {
    using namespace bgmm;
    if (n <= 0 || K < 1 || K > 32 || lnrho == nullptr || lnpi == nullptr || lna == nullptr || omega == nullptr ||
        phi == nullptr || path == nullptr) {
        set_error("bgmm_hmm_viterbi: bad argument (n=%lld K=%d, K <= 32)", (long long)n, K);
        return BGMM_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t smem_f = (size_t)2 * VT_TILE * K * sizeof(double);
    const size_t smem_b = (size_t)1024 * K * sizeof(int32_t);
    cudaError_t e = cudaFuncSetAttribute(hmm_viterbi_back_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(1024 * 32 * 4));
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(viterbi_back)");
#define BGMM_VIT(KP)                                                                                                   \
    do {                                                                                                               \
        e = cudaFuncSetAttribute(hmm_viterbi_fwd_kernel<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);  \
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(viterbi_fwd)");                                \
        launch(hmm_viterbi_fwd_kernel<KP>, 1, SEQ_T, smem_f, s, n, K, lnrho, lnpi, lna, omega, phi);                     \
    } while (0)
    if (K <= 2) BGMM_VIT(2);
    else if (K <= 4) BGMM_VIT(4);
    else if (K <= 8) BGMM_VIT(8);
    else if (K <= 16) BGMM_VIT(16);
    else BGMM_VIT(32);
#undef BGMM_VIT
    launch(hmm_viterbi_back_kernel, 1, SEQ_T, smem_b, s, n, K, omega, phi, path);
    return check_cuda(cudaGetLastError(), "viterbi launch");
}

extern "C" int64_t bgmm_hmm_scan_workspace_doubles(int K, int64_t n) {
    if (K <= 0 || K > 32 || n <= 0) return 0;
    const int L = bgmm::hmm_chunk_len(n);
    return bgmm::scan_ws_doubles(K, n, (n + L - 1) / L);
}

// Several sequences: every sequence is cut into chunks of hmm_chunk_len(n), the last one shorter, so there are at most
// ceil(n / L) + n_seqs chunks; plus G0's per-chunk partials.
extern "C" int64_t bgmm_hmm_seq_workspace_doubles(int K, int64_t n, int64_t n_seqs) {
    if (K <= 0 || K > 32 || n <= 0 || n_seqs < 1 || n_seqs > n) return 0;
    const int L = bgmm::hmm_chunk_len(n);
    const int64_t nch = (n + L - 1) / L + n_seqs;
    return bgmm::scan_ws_doubles(K, n, nch) + nch * K;
}

// The chunk table of bgmm_hmm_pass_seqs (int64):
//   [0] n  [1] n_seqs  [2] L  [3] nch  [4] nshort  [5] nlong  [6] size  [7] 0
//   coff[nch + 1] | sst[nch] | sen[nch] | segs[nshort + nlong][2] | starts[n_seqs]
// chunk c = elements [coff[c], coff[c+1]) of the sequence [sst[c], sen[c]); segs = (first chunk, chunk count) of every
// sequence with more than one chunk, those swept by one CTA (nshort) before those long enough for the two-level sweep.
extern "C" int64_t bgmm_hmm_seq_plan(int64_t n, int64_t n_seqs, const int64_t* seq_starts, int64_t* plan, int64_t cap) {
    using namespace bgmm;
    if (n <= 0 || n_seqs < 1 || seq_starts == nullptr) {
        set_error("bgmm_hmm_seq_plan: bad argument (n=%lld n_seqs=%lld)", (long long)n, (long long)n_seqs);
        return BGMM_EINVAL;
    }
    if (seq_starts[0] != 0) { set_error("bgmm_hmm_seq_plan: seq_starts[0] must be 0"); return BGMM_EINVAL; }
    const int64_t L = hmm_chunk_len(n);
    int64_t nch = 0, nseg = 0;
    for (int64_t q = 0; q < n_seqs; ++q) {
        const int64_t a = seq_starts[q], b = q + 1 < n_seqs ? seq_starts[q + 1] : n;
        if (!(b > a) || b > n) {
            set_error("bgmm_hmm_seq_plan: seq_starts must increase strictly and stay below n (index %lld)", (long long)q);
            return BGMM_EINVAL;
        }
        const int64_t m = (b - a + L - 1) / L;
        nch += m;
        nseg += m > 1;
    }
    const int64_t size = 8 + 3 * nch + 1 + 2 * nseg + n_seqs;
    if (plan == nullptr || cap < size) return size;
    int64_t* coff = plan + 8;
    int64_t* sst = coff + nch + 1;
    int64_t* sen = sst + nch;
    int64_t* segs = sen + nch;
    int64_t* starts = segs + 2 * nseg;
    int64_t c = 0, ns = 0, nl = 0, nshort = 0;
    for (int64_t q = 0; q < n_seqs; ++q) {
        const int64_t m = ((q + 1 < n_seqs ? seq_starts[q + 1] : n) - seq_starts[q] + L - 1) / L;
        nshort += m > 1 && !two_level_sweep(m - 1);
    }
    for (int64_t q = 0; q < n_seqs; ++q) {
        const int64_t a = seq_starts[q], b = q + 1 < n_seqs ? seq_starts[q + 1] : n, m = (b - a + L - 1) / L;
        if (m > 1) {
            const bool lng = two_level_sweep(m - 1);
            int64_t* sg = segs + 2 * (lng ? nshort + nl++ : ns++);
            sg[0] = c;
            sg[1] = m;
        }
        for (int64_t j = 0; j < m; ++j, ++c) {
            coff[c] = a + j * L;
            sst[c] = a;
            sen[c] = b;
        }
        starts[q] = a;
    }
    coff[nch] = n;
    plan[0] = n; plan[1] = n_seqs; plan[2] = L; plan[3] = nch; plan[4] = nshort; plan[5] = nseg - nshort;
    plan[6] = size; plan[7] = 0;
    return size;
}

extern "C" int bgmm_hmm_supported(int K, int D) {
    return (K >= 1 && K <= 32 && bgmm::large_supported(K, D, BGMM_F64)) ? 1 : 0;
}

namespace bgmm {
// plan / plan_dev: NULL (one sequence), or bgmm_hmm_seq_plan's table on the host and the same table on the device
static int hmm_pass(const void* x, int64_t n, int K, int D, double* state, double* hst, double* workspace, double* scan_ws,
                    double* lnrho, double* alpha, double* gamma, double* cs, double* beta_out, int mode, int force,
                    void* stream, const int64_t* plan, const int64_t* plan_dev) {
    if (!bgmm_hmm_supported(K, D)) {
        set_error("bgmm_hmm_pass: unsupported shape K=%d D=%d (float64, K <= 32, D <= 128)", K, D);
        return BGMM_ENOSUP;
    }
    if (x == nullptr || n <= 0 || state == nullptr || hst == nullptr || workspace == nullptr ||
        (mode != BGMM_HMM_EMISSION_ONLY && gamma == nullptr) ||
        (mode == BGMM_HMM_FULL && (scan_ws == nullptr || lnrho == nullptr || alpha == nullptr || cs == nullptr))) {
        set_error("bgmm_hmm_pass: NULL buffer or n <= 0");
        return BGMM_EINVAL;
    }
    if (mode == BGMM_HMM_EMISSION_ONLY) {                        // ln rho of x under the current parameter set, nothing else
        if (lnrho == nullptr) { set_error("bgmm_hmm_pass: lnrho is NULL"); return BGMM_EINVAL; }
        const int rs = launch_emit_small(x, n, K, D, state, make_layout(K, D, 1), force, lnrho, nullptr, nullptr,
                                         (cudaStream_t)stream);
        if (rs != -1) return rs;
        PassArgs ea{x, n, state, workspace, nullptr, lnrho, nullptr, nullptr, force};
        ea.ignore_robust = 1;                                    // the hidden-Markov path has no DIRECT kernel (DESIGN §2)
        ea.lnrho_only = 1;
        return launch_pass_large_part(ea, K, D, BGMM_F64, 1, (cudaStream_t)stream);
    }
    if (mode != BGMM_HMM_FULL && mode != BGMM_HMM_STATS_FROM_GAMMA) {
        set_error("bgmm_hmm_pass: unknown mode %d", mode);
        return BGMM_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const Layout L = make_layout(K, D, 1);
    const HmmLayout H = make_hmm_layout(K);
    PassArgs a{x, n, state, workspace, nullptr, lnrho, nullptr, nullptr, force};
    a.ignore_robust = 1;
    int rc;
    if (mode == BGMM_HMM_FULL) {
        ScanPlan sp;
        sp.n = n; sp.K = K; sp.L = hmm_chunk_len(n); sp.nch = (int)((n + sp.L - 1) / sp.L);
        if (plan != nullptr) sp.nch = (int)plan[3];
        const char* wc = getenv("BGMM_HMM_WINDOW_CAP");          // tests / experiments: 0 forces the basis + sweep path
        sp.window_cap = wc != nullptr ? atoi(wc) : 16384;
        const int64_t KK = (int64_t)K * K, nch = sp.nch;
        ScanBufs B;
        B.lnrho = lnrho; B.alpha = alpha; B.gamma = gamma; B.cs = cs; B.beta_out = beta_out;
        B.tf = scan_ws; B.ls = B.tf + nch * KK; B.vb = B.ls + nch * K; B.ps = B.vb + nch * K;
        B.plc = B.ps + nch * KK; B.pgl = B.plc + nch;
        double* rh = B.pgl + nch;
        B.rhohat = rh; B.chat = rh + n * K;
        double* rmx = B.chat + n;
        B.rowmax = rmx;
        B.ichat = rmx + n;
        B.seq2 = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(B.ichat + n) + 15) & ~uintptr_t(15));   // cp.async 16
        SeqTable T{nullptr, nullptr, nullptr, nullptr};
        if (plan != nullptr) {
            T.coff = plan_dev + 8;
            T.sst = T.coff + sp.nch + 1;
            T.sen = T.sst + sp.nch;
            T.pg0 = B.seq2 + 72 * (KK + 2 * K);
        }
        a.rhohat_out = rh; a.rowmax_out = rmx;
        rc = launch_emit_small(x, n, K, D, state, L, force, lnrho, rh, rmx, s);
        if (rc == -1) {
            a.lnrho_only = 1;
            rc = launch_pass_large_part(a, K, D, BGMM_F64, 1, s);
        }
        if (rc) return rc;
        const int64_t* segs_dev = plan != nullptr ? plan_dev + 8 + 3 * plan[3] + 1 : nullptr;
#define BGMM_SCAN(KP) (plan != nullptr ? launch_scan<KP, true>(sp, state, L, hst, H, force, B, T, s, plan, segs_dev) \
                                        : launch_scan<KP, false>(sp, state, L, hst, H, force, B, NoSeqTable{}, s, nullptr, nullptr))
        if (K <= 2) rc = BGMM_SCAN(2);
        else if (K <= 4) rc = BGMM_SCAN(4);
        else if (K <= 8) rc = BGMM_SCAN(8);
        else if (K <= 16) rc = BGMM_SCAN(16);
        else rc = BGMM_SCAN(32);
#undef BGMM_SCAN
        if (rc) return rc;
    }
    a.lnrho_only = 0;
    a.lnrho_out = nullptr;
    a.r_out = gamma;
    return launch_pass_large_part(a, K, D, BGMM_F64, 2, s);
}
}  // namespace bgmm

extern "C" int bgmm_hmm_pass(const void* x, int64_t n, int K, int D, double* state, double* hst, double* workspace,
                             double* scan_ws, double* lnrho, double* alpha, double* gamma, double* cs, double* beta_out,
                             int mode, int force, void* stream) {
    return bgmm::hmm_pass(x, n, K, D, state, hst, workspace, scan_ws, lnrho, alpha, gamma, cs, beta_out, mode, force, stream,
                          nullptr, nullptr);
}

extern "C" int bgmm_hmm_pass_seqs(const void* x, int64_t n, int K, int D, double* state, double* hst, double* workspace,
                                  double* scan_ws, double* lnrho, double* alpha, double* gamma, double* cs, double* beta_out,
                                  int mode, int force, const int64_t* plan, const int64_t* plan_dev, void* stream) {
    using namespace bgmm;
    if (plan == nullptr || plan_dev == nullptr || plan[0] != n || plan[1] < 1 || plan[3] < plan[1] ||
        plan[6] != 8 + 3 * plan[3] + 1 + 2 * (plan[4] + plan[5]) + plan[1] || plan[2] != hmm_chunk_len(n)) {
        set_error("bgmm_hmm_pass_seqs: plan is NULL or not bgmm_hmm_seq_plan's table for n=%lld", (long long)n);
        return BGMM_EINVAL;
    }
    return hmm_pass(x, n, K, D, state, hst, workspace, scan_ws, lnrho, alpha, gamma, cs, beta_out, mode, force, stream,
                    plan, plan_dev);
}
