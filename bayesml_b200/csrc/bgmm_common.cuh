// Shared device/host helpers for libbgmm (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/bgmm.h"

namespace bgmm {

__host__ __device__ inline int feat_count(int D) { return 1 + D + D * (D + 1) / 2; }
__host__ __device__ inline int feat_pitch(int D) { return (feat_count(D) + 7) & ~7; }

// State-block layout (units: doubles).  Mirrors bgmm_layout(); kept in one place so kernels and host agree.
struct Layout {
    int K, D, P, pitch, hist_len;
    int64_t center, alpha0, kappa0, nu0, m0, w0inv, lnb0, lnc0, params[2], stats, ns, xbar, smats, vlk, vlterms,
        vlhist, ctrl, total, stats_len, params_len, shift;
    // offsets inside one parameter set
    int64_t p_alpha, p_kappa, p_nu, p_m, p_winv, p_w, p_elnpi, p_elndet, p_lnb, p_coef, p_acst, p_linv;
};

__host__ __device__ inline int64_t align8(int64_t v) { return (v + 7) & ~int64_t(7); }

__host__ __device__ inline Layout make_layout(int K, int D, int hist_len) {
    Layout L;
    L.K = K; L.D = D; L.P = feat_count(D); L.pitch = feat_pitch(D); L.hist_len = hist_len;
    const int64_t KD = (int64_t)K * D, KDD = KD * D;
    int64_t o = 0;
    L.p_alpha = o;  o += align8(K);
    L.p_kappa = o;  o += align8(K);
    L.p_nu = o;     o += align8(K);
    L.p_m = o;      o += align8(KD);
    L.p_winv = o;   o += align8(KDD);
    L.p_w = o;      o += align8(KDD);
    L.p_elnpi = o;  o += align8(K);
    L.p_elndet = o; o += align8(K);
    L.p_lnb = o;    o += align8(K);
    L.p_coef = o;   o += (int64_t)K * L.pitch;
    L.p_acst = o;   o += align8(K);
    L.p_linv = o;   o += align8(KDD);
    L.params_len = o;
    o = 0;
    L.center = o;  o += align8(D);
    L.alpha0 = o;  o += align8(K);
    L.kappa0 = o;  o += align8(K);
    L.nu0 = o;     o += align8(K);
    L.m0 = o;      o += align8(KD);
    L.w0inv = o;   o += align8(KDD);
    L.lnb0 = o;    o += align8(K);
    L.lnc0 = o;    o += 8;
    L.params[0] = o; o += L.params_len;
    L.params[1] = o; o += L.params_len;
    L.stats_len = (int64_t)K * L.pitch + 8;
    L.stats = o;   o += L.stats_len;
    L.ns = o;      o += align8(K);
    L.xbar = o;    o += align8(KD);
    L.smats = o;   o += align8(KDD);
    L.vlk = o;     o += (int64_t)K * 8;
    L.vlterms = o; o += 8;
    L.ctrl = o;    o += BGMM_N_CTRL / 2;  // int32[16]
    L.shift = o;   o += align8(KD);
    L.vlhist = o;  o += align8(hist_len); // variable length: keep it LAST so no other offset depends on hist_len
    L.total = o;
    return L;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block-wide sum; result valid in every thread.  `scratch` holds >= 33 doubles of shared memory.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect scratch from a previous call
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double t = (lane < nwarp) ? scratch[lane] : 0.0;
        t = warp_sum(t);
        if (lane == 0) scratch[32] = t;
    }
    __syncthreads();
    return scratch[32];
}

// Block-wide max (fmax, so the order does not matter); result valid in every thread.  `scratch` as for block_sum.
__device__ __forceinline__ double block_max(double v, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();  // protect scratch from a previous call
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    v = scratch[0];
    for (int w = 1; w < nwarp; ++w) v = fmax(v, scratch[w]);
    __syncthreads();
    return v;
}

// Device-resident descriptor of the peer-memory exchange (bgmm_comm.cu); mirrors the layout documented in bgmm.h.
struct CommDesc {
    int world, rank;
    int64_t reserved;
    double* xchg[BGMM_MAX_RANKS];      // exchange block of every rank as mapped in THIS process ([rank] = own block)
};

// Four block-wide sums with one set of barriers (deterministic; results valid in every thread, written back in place).
// The four partials of warp w go to scratch[4w .. 4w+3] (<= 32 doubles for <= 8 warps); every thread then adds them in warp order.
__device__ __forceinline__ void block_sum4(double& a, double& b, double& c, double& d, double* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
    a = warp_sum(a); b = warp_sum(b); c = warp_sum(c); d = warp_sum(d);
    __syncthreads();
    if (lane == 0) { scratch[4 * warp] = a; scratch[4 * warp + 1] = b; scratch[4 * warp + 2] = c; scratch[4 * warp + 3] = d; }
    __syncthreads();
    double ta = 0.0, tb = 0.0, tc = 0.0, td = 0.0;
    for (int w = 0; w < nwarp; ++w) { ta += scratch[4 * w]; tb += scratch[4 * w + 1]; tc += scratch[4 * w + 2]; td += scratch[4 * w + 3]; }
    __syncthreads();
    a = ta; b = tb; c = tc; d = td;
}

// Member states of a batched pass (bgmm_pass_batched): device pointers of R state blocks that share X.
struct BatchDesc {
    double* st[BGMM_MAX_BATCH];
    int R;
};

// Arguments of one pass launch (see bgmm_pass in include/bgmm.h).
struct PassArgs {
    const void* x;
    int64_t n;
    double* state;
    double* workspace;
    double* r_out;
    double* lnrho_out;
    int32_t* argmax_out;
    const double* r_in;
    int force;
    int no_publish = 0;   // 1: leave the peer-exchange block alone even if ctrl.comm is set (BGMM_FORCE_NO_PUBLISH)
    // conditioning guard (ctrl.ROBUST): 0 = feature-map kernel, returns at once when the flag is set (the DIRECT kernel
    // launched behind it does the pass); 1 = ignore the flag (given responsibilities, hidden-Markov path, forced variant)
    int ignore_robust = 0;
    int crit_limit = 0;   // > 0: this pass hands over to the DIRECT kernel when ctrl.CRIT exceeds it (fp32-mode kernels have a
                          // lower limit than the fp64 threshold behind ctrl.ROBUST); 0: ctrl.ROBUST decides
    int lnrho_only = 0;   // large-regime E kernel: write ln rho only (no softmax / r / entropy): the HMM emission pass
    double* rhohat_out = nullptr;   // with lnrho_only: exp(ln rho - row max) [n][K] and the row max [n] (scan inputs)
    double* rowmax_out = nullptr;
};

// HMM extension block ("hst", doubles) next to the state block: transition-matrix hyperparameters and features, the
// statistics the forward-backward scan produces, and the HMM-specific ELBO terms (include/bgmm.h: bgmm_hmm_layout).
struct HmmLayout {
    int K;
    int64_t KK, zeta0, lncz0, set[2], s_zeta, s_lna, s_at, s_misc, ms, g0, sc, vlx, total;
};
__host__ __device__ inline HmmLayout make_hmm_layout(int K) {
    HmmLayout H;
    H.K = K;
    H.KK = align8((int64_t)K * K);
    H.s_zeta = 0; H.s_lna = H.KK; H.s_at = 2 * H.KK; H.s_misc = 3 * H.KK;   // misc: [0] max ln a~, [1] ln C(zeta) sum
    const int64_t setlen = 3 * H.KK + 8;
    int64_t o = 0;
    H.zeta0 = o; o += H.KK;
    H.lncz0 = o; o += 8;
    H.set[0] = o; o += setlen;
    H.set[1] = o; o += setlen;
    H.ms = o; o += H.KK;
    H.g0 = o; o += align8(K);
    H.sc = o; o += 8;        // [0] sum ln c_i   [1] sum gamma . ln rho
    H.vlx = o; o += 8;       // [0] E ln p(z)  [1] E ln p(A)  [2] -E ln q(z)  [3] -E ln q(A)
    H.total = o;
    return H;
}

// Chunk length of the HMM scans and of the chain sampler: <= 4096 chunks (the length of their phase B), at least 32
// elements each.
__host__ __device__ inline int hmm_chunk_len(int64_t n) {
    int64_t L = (n + 4095) / 4096;
    if (L < 32) L = 32;
    return (int)((L + 7) & ~int64_t(7));
}

// Entry test of every pass kernel: queued launches after convergence are no-ops (ctrl.done), and the feature-map kernels
// stand down when bgmm_small has flagged the current parameter set as ill-conditioned (ctrl.robust): the DIRECT kernel
// launched behind them does that pass.
__device__ __forceinline__ bool robust_set(const volatile int* ctrl, int crit_limit) {
    return crit_limit > 0 ? ctrl[BGMM_CTRL_CRIT] > crit_limit : ctrl[BGMM_CTRL_ROBUST] != 0;
}
__device__ __forceinline__ bool pass_skip(const volatile int* ctrl, int force, int ignore_robust, int crit_limit = 0) {
    return (!force && ctrl[BGMM_CTRL_DONE]) || (!ignore_robust && robust_set(ctrl, crit_limit));
}

double robust_threshold();

// ---- programmatic dependent launch (PDL) ----
// Every kernel of the VB loop is launched with the programmatic-stream-serialization attribute and begins with
// pdl_trigger(); pdl_wait():  the next kernel's CTAs are scheduled as soon as SM resources free up and sit in
// griddepcontrol.wait until the previous grid has completed and its memory is visible, so the launch latency of each
// kernel boundary (~3 us, five boundaries per iteration) disappears from the critical path.  Without a programmatic
// dependency both instructions are no-ops.  BGMM_PDL=0 in the environment restores plain launches.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();

// Kernels launched from this host thread (bgmm_launch_count).  Every kernel of libbgmm is launched through launch() or
// launch_pdl(), which count it, so the library, not its callers, knows what each entry point launched.
extern thread_local int64_t g_launches;

template <typename... KArgs, typename... Args>
inline cudaError_t launch_counted(const cudaLaunchConfig_t& cfg, void (*kern)(KArgs...), Args... args) {
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
    if (e == cudaSuccess) ++g_launches;
    return e;
}

// A plain launch: no attributes, the kernel starts once its predecessor on the stream has completed.
template <typename... KArgs, typename... Args>
inline cudaError_t launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    return launch_counted(cfg, kern, args...);
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return launch_counted(cfg, kern, args...);
}

// ---- the end of a pass: hand its statistics over ----
// Every pass leaves per-CTA partial statistics [grid][stats_len] in the workspace.  The CTA that finishes last (of the pass
// kernel itself, or of reduce_partials_kernel behind it) sums them into state.STATS and, in a row-sharded fit, publishes
// the result to the peers (bgmm_comm.cu), where the next bgmm_small picks it up.

// Last-CTA election on ctrl.PASS_TICKET: true in every thread of the CTA that arrives last, which then sees the stores of
// every other CTA.  That CTA resets the ticket for the next pass.
__device__ __forceinline__ bool last_cta(volatile int* ctrl) {
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const int t = atomicAdd(const_cast<int*>(&ctrl[BGMM_CTRL_PASS_TICKET]), 1);
        is_last = (t == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
    if (threadIdx.x == 0) ctrl[BGMM_CTRL_PASS_TICKET] = 0;
    return true;
}

// state.STATS = the sum of the gridDim.x partials in CTA order (deterministic), with the pass's row count and `format`
// (BGMM_STATS_FORMAT: 1 = moments about state.SHIFT, 0 = about the centre) in the tail.
__device__ __forceinline__ void sum_partials(const PassArgs& a, const Layout& L, double format) {
    const int64_t len = L.stats_len, tail = (int64_t)L.K * L.pitch;
    double* out = a.state + L.stats;
    for (int64_t o = threadIdx.x; o < len; o += blockDim.x) {
        double acc = 0.0;
        for (int b = 0; b < (int)gridDim.x; ++b) acc += __ldcg(&a.workspace[(int64_t)b * len + o]);
        if (o == tail + BGMM_STATS_ROWS) acc = (double)a.n;
        if (o == tail + BGMM_STATS_FORMAT) acc = format;
        out[o] = acc;
    }
}

// The peer-exchange descriptor a pass publishes to: the one in ctrl.COMM unless the call set BGMM_FORCE_NO_PUBLISH.
// nullptr: one GPU, or the caller exchanges state.STATS itself (NCCL).
__device__ __forceinline__ const CommDesc* publish_target(const volatile int* ctrl, int no_publish) {
    if (no_publish) return nullptr;
    const unsigned long long lo = (unsigned int)ctrl[BGMM_CTRL_COMM_LO], hi = (unsigned int)ctrl[BGMM_CTRL_COMM_HI];
    return reinterpret_cast<const CommDesc*>((hi << 32) | lo);
}

// Run by the elected CTA once state.STATS holds the reduced statistics: copy them into the own exchange block, fence at
// system scope, stamp every peer, bump ctrl.SEQ.  Nothing to do without a descriptor.
__device__ __forceinline__ void publish_stats(double* __restrict__ st, const Layout& L, const CommDesc* cd) {
    if (cd == nullptr) return;
    __threadfence();
    __syncthreads();
    volatile int* ctrl = reinterpret_cast<volatile int*>(st + L.ctrl);
    const int seq = ctrl[BGMM_CTRL_SEQ];
    const int64_t len = L.stats_len;
    double* mine = cd->xchg[cd->rank] + (int64_t)(seq & 1) * len;
    const volatile double* src = st + L.stats;
    for (int64_t o = threadIdx.x; o < len; o += blockDim.x) mine[o] = src[o];
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < cd->world) {
        // stamp seq+1 into slot [parity][my rank] of peer `threadIdx.x` (release at system scope)
        unsigned long long* flag = reinterpret_cast<unsigned long long*>(cd->xchg[threadIdx.x] + 2 * len) +
                                   (seq & 1) * BGMM_MAX_RANKS + cd->rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"((unsigned long long)(seq + 1)) : "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) ctrl[BGMM_CTRL_SEQ] = seq + 1;
}

// The finish of a pass kernel that reduces its own partials (the simple, DIRECT and fp32 kernels).
__device__ __forceinline__ void finish_pass(const PassArgs& a, const Layout& L, volatile int* ctrl, double format) {
    if (!last_cta(ctrl)) return;
    sum_partials(a, L, format);
    publish_stats(a.state, L, publish_target(ctrl, a.no_publish));
}

// sum of `nparts` per-CTA partial statistics buffers (workspace) into state.STATS, fixed order (bgmm_pass_dmma.cu)
void launch_reduce_partials(const PassArgs& a, const Layout& L, int nparts, cudaStream_t stream);

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

}  // namespace bgmm
