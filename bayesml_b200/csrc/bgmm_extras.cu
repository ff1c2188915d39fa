// Widening rows of SURVEY.md §8(f): per-row work either side of the VB loop that the reference does on the host.
//
//   bgmm_pred_logdensity  f3: ln p(x_new | x^n) of every row under the predictive mixture of Student-t distributions
//                         (formula: /root/reference/bayesml/gaussianmixture/__init__.py:86-97; the reference evaluates the
//                         same density through scipy.stats.multivariate_t at _gaussianmixture.py:1086-1099, one point at a
//                         time).  The quadratic forms (x - mu_k)^T Lambda_k (x - mu_k) come from bgmm_pass (ln rho output of
//                         a parameter set whose Lambda is p_lambda_mats); this kernel is the Student-t / log-sum-exp epilogue.
//   bgmm_dirichlet1       f2: r_n ~ Dirichlet(1_K) per row on the device (`_init_random_responsibility` :734-736 draws them
//                         with numpy's PCG64 + ziggurat stream, 3.2e8 variates on the host at BASELINE config C2).  Counter-
//                         based Philox4x32-10 keyed by (seed, global row): the draw of a row does not depend on how the rows
//                         are sharded.  NOT the reference's random stream — an opt-in (`device_init=True`); same distribution.
//   bgmm_hmm_init_random  the hidden-Markov `random_responsibility` initial state (gamma, sum xi, gamma at the sequence
//                         starts) from Dirichlet(1_{K^2}) transition draws, Philox keyed by (seed, element); same opt-in.
#include "bgmm_common.cuh"
#include <math.h>

namespace bgmm {

__global__ void __launch_bounds__(256) pred_logdensity_kernel(const double* __restrict__ lnrho, const int64_t n, const int K,
                                                              const double* __restrict__ acst, const double* __restrict__ ck,
                                                              const double* __restrict__ hk, const double* __restrict__ nuk,
                                                              double* __restrict__ out) {
    // one warp per row: lane k (k += 32) evaluates component k, then a log-sum-exp over the warp
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= n) return;
    double mx = -INFINITY, t[2] = {-INFINITY, -INFINITY};       // K <= 64
    for (int k = lane, s = 0; k < K; k += 32, ++s) {
        // ln rho = a_k - 0.5 * Delta^2  ->  Delta^2 >= 0 up to rounding
        const double d2 = fmax(0.0, -2.0 * (lnrho[row * K + k] - acst[k]));
        t[s] = ck[k] - hk[k] * log1p(d2 / nuk[k]);
        mx = fmax(mx, t[s]);
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    double sum = 0.0;
    for (int s = 0; s < 2; ++s)
        if (t[s] > -INFINITY) sum += exp(t[s] - mx);
    sum = warp_sum(sum);
    if (lane == 0) out[row] = mx + log(sum);
}

// Philox4x32-10 (Salmon et al. 2011): counter (c0..c3), key (k0, k1) -> 4 x 32 random bits
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 key) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return c;
}

__device__ __forceinline__ double uniform_open(uint32_t hi, uint32_t lo) {       // (0, 1): 53 random bits, never 0
    const unsigned long long u = ((unsigned long long)hi << 32) | lo;
    return ((double)(u >> 11) + 0.5) * (1.0 / 9007199254740992.0);
}

__global__ void __launch_bounds__(256) dirichlet1_kernel(double* __restrict__ r, const int64_t n, const int K,
                                                         const unsigned long long seed, const int64_t row_offset) {
    // one thread per row: K standard exponentials -ln(u), normalised (Dirichlet(1,..,1) = normalised Gamma(1) draws)
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const unsigned long long g = (unsigned long long)(row_offset + i);
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    double* out = r + i * K;
    double sum = 0.0;
    for (int j = 0; j < K; j += 2) {
        const uint4 v = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)(j >> 1), 0x42474d4du), key);
        const double e0 = -log(uniform_open(v.x, v.y));
        out[j] = e0;
        sum += e0;
        if (j + 1 < K) {
            const double e1 = -log(uniform_open(v.z, v.w));
            out[j + 1] = e1;
            sum += e1;
        }
    }
    const double inv = 1.0 / sum;
    for (int j = 0; j < K; ++j) out[j] *= inv;
}

// One generated element: class k = pick(u) with u the uniform of Philox word 0 of the counter (g, 0, tag) under `key`,
// then x[i] = mu_k + L_k eps (L_k = chol[k], lower [D][D]) with eps ~ N(0, I_D) by Box-Muller from words 1, 2, ... of
// the same counter.  `eps` holds D doubles of this thread's scratch.  Returns k.
template <class Pick>
__device__ __forceinline__ int gauss_sample(double* __restrict__ x, const int64_t i, double* eps, const int D,
                                            const double* __restrict__ mu, const double* __restrict__ chol,
                                            const unsigned long long g, const uint2 key, const uint32_t tag, Pick pick) {
    const uint4 v0 = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), 0u, tag), key);
    const int k = pick(uniform_open(v0.x, v0.y));
    for (int j = 0; j < D; j += 2) {
        const uint4 v = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)(1 + (j >> 1)), tag), key);
        const double rad = sqrt(-2.0 * log(uniform_open(v.x, v.y))), ang = 6.283185307179586476925286766559 * uniform_open(v.z, v.w);
        double sn, cs;
        sincos(ang, &sn, &cs);
        eps[j] = rad * cs;
        if (j + 1 < D) eps[j + 1] = rad * sn;
    }
    const double* L = chol + (int64_t)k * D * D;
    const double* m = mu + (int64_t)k * D;
    for (int a = 0; a < D; ++a) {
        double acc = m[a];
        for (int b = 0; b <= a; ++b) acc = fma(L[a * D + b], eps[b], acc);
        x[i * D + a] = acc;
    }
    return k;
}

// GenModel.gen_sample on the device (/root/reference/bayesml/gaussianmixture/_gaussianmixture.py:241-264: a Python loop,
// one `rng.choice` + one `rng.multivariate_normal` per sample): one thread per sample, class from the inverse CDF of pi,
// x = mu_z + L_z eps with L_z = chol(Lambda_z^-1) and Box-Muller normals from Philox keyed by (seed, global row).
__global__ void __launch_bounds__(128) gen_sample_kernel(double* __restrict__ x, int32_t* __restrict__ z, const int64_t n,
                                                         const int K, const int D, const double* __restrict__ cdf,
                                                         const double* __restrict__ mu, const double* __restrict__ chol,
                                                         const unsigned long long seed, const int64_t row_offset) {
    extern __shared__ double eps_s[];                           // [128][D + 1]: this thread's standard normals
    const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (i >= n) return;
    const unsigned long long g = (unsigned long long)(row_offset + i);
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    double* eps = eps_s + threadIdx.x * (D + 1);
    z[i] = gauss_sample(x, i, eps, D, mu, chol, g, key, 0x47454e53u, [&](double u) {
        int k = 0;
        while (k < K - 1 && u > cdf[k]) ++k;
        return k;
    });
}

// ---- hidden-Markov chains (bgmm_hmm_gen_sample) ----
// Element i of a chain is z_i = f_i(z_{i-1}) with f_i(s) = inverse CDF of row s of A at u_i, or at a sequence start the
// constant map "inverse CDF of pi at u_i".  Maps on {0..K-1} compose associatively, so the chain is sampled exactly in
// three phases over chunks of L elements:  A: per chunk, the composed map F_c (lane s of the chunk's warp runs the chunk
// from state s);  B: one CTA sweeps the <= 4096 maps staged in shared memory, in_c = F_{c-1}(in_{c-1});  C: per chunk,
// the run from in_c writes z.  u_i is Philox word 0 of (seed, i, HMM_GEN_TAG), so z does not depend on L.
constexpr uint32_t HMM_GEN_TAG = 0x484d4d47u;                    // "HMMG"
constexpr int HMM_GEN_MAX_CHUNKS = 4096;

__host__ __device__ inline int pow2_ceil(int K) {
    int p = 1;
    while (p < K) p <<= 1;
    return p;
}

// The (K + 1) inverse-CDF rows in shared memory, stride KP + 1 doubles (KP = pow2_ceil(K)): entry k < K - 1 is the running
// max of cdf[r][0..k], every later entry +inf.  The running max does not change "the first k with u <= cdf[r][k]" (every
// earlier entry is < u), makes the row sorted for a binary search, and k = K - 1 is the clamp of gen_sample_kernel.
__device__ __forceinline__ void stage_cdf(double* tab, const double* __restrict__ cdf, const int K, const int KP) {
    for (int e = threadIdx.x; e < (K + 1) * KP; e += blockDim.x) {
        const int r = e / KP, k = e - r * KP;
        double v = INFINITY;
        if (k < K - 1) {
            v = cdf[r * K];
            for (int j = 1; j <= k; ++j) v = fmax(v, cdf[r * K + j]);
        }
        tab[r * (KP + 1) + k] = v;
    }
}

__device__ __forceinline__ int inv_cdf(const double* row, const double u, const int KP) {
    int k = 0;
    for (int step = KP >> 1; step > 0; step >>= 1)
        if (row[k + step - 1] < u) k += step;
    return k;
}

// Phases A (WRITE_Z = false: maps[c][s] = F_c(s)) and C (WRITE_Z: z of chunk c from in[c]); one warp per chunk.  The
// lanes draw the uniforms of 32 elements at a time and the chain steps through them by broadcast; `starts` (sorted,
// starts[0] = 0) is searched once per chunk and then read 32 entries per batch into a bit mask of the batch's starts.
template <bool WRITE_Z>
__global__ void __launch_bounds__(256) hmm_chain_kernel(const int64_t n, const int K, const int KP, const int64_t L,
                                                        const int nch, const double* __restrict__ cdf,
                                                        const int64_t* __restrict__ starts, const int64_t n_seqs,
                                                        const unsigned long long seed, uint8_t* __restrict__ maps,
                                                        const uint8_t* __restrict__ in, int32_t* __restrict__ z) {
    extern __shared__ double tab[];                             // [K + 1][KP + 1]
    stage_cdf(tab, cdf, K, KP);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c >= nch) return;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const int64_t b = (int64_t)c * L, e = min(n, b + L);
    int64_t lo = 0, hi = n_seqs;                                // p = first sequence start >= b
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (starts[mid] < b) lo = mid + 1; else hi = mid;
    }
    int64_t p = lo;
    int s = WRITE_Z ? (int)in[c] : min(lane, K - 1);
    for (int64_t base = b; base < e; base += 32) {
        const unsigned long long g = (unsigned long long)(base + lane);
        const uint4 v = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), 0u, HMM_GEN_TAG), key);
        const double u_mine = uniform_open(v.x, v.y);
        const int64_t st = p + lane < n_seqs ? starts[p + lane] : n;
        const bool hit = st < base + 32;
        const unsigned smask = __reduce_or_sync(0xffffffffu, hit ? 1u << (int)(st - base) : 0u);
        p += __popc(__ballot_sync(0xffffffffu, hit));
        const int cnt = (int)min((int64_t)32, e - base);
        int zi = 0;
        for (int j = 0; j < cnt; ++j) {
            const double u = __shfl_sync(0xffffffffu, u_mine, j);
            s = inv_cdf(tab + ((smask >> j) & 1u ? 0 : s + 1) * (KP + 1), u, KP);
            if (WRITE_Z && lane == j) zi = s;
        }
        if (WRITE_Z && lane < cnt) z[base + lane] = zi;
    }
    if (!WRITE_Z && lane < K) maps[(int64_t)c * K + lane] = (uint8_t)s;
}

// Phase B in one CTA of 1024 threads, on maps staged in shared memory (a chain of dependent global loads would cost one
// L2 round trip per chunk): the nch maps are cut into nseg segments; thread (seg, s) composes its segment's maps from s,
// thread 0 sweeps the nseg segment maps, and thread seg then writes in[c] along its segment.
__global__ void __launch_bounds__(1024) hmm_chain_sweep_kernel(const uint8_t* __restrict__ maps, const int nch, const int K,
                                                               const int nseg, uint8_t* __restrict__ in) {
    extern __shared__ uint4 sweep_s[];
    uint8_t* mp = reinterpret_cast<uint8_t*>(sweep_s);          // [nch][K] padded to 16 bytes | [nseg][K] | [nseg]
    const int mbytes = (nch * K + 15) & ~15;
    uint8_t* segm = mp + mbytes;
    uint8_t* segin = segm + nseg * K;
    for (int o = threadIdx.x; o < mbytes / 16; o += blockDim.x) sweep_s[o] = reinterpret_cast<const uint4*>(maps)[o];
    __syncthreads();
    const int t = threadIdx.x, sl = (nch + nseg - 1) / nseg;
    const int seg = t / K, s0 = t - seg * K;
    if (seg < nseg) {
        int s = s0;
        for (int c = seg * sl; c < min(nch, seg * sl + sl); ++c) s = mp[c * K + s];
        segm[seg * K + s0] = (uint8_t)s;
    }
    __syncthreads();
    if (t == 0) {
        int s = 0;                                              // chunk 0 begins with a sequence start: any state
        for (int q = 0; q < nseg; ++q) {
            segin[q] = (uint8_t)s;
            s = segm[q * K + s];
        }
    }
    __syncthreads();
    if (t < nseg) {
        int s = segin[t];
        for (int c = t * sl; c < min(nch, t * sl + sl); ++c) {
            in[c] = (uint8_t)s;
            s = mp[c * K + s];
        }
    }
}

// Emission: one thread per element, x_i = mu_{z_i} + L_{z_i} eps_i (64 threads: [64][D + 1] doubles of scratch, D <= 256).
__global__ void __launch_bounds__(64) hmm_emit_kernel(double* __restrict__ x, const int32_t* __restrict__ z, const int64_t n,
                                                      const int D, const double* __restrict__ mu,
                                                      const double* __restrict__ chol, const unsigned long long seed) {
    extern __shared__ double eps_s[];
    const int64_t i = (int64_t)blockIdx.x * 64 + threadIdx.x;
    if (i >= n) return;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    gauss_sample(x, i, eps_s + threadIdx.x * (D + 1), D, mu, chol, (unsigned long long)i, key, HMM_GEN_TAG,
                 [&](double) { return (int)z[i]; });
}

// Workspace of bgmm_hmm_gen_sample (bytes, 256-aligned parts): starts [n_seqs] int64 | maps [nch][K] | in [nch].
struct HmmGenWs {
    int64_t nch, starts, maps, in, total;
};
inline int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }
inline bool hmm_gen_ws(int K, int64_t n, int64_t n_seqs, int64_t chunk_len, HmmGenWs& w) {
    if (K <= 0 || K > 32 || n < 0) return false;
    const int64_t L = chunk_len == 0 ? hmm_chunk_len(n) : chunk_len;
    if (L <= 0) return false;
    w.nch = (n + L - 1) / L;
    if (w.nch > HMM_GEN_MAX_CHUNKS) return false;
    w.starts = 0;
    w.maps = align256((n_seqs > 1 ? n_seqs : 1) * 8);
    w.in = w.maps + align256(w.nch * K);
    w.total = w.in + align256(w.nch);
    return true;
}

// ---- hidden-Markov 'random_responsibility' initial state (bgmm_hmm_init_random) ----
// Element i draws xt_i[j][k] (j, k < K), K^2 standard exponentials -ln u, and xi_i = xt_i / T_i with T_i the sum of all
// K^2 entries: Dirichlet(1_{K^2}) as a K x K matrix.  Counter mapping: pair p = r * K + k (r < ceil(K / 2)) holds the
// entries (2r, k) and (2r + 1, k); Philox4x32-10 of counter (i lo, i hi, p, HMM_INIT_TAG) under key (seed lo, seed hi)
// gives (2r, k) from words (0, 1) and (2r + 1, k) from words (2, 3), which stay unused when 2r + 1 = K.
// Rules (those of hiddenmarkovnormal._init_random_responsibility): gamma_i = column sums of xi_i, except at a sequence
// start s, where gamma_s = row sums of xi_{s+1} (its sequence is longer than 1) or of xi_s (length 1); MS = sum of xi_i
// over the elements that are not starts, G0 = sum of gamma over the starts.  n = 1: gamma_0 = row 0 of xt_0 normalised
// by its own sum (K exponentials: Dirichlet(1_K)), MS = 0.
// Layout: a group of KP lanes (KP = max(2, pow2_ceil(K))) per element, lane k of the group owns column k, so a warp
// takes 32 / KP consecutive elements per step.  Every warp runs a fixed contiguous span of elements and keeps MS in KP
// registers per lane; the per-block partials are summed in block order by hmm_init_finish_kernel.  The grid depends
// only on (n, K), so the sums come out the same bits on every run and every GPU.  A start's xi_{s+1} is redrawn.
constexpr uint32_t HMM_INIT_TAG = 0x484d4d49u;                   // "HMMI"
constexpr int HMM_INIT_WARPS = 8;
constexpr int HMM_INIT_MAX_BLOCKS = 1024;

struct HmmInitGrid {
    int KP, nblk;
    int64_t span;                                               // elements per warp, a multiple of 32 / KP
};
inline bool hmm_init_grid(int K, int64_t n, HmmInitGrid& g) {
    if (K < 1 || K > 32 || n < 1) return false;
    g.KP = K <= 2 ? 2 : pow2_ceil(K);
    const int64_t per = 32 / g.KP, steps = (n + per - 1) / per;
    g.nblk = (int)min((int64_t)HMM_INIT_MAX_BLOCKS, (steps + HMM_INIT_WARPS - 1) / HMM_INIT_WARPS);
    const int64_t warps = (int64_t)g.nblk * HMM_INIT_WARPS;
    g.span = (steps + warps - 1) / warps * per;
    return true;
}

// 1 / t for a positive normal t, within an ulp of the rounded quotient: the reciprocal estimate and two Newton steps,
// without the slow-path call of the IEEE division (a call makes ptxas spill values that live across it)
__device__ __forceinline__ double recip_pos(const double t) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(t));
    r = fma(r, fma(-t, r, 1.0), r);
    return fma(r, fma(-t, r, 1.0), r);
}

template <int KP>
__device__ __forceinline__ double group_sum(double v) {         // over the KP lanes of a group; every lane gets the sum
#pragma unroll
    for (int o = KP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Column k of xt_i into e[0..K-1] (zeros beyond K, and in lanes k >= K); returns its sum.
template <int KP>
__device__ __forceinline__ double init_draw(double (&e)[KP], const unsigned long long i, const int K, const int k,
                                            const uint2 key) {
    double col = 0.0;
#pragma unroll
    for (int r = 0; r < KP / 2; ++r) {
        e[2 * r] = e[2 * r + 1] = 0.0;
        if (2 * r < K && k < K) {
            const uint4 v = philox4x32_10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)(r * K + k), HMM_INIT_TAG), key);
            e[2 * r] = -log(uniform_open(v.x, v.y));
            if (2 * r + 1 < K) e[2 * r + 1] = -log(uniform_open(v.z, v.w));
        }
    }
#pragma unroll
    for (int j = 0; j < KP; ++j) col += e[j];
    return col;
}

template <int KP>
__global__ void __launch_bounds__(HMM_INIT_WARPS * 32) hmm_init_random_kernel(const int64_t n, const int K,
                                                                             const unsigned long long seed,
                                                                             const int64_t* __restrict__ starts,
                                                                             const int64_t n_seqs, const int64_t span,
                                                                             double* __restrict__ gamma,
                                                                             double* __restrict__ part) {
    constexpr int G = 32 / KP;                                  // elements per warp step
    __shared__ double red[KP * KP + KP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane / KP, k = lane % KP;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    const int64_t b = min(n, ((int64_t)blockIdx.x * HMM_INIT_WARPS + warp) * span), e = min(n, b + span);
    // starts == NULL: one sequence, start 0
    auto start = [&](int64_t q) { return q >= n_seqs ? INT64_MAX : starts != nullptr ? starts[q] : (int64_t)0; };
    int64_t lo = 0, hi = n_seqs;                                // p = first sequence start >= b
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (start(mid) < b) lo = mid + 1; else hi = mid;
    }
    int64_t p = lo;
    double acc[KP], g0 = 0.0;
#pragma unroll
    for (int j = 0; j < KP; ++j) acc[j] = 0.0;
    for (int64_t base = b; base < e; base += G) {
        // bit t of smask: element base + t is a sequence start (t <= G, so the start after the last element is seen)
        const int64_t st = start(p + lane);
        const unsigned smask = __reduce_or_sync(0xffffffffu, st <= base + G ? 1u << (int)(st - base) : 0u);
        p += __popc(__ballot_sync(0xffffffffu, st < base + G));
        const int64_t i = base + g;
        const bool valid = i < e, first = valid && ((smask >> g) & 1u);
        double ev[KP];
        const double col = init_draw<KP>(ev, (unsigned long long)i, K, k, key);
        double inv = recip_pos(group_sum<KP>(col));
        if (valid && !first) {
#pragma unroll
            for (int j = 0; j < KP; ++j) acc[j] += ev[j] * inv;
            if (k < K) gamma[i * K + k] = col * inv;
        }
        if (__any_sync(0xffffffffu, first)) {                   // warp-uniform: every lane takes part in the shuffles
            const bool redraw = first && !(i + 1 == n || ((smask >> (g + 1)) & 1u));
            const double col1 = redraw ? init_draw<KP>(ev, (unsigned long long)(i + 1), K, k, key) : 0.0;
            const double t1 = group_sum<KP>(col1);
            if (redraw) inv = recip_pos(t1);
            double row = 0.0, row0 = 0.0;
#pragma unroll
            for (int j = 0; j < KP; ++j) {
                const double s = group_sum<KP>(ev[j]);
                if (k == j) row = s;
                if (j == 0) row0 = s;
            }
            const double gm = n == 1 ? ev[0] * recip_pos(row0) : row * inv;
            if (first && k < K) {
                gamma[i * K + k] = gm;
                g0 += gm;
            }
        }
    }
    // the warp's groups, then the block's warps in order
#pragma unroll
    for (int j = 0; j < KP; ++j)
        for (int o = KP; o < 32; o <<= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
    for (int o = KP; o < 32; o <<= 1) g0 += __shfl_xor_sync(0xffffffffu, g0, o);
    for (int w = 0; w < HMM_INIT_WARPS; ++w) {
        if (warp == w && lane < K) {
#pragma unroll
            for (int j = 0; j < KP; ++j)
                if (j < K) red[j * K + lane] = (w == 0 ? 0.0 : red[j * K + lane]) + acc[j];
            red[K * K + lane] = (w == 0 ? 0.0 : red[K * K + lane]) + g0;
        }
        __syncthreads();
    }
    const int len = K * K + K;
    for (int t = threadIdx.x; t < len; t += blockDim.x) part[(int64_t)blockIdx.x * len + t] = red[t];
}

// MS, G0 = the per-block partials summed in block order; SC = 0.
__global__ void __launch_bounds__(128) hmm_init_finish_kernel(const double* __restrict__ part, const int nblk, const int K,
                                                              double* __restrict__ ms, double* __restrict__ g0,
                                                              double* __restrict__ sc) {
    const int len = K * K + K, t = blockIdx.x * 128 + threadIdx.x;
    if (t < 8) sc[t] = 0.0;
    if (t >= len) return;
    double s = 0.0;
    for (int blk = 0; blk < nblk; ++blk) s += part[(int64_t)blk * len + t];
    if (t < K * K) ms[t] = s; else g0[t - K * K] = s;
}

template <int KP>
int launch_hmm_init_random(const HmmInitGrid& gr, int64_t n, int K, unsigned long long seed, const int64_t* starts,
                           int64_t n_seqs, double* gamma, double* part, cudaStream_t st) {
    launch(hmm_init_random_kernel<KP>, (unsigned)gr.nblk, HMM_INIT_WARPS * 32, 0, st, n, K, seed, starts, n_seqs, gr.span,
           gamma, part);
    return check_cuda(cudaGetLastError(), "hmm_init_random_kernel launch");
}

}  // namespace bgmm

using namespace bgmm;

extern "C" int bgmm_gen_sample(double* x_out, int32_t* z_out, int64_t n, int K, int D, const double* cdf, const double* mu,
                               const double* chol, uint64_t seed, int64_t row_offset, void* stream) {
    if (n < 0 || K <= 0 || D <= 0 || D > 256 || row_offset < 0 || cdf == nullptr || mu == nullptr || chol == nullptr ||
        ((x_out == nullptr || z_out == nullptr) && n > 0)) {
        set_error("bgmm_gen_sample: bad argument (n=%lld K=%d D=%d; D <= 256)", (long long)n, K, D);
        return BGMM_EINVAL;
    }
    if (n == 0) return BGMM_OK;
    const size_t smem = sizeof(double) * 128 * (size_t)(D + 1);
    if (smem > 48 * 1024) {
        int rc = check_cuda(cudaFuncSetAttribute(gen_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                            "cudaFuncSetAttribute(gen_sample_kernel)");
        if (rc) return rc;
    }
    launch(gen_sample_kernel, (unsigned)((n + 127) / 128), 128, smem, (cudaStream_t)stream, x_out, z_out, n, K, D, cdf, mu, chol,
           (unsigned long long)seed, row_offset);
    return check_cuda(cudaGetLastError(), "gen_sample_kernel launch");
}

extern "C" int64_t bgmm_hmm_gen_workspace_bytes(int K, int64_t n, int64_t n_seqs, int64_t chunk_len) {
    HmmGenWs w;
    return hmm_gen_ws(K, n, n_seqs, chunk_len, w) ? w.total : 0;
}

extern "C" int bgmm_hmm_gen_sample(double* x_out, int32_t* z_out, int64_t n, int K, int D, const double* cdf, const double* mu,
                                   const double* chol, const int64_t* seq_starts, int64_t n_seqs, uint64_t seed,
                                   int64_t chunk_len, void* workspace, void* stream) {
    HmmGenWs w;
    if (seq_starts == nullptr || n_seqs < 1) n_seqs = 1;
    if (n < 0 || K <= 0 || K > 32 || D <= 0 || D > 256 || chunk_len < 0 || cdf == nullptr || mu == nullptr ||
        chol == nullptr || ((x_out == nullptr || z_out == nullptr || workspace == nullptr) && n > 0)) {
        set_error("bgmm_hmm_gen_sample: bad argument (n=%lld K=%d D=%d; K <= 32, D <= 256)", (long long)n, K, D);
        return BGMM_EINVAL;
    }
    if (!hmm_gen_ws(K, n, n_seqs, chunk_len, w)) {
        set_error("bgmm_hmm_gen_sample: chunk_len=%lld gives more than %d chunks of n=%lld", (long long)chunk_len,
                  HMM_GEN_MAX_CHUNKS, (long long)n);
        return BGMM_EINVAL;
    }
    if (seq_starts != nullptr && n_seqs > 1) {
        bool ok = seq_starts[0] == 0 && n_seqs <= n;
        for (int64_t q = 1; ok && q < n_seqs; ++q) ok = seq_starts[q] > seq_starts[q - 1] && seq_starts[q] < n;
        if (!ok) {
            set_error("bgmm_hmm_gen_sample: seq_starts must begin with 0, increase strictly and stay below n=%lld",
                      (long long)n);
            return BGMM_EINVAL;
        }
    }
    if (n == 0) return BGMM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    int64_t* starts = reinterpret_cast<int64_t*>(ws + w.starts);
    int rc = n_seqs > 1 ? check_cuda(cudaMemcpyAsync(starts, seq_starts, sizeof(int64_t) * n_seqs, cudaMemcpyHostToDevice, st),
                                     "cudaMemcpyAsync(seq_starts)")
                        : check_cuda(cudaMemsetAsync(starts, 0, sizeof(int64_t), st), "cudaMemsetAsync(seq_starts)");
    if (rc) return rc;
    const int KP = pow2_ceil(K), nch = (int)w.nch;
    const int64_t L = chunk_len == 0 ? hmm_chunk_len(n) : chunk_len;
    const size_t tab_smem = sizeof(double) * (K + 1) * (KP + 1);
    const unsigned grid = (unsigned)((nch + 7) / 8);
    uint8_t* maps = ws + w.maps;
    uint8_t* in = ws + w.in;
    launch(hmm_chain_kernel<false>, grid, 256, tab_smem, st, n, K, KP, L, nch, cdf, starts, n_seqs, (unsigned long long)seed,
           maps, nullptr, nullptr);
    if ((rc = check_cuda(cudaGetLastError(), "hmm_chain_kernel<maps> launch"))) return rc;
    int nseg = 1;
    while ((nseg + 1) * (nseg + 1) <= nch) ++nseg;              // ~sqrt(nch) segments of ~sqrt(nch) maps
    nseg = min(nseg, 1024 / K);
    const size_t sweep_smem = (size_t)((nch * K + 15) & ~15) + (size_t)nseg * (K + 1);
    if (sweep_smem > 48 * 1024) {
        rc = check_cuda(cudaFuncSetAttribute(hmm_chain_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sweep_smem),
                        "cudaFuncSetAttribute(hmm_chain_sweep_kernel)");
        if (rc) return rc;
    }
    launch(hmm_chain_sweep_kernel, 1, 1024, sweep_smem, st, maps, nch, K, nseg, in);
    if ((rc = check_cuda(cudaGetLastError(), "hmm_chain_sweep_kernel launch"))) return rc;
    launch(hmm_chain_kernel<true>, grid, 256, tab_smem, st, n, K, KP, L, nch, cdf, starts, n_seqs, (unsigned long long)seed,
           nullptr, in, z_out);
    if ((rc = check_cuda(cudaGetLastError(), "hmm_chain_kernel<z> launch"))) return rc;
    const size_t emit_smem = sizeof(double) * 64 * (size_t)(D + 1);
    if (emit_smem > 48 * 1024) {
        rc = check_cuda(cudaFuncSetAttribute(hmm_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)emit_smem),
                        "cudaFuncSetAttribute(hmm_emit_kernel)");
        if (rc) return rc;
    }
    launch(hmm_emit_kernel, (unsigned)((n + 63) / 64), 64, emit_smem, st, x_out, z_out, n, D, mu, chol, (unsigned long long)seed);
    return check_cuda(cudaGetLastError(), "hmm_emit_kernel launch");
}

extern "C" int64_t bgmm_hmm_init_random_workspace_doubles(int K, int64_t n) {
    HmmInitGrid gr;
    return hmm_init_grid(K, n, gr) ? (int64_t)gr.nblk * (K * K + K) : 0;
}

extern "C" int bgmm_hmm_init_random(int64_t n, int K, uint64_t seed, const int64_t* seq_starts_host,
                                    const int64_t* seq_starts, int64_t n_seqs, double* gamma, double* hst, double* workspace,
                                    void* stream) {
    HmmInitGrid gr;
    if (!hmm_init_grid(K, n, gr) || n_seqs < 1 || gamma == nullptr || hst == nullptr || workspace == nullptr ||
        (n_seqs > 1 && (seq_starts_host == nullptr || seq_starts == nullptr || n_seqs > n))) {
        set_error("bgmm_hmm_init_random: bad argument (n=%lld K=%d n_seqs=%lld; n >= 1, 1 <= K <= 32, 1 <= n_seqs <= n)",
                  (long long)n, K, (long long)n_seqs);
        return BGMM_EINVAL;
    }
    if (n_seqs > 1) {
        bool ok = seq_starts_host[0] == 0;
        for (int64_t q = 1; ok && q < n_seqs; ++q) ok = seq_starts_host[q] > seq_starts_host[q - 1] && seq_starts_host[q] < n;
        if (!ok) {
            set_error("bgmm_hmm_init_random: seq_starts must begin with 0, increase strictly and stay below n=%lld",
                      (long long)n);
            return BGMM_EINVAL;
        }
    } else {
        seq_starts = nullptr;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long s = (unsigned long long)seed;
    int rc;
    switch (gr.KP) {
        case 2: rc = launch_hmm_init_random<2>(gr, n, K, s, seq_starts, n_seqs, gamma, workspace, st); break;
        case 4: rc = launch_hmm_init_random<4>(gr, n, K, s, seq_starts, n_seqs, gamma, workspace, st); break;
        case 8: rc = launch_hmm_init_random<8>(gr, n, K, s, seq_starts, n_seqs, gamma, workspace, st); break;
        case 16: rc = launch_hmm_init_random<16>(gr, n, K, s, seq_starts, n_seqs, gamma, workspace, st); break;
        default: rc = launch_hmm_init_random<32>(gr, n, K, s, seq_starts, n_seqs, gamma, workspace, st); break;
    }
    if (rc) return rc;
    const HmmLayout H = make_hmm_layout(K);
    launch(hmm_init_finish_kernel, (unsigned)((K * K + K + 127) / 128), 128, 0, st, (const double*)workspace, gr.nblk, K,
           hst + H.ms, hst + H.g0, hst + H.sc);
    return check_cuda(cudaGetLastError(), "hmm_init_finish_kernel launch");
}

extern "C" int bgmm_pred_logdensity(const double* lnrho, int64_t n, int K, const double* acst, const double* ck,
                                    const double* hk, const double* nuk, double* out, void* stream) {
    if (n < 0 || K <= 0 || K > 64 || ((lnrho == nullptr || out == nullptr) && n > 0) || acst == nullptr || ck == nullptr ||
        hk == nullptr || nuk == nullptr) {
        set_error("bgmm_pred_logdensity: bad argument (n=%lld K=%d; K <= 64)", (long long)n, K);
        return BGMM_EINVAL;
    }
    if (n == 0) return BGMM_OK;
    launch(pred_logdensity_kernel, (unsigned)((n + 7) / 8), 256, 0, (cudaStream_t)stream, lnrho, n, K, acst, ck, hk, nuk, out);
    return check_cuda(cudaGetLastError(), "pred_logdensity_kernel launch");
}

extern "C" int bgmm_dirichlet1(double* r_out, int64_t n, int K, uint64_t seed, int64_t row_offset, void* stream) {
    if (n < 0 || K <= 0 || row_offset < 0 || (r_out == nullptr && n > 0)) {
        set_error("bgmm_dirichlet1: bad argument (n=%lld K=%d)", (long long)n, K);
        return BGMM_EINVAL;
    }
    if (n == 0) return BGMM_OK;
    launch(dirichlet1_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream, r_out, n, K, (unsigned long long)seed,
           row_offset);
    return check_cuda(cudaGetLastError(), "dirichlet1_kernel launch");
}
