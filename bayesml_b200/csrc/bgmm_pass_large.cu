// bgmm_pass, large K*P regime (BGMM_PASS_LARGE): fp64, any D <= 128, K <= 64 — BASELINE configs C4 (D=128, K=64) and
// C5 (D=32, K=16), where the K x P statistics accumulators (P = 1 + D + D(D+1)/2) no longer fit on one SM.
//
// Two tiled GEMM kernels on the FP64 tensor pipe (mma.sync.m8n8k4.f64 = DMMA.8x8x4), the feature tile Phi generated on the
// fly in 64-column chunks from the X tile held in shared memory (Phi itself never exists in HBM):
//   e_large_kernel : ln rho[64 rows][K] = sum over 64-feature chunks Phi_chunk . coef_chunk^T; the A (Phi) fragments are
//                    built in registers from the X tile (each 8-row block belongs to one warp), the coefficient chunks
//                    come by TMA from a pre-swizzled image (one extra warp, two stages),
//                    softmax in the accumulator fragments, entropy term, r written to HBM ([N][K] fp64, the only
//                    intermediate that leaves the chip: K*8 bytes per sample against (D^2+3D) K flops),
//   m_large_kernel : raw[K][128-feature chunk] += R^T . Phi_chunk, output-stationary: a CTA owns one feature chunk for a
//                    contiguous range of rows (grid = chunks x row splits), accumulators in registers, the B (Phi)
//                    fragments built in registers from TMA-prefetched X tiles,
// then reduce_partials_kernel sums the row splits in a fixed order (deterministic).
// Same shared-memory fragment layout (k-step-pair permutation + XOR swizzle) as the fused kernel (bgmm_mma.cuh).
// Replaces `_update_q_z` :772-784, `_calc_n_x_bar_s` :725-732, `xlogy` :704 of the reference GMM file for these shapes.
#include "bgmm_common.cuh"
#include "bgmm_mma.cuh"
#include <math.h>

namespace bgmm {

constexpr int LG_THREADS = 256;
constexpr int LG_ETILE = 64;      // rows per E tile (8 m-blocks, one per warp)
constexpr int LG_CW = 64;         // E: feature columns per chunk
constexpr int LG_MSUB = 32;       // M: rows per step
constexpr int LG_MCW = 128;       // M: feature columns owned by one CTA

// logical feature p -> kind/indices: 0 constant, 1 linear (i), 2 quadratic (i >= j), 3 padding (zero)
__device__ __forceinline__ void feat_decode(int p, int D, int P, int& kind, int& i, int& j) {
    i = 0; j = 0;
    if (p >= P) { kind = 3; return; }
    if (p == 0) { kind = 0; return; }
    if (p <= D) { kind = 1; i = p - 1; return; }
    const int q = p - 1 - D;
    int r = (int)((sqrtf(8.0f * q + 1.0f) - 1.0f) * 0.5f);
    while (r * (r + 1) / 2 > q) --r;
    while ((r + 1) * (r + 2) / 2 <= q) ++r;
    kind = 2; i = r; j = q - r * (r + 1) / 2;
}
__device__ __forceinline__ double feat_value(int kind, int i, int j, const double* xr) {
    return kind == 2 ? xr[i] * xr[j] : (kind == 1 ? xr[i] : (kind == 0 ? 1.0 : 0.0));
}

// Coefficient image for the E kernel: chunk c = the [8*KB][64] shared-memory tile (k-step-pair permutation + swizzle, zero /
// -1e300 padding applied) stored contiguously, so that the E kernel fetches a chunk with ONE TMA bulk copy.
template <int KB>
__global__ void __launch_bounds__(LG_THREADS) coef_pack_kernel(const double* __restrict__ st, const Layout L,
                                                               double* __restrict__ packed, const int force,
                                                               const int ignore_robust) {
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (pass_skip(ctrl, force, ignore_robust)) return;
    const double* __restrict__ coef_g = st + L.params[ctrl[BGMM_CTRL_CUR]] + L.p_coef;
    const int c = blockIdx.x;
    double* out = packed + (int64_t)c * 8 * KB * LG_CW;
    for (int e = threadIdx.x; e < 8 * KB * LG_CW; e += LG_THREADS) {
        const int k = e >> 6, f2 = e & (LG_CW - 1), p2 = LG_CW * c + f2;
        double v = 0.0;
        if (k < L.K) { if (p2 < L.P) v = coef_g[(int64_t)k * L.pitch + p2]; }
        else if (p2 == 0) v = -1.0e300;                        // padded components: r == 0 exactly
        out[k * LG_CW + (phys_col(f2) ^ fsw(k))] = v;
    }
}

constexpr int LG_ETHREADS = 288;   // E kernel: 8 GEMM warps + 1 warp that streams the coefficient chunks by TMA

// Every logical feature as a product x[a] * x[b] of two columns of the X tile EXTENDED by the constant columns
// x[D] = 1 and x[D + 1] = 0 (they live in the tile's row padding): quadratic (i, j), linear (D, i), constant (D, D), padding
// (D + 1, D + 1).  Packed (a << 8) | b.  The fragment generation is then branch-free and still exact (1 * x = x).
__global__ void __launch_bounds__(256) feat_table_kernel(unsigned short* __restrict__ tab, const int D, const int P,
                                                         const int n) {
    const int p = blockIdx.x * 256 + threadIdx.x;
    if (p >= n) return;
    int kind, i, j;
    feat_decode(p, D, P, kind, i, j);
    const int fa = kind == 2 ? i : (kind == 3 ? D + 1 : D);
    const int fb = kind == 2 ? j : (kind == 1 ? i : (kind == 0 ? D : D + 1));
    tab[p] = (unsigned short)((fa << 8) | fb);
}

// In the E-GEMM every 8-row block of Phi is consumed by exactly one warp, so Phi is never staged in shared memory: each
// thread builds its A fragments (row g of its block, the features of its quad lane q) from the X tile in registers, one
// in-stream DMUL per fragment.  (A separate producer starves: its DMULs queue behind the GEMM warps' DMMAs on the in-order
// FP64 pipe, ~250 cycles each — measured, profiles/.)  The X tile has a padded row pitch (conflict-free column reads).
// GB = 8-component blocks per softmax GROUP.  GB == KB: one mixture (the usual case).  GB < KB: the K components are
// NG = KB / GB independent mixtures of 8*GB components each that share X (batched restarts, bgmm_pass_batched): one X read
// and one Phi fragment generation serve all of them; the softmax, the entropy term and r are per group.
template <int KB, int GB>
__global__ void __launch_bounds__(LG_ETHREADS, 1)
e_large_kernel(const PassArgs a, const Layout L, double* __restrict__ ews, const double* __restrict__ packed,
               const unsigned short* __restrict__ ftab) {
    constexpr int NG = KB / GB;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int K = L.K, D = L.D, P = L.P;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust)) return;
    const double* __restrict__ x = static_cast<const double*>(a.x);

    const int nchunk = (P + LG_CW - 1) / LG_CW;
    const int XP = D + 2;                                      // padded pitch: 8 rows x same column -> 8 distinct bank groups
    double* coefS = reinterpret_cast<double*>(smem_raw);       // [2 stages][8*KB][64] swizzled (TMA destination)
    double* xs = coefS + 2 * 8 * KB * LG_CW;                   // [64][D + 2]
    double* red = xs + LG_ETILE * XP;                          // [40]
    uint64_t* cfull = reinterpret_cast<uint64_t*>(red + 40);   // [2]  coefficient chunk landed (TMA tx)
    uint64_t* cempty = cfull + 2;                              // [2]  stage consumed (256 arrivals)
    unsigned short* tabS = reinterpret_cast<unsigned short*>(cempty + 2);   // [nchunk * 64]
    constexpr uint32_t kChunkBytes = 8 * KB * LG_CW * sizeof(double);
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) { mbar_init(&cfull[i], 1); mbar_init(&cempty[i], 256); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int p = tid; p < nchunk * LG_CW; p += LG_ETHREADS) tabS[p] = ftab[p];
    __syncthreads();

    const int64_t ntiles = (a.n + LG_ETILE - 1) / LG_ETILE;
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    double ent[NG];
#pragma unroll
    for (int gi = 0; gi < NG; ++gi) ent[gi] = 0.0;

    if (warp == 8) {
        // =========================== TMA WARP: coefficient chunks, two stages ===========================
        // the whole warp walks the loop (convergent at the final block barrier); lane 0 issues the copies
        const int64_t total = my_tiles * nchunk;
        int c = 0;
        for (int64_t cc = 0; cc < total; ++cc) {
            const int b = (int)(cc & 1);
            if (cc >= 2) mbar_wait(&cempty[b], (uint32_t)(((cc >> 1) - 1) & 1));
            if (lane == 0) {
                mbar_expect_tx(&cfull[b], kChunkBytes);
                tma_load_1d(coefS + b * 8 * KB * LG_CW, packed + (int64_t)c * 8 * KB * LG_CW, kChunkBytes, &cfull[b]);
            }
            __syncwarp();
            if (++c == nchunk) c = 0;
        }
    } else {
        // =========================== GEMM WARPS ===========================
        const int fg = fsw(g);
        const int lrow = 8 * warp + g;
        const int eo0 = (2 * q) ^ fg, eo1 = (8 + 2 * q) ^ fg;
        const double* xr = xs + lrow * XP;                     // this thread's row of the X tile
        for (int r = tid; r < LG_ETILE; r += 256) { xs[r * XP + D] = 1.0; xs[r * XP + D + 1] = 0.0; }   // constant columns
        double sprod[NG];
#pragma unroll
        for (int gi = 0; gi < NG; ++gi) sprod[gi] = 1.0;
        int64_t cc = 0;
        int it = 0;
        // D <= 32: a 64-row tile is <= 8 elements per thread, so the NEXT tile is fetched into registers before this
        // tile's GEMM and only stored to shared memory at the top of the next iteration (the global round trip, otherwise
        // exposed once per tile, hides behind the GEMM; at small D it is most of the kernel's time)
        const bool reg_prefetch = D <= 32;
        double pre[8];
        auto fetch_tile = [&](int64_t tt) {
            const int64_t r0 = tt * LG_ETILE;
            const int64_t lim = tt < ntiles ? min((int64_t)LG_ETILE, a.n - r0) * D : 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int e = tid + 256 * j;
                pre[j] = e < lim ? x[r0 * D + e] : 0.0;
            }
        };
        if (reg_prefetch) fetch_tile(blockIdx.x);
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
            const int64_t row0 = t * LG_ETILE;
            const int rows = (int)min((int64_t)LG_ETILE, a.n - row0);
            asm volatile("bar.sync 1, 256;" ::: "memory");     // every GEMM warp is done with the previous X tile
            if (reg_prefetch) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int e = tid + 256 * j;
                    if (e < LG_ETILE * D) {
                        const int r = e / D, c = e - r * D;
                        xs[r * XP + c] = pre[j];
                    }
                }
                fetch_tile(t + gridDim.x);
            } else {
                for (int e = tid; e < LG_ETILE * D; e += 256) {
                    const int r = e / D, c = e - r * D;
                    xs[r * XP + c] = (e < rows * D) ? x[row0 * D + e] : 0.0;
                }
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            double acc[2][KB][2];
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) { acc[m][kb][0] = 0.0; acc[m][kb][1] = 0.0; }
            for (int c = 0; c < nchunk; ++c, ++cc) {
                const int b = (int)(cc & 1);
                // A fragments of this chunk: logical features 64c + 16w + {q, 4+q, 8+q, 12+q}, w = 0..3
                double af[4][4];
                const unsigned short* tb = tabS + LG_CW * c + q;
#pragma unroll
                for (int w = 0; w < 4; ++w)
#pragma unroll
                    for (int h = 0; h < 4; ++h) {
                        const unsigned int code = tb[16 * w + 4 * h];
                        af[w][h] = xr[code >> 8] * xr[code & 0xFF];     // columns D, D + 1 of the tile hold 1 and 0
                    }
                mbar_wait(&cfull[b], (uint32_t)((cc >> 1) & 1));
                const double* eB = coefS + b * 8 * KB * LG_CW + g * LG_CW;
#pragma unroll
                for (int w = 0; w < LG_CW / 16; ++w) {
#pragma unroll
                    for (int kb = 0; kb < KB; ++kb) {
                        const double2 b0 = lds2(eB + kb * 8 * LG_CW + 16 * w + eo0);
                        const double2 b1 = lds2(eB + kb * 8 * LG_CW + 16 * w + eo1);
                        dmma(acc[0][kb][0], acc[0][kb][1], af[w][0], b0.x);      // feature 16w + q
                        dmma(acc[1][kb][0], acc[1][kb][1], af[w][1], b0.y);      // feature 16w + 4 + q
                        dmma(acc[0][kb][0], acc[0][kb][1], af[w][2], b1.x);      // feature 16w + 8 + q
                        dmma(acc[1][kb][0], acc[1][kb][1], af[w][3], b1.y);      // feature 16w + 12 + q
                    }
                }
                mbar_arrive(&cempty[b]);
            }
            double lr[KB][2];
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) {
                lr[kb][0] = acc[0][kb][0] + acc[1][kb][0];
                lr[kb][1] = acc[0][kb][1] + acc[1][kb][1];
            }
            // ---- softmax over k for row lrow; this thread holds components 8kb + 2q + {0,1} ----
            const int64_t grow = row0 + lrow;
            const bool valid = lrow < rows;
            if constexpr (NG > 1) {
                // batched mixtures: one softmax per group of GB blocks; r -> HBM, entropy per group; nothing else is produced
#pragma unroll
                for (int gi = 0; gi < NG; ++gi) {
                    double gmx = -INFINITY;
#pragma unroll
                    for (int kb = gi * GB; kb < (gi + 1) * GB; ++kb) gmx = fmax(gmx, fmax(lr[kb][0], lr[kb][1]));
                    gmx = fmax(gmx, __shfl_xor_sync(0xffffffffu, gmx, 1));
                    gmx = fmax(gmx, __shfl_xor_sync(0xffffffffu, gmx, 2));
                    double gsum = 0.0, gdot = 0.0;
#pragma unroll
                    for (int kb = gi * GB; kb < (gi + 1) * GB; ++kb)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double z = lr[kb][e] - gmx;
                            const double ex = exp_nonpos(z);
                            lr[kb][e] = ex;
                            gsum += ex;
                            gdot = fma(ex, z, gdot);
                        }
                    gsum += __shfl_xor_sync(0xffffffffu, gsum, 1);
                    gsum += __shfl_xor_sync(0xffffffffu, gsum, 2);
                    gdot += __shfl_xor_sync(0xffffffffu, gdot, 1);
                    gdot += __shfl_xor_sync(0xffffffffu, gdot, 2);
                    const double ginv = valid ? 1.0 / gsum : 0.0;
                    if (valid && q == 0) { ent[gi] = fma(gdot, ginv, ent[gi]); sprod[gi] *= gsum; }
                    if ((it & 7) == 7) { ent[gi] -= log(sprod[gi]); sprod[gi] = 1.0; }
#pragma unroll
                    for (int kb = gi * GB; kb < (gi + 1) * GB; ++kb)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int k = 8 * kb + 2 * q + e;
                            if (valid && k < K) a.r_out[grow * K + k] = lr[kb][e] * ginv;
                        }
                }
                continue;
            }
            double mx = -INFINITY;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) mx = fmax(mx, fmax(lr[kb][0], lr[kb][1]));
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
            mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
            if (a.lnrho_out != nullptr && valid) {
#pragma unroll
                for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int k = 8 * kb + 2 * q + e;
                        if (k < K) a.lnrho_out[grow * K + k] = lr[kb][e];
                    }
            }
            if (a.lnrho_only) {                             // HMM emission pass: the scan kernels take over from here
                if (valid && a.rhohat_out != nullptr) {
#pragma unroll
                    for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int k = 8 * kb + 2 * q + e;
                            if (k < K) a.rhohat_out[grow * K + k] = exp_nonpos(lr[kb][e] - mx);
                        }
                    if (q == 0) a.rowmax_out[grow] = mx;
                }
                continue;
            }
            double sum = 0.0, dot = 0.0;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double z = lr[kb][e] - mx;
                    const double ex = exp_nonpos(z);
                    lr[kb][e] = ex;
                    sum += ex;
                    dot = fma(ex, z, dot);
                }
            sum += __shfl_xor_sync(0xffffffffu, sum, 1);
            sum += __shfl_xor_sync(0xffffffffu, sum, 2);
            dot += __shfl_xor_sync(0xffffffffu, dot, 1);
            dot += __shfl_xor_sync(0xffffffffu, dot, 2);
            const double inv = valid ? 1.0 / sum : 0.0;
            if (valid && q == 0) { ent[0] = fma(dot, inv, ent[0]); sprod[0] *= sum; }
            if ((it & 7) == 7) { ent[0] -= log(sprod[0]); sprod[0] = 1.0; }
            int best = 0x7fffffff;
            double bestv = -1.0;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double r = lr[kb][e] * inv;
                    const int k = 8 * kb + 2 * q + e;
                    if (r > bestv) { bestv = r; best = k; }
                    if (valid && k < K) a.r_out[grow * K + k] = r;      // r_out is mandatory in this regime (the M kernel's input)
                }
            if (a.argmax_out != nullptr) {
#pragma unroll
                for (int o = 1; o <= 2; o <<= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bestv, o);
                    const int ok = __shfl_xor_sync(0xffffffffu, best, o);
                    if (ov > bestv || (ov == bestv && ok < best)) { bestv = ov; best = ok; }
                }
                if (valid && q == 0) a.argmax_out[grow] = best;
            }
        }
#pragma unroll
        for (int gi = 0; gi < NG; ++gi) ent[gi] -= log(sprod[gi]);
    }
#pragma unroll
    for (int gi = 0; gi < NG; ++gi) {
        const double v = block_sum(ent[gi], red);
        if (tid == 0) ews[(int64_t)blockIdx.x * 8 + gi] = v;          // per CTA: 8 slots, one per group
    }
}

// Output-stationary statistics GEMM.  A CTA owns the 128-feature chunk cx for the rows of split ry; warp w owns the
// feature blocks 2w, 2w+1 and thread column g of each, i.e. two FIXED features per thread, whose Phi values (the B
// fragments) it forms in registers from the X tile: two in-stream DMULs per 2*KB DMMAs, no Phi tile in shared memory.
// X tiles (double buffered) and r tiles arrive by TMA one step ahead; r is re-laid out into the swizzled A-fragment tile.
template <int KB>
__global__ void __launch_bounds__(LG_THREADS, 2)
m_large_kernel(const PassArgs a, const Layout L, const double* __restrict__ ews, const int n_ews, const int nsplit) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int RP = (8 * KB < 16) ? 16 : 8 * KB;
    const int K = L.K, D = L.D, P = L.P;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust)) return;
    const double* __restrict__ x = static_cast<const double*>(a.x);
    const double* __restrict__ rws = a.r_out;

    double* rS = reinterpret_cast<double*>(smem_raw);          // [32][RP] swizzled A-fragment tile
    double* xs = rS + LG_MSUB * RP;                            // [2 stages][32][D]   TMA destination
    double* rst = xs + 2 * LG_MSUB * D;                        // [32][K]             TMA destination (row-major, as in HBM)
    uint64_t* bars = reinterpret_cast<uint64_t*>(rst + ((LG_MSUB * K + 1) & ~1));   // [2]
    const uint32_t xbytes = (uint32_t)(LG_MSUB * D * sizeof(double)), rbytes = (uint32_t)(LG_MSUB * K * sizeof(double));
    if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    uint32_t ph[2] = {0u, 0u};

    const int cx = blockIdx.x, ry = blockIdx.y;
    const int64_t nsub = (a.n + LG_MSUB - 1) / LG_MSUB;
    const int64_t per = (nsub + nsplit - 1) / nsplit;
    const int64_t s_begin = ry * per, s_end = min(nsub, s_begin + per);

    // this thread's two features (logical order: B column g of block b is feature 128cx + 8b + g)
    // as x[a] * x[b] with unconditional loads and selects for the constant factors (no branches in the GEMM loop)
    int kind0, i0, j0, kind1, i1, j1;
    feat_decode(LG_MCW * cx + 8 * (2 * warp) + g, D, P, kind0, i0, j0);
    feat_decode(LG_MCW * cx + 8 * (2 * warp + 1) + g, D, P, kind1, i1, j1);
    const bool ua0 = kind0 == 1 || kind0 == 2, ub0 = kind0 == 2, ua1 = kind1 == 1 || kind1 == 2, ub1 = kind1 == 2;
    const double cb0 = kind0 == 3 ? 0.0 : 1.0, cb1 = kind1 == 3 ? 0.0 : 1.0;
    for (int e = tid; e < LG_MSUB * RP; e += LG_THREADS) rS[e] = 0.0;     // padded components stay zero

    double macc[2][KB][2];
#pragma unroll
    for (int l = 0; l < 2; ++l)
#pragma unroll
        for (int kb = 0; kb < KB; ++kb) { macc[l][kb][0] = 0.0; macc[l][kb][1] = 0.0; }
    const int fq = fsw(q);
    const double* mR = rS + q * RP + ((2 * g) ^ fq);

    auto issue = [&](int64_t sb, int b) {                      // full 32-row steps only; a ragged last step uses plain loads
        const int64_t row0 = sb * LG_MSUB;
        if (sb < s_end && row0 + LG_MSUB <= a.n) {
            mbar_expect_tx(&bars[b], xbytes + rbytes);
            tma_load_1d(xs + b * LG_MSUB * D, x + row0 * D, xbytes, &bars[b]);
            tma_load_1d(rst, rws + row0 * K, rbytes, &bars[b]);
        }
    };
    __syncthreads();
    if (tid == 0) issue(s_begin, 0);
    int it = 0;
    for (int64_t sb = s_begin; sb < s_end; ++sb, ++it) {
        const int b = it & 1;
        const int64_t row0 = sb * LG_MSUB;
        const int rows = (int)min((int64_t)LG_MSUB, a.n - row0);
        double* xt = xs + b * LG_MSUB * D;
        if (rows == LG_MSUB) {
            mbar_wait(&bars[b], ph[b]);
            ph[b] ^= 1u;
        } else {
            for (int e = tid; e < LG_MSUB * D; e += LG_THREADS) xt[e] = (e < rows * D) ? x[row0 * D + e] : 0.0;
            for (int e = tid; e < LG_MSUB * K; e += LG_THREADS) rst[e] = (e < rows * K) ? rws[row0 * K + e] : 0.0;
            __syncthreads();
        }
        for (int e = tid; e < LG_MSUB * K; e += LG_THREADS) {
            const int r = e / K, k = e - r * K;
            const int kb = k >> 3, cc = k & 7;
            rS[r * RP + ((16 * (kb >> 1) + 2 * cc + (kb & 1)) ^ fsw(r))] = rst[e];
        }
        __syncthreads();                                       // rS built, rst free; every warp finished the previous GEMM
        if (tid == 0) issue(sb + 1, b ^ 1);                    // prefetch the next step (other X stage, the r staging tile)
#pragma unroll
        for (int ks = 0; ks < LG_MSUB / 4; ++ks) {
            double ra[KB];
            if constexpr (KB >= 2) {
#pragma unroll
                for (int v = 0; v < KB / 2; ++v) {
                    const double2 r2 = lds2(mR + ks * 4 * RP + 16 * v);
                    ra[2 * v] = r2.x;
                    ra[2 * v + 1] = r2.y;
                }
            } else {
                ra[0] = mR[ks * 4 * RP];
            }
            const double* xr = xt + (4 * ks + q) * D;
            const double xa0 = xr[i0], xb0 = xr[j0], xa1 = xr[i1], xb1 = xr[j1];
            const double b0 = (ua0 ? xa0 : 1.0) * (ub0 ? xb0 : cb0), b1 = (ua1 ? xa1 : 1.0) * (ub1 ? xb1 : cb1);
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) {
                dmma(macc[0][kb][0], macc[0][kb][1], ra[kb], b0);
                dmma(macc[1][kb][0], macc[1][kb][1], ra[kb], b1);
            }
        }
        __syncthreads();                                       // GEMM finished: rS may be rebuilt, this X stage refilled
    }

    // ---- partial of this row split (logical layout [K][pitch]); split 0 also carries the entropy term ----
    const int64_t len = L.stats_len;
    double* part = a.workspace + (int64_t)ry * len;
#pragma unroll
    for (int l = 0; l < 2; ++l) {
        const int bb = 2 * warp + l;
#pragma unroll
        for (int kb = 0; kb < KB; ++kb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int k = 8 * kb + g;                              // C fragment: row g = component, cols 2q+e = feature 8bb + 2q + e
                const int p = LG_MCW * cx + 8 * bb + 2 * q + e;
                if (k < K && p < L.pitch) part[(int64_t)k * L.pitch + p] = macc[l][kb][e];
            }
    }
    if (cx == 0 && tid < 8) {
        double v = 0.0;
        if (tid == BGMM_STATS_ENTROPY && ry == 0)
            for (int i = 0; i < n_ews; ++i) v += ews[(int64_t)i * 8];   // fixed order: deterministic (group 0; the other
                                                                        // groups of a batched pass are summed by batch_scatter)
        part[(int64_t)K * L.pitch + tid] = v;                           // the rest of the tail: 0
    }
}

// ---- host side ----
static int large_kb(int K) { return K <= 8 ? 1 : (K <= 16 ? 2 : (K <= 32 ? 4 : 8)); }

bool large_supported(int K, int D, int dtype) { return dtype == BGMM_F64 && K >= 1 && K <= 64 && D >= 1 && D <= 128; }

// upper bound of the M kernel's row splits (= partial statistics buffers in the workspace): few feature chunks (small D)
// need many splits to fill the GPU, many chunks need few
static int large_max_split(int D) {
    const int n_chunks = (feat_pitch(D) + LG_MCW - 1) / LG_MCW;
    const int s = 320 / n_chunks;
    return s < 4 ? 4 : s;
}

static void large_plan(int K, int D, int64_t n, int& grid_e, int& n_chunks, int& nsplit) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t ntiles = (n + LG_ETILE - 1) / LG_ETILE;
    grid_e = (int)(ntiles < 1 ? 1 : (ntiles < sms ? ntiles : sms));
    n_chunks = (feat_pitch(D) + LG_MCW - 1) / LG_MCW;
    const int64_t nsub = (n + LG_MSUB - 1) / LG_MSUB;
    int64_t s = (2 * sms) / n_chunks;                                   // ONE resident wave (2 CTAs per SM): no tail wave
    if (s > large_max_split(D)) s = large_max_split(D);
    if (s > nsub) s = nsub;
    if (s < 1) s = 1;
    nsplit = (int)s;
}

int64_t large_workspace_doubles(int K, int D) {
    if (K > 64 || D > 128) return 0;
    const int64_t nchunk = (feat_count(D) + LG_CW - 1) / LG_CW;
    // <= 64 row splits + E-kernel entropy partials (8 group slots per CTA) + the packed coefficient image
    // (nchunk x [8*KB][64]) + the (i, j) table
    return (int64_t)large_max_split(D) * ((int64_t)K * feat_pitch(D) + 8) + 8 * 160 + nchunk * 64 * LG_CW +
           (nchunk * LG_CW + 3) / 4 + 8;
}

// which = 1: E kernel (+ coefficient image / feature table), 2: M kernel (+ reduction over the row splits), 3: both
template <int KB, int GB>
static int launch_large_t(const PassArgs& a, const Layout& L, int which, cudaStream_t stream) {
    int grid_e, n_chunks, nsplit;
    large_plan(L.K, L.D, a.n, grid_e, n_chunks, nsplit);
    const int64_t len = L.stats_len;
    double* ews = a.workspace + (int64_t)large_max_split(L.D) * len;
    double* packed = ews + 8 * 160;
    const int nchunk_e = (L.P + LG_CW - 1) / LG_CW;
    unsigned short* ftab = reinterpret_cast<unsigned short*>(packed + (int64_t)nchunk_e * 8 * KB * LG_CW);
    if (which & 1) {
        const size_t smem_e = sizeof(double) * ((size_t)2 * 8 * KB * LG_CW + (size_t)LG_ETILE * (L.D + 2) + 40) +
                              4 * sizeof(uint64_t) + sizeof(unsigned short) * (size_t)nchunk_e * LG_CW + 128;
        cudaError_t e = cudaFuncSetAttribute(e_large_kernel<KB, GB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_e);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(e_large)");
        launch(coef_pack_kernel<KB>, nchunk_e, LG_THREADS, 0, stream, a.state, L, packed, a.force, a.ignore_robust);
        launch(feat_table_kernel, (nchunk_e * LG_CW + 255) / 256, 256, 0, stream, ftab, L.D, L.P, nchunk_e * LG_CW);
        launch(e_large_kernel<KB, GB>, grid_e, LG_ETHREADS, smem_e, stream, a, L, ews, packed, ftab);
    }
    if (which & 2) {
        constexpr int RP = (8 * KB < 16) ? 16 : 8 * KB;
        const size_t smem_m = sizeof(double) * ((size_t)LG_MSUB * RP + (size_t)2 * LG_MSUB * L.D + (size_t)LG_MSUB * L.K + 2) +
                              2 * sizeof(uint64_t) + 128;
        cudaError_t e = cudaFuncSetAttribute(m_large_kernel<KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(m_large)");
        launch(m_large_kernel<KB>, dim3(n_chunks, nsplit), LG_THREADS, smem_m, stream, a, L, ews, grid_e, nsplit);
        launch_reduce_partials(a, L, nsplit, stream);
    }
    return check_cuda(cudaGetLastError(), "pass_large launch");
}

int launch_pass_large_part(const PassArgs& a, int K, int D, int dtype, int which, cudaStream_t stream, int group_blocks) {
    if (!large_supported(K, D, dtype)) {
        set_error("bgmm_pass(large): unsupported shape K=%d D=%d dtype=%d", K, D, dtype);
        return BGMM_ENOSUP;
    }
    if ((which & 2) && a.r_out == nullptr) {
        set_error("bgmm_pass(large): r_out ([n][K] float64) is required in this regime (it is the M kernel's input)");
        return BGMM_EINVAL;
    }
    const Layout L = make_layout(K, D, 1);
    const int kb = large_kb(K), gb = group_blocks > 0 ? group_blocks : kb;      // gb < kb: batched mixtures (softmax groups)
#define BGMM_LG_CASE(KBv, GBv) if (kb == KBv && gb == GBv) return launch_large_t<KBv, GBv>(a, L, which, stream);
    BGMM_LG_CASE(1, 1)
    BGMM_LG_CASE(2, 2) BGMM_LG_CASE(2, 1)
    BGMM_LG_CASE(4, 4) BGMM_LG_CASE(4, 2) BGMM_LG_CASE(4, 1)
    BGMM_LG_CASE(8, 8) BGMM_LG_CASE(8, 4) BGMM_LG_CASE(8, 2) BGMM_LG_CASE(8, 1)
#undef BGMM_LG_CASE
    set_error("bgmm_pass(large): no instantiation for %d component blocks in groups of %d", kb, gb);
    return BGMM_ENOSUP;
}

int launch_pass_large(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream) {
    return launch_pass_large_part(a, K, D, dtype, 3, stream, 0);
}

// ---- batched mixtures (bgmm_pass_batched): R member states share one sweep over X through a "super" state block ----
// gather: coefficient rows of every member's current parameter set -> rows [r * Kp, r * Kp + K) of the super state's set 0
// (rows K..Kp-1 of each group: ln rho = -1e300, i.e. r == 0 exactly); super ctrl.done = every member is done.
__global__ void __launch_bounds__(128) batch_gather_kernel(const BatchDesc bd, double* __restrict__ sup, const Layout Ls,
                                                           const Layout Lm, const int Kp) {
    const int ke = blockIdx.x, r = ke / Kp, k = ke - r * Kp;
    const double* st = bd.st[r];
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + Lm.ctrl);
    double* dst = sup + Ls.params[0] + Ls.p_coef + (int64_t)ke * Ls.pitch;
    if (k < Lm.K) {
        const double* src = st + Lm.params[ctrl[BGMM_CTRL_CUR]] + Lm.p_coef + (int64_t)k * Lm.pitch;
        for (int p = threadIdx.x; p < Ls.pitch; p += 128) dst[p] = src[p];
    } else {
        for (int p = threadIdx.x; p < Ls.pitch; p += 128) dst[p] = p == 0 ? -1.0e300 : 0.0;
    }
    if (ke == 0 && threadIdx.x == 0) {
        int all_done = 1;
        for (int i = 0; i < bd.R; ++i)
            all_done &= reinterpret_cast<const volatile int*>(bd.st[i] + Lm.ctrl)[BGMM_CTRL_DONE] != 0;
        volatile int* sc = reinterpret_cast<volatile int*>(sup + Ls.ctrl);
        sc[BGMM_CTRL_CUR] = 0; sc[BGMM_CTRL_DONE] = all_done; sc[BGMM_CTRL_ROBUST] = 0;
    }
}

// scatter: statistics rows of group r -> member r's STATS (+ tail: the group's entropy term summed over the E kernel's
// CTAs in a fixed order, the row count, format 0).  Members that are done keep their last statistics.
__global__ void __launch_bounds__(128) batch_scatter_kernel(const BatchDesc bd, const double* __restrict__ sup, const Layout Ls,
                                                            const Layout Lm, const int Kp, const double* __restrict__ ews,
                                                            const int n_ews, const double rows) {
    const volatile int* sc = reinterpret_cast<const volatile int*>(sup + Ls.ctrl);
    if (sc[BGMM_CTRL_DONE]) return;
    const int r = blockIdx.x / (Lm.K + 1), k = blockIdx.x - r * (Lm.K + 1);
    double* st = bd.st[r];
    if (reinterpret_cast<const volatile int*>(st + Lm.ctrl)[BGMM_CTRL_DONE]) return;
    if (k < Lm.K) {
        const double* src = sup + Ls.stats + (int64_t)(r * Kp + k) * Ls.pitch;
        double* dst = st + Lm.stats + (int64_t)k * Lm.pitch;
        for (int p = threadIdx.x; p < Lm.pitch; p += 128) dst[p] = src[p];
    } else if (threadIdx.x == 0) {
        double v = 0.0;
        for (int i = 0; i < n_ews; ++i) v += ews[(int64_t)i * 8 + r];
        double* tail = st + Lm.stats + (int64_t)Lm.K * Lm.pitch;
        tail[BGMM_STATS_ENTROPY] = v; tail[BGMM_STATS_ROWS] = rows; tail[BGMM_STATS_FORMAT] = 0.0;
        for (int o = BGMM_STATS_FORMAT + 1; o < 8; ++o) tail[o] = 0.0;
    }
}

int launch_pass_batched(const void* x, int64_t n, int K, int D, const BatchDesc& bd, double* sup, double* workspace,
                        double* r_scratch, cudaStream_t stream) {
    const int Kp = (K + 7) & ~7, Ke = bd.R * Kp;
    if (!large_supported(Ke, D, BGMM_F64) || bd.R < 2 || bd.R > BGMM_MAX_BATCH) {
        set_error("bgmm_pass_batched: unsupported batch (K=%d -> %d per group, R=%d, D=%d; R * Kp <= 64)", K, Kp, bd.R, D);
        return BGMM_ENOSUP;
    }
    const Layout Ls = make_layout(Ke, D, 1), Lm = make_layout(K, D, 1);
    launch(batch_gather_kernel, Ke, 128, 0, stream, bd, sup, Ls, Lm, Kp);
    PassArgs a{x, n, sup, workspace, r_scratch, nullptr, nullptr, nullptr, 0};
    a.ignore_robust = 1;                                        // a flagged member is redone by its own DIRECT pass (caller)
    const int rc = launch_pass_large_part(a, Ke, D, BGMM_F64, 3, stream, Kp / 8);
    if (rc) return rc;
    int grid_e, n_chunks, nsplit;
    large_plan(Ke, D, n, grid_e, n_chunks, nsplit);
    const double* ews = workspace + (int64_t)large_max_split(D) * Ls.stats_len;
    launch(batch_scatter_kernel, bd.R * (K + 1), 128, 0, stream, bd, sup, Ls, Lm, Kp, ews, grid_e, (double)n);
    return check_cuda(cudaGetLastError(), "pass_batched launch");
}

}  // namespace bgmm
