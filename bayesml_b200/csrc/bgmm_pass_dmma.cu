// bgmm_pass, fp64 tensor-pipe variant (BGMM_PASS_DMMA) for sm_100a.
//
// One fused sweep over the centred rows of X per VB iteration; r never touches HBM (HBM traffic = X once).
// Persistent, warp-specialised CTA (one per SM, 384 threads = 3 warpgroups) working on 32-sample sub-tiles:
//
//   producer warpgroup (warps 8-11)
//     - keeps a 2-stage ring of X sub-tiles filled by TMA bulk copies (cp.async.bulk + mbarrier complete_tx),
//     - expands each sub-tile into the feature tile Phi[32][SP] (phi = [1, x, x_i x_j (i>=j)], zero padded) in a
//       4-stage shared-memory ring (full/empty mbarriers towards the consumers);
//   consumer warpgroups A (warps 0-3) and B (warps 4-7), ping-pong on alternate sub-tiles, each doing
//     - E-GEMM on the FP64 tensor pipe:  ln rho[32][K] = Phi . coef^T   (mma.sync.m8n8k4.f64 = SASS DMMA.8x8x4;
//       warp = one 8-row m-block x all K components x the full feature range, no cross-warp reduction),
//     - softmax over k in the accumulator fragments (quad shuffles), entropy term, optional r / ln rho / argmax
//       stores, r tile -> shared memory (one buffer per warpgroup),
//     - M-GEMM on the same pipe:  raw[K][SP] += R^T . Phi   with the K x SP accumulators resident in registers for
//       the whole sweep (warp = all K components x SP/32 feature blocks).
//   While one consumer warpgroup is in its (non-DMMA) softmax, the other one and the producer keep the DMMA pipe and
//   the LSU busy.  At the end the two consumer warpgroups merge their accumulators through shared memory, the CTA
//   writes ONE partial statistics buffer, and reduce_partials_kernel sums the partials in a fixed order (deterministic).
//
// Replaces `_update_q_z` :772-784 (incl. the K-loop of N x D temporaries), `_calc_n_x_bar_s` :725-732 and the
// `xlogy` term :704 of /root/reference/bayesml/gaussianmixture/_gaussianmixture.py.
//
// Shared-memory layout: rows of Phi / coef / R are stored with a "k-step pair" column permutation
// (logical feature p = 8u + 4h + q  ->  physical column 8u + 2q + h) so that one LDS.128 yields the A (or B)
// fragments of two consecutive k-steps, and with a 16-byte-chunk XOR swizzle  f(row) = ((row&1)<<2)|(row&2)
// that makes every fragment load (LDS.128 by quarter-warp, LDS.64 by half-warp) bank-conflict free.  All fragment
// addresses are loop-invariant pointers plus immediates.
#include "bgmm_common.cuh"
#include "bgmm_mma.cuh"
#include <math.h>

namespace bgmm {

constexpr int DM_THREADS = 384;      // consumer warpgroups A, B + producer warpgroup
constexpr int DM_TILE = 32;          // samples per sub-tile = 4 m-blocks (one per consumer warp)
constexpr int DM_NXS = 2;            // stages of the X ring (TMA); small, so that the Phi ring can have 4 stages
constexpr int DM_XPAD = 4;           // doubles of slack after each X stage (vector loads past the last row)
constexpr int DM_MAXG = 64;          // entries of the Phi-expansion group table

template <int KB, int SP, int NPS>
__global__ void __launch_bounds__(DM_THREADS, 1)
pass_dmma_kernel(const PassArgs a, const Layout L) {
    constexpr int RP = (8 * KB < 16) ? 16 : 8 * KB;          // pitch of the r tile (multiple of 16)
    constexpr int MAXNB = SP / 32;                            // M-GEMM n-blocks (8 features) owned by one consumer warp
    constexpr int EG = SP / 16;                               // E-GEMM: groups of 16 physical columns (4 k-steps each)
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int K = L.K, D = L.D, P = L.P;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
    const int wg = warp >> 2, wq = warp & 3;                  // warpgroup (0,1 consumers; 2 producer), warp in group
    pdl_trigger();
    pdl_wait();
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust)) return;
    const double* __restrict__ coef_g = a.state + L.params[ctrl[BGMM_CTRL_CUR]] + L.p_coef;
    const double* __restrict__ x = static_cast<const double*>(a.x);

    // ---- carve shared memory ----
    const int xstage = DM_TILE * D + DM_XPAD;
    double* phiS = reinterpret_cast<double*>(smem_raw);                  // [NPS][32][SP]
    double* coefS = phiS + NPS * DM_TILE * SP;                           // [8*KB][SP]
    double* rS = coefS + 8 * KB * SP;                                    // [2 groups][32][RP]
    double* xS = rS + 2 * DM_TILE * RP;                                  // [NXS][32*D + pad]
    double* red = xS + DM_NXS * xstage;                                  // [40]
    uint64_t* xfull = reinterpret_cast<uint64_t*>(red + 40);             // [NXS]
    uint64_t* pfull = xfull + DM_NXS;                                    // [NPS]
    uint64_t* pempty = pfull + NPS;                                      // [NPS]
    uint2* gtab = reinterpret_cast<uint2*>(pempty + NPS);                // [DM_MAXG]

    const int64_t nsub = (a.n + DM_TILE - 1) / DM_TILE;                  // sub-tiles in this rank's rows
    const int nloc = (int)((nsub - blockIdx.x + gridDim.x - 1) / gridDim.x);   // sub-tiles of this CTA (>= 0)
    const uint32_t tile_bytes = (uint32_t)(DM_TILE * D * sizeof(double));

    if (tid == 0) {
        for (int i = 0; i < DM_NXS; ++i) mbar_init(&xfull[i], 1);
        for (int i = 0; i < NPS; ++i) { mbar_init(&pfull[i], 128); mbar_init(&pempty[i], 128); }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");

    // ---- one-time: swizzled coefficient matrix; tile-invariant columns of Phi (constant 1, zero padding);
    //      group table of the Phi expansion: entry = (i, 4*jb, flags) + 4 physical columns (0xFF = masked) ----
    for (int e = tid; e < 8 * KB * SP; e += DM_THREADS) {
        const int k = e / SP, p = e - k * SP;
        double v = 0.0;
        if (k < K) { if (p < P) v = coef_g[(int64_t)k * L.pitch + p]; }
        else if (p == 0) v = -1.0e300;                                    // padded components: r == 0 exactly
        coefS[swz(k, phys_col(p), SP)] = v;
    }
    for (int e = tid; e < NPS * DM_TILE * (SP - P + 1); e += DM_THREADS) {
        const int r = e / (SP - P + 1), c = e - r * (SP - P + 1);        // r runs over all rows of all stages
        if (c == 0) phiS[swz(r, phys_col(0), SP)] = 1.0;
        else phiS[swz(r, phys_col(P + c - 1), SP)] = 0.0;
    }
    const int nlin = (D + 3) / 4;                                         // linear groups: x_j * 1
    int ngq = 0;
    for (int i = 0; i < D; ++i) ngq += i / 4 + 1;                         // quadratic groups: x_i * x_{4jb..4jb+3}, j <= i
    const int ngt = nlin + ngq;
    for (int gi = tid; gi < ngt; gi += DM_THREADS) {
        uint32_t lo, hi = 0;
        if (gi < nlin) {
            lo = 0xFFu | ((uint32_t)(4 * gi) << 8);                       // i = 0xFF: multiplier 1.0
            for (int c = 0; c < 4; ++c) {
                const int j = 4 * gi + c;
                hi |= (uint32_t)(j < D ? phys_col(1 + j) : 0xFF) << (8 * c);
            }
        } else {
            int rem = gi - nlin, i = 0;
            while (rem >= i / 4 + 1) { rem -= i / 4 + 1; ++i; }
            lo = (uint32_t)i | ((uint32_t)(4 * rem) << 8);
            for (int c = 0; c < 4; ++c) {
                const int j = 4 * rem + c;
                hi |= (uint32_t)(j <= i ? phys_col(1 + D + i * (i + 1) / 2 + j) : 0xFF) << (8 * c);
            }
        }
        gtab[gi] = make_uint2(lo, hi);
    }
    __syncthreads();

    double ent = 0.0;
    const int64_t len = L.stats_len;

    if (wg == 2) {
        // =========================== PRODUCER WARPGROUP ===========================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");      // hand registers to the consumer warpgroups
        const int ptid = tid - 256;
        auto issue_tile = [&](int j) {                                    // local sub-tile j -> X stage j % NXS (full tiles only)
            const int64_t row0 = ((int64_t)blockIdx.x + (int64_t)j * gridDim.x) * DM_TILE;
            if (j < nloc && row0 + DM_TILE <= a.n) {
                const int st = j % DM_NXS;
                mbar_expect_tx(&xfull[st], tile_bytes);
                tma_load_1d(xS + st * xstage, x + row0 * D, tile_bytes, &xfull[st]);
            }
        };
        if (ptid == 0)
            for (int j = 0; j < DM_NXS; ++j) issue_tile(j);
        const int q128 = 128 / ngt, r128 = 128 % ngt;
        const bool even_d = (D & 1) == 0;
        for (int j = 0; j < nloc; ++j) {
            const int xs = j % DM_NXS, ps = j % NPS;
            const int64_t row0 = ((int64_t)blockIdx.x + (int64_t)j * gridDim.x) * DM_TILE;
            const int rows = (int)min((int64_t)DM_TILE, a.n - row0);
            double* xt = xS + xs * xstage;
            if (rows == DM_TILE) {
                mbar_wait(&xfull[xs], (uint32_t)((j / DM_NXS) & 1));
            } else {                                                      // ragged last sub-tile: plain loads, zero fill
                for (int e = ptid; e < DM_TILE * D; e += 128) xt[e] = (e < rows * D) ? x[row0 * D + e] : 0.0;
                wg_sync(1);
            }
            if (j >= NPS) mbar_wait(&pempty[ps], (uint32_t)(((j / NPS) - 1) & 1));
            double* ph = phiS + ps * DM_TILE * SP;
            int r = ptid / ngt, gi = ptid - r * ngt;
            while (r < DM_TILE) {
                const uint2 e = gtab[gi];
                const int i = e.x & 0xFF, j4 = (e.x >> 8) & 0xFF;
                const double* xr = xt + r * D;
                const double xi = (i == 0xFF) ? 1.0 : xr[i];
                double v0, v1, v2, v3;
                if (even_d) {
                    const double2 u0 = lds2(xr + j4), u1 = lds2(xr + j4 + 2);
                    v0 = u0.x; v1 = u0.y; v2 = u1.x; v3 = u1.y;
                } else {
                    v0 = xr[j4]; v1 = xr[j4 + 1]; v2 = xr[j4 + 2]; v3 = xr[j4 + 3];
                }
                double* pr = ph + r * SP;
                const int f = fsw(r);
                const int c0 = e.y & 0xFF, c1 = (e.y >> 8) & 0xFF, c2 = (e.y >> 16) & 0xFF, c3 = e.y >> 24;
                if (c0 != 0xFF) pr[c0 ^ f] = xi * v0;
                if (c1 != 0xFF) pr[c1 ^ f] = xi * v1;
                if (c2 != 0xFF) pr[c2 ^ f] = xi * v2;
                if (c3 != 0xFF) pr[c3 ^ f] = xi * v3;
                gi += r128; r += q128;
                if (gi >= ngt) { gi -= ngt; ++r; }
            }
            mbar_arrive(&pfull[ps]);                                      // 128 arrivals complete the phase
            wg_sync(1);                                                   // every producer thread is done with this X stage
            if (ptid == 0) issue_tile(j + DM_NXS);
        }
    } else {
        // =========================== CONSUMER WARPGROUPS ===========================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");     // 2*128*208 + 128*88 = 64512 <= 65536 registers
        double macc[MAXNB][KB][2];
#pragma unroll
        for (int l = 0; l < MAXNB; ++l)
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) { macc[l][kb][0] = 0.0; macc[l][kb][1] = 0.0; }

        // loop-invariant fragment offsets (all swizzles resolved here; the loops below use immediates only)
        const int fg = fsw(g), fq = fsw(q);
        const int lrow = 8 * wq + g;                          // row of the sub-tile this thread finalises in the softmax
        const int eAo = lrow * SP;
        const double* eB = coefS + g * SP;
        const int eo0 = (2 * q) ^ fg, eo1 = (8 + 2 * q) ^ fg;
        const int rsto = lrow * RP + ((4 * q) ^ fg);
        const int mRo = q * RP + ((2 * g) ^ fq);
        int mPo[MAXNB];
#pragma unroll
        for (int l = 0; l < MAXNB; ++l) mPo[l] = q * SP + ((8 * (wq + 4 * l) + g) ^ fq);   // n-block b = wq + 4l

        int jj = 0;
        double sprod = 1.0;
        for (int j = wg; j < nloc; j += 2, ++jj) {
            const int ps = j % NPS;
            const int64_t row0 = ((int64_t)blockIdx.x + (int64_t)j * gridDim.x) * DM_TILE;
            const int rows = (int)min((int64_t)DM_TILE, a.n - row0);
            const double* ph = phiS + ps * DM_TILE * SP;
            double* rb = rS + wg * DM_TILE * RP;
            mbar_wait(&pfull[ps], (uint32_t)((j / NPS) & 1));

            // ---- E-GEMM: m-block wq, all KB n-blocks, all EG column groups; two accumulator sets for ILP ----
            double acc[2][KB][2];
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) { acc[m][kb][0] = 0.0; acc[m][kb][1] = 0.0; }
            const double* eA = ph + eAo;
#pragma unroll
            for (int w = 0; w < EG; ++w) {
                const double2 a0 = lds2(eA + 16 * w + eo0), a1 = lds2(eA + 16 * w + eo1);
                double2 b0[KB], b1[KB];
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    b0[kb] = lds2(eB + kb * 8 * SP + 16 * w + eo0);
                    b1[kb] = lds2(eB + kb * 8 * SP + 16 * w + eo1);
                }
                // the .x and .y k-steps of one LDS.128 accumulate into different sets: whatever order ptxas picks,
                // two consecutive DMMAs never depend on each other (DMMA latency ~29 cycles, issue interval 16)
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    dmma(acc[0][kb][0], acc[0][kb][1], a0.x, b0[kb].x);
                    dmma(acc[1][kb][0], acc[1][kb][1], a0.y, b0[kb].y);
                }
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    dmma(acc[0][kb][0], acc[0][kb][1], a1.x, b1[kb].x);
                    dmma(acc[1][kb][0], acc[1][kb][1], a1.y, b1[kb].y);
                }
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
            double sum = 0.0, dot = 0.0;
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double z = lr[kb][e] - mx;
                    const double ex = exp_nonpos(z);
                    lr[kb][e] = ex;
                    sum += ex;
                    dot = fma(ex, z, dot);              // z is finite (padding uses -1e300), so 0 * z == 0
                }
            sum += __shfl_xor_sync(0xffffffffu, sum, 1);
            sum += __shfl_xor_sync(0xffffffffu, sum, 2);
            dot += __shfl_xor_sync(0xffffffffu, dot, 1);
            dot += __shfl_xor_sync(0xffffffffu, dot, 2);
            const double inv = valid ? 1.0 / sum : 0.0;     // rows past the end contribute r = 0
            // sum_k r ln r = dot/sum - ln(sum); 1 <= sum <= K, so the logs of up to 8 rows are taken as one log of a product
            if (valid && q == 0) { ent = fma(dot, inv, ent); sprod *= sum; }
            if ((jj & 7) == 7) { ent -= log(sprod); sprod = 1.0; }
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) { lr[kb][0] *= inv; lr[kb][1] *= inv; }
            // r tile: physical column 16(kb>>1) + 4q + 2e + (kb&1), swizzle folded into rsto
            double* rst = rb + rsto;
            if constexpr (KB >= 2) {
#pragma unroll
                for (int v = 0; v < KB / 2; ++v)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                        *reinterpret_cast<double2*>(rst + 16 * v + 2 * e) = make_double2(lr[2 * v][e], lr[2 * v + 1][e]);
            } else {
                rst[0] = lr[0][0];
                rst[2] = lr[0][1];
            }
            if (a.r_out != nullptr && valid) {
#pragma unroll
                for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int k = 8 * kb + 2 * q + e;
                        if (k < K) a.r_out[grow * K + k] = lr[kb][e];
                    }
            }
            if (a.argmax_out != nullptr) {
                int best = 0x7fffffff;
                double bestv = -1.0;
#pragma unroll
                for (int kb = 0; kb < KB; ++kb)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                        if (lr[kb][e] > bestv) { bestv = lr[kb][e]; best = 8 * kb + 2 * q + e; }   // ascending k: first wins
#pragma unroll
                for (int o = 1; o <= 2; o <<= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, bestv, o);
                    const int ok = __shfl_xor_sync(0xffffffffu, best, o);
                    if (ov > bestv || (ov == bestv && ok < best)) { bestv = ov; best = ok; }
                }
                if (valid && q == 0) a.argmax_out[grow] = best;
            }
            wg_sync(2 + wg);          // r tile of this warpgroup complete

            // ---- M-GEMM: raw[k][p] += sum_n r[n][k] phi[n][p]; A = R^T (8 comps x 4 samples), B = Phi (4 x 8) ----
            const double* mR = rb + mRo;
#pragma unroll
            for (int ks = 0; ks < DM_TILE / 4; ++ks) {
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
                double bfr[MAXNB];
#pragma unroll
                for (int l = 0; l < MAXNB; ++l) bfr[l] = ph[mPo[l] + ks * 4 * SP];
#pragma unroll
                for (int l = 0; l < MAXNB; ++l)
#pragma unroll
                    for (int kb = 0; kb < KB; ++kb) dmma(macc[l][kb][0], macc[l][kb][1], ra[kb], bfr[l]);
            }
            mbar_arrive(&pempty[ps]);                                     // this thread is done with the Phi stage
            wg_sync(2 + wg);          // every warp of the group has read the r tile: it may be overwritten (single buffer)
        }

        ent -= log(sprod);

        // ---- merge the two warpgroups' accumulators through shared memory (the Phi ring is free now) and write ONE
        //      partial per CTA (logical layout [K][pitch]); the cross-CTA sum is done by reduce_partials_kernel ----
        wg_sync(2 + wg);
        asm volatile("bar.sync 4, 256;" ::: "memory");        // both consumer warpgroups are done with every Phi stage
        double* mrg = phiS;                                    // [8*KB][SP] in (component, physical column) order
        if (wg == 1) {
#pragma unroll
            for (int l = 0; l < MAXNB; ++l)
#pragma unroll
                for (int kb = 0; kb < KB; ++kb)
                    *reinterpret_cast<double2*>(&mrg[(8 * kb + g) * SP + 8 * (wq + 4 * l) + 2 * q]) =
                        make_double2(macc[l][kb][0], macc[l][kb][1]);
        }
        asm volatile("bar.sync 4, 256;" ::: "memory");
        if (wg == 0) {
            double* part = a.workspace + (int64_t)blockIdx.x * len;
#pragma unroll
            for (int l = 0; l < MAXNB; ++l) {
                const int b = wq + 4 * l;
#pragma unroll
                for (int kb = 0; kb < KB; ++kb) {
                    const double2 o = lds2(&mrg[(8 * kb + g) * SP + 8 * b + 2 * q]);
                    const int k = 8 * kb + g;              // C fragment: row g = component, cols 2q+e = physical 8b+2q+e
                    const int p0 = 8 * b + q;              // physical 8b + 2q + e  <->  logical 8b + 4e + q
                    if (k < K && p0 < L.pitch) part[(int64_t)k * L.pitch + p0] = macc[l][kb][0] + o.x;
                    if (k < K && p0 + 4 < L.pitch) part[(int64_t)k * L.pitch + p0 + 4] = macc[l][kb][1] + o.y;
                }
            }
        }
    }
    ent = block_sum(ent, red);
    if (tid == 0) {
        double* part = a.workspace + (int64_t)blockIdx.x * len;
        part[(int64_t)K * L.pitch + BGMM_STATS_ENTROPY] = ent;
        for (int o = 1; o < 8; ++o) part[(int64_t)K * L.pitch + o] = 0.0;
    }
}

// Cross-CTA reduction of the per-CTA partial statistics, fully parallel and in a fixed order (deterministic):
// out[o] = sum_b ws[b][o].  A 256-thread CTA owns 32 outputs; its 8 warps each sum one slice of the partials (short
// dependency chains, 256-byte coalesced loads) and warp 0 adds the 8 slice sums in slice order.
// The tail of the statistics gets the local row count and format 0.  With a peer-exchange descriptor in ctrl.comm the last
// CTA to finish publishes the reduced buffer to the peers.
__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ ws, const int nparts,
                                                              const int64_t len, double* __restrict__ st, const Layout L,
                                                              const double rows, const int force, const int ignore_robust,
                                                              const int no_publish, const int crit_limit) {
    pdl_trigger();
    pdl_wait();
    volatile int* ctrl = reinterpret_cast<volatile int*>(st + L.ctrl);
    if (pass_skip(ctrl, force, ignore_robust, crit_limit)) return;
    double* __restrict__ out = st + L.stats;
    const int64_t tail = (int64_t)L.K * L.pitch;
    const CommDesc* cd = publish_target(ctrl, no_publish);
    __shared__ double slice[8][32];
    const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int64_t o = (int64_t)blockIdx.x * 32 + lane;
    const int per = (nparts + 7) / 8, b0 = sl * per, b1 = min(nparts, b0 + per);
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (o < len) {
        int b = b0;
        for (; b + 3 < b1; b += 4) {
            s0 += ws[(int64_t)(b + 0) * len + o];
            s1 += ws[(int64_t)(b + 1) * len + o];
            s2 += ws[(int64_t)(b + 2) * len + o];
            s3 += ws[(int64_t)(b + 3) * len + o];
        }
        for (; b < b1; ++b) s0 += ws[(int64_t)b * len + o];
    }
    slice[sl][lane] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (sl == 0 && o < len) {
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) acc += slice[i][lane];
        if (o == tail + BGMM_STATS_ROWS) acc = rows;
        if (o == tail + BGMM_STATS_FORMAT) acc = 0.0;     // moments about the centre (feature-map kernels)
        out[o] = acc;
    }
    if (cd != nullptr && last_cta(ctrl)) publish_stats(st, L, cd);      // one GPU: no election
}

// ---- host side ----
void launch_reduce_partials(const PassArgs& a, const Layout& L, int nparts, cudaStream_t stream) {
    const int64_t len = L.stats_len;
    launch_pdl(reduce_partials_kernel, dim3((unsigned)((len + 31) / 32)), dim3(256), 0, stream, (const double*)a.workspace,
               nparts, len, a.state, L, (double)a.n, a.force, a.ignore_robust, a.no_publish, a.crit_limit);
}

struct DmmaPlan {
    bool ok;
    int KB, SP, RP, NPS;
    size_t smem;
};

static size_t dmma_smem(int KB, int SP, int RP, int NPS, int D) {
    return sizeof(double) * ((size_t)NPS * DM_TILE * SP + (size_t)8 * KB * SP + (size_t)2 * DM_TILE * RP +
                             (size_t)DM_NXS * (DM_TILE * D + DM_XPAD) + 40) +
           sizeof(uint64_t) * (DM_NXS + 2 * NPS) + sizeof(uint2) * DM_MAXG + 128;
}

static DmmaPlan plan_dmma(int K, int D) {
    DmmaPlan p{};
    const int P = feat_count(D);
    p.SP = (P + 31) & ~31;
    p.KB = K <= 8 ? 1 : (((K + 15) & ~15) / 8);
    p.RP = 8 * p.KB < 16 ? 16 : 8 * p.KB;
    int ng = (D + 3) / 4;
    for (int i = 0; i < D; ++i) ng += i / 4 + 1;
    const size_t cap = 227 * 1024 - 512;
    p.NPS = dmma_smem(p.KB, p.SP, p.RP, 4, D) <= cap ? 4 : (dmma_smem(p.KB, p.SP, p.RP, 3, D) <= cap ? 3 : 2);
    p.smem = dmma_smem(p.KB, p.SP, p.RP, p.NPS, D);
    p.ok = ng <= DM_MAXG && ng <= 128 && (p.KB == 1 || p.KB == 2 || p.KB == 4) && p.SP <= 192 && p.smem <= cap &&
           (D * sizeof(double) * DM_TILE) % 16 == 0;
    return p;
}

bool dmma_supported(int K, int D, int dtype) { return dtype == BGMM_F64 && plan_dmma(K, D).ok; }

static int dmma_grid(int64_t n) {
    const int64_t ntiles = (n + 2 * DM_TILE - 1) / (2 * DM_TILE);   // at least two sub-tiles per CTA when possible
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)(ntiles < 1 ? 1 : (ntiles < sms ? ntiles : sms));
}

int64_t dmma_workspace_doubles(int K, int D) {
    if (!plan_dmma(K, D).ok) return 0;
    return (int64_t)160 * ((int64_t)K * feat_pitch(D) + 8);   // one partial per CTA, >= SM count of any sm_100 part
}

template <int KB, int SP, int NPS>
static int launch_cfg(const PassArgs& a, const Layout& L, const DmmaPlan& p, cudaStream_t stream) {
    auto kern = pass_dmma_kernel<KB, SP, NPS>;
    // per launch: the attribute is per device and a process may drive several devices
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 512);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(pass_dmma)");
    const int grid = dmma_grid(a.n);
    e = launch_pdl(kern, dim3(grid), dim3(DM_THREADS), p.smem, stream, a, L);
    if (e != cudaSuccess) return check_cuda(e, "pass_dmma_kernel launch");
    launch_reduce_partials(a, L, grid, stream);
    return check_cuda(cudaGetLastError(), "pass_dmma_kernel launch");
}

int launch_pass_dmma(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream) {
    const DmmaPlan p = plan_dmma(K, D);
    if (dtype != BGMM_F64 || !p.ok) {
        set_error("bgmm_pass(dmma): unsupported shape K=%d D=%d dtype=%d", K, D, dtype);
        return BGMM_ENOSUP;
    }
    if ((reinterpret_cast<uintptr_t>(a.x) & 15) != 0) {
        set_error("bgmm_pass(dmma): x must be 16-byte aligned");
        return BGMM_EINVAL;
    }
    const Layout L = make_layout(K, D, 1);
#define BGMM_DM_CASE(kb, sp, nps) if (p.KB == kb && p.SP == sp && p.NPS == nps) return launch_cfg<kb, sp, nps>(a, L, p, stream);
#define BGMM_DM_ROW(kb) BGMM_DM_CASE(kb, 32, 4) BGMM_DM_CASE(kb, 64, 4) BGMM_DM_CASE(kb, 96, 4) BGMM_DM_CASE(kb, 128, 4) \
                        BGMM_DM_CASE(kb, 160, 4) BGMM_DM_CASE(kb, 192, 4) BGMM_DM_CASE(kb, 192, 3) BGMM_DM_CASE(kb, 160, 3)
    BGMM_DM_ROW(1) BGMM_DM_ROW(2) BGMM_DM_ROW(4)
#undef BGMM_DM_ROW
#undef BGMM_DM_CASE
    set_error("bgmm_pass(dmma): no instantiation for KB=%d SP=%d NPS=%d", p.KB, p.SP, p.NPS);
    return BGMM_ENOSUP;
}

}  // namespace bgmm
