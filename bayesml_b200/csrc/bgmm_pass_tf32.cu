// bgmm_pass, fp32-mode tensor-core variant (BGMM_PASS_TF32) for sm_100a: tcgen05.mma kind::tf32 with 3xTF32 operands,
// fp32 accumulators in tensor memory, read back with tcgen05.ld.  X is float32 ("fp32 mode", BASELINE.json north_star (1)).
//
// Which formulation (profiles/r02_fp32_precision_study.json, tools/fp32_precision_study.py): in fp32 the feature-map E-step
// loses eps32 * crit (2e-4 in ln rho at C2's geometry with a 3xTF32 split), the WHITENED form does not:
//     y_nk = sqrt(nu_k) Linv_k (x_n - m_k)      ln rho_nk = a_k - |y_nk|^2 / 2          (7e-6 at C2 in fp32)
// and it is one GEMM:  Y[n][(k, j)] = [x_n, 1] . B,  B[(k, j)][i] = s_k Linv_k[j][i],  B[(k, j)][D] = -s_k (Linv_k m_k)[j],
// s_k = sqrt(nu_k log2(e) / 2)  (so ln rho in base 2 is a2_k - |y|^2), with the row norms, the softmax over k, the entropy
// term and r in the epilogue of the thread that owns the row (a TMEM lane is a sample: no shuffles at all).
//
//   tf32_prep_kernel    per iteration: B (hi / lo parts, already in the shared-memory operand layout) and a2 from the
//                       parameter set (Linv comes from bgmm_small: BGMM_P_LINV);
//   pass_tf32_e_kernel  persistent, one CTA (544 threads) per SM, 128-sample tiles: 16 epilogue / staging warps split the
//                       [x, 1] tile into tf32 hi + lo and stage it K-major in shared memory (two stages, x prefetched one
//                       tile ahead); a 17th warp issues, per 256-column chunk of (component, dimension) pairs, the three
//                       products hi.hi + hi.lo + lo.hi into one of two TMEM buffers and commits to an mbarrier; the four
//                       warps of a TMEM lane quarter split the chunk's columns (tcgen05.ld, lane = sample), accumulate |y|^2
//                       per component and combine max / sum / entropy through shared memory; the next chunk's MMAs run
//                       meanwhile; r (float32, [n][KP]) goes to HBM for the statistics kernel — 4 KP bytes per sample.
//   pass_tf32_m_kernel  persistent, 544 threads: raw = R^T . Phi with R^T in TENSOR MEMORY (staging warps), Phi generated
//                       into 128-byte-swizzled shared-memory stages (generator warps), one issuing warp; see its header.
// E-kernel operands are staged K-major in the no-swizzle canonical layout, Phi in the SWIZZLE_128B layout (bgmm_tc.cuh; both
// verified on the B200 by tests/test_gpu_tc.py).  Replaces `_update_q_z` :772-783 and `_calc_n_x_bar_s` :725-732 of the
// reference GMM file in fp32 mode; bar 1e-4.
#include "bgmm_common.cuh"
#include "bgmm_mma.cuh"
#include "bgmm_tc.cuh"
#include <math.h>

namespace bgmm {

constexpr int TF_TILE = 128;                 // samples per tile = TMEM lanes = threads
constexpr int TF_NMAX = 256;                 // columns of one MMA / one TMEM buffer

struct Tf32Plan {
    bool ok;
    int D, K, DP, KD, KP, cpc, nchunks, nmma;    // padded dims; components per chunk; chunk count; MMA N
    size_t smem_e;
};

static Tf32Plan plan_tf32(int K, int D) {
    Tf32Plan p{};
    p.D = D; p.K = K;
    p.DP = D <= 4 ? 4 : (D <= 8 ? 8 : (D <= 16 ? 16 : 32));
    p.KD = (D + 1 + 7) & ~7;
    p.KP = (K + 3) & ~3;
    p.cpc = (TF_NMAX / p.DP) & ~3;
    if (p.cpc > p.KP) p.cpc = p.KP;
    p.nchunks = (p.KP + p.cpc - 1) / p.cpc;
    p.nmma = p.cpc * p.DP;
    // B (hi, lo) for every chunk + two stages of A (hi, lo) + a2 + barriers
    p.smem_e = sizeof(float) * ((size_t)2 * p.nchunks * p.nmma * p.KD + (size_t)2 * 2 * TF_TILE * p.KD + 64 + 12 * TF_TILE + TF_TILE * 68) + 256;
    p.ok = D >= 1 && D <= 31 && K >= 1 && K <= 64 && p.KD <= 32 && p.smem_e <= 220 * 1024 && (p.nmma % 16) == 0;
    return p;
}

bool tf32_supported(int K, int D, int dtype) { return dtype == BGMM_F32 && plan_tf32(K, D).ok; }

// floats of global scratch: the operand image of B (hi, lo) + a2
int64_t tf32_image_floats(int K, int D) {
    const Tf32Plan p = plan_tf32(K, D);
    return p.ok ? (int64_t)2 * p.nchunks * p.nmma * p.KD + 64 : 0;
}

// ---- per iteration: the whitening operand, split and laid out as the E kernel's shared-memory image ----
// image = [part (hi, lo)][chunk][K-major tile: nmma rows x KD cols, LBO = 128 B, SBO = (KD / 4) * 128 B] then a2[64]
__global__ void __launch_bounds__(256) tf32_prep_kernel(const double* __restrict__ st, const Layout L, float* __restrict__ img,
                                                        const int DP, const int KD, const int KP, const int cpc,
                                                        const int nchunks, const int nmma, const int force,
                                                        const int crit_limit) {
    pdl_trigger();
    pdl_wait();
    const volatile int* ctrl = reinterpret_cast<const volatile int*>(st + L.ctrl);
    if (pass_skip(ctrl, force, 0, crit_limit)) return;
    const int K = L.K, D = L.D;
    const double* Pc = st + L.params[ctrl[BGMM_CTRL_CUR]];
    const int64_t part = (int64_t)nchunks * nmma * KD;
    const int lbo_f = 32, sbo_f = (KD / 4) * 32;
    const int total = nchunks * nmma * KD;
    for (int e = blockIdx.x * 256 + threadIdx.x; e < total; e += gridDim.x * 256) {
        const int ch = e / (nmma * KD), rem = e - ch * nmma * KD;
        const int n = rem / KD, i = rem - n * KD;                // row n = (local component, dimension j), column i
        const int c = ch * cpc + n / DP, j = n % DP;
        double v = 0.0;
        if (c < K && j < D) {
            const double s = sqrt(Pc[L.p_nu + c] * (0.5 * 1.4426950408889634074));
            const double* Li = Pc + L.p_linv + (int64_t)c * D * D + (int64_t)j * D;      // row j of Linv_c
            if (i < D) v = s * Li[i];
            else if (i == D) {
                const double* m = Pc + L.p_m + (int64_t)c * D;
                double acc = 0.0;
                for (int l = 0; l <= j; ++l) acc += Li[l] * m[l];
                v = -s * acc;
            }
        }
        const float hi = tc::tf32_hi((float)v);
        const float lo = (float)(v - (double)hi);
        const int64_t o = (int64_t)ch * nmma * KD + tc::kmajor_off(n, i, lbo_f, sbo_f);
        img[o] = hi;
        img[part + o] = lo;
    }
    if (blockIdx.x == 0 && threadIdx.x < 64) {
        const int c = threadIdx.x;
        img[2 * part + c] = c < K ? (float)(Pc[L.p_acst + c] * 1.4426950408889634074) : -1.0e30f;
    }
}

__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2f(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// r_f32 [n][KP] float32: the hand-over to the statistics kernel.  Optional float64 outputs as in the other variants.
// 512 threads = 4 groups of 4 warps.  A TMEM lane (= sample row) is readable by the warps w with w % 4 == lane / 32, so the
// four groups share every row and split its COLUMNS: group q reads the q-th 64-column batch of every chunk.  One warp per
// scheduler (the first version, 128 threads) left the epilogue latency bound at ~11 cycles per instruction — 4.1 ms at C2
// against 0.6 ms of tensor-core time; four warps per scheduler hide it.  The softmax over k then spans four threads:
// max, sum and the entropy dot product are combined through shared memory ([4][128] floats, two block barriers).
constexpr int TE_THREADS = 512;               // epilogue / staging threads
constexpr int TE_BLOCK = TE_THREADS + 32;    // + one warp whose elected lane issues the MMAs (no block barrier in the tile loop)

// OUT = false: the loop instantiation (no float64 ln rho / r / arg-max outputs: their predicated-off stores and conversions
// were 11 % of the issue slots of the first version).
template <int DP, int KD, bool OUT>
__global__ void __launch_bounds__(TE_BLOCK, 1)
pass_tf32_e_kernel(const PassArgs a, const Layout L, const float* __restrict__ img, float* __restrict__ r_f32,
                   double* __restrict__ ews, const int KP, const int cpc, const int nchunks, const int nmma, const int dbg) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    pdl_trigger();
    pdl_wait();
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust, a.crit_limit)) return;
    const int K = L.K, D = L.D, tid = threadIdx.x, warp = tid >> 5;
    const int rowt = tid & 127, gq = tid >> 7;                  // sample row of the tile; column group
    const float* __restrict__ x = static_cast<const float*>(a.x);
    constexpr int KCH = KD / 4, KGR = KD / 8;
    constexpr int A_LBO = 32, A_SBO = KCH * 32;                 // floats: k-chunks adjacent, then the next 8-row group
    constexpr int CPCMAX = TF_NMAX / DP, NCHMAX = DP / 4;       // CPCMAX * NCHMAX = 64 components at most
    constexpr int CPB = 64 / DP > 0 ? 64 / DP : 1;              // components per 64-column batch
    constexpr int NL = NCHMAX * CPB;                            // components this thread can own (<= 16)
    const int64_t bpart = (int64_t)nchunks * nmma * KD;
    float* Bs = reinterpret_cast<float*>(smem_raw);            // [2 parts][nchunks][nmma x KD]
    float* As = Bs + 2 * bpart;                                // [2 stages][2 parts][128 x KD]
    float* a2s = As + 2 * 2 * TF_TILE * KD;                    // [64]
    float* xch = a2s + 64;                                     // [3][4][128]: max, sum, dot of every column group
    float* rst = xch + 3 * 4 * TF_TILE;                        // [128][KP + 4]: r tile staged for coalesced row stores
    const int RSP = KP + 4;                                    // pitch: 16-byte aligned, rows 4 banks apart
    uint64_t* mbar = reinterpret_cast<uint64_t*>(rst + TF_TILE * (64 + 4));  // [2] MMAs of TMEM buffer b complete
    uint64_t* tfree = mbar + 2;                                // [2] TMEM buffer b drained by all 16 epilogue warps
    uint64_t* astaged = mbar + 4;                              // [2] A stage s written (one arrival per staging warp)
    uint32_t* tslot = reinterpret_cast<uint32_t*>(mbar + 6);
    __shared__ double red[40];

    for (int64_t e = tid; e < 2 * bpart; e += TE_BLOCK) Bs[e] = img[e];
    for (int e = tid; e < 64; e += TE_BLOCK) a2s[e] = img[2 * bpart + e];
    if (tid == 0) {
        mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1);
        mbar_init(&tfree[0], TE_THREADS / 32); mbar_init(&tfree[1], TE_THREADS / 32);
        mbar_init(&astaged[0], TE_THREADS / 32); mbar_init(&astaged[1], TE_THREADS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (warp == 0) tc::tmem_alloc<512>(tslot);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tbase = *tslot;
    const uint32_t idesc = tc::make_idesc_tf32(128, nmma, 0, 0);
    // the last chunk may hold fewer components: its MMAs cover only their columns (C2: 8 of 16 -> N = 128, a quarter less
    // tensor-core time per tile)
    const int n_last = (((KP - (nchunks - 1) * cpc) * DP) + 15) & ~15;
    const uint32_t idesc_last = tc::make_idesc_tf32(128, n_last < nmma ? n_last : nmma, 0, 0);
    const uint32_t b_lbo = 4 * 32, b_sbo = 4 * KCH * 32, a_lbo = 4 * A_LBO, a_sbo = 4 * A_SBO;    // bytes

    const int64_t ntiles = (a.n + TF_TILE - 1) / TF_TILE;
    const int64_t my_tiles = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t total_g = my_tiles * nchunks;                 // chunks of this CTA, in issue order

    // this thread's part of a tile's [x, 1] rows: k-chunks kc = gq, gq + 4, ..  The global loads are issued ONE TILE AHEAD of
    // the staging (fetch_tile(lt + 1) right after stage_tile(lt)): their latency was 17 % of the kernel as a long-scoreboard stall
    constexpr int NKC = (KCH + 3) / 4;
    float xpre[NKC][4];
    auto fetch_tile = [&](int64_t lt) {
        const int64_t row = (blockIdx.x + lt * gridDim.x) * TF_TILE + rowt;
        const bool valid = lt < my_tiles && row < a.n;
#pragma unroll
        for (int u = 0; u < NKC; ++u) {
            const int kc = 4 * u + gq;
            if (valid && (D & 3) == 0 && 4 * kc + 3 < D) {         // a whole 16-byte chunk of the row: one load
                const float4 f = __ldg(reinterpret_cast<const float4*>(x + row * D) + kc);
                xpre[u][0] = f.x; xpre[u][1] = f.y; xpre[u][2] = f.z; xpre[u][3] = f.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = 4 * kc + q;
                    xpre[u][q] = (valid && i < D) ? __ldg(x + row * D + i) : ((valid && i == D) ? 1.0f : 0.0f);
                }
            }
        }
    };
    auto stage_tile = [&](int64_t lt) {                         // local tile lt -> A stage lt & 1, from the prefetched registers
        float* Ah = As + (size_t)(lt & 1) * 2 * TF_TILE * KD;
        float* Al = Ah + TF_TILE * KD;
#pragma unroll
        for (int u = 0; u < NKC; ++u) {
            const int kc = 4 * u + gq;
            if (kc < KCH) {
                float h[4], l[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    h[q] = tc::tf32_hi(xpre[u][q]);
                    l[q] = xpre[u][q] - h[q];
                }
                const int o = tc::kmajor_off(rowt, 4 * kc, A_LBO, A_SBO);
                *reinterpret_cast<float4*>(Ah + o) = make_float4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<float4*>(Al + o) = make_float4(l[0], l[1], l[2], l[3]);
            }
        }
    };
    // descriptor low words (address | LBO) of A stage 0 / B chunk 0 per part and k-step; stage, chunk are address offsets
    uint32_t alo[2][KGR], blo[2][KGR];
#pragma unroll
    for (int pt = 0; pt < 2; ++pt)
#pragma unroll
        for (int ks = 0; ks < KGR; ++ks) {
            const uint32_t aaddr = tc::smem_u32(As + (size_t)pt * TF_TILE * KD) + 2 * ks * a_lbo;
            const uint32_t baddr = tc::smem_u32(Bs) + (pt ? 4 * (uint32_t)bpart : 0u) + 2 * ks * b_lbo;
            alo[pt][ks] = ((aaddr >> 4) & 0x3FFFu) | (((a_lbo >> 4) & 0x3FFFu) << 16);
            blo[pt][ks] = ((baddr >> 4) & 0x3FFFu) | (((b_lbo >> 4) & 0x3FFFu) << 16);
        }
    const uint32_t ahi = ((a_sbo >> 4) & 0x3FFFu) | (1u << 14), bhi = ((b_sbo >> 4) & 0x3FFFu) | (1u << 14);
    const uint32_t a_stage_step = (uint32_t)(2 * TF_TILE * KD * 4) >> 4, b_chunk_step = (uint32_t)(nmma * KD * 4) >> 4;
    auto issue_chunk = [&](int64_t g) {                          // thread 0 only
        tc::fence_after_sync();
        const int64_t lt = g / nchunks;
        const int ch = (int)(g - lt * nchunks);
        const uint32_t d_tmem = tbase + (uint32_t)(g & 1) * TF_NMAX;
        const uint32_t aoff = (lt & 1) ? a_stage_step : 0u, boff = (uint32_t)ch * b_chunk_step;
        const uint32_t id = ch == nchunks - 1 ? idesc_last : idesc;
        uint32_t accum = 0;
#pragma unroll
        for (int s = 0; s < 3; ++s) {                            // hi.hi, hi.lo, lo.hi
            if (dbg == 2 && s > 0) continue;                     // never taken: dbg is 0 (see launch_e_t)
#pragma unroll
            for (int ks = 0; ks < KGR; ++ks) {
                tc::mma_tf32_w(d_tmem, alo[s == 2 ? 1 : 0][ks] + aoff, ahi, blo[s == 1 ? 1 : 0][ks] + boff, bhi, id, accum);
                accum = 1;
            }
        }
        tc::mma_commit(&mbar[g & 1]);
    };

    float ent = 0.f;
    if (warp == TE_THREADS / 32) {
        // =========================== MMA WARP ===========================
        // chunk g (tile g / nchunks) goes to TMEM buffer g & 1 as soon as that buffer has been drained (tfree) and the tile's
        // A stage is written (astaged); the whole warp walks the loop, one elected lane issues
        for (int64_t g = 0; g < total_g; ++g) {
            const int64_t lt = g / nchunks;
            if (g - lt * nchunks == 0) mbar_wait(&astaged[lt & 1], (uint32_t)((lt >> 1) & 1));
            if (g >= 2) mbar_wait(&tfree[g & 1], (uint32_t)(((g >> 1) - 1) & 1));
            if ((tid & 31) == 0) issue_chunk(g);
            __syncwarp();
        }
    } else {
        // =========================== EPILOGUE / STAGING WARPS ===========================
        const int qbar = 1 + (warp & 3);                         // named barrier of the four warps that share this row quarter
        const int st_t128 = (tid & 31) + 32 * gq, st_q4 = KP / 4;
        const int st_rr0 = st_t128 / st_q4, st_c40 = st_t128 - st_rr0 * st_q4, st_drr = 128 / st_q4, st_dc4 = 128 - st_drr * st_q4;
        if (my_tiles > 0) {
            fetch_tile(0);
            stage_tile(0);
            fetch_tile(1);
            tc::fence_proxy_async();
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&astaged[0]);
        }
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
            // stage the next tile now: its MMAs can start as soon as a TMEM buffer frees up.  (Its stage was last read by tile
            // lt - 1, whose chunks this thread has already seen complete.)
            if (lt + 1 < my_tiles) {
                stage_tile(lt + 1);
                fetch_tile(lt + 2);
                tc::fence_proxy_async();
                __syncwarp();
                if ((tid & 31) == 0) mbar_arrive(&astaged[(lt + 1) & 1]);
            }
            const int64_t row = (blockIdx.x + lt * gridDim.x) * TF_TILE + rowt;
            const bool valid = row < a.n;
            // this thread's components: chunk ch, batch gq, u = 0 .. CPB-1 -> component ch * cpc + gq * CPB + u (local slot ch * CPB + u)
            float l2[NL];
#pragma unroll
            for (int c = 0; c < NL; ++c) l2[c] = -1.0e30f;
#pragma unroll
            for (int ch = 0; ch < NCHMAX; ++ch) {
                if (ch < nchunks) {                              // uniform
                    const int64_t g = lt * nchunks + ch;
                    mbar_wait(&mbar[g & 1], (uint32_t)((g >> 1) & 1));
                    tc::fence_after_sync();
                    const uint32_t t0 = tbase + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)(g & 1) * TF_NMAX + 64 * gq;
                    if (gq * CPB < cpc && ch * cpc + gq * CPB < KP && dbg != 1) {   // uniform per warp: this 64-column batch holds components
                        if constexpr (DP == 16) {
                            // two 32-column halves: 32 live accumulator registers instead of 64 (the 120-register cap of a
                            // 544-thread CTA made the one-batch form spill)
#pragma unroll
                            for (int hb = 0; hb < 2; ++hb) {
                                uint32_t v[2][16];
                                tc::tmem_ld16_async(t0 + 32 * hb, v[0]);
                                tc::tmem_ld16_async(t0 + 32 * hb + 16, v[1]);
                                tc::tmem_wait_ld();
#pragma unroll
                                for (int u = 0; u < 2; ++u) {
                                    float q0 = 0.f, q1 = 0.f;
#pragma unroll
                                    for (int j = 0; j < 16; j += 2) {
                                        const float y0 = __uint_as_float(v[u][j]), y1 = __uint_as_float(v[u][j + 1]);
                                        q0 = fmaf(y0, y0, q0);
                                        q1 = fmaf(y1, y1, q1);
                                    }
                                    l2[ch * CPB + 2 * hb + u] = a2s[ch * cpc + gq * CPB + 2 * hb + u] - (q0 + q1);
                                }
                            }
                        } else if constexpr (DP >= 16) {
                            uint32_t v[4][16];
#pragma unroll
                            for (int h = 0; h < 4; ++h) tc::tmem_ld16_async(t0 + 16 * h, v[h]);
                            tc::tmem_wait_ld();
#pragma unroll
                            for (int u = 0; u < CPB; ++u) {
                                float q0 = 0.f, q1 = 0.f;
#pragma unroll
                                for (int h = 0; h < DP / 16; ++h)
#pragma unroll
                                    for (int j = 0; j < 16; j += 2) {
                                        const float y0 = __uint_as_float(v[u * (DP / 16) + h][j]);
                                        const float y1 = __uint_as_float(v[u * (DP / 16) + h][j + 1]);
                                        q0 = fmaf(y0, y0, q0);
                                        q1 = fmaf(y1, y1, q1);
                                    }
                                l2[ch * CPB + u] = a2s[ch * cpc + gq * CPB + u] - (q0 + q1);
                            }
                        } else {
                            uint32_t v[4][16];
#pragma unroll
                            for (int h = 0; h < 4; ++h) tc::tmem_ld16_async(t0 + 16 * h, v[h]);
                            tc::tmem_wait_ld();
                            constexpr int PER = 16 / DP;         // components per 16-column load
#pragma unroll
                            for (int h = 0; h < 4; ++h)
#pragma unroll
                                for (int u = 0; u < PER; ++u) {
                                    float q = 0.f;
#pragma unroll
                                    for (int j = 0; j < DP; ++j) {
                                        const float y = __uint_as_float(v[h][u * DP + j]);
                                        q = fmaf(y, y, q);
                                    }
                                    l2[ch * CPB + h * PER + u] = a2s[ch * cpc + gq * CPB + h * PER + u] - q;
                                }
                        }
                    }
                    tc::fence_before_sync();
                    __syncwarp();
                    if ((tid & 31) == 0) mbar_arrive(&tfree[g & 1]);      // this warp has drained TMEM buffer g & 1
                }
            }
            // ---- softmax over k: four threads per row (one per column group), combined through shared memory; only the
            //      four warps that share the row quarter synchronise (named barrier, 128 threads) ----
            float mx = -3.0e38f;
            // slots of chunks this launch does not have (ch >= nchunks, uniform) are skipped, not carried as -1e30 padding: at
            // C2 that is half of the exponentials
#pragma unroll
            for (int ch = 0; ch < NCHMAX; ++ch)
                if (ch < nchunks) {
#pragma unroll
                    for (int u = 0; u < CPB; ++u) mx = fmaxf(mx, l2[ch * CPB + u]);
                }
            xch[gq * TF_TILE + rowt] = mx;
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            mx = fmaxf(fmaxf(xch[rowt], xch[TF_TILE + rowt]), fmaxf(xch[2 * TF_TILE + rowt], xch[3 * TF_TILE + rowt]));
            float s = 0.f, dot = 0.f;
#pragma unroll
            for (int c = 0; c < NL; ++c) {
                if ((c / CPB) >= nchunks) { l2[c] = 0.f; continue; }   // uniform
                const float z = l2[c] - mx;
                const float e = ex2f(z);                         // padded slots: z ~ -1e30 -> 0
                if (OUT && a.lnrho_out != nullptr && valid) {
                    const int comp = (c / CPB) * cpc + gq * CPB + (c % CPB);
                    if (gq * CPB < cpc && comp < K) a.lnrho_out[row * K + comp] = (double)l2[c] * 0.693147180559945309417232121458;
                }
                l2[c] = e;
                s += e;
                dot = fmaf(e, fmaxf(z, -1.0e4f), dot);           // e == 0 there: keep 0 * z finite
            }
            xch[(4 + gq) * TF_TILE + rowt] = s;
            xch[(8 + gq) * TF_TILE + rowt] = dot;
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            s = (xch[4 * TF_TILE + rowt] + xch[5 * TF_TILE + rowt]) + (xch[6 * TF_TILE + rowt] + xch[7 * TF_TILE + rowt]);
            dot = (xch[8 * TF_TILE + rowt] + xch[9 * TF_TILE + rowt]) + (xch[10 * TF_TILE + rowt] + xch[11 * TF_TILE + rowt]);
            const float inv = valid ? 1.0f / s : 0.f;
            if (valid && gq == 0) ent += 0.693147180559945309f * (dot * inv - lg2f(s));
            // r: this thread's CPB consecutive components of every chunk, staged for coalesced row stores
#pragma unroll
            for (int ch = 0; ch < NCHMAX; ++ch) {
                if (ch < nchunks && gq * CPB < cpc) {
                    const int c0 = ch * cpc + gq * CPB;
#pragma unroll
                    for (int u = 0; u < CPB; ++u) {
                        const float rv = l2[ch * CPB + u] * inv;
                        if (CPB != 4 && c0 + u < KP) rst[rowt * RSP + c0 + u] = rv;
                        if (OUT && a.r_out != nullptr && valid && c0 + u < K) a.r_out[row * K + c0 + u] = (double)rv;
                        l2[ch * CPB + u] = rv;
                    }
                    if (CPB == 4 && c0 < KP)                     // KP, c0 and the pitch are multiples of 4: one 16-byte store
                        *reinterpret_cast<float4*>(rst + rowt * RSP + c0) =
                            make_float4(l2[ch * CPB], l2[ch * CPB + 1], l2[ch * CPB + 2], l2[ch * CPB + 3]);
                }
            }
            if (OUT && a.argmax_out != nullptr) {                // final pass only: arg max over the four column groups
                int best = 0x7fffffff;
                float bestv = -1.f;
#pragma unroll
                for (int c = 0; c < NL; ++c) {
                    const int comp = (c / CPB) * cpc + gq * CPB + (c % CPB);
                    if ((c / CPB) < nchunks && gq * CPB < cpc && comp < K && (l2[c] > bestv || (l2[c] == bestv && comp < best))) {
                        bestv = l2[c]; best = comp;
                    }
                }
                xch[gq * TF_TILE + rowt] = bestv;
                xch[(4 + gq) * TF_TILE + rowt] = __int_as_float(best);
            }
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");
            {   // this quarter's 32 rows of r are contiguous in r_f32 (32 x KP floats): 16-byte stores by its 128 threads
                const int qtr = warp & 3, t128 = (tid & 31) + 32 * gq;
                const int64_t row0 = (blockIdx.x + lt * gridDim.x) * TF_TILE + 32 * qtr;
                const int rows_here = (int)max((int64_t)0, min((int64_t)32, a.n - row0));
                const int q4 = KP / 4;
                int rr = st_rr0, c4 = st_c40;                    // (t128 / q4, t128 % q4), advanced by (128 / q4, 128 % q4)
                for (int e = t128; e < rows_here * q4; e += 128) {
                    *reinterpret_cast<float4*>(r_f32 + (row0 + rr) * KP + 4 * c4) =
                        *reinterpret_cast<const float4*>(rst + (32 * qtr + rr) * RSP + 4 * c4);
                    rr += st_drr; c4 += st_dc4;
                    if (c4 >= q4) { c4 -= q4; ++rr; }
                }
            }
            if (OUT && a.argmax_out != nullptr && gq == 0 && valid) {
                int best = __float_as_int(xch[4 * TF_TILE + rowt]);
                float bestv = xch[rowt];
                for (int o = 1; o < 4; ++o) {
                    const float ov = xch[o * TF_TILE + rowt];
                    const int ok = __float_as_int(xch[(4 + o) * TF_TILE + rowt]);
                    if (ov > bestv || (ov == bestv && ok < best)) { bestv = ov; best = ok; }
                }
                a.argmax_out[row] = best;
            }
            asm volatile("bar.sync %0, 128;" ::"r"(qbar) : "memory");      // xch / rst rows of this quarter are reused by the next tile
        }
    }
    const double e_cta = block_sum((double)ent, red);
    if (tid == 0) ews[blockIdx.x] = e_cta;
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tbase);
}

// ---- statistics: raw[k][p] = sum_n r_nk phi_p(x'_n) as  D[component][feature] = R^T . Phi  on the tensor cores -------
// Contraction over SAMPLES: a 64-sample sub-tile is 8 MMA k-steps.  What bounds this GEMM is the tensor core's operand
// bandwidth from shared memory (~64 B/clk measured: the first version, both operands in shared memory with the features on
// M, spent 68 % of its time waiting for 48 small MMAs per sub-tile).  So:
//   A = R^T lives in TENSOR MEMORY (lane = component, column = sample; written by the warp whose lanes are the components:
//       lane c reads r[row][c], a coalesced 128-byte row per sample, and stores 8 samples per tcgen05.st) — no shared-memory
//       traffic for A; rows K .. 127 of the M = 128 tile are zero;
//   B = Phi (N = features, all of them in one MMA: P <= 256) is staged K-major in the 128-byte-swizzle layout (a feature
//       row holds 32 samples; bgmm_tc.cuh), i.e. TRANSPOSED with respect to the thread that produces it: generator warp g
//       owns the features p = g (mod 8) — one row of every 8-row swizzle atom — and a lane two consecutive samples:
//       conflict-free 8-byte stores; two stages, so the generation of sub-tile t + 1 overlaps the MMAs of sub-tile t;
//       the x rows arrive by cp.async two sub-tiles ahead (five buffers, one mbarrier each).
//   K <= 32: the hi parts of R^T sit in TMEM lanes 0-31, the lo parts in lanes 64-95 of the same columns: two MMAs per
//       k-step (against Phi_hi and Phi_lo) give all four split products.
// Every value is split into tf32 hi (truncated: one LOP3) + the exact remainder lo; the split products accumulate in fp32 in tensor
// memory over TF_FLUSH sub-tiles and are then added into a float64 CTA-private array (feature-major, so a warp's lanes =
// components are contiguous), so the fp32 error of a partial sum never exceeds that of 2048 samples.  Moments are about
// the global centre (format 0), reduced over the CTAs by reduce_partials_kernel.
constexpr int TM_SUB = 64;                   // samples per sub-tile
constexpr int TF_FLUSH = 32;                 // sub-tiles between TMEM -> fp64 flushes (2048 samples)
constexpr int TM_GEN = 256;                  // generator threads: four per sample
constexpr int TM_STG = 256;                  // staging threads: warps w with (w & 3) = 0 own TMEM lanes 0-31 (components 0-31),
                                             // (w & 3) = 1 lanes 32-63; four warps per lane quarter, 16 samples each — ONE warp
                                             // splitting all 64 samples of its component into hi / lo was the critical path
constexpr int TM_BLOCK = TM_GEN + TM_STG + 32;   // warps 0-15 with (w & 3) >= 2 generate Phi; warp 16 only issues the MMAs

// Phi rows of ONE sample into the hi / lo staging tiles, features with (p & 3) == Q only; D is a compile-time constant so
// every product index and every shared-memory offset is static (5 instructions per feature: mul, cvt, sub, 2 stores)
// A generator warp owns the features p = FG (mod 8) — one row of every swizzled 8-row atom, so the XOR of the chunk index is
// a per-thread constant — and a lane two consecutive samples: 8-byte stores, 4 instructions per (sample, feature).
// o0 = float offset of (row FG of atom row-group 0, this lane's sample pair).
// explicit shared-space accesses: the staging pointers come out of a 1024-byte round-up of the dynamic shared memory base,
// through which the compiler loses the address space and emits generic LD / ST (4.5 % of the executed instructions)
__device__ __forceinline__ void sts64(uint32_t addr, float a, float b) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void sts32(uint32_t addr, float a) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(a) : "memory"); }
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// Bh / Bl: 32-bit shared addresses of the hi / lo staging tiles
template <int DT, int FG>
__device__ __forceinline__ void gen_features(const float (&xa)[DT > 0 ? DT : 1], const float (&xb)[DT > 0 ? DT : 1],
                                             const uint32_t Bh, const uint32_t Bl, const int o0) {
    auto put = [&](int p, float va, float vb) {
        const float ha = tc::tf32_trunc(va), hb = tc::tf32_trunc(vb);
        const uint32_t o = 4u * (uint32_t)((p >> 3) * 256 + o0);
        sts64(Bh + o, ha, hb);
        sts64(Bl + o, va - ha, vb - hb);
    };
    if (FG == 0) put(0, 1.0f, 1.0f);
#pragma unroll
    for (int i = 0; i < DT; ++i)
        if (((1 + i) & 7) == FG) put(1 + i, xa[i], xb[i]);
#pragma unroll
    for (int i = 0; i < DT; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j)
            if (((1 + DT + i * (i + 1) / 2 + j) & 7) == FG) put(1 + DT + i * (i + 1) / 2 + j, xa[i] * xa[j], xb[i] * xb[j]);
}

// DT = compile-time D (0: run-time D through a table); NF = features rounded up to 16 (the MMA N), passed at run time
template <int DT>
__global__ void __launch_bounds__(TM_BLOCK, 1)
pass_tf32_m_kernel(const PassArgs a, const Layout L, const float* __restrict__ r_f32, const int KP, const int NF, const int nst,
                   double* __restrict__ acct, const double* __restrict__ ews, const int n_ews) {
    extern __shared__ __align__(128) unsigned char smem_raw_m[];
    pdl_trigger();
    pdl_wait();
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (pass_skip(ctrl, a.force, a.ignore_robust, a.crit_limit)) return;
    const int K = L.K, D = DT > 0 ? DT : L.D, P = L.P, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const float* __restrict__ x = static_cast<const float*>(a.x);
    const int bpart = NF * TM_SUB;                             // floats of one part (hi or lo) of one stage
    // [nst stages][2 parts][2 k-atoms of 32 samples][NF / 8 row groups][8 features][128 bytes, chunks swizzled]
    float* Bs = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(smem_raw_m) + 1023) & ~uintptr_t(1023));
    float* xs = Bs + 2 * nst * bpart;                                // [64][D + 2]: x', 1, 0   (run-time D only)
    // compile-time D: xs = XNB buffers of 32 row PAIRS, pitch 2 D + 4 floats (16-byte aligned, conflict-free for LDS.128).
    // Five buffers, filled two sub-tiles ahead: a generator warp can be up to two iterations behind the fastest one (each
    // waits for the MMAs of sub-tile t - 2 only), so the tiles t - 2 .. t + 2 must be distinct buffers — then no block
    // barrier is needed around the tile (the 256-thread barrier of the two-buffer form cost ~500 cycles of skew per sub-tile).
    constexpr int XPP = DT > 0 ? 2 * DT + 4 : 0;
    constexpr int XNB = 5;
    unsigned short* ftab = reinterpret_cast<unsigned short*>(xs + (DT > 0 ? XNB * 32 * XPP : TM_SUB * (D + 2)));   // [P] (run-time D only)
    uint64_t* mbar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(ftab + (DT > 0 ? 0 : ((P + 7) & ~7))) + 15) & ~uintptr_t(15));
    uint64_t* mdone = mbar;                                    // [2] MMAs of sub-tile parity b complete (B stage + A buffer free)
    uint64_t* bfull = mbar + 2;                                // [2] B stage b written (one arrival per generator warp: 256
                                                               //     per-thread arrivals on one mbarrier cost ~1000 cycles a sub-tile)
    uint64_t* afull = mbar + 4;                                // [2] A buffer b written (one arrival per staging warp)
    uint64_t* xfull = mbar + 6;                                // [5] x tile buffer filled (cp.async arrivals of the 256 generator threads)
    uint32_t* tslot = reinterpret_cast<uint32_t*>(mbar + 11);
    const int KW = (KP + 31) / 32;                             // component warps with real rows (1 or 2)
    double* acc = acct + (int64_t)blockIdx.x * 256 * 64;      // CTA-private [NF][64] float64, feature-major

    if (DT == 0) {
        // feature table: phi_p = xs[.][i] * xs[.][j] with the constant columns xs[.][D] = 1, xs[.][D + 1] = 0
        for (int p = tid; p < P; p += TM_BLOCK) {
            int i, j;
            if (p == 0) { i = D; j = D; }
            else if (p <= D) { i = p - 1; j = D; }
            else {
                const int q = p - 1 - D;
                int r = (int)((sqrtf(8.0f * q + 1.0f) - 1.0f) * 0.5f);
                while (r * (r + 1) / 2 > q) --r;
                while ((r + 1) * (r + 2) / 2 <= q) ++r;
                i = r; j = q - r * (r + 1) / 2;
            }
            ftab[p] = (unsigned short)((i << 8) | j);
        }
    }
    for (int e = tid; e < 2 * nst * bpart; e += TM_BLOCK) Bs[e] = 0.f;    // feature rows P .. NF-1 are never written
    for (int e = tid; e < NF * 64; e += TM_BLOCK) acc[e] = 0.0;
    if (tid == 0) {
        mbar_init(&mdone[0], 1); mbar_init(&mdone[1], 1);
        mbar_init(&bfull[0], TM_GEN / 32); mbar_init(&bfull[1], TM_GEN / 32);
        mbar_init(&afull[0], TM_STG / 32); mbar_init(&afull[1], TM_STG / 32);
        for (int i = 0; i < 5; ++i) mbar_init(&xfull[i], TM_GEN);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (warp == 0) tc::tmem_alloc<512>(tslot);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tbase = *tslot;
    // TMEM columns: A stage s hi at 128 s, lo at 128 s + 64; D at 256 .. 256 + NF
    if (warp < 4) {                                             // rows K .. 127 of A stay zero: clear all 128 lanes once
        const float z[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < 256; c += 8) tc::tmem_st8(tbase + ((uint32_t)(32 * warp) << 16) + c, z);
        tc::tmem_wait_st();
    }
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t idesc = tc::make_idesc_tf32(128, NF, 0, 0);
    const int64_t nsub = (a.n + TM_SUB - 1) / TM_SUB;
    const int64_t my_sub = blockIdx.x < nsub ? (nsub - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    // K <= 32: the hi parts of R^T sit in TMEM lanes 0-31 and the lo parts in lanes 64-95 of the SAME columns, so one MMA
    // against Phi_hi yields r_hi.Phi_hi and r_lo.Phi_hi in different accumulator rows, one against Phi_lo the other two
    // products: two MMAs per k-step instead of three (and r_lo.Phi_lo comes for free).  Staging warps are then the even
    // ones (lane quarters 0 and 2), generators the odd ones.  K > 32: components 32-63 need lanes 32-63, three MMAs.
    const bool two = KW == 1;
    const int wq = warp & 3;

    if (warp == TM_BLOCK / 32 - 1) {
        // =========================== ISSUER: one thread feeds the tensor core and nothing else ===========================
        int since_flush = 0;
        // descriptor low words (address field | LBO) of stage 0, per part and k-step; the high word (SBO = 1024 B, version,
        // SWIZZLE_128B) is constant and the other stage is a constant offset in the address field
        uint32_t blo[2][TM_SUB / 8];
#pragma unroll
        for (int pt = 0; pt < 2; ++pt)
#pragma unroll
            for (int ks = 0; ks < TM_SUB / 8; ++ks) {
                const uint32_t addr = tc::smem_u32(Bs + (size_t)pt * bpart) + (uint32_t)((ks >> 2) * (NF * 128) + (ks & 3) * 32);
                blo[pt][ks] = ((addr >> 4) & 0x3FFFu) | 0x10000u;
            }
        const uint32_t bhi = (1024u >> 4) | (1u << 14) | (2u << 29);
        const uint32_t stage_step = nst == 2 ? (uint32_t)((2 * bpart * 4) >> 4) : 0u;
        for (int64_t t = 0; t < my_sub; ++t) {
            if (since_flush == TF_FLUSH) since_flush = 0;       // the staging warps flushed before they signalled afull
            mbar_wait(&afull[t & 1], (uint32_t)((t >> 1) & 1));
            mbar_wait(&bfull[t & 1], (uint32_t)((t >> 1) & 1));
            tc::fence_after_sync();
            if (lane == 0) {
                const uint32_t soff = (t & 1) ? stage_step : 0u;
                const uint32_t ah = tbase + 128 * (uint32_t)(t & 1), al = ah + 64, dt = tbase + 256;
                tc::mma_tf32_ts_w(dt, ah, blo[0][0] + soff, bhi, idesc, since_flush > 0 ? 1u : 0u);
#pragma unroll
                for (int ks = 1; ks < TM_SUB / 8; ++ks) tc::mma_tf32_ts_w(dt, ah + 8 * ks, blo[0][ks] + soff, bhi, idesc, 1u);
#pragma unroll
                for (int ks = 0; ks < TM_SUB / 8; ++ks) tc::mma_tf32_ts_w(dt, ah + 8 * ks, blo[1][ks] + soff, bhi, idesc, 1u);   // hi.lo
                if (!two) {
#pragma unroll
                    for (int ks = 0; ks < TM_SUB / 8; ++ks) tc::mma_tf32_ts_w(dt, al + 8 * ks, blo[0][ks] + soff, bhi, idesc, 1u);   // lo.hi
                }
                tc::mma_commit(&mdone[t & 1]);
            }
            __syncwarp();
            ++since_flush;
        }
    } else if (two ? (wq & 1) : wq >= 2) {
        // =========================== GENERATOR WARPS: Phi of sub-tile t into B stage t & 1 ===========================
        const int gtid = (((warp >> 2) << 1) + (two ? wq >> 1 : wq - 2)) * 32 + lane;     // 0 .. 255 over the generator warps
        // run-time D: four threads per sample, features by index mod 4; xo[r] = the sample's word offset inside row r of a
        // swizzled atom.  Compile-time D: warp gw owns the features p = gw (mod 8), lane l the samples 2 l and 2 l + 1.
        const int s_loc = DT > 0 ? 2 * lane : (gtid & 63), qd = gtid >> 6, gw = gtid >> 5;
        int xo[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) xo[r] = (s_loc >> 5) * (NF * 32) + (((((s_loc & 31) >> 2) ^ r)) << 2) + (s_loc & 3);
        const int o0 = (s_loc >> 5) * (NF * 32) + gw * 32 + (((((s_loc & 31) >> 2) ^ gw)) << 2) + (s_loc & 3);
        // compile-time D (a multiple of 4): the 64 x rows of a sub-tile (256 D contiguous bytes) come in by cp.async TWO sub-tiles
        // ahead into one of five buffers (see XNB above).  Global loads issued at the top of the iteration that consumes them
        // were 60 % of the generators' stall samples, and an L1 prefetch did not remove them.  Chunk c (16 bytes) of the tile
        // goes to row pair c / (D / 2).
        // per-thread constants of the tile fetch: at most one 16-byte chunk per generator thread (32 D/2 <= 256 chunks)
        constexpr int CPP = DT > 0 ? DT / 2 : 1;                // 16-byte chunks per row pair
        const bool has_chunk = DT > 0 && gtid < 32 * CPP;
        const uint32_t xdst0 = tc::smem_u32(xs + (gtid / CPP) * XPP + 4 * (gtid % CPP));
        const float* xsrc = x + (int64_t)blockIdx.x * TM_SUB * DT + (int64_t)gtid * 4;   // this thread's chunk of the next tile
        const int64_t xsrc_step = (int64_t)gridDim.x * TM_SUB * DT;
        uint32_t xbuf = 0, xbar = tc::smem_u32(xfull);          // next tile's buffer (byte offset) and its barrier
        int64_t xtt = 0;                                        // index of the next tile to fetch
        auto fetch_x = [&]() {
            if (DT > 0) {
                if (has_chunk) {
                    // every row of a tile exists unless it is this CTA's last one: then test the chunk (rows past the end: zero fill)
                    const int nbytes = (xtt + 1 < my_sub || (xtt < my_sub && xsrc < x + a.n * DT)) ? 16 : 0;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(xdst0 + xbuf), "l"(nbytes ? xsrc : x), "r"(nbytes)
                                 : "memory");
                }
                // arrives on the buffer's barrier when this thread's copies have landed (threads without a chunk at once)
                asm volatile("cp.async.mbarrier.arrive.noinc.shared.b64 [%0];" ::"r"(xbar) : "memory");
                xsrc += xsrc_step;
                ++xtt;
                xbuf += 32u * XPP * 4u;
                xbar += 8u;
                if (xbuf == XNB * 32u * XPP * 4u) { xbuf = 0; xbar -= 8u * XNB; }
            }
        };
        fetch_x();
        fetch_x();
        for (int64_t t = 0; t < my_sub; ++t) {
            const int64_t sb = blockIdx.x + t * gridDim.x;
            float xa[DT > 0 ? DT : 1], xb[DT > 0 ? DT : 1];
            if (DT > 0) {
                mbar_wait(&xfull[t % XNB], (uint32_t)((t / XNB) & 1));   // every generator thread's chunk of tile t has landed
                const uint32_t pp = tc::smem_u32(xs + (size_t)(t % XNB) * 32 * XPP + lane * XPP);
#pragma unroll
                for (int i = 0; i < DT / 4; ++i) {
                    const float4 fa = lds128(pp + 16 * i), fb = lds128(pp + 16 * (DT / 4 + i));
                    xa[4 * i] = fa.x; xa[4 * i + 1] = fa.y; xa[4 * i + 2] = fa.z; xa[4 * i + 3] = fa.w;
                    xb[4 * i] = fb.x; xb[4 * i + 1] = fb.y; xb[4 * i + 2] = fb.z; xb[4 * i + 3] = fb.w;
                }
                fetch_x();                                                 // buffer (t + 2) % 5: last read (tile t - 3) by every warp
            }
            // the MMAs that read this stage are done: sub-tile t - 2 with two stages, t - 1 with one (large feature counts)
            if (nst == 2) { if (t >= 2) mbar_wait(&mdone[t & 1], (uint32_t)(((t >> 1) - 1) & 1)); }
            else if (t >= 1) mbar_wait(&mdone[(t - 1) & 1], (uint32_t)(((t - 1) >> 1) & 1));
            const uint32_t Bh = tc::smem_u32(Bs + (size_t)(nst == 2 ? (t & 1) : 0) * 2 * bpart), Bl = Bh + 4u * (uint32_t)bpart;
            if (DT > 0) {
                switch (gw) {                     // warp-uniform
                    case 0: gen_features<DT, 0>(xa, xb, Bh, Bl, o0); break;
                    case 1: gen_features<DT, 1>(xa, xb, Bh, Bl, o0); break;
                    case 2: gen_features<DT, 2>(xa, xb, Bh, Bl, o0); break;
                    case 3: gen_features<DT, 3>(xa, xb, Bh, Bl, o0); break;
                    case 4: gen_features<DT, 4>(xa, xb, Bh, Bl, o0); break;
                    case 5: gen_features<DT, 5>(xa, xb, Bh, Bl, o0); break;
                    case 6: gen_features<DT, 6>(xa, xb, Bh, Bl, o0); break;
                    default: gen_features<DT, 7>(xa, xb, Bh, Bl, o0); break;
                }
            } else {
                asm volatile("bar.sync 1, 256;" ::: "memory");  // xs free (previous sub-tile's products formed)
                for (int e = gtid; e < TM_SUB * (D + 2); e += TM_GEN) {
                    const int sr = e / (D + 2), c = e - sr * (D + 2);
                    const int64_t rr = sb * TM_SUB + sr;
                    xs[e] = c < D ? (rr < a.n ? __ldg(x + rr * D + c) : 0.f) : (c == D ? 1.f : 0.f);
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                const float* xr = xs + s_loc * (D + 2);
                for (int p = qd; p < P; p += 4) {
                    const unsigned int code = ftab[p];
                    const float v = xr[code >> 8] * xr[code & 0xFF];
                    const float h = tc::tf32_trunc(v);
                    const uint32_t o = 4u * (uint32_t)((p >> 3) * 256 + (p & 7) * 32 + xo[p & 7]);
                    sts32(Bh + o, h);
                    sts32(Bl + o, v - h);
                }
            }
            tc::fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bfull[t & 1]);
        }
    } else {
        // =========================== STAGING WARPS: R^T into TMEM, MMA issue, flushes ===========================
        const int sq = warp >> 2;                               // which 16 of the 64 samples (and which features of a flush)
        const int c = two ? lane : 32 * wq + lane;              // the component of this lane
        const bool lo_part = two && wq == 2;                    // this warp stages (and flushes) the lo parts
        const int acol = two ? 32 * (wq >> 1) + lane : c;       // column of the float64 accumulator array
        const uint32_t lane_base = tbase + ((uint32_t)(32 * wq) << 16);
        int since_flush = 0;
        auto flush = [&]() {                                    // D rows (lane = component) -> float64, feature-major
            {
                for (int p0 = 16 * sq; p0 < NF; p0 += 64) {
                    float v[16];
                    double o[16];
                    double* ap = acc + (int64_t)p0 * 64 + acol;
#pragma unroll
                    for (int j = 0; j < 16; ++j) o[j] = __ldcg(ap + j * 64);     // 16 independent loads in flight
                    tc::tmem_ld16(lane_base + 256 + p0, v);
#pragma unroll
                    for (int j = 0; j < 16; ++j) __stcg(ap + j * 64, o[j] + (double)v[j]);
                }
            }
        };
        // this component's responsibilities of 16 samples (a warp reads one 128-byte row of r per sample), one sub-tile ahead
        float rv[2][8];
        auto load_r = [&](int64_t t) {
            const int64_t row0 = (blockIdx.x + t * gridDim.x) * TM_SUB + 16 * sq;
            if (t < my_sub && row0 + 16 <= a.n && c < KP) {            // all 16 rows exist: no per-row 64-bit compares
                const float* p = r_f32 + row0 * KP + c;
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int u = 0; u < 8; ++u) rv[j][u] = __ldg(p + (8 * j + u) * KP);
            } else {
#pragma unroll
                for (int j = 0; j < 2; ++j)
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int64_t row = row0 + 8 * j + u;
                        rv[j][u] = (t < my_sub && row < a.n && c < KP) ? __ldg(r_f32 + row * KP + c) : 0.f;
                    }
            }
        };
        load_r(0);
        for (int64_t t = 0; t < my_sub; ++t) {
            if (!lo_part && t + 3 < my_sub && 128 * lane < 16 * KP * 4) {
                // r rows of sub-tile t + 2 (this warp's 16 rows = 64 KP bytes, contiguous) towards L2 / L1; sub-tile t + 2 is
                // not the CTA's last, so all of its rows exist
                const char* pr = reinterpret_cast<const char*>(r_f32 + ((blockIdx.x + (t + 2) * gridDim.x) * TM_SUB + 16 * sq) * KP);
                asm volatile("prefetch.global.L1 [%0];" ::"l"(pr + 128 * lane));
            }
            if (t >= 2) mbar_wait(&mdone[t & 1], (uint32_t)(((t >> 1) - 1) & 1));     // A buffer t & 1 free
            tc::fence_after_sync();
            if (since_flush == TF_FLUSH) {
                // every MMA issued so far has completed?  sub-tile t - 1 must be waited for explicitly
                mbar_wait(&mdone[(t - 1) & 1], (uint32_t)(((t - 1) >> 1) & 1));
                tc::fence_after_sync();
                flush();
                since_flush = 0;
                tc::fence_before_sync();
            }
            {
                const uint32_t abase = lane_base + 128 * (uint32_t)(t & 1);
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    float h[8], l[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) { h[u] = tc::tf32_trunc(rv[j][u]); l[u] = rv[j][u] - h[u]; }
                    if (two) {
                        tc::tmem_st8(abase + 16 * sq + 8 * j, lo_part ? l : h);
                    } else {
                        tc::tmem_st8(abase + 16 * sq + 8 * j, h);
                        tc::tmem_st8(abase + 64 + 16 * sq + 8 * j, l);
                    }
                }
                load_r(t + 1);
                tc::tmem_wait_st();
            }
            tc::fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&afull[t & 1]);          // this warp's part of A is in place (and its flush is done)
            ++since_flush;
        }
        if (my_sub > 0) {
            mbar_wait(&mdone[(my_sub - 1) & 1], (uint32_t)(((my_sub - 1) >> 1) & 1));
            tc::fence_after_sync();
            if (since_flush > 0) flush();
        }
    }
    __threadfence_block();
    __syncthreads();
    // ---- per-CTA partial (logical layout [K][pitch] float64) ----
    const int64_t len = L.stats_len;
    double* part = a.workspace + (int64_t)blockIdx.x * len;
    for (int64_t o = tid; o < len; o += TM_BLOCK) part[o] = 0.0;
    __syncthreads();
    for (int e = tid; e < K * P; e += TM_BLOCK) {
        const int k = e / P, p = e - k * P;
        part[(int64_t)k * L.pitch + p] = acc[(int64_t)p * 64 + k] + (two ? acc[(int64_t)p * 64 + 32 + k] : 0.0);
    }
    if (blockIdx.x == 0 && tid == 0) {
        double v = 0.0;
        for (int i = 0; i < n_ews; ++i) v += ews[i];              // fixed order: deterministic
        part[(int64_t)K * L.pitch + BGMM_STATS_ENTROPY] = v;
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tbase);
}

// ---- host side ----
static int tf32_grid(int64_t units) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)(units < 1 ? 1 : (units < sms ? units : sms));
}

struct Tf32MPlan { bool ok; int NF, nst; size_t smem; };
static Tf32MPlan plan_tf32_m(int K, int D) {
    Tf32MPlan m{};
    const int P = feat_count(D);
    m.NF = (P + 15) & ~15;
    auto bytes = [&](int nst) {
        return sizeof(float) * ((size_t)2 * nst * m.NF * TM_SUB + (size_t)TM_SUB * (D + 2) + 5 * 32 * (2 * 16 + 4)) +
               sizeof(unsigned short) * ((P + 7) & ~7) + 128 + 1024;
    };
    m.nst = bytes(2) <= 220 * 1024 ? 2 : 1;                    // two Phi stages when they fit (P <= ~190), else one
    m.smem = bytes(m.nst);
    m.ok = m.NF <= 256 && K <= 64 && m.smem <= 220 * 1024;
    return m;
}

bool tf32_pass_supported(int K, int D, int dtype) { return tf32_supported(K, D, dtype) && plan_tf32_m(K, D).ok && K >= 2; }

// doubles of workspace: per-CTA partial statistics + entropy partials + the operand image + the CTA-private float64
// accumulators of the statistics kernel + r (float32 [n][KP])
static int64_t tf32_fixed_doubles(int K, int D) {
    return (int64_t)160 * ((int64_t)K * feat_pitch(D) + 8) + 160 + (tf32_image_floats(K, D) + 1) / 2 + 8 + (int64_t)160 * 256 * 64;
}
int64_t tf32_workspace_doubles(int K, int D, int64_t n) {
    if (!tf32_pass_supported(K, D, BGMM_F32)) return 0;
    const Tf32Plan p = plan_tf32(K, D);
    return tf32_fixed_doubles(K, D) + (n * p.KP + 1) / 2 + 8;
}

template <int DP, int KD, bool OUT>
static cudaError_t launch_e_t(const Tf32Plan& p, const PassArgs& a, const Layout& L, const float* img, float* r_f32, double* ews,
                              int grid, cudaStream_t stream) {
    auto kern = pass_tf32_e_kernel<DP, KD, OUT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_e);
    if (e != cudaSuccess) return e;
    // dbg is always 0.  Removing the parameter and its two tests changes the kernel's register allocation and made the c2f32
    // step 1.4 % slower on a B200 at 1000 W (2.575 against 2.538 ms), so the runtime zero stays until the epilogue is re-tuned.
    return launch_pdl(kern, dim3(grid), dim3(TE_BLOCK), p.smem_e, stream, a, L, img, r_f32, ews, p.KP, p.cpc, p.nchunks, p.nmma, 0);
}
template <int DP, int KD>
static cudaError_t launch_e(const Tf32Plan& p, const PassArgs& a, const Layout& L, const float* img, float* r_f32, double* ews,
                            int grid, cudaStream_t stream) {
    const bool out = a.r_out != nullptr || a.lnrho_out != nullptr || a.argmax_out != nullptr;
    return out ? launch_e_t<DP, KD, true>(p, a, L, img, r_f32, ews, grid, stream)
               : launch_e_t<DP, KD, false>(p, a, L, img, r_f32, ews, grid, stream);
}

template <int DT>
static cudaError_t launch_m_t(const Tf32MPlan& m, const PassArgs& a, const Layout& L, const float* r_f32, int KP, double* acct,
                              const double* ews, int n_ews, int grid, cudaStream_t stream) {
    auto kern = pass_tf32_m_kernel<DT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m.smem);
    if (e != cudaSuccess) return e;
    return launch_pdl(kern, dim3(grid), dim3(TM_BLOCK), m.smem, stream, a, L, r_f32, KP, m.NF, m.nst, acct, ews, n_ews);
}

int launch_pass_tf32(const PassArgs& a, int K, int D, int dtype, cudaStream_t stream) {
    if (!tf32_pass_supported(K, D, dtype)) {
        set_error("bgmm_pass(tf32): unsupported shape K=%d D=%d dtype=%d (float32 X, 2 <= K <= 64, D <= 31, K * P accumulators "
                  "in 128 TMEM columns)", K, D, dtype);
        return BGMM_ENOSUP;
    }
    const Tf32Plan p = plan_tf32(K, D);
    const Tf32MPlan m = plan_tf32_m(K, D);
    const Layout L = make_layout(K, D, 1);
    const int64_t len = L.stats_len;
    double* ews = a.workspace + (int64_t)160 * len;
    float* img = reinterpret_cast<float*>(ews + 160);
    double* acct = ews + 160 + (tf32_image_floats(K, D) + 1) / 2 + 8;
    float* r_f32 = reinterpret_cast<float*>(a.workspace + tf32_fixed_doubles(K, D));
    const int grid_e = tf32_grid((a.n + TF_TILE - 1) / TF_TILE), grid_m = tf32_grid((a.n + TM_SUB - 1) / TM_SUB);
    cudaError_t e = launch_pdl(tf32_prep_kernel, dim3(32), dim3(256), 0, stream, (const double*)a.state, L, img, p.DP, p.KD,
                               p.KP, p.cpc, p.nchunks, p.nmma, a.force, a.crit_limit);
    if (e != cudaSuccess) return check_cuda(e, "tf32_prep_kernel launch");
#define BGMM_TF_E(dp, kd) if (p.DP == dp && p.KD == kd) e = launch_e<dp, kd>(p, a, L, img, r_f32, ews, grid_e, stream);
    BGMM_TF_E(4, 8) else BGMM_TF_E(8, 8) else BGMM_TF_E(8, 16) else BGMM_TF_E(16, 16) else BGMM_TF_E(16, 24)
    else BGMM_TF_E(32, 24) else BGMM_TF_E(32, 32)
    else { set_error("bgmm_pass(tf32): no E instantiation for DP=%d KD=%d", p.DP, p.KD); return BGMM_ENOSUP; }
#undef BGMM_TF_E
    if (e != cudaSuccess) return check_cuda(e, "pass_tf32_e_kernel launch");
    // compile-time D for the common dimensions (static feature indices), the table-driven instantiation otherwise
    if (D == 16) e = launch_m_t<16>(m, a, L, r_f32, p.KP, acct, ews, grid_e, grid_m, stream);
    else if (D == 8) e = launch_m_t<8>(m, a, L, r_f32, p.KP, acct, ews, grid_e, grid_m, stream);
    else if (D == 4) e = launch_m_t<4>(m, a, L, r_f32, p.KP, acct, ews, grid_e, grid_m, stream);
    else e = launch_m_t<0>(m, a, L, r_f32, p.KP, acct, ews, grid_e, grid_m, stream);
    if (e != cudaSuccess) return check_cuda(e, "pass_tf32_m_kernel launch");
    launch_reduce_partials(a, L, grid_m, stream);
    return check_cuda(cudaGetLastError(), "pass_tf32 launch");
}

}  // namespace bgmm
