// bgmm_pass, generic variant (BGMM_PASS_SIMPLE): scalar fp64 FMA, any K and D.
//
// One thread owns one sample for the E-step (ln rho_nk = coef_k . phi(x'_n), softmax over k, entropy term);
// the statistics raw_k = sum_n r_nk phi(x'_n) are then accumulated with one thread per OUTPUT element over the
// tile held in shared memory, so no atomics are needed and the result is deterministic.
// Replaces `_update_q_z` :772-784, `_calc_n_x_bar_s` :725-732 and the `xlogy` term :704 of
// /root/reference/bayesml/gaussianmixture/_gaussianmixture.py.  This is the correctness baseline on the GPU
// and the path for shapes the tensor-pipe kernel does not cover; the fast path is bgmm_pass_dmma.cu.
//
// DIRECT instantiation (BGMM_PASS_DIRECT): the conditioning-safe form of the same sweep.  ln rho_nk is evaluated from the
// explicit differences d = x' - m'_k  (a_k + sum_{i>=j} coefq_ij d_i d_j: the reference's (x - m_k)^T Lambda_k (x - m_k),
// :775-781) and the statistics are the moments of (x' - shift_k) with shift_k ~ the component's own mean (state.SHIFT), i.e.
// the reference's two-pass centred form (:730-732) up to a shift that bgmm_small removes.  No term grows with the distance
// of a component from the global centre, at twice the arithmetic of the feature-map form.  It runs in place of the
// requested variant whenever bgmm_small has raised ctrl.ROBUST for the current parameter set.
#include "bgmm_common.cuh"
#include <math.h>

namespace bgmm {

constexpr int SIMPLE_THREADS = 128;


template <typename T, bool DIRECT>
__global__ void __launch_bounds__(SIMPLE_THREADS) pass_simple_kernel(const PassArgs a, const Layout L, const int tile) {
    extern __shared__ double sm[];
    const int K = L.K, D = L.D, P = L.P, tid = threadIdx.x;
    pdl_trigger();
    pdl_wait();
    volatile int* ctrl = reinterpret_cast<volatile int*>(a.state + L.ctrl);
    if (!a.force && ctrl[BGMM_CTRL_DONE]) return;
    if (!a.ignore_robust && robust_set(ctrl, a.crit_limit) != DIRECT) return;   // the other form does this pass
    const double* __restrict__ Pc = a.state + L.params[ctrl[BGMM_CTRL_CUR]];
    const double* __restrict__ coef = Pc + L.p_coef;
    const double* __restrict__ mvec = Pc + L.p_m;              // [K][D] (DIRECT)
    const double* __restrict__ acst = Pc + L.p_acst;           // [K]    (DIRECT)
    const double* __restrict__ shift = a.state + L.shift;      // [K][D] (DIRECT)
    const T* __restrict__ x = static_cast<const T*>(a.x);

    const int xp = D + 1;                 // padded row pitch: conflict-free per-thread rows
    double* xs = sm;                      // [tile][D+1]
    double* rs = xs + (size_t)tile * xp;  // [tile][K]
    double* scratch = rs + (size_t)tile * K;  // [40]

    const int64_t len = L.stats_len;
    double* part = a.workspace + (int64_t)blockIdx.x * len;
    for (int64_t o = tid; o < len; o += SIMPLE_THREADS) part[o] = 0.0;
    double ent = 0.0;

    const int64_t ntiles = (a.n + tile - 1) / tile;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * tile;
        const int rows = (int)min((int64_t)tile, a.n - row0);
        __syncthreads();
        for (int e = tid; e < rows * D; e += SIMPLE_THREADS) {
            const int s = e / D, d = e - s * D;
            xs[s * xp + d] = (double)x[row0 * D + e];
        }
        __syncthreads();
        for (int s = tid; s < rows; s += SIMPLE_THREADS) {
            const double* xr = xs + s * xp;
            double* rr = rs + (size_t)s * K;
            if (a.r_in != nullptr) {
                double e_loc = 0.0;
                for (int k = 0; k < K; ++k) {
                    const double r = a.r_in[(row0 + s) * K + k];
                    rr[k] = r;
                    if (r > 0.0) e_loc += r * log(r);   // xlogy(r, r), :704
                }
                ent += e_loc;
                continue;
            }
            double mx = -INFINITY;
            for (int k = 0; k < K; ++k) {
                const double* c = coef + (int64_t)k * L.pitch;
                double acc;
                int q = 1 + D;
                if constexpr (DIRECT) {
                    const double* mk = mvec + (int64_t)k * D;
                    acc = acst[k];
                    for (int i = 0; i < D; ++i) {
                        double row = 0.0;
                        for (int j = 0; j <= i; ++j) row = fma(c[q + j], xr[j] - mk[j], row);
                        acc = fma(row, xr[i] - mk[i], acc);
                        q += i + 1;
                    }
                } else {
                    acc = c[0];
                    for (int i = 0; i < D; ++i) acc = fma(c[1 + i], xr[i], acc);
                    for (int i = 0; i < D; ++i) {
                        const double xi = xr[i];
                        double row = 0.0;
                        for (int j = 0; j <= i; ++j) row = fma(c[q + j], xr[j], row);
                        acc = fma(row, xi, acc);
                        q += i + 1;
                    }
                }
                rr[k] = acc;
                mx = fmax(mx, acc);
            }
            if (a.lnrho_out != nullptr)
                for (int k = 0; k < K; ++k) a.lnrho_out[(row0 + s) * K + k] = rr[k];
            double sum = 0.0, dot = 0.0;
            for (int k = 0; k < K; ++k) {
                const double z = rr[k] - mx;
                const double e = exp(z);
                rr[k] = e;
                sum += e;
                if (e > 0.0) dot = fma(e, z, dot);
            }
            // sum_k r ln r = sum_k r_k (ln rho_k - max) - ln(sum)   [sum_k r_k = 1]
            ent += dot / sum - log(sum);
            int best = 0;
            double bestv = -1.0;
            for (int k = 0; k < K; ++k) {
                const double r = rr[k] / sum;
                rr[k] = r;
                if (r > bestv) { bestv = r; best = k; }   // first index on ties, as np.argmax (:1191)
            }
            if (a.r_out != nullptr)
                for (int k = 0; k < K; ++k) a.r_out[(row0 + s) * K + k] = rr[k];
            if (a.argmax_out != nullptr) a.argmax_out[row0 + s] = best;
        }
        __syncthreads();
        // statistics: one thread per output (k, p)
        for (int o = tid; o < K * P; o += SIMPLE_THREADS) {
            const int k = o / P, p = o - k * P;
            double acc = 0.0;
            const double* sk = shift + (int64_t)k * D;
            if (p == 0) {
                for (int s = 0; s < rows; ++s) acc += rs[(size_t)s * K + k];
            } else if (p <= D) {
                const int i = p - 1;
                const double si = DIRECT ? sk[i] : 0.0;
                for (int s = 0; s < rows; ++s) acc = fma(rs[(size_t)s * K + k], xs[s * xp + i] - si, acc);
            } else {
                const int q = p - 1 - D;
                int i = (int)((sqrt(8.0 * q + 1.0) - 1.0) * 0.5);
                while (i * (i + 1) / 2 > q) --i;
                while ((i + 1) * (i + 2) / 2 <= q) ++i;
                const int j = q - i * (i + 1) / 2;
                const double si = DIRECT ? sk[i] : 0.0, sj = DIRECT ? sk[j] : 0.0;
                for (int s = 0; s < rows; ++s)
                    acc = fma(rs[(size_t)s * K + k], (xs[s * xp + i] - si) * (xs[s * xp + j] - sj), acc);
            }
            part[(int64_t)k * L.pitch + p] += acc;
        }
    }
    ent = block_sum(ent, scratch);
    if (tid == 0) part[(int64_t)K * L.pitch + BGMM_STATS_ENTROPY] = ent;
    finish_pass(a, L, ctrl, DIRECT ? 1.0 : 0.0);
}

static int simple_tile(int K, int D) {
    // shared memory per sample: (D+1) + K doubles; keep the tile a multiple of 32 and <= 128
    const size_t per = sizeof(double) * ((size_t)D + 1 + K);
    int tile = (int)((200 * 1024 - 40 * sizeof(double)) / per);
    if (tile > SIMPLE_THREADS) tile = SIMPLE_THREADS;
    if (tile >= 32) tile &= ~31;
    return tile;
}

int simple_grid_cap(int K, int D) {
    const int64_t len = (int64_t)K * feat_pitch(D) + 8;
    int64_t cap = ((int64_t)256 << 20) / (8 * len);   // <= 256 MiB of partials
    if (cap > 148 * 4) cap = 148 * 4;
    if (cap < 1) cap = 1;
    return (int)cap;
}

int launch_pass_simple(const PassArgs& a, int K, int D, int dtype, int direct, cudaStream_t stream) {
    const Layout L = make_layout(K, D, 1);  // offsets used by the pass do not depend on hist_len
    const int tile = simple_tile(K, D);
    if (tile < 1) {
        set_error("bgmm_pass(simple): K=%d D=%d does not fit in shared memory", K, D);
        return BGMM_ENOSUP;
    }
    const size_t smem = sizeof(double) * ((size_t)tile * (D + 1 + K) + 40);
    const int64_t ntiles = (a.n + tile - 1) / tile;
    int64_t grid64 = ntiles < 1 ? 1 : ntiles;
    if (grid64 > simple_grid_cap(K, D)) grid64 = simple_grid_cap(K, D);
    const int grid = (int)grid64;
    auto go = [&](auto kern) -> int {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(pass_simple)");
        return check_cuda(launch_pdl(kern, dim3(grid), dim3(SIMPLE_THREADS), smem, stream, a, L, tile),
                          "pass_simple_kernel launch");
    };
    if (dtype == BGMM_F64) return direct ? go(pass_simple_kernel<double, true>) : go(pass_simple_kernel<double, false>);
    return direct ? go(pass_simple_kernel<float, true>) : go(pass_simple_kernel<float, false>);
}

}  // namespace bgmm
