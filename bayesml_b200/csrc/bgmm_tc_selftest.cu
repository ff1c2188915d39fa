// bgmm_tc_selftest: D[128][N] = A[128][Kd] . B[N][Kd]^T on the 5th-generation tensor cores (tcgen05.mma kind::tf32,
// operands in shared memory, accumulator in tensor memory) for either operand layout — the unit test of the descriptor
// conventions in bgmm_tc.cuh that the fp32-mode kernels rely on (tests/test_gpu_tc.py compares with a tf32-truncated matmul).
#include "bgmm_common.cuh"
#include "bgmm_mma.cuh"
#include "bgmm_tc.cuh"

namespace bgmm {

__global__ void __launch_bounds__(128) tc_selftest_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                          float* __restrict__ Dout, const int N, const int Kd,
                                                          const int a_mn, const int b_mn_arg) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t mbar;
    __shared__ uint32_t tmem_slot;
    float* As = reinterpret_cast<float*>(smem_raw);            // 128 x Kd
    float* Bs = As + 128 * Kd;                                 // N x Kd
    const int b_mn = b_mn_arg >= 4 ? 0 : b_mn_arg;             // 4 / 5: the latency / throughput probes, K-major no-swizzle B
    const bool b_sw = b_mn == 3;                               // B K-major in the 128-byte-swizzle layout (Kd % 32 == 0)
    if (b_sw) Bs = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(Bs) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, warp = tid >> 5;
    const int kch = Kd / 4, kgr = Kd / 8;
    // K-major: row-group major, k-chunks contiguous -> LBO = 128 B, SBO = kch * 128 B
    // MN-major: k-group major over mn-chunks          -> SBO = 128 B (next 4 m), LBO = (rows / 4) * 128 B (next 8 k)
    const int a_lbo = a_mn ? (128 / 4) * 32 : 32, a_sbo = a_mn ? 32 : kch * 32;      // in floats
    const int b_lbo = b_mn ? (N / 4) * 32 : 32, b_sbo = b_mn ? 32 : kch * 32;
    for (int e = tid; e < 128 * Kd; e += 128) {
        const int r = e / Kd, c = e - r * Kd;
        As[a_mn ? tc::mnmajor_off(c, r, a_lbo, a_sbo) : tc::kmajor_off(r, c, a_lbo, a_sbo)] = A[e];
    }
    for (int e = tid; e < N * Kd; e += 128) {
        const int r = e / Kd, c = e - r * Kd;
        if (b_sw) Bs[(c >> 5) * (N / 8) * 256 + tc::sw128_off(r, c & 31)] = B[e];
        else Bs[b_mn ? tc::mnmajor_off(c, r, b_lbo, b_sbo) : tc::kmajor_off(r, c, b_lbo, b_sbo)] = B[e];
    }
    if (tid == 0) mbar_init(&mbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (warp == 0) tc::tmem_alloc<512>(&tmem_slot);
    tc::fence_proxy_async();
    tc::fence_before_sync();
    __syncthreads();
    tc::fence_after_sync();
    const uint32_t tbase = tmem_slot;
    if (a_mn == 2) {
        // A in TENSOR MEMORY: every thread stores its own row (lane = m) at columns 256 + k
        for (int ks = 0; ks < kgr; ++ks) {
            float v[8];
            for (int j = 0; j < 8; ++j) v[j] = A[tid * Kd + 8 * ks + j];
            tc::tmem_st8(tbase + ((uint32_t)(32 * warp) << 16) + 256 + 8 * ks, v);
        }
        tc::tmem_wait_st();
        tc::fence_before_sync();
        __syncthreads();
        tc::fence_after_sync();
    }
    if (tid == 0 && a_mn == 2) {
        const uint32_t idesc = tc::make_idesc_tf32(128, N, 0, b_sw ? 0 : b_mn);
        for (int ks = 0; ks < kgr; ++ks) {
            const uint32_t b_addr = tc::smem_u32(Bs) + 4 * (b_mn ? ks * b_lbo : 2 * ks * b_lbo);
            const uint64_t bd = b_sw ? tc::make_smem_desc_sw128(tc::smem_u32(Bs) + (ks >> 2) * (N / 8) * 1024 + (ks & 3) * 32, 1024)
                                     : tc::make_smem_desc(b_addr, 4 * b_lbo, 4 * b_sbo);
            tc::mma_tf32_ts(tbase, tbase + 256 + 8 * ks, bd, idesc, ks > 0 ? 1u : 0u);
        }
        tc::mma_commit(&mbar);
    } else if (tid == 0) {
        const uint32_t idesc = tc::make_idesc_tf32(128, N, a_mn, b_mn);
        for (int ks = 0; ks < kgr; ++ks) {
            // one MMA consumes 8 k: K-major -> two k-chunks (advance 2 * LBO), MN-major -> one k-group (advance LBO)
            const uint32_t a_addr = tc::smem_u32(As) + 4 * (a_mn ? ks * a_lbo : 2 * ks * a_lbo);
            const uint32_t b_addr = tc::smem_u32(Bs) + 4 * (b_mn ? ks * b_lbo : 2 * ks * b_lbo);
            tc::mma_tf32(tbase, tc::make_smem_desc(a_addr, 4 * a_lbo, 4 * a_sbo), tc::make_smem_desc(b_addr, 4 * b_lbo, 4 * b_sbo),
                         idesc, ks > 0 ? 1u : 0u);
        }
        tc::mma_commit(&mbar);
    }
    mbar_wait(&mbar, 0);
    tc::fence_after_sync();
    if (a_mn == 2 && b_mn_arg >= 4) {
        // latency probe (tests/test_gpu_tc.py::test_tcgen05_round_trip_latency): ONE thread issues one MMA, commits and waits for
        // the mbarrier, 256 times back to back; Dout[0] = cycles per round trip (issue -> complete -> commit -> arrival seen)
        if (tid == 0) {
            const uint32_t idesc = tc::make_idesc_tf32(128, N, 0, 0);
            const uint64_t bd = tc::make_smem_desc(tc::smem_u32(Bs), 4 * 32, 4 * (Kd / 4) * 32);
            uint32_t phase = 1;
            const long long t0 = clock64();
            const int per_commit = b_mn_arg == 5 ? 16 : 1;     // 5: sixteen MMAs back to back per commit (throughput)
            for (int it = 0; it < 256; ++it) {
                for (int j = 0; j < per_commit; ++j) tc::mma_tf32_ts(tbase, tbase + 256, bd, idesc, 1u);
                tc::mma_commit(&mbar);
                mbar_wait(&mbar, phase);
                phase ^= 1u;
            }
            const long long t1 = clock64();
            Dout[0] = (float)((t1 - t0) / 256.0);
        }
        __syncthreads();
        tc::fence_before_sync();
        __syncthreads();
        if (warp == 0) tc::tmem_dealloc<512>(tbase);
        return;
    }
    for (int c0 = 0; c0 < N; c0 += 16) {
        float v[16];
        tc::tmem_ld16(tbase + ((uint32_t)(32 * warp) << 16) + c0, v);
        const int row = tid;
#pragma unroll
        for (int j = 0; j < 16; ++j) Dout[row * N + c0 + j] = v[j];
    }
    tc::fence_before_sync();
    __syncthreads();
    if (warp == 0) tc::tmem_dealloc<512>(tbase);
}

}  // namespace bgmm

extern "C" int bgmm_tc_selftest(const float* A, const float* B, float* D, int N, int Kd, int a_mn_major, int b_mn_major,
                                void* stream) {
    using namespace bgmm;
    if (A == nullptr || B == nullptr || D == nullptr || N < 16 || N > 256 || (N % 16) != 0 || Kd < 8 || (Kd % 8) != 0 ||
        Kd > 64) {
        set_error("bgmm_tc_selftest: bad argument (N=%d multiple of 16 in [16, 256], Kd=%d multiple of 8 in [8, 64])", N, Kd);
        return BGMM_EINVAL;
    }
    if (b_mn_major == 3 && (a_mn_major != 2 || (Kd % 32) != 0)) {
        set_error("bgmm_tc_selftest: the swizzled B layout (3) needs A in tensor memory (2) and Kd a multiple of 32");
        return BGMM_EINVAL;
    }
    const size_t smem = sizeof(float) * (size_t)(128 + N) * Kd + 128 + 1024;
    cudaError_t e = cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(tc_selftest)");
    launch(tc_selftest_kernel, 1, 128, smem, (cudaStream_t)stream, A, B, D, N, Kd, a_mn_major, b_mn_major);
    return check_cuda(cudaGetLastError(), "tc_selftest_kernel launch");
}
