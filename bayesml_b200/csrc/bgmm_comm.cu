// Peer-memory exchange of the sufficient statistics between the GPUs of one NVLink/NVSwitch box.
//
// The per-iteration collective of the row-sharded fit is an all-reduce of K*PITCH+8 doubles (41 KB at K=32, D=16) that
// is followed immediately by bgmm_small.  Instead of an NCCL call between the two kernels, every rank PUBLISHES its
// local statistics into an exchange block that its peers have mapped through CUDA IPC (the last CTA of every bgmm_pass's
// reduction: copy + system fence + a stamp written into every peer's flag array, publish_stats in bgmm_common.cuh), and
// bgmm_small itself waits for the stamps and sums the peers' blocks straight out of peer memory, in rank order — so the
// reduced values are bit-identical on every rank and the transfer is fused into the kernels on either side (no extra
// launch, no ring/tree latency).
// Two exchange buffers (sequence parity) make the protocol safe without a second barrier: a rank can run at most one
// exchange ahead of the slowest peer, because its next bgmm_small needs that peer's next stamp.
#include "bgmm_common.cuh"
#include <string.h>

using namespace bgmm;

extern "C" int64_t bgmm_comm_block_doubles(int K, int D) {
    if (K <= 0 || D <= 0) return 0;
    return 2 * ((int64_t)K * feat_pitch(D) + 8) + 2 * BGMM_MAX_RANKS;
}

extern "C" int bgmm_comm_alloc(int64_t doubles, void** base_out, void* ipc_handle_out) {
    if (doubles <= 0 || base_out == nullptr || ipc_handle_out == nullptr) {
        set_error("bgmm_comm_alloc: bad argument");
        return BGMM_EINVAL;
    }
    void* p = nullptr;
    int rc = check_cuda(cudaMalloc(&p, (size_t)doubles * sizeof(double)), "cudaMalloc(exchange block)");
    if (rc) return rc;
    rc = check_cuda(cudaMemset(p, 0, (size_t)doubles * sizeof(double)), "cudaMemset(exchange block)");
    if (rc) { cudaFree(p); return rc; }
    cudaIpcMemHandle_t h;
    rc = check_cuda(cudaIpcGetMemHandle(&h, p), "cudaIpcGetMemHandle");
    if (rc) { cudaFree(p); return rc; }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(ipc_handle_out, &h, sizeof(h));
    *base_out = p;
    return BGMM_OK;
}

extern "C" int bgmm_comm_open(const void* ipc_handle, void** ptr_out) {
    if (ipc_handle == nullptr || ptr_out == nullptr) { set_error("bgmm_comm_open: bad argument"); return BGMM_EINVAL; }
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle, sizeof(h));
    return check_cuda(cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
}

extern "C" int bgmm_comm_close(void* ptr) { return check_cuda(cudaIpcCloseMemHandle(ptr), "cudaIpcCloseMemHandle"); }
extern "C" int bgmm_comm_free(void* base) { return check_cuda(cudaFree(base), "cudaFree(exchange block)"); }
