// nb2_peer.cu - end-of-frame state gather across the GPUs of one node WITHOUT compute kernels (SURVEY.md §8(e)).
//
// The reference design is an ncclAllGather of body_q / body_qd after every frame.  NCCL's all-gather runs as kernels: on a GPU
// whose solver kernel needs every SM to stay a single wave (13.8 one-warp CTAs per SM at 4096 envs) those kernels push the tail
// of the wave out (round 1: 90 % weak scaling at N = 8, DESIGN.md §6).  Here every rank owns a symmetric receive buffer
// (cudaMalloc + CUDA IPC, mapped by all peers); after a frame a rank WRITES its slice into every peer's buffer with the copy
// engines (cudaMemcpyAsync on peer-mapped pointers: NVLink DMA, no SM), then publishes the frame's sequence number in the
// peer's flag word; a consumer waits on its own flag words with a stream memory operation (cuStreamWaitValue32: no SM either).
// Two receive slots (sequence parity) let frame f+1 land while frame f is still being read.
#include <cuda.h>

#include <cstring>

#include "nb2_internal.cuh"

struct nb2_peer_gather {
    int device = 0, rank = 0, world = 1;
    size_t bytes_per_rank = 0;
    char* recv = nullptr;      // [2 slots][world][bytes_per_rank]
    int* flags = nullptr;      // [2 slots][world] sequence numbers
    std::vector<char*> peer_recv;  // peer-mapped addresses (own rank: the local pointers)
    std::vector<int*> peer_flags;
    int** d_peer_flags = nullptr;  // device copy of peer_flags for the signal kernel
    CUresult (*wait32)(CUstream, CUdeviceptr, cuuint32_t, unsigned int) = nullptr;
};

namespace nb2 {

__global__ void peer_signal_kernel(int** flags, int world, int index, int value) {
    __threadfence_system();
    for (int p = threadIdx.x; p < world; p += blockDim.x) {
        volatile int* f = flags[p] + index;
        *f = value;
    }
    __threadfence_system();
}
__global__ void peer_wait_kernel(const int* flags, int world, int value) {  // fallback when stream memory operations are unavailable
    for (int p = threadIdx.x; p < world; p += blockDim.x) {
        const volatile int* f = flags + p;
        while (*f - value < 0) __nanosleep(200);
    }
}

}  // namespace nb2

using namespace nb2;

extern "C" {

size_t nb2_peer_gather_handle_bytes(void) { return 2 * sizeof(cudaIpcMemHandle_t); }

nb2_status nb2_peer_gather_create(int32_t device, int32_t rank, int32_t world_size, size_t bytes_per_rank, nb2_peer_gather** out) {
    if (!out || world_size < 1 || rank < 0 || rank >= world_size || bytes_per_rank == 0) {
        set_error("nb2_peer_gather_create: invalid argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    *out = nullptr;
    int prev = -1;
    cudaGetDevice(&prev);
    NB2_CUDA_CHECK(cudaSetDevice(device));
    nb2_peer_gather* g = new nb2_peer_gather();
    g->device = device;
    g->rank = rank;
    g->world = world_size;
    g->bytes_per_rank = (bytes_per_rank + 15) & ~size_t(15);
    void* p = nullptr;
    NB2_CUDA_CHECK(cudaMalloc(&p, 2 * size_t(world_size) * g->bytes_per_rank));
    g->recv = static_cast<char*>(p);
    NB2_CUDA_CHECK(cudaMalloc(&p, 2 * size_t(world_size) * sizeof(int)));
    g->flags = static_cast<int*>(p);
    NB2_CUDA_CHECK(cudaMemset(g->flags, 0, 2 * size_t(world_size) * sizeof(int)));
    NB2_CUDA_CHECK(cudaMalloc(&p, size_t(world_size) * sizeof(int*)));
    g->d_peer_flags = static_cast<int**>(p);
    g->peer_recv.assign(size_t(world_size), nullptr);
    g->peer_flags.assign(size_t(world_size), nullptr);
    g->peer_recv[rank] = g->recv;
    g->peer_flags[rank] = g->flags;
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
        g->wait32 = reinterpret_cast<decltype(g->wait32)>(fn);
    cudaGetLastError();
    if (prev >= 0 && prev != device) cudaSetDevice(prev);
    *out = g;
    return NB2_OK;
}

void* nb2_peer_gather_buffer(nb2_peer_gather* g, int32_t slot) {
    return g ? g->recv + size_t(slot & 1) * size_t(g->world) * g->bytes_per_rank : nullptr;
}
size_t nb2_peer_gather_stride(const nb2_peer_gather* g) { return g ? g->bytes_per_rank : 0; }

nb2_status nb2_peer_gather_export(nb2_peer_gather* g, void* handle_out) {
    if (!g || !handle_out) {
        set_error("nb2_peer_gather_export: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    cudaIpcMemHandle_t h[2];
    NB2_CUDA_CHECK(cudaIpcGetMemHandle(&h[0], g->recv));
    NB2_CUDA_CHECK(cudaIpcGetMemHandle(&h[1], g->flags));
    std::memcpy(handle_out, h, sizeof(h));
    return NB2_OK;
}

// all_handles: world_size entries of nb2_peer_gather_handle_bytes() each, in rank order (exchanged by the host, e.g.
// torch.distributed.all_gather_object); peers must live on other devices of the same node with P2P access
nb2_status nb2_peer_gather_connect(nb2_peer_gather* g, const void* all_handles) {
    if (!g || !all_handles) {
        set_error("nb2_peer_gather_connect: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    int prev = -1;
    cudaGetDevice(&prev);
    NB2_CUDA_CHECK(cudaSetDevice(g->device));
    const char* base = static_cast<const char*>(all_handles);
    for (int p = 0; p < g->world; ++p) {
        if (p == g->rank) continue;
        cudaIpcMemHandle_t h[2];
        std::memcpy(h, base + size_t(p) * sizeof(h), sizeof(h));
        void* a = nullptr;
        void* b = nullptr;
        NB2_CUDA_CHECK(cudaIpcOpenMemHandle(&a, h[0], cudaIpcMemLazyEnablePeerAccess));
        NB2_CUDA_CHECK(cudaIpcOpenMemHandle(&b, h[1], cudaIpcMemLazyEnablePeerAccess));
        g->peer_recv[p] = static_cast<char*>(a);
        g->peer_flags[p] = static_cast<int*>(b);
    }
    NB2_CUDA_CHECK(cudaMemcpy(g->d_peer_flags, g->peer_flags.data(), size_t(g->world) * sizeof(int*), cudaMemcpyHostToDevice));
    if (prev >= 0 && prev != g->device) cudaSetDevice(prev);
    return NB2_OK;
}

// Copies `bytes` (<= bytes_per_rank) from `src` (device memory of this rank) into slot (sequence & 1), position `rank`, of EVERY
// rank's receive buffer, then publishes `sequence` (> 0, increasing) there.  Everything is enqueued on `cuda_stream`.
nb2_status nb2_peer_gather_push(nb2_peer_gather* g, const void* src, size_t bytes, int32_t sequence, void* cuda_stream) {
    if (!g || !src || bytes > g->bytes_per_rank || sequence <= 0) {
        set_error("nb2_peer_gather_push: invalid argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
    const size_t slot_off = size_t(sequence & 1) * size_t(g->world) * g->bytes_per_rank + size_t(g->rank) * g->bytes_per_rank;
    const int flag_index = (sequence & 1) * g->world + g->rank;
    for (int k = 0; k < g->world; ++k) {
        const int p = (g->rank + k) % g->world;  // start with the local copy, then round-robin: ranks do not all hit rank 0 first
        if (!g->peer_recv[p]) {
            set_error("nb2_peer_gather_push: nb2_peer_gather_connect has not been called");
            return NB2_ERR_INVALID_ARGUMENT;
        }
        NB2_CUDA_CHECK(cudaMemcpyAsync(g->peer_recv[p] + slot_off, src, bytes, cudaMemcpyDefault, s));
    }
    // The flag is published by a small kernel: publishing it with cuStreamWriteValue32 instead was not faster (0.7449 vs 0.7436 ms
    // per frame at N = 2, DESIGN.md section 6).
    peer_signal_kernel<<<1, 32, 0, s>>>(g->d_peer_flags, g->world, flag_index, sequence);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// Makes `cuda_stream` wait until the slices of ALL ranks for `sequence` have landed in this rank's buffer (slot sequence & 1).
nb2_status nb2_peer_gather_wait(nb2_peer_gather* g, int32_t sequence, void* cuda_stream) {
    if (!g || sequence <= 0) {
        set_error("nb2_peer_gather_wait: invalid argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t s = static_cast<cudaStream_t>(cuda_stream);
    const int* f = g->flags + (sequence & 1) * g->world;
    if (g->wait32) {
        for (int p = 0; p < g->world; ++p) {
            const CUresult r = g->wait32(s, reinterpret_cast<CUdeviceptr>(f + p), cuuint32_t(sequence), CU_STREAM_WAIT_VALUE_GEQ);
            if (r != CUDA_SUCCESS) {
                g->wait32 = nullptr;  // not supported on this device / driver: fall back to the polling kernel
                break;
            }
            if (p == g->world - 1) return NB2_OK;
        }
    }
    peer_wait_kernel<<<1, 32, 0, s>>>(f, g->world, sequence);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

void nb2_peer_gather_destroy(nb2_peer_gather* g) {
    if (!g) return;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(g->device);
    for (int p = 0; p < g->world; ++p) {
        if (p == g->rank) continue;
        if (g->peer_recv[p]) cudaIpcCloseMemHandle(g->peer_recv[p]);
        if (g->peer_flags[p]) cudaIpcCloseMemHandle(g->peer_flags[p]);
    }
    cudaFree(g->recv);
    cudaFree(g->flags);
    cudaFree(g->d_peer_flags);
    if (prev >= 0 && prev != g->device) cudaSetDevice(prev);
    delete g;
}

}  // extern "C"
