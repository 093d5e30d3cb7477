// v2p_mapped.cuh -- small device -> host hand-offs (totals, status blocks, per-file offsets) WITHOUT the copy engine.
//
// While a chunk's result tape streams back over PCIe (a ~1 GB cudaMemcpyAsync), every other D2H copy -- even 8 bytes --
// queues behind it on the device-to-host copy engine, which serialises the next chunk's kernels with the copy-back
// (measured: 20 chunks x 19 ms of "generation" that is 1 ms of kernels).  These helpers publish small results with a
// one-warp kernel that stores straight into mapped pinned host memory (posted PCIe writes from the SM), so the host
// only waits for the stream the kernels run on.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

namespace v2p {

struct PubList {
    const unsigned long long* src[8];
    int n;
};

// dst[i] = *src[i]  (scattered 8-byte scalars)
static __global__ void k_publish_list(unsigned long long* __restrict__ dst, PubList l) {
    if ((int)threadIdx.x < l.n) dst[threadIdx.x] = *l.src[threadIdx.x];
    __threadfence_system();
}

// dst[0..n) = src[0..n)  (a small array of 8-byte words)
static __global__ void k_publish_words(unsigned long long* __restrict__ dst, const unsigned long long* __restrict__ src, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[i];
    __threadfence_system();
}

// pinned + mapped host scratch, freed by the destructor; under unified addressing the device uses the same pointer
struct MappedBuf {
    unsigned long long* p = nullptr;
    size_t words = 0;

    MappedBuf() = default;
    MappedBuf(const MappedBuf&) = delete;
    MappedBuf& operator=(const MappedBuf&) = delete;
    MappedBuf(MappedBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), words(std::exchange(o.words, 0)) {}
    MappedBuf& operator=(MappedBuf&& o) noexcept {
        std::swap(p, o.p), std::swap(words, o.words);
        return *this;
    }
    ~MappedBuf() {
        if (p) cudaFreeHost(p);
    }

    cudaError_t reserve(size_t n) {
        n = n < 64 ? 64 : n;
        if (words >= n) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr, words = 0;
        cudaError_t st = cudaHostAlloc((void**)&p, (n + n / 4) * 8, cudaHostAllocMapped | cudaHostAllocPortable);
        if (st == cudaSuccess) words = n + n / 4;
        return st;
    }
};

inline cudaError_t publish_words(unsigned long long* dst_mapped, const void* src_dev, uint64_t n, cudaStream_t s) {
    if (!n) return cudaSuccess;
    const unsigned grid = (unsigned)((n + 255) / 256 > 64 ? 64 : (n + 255) / 256);
    k_publish_words<<<grid, 256, 0, s>>>(dst_mapped, (const unsigned long long*)src_dev, n);
    return cudaGetLastError();
}

}  // namespace v2p
