// v2p_hostres.cuh -- the host-side scaffolding every C ABI object of the library shares: buffers that own their
// memory, the error message of the last failed call, the CUDA-check macros, and the CUB scan the host code launches.
// Host code only; no kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <utility>

#include "v2p_engine.h"

namespace v2p {

// Grow-only buffer that owns its memory (freed by the destructor); need() does not keep the contents when it grows.
//   device:      at least 256 bytes, allocated with bytes/8 + 256 of slack, so kernels that read 16-byte vectors past
//                a logical end stay inside the allocation
//   pinned host: at least 4096 bytes, allocated with bytes/4 of slack, portable to every device
template <bool kPinned>
struct OwnedBuf {
    void* p = nullptr;
    size_t cap = 0;

    OwnedBuf() = default;
    OwnedBuf(const OwnedBuf&) = delete;
    OwnedBuf& operator=(const OwnedBuf&) = delete;
    OwnedBuf(OwnedBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    OwnedBuf& operator=(OwnedBuf&& o) noexcept {
        std::swap(p, o.p), std::swap(cap, o.cap);
        return *this;
    }
    ~OwnedBuf() {
        if (p) dealloc(p);
    }

    cudaError_t need(size_t bytes) {
        bytes = std::max<size_t>(bytes, kPinned ? 4096 : 256);
        if (cap >= bytes) return cudaSuccess;
        if (p) {
            const cudaError_t st = dealloc(p);
            if (st != cudaSuccess) return st;
            p = nullptr, cap = 0;
        }
        const size_t want = kPinned ? bytes + bytes / 4 : bytes + bytes / 8 + 256;
        const cudaError_t st = kPinned ? cudaHostAlloc(&p, want, cudaHostAllocPortable) : cudaMalloc(&p, want);
        if (st != cudaSuccess) return p = nullptr, st;
        cap = want;
        return cudaSuccess;
    }

private:
    static cudaError_t dealloc(void* q) { return kPinned ? cudaFreeHost(q) : cudaFree(q); }
};
using DevBuf = OwnedBuf<false>;
using PinnedBuf = OwnedBuf<true>;

// b.need(bytes + 16), then `bytes` from the host on stream s (the 16 bytes past the end are for 16-byte vector loads)
inline cudaError_t upload(DevBuf& b, const void* h, size_t bytes, cudaStream_t s) {
    cudaError_t st = b.need(bytes + 16);
    if (st == cudaSuccess && bytes) st = cudaMemcpyAsync(b.p, h, bytes, cudaMemcpyHostToDevice, s);
    return st;
}

// printf-style formatting into a string of whatever length the message takes
inline std::string vformat(const char* fmt, va_list ap) {
    va_list ap2;
    va_copy(ap2, ap);
    const int n = vsnprintf(nullptr, 0, fmt, ap2);
    va_end(ap2);
    if (n <= 0) return std::string();
    std::string s((size_t)n, '\0');
    vsnprintf(&s[0], (size_t)n + 1, fmt, ap);
    return s;
}

// the message of a failed call into its object's error string; returns the status code
inline int fail(std::string& dst, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    dst = vformat(fmt, ap);
    va_end(ap);
    return code;
}

}  // namespace v2p

// return V2P_ERR_CUDA from the enclosing function when `call` does not return cudaSuccess, with the message in `dst`
#define CU(dst, call)                                                                                                  \
    do {                                                                                                               \
        const cudaError_t _st = (call);                                                                                \
        if (_st != cudaSuccess)                                                                                        \
            return ::v2p::fail((dst), V2P_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), __FILE__, \
                               __LINE__);                                                                              \
    } while (0)

// the same inside a loop that must not return (the pipeline's chunk loop, whose drain must still wait for every copy in
// flight): the status goes to `rc` and the loop is left
#define CU_BREAK(dst, rc, call)                                                                                      \
    {                                                                                                                \
        const cudaError_t _st = (call);                                                                              \
        if (_st != cudaSuccess) {                                                                                    \
            (rc) = ::v2p::fail((dst), V2P_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), __FILE__, \
                               __LINE__);                                                                            \
            break;                                                                                                   \
        }                                                                                                            \
    }

namespace v2p {

inline unsigned blocks(uint64_t n) { return (unsigned)((n + 255) / 256); }  // 256-thread blocks over n items

// CUB exclusive sum of n items on stream s; `tmp` is its grow-only scratch.  In and Out reach CUB unchanged: each pair
// of iterator types instantiates scan kernels of its own.  Defined only in files that include CUB before this header:
// any CUB header adds a kernel (cub::EmptyKernel) to a file's device code, so this header does not include one.
#ifdef CUB_VERSION
template <class In, class Out>
int exclusive_sum(std::string& err, DevBuf& tmp, In in, Out out, uint64_t n, cudaStream_t s) {
    size_t bytes = 0;
    CU(err, cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, (int64_t)n, s));
    CU(err, tmp.need(bytes));
    CU(err, cub::DeviceScan::ExclusiveSum(tmp.p, bytes, in, out, (int64_t)n, s));
    return V2P_OK;
}
#endif

}  // namespace v2p
