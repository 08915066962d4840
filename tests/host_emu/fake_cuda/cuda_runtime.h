// A stand-in for the CUDA runtime's allocator so that host code owning device memory (csrc/rt_devbuf.h) compiles with g++ and its
// ownership rules can be checked on the CPU (test infrastructure only). It records every live block with its size, counts
// allocations and frees, fails the n-th cudaMalloc on request and keeps a last error that cudaGetLastError reads and clears.
#pragma once
#include <cstddef>
#include <cstdlib>
#include <map>

enum cudaError_t { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2 };

namespace fake_cuda {
inline long mallocs = 0, frees = 0, bad_frees = 0;   // bad_frees: pointers that were not live (double or foreign frees)
inline long fail_in = 0;                             // > 0: the fail_in-th cudaMalloc from now fails
inline cudaError_t last_error = cudaSuccess;
inline std::map<void*, size_t> live;                 // block -> bytes

inline void reset() {
    for (auto& b : live) std::free(b.first);
    live.clear();
    mallocs = frees = bad_frees = fail_in = 0;
    last_error = cudaSuccess;
}
inline size_t bytes_of(const void* p) {
    auto it = live.find(const_cast<void*>(p));
    return it == live.end() ? 0 : it->second;
}
}  // namespace fake_cuda

inline cudaError_t cudaMalloc(void** p, size_t bytes) {
    if (fake_cuda::fail_in > 0 && --fake_cuda::fail_in == 0) {
        *p = reinterpret_cast<void*>(0xdead0);           // the runtime promises nothing about *p after a failure
        fake_cuda::last_error = cudaErrorMemoryAllocation;
        return cudaErrorMemoryAllocation;
    }
    *p = std::malloc(bytes ? bytes : 1);
    ++fake_cuda::mallocs;
    fake_cuda::live[*p] = bytes;
    return cudaSuccess;
}

inline cudaError_t cudaFree(void* p) {
    if (!p) return cudaSuccess;
    if (!fake_cuda::live.erase(p)) { ++fake_cuda::bad_frees; return cudaErrorInvalidValue; }
    std::free(p);
    ++fake_cuda::frees;
    return cudaSuccess;
}

inline cudaError_t cudaGetLastError() {
    const cudaError_t e = fake_cuda::last_error;
    fake_cuda::last_error = cudaSuccess;
    return e;
}
