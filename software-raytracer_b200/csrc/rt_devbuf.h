// rt_devbuf.h - DeviceArray<T>, the owner of every device buffer of a context (rt_ctx.h) and of the wavefront pipeline's state
// (rt_wavefront.cu): one cudaMalloc allocation of capacity() elements, freed when the array is reset, replaced or destroyed.
// Host code only; it includes nothing but the CUDA runtime so the ownership rules can be tested with g++ (tests/test_devbuf_cpu.py).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

namespace rtb {

template <typename T>
class DeviceArray {
public:
    DeviceArray() = default;
    DeviceArray(const DeviceArray&) = delete;
    DeviceArray& operator=(const DeviceArray&) = delete;
    DeviceArray(DeviceArray&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DeviceArray& operator=(DeviceArray&& o) noexcept {
        if (this != &o) { reset(); p_ = o.p_; n_ = o.n_; o.p_ = nullptr; o.n_ = 0; }
        return *this;
    }
    ~DeviceArray() { reset(); }

    T* get() const { return p_; }
    size_t capacity() const { return n_; }

    // Room for n elements: an allocation that has it is kept, else it is freed and exactly n elements are allocated. On failure the
    // array is empty and the thread's last error is cleared, so that the next launch check does not report the failed allocation.
    // Callers synchronise the stream first when kernels may still use the old allocation.
    cudaError_t reserve(size_t n) {
        if (n <= n_) return cudaSuccess;
        reset();
        const cudaError_t e = cudaMalloc((void**)&p_, n * sizeof(T));
        if (e != cudaSuccess) { p_ = nullptr; cudaGetLastError(); return e; }
        n_ = n;
        return cudaSuccess;
    }
    void reset() {
        if (p_) cudaFree(p_);
        p_ = nullptr; n_ = 0;
    }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

// n elements in every array of a group that is used together, or none: a failure leaves every array of the group empty
template <typename... A>
cudaError_t reserve_all(size_t n, A&... arrays) {
    cudaError_t e = cudaSuccess;
    ((e = e == cudaSuccess ? arrays.reserve(n) : e), ...);
    if (e != cudaSuccess) (arrays.reset(), ...);
    return e;
}

}  // namespace rtb
