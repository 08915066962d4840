// Host build of csrc/rt_devbuf.h against the fake CUDA allocator in fake_cuda/cuda_runtime.h (test infrastructure only). Each
// check returns 0 when it holds, else the line of the first failed condition.
#include <cuda_runtime.h>

#include <utility>

#include "../../software-raytracer_b200/csrc/rt_devbuf.h"

using namespace rtb;
using namespace fake_cuda;

#define CHECK(cond) do { if (!(cond)) return __LINE__; } while (0)

namespace {
struct Rec { float v[7]; };   // an element size that is neither a power of two nor a multiple of 4 words
}

extern "C" {

// a reserve within capacity keeps the allocation; a new one holds exactly n elements, no headroom
int devbuf_reserve_within_capacity() {
    reset();
    {
        DeviceArray<Rec> a;
        CHECK(a.get() == nullptr && a.capacity() == 0);
        CHECK(a.reserve(0) == cudaSuccess && a.get() == nullptr && mallocs == 0);
        CHECK(a.reserve(100) == cudaSuccess && a.get() != nullptr && a.capacity() == 100);
        CHECK(bytes_of(a.get()) == 100 * sizeof(Rec));
        Rec* p = a.get();
        CHECK(a.reserve(100) == cudaSuccess && a.get() == p && a.capacity() == 100);
        CHECK(a.reserve(1) == cudaSuccess && a.get() == p && a.capacity() == 100);
        CHECK(a.reserve(0) == cudaSuccess && a.get() == p);
        CHECK(mallocs == 1 && frees == 0);
    }
    CHECK(mallocs == 1 && frees == 1 && bad_frees == 0 && live.empty());
    return 0;
}

// growth frees the old block exactly once, before the new one is allocated
int devbuf_growth_frees_old_once() {
    reset();
    DeviceArray<int> a;
    CHECK(a.reserve(8) == cudaSuccess);
    void* old = a.get();
    CHECK(a.reserve(9) == cudaSuccess && a.capacity() == 9 && bytes_of(a.get()) == 9 * sizeof(int));
    CHECK(mallocs == 2 && frees == 1 && bad_frees == 0);
    CHECK(live.size() == 1 && live.count(a.get()) == 1 && (a.get() == old || live.count(old) == 0));
    a.reset();
    CHECK(a.get() == nullptr && a.capacity() == 0 && frees == 2 && live.empty());
    a.reset();
    CHECK(frees == 2 && bad_frees == 0);
    return 0;
}

// a failed reserve leaves the array empty, the old block freed and the last error cleared; the array stays usable
int devbuf_failed_reserve_leaves_empty() {
    reset();
    DeviceArray<double> a;
    CHECK(a.reserve(4) == cudaSuccess);
    fail_in = 1;
    CHECK(a.reserve(100) == cudaErrorMemoryAllocation);
    CHECK(a.get() == nullptr && a.capacity() == 0);
    CHECK(cudaGetLastError() == cudaSuccess);
    CHECK(frees == 1 && live.empty());
    fail_in = 1;
    CHECK(a.reserve(1) == cudaErrorMemoryAllocation && a.get() == nullptr && cudaGetLastError() == cudaSuccess);
    CHECK(a.reserve(100) == cudaSuccess && a.capacity() == 100 && live.size() == 1);
    return 0;
}

// a move leaves the source empty; a move assignment frees what the target held
int devbuf_move_leaves_source_empty() {
    reset();
    DeviceArray<int> a;
    CHECK(a.reserve(5) == cudaSuccess);
    int* p = a.get();
    DeviceArray<int> b(std::move(a));
    CHECK(a.get() == nullptr && a.capacity() == 0 && b.get() == p && b.capacity() == 5);
    DeviceArray<int> c;
    CHECK(c.reserve(3) == cudaSuccess);
    void* q = c.get();
    c = std::move(b);
    CHECK(b.get() == nullptr && b.capacity() == 0 && c.get() == p && c.capacity() == 5);
    CHECK(frees == 1 && live.count(q) == 0 && live.size() == 1);
    a.reset(); b.reset();
    CHECK(frees == 1 && bad_frees == 0);
    return 0;
}

// a grouped allocation that fails at any member leaves none of the group allocated, also when the group held smaller blocks
int devbuf_group_all_or_nothing() {
    for (int k = 1; k <= 3; ++k) {
        for (int held = 0; held < 2; ++held) {
            reset();
            DeviceArray<float> a, b; DeviceArray<int> c;
            if (held) CHECK(reserve_all(4, a, b, c) == cudaSuccess && live.size() == 3);
            fail_in = k;
            CHECK(reserve_all(10, a, b, c) == cudaErrorMemoryAllocation);
            CHECK(a.get() == nullptr && b.get() == nullptr && c.get() == nullptr);
            CHECK(a.capacity() == 0 && b.capacity() == 0 && c.capacity() == 0);
            CHECK(live.empty() && bad_frees == 0 && cudaGetLastError() == cudaSuccess);
            CHECK(mallocs == frees);
        }
    }
    reset();
    DeviceArray<float> a, b; DeviceArray<int> c;
    CHECK(reserve_all(10, a, b, c) == cudaSuccess && mallocs == 3);
    CHECK(bytes_of(a.get()) == 40 && bytes_of(b.get()) == 40 && bytes_of(c.get()) == 40);
    CHECK(reserve_all(10, a, b, c) == cudaSuccess && mallocs == 3 && frees == 0);
    return 0;
}

// every allocation is freed exactly once by the time the arrays are destroyed, whatever happened to them before
int devbuf_everything_freed_once() {
    reset();
    {
        DeviceArray<int> a, b[2];
        DeviceArray<Rec> r;
        CHECK(a.reserve(3) == cudaSuccess && a.reserve(30) == cudaSuccess);
        CHECK(reserve_all(7, b[0], b[1], r) == cudaSuccess);
        fail_in = 2;
        CHECK(reserve_all(70, b[0], b[1], r) == cudaErrorMemoryAllocation);
        CHECK(reserve_all(70, b[0], b[1]) == cudaSuccess);
        DeviceArray<int> m(std::move(a));
        a = std::move(m);
        m = std::move(b[1]);
        CHECK(r.reserve(1) == cudaSuccess);
    }
    CHECK(mallocs > 0 && mallocs == frees && bad_frees == 0 && live.empty());
    return 0;
}

}  // extern "C"
