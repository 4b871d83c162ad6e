// TEST INFRASTRUCTURE — armour_b200/csrc/device_buffer.h compiled with g++ against stand-ins of cudaMalloc / cudaFree that
// count the live allocations and can be told to fail.  Built and driven by tests/test_device_buffer.py; never part of the
// product.
#include <cstddef>
#include <cstdlib>
#include <set>
#include <utility>

enum cudaError_t { cudaSuccess = 0, cudaErrorMemoryAllocation = 2 };

namespace {
std::set<void*> g_live;
long g_mallocs = 0, g_frees = 0, g_bad_frees = 0;
size_t g_last_bytes = 0;
int g_fail = 0;  // the next g_fail allocations fail
}  // namespace

cudaError_t cudaMalloc(void** p, size_t bytes) {
    if (g_fail > 0) {
        g_fail--;
        *p = reinterpret_cast<void*>(0x10);  // what the runtime leaves in *p on failure is not specified
        return cudaErrorMemoryAllocation;
    }
    *p = std::malloc(bytes ? bytes : 1);
    g_live.insert(*p);
    g_mallocs++;
    g_last_bytes = bytes;
    return cudaSuccess;
}

cudaError_t cudaFree(void* p) {
    g_frees++;
    if (g_live.erase(p) == 0) {  // not a live allocation: a second free, or a pointer that was never allocated
        g_bad_frees++;
        return cudaSuccess;
    }
    std::free(p);
    return cudaSuccess;
}

#include "../../armour_b200/csrc/device_buffer.h"

using Buf = armour::DeviceBuffer<double>;

extern "C" {
Buf* buf_new() { return new Buf; }
void buf_delete(Buf* b) { delete b; }
int buf_reserve(Buf* b, size_t n) { return b->reserve(n); }
size_t buf_capacity(const Buf* b) { return b->capacity(); }
void* buf_get(const Buf* b) { return b->get(); }
Buf* buf_move_new(Buf* src) { return new Buf(std::move(*src)); }
void buf_move_assign(Buf* dst, Buf* src) { *dst = std::move(*src); }

void stub_fail_next(int n) { g_fail = n; }
long stub_live() { return long(g_live.size()); }
long stub_mallocs() { return g_mallocs; }
long stub_frees() { return g_frees; }
long stub_bad_frees() { return g_bad_frees; }
size_t stub_last_bytes() { return g_last_bytes; }
}
