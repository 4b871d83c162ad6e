// Owning handle of one device allocation, used for every device buffer of the C API's contexts: each buffer is freed
// exactly once, by its owner's destructor, and a failed allocation never leaves a capacity behind without memory.
// Like the kernel headers it relies on the CUDA runtime declarations (cudaMalloc, cudaFree, cudaError_t) being in scope;
// tests/test_device_buffer.py compiles it against stubs of them.
#pragma once
#include <cstddef>
#include <utility>

namespace armour {

template <class T>
class DeviceBuffer {  // move-only
  public:
    DeviceBuffer() = default;
    DeviceBuffer(DeviceBuffer&& o) noexcept : p_(std::exchange(o.p_, nullptr)), n_(std::exchange(o.n_, 0)) {}
    DeviceBuffer& operator=(DeviceBuffer&& o) noexcept {
        if (this != &o) {
            release();
            p_ = std::exchange(o.p_, nullptr);
            n_ = std::exchange(o.n_, 0);
        }
        return *this;
    }
    ~DeviceBuffer() { release(); }

    T* get() const { return p_; }
    size_t capacity() const { return n_; }  // elements

    // At least n elements.  Grows only, and does not keep the contents when it grows: the old allocation is freed, then n
    // elements are allocated.  On failure the buffer is empty (null, capacity 0), so the next reserve allocates.
    cudaError_t reserve(size_t n) {
        if (n <= n_) return cudaSuccess;
        release();
        void* p = nullptr;
        const cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e != cudaSuccess) return e;
        p_ = static_cast<T*>(p);
        n_ = n;
        return cudaSuccess;
    }

  private:
    void release() {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
    }
    T* p_ = nullptr;
    size_t n_ = 0;
};

}  // namespace armour
