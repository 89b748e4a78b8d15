// scan3d_device_buffer.h -- the one owner of the context's device memory (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace s3d {

// n elements of device memory, owned: not copyable, movable and std::swap-able with the capacity travelling with the
// pointer, freed by the destructor.  ensure(n) grows it, never shrinks it, and does not keep the contents: every
// buffer grown this way is scratch or an output.
template <class T>
class DeviceBuffer {
public:
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    DeviceBuffer(DeviceBuffer&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DeviceBuffer& operator=(DeviceBuffer&& o) noexcept
    {
        if (this != &o) {
            release();
            p_ = o.p_; n_ = o.n_;
            o.p_ = nullptr; o.n_ = 0;
        }
        return *this;
    }
    ~DeviceBuffer() { release(); }

    // at least n elements: nothing when it holds them, else the old memory is freed before the new is allocated;
    // after a failure the buffer is empty
    cudaError_t ensure(size_t n)
    {
        if (n <= n_) return cudaSuccess;
        release();
        const cudaError_t e = cudaMalloc((void**)&p_, n * sizeof(T));
        if (e != cudaSuccess) { p_ = nullptr; return e; }
        n_ = n;
        return cudaSuccess;
    }
    void release()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
    }
    size_t size() const { return n_; }
    T* get() const { return p_; }
    operator T*() const { return p_; }

private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

// One member of grow_group: a buffer and the elements it must hold.
template <class T>
struct Grow {
    Grow(DeviceBuffer<T>& b, size_t count) : buf(b), n(count) {}
    DeviceBuffer<T>& buf;
    size_t n;
};

// Buffers sized together grow as one group: every member too small for its count is released before any is
// allocated, so the group never holds its old and its new memory at once.  Stops at the first failure.
template <class... T>
cudaError_t grow_group(Grow<T>... m)
{
    ((m.buf.size() < m.n ? m.buf.release() : void()), ...);
    cudaError_t e = cudaSuccess;
    (void)(((e = m.buf.ensure(m.n)) == cudaSuccess) && ...);
    return e;
}

}  // namespace s3d
