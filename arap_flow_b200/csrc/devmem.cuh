// devmem.cuh -- who owns host-side device memory (DESIGN.md 4.7): DevBuf, one exact-size device array; GrowBuf, one
// grow-only block of device or pinned host memory; Workspace, a GrowBuf per device shared by the stand-alone calls;
// Layout, the 256-byte-aligned carve of one block into many.  And guarded, which turns a failure into a return code.
//
// Layout is plain integer arithmetic and compiles without CUDA (tests/devmem_host.cpp); the rest needs nvcc.
#pragma once
#include <cstddef>

namespace arapb200 {

// Blocks of one buffer, each starting on a 256-byte boundary: take(bytes) returns the next block's offset and bytes()
// the total so far.  One description of the blocks both sizes the buffer and places the pointers in it.  A block of 0
// bytes takes no space.
class Layout {
public:
    size_t take(size_t bytes)
    {
        const size_t at = end_;
        end_ += (bytes + 255) & ~(size_t)255;
        return at;
    }
    size_t bytes() const { return end_; }

private:
    size_t end_ = 0;
};

} // namespace arapb200

#ifdef __CUDACC__
#include "common.cuh"
#include <exception>
#include <mutex>
#include <utility>

namespace arapb200 {

// count elements of device memory (at least one, so that p is never null), freed by the destructor
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    explicit DevBuf(size_t count) : n(count) { ARAP_CUDA_CHECK(cudaMalloc(&p, (count ? count : 1) * sizeof(T))); }
    ~DevBuf()
    {
        if (p) cudaFree(p);
    }
    DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
    DevBuf& operator=(DevBuf&& o) noexcept
    {
        std::swap(p, o.p);
        std::swap(n, o.n);
        return *this;
    }
    void up(const T* h, cudaStream_t s = nullptr)
    {
        ARAP_CUDA_CHECK(cudaMemcpyAsync(p, h, n * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void down(T* h, cudaStream_t s = nullptr)
    {
        ARAP_CUDA_CHECK(cudaMemcpyAsync(h, p, n * sizeof(T), cudaMemcpyDeviceToHost, s));
    }
};

// A block of device (cudaMalloc) or pinned host (cudaMallocHost) memory that only grows.  reserve() keeps the block
// when it is large enough; otherwise it frees it and leaves the buffer empty (null, capacity 0) before it allocates, so
// a failed allocation throws with nothing stale behind it.
class GrowBuf {
public:
    enum Kind { Device, Pinned };
    explicit GrowBuf(Kind kind = Device) : kind_(kind) {}
    ~GrowBuf() { release(); }
    GrowBuf(GrowBuf&& o) noexcept
        : kind_(o.kind_), p_(std::exchange(o.p_, nullptr)), cap_(std::exchange(o.cap_, 0)) {}
    GrowBuf& operator=(GrowBuf&& o) noexcept
    {
        std::swap(kind_, o.kind_);
        std::swap(p_, o.p_);
        std::swap(cap_, o.cap_);
        return *this;
    }
    unsigned char* reserve(size_t bytes)
    {
        if (bytes > cap_) {
            ARAP_CUDA_CHECK(release());
            void* q = nullptr;
            ARAP_CUDA_CHECK(kind_ == Pinned ? cudaMallocHost(&q, bytes) : cudaMalloc(&q, bytes));
            p_ = (unsigned char*)q;
            cap_ = bytes;
        }
        return p_;
    }
    unsigned char* data() const { return p_; }
    size_t capacity() const { return cap_; }

private:
    cudaError_t release()
    {
        void* q = std::exchange(p_, nullptr);
        cap_ = 0;
        if (!q) return cudaSuccess;
        return kind_ == Pinned ? cudaFreeHost(q) : cudaFree(q);
    }
    Kind kind_;
    unsigned char* p_ = nullptr;
    size_t cap_ = 0;
};

// Device workspace of a stand-alone call, kept for the life of the process: a cudaMalloc / cudaFree per call costs more
// than the kernels, and cudaFree synchronises the device.  A caller holds mu until its last copy out of buf has
// returned.  stream: a non-blocking stream of the workspace's own, for a caller that creates and uses one.
struct Workspace {
    std::mutex mu;
    GrowBuf buf;
    cudaStream_t stream = nullptr;
};

// One Workspace per device ordinal, created on first use and never freed: it outlives the CUDA context teardown at
// exit.
class WorkspaceTable {
public:
    Workspace& current()
    {
        int dev = 0;
        ARAP_CUDA_CHECK(cudaGetDevice(&dev));
        if (dev < 0 || dev >= kMaxDevices) arap_fail(1, "device ordinal %d out of range", dev);
        std::lock_guard<std::mutex> g(mu_);
        if (!table_[dev]) table_[dev] = new Workspace;
        return *table_[dev];
    }

private:
    static constexpr int kMaxDevices = 64;
    std::mutex mu_;
    Workspace* table_[kMaxDevices] = {};
};

// every extern "C" entry point runs its body through this: an ArapError (CUDA failure, watchdog, capacity) becomes the
// function's non-zero return code instead of taking the host process down
template <class F>
int guarded(F&& f)
{
    try {
        return f();
    } catch (const ArapError& e) {
        return e.code;
    } catch (const std::exception& e) {
        fprintf(stderr, "arapb200: %s\n", e.what());
        return 2;
    } catch (...) {
        return 2;
    }
}

} // namespace arapb200
#endif
