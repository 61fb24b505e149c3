// Owners of the CUDA resources the host code holds (capi.cu, ingest.cu): every allocation, stream and event belongs to one
// object whose destructor releases it.  An error thrown between two CUDA calls therefore leaks nothing, and a failed
// allocation leaves an empty owner behind, never a freed pointer or a stale capacity.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #call); \
    } while (0)

// library internals: shared by the objects of libdrprg_cuda.so, not exported from it
#pragma GCC visibility push(hidden)
namespace drprg {

inline double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

enum class Mem { device, pinned };

// cap elements of device (cudaMalloc) or pinned host (cudaMallocHost) memory
template <class T, Mem M>
struct CudaBuf {
    T* p = nullptr;
    size_t cap = 0;
    CudaBuf() = default;
    CudaBuf(CudaBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    CudaBuf& operator=(CudaBuf&& o) noexcept {
        if (this != &o) {
            release();
            p = std::exchange(o.p, nullptr);
            cap = std::exchange(o.cap, 0);
        }
        return *this;
    }
    ~CudaBuf() { release(); }
    // grow-only: keeps the buffer when n elements fit, else allocates `want` (>= n) elements afresh (contents are lost)
    void reserve(size_t n, size_t want) {
        if (n <= cap) return;
        release();
        void* q = nullptr;
        if (M == Mem::device) CK(cudaMalloc(&q, want * sizeof(T)));
        else CK(cudaMallocHost(&q, want * sizeof(T)));
        p = static_cast<T*>(q);
        cap = want;
    }
    void release() {
        if (p && M == Mem::device) cudaFree(p);
        if (p && M == Mem::pinned) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

template <class T>
struct DBuf : CudaBuf<T, Mem::device> {  // grow-only device workspace
    void ensure(size_t n) { this->reserve(n, n + n / 4 + 1024); }
    // exactly max(1, v.size()) elements holding v
    void assign(const std::vector<T>& v) {
        const size_t n = std::max<size_t>(1, v.size());
        this->release();
        this->reserve(n, n);
        if (!v.empty()) CK(cudaMemcpy(this->p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    }
};

template <class T>
struct PinnedBuf : CudaBuf<T, Mem::pinned> {  // grow-only pinned host buffer: async D2H into pageable memory would block the host
    size_t n = 0;
    void resize(size_t want) {
        n = 0;
        this->reserve(want, want + want / 4 + 256);
        n = want;
    }
    T* data() { return this->p; }
    size_t size() const { return n; }
    T* begin() { return this->p; }
    T* end() { return this->p + n; }
};

struct StreamDestroy {
    void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
};
struct EventDestroy {
    void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;

inline Stream new_stream() {  // non-blocking: does not synchronise with the legacy default stream
    cudaStream_t s = nullptr;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    return Stream(s);
}
inline Event new_event(unsigned flags) {
    cudaEvent_t e = nullptr;
    CK(cudaEventCreateWithFlags(&e, flags));
    return Event(e);
}

// freed batch buffers are parked here and reused by the next upload: cudaFree synchronises the device and
// cudaMalloc costs ~0.1-1 ms, both of which would sit inside every end-to-end step
struct DevPool {
    struct Slot { void* p; size_t bytes; int device; };
    std::vector<Slot> free_;
    std::mutex m_;
    void* get(size_t bytes, int device) {
        std::lock_guard<std::mutex> g(m_);
        size_t best = free_.size();
        for (size_t i = 0; i < free_.size(); ++i)
            if (free_[i].device == device && free_[i].bytes >= bytes && (best == free_.size() || free_[i].bytes < free_[best].bytes)) best = i;
        if (best != free_.size() && free_[best].bytes <= bytes * 2 + (1 << 20)) {
            void* p = free_[best].p;
            free_.erase(free_.begin() + best);
            return p;
        }
        void* p = nullptr;
        CK(cudaMalloc(&p, bytes));
        return p;
    }
    void put(void* p, size_t bytes, int device) {
        std::lock_guard<std::mutex> g(m_);
        if (free_.size() >= 16) {
            cudaFree(free_.front().p);
            free_.erase(free_.begin());
        }
        free_.push_back({p, bytes, device});
    }
};
// never destroyed: static teardown may run after the CUDA runtime has been unloaded
inline DevPool& g_pool = *new DevPool;

struct PoolReturn {  // deleter of a PoolBuf: the buffer goes back to g_pool
    size_t bytes = 0;
    int device = -1;
    void operator()(void* p) const { g_pool.put(p, bytes, device); }
};
template <class T>
using PoolBuf = std::unique_ptr<T, PoolReturn>;
template <class T>
PoolBuf<T> pool_get(size_t bytes, int device) {
    return PoolBuf<T>(static_cast<T*>(g_pool.get(bytes, device)), PoolReturn{bytes, device});
}

}  // namespace drprg
#pragma GCC visibility pop
