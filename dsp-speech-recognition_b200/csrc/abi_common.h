// Shared plumbing of the C-ABI translation units (error reporting, CUDA call checking, owners of CUDA resources).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/dspfe.h"

namespace dspfe {
inline thread_local std::string g_err;
inline int fail(int code, const std::string& msg) { g_err = msg; return code; }
}  // namespace dspfe

// After a kernel launch: always check the launch status; with DSPFE_DEBUG_SYNC=1 in the environment also wait for
// the kernel and name it if it faulted (debug aid, off by default: the entry points never synchronise).
namespace dspfe {
inline bool debug_sync() { static const bool v = [] { const char* e = getenv("DSPFE_DEBUG_SYNC"); return e && e[0] == '1'; }(); return v; }
}
// Optional per-kernel timing (dspfe_timing_begin / dspfe_timing_end, include/dspfe.h): while a collection is open on a
// stream, every kernel the library launches on that stream is followed by an event; a kernel's time is the distance
// between its event and the previous one (launches on one stream are serial).  Off by default: one predictable branch.
namespace dspfe {
struct StageTimer {
    bool on = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t start = nullptr;
    std::vector<std::pair<const char*, cudaEvent_t>> marks;
    long long launches = 0;          // every LAUNCH_CHECK since the library was loaded (for reports)
    cudaError_t ensure_start() { return start ? cudaSuccess : cudaEventCreate(&start); }
    void clear_marks() { for (auto& m : marks) cudaEventDestroy(m.second); marks.clear(); }
};
inline StageTimer g_timer;
inline void timer_mark(const char* name, cudaStream_t st) {
    ++g_timer.launches;
    if (!g_timer.on || st != g_timer.stream) return;
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, st);
    g_timer.marks.emplace_back(name, e);
}
}  // namespace dspfe
#define LAUNCH_CHECK(name, stream)                                                                      \
    do {                                                                                                \
        ::dspfe::timer_mark(name, stream);                                                              \
        cudaError_t e_ = cudaGetLastError();                                                            \
        if (e_ == cudaSuccess && ::dspfe::debug_sync()) e_ = cudaStreamSynchronize(stream);             \
        if (e_ != cudaSuccess)                                                                          \
            return ::dspfe::fail(DSPFE_ERR_CUDA, std::string(name) + ": " + cudaGetErrorString(e_));    \
    } while (0)

#define CUDA_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t e_ = (expr);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return ::dspfe::fail(DSPFE_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));   \
    } while (0)

// Owners of the memory, streams and events the plans keep between calls.  Each releases its resource in its destructor,
// so `delete plan` frees a plan, or what a failed create had made so far.  Members are released in reverse order of
// declaration: a plan declares its streams and events before the buffers used on them.
namespace dspfe {

struct NoCopy {
    NoCopy() = default;
    NoCopy(const NoCopy&) = delete;
    NoCopy& operator=(const NoCopy&) = delete;
};

// Grow-only array of T in device memory (cudaMalloc) or pinned host memory (cudaHostAlloc).  reserve(n, floor) keeps the
// block when it holds n elements; otherwise it frees the block, whose contents are not kept, and allocates max(n, floor).
// cudaFree synchronises the device, so a block that queued work on another stream still uses is not freed under it.
template <class T, bool kPinned>
class Array : NoCopy {
public:
    ~Array() { release(); }
    int reserve(int64_t n, int64_t floor = 0) {
        if (n <= cap_) return DSPFE_OK;
        release();
        const int64_t m = std::max(n, floor);
        void* q = nullptr;
        const cudaError_t e = kPinned ? cudaHostAlloc(&q, m * sizeof(T), cudaHostAllocDefault) : cudaMalloc(&q, m * sizeof(T));
        if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string(kPinned ? "cudaHostAlloc: " : "cudaMalloc: ") + cudaGetErrorString(e));
        p_ = static_cast<T*>(q); cap_ = m;
        return DSPFE_OK;
    }
    T* get() const { return p_; }
    int64_t capacity() const { return cap_; }
private:
    void release() {
        if (p_) { if (kPinned) cudaFreeHost(p_); else cudaFree(p_); }
        p_ = nullptr; cap_ = 0;
    }
    T* p_ = nullptr;
    int64_t cap_ = 0;
};
template <class T> using DeviceArray = Array<T, false>;
template <class T> using PinnedArray = Array<T, true>;

// A non-blocking stream, created by the first ensure().
class Stream : NoCopy {
public:
    ~Stream() { if (s_) cudaStreamDestroy(s_); }
    cudaError_t ensure() { return s_ ? cudaSuccess : cudaStreamCreateWithFlags(&s_, cudaStreamNonBlocking); }
    cudaStream_t get() const { return s_; }
private:
    cudaStream_t s_ = nullptr;
};

// An event without timing (ordering only), created by the first ensure().
class Event : NoCopy {
public:
    ~Event() { if (e_) cudaEventDestroy(e_); }
    cudaError_t ensure() { return e_ ? cudaSuccess : cudaEventCreateWithFlags(&e_, cudaEventDisableTiming); }
    cudaEvent_t get() const { return e_; }
private:
    cudaEvent_t e_ = nullptr;
};

// A per-call temporary: alloc() takes it from the stream-ordered pool of `st`, and it goes back on the same stream when
// the owner leaves scope, on every return path.
template <class T>
class StreamTemp : NoCopy {
public:
    ~StreamTemp() { if (p_) cudaFreeAsync(p_, st_); }
    cudaError_t alloc(int64_t n, cudaStream_t st) {
        st_ = st;
        const cudaError_t e = cudaMallocAsync(&p_, n * sizeof(T), st);
        if (e != cudaSuccess) p_ = nullptr;
        return e;
    }
    T* get() const { return p_; }
private:
    T* p_ = nullptr;
    cudaStream_t st_ = nullptr;
};

}  // namespace dspfe
