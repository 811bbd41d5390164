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

// The argument check of every batched entry point on device samples, in one order: a null plan, offsets or required output
// (`args_ok` false) or a negative count -> DSPFE_ERR_INVALID_ARG; a plan that cannot run this entry point (`unsupported`, the
// message, or null) -> DSPFE_ERR_UNSUPPORTED; an empty batch -> DSPFE_OK, and the caller returns before it queues anything;
// null samples with total_samples > 0, or samples not 16-byte aligned -> DSPFE_ERR_INVALID_ARG.
inline int check_batch(bool args_ok, int64_t n_utt, int64_t total_samples, const void* d_pcm, const char* unsupported = nullptr) {
    if (!args_ok || n_utt < 0 || total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (unsupported) return fail(DSPFE_ERR_UNSUPPORTED, unsupported);
    if (n_utt == 0) return DSPFE_OK;
    if (!d_pcm && total_samples > 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm is null");
    if (((uintptr_t)d_pcm & 15) != 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm must be 16-byte aligned");
    return DSPFE_OK;
}

// The same for the host-buffer forms: bad arguments, then `unsupported`, then every offset of the batch non-decreasing
// (h_offsets[0 .. n_utt]); DSPFE_OK for an empty batch.
inline int check_host_batch(bool args_ok, const int64_t* h_offsets, int32_t n_utt, const char* unsupported = nullptr) {
    if (!args_ok || !h_offsets || n_utt < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (unsupported) return fail(DSPFE_ERR_UNSUPPORTED, unsupported);
    for (int32_t u = 0; u < n_utt; ++u)
        if (h_offsets[u + 1] < h_offsets[u]) return fail(DSPFE_ERR_INVALID_ARG, "offsets must be non-decreasing");
    return DSPFE_OK;
}
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

// The staging of a plan's host-buffer forms: a stream, and on the device the samples of a host batch from h_offsets[0] on
// and the offsets relative to the first.
class HostBatch : NoCopy {
public:
    // Copies the batch on the stream.  frames(u, len) is the frame count of utterance u of len samples: their prefix sums go
    // to h_frame_off (optional, [n_utt + 1]), and *total / *n_frames receive the batch's samples and frames.
    template <class Frames>
    int stage(const void* h_pcm, int64_t esz, const int64_t* h_offsets, int32_t n_utt, Frames frames, int64_t* h_frame_off,
              int64_t* total, int64_t* n_frames) {
        const int64_t base = h_offsets[0];
        *total = h_offsets[n_utt] - base;
        CUDA_TRY(stream_.ensure());
        int rc = pcm_.reserve((*total + 8) * esz);
        if (!rc) rc = off_.reserve(n_utt + 1);
        if (rc) return rc;
        std::vector<int64_t> rel(n_utt + 1);
        int64_t f = 0;
        for (int32_t u = 0; u < n_utt; ++u) {
            rel[u] = h_offsets[u] - base;
            if (h_frame_off) h_frame_off[u] = f;
            f += frames(u, h_offsets[u + 1] - h_offsets[u]);
        }
        rel[n_utt] = *total;
        if (h_frame_off) h_frame_off[n_utt] = f;
        *n_frames = f;
        const cudaStream_t st = stream_.get();
        if (*total > 0) CUDA_TRY(cudaMemcpyAsync(pcm_.get(), (const char*)h_pcm + base * esz, *total * esz, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(off_.get(), rel.data(), (n_utt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        return DSPFE_OK;
    }
    cudaStream_t stream() const { return stream_.get(); }
    template <class T = void> const T* pcm() const { return reinterpret_cast<const T*>(pcm_.get()); }
    const int64_t* offsets() const { return off_.get(); }
private:
    Stream stream_;
    DeviceArray<unsigned char> pcm_;
    DeviceArray<int64_t> off_;
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
