// Owners of the library's CUDA resources (host C++): device memory, pinned host memory, events and owned streams.
// A handle's buffers are replaced only after all their allocations have succeeded: new buffers go into locals first, a
// failure releases the locals and leaves the handle as it was.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <memory>
#include <utility>

namespace hbd {

struct DevFree { void operator()(void* p) const { cudaFree(p); } };
struct HostFree { void operator()(void* p) const { cudaFreeHost(p); } };
struct EventFree { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
struct StreamFree { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };

template <typename T> using DevPtr = std::unique_ptr<T, DevFree>;
template <typename T> using HostPtr = std::unique_ptr<T, HostFree>;
using Event = std::unique_ptr<CUevent_st, EventFree>;
using Stream = std::unique_ptr<CUstream_st, StreamFree>;

// Each of these fills `out` on success and leaves it untouched on failure.  Allocations hold at least one element.  A
// refused allocation is returned here and cleared from the runtime's last error, so that the launch check of the next
// kernel (cudaGetLastError) does not report it a second time.
template <typename T> cudaError_t dev_alloc(DevPtr<T>& out, size_t count)
{
    void* p = nullptr;
    const cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) out.reset(static_cast<T*>(p)); else cudaGetLastError();
    return e;
}
template <typename T> cudaError_t host_alloc(HostPtr<T>& out, size_t count)
{
    void* p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, std::max<size_t>(count, 1) * sizeof(T), cudaHostAllocDefault);
    if (e == cudaSuccess) out.reset(static_cast<T*>(p)); else cudaGetLastError();
    return e;
}
inline cudaError_t event_create(Event& out, unsigned flags = cudaEventDisableTiming)
{
    cudaEvent_t ev = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&ev, flags);
    if (e == cudaSuccess) out.reset(ev);
    return e;
}
inline cudaError_t stream_create(Stream& out, int priority = 0)
{
    cudaStream_t s = nullptr;
    const cudaError_t e = cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, priority);
    if (e == cudaSuccess) out.reset(s);
    return e;
}

// K device matrices [rows][pitch] of T under one pitch (K = 2: the two halves of a ping-pong pair)
template <typename T, int K = 1> struct Rows {
    DevPtr<T> p[K];
    size_t pitch = 0;
    T* get(int i = 0) const { return p[i].get(); }

    // Enqueue the next generation into `next`: [rows][new_pitch], zeroed, the first `keep` elements of every row copied
    // from this one.  `next` stays empty when this one is already wide enough.  The caller synchronises `s`, then commits.
    cudaError_t regrow(Rows& next, size_t new_pitch, size_t rows, size_t keep, cudaStream_t s) const
    {
        if (new_pitch <= pitch && p[0]) return cudaSuccess;
        for (int i = 0; i < K; ++i) {
            cudaError_t e = dev_alloc(next.p[i], rows * new_pitch);
            if (e == cudaSuccess) e = cudaMemsetAsync(next.get(i), 0, rows * new_pitch * sizeof(T), s);
            if (e == cudaSuccess && p[i] && keep)
                e = cudaMemcpy2DAsync(next.get(i), new_pitch * sizeof(T), get(i), pitch * sizeof(T), std::min(keep, pitch) * sizeof(T), rows,
                                      cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) return e;
        }
        next.pitch = new_pitch;
        return cudaSuccess;
    }
    void commit(Rows& next) { if (next.p[0]) *this = std::move(next); }
    // regrow, synchronise, commit; changes nothing on failure
    cudaError_t grow(size_t new_pitch, size_t rows, size_t keep, cudaStream_t s)
    {
        Rows next;
        cudaError_t e = regrow(next, new_pitch, rows, keep, s);
        if (e == cudaSuccess && next.p[0]) e = cudaStreamSynchronize(s);
        if (e == cudaSuccess) commit(next);
        return e;
    }
};

} // namespace hbd
