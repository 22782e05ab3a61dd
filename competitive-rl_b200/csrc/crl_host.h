// crl_host.h -- host-side plumbing shared by the C ABI translation units (crl_abi.cu, crl_car_abi.cu, pong_opponent.cu).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "../../include/crl_b200.h"

// Defined in crl_abi.cu: sets the calling thread's crl_last_error text and returns `code`; adds to crl_launch_count.
int crl_set_error(int code, const char* fmt, ...);
void crl_count_launch(int n);

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) return crl_set_error(CRL_E_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)
// n = the number of kernels the call launches
#define LAUNCH(expr, n)      \
    do {                     \
        CUDA_TRY(expr);      \
        crl_count_launch(n); \
    } while (0)

// Every ABI entry point runs on the handle's device and leaves the caller's current device as it found it
// (a process that drives several GPUs must not have its current device flipped by an env on another GPU,
// including when a handle is destroyed at garbage-collection time).
struct CrlDeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit CrlDeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) {
            err = cudaSetDevice(device);
            switched = (err == cudaSuccess);
        }
    }
    ~CrlDeviceGuard() {
        if (switched) cudaSetDevice(prev);
    }
    CrlDeviceGuard(const CrlDeviceGuard&) = delete;
    CrlDeviceGuard& operator=(const CrlDeviceGuard&) = delete;
};

#define CHECK_HANDLE(h, device)                                       \
    do {                                                              \
        if (!(h)) return crl_set_error(CRL_E_INVALID, "null handle"); \
    } while (0);                                                      \
    CrlDeviceGuard crl_guard_(device);                                \
    CUDA_TRY(crl_guard_.err)

// The device check of every *_create.
inline int crl_check_device(int device) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return crl_set_error(CRL_E_CUDA, "no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return crl_set_error(CRL_E_INVALID, "device %d out of range", device);
    return CRL_OK;
}

// `count` device counters -> stats_host.  Synchronises `s`.
inline int crl_read_counters(const unsigned long long* counters_dev, uint64_t* stats_host, int count, cudaStream_t s) {
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "counters are copied as they are");
    CUDA_TRY(cudaMemcpyAsync(stats_host, counters_dev, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return CRL_OK;
}

// The device memory a handle owns.  Every buffer is zero-filled and has 16 bytes of slack past its end (kernels may load
// a whole 16-byte chunk across it).
class DeviceAllocs {
    std::vector<void*> ptrs_;

public:
    template <typename T>
    cudaError_t alloc(T** p, size_t count) {
        void* q = nullptr;
        cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 16);
        if (e != cudaSuccess) return e;
        ptrs_.push_back(q);
        *p = (T*)q;
        return cudaMemset(q, 0, count * sizeof(T) + 16);
    }
    // A buffer superseded by a re-upload; nullptr is ignored.  Only once no queued work can still read it.
    cudaError_t free(const void* p) {
        auto it = std::find(ptrs_.begin(), ptrs_.end(), p);
        if (it == ptrs_.end()) return cudaSuccess;
        ptrs_.erase(it);
        return cudaFree(const_cast<void*>(p));
    }
    void free_all() {
        for (void* p : ptrs_) cudaFree(p);
        ptrs_.clear();
    }
};

// A stream beside the caller's, created on first use: fork(s) starts it behind everything queued on s so far, join(s)
// makes s wait for everything queued on it so far.
struct SideStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;

    // All three objects or none: a failed creation is tried again by the next call.
    cudaError_t ensure(bool high_priority) {
        if (stream) return cudaSuccess;
        int lo = 0, hi = 0;
        cudaError_t e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&stream, cudaStreamNonBlocking, high_priority ? hi : 0);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming);
        if (e != cudaSuccess) destroy();
        return e;
    }
    cudaError_t fork(cudaStream_t s) {
        cudaError_t e = cudaEventRecord(ev_fork, s);
        return e == cudaSuccess ? cudaStreamWaitEvent(stream, ev_fork, 0) : e;
    }
    cudaError_t join(cudaStream_t s) {
        cudaError_t e = cudaEventRecord(ev_join, stream);
        return e == cudaSuccess ? cudaStreamWaitEvent(s, ev_join, 0) : e;
    }
    cudaError_t sync() { return stream ? cudaStreamSynchronize(stream) : cudaSuccess; }
    void destroy() {
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (stream) cudaStreamDestroy(stream);
        stream = nullptr;
        ev_fork = ev_join = nullptr;
    }
};
