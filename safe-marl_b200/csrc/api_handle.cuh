// api_handle.cuh -- what the C-ABI host layers share for their handles (FpHandle: flex_api.cu, FpPolicy: policy.cu,
// FpReplay: predictor.cu), each of which has `int device` and `std::string err`: error reporting, the device guard,
// checked CUDA calls, all-or-nothing allocation, launch counting.  Host code only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <initializer_list>
#include <string>

#include "../../include/flexgpu.h"

// The last failed create of a handle of type H on this thread: its *_last_error(NULL).
template <class H>
std::string& create_error() {
    static thread_local std::string msg;
    return msg;
}

template <class H>
int fail(H* h, int code, const std::string& msg) {
    (h ? h->err : create_error<H>()) = msg;
    return code;
}

// Makes `device` current until the end of the scope, then the caller's current device again (best effort: a destructor
// cannot report).  Selecting the device that is already current costs no cudaSetDevice.
class DeviceGuard {
  public:
    explicit DeviceGuard(int device) : dev_(device) {
        if ((err_ = cudaGetDevice(&prev_)) != cudaSuccess) prev_ = -1;
        else if (prev_ != device) err_ = cudaSetDevice(device);
    }
    ~DeviceGuard() { if (prev_ >= 0 && prev_ != dev_) cudaSetDevice(prev_); }
    cudaError_t error() const { return err_; }

  private:
    int prev_ = -1, dev_;
    cudaError_t err_;
};

// The rest of the entry point runs on handle h's device; the caller's current device is current again on return.
#define USE_DEVICE(h)                                                                                     \
    const DeviceGuard device_guard_((h)->device);                                                         \
    if (const cudaError_t e_ = device_guard_.error())                                                     \
        return fail((h), FP_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e_))

#define CUDA_TRY(h, expr)                                                                                 \
    do {                                                                                                  \
        cudaError_t e_ = (expr);                                                                          \
        if (e_ != cudaSuccess) return fail((h), FP_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
    } while (0)

struct GroupBuf {
    void** p; size_t bytes;
    template <class T> GroupBuf(T** q, size_t b) : p(reinterpret_cast<void**>(q)), bytes(b) {}
};

// Allocates (and with zero, clears) a group of buffers used together, all null on entry.  On any failure every buffer
// of the group is freed back to null, so the next call retries the whole group.
inline cudaError_t alloc_group(std::initializer_list<GroupBuf> group, bool zero = false) {
    cudaError_t e = cudaSuccess;
    for (const GroupBuf& b : group)
        if (e == cudaSuccess && (e = cudaMalloc(b.p, b.bytes)) == cudaSuccess && zero) e = cudaMemset(*b.p, 0, b.bytes);
    if (e != cudaSuccess) for (const GroupBuf& b : group) { cudaFree(*b.p); *b.p = nullptr; }
    return e;
}

// After `k` kernel launches: a launch error goes to the handle, otherwise the handle (with `int64_t launches`) counts them.
template <class H>
int launched(H* h, const char* what, int64_t k = 1) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(h, FP_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
    h->launches += k;
    return FP_OK;
}

// Grid of a grid-stride kernel of 256-thread CTAs over `total` elements: at most 16 CTAs per SM of a B200.
inline int grid_for(int64_t total) {
    const int64_t g = (total + 255) / 256;
    return (int)(g < 1 ? 1 : (g > 148 * 16 ? 148 * 16 : g));
}
