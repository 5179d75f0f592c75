// Host-side helpers shared by the translation units of libmvrl.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/mvrl.h"

int mvrl_fail(int code, const char* fmt, ...);

#define MVRL_CUDA(call)                                                                     \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return mvrl_fail(MVRL_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Every entry point runs on the device its handle (or its pointers) lives on and leaves the CALLER's current device
// untouched: a process driving several GPUs from one thread must not find torch's current device switched by a step.
struct MvrlDeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit MvrlDeviceGuard(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && device >= 0 && prev != device) {
            err = cudaSetDevice(device);
            switched = (err == cudaSuccess);
        }
    }
    ~MvrlDeviceGuard() { if (switched) cudaSetDevice(prev); }
    MvrlDeviceGuard(const MvrlDeviceGuard&) = delete;
    MvrlDeviceGuard& operator=(const MvrlDeviceGuard&) = delete;
};
#define MVRL_ON_DEVICE(device)                                                                               \
    MvrlDeviceGuard mvrl_guard_(device);                                                                     \
    if (mvrl_guard_.err != cudaSuccess)                                                                      \
        return mvrl_fail(MVRL_ECUDA, "cannot select device %d: %s", (int)(device), cudaGetErrorString(mvrl_guard_.err))

// device ordinal a pointer lives on (device or managed memory), -1 when it cannot be told (host pointer, null)
static inline int mvrl_device_of(const void* p) {
    if (!p) return -1;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return -1; }
    return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) ? at.device : -1;
}
// MVRL_EINVAL unless every non-null ptrs[j] is device memory on `device`; the message names names[j], or "argument j" without
// names.  cudaPointerGetAttributes does not synchronise and may be called during stream capture.
template <class T>
static inline int mvrl_check_device_ptrs(int device, T* const* ptrs, const char* const* names, int count, const char* who) {
    for (int j = 0; j < count; ++j)
        if (ptrs[j] && mvrl_device_of(ptrs[j]) != device)
            return names ? mvrl_fail(MVRL_EINVAL, "%s: %s is not device memory on device %d", who, names[j], device)
                         : mvrl_fail(MVRL_EINVAL, "%s: argument %d is not device memory on device %d", who, j, device);
    return MVRL_OK;
}
// stateless entry points (no handle): run where their output lives; fail when the pointers disagree
#define MVRL_ON_DEVICE_OF(out_ptr, in_ptr, who)                                                              \
    const int mvrl_dev_out_ = mvrl_device_of(out_ptr), mvrl_dev_in_ = mvrl_device_of(in_ptr);                \
    if (mvrl_dev_out_ < 0) return mvrl_fail(MVRL_EINVAL, "%s: output is not a device pointer", who);         \
    if (mvrl_dev_in_ >= 0 && mvrl_dev_in_ != mvrl_dev_out_)                                                  \
        return mvrl_fail(MVRL_EINVAL, "%s: input lives on device %d, output on device %d", who, mvrl_dev_in_, mvrl_dev_out_); \
    MVRL_ON_DEVICE(mvrl_dev_out_)

static inline unsigned mvrl_grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

static inline int mvrl_check_launch(const char* what) {
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) { cudaGetLastError(); return mvrl_fail(MVRL_ECUDA, "%s launch failed: %s", what, cudaGetErrorString(e)); }
    return MVRL_OK;
}

// shared by every create(): validates the device ordinal, fails without a GPU (no CPU path)
int mvrl_require_device(int device);
bool mvrl_invert_n(const double* a, double* out, int n);
