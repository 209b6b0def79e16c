// handle.cuh - the host plumbing every library handle shares (uavenv in uavenv_capi.cu, uavpolicy in policy_forward.cu,
// uavtrain in policy_train.cu): error messages, tracked device allocations, the checks every *_create makes, and
// teardown.  Return codes are those of include/uavenv_b200.h: -1 bad argument, -2 CUDA failure, -3 out of memory.
#pragma once
#include <cstdarg>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

namespace capi {

struct Handle {
    int device = 0;
    std::vector<void *> allocs;   // freed together by destroy_handle
    std::string err;              // *_last_error(handle)
};

// *_last_error(NULL): the last failure of this thread that had no handle to record it; one string per handle type
template <typename H>
std::string &handle_free_error() {
    static thread_local std::string s;
    return s;
}

template <typename H>
const char *last_error(const H *h) { return h ? h->err.c_str() : handle_free_error<H>().c_str(); }

inline void record(std::string &err, const char *fmt, va_list ap) {
    char buf[512];
    vsnprintf(buf, sizeof buf, fmt, ap);
    err = buf;
}

// records the message for *_last_error(h), or for *_last_error(NULL) when h is NULL, and returns code
template <typename H>
int fail(H *h, int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    record(h ? h->err : handle_free_error<H>(), fmt, ap);
    va_end(ap);
    return code;
}

// fail<H>(nullptr, ...): a failure with no handle, recorded for *_last_error(NULL) of handle type H.  H may be an
// incomplete type here, as in the env library's handle-free entry points, which never see struct uavenv.
template <typename H>
int fail(std::nullptr_t, int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    record(handle_free_error<H>(), fmt, ap);
    va_end(ap);
    return code;
}

// returns from the enclosing function when a CUDA call fails: -3 when the device ran out of memory, -2 otherwise
#define CU_TRY(h, expr)                                                                              \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return capi::fail(h, e_ == cudaErrorMemoryAllocation ? -3 : -2, "%s failed: %s", #expr,  \
                              cudaGetErrorString(e_));                                               \
    } while (0)

// for an entry point without a handle: 0 when e is cudaSuccess, otherwise -2 with "<fn>: <what> failed: <error>" for
// *_last_error(NULL) of handle type H
template <typename H>
int check_cuda(cudaError_t e, const char *fn, const char *what) {
    return e == cudaSuccess ? 0 : fail<H>(nullptr, -2, "%s: %s failed: %s", fn, what, cudaGetErrorString(e));
}

// cudaMalloc of n elements (at least one), freed with the handle
template <typename T>
cudaError_t alloc(Handle *h, T **ptr, size_t n) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, (n ? n : 1) * sizeof(T));
    if (e == cudaSuccess) { h->allocs.push_back(q); *ptr = static_cast<T *>(q); }
    return e;
}

// The checks of fn (= "<api>_create") that need no device: out, and its size argument `size`, named size_name.
// On success *out is NULL until the caller hands a handle over.
template <typename H>
int check_create_args(const char *fn, const char *size_name, int32_t size, H **out) {
    if (!out) return fail<H>(nullptr, -1, "%s: out is NULL", fn);
    *out = nullptr;
    if (size <= 0) return fail<H>(nullptr, -1, "%s: %s must be > 0 (got %d)", fn, size_name, size);
    return 0;
}

// The device checks of fn, after its argument checks.  On success p is a new handle for `device`.
template <typename H>
int new_handle(const char *fn, int32_t device, H *&p) {
    p = nullptr;
    int ndev = 0;
    const cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(p, -2, "%s: no CUDA device (%s); there is no CPU fallback", fn,
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return fail(p, -1, "%s: device %d out of range", fn, device);
    p = new (std::nothrow) H();
    if (!p) return fail(p, -3, "%s: out of host memory", fn);
    p->device = device;
    return 0;
}

// frees a handle whose create failed, keeping its message for *_last_error(NULL); returns code
template <typename H>
int abandon_handle(H *p, int code) {
    handle_free_error<H>() = p->err;
    for (void *q : p->allocs) cudaFree(q);
    delete p;
    return code;
}

template <typename H>
int destroy_handle(H *p) {
    if (!p) return 0;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    for (void *q : p->allocs) cudaFree(q);
    delete p;
    return 0;
}

}  // namespace capi
