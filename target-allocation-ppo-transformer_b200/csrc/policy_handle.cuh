// policy_handle.cuh - the host plumbing both policy handles share (uavpolicy in policy_forward.cu, uavtrain in
// policy_train.cu): error messages, tracked device allocations, the checks every *_create makes, and teardown.
#pragma once
#include <cstdarg>
#include <cstdio>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

namespace uavp {

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

// records the message for *_last_error and returns code
template <typename H>
int fail(H *h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    (h ? h->err : handle_free_error<H>()) = buf;
    return code;
}

#define UAVP_TRY(h, expr)                                                                                  \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess) return uavp::fail(h, -2, "%s failed: %s", #expr, cudaGetErrorString(e_));   \
    } while (0)

// cudaMalloc of n elements (at least one), freed with the handle
template <typename T>
cudaError_t alloc(Handle *h, T **ptr, size_t n) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, (n ? n : 1) * sizeof(T));
    if (e == cudaSuccess) { h->allocs.push_back(q); *ptr = static_cast<T *>(q); }
    return e;
}

// The checks of fn (= "<api>_create") before it allocates anything; `size` is its size argument, named size_name.
// On success p is a new handle for `device` and *out is NULL until the caller hands p over.
template <typename H>
int new_handle(const char *fn, const char *size_name, int32_t device, int32_t size, H **out, H *&p) {
    p = nullptr;
    if (!out) return fail(p, -1, "%s: out is NULL", fn);
    *out = nullptr;
    if (size <= 0) return fail(p, -1, "%s: %s must be > 0", fn, size_name);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(p, -2, "%s: no CUDA device; there is no CPU fallback", fn);
    if (device < 0 || device >= ndev) return fail(p, -1, "%s: device %d out of range", fn, device);
    p = new (std::nothrow) H();
    if (!p) return fail(p, -3, "out of host memory");
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

}  // namespace uavp
