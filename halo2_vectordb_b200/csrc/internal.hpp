// internal.hpp -- helpers shared by the translation units of libh2v.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "h2v.h"

namespace h2v {
int set_error(int code, const char *msg);     // h2v.cu: records the thread-local h2v_last_error() text
void count_launches(uint64_t n);              // h2v.cu: h2v_launch_count()
int current_device();

inline int failf(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    return set_error(code, buf);
}

// a device allocation that grows on demand and keeps its size between calls
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return H2V_OK;
        release();
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            return failf(H2V_ENOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
        }
        cap = bytes;
        return H2V_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
}  // namespace h2v

#define H2V_CU(x)                                                                                                  \
    do {                                                                                                           \
        cudaError_t e_ = (x);                                                                                      \
        if (e_ != cudaSuccess) return h2v::failf(H2V_ECUDA, "%s failed: %s", #x, cudaGetErrorString(e_));          \
    } while (0)
#define H2V_LAUNCHED()                                                                                             \
    do {                                                                                                           \
        h2v::count_launches(1);                                                                                    \
        cudaError_t e_ = cudaGetLastError();                                                                       \
        if (e_ != cudaSuccess)                                                                                     \
            return h2v::failf(H2V_ECUDA, "kernel launch failed (%s:%d): %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
    } while (0)
#define H2V_TRY(x)                  \
    do {                            \
        int rc_ = (x);              \
        if (rc_) return rc_;        \
    } while (0)
