// Shared plumbing for libqmri_b200: context, error reporting, launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string>
#include <vector>

#include "../../include/qmri.h"

struct qmri_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    int64_t launches = 0;
    int sm_count = 148;
    size_t l2_bytes = 0;
};

extern thread_local char g_qmri_err[512];

// per-device caches (cudaFuncSetAttribute opt-ins, occupancy queries) are indexed by qmri_ctx::device: the attribute is per device
// and one process may hold contexts on several GPUs
constexpr int QMRI_MAX_DEV = 64;
static inline int qmri_dev_slot(const qmri_ctx* ctx) { return ctx->device & (QMRI_MAX_DEV - 1); }

static inline int qmri_fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_qmri_err, sizeof(g_qmri_err), fmt, ap);
    va_end(ap);
    return code;
}

#define QCUDA(expr)                                                                                   \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess)                                                                        \
            return qmri_fail(QMRI_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                             __FILE__, __LINE__);                                                     \
    } while (0)

#define QCHECK(expr)              \
    do {                          \
        int _r = (expr);          \
        if (_r != QMRI_OK) return _r; \
    } while (0)

#define QLAUNCH_CHECK(ctx)                                                                            \
    do {                                                                                              \
        (ctx)->launches++;                                                                            \
        cudaError_t _e = cudaGetLastError();                                                          \
        if (_e != cudaSuccess)                                                                        \
            return qmri_fail(QMRI_ECUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),  \
                             __FILE__, __LINE__);                                                     \
    } while (0)

struct DevSetter {
    int prev = -1;
    explicit DevSetter(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DevSetter() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

template <typename T>
static inline int dev_alloc(T** p, size_t n) {
    cudaError_t e = cudaMalloc((void**)p, n * sizeof(T));
    if (e != cudaSuccess) return qmri_fail(QMRI_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e));
    return QMRI_OK;
}

static inline int dtype_is_complex(int dt) { return dt == QMRI_C64 || dt == QMRI_C128; }
static inline size_t dtype_size(int dt) {
    switch (dt) {
        case QMRI_F32: return 4;
        case QMRI_F64: return 8;
        case QMRI_C64: return 8;
        case QMRI_C128: return 16;
    }
    return 0;
}

// ordered-int encoding of floats for atomicMin/atomicMax
__host__ __device__ static inline int float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    int b = __float_as_int(f);
#else
    int b;
    memcpy(&b, &f, 4);
#endif
    return b >= 0 ? b : b ^ 0x7fffffff;
}
__host__ __device__ static inline float ordered_to_float(int k) {
    int b = k >= 0 ? k : k ^ 0x7fffffff;
#ifdef __CUDA_ARCH__
    return __int_as_float(b);
#else
    float f;
    memcpy(&f, &b, 4);
    return f;
#endif
}

#ifdef __CUDACC__
// Sum of v over a block of THREADS threads in a fixed order (a butterfly within each warp, then the warps in order), so that the
// result does not depend on scheduling: no atomics.  Valid in thread 0.  Every thread of the block must call it.
template <int THREADS>
__device__ __forceinline__ double block_sum_fixed(double v) {
    static_assert(THREADS % 32 == 0, "whole warps");
    __shared__ double red[THREADS / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < THREADS / 32; ++w) v += red[w];
    return v;
}
#endif
