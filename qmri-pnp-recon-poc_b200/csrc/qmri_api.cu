// libqmri_b200 - the C ABI of include/qmri.h: context, acquisition operator, x-update,
// ADMM loop driver, denoiser and dictionary-matching entry points.  Each entry point's
// reference counterpart is cited in include/qmri.h.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "aux_kernels.h"
#include "common.cuh"
#include "conv_kernels.h"
#include "lrtv_kernels.h"
#include "match_kernel.h"
#include "op_tables.h"
#include "unetres.h"
#include "xupdate_kernel.h"

thread_local char g_qmri_err[512] = "";

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n) {
        if (n <= bytes) return QMRI_OK;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&p, n);
        if (e != cudaSuccess) return qmri_fail(QMRI_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", n, cudaGetErrorString(e));
        bytes = n;
        return QMRI_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    template <typename T>
    T* as() const { return reinterpret_cast<T*>(p); }
};

namespace {

// host-layout array (already on the device as raw bytes) -> planar fp32
template <typename T>
__global__ void unpack_kernel(const T* __restrict__ src, float* __restrict__ re, float* __restrict__ im, size_t n, int cplx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (cplx) {
        re[i] = (float)src[2 * i];
        if (im) im[i] = (float)src[2 * i + 1];
    } else {
        re[i] = (float)src[i];
        if (im) im[i] = 0.f;
    }
}
template <typename T>
__global__ void pack_kernel(T* __restrict__ dst, const float* __restrict__ re, const float* __restrict__ im, size_t n, int cplx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (cplx) {
        dst[2 * i] = (T)re[i];
        dst[2 * i + 1] = im ? (T)im[i] : (T)0;
    } else {
        dst[i] = (T)re[i];
    }
}
// interleaved complex <-> float2
template <typename T>
__global__ void cvt_c_in_kernel(const T* __restrict__ src, float2* __restrict__ dst, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = make_float2((float)src[2 * i], (float)src[2 * i + 1]);
}
template <typename T>
__global__ void cvt_c_out_kernel(T* __restrict__ dst, const float2* __restrict__ src, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        dst[2 * i] = (T)src[i].x;
        dst[2 * i + 1] = (T)src[i].y;
    }
}
// z = v - u (u optional)
__global__ void sub_kernel(const float* vr, const float* vi, const float* ur, const float* ui, float* zr, float* zi, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    zr[i] = vr[i] - (ur ? ur[i] : 0.f);
    zi[i] = (vi ? vi[i] : 0.f) - (ui ? ui[i] : 0.f);
}
// w = x + u (u optional) with per-slice min/max of Re(w); w may be null (min/max only)
__global__ void add_minmax_kernel(const float* xr, const float* xi, const float* ur, const float* ui, float* wr, float* wi,
                                  size_t per_slice, int* minmax) {
    __shared__ float smin[8], smax[8];
    const int s = blockIdx.y;
    float lmin = INFINITY, lmax = -INFINITY;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_slice; i += (size_t)gridDim.x * blockDim.x) {
        size_t g = (size_t)s * per_slice + i;
        float a = xr[g] + (ur ? ur[g] : 0.f);
        if (wr) {
            wr[g] = a;
            wi[g] = xi[g] + (ui ? ui[g] : 0.f);
        }
        lmin = fminf(lmin, a);
        lmax = fmaxf(lmax, a);
    }
    for (int o = 16; o > 0; o >>= 1) {
        lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((threadIdx.x & 31) == 0) {
        smin[threadIdx.x >> 5] = lmin;
        smax[threadIdx.x >> 5] = lmax;
    }
    __syncthreads();
    if (threadIdx.x == 0 && minmax) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
            lmin = fminf(lmin, smin[w]);
            lmax = fmaxf(lmax, smax[w]);
        }
        atomicMin(minmax + 2 * s, float_to_ordered(lmin));
        atomicMax(minmax + 2 * s + 1, float_to_ordered(lmax));
    }
}
// ordered-int keys -> floats, and re-arm the keys for the next iteration
__global__ void minmax_finalize_kernel(int* ord, float* mm, int S) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < S) {
        mm[2 * i] = ordered_to_float(ord[2 * i]);
        mm[2 * i + 1] = ordered_to_float(ord[2 * i + 1]);
        ord[2 * i] = 0x7fffffff;
        ord[2 * i + 1] = (int)0x80000000;
    }
}

inline unsigned nblk(size_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

// PnP-ADMM progress monitor (PnP_ADMM.m:106-109).  Per-slice sum of squares of a [S][len] (+ b) fp32 array: one block per slice,
// a fixed summation order (no atomics), so the denominators of the history are the same bits on every run.
constexpr int MON_THREADS = 256;
__global__ void __launch_bounds__(MON_THREADS) slice_sumsq_kernel(const float* a, const float* b, size_t len, double* out) {
    const int s = blockIdx.x;
    double acc = 0.0;
    for (size_t i = threadIdx.x; i < len; i += MON_THREADS) {
        const double u = a[(size_t)s * len + i], w = b ? b[(size_t)s * len + i] : 0.f;
        acc += u * u + w * w;
    }
    acc = block_sum_fixed<MON_THREADS>(acc);
    if (threadIdx.x == 0) out[s] = acc;
}
// Row k of the history from the monitored x-update's partial sums (stream_solve_kernel: [S][C], stream_adj_kernel: [S][C][G]),
// each slice's summed in a fixed order.  k is a device-side counter, zeroed by qmri_admm_run and advanced here, because a replayed
// CUDA graph cannot take a new argument per iteration.  One block, so that every slice is written before the counter moves.
// dc_scale = (rho / (1 + rho))^2 turns |y - A z|^2 into |y - A x|^2.  A zero denominator gives NaN.
__global__ void __launch_bounds__(MON_THREADS) monitor_finalize_kernel(const double* dc_part, const double* gt_part, const double* y2,
                                                                       const double* gt2, int* counter, double* h_dc, double* h_gt,
                                                                       int S, int dc_n, int gt_n, int rows, double dc_scale) {
    const int k = *counter;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (k < rows) {
        for (int s = threadIdx.x; s < S; s += MON_THREADS) {
            double a = 0.0;
            for (int i = 0; i < dc_n; ++i) a += dc_part[(size_t)s * dc_n + i];
            h_dc[(size_t)k * S + s] = y2[s] > 0.0 ? sqrt(a * dc_scale / y2[s]) : nan;
            if (h_gt) {
                double b = 0.0;
                for (int i = 0; i < gt_n; ++i) b += gt_part[(size_t)s * gt_n + i];
                h_gt[(size_t)k * S + s] = gt2[s] > 0.0 ? sqrt(b / gt2[s]) : nan;
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) *counter = k + 1;
}

int unpack_async(qmri_ctx* ctx, const void* dev_raw, int dtype, float* re, float* im, size_t n) {
    if (n == 0) return QMRI_OK;
    int cplx = dtype_is_complex(dtype);
    if (dtype == QMRI_F32 || dtype == QMRI_C64)
        unpack_kernel<float><<<nblk(n), 256, 0, ctx->stream>>>((const float*)dev_raw, re, im, n, cplx);
    else
        unpack_kernel<double><<<nblk(n), 256, 0, ctx->stream>>>((const double*)dev_raw, re, im, n, cplx);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
int pack_async(qmri_ctx* ctx, void* dev_raw, int dtype, const float* re, const float* im, size_t n) {
    if (n == 0) return QMRI_OK;
    int cplx = dtype_is_complex(dtype);
    if (dtype == QMRI_F32 || dtype == QMRI_C64)
        pack_kernel<float><<<nblk(n), 256, 0, ctx->stream>>>((float*)dev_raw, re, im, n, cplx);
    else
        pack_kernel<double><<<nblk(n), 256, 0, ctx->stream>>>((double*)dev_raw, re, im, n, cplx);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

bool valid_dtype(int dt) { return dt >= QMRI_F32 && dt <= QMRI_C128; }

}  // namespace

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
extern "C" int qmri_version(void) { return QMRI_VERSION; }
extern "C" const char* qmri_last_error(void) { return g_qmri_err; }

extern "C" int qmri_ctx_create(qmri_ctx** out, int device_id) {
    if (!out) return qmri_fail(QMRI_EINVAL, "qmri_ctx_create: out is null");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return qmri_fail(QMRI_ECUDA, "no CUDA device available (%s); libqmri_b200 has no CPU fallback",
                         e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device_id < 0 || device_id >= ndev) return qmri_fail(QMRI_EINVAL, "device %d out of range [0,%d)", device_id, ndev);
    cudaDeviceProp prop;
    QCUDA(cudaGetDeviceProperties(&prop, device_id));
    if (prop.major != 10)
        return qmri_fail(QMRI_EUNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device_id,
                         prop.major, prop.minor);
    qmri_ctx* ctx = new qmri_ctx();
    ctx->device = device_id;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    DevSetter ds(device_id);
    QCUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    *out = ctx;
    return QMRI_OK;
}
extern "C" int qmri_ctx_destroy(qmri_ctx* ctx) {
    if (!ctx) return QMRI_OK;
    DevSetter ds(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return QMRI_OK;
}
extern "C" int qmri_ctx_set_stream(qmri_ctx* ctx, void* cuda_stream) {
    if (!ctx) return qmri_fail(QMRI_EINVAL, "null ctx");
    DevSetter ds(ctx->device);
    if (ctx->own_stream && ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        QCUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return QMRI_OK;
}
extern "C" int qmri_ctx_synchronize(qmri_ctx* ctx) {
    if (!ctx) return qmri_fail(QMRI_EINVAL, "null ctx");
    DevSetter ds(ctx->device);
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}
extern "C" int64_t qmri_ctx_launch_count(qmri_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------
// acquisition operator
// ------------------------------------------------------------------------------------------
// device copy of one set of streaming-kernel tables (general V: one per part of the union mask)
struct StreamDev {
    float2 *tw2 = nullptr, *tw448 = nullptr;
    uint32_t *itA = nullptr, *itB = nullptr, *ent = nullptr;
    uint16_t* rowmask = nullptr;
    int* frame_ptr = nullptr;
    int ns_max = 0, n_ovf = 0;
    int upload(const optab::K1Tables& t) {
        int r = 0;
        r |= dev_alloc(&tw2, (size_t)256);
        r |= dev_alloc(&tw448, t.tw448.size() / 2);
        r |= dev_alloc(&itA, t.itA.size());
        r |= dev_alloc(&itB, t.itB.size());
        r |= dev_alloc(&ent, t.ent.size());
        r |= dev_alloc(&rowmask, t.rowmask.size());
        r |= dev_alloc(&frame_ptr, t.frame_ptr.size());
        if (r) return QMRI_ENOMEM;
        cudaMemcpy(tw2, t.tw2.data(), sizeof(float) * t.tw2.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(tw448, t.tw448.data(), sizeof(float) * t.tw448.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(itA, t.itA.data(), sizeof(uint32_t) * t.itA.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(itB, t.itB.data(), sizeof(uint32_t) * t.itB.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(ent, t.ent.data(), sizeof(uint32_t) * t.ent.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(rowmask, t.rowmask.data(), sizeof(uint16_t) * t.rowmask.size(), cudaMemcpyHostToDevice);
        cudaError_t e = cudaMemcpy(frame_ptr, t.frame_ptr.data(), sizeof(int) * t.frame_ptr.size(), cudaMemcpyHostToDevice);
        ns_max = t.ns_max;
        n_ovf = t.n_ovf;
        return e == cudaSuccess ? QMRI_OK : qmri_fail(QMRI_ECUDA, "operator table upload failed: %s", cudaGetErrorString(e));
    }
    void release() {
        cudaFree(tw2); cudaFree(tw448); cudaFree(itA); cudaFree(itB); cudaFree(ent); cudaFree(rowmask); cudaFree(frame_ptr);
        tw2 = tw448 = nullptr; itA = itB = ent = nullptr; rowmask = nullptr; frame_ptr = nullptr;
    }
};

struct qmri_op {
    qmri_ctx* ctx = nullptr;
    int N = 0, M = 0, C = 0, L = 0;
    int k1_mc = 28;
    optab::K1Tables t;
    // device tables
    float2* d_tw = nullptr;
    int* d_frame_ptr = nullptr;
    uint16_t* d_samp = nullptr;
    uint32_t* d_p4tab = nullptr;
    float2* d_tw2 = nullptr;
    float2* d_tw448 = nullptr;
    uint32_t* d_itA = nullptr;
    uint32_t* d_itB = nullptr;
    uint32_t* d_ent = nullptr;
    uint16_t* d_rowmask = nullptr;
    uint32_t *d_ritA = nullptr, *d_ritB = nullptr, *d_rent = nullptr;  // real-image streaming kernels (folded rows)
    uint16_t* d_rrowmask = nullptr;
    int k1_kernel = 0;  // 0 = choose by batch size, 1 = cluster kernel, 2 = streaming kernel (QMRI_K1_KERNEL=cluster|stream)
    // general V (not the identity): channels are transformed on the union of the masks and mixed per k-space location
    bool general = false;
    optab::GeneralTables g;
    std::vector<StreamDev> gparts;
    float* d_V = nullptr;
    int *d_memb_ptr = nullptr, *d_memb_frame = nullptr, *d_memb_meas = nullptr, *d_meas_u = nullptr, *d_meas_frame = nullptr;
    float* d_minv = nullptr;      // [nU][C][C] (G_u + rho I)^{-1} for minv_rho
    double minv_rho = -1.0;
    // scratch for the host entry points
    DevBuf stage, a_re, a_im, b_re, b_im, c_re, c_im, ybuf, mm_ord, mm_f;
    DevBuf k1_part, k1_cbuf;  // streaming x-update: partial sample sums / solved samples
    // the bare sampling matrix (P.for / P.adj): uploaded on first use
    std::vector<double> hV;   // L x C column-major (empty: identity)
    DevBuf p_idx, p_fp, p_V, p_k, p_y, p_stage;
    size_t plane() const { return (size_t)N * M * C; }
};

static int op_from_frames(qmri_ctx* ctx, int N, int M, int C, int L, const std::vector<std::vector<int32_t>>& frames,
                          const double* V, qmri_op** out) {
    if (!ctx || !out) return qmri_fail(QMRI_EINVAL, "operator: null argument");
    if (N != M || (N != 224 && N != 256))
        return qmri_fail(QMRI_EUNSUPPORTED, "this build supports N == M == 224 or 256 (got %d x %d)", N, M);
    if (C < 1 || C > 64) return qmri_fail(QMRI_EINVAL, "C = %d out of range", C);
    bool identity = (L == C);
    if (V && identity) {
        for (int i = 0; i < L && identity; ++i)
            for (int c = 0; c < C; ++c)
                if (fabs(V[i + (size_t)L * c] - (i == c ? 1.0 : 0.0)) > 1e-12) {
                    identity = false;
                    break;
                }
    }
    if (!identity && !V) return qmri_fail(QMRI_EINVAL, "operator: V must be given when size(V,1) != C");
    if (!identity && C > 16) return qmri_fail(QMRI_EUNSUPPORTED, "general V: at most 16 channels (got %d)", C);
    if ((int)frames.size() != L) return qmri_fail(QMRI_EINVAL, "operator: %zu frames for size(V,1) = %d", frames.size(), L);
    for (int f = 0; f < L; ++f) {
        if (frames[f].size() > 4096) return qmri_fail(QMRI_EUNSUPPORTED, "frame %d samples %zu k-space locations; limit 4096", f, frames[f].size());
        for (size_t j = 0; j < frames[f].size(); ++j) {
            if (frames[f][j] < 0 || frames[f][j] >= N * M) return qmri_fail(QMRI_EINVAL, "k index out of range in frame %d", f);
            if (j && frames[f][j] <= frames[f][j - 1]) return qmri_fail(QMRI_EINVAL, "k indices must ascend inside frame %d", f);
        }
    }
    DevSetter ds(ctx->device);
    qmri_op* op = new qmri_op();
    op->ctx = ctx;
    op->N = N; op->M = M; op->C = C; op->L = L;
    const char* env = getenv("QMRI_K1_MC");
    if (env && atoi(env) == 56) op->k1_mc = 56;
    env = getenv("QMRI_K1_KERNEL");
    if (env && !strcmp(env, "cluster")) op->k1_kernel = 1;
    if (env && !strcmp(env, "stream")) op->k1_kernel = 2;
    env = getenv("QMRI_K1_QMIN");  // tuning knob: smallest chunk size tried for the streaming kernel's work items
    const int q_min = env ? atoi(env) : 8;  // 8: measured best on the spiral masks (fewer overflow partials)
    optab::build_k1_tables(N, frames, op->t, q_min);
    if (N == 256 && identity && !op->t.stream_ok) {  // 256: the streaming kernels are the only x-update kernels
        const int max_row = op->t.max_row;
        delete op;
        return qmri_fail(QMRI_EUNSUPPORTED, "N == M == 256: the mask does not fit the streaming kernel's work-item tables (densest k-space "
                         "row: %d samples)", max_row);
    }
    op->general = !identity;
    if (!identity) op->hV.assign(V, V + (size_t)L * C);
    if (op->general) {
        optab::build_general_tables(N, frames, V, L, C, op->g, q_min);
        if (!op->g.ok) {
            const int nU = op->g.nU;
            delete op;
            return qmri_fail(QMRI_EUNSUPPORTED, "general V: the union of the %d masks (%d k-space locations) does not fit the streaming "
                             "kernels' work-item tables even in 32 parts - SURVEY.md 8f-2", L, nU);
        }
    }
    const optab::K1Tables& t = op->t;
    size_t nm = std::max(1, t.nmeas);
    int r = 0;
    r |= dev_alloc(&op->d_tw, (size_t)N);
    r |= dev_alloc(&op->d_frame_ptr, t.frame_ptr.size());
    r |= dev_alloc(&op->d_samp, nm);
    r |= dev_alloc(&op->d_p4tab, std::max<size_t>(t.p4tab.size(), 1));
    r |= dev_alloc(&op->d_tw2, (size_t)256);
    r |= dev_alloc(&op->d_tw448, (size_t)2 * N);
    r |= dev_alloc(&op->d_itA, t.itA.size());
    r |= dev_alloc(&op->d_itB, t.itB.size());
    r |= dev_alloc(&op->d_ent, t.ent.size());
    r |= dev_alloc(&op->d_rowmask, t.rowmask.size());
    r |= dev_alloc(&op->d_ritA, t.r_itA.size());
    r |= dev_alloc(&op->d_ritB, t.r_itB.size());
    r |= dev_alloc(&op->d_rent, t.r_ent.size());
    r |= dev_alloc(&op->d_rrowmask, t.r_rowmask.size());
    if (op->general) {
        const optab::GeneralTables& g = op->g;
        const size_t nmf = std::max<size_t>(g.memb_frame.size(), 1);
        r |= dev_alloc(&op->d_V, g.V.size());
        r |= dev_alloc(&op->d_memb_ptr, g.memb_ptr.size());
        r |= dev_alloc(&op->d_memb_frame, nmf);
        r |= dev_alloc(&op->d_memb_meas, nmf);
        r |= dev_alloc(&op->d_meas_u, nmf);
        r |= dev_alloc(&op->d_meas_frame, nmf);
        r |= dev_alloc(&op->d_minv, std::max<size_t>((size_t)g.nU * C * C, 1));
        op->gparts.resize(g.parts.size());
        for (size_t pi = 0; pi < g.parts.size() && !r; ++pi) r |= op->gparts[pi].upload(g.parts[pi]);
        if (!r) {
            cudaMemcpy(op->d_V, g.V.data(), sizeof(float) * g.V.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(op->d_memb_ptr, g.memb_ptr.data(), sizeof(int) * g.memb_ptr.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(op->d_memb_frame, g.memb_frame.data(), sizeof(int) * g.memb_frame.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(op->d_memb_meas, g.memb_meas.data(), sizeof(int) * g.memb_meas.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(op->d_meas_u, g.meas_u.data(), sizeof(int) * g.meas_u.size(), cudaMemcpyHostToDevice);
            cudaMemcpy(op->d_meas_frame, g.meas_frame.data(), sizeof(int) * g.meas_frame.size(), cudaMemcpyHostToDevice);
        }
    }
    if (r) {
        qmri_op_destroy(op);
        return QMRI_ENOMEM;
    }
    cudaMemcpy(op->d_tw, t.tw.data(), sizeof(float) * 2 * N, cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_frame_ptr, t.frame_ptr.data(), sizeof(int) * t.frame_ptr.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_samp, t.samp.data(), sizeof(uint16_t) * t.nmeas, cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_tw2, t.tw2.data(), sizeof(float) * t.tw2.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_tw448, t.tw448.data(), sizeof(float) * t.tw448.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_itA, t.itA.data(), sizeof(uint32_t) * t.itA.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_itB, t.itB.data(), sizeof(uint32_t) * t.itB.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_ent, t.ent.data(), sizeof(uint32_t) * t.ent.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_rowmask, t.rowmask.data(), sizeof(uint16_t) * t.rowmask.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_ritA, t.r_itA.data(), sizeof(uint32_t) * t.r_itA.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_ritB, t.r_itB.data(), sizeof(uint32_t) * t.r_itB.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_rent, t.r_ent.data(), sizeof(uint32_t) * t.r_ent.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(op->d_rrowmask, t.r_rowmask.data(), sizeof(uint16_t) * t.r_rowmask.size(), cudaMemcpyHostToDevice);
    cudaError_t e = cudaMemcpy(op->d_p4tab, t.p4tab.data(), sizeof(uint32_t) * t.p4tab.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        qmri_op_destroy(op);
        return qmri_fail(QMRI_ECUDA, "operator table upload failed: %s", cudaGetErrorString(e));
    }
    *out = op;
    return QMRI_OK;
}

extern "C" int qmri_op_spiral(qmri_ctx* ctx, int N, int M, int S_curve, const double* V, int L, int C, qmri_op** out) {
    if (N != M) return qmri_fail(QMRI_EINVAL, "setup_subsampling_spiralgrided assumes N == M (zeros(N), line 31)");
    if (S_curve < 2 || L < 1) return qmri_fail(QMRI_EINVAL, "spiral: need S >= 2 and L >= 1");
    std::vector<std::vector<int32_t>> frames;
    optab::spiral_frames(N, S_curve, L, frames);
    return op_from_frames(ctx, N, M, C, L, frames, V, out);
}
extern "C" int qmri_op_epi(qmri_ctx* ctx, int N, int M, double percentage, const double* V, int L, int C, qmri_op** out) {
    if (!(percentage > 0.0) || percentage > 1.0 || L < 1) return qmri_fail(QMRI_EINVAL, "epi: percentage must be in (0,1]");
    std::vector<std::vector<int32_t>> frames;
    optab::epi_frames(N, M, percentage, L, frames);
    return op_from_frames(ctx, N, M, C, L, frames, V, out);
}
extern "C" int qmri_op_create(qmri_ctx* ctx, int N, int M, int C, int L, const int32_t* idx, const int64_t* frame_ptr,
                              const double* V, qmri_op** out) {
    if (!idx || !frame_ptr || L < 1) return qmri_fail(QMRI_EINVAL, "qmri_op_create: null idx / frame_ptr");
    std::vector<std::vector<int32_t>> frames(L);
    for (int f = 0; f < L; ++f) {
        if (frame_ptr[f + 1] < frame_ptr[f]) return qmri_fail(QMRI_EINVAL, "frame_ptr must be non-decreasing");
        frames[f].assign(idx + frame_ptr[f], idx + frame_ptr[f + 1]);
    }
    return op_from_frames(ctx, N, M, C, L, frames, V, out);
}
extern "C" int qmri_op_destroy(qmri_op* op) {
    if (!op) return QMRI_OK;
    DevSetter ds(op->ctx->device);
    cudaStreamSynchronize(op->ctx->stream);
    cudaFree(op->d_tw); cudaFree(op->d_frame_ptr); cudaFree(op->d_samp);
    cudaFree(op->d_p4tab);
    cudaFree(op->d_V); cudaFree(op->d_memb_ptr); cudaFree(op->d_memb_frame); cudaFree(op->d_memb_meas); cudaFree(op->d_meas_u);
    cudaFree(op->d_meas_frame); cudaFree(op->d_minv);
    for (auto& sd : op->gparts) sd.release();
    cudaFree(op->d_tw2); cudaFree(op->d_tw448); cudaFree(op->d_itA); cudaFree(op->d_itB); cudaFree(op->d_ent); cudaFree(op->d_rowmask);
    cudaFree(op->d_ritA); cudaFree(op->d_ritB); cudaFree(op->d_rent); cudaFree(op->d_rrowmask);
    op->stage.release(); op->a_re.release(); op->a_im.release(); op->b_re.release(); op->b_im.release();
    op->c_re.release(); op->c_im.release(); op->ybuf.release(); op->mm_ord.release(); op->mm_f.release();
    op->k1_part.release(); op->k1_cbuf.release();
    op->p_idx.release(); op->p_fp.release(); op->p_V.release(); op->p_k.release(); op->p_y.release(); op->p_stage.release();
    delete op;
    return QMRI_OK;
}
extern "C" int64_t qmri_op_nmeas(const qmri_op* op) { return op ? op->t.nmeas : -1; }
extern "C" int qmri_op_indices(const qmri_op* op, int32_t* idx, int64_t* frame_ptr) {
    if (!op) return qmri_fail(QMRI_EINVAL, "null op");
    if (idx) memcpy(idx, op->t.idx.data(), sizeof(int32_t) * op->t.nmeas);
    if (frame_ptr)
        for (int f = 0; f <= op->L; ++f) frame_ptr[f] = op->t.frame_ptr[f];
    return QMRI_OK;
}

// Kernel choice for one x-update launch: the streaming kernels (xupdate_stream.cu: forward / solve / adjoint, up to 16 CTAs
// per slice-channel image) from about two slices on, the single cluster kernel (xupdate_kernel.cu: the image stays in the
// shared memory of eight CTAs) below that - measured on B200: 23.8 vs 27.0 us at one slice, 16.2 vs 15.5 us at two, 9.1 vs
// 7.4 us at eight, 6.97 vs 4.13 us per slice at 120.  QMRI_K1_KERNEL=cluster|stream forces one (tests, profiling).
// N == M == 256: the cluster kernel is built for 224 only, so the streaming kernels run at every batch size.
// part / cbuf: scratch of the streaming kernels.  The host entry points use the operator's; an ADMM session brings its own,
// sized once for its batch, because its CUDA graph keeps the addresses.
// General V: forward transform of every channel on the union mask (one launch per part of the union) -> per-location channel
// mixing -> adjoint transform (the parts' corrections accumulate: the first pass runs the caller's mode, the others add in place).
static int k1_general_dispatch(qmri_op* op, K1Params p, int S, DevBuf* part, DevBuf* cbuf) {
    qmri_ctx* ctx = op->ctx;
    const optab::GeneralTables& g = op->g;
    const int nU = g.nU, P = (int)g.parts.size();
    // monitored PnP-ADMM session: the residual comes from the per-location solve (mix_residual_kernel), the ground-truth error
    // from the adjoint launch that completes x
    double* const mon_dc = p.mon_dc;
    double* const mon_gt = p.mon_gt;
    p.mon_dc = p.mon_gt = nullptr;
    p.shared_mask = 1;
    p.G = k1_stream_groups(S, op->C, ctx->sm_count);
    p.slot_stride = nU;
    QCHECK(part->ensure(std::max<size_t>(k1_stream_part_elems(S, op->C, p.G, nU), 1) * sizeof(float2)));
    QCHECK(cbuf->ensure(std::max<size_t>(k1_stream_cbuf_elems(S, op->C, nU), 1) * sizeof(float2)));
    p.part = part->as<float2>();
    p.cbuf = cbuf->as<float2>();
    GeneralMix m = {};
    m.part = p.part; m.cbuf = p.cbuf; m.y = p.y; m.y_out = p.y_out;
    m.V = op->d_V; m.Minv = op->d_minv;
    m.memb_ptr = op->d_memb_ptr; m.memb_frame = op->d_memb_frame; m.memb_meas = op->d_memb_meas;
    m.meas_u = op->d_meas_u; m.meas_frame = op->d_meas_frame;
    m.S = S; m.C = op->C; m.L = op->L; m.G = p.G; m.nU = nU; m.nmeas = op->t.nmeas;
    m.inv_n = 1.0f / (float)op->N;
    m.mon_dc = mon_dc;
    auto use_part = [&](K1Params& q, int pi) {
        const StreamDev& sd = op->gparts[pi];
        q.tw2 = sd.tw2; q.tw448 = sd.tw448; q.itA = sd.itA; q.itB = sd.itB; q.ent = sd.ent; q.rowmask = sd.rowmask;
        q.frame_ptr = sd.frame_ptr; q.n_ovf = sd.n_ovf;
        q.slot_off = g.part_off[pi];
        return sd.ns_max;
    };
    auto forward_all = [&]() -> int {
        K1Params q = p;
        q.stage = K1_STAGE_FWD_ONLY;
        for (int pi = 0; pi < P; ++pi) {
            const int ns = use_part(q, pi);
            QCHECK(k1_stream_launch(ctx, q, S, ns));
        }
        return QMRI_OK;
    };
    // pass 0 writes `mode`'s result, passes 1.. add their part of the correction in place (SOLVE mode: out = in + corr)
    auto adjoint_all = [&]() -> int {
        for (int pi = 0; pi < P; ++pi) {
            K1Params q = p;
            q.stage = K1_STAGE_ADJ_ONLY;
            const int ns = use_part(q, pi);
            const bool last = pi == P - 1;
            if (pi > 0) {
                q.mode = K1_SOLVE;
                q.in_re = p.out_re; q.in_im = p.out_im;
                q.x_re = q.x_im = nullptr;
            }
            if (!last) q.minmax = nullptr;  // min / max of the finished image only
            // x is complete after the last pass: SOLVE mode's output, or ADMM mode's x of a one-part union
            if (last && (p.mode == K1_SOLVE || (pi == 0 && p.x_re))) q.mon_gt = mon_gt;
            QCHECK(k1_stream_launch(ctx, q, S, ns));
            if (pi > 0 && p.mode == K1_ADMM && p.x_re) {  // last iteration: x receives the same corrections
                K1Params qx = q;
                qx.in_re = p.x_re; qx.in_im = p.x_im; qx.out_re = p.x_re; qx.out_im = p.x_im;
                qx.minmax = nullptr;
                qx.mon_gt = last ? mon_gt : nullptr;
                QCHECK(k1_stream_launch(ctx, qx, S, ns));
            }
        }
        return QMRI_OK;
    };
    if (p.mode == K1_FORWARD) {
        QCHECK(forward_all());
        return k1_general_mix_forward(ctx, m);
    }
    if (p.mode == K1_ADJOINT) {
        QCHECK(k1_general_mix_adjoint(ctx, m));
        return adjoint_all();
    }
    if (!(p.rho > 0.0)) return qmri_fail(QMRI_EINVAL, "x-update: rho must be positive");
    if (op->minv_rho != p.rho) {  // happens on the first x-update of a run, i.e. before any CUDA-graph capture of the loop
        std::vector<float> minv;
        optab::general_inverses(g, p.rho, minv);
        QCUDA(cudaStreamSynchronize(ctx->stream));
        QCUDA(cudaMemcpy(op->d_minv, minv.data(), sizeof(float) * minv.size(), cudaMemcpyHostToDevice));
        op->minv_rho = p.rho;
    }
    QCHECK(forward_all());
    QCHECK(k1_general_mix_solve(ctx, m));
    if (mon_dc) QCHECK(k1_general_mix_residual(ctx, m));
    return adjoint_all();
}

// A monitored PnP-ADMM session (qmri_admm_monitor) runs its x-update on the streaming kernels at every batch size: they carry the
// monitor's reductions, the cluster kernel does not.
static int k1_monitor_supported(const qmri_op* op) {
    if (op->general) return QMRI_OK;  // the general-V path always runs the streaming transforms
    if (op->k1_kernel == 1)
        return qmri_fail(QMRI_EUNSUPPORTED, "QMRI_K1_KERNEL=cluster: the convergence history (qmri_admm_monitor) is computed by the streaming "
                         "x-update kernels only");
    if (!op->t.stream_ok)
        return qmri_fail(QMRI_EUNSUPPORTED, "qmri_admm_monitor: this mask does not fit the streaming kernel's work-item tables (densest "
                         "k-space row: %d samples)", op->t.max_row);
    return QMRI_OK;
}

static int k1_dispatch(qmri_op* op, const K1Params& p_in, int S, DevBuf* part = nullptr, DevBuf* cbuf = nullptr) {
    K1Params p = p_in;
    if (!part) part = &op->k1_part;
    if (!cbuf) cbuf = &op->k1_cbuf;
    const bool monitored = p.mon_dc || p.mon_gt;
    if (monitored) {
        const int rc = k1_monitor_supported(op);
        if (rc) return rc;
    }
    if (op->general) return k1_general_dispatch(op, p, S, part, cbuf);
    qmri_ctx* ctx = op->ctx;
    const bool can_stream = op->t.stream_ok;
    bool stream = can_stream && (long long)S * op->C * K1_STREAM_MIN_IMAGES_DIV >= (long long)ctx->sm_count;
    if (op->N == 256 || monitored) {
        if (op->k1_kernel == 1 && op->N == 256)
            return qmri_fail(QMRI_EUNSUPPORTED, "QMRI_K1_KERNEL=cluster: the cluster x-update kernel supports N == M == 224 only (operator is "
                             "%d x %d)", op->N, op->M);
        stream = true;  // stream_ok: checked when the operator was built (256) or by k1_monitor_supported
    }
    if (op->k1_kernel == 1) stream = false;
    if (op->k1_kernel == 2) {
        if (!can_stream)
            return qmri_fail(QMRI_EUNSUPPORTED, "QMRI_K1_KERNEL=stream: this mask does not fit the streaming kernel's work-item tables (densest k-space row: %d samples)", op->t.max_row);
        stream = true;
    }
    if (stream) {
        p.G = k1_stream_groups(S, op->C, ctx->sm_count);
        // allocation happens on the first launch of a batch size, i.e. before any CUDA-graph capture of the loop
        QCHECK(part->ensure(k1_stream_part_elems(S, op->C, p.G, op->t.ns_max) * sizeof(float2)));
        QCHECK(cbuf->ensure(k1_stream_cbuf_elems(S, op->C, op->t.ns_max) * sizeof(float2)));
        p.part = part->as<float2>();
        p.cbuf = cbuf->as<float2>();
        return k1_stream_launch(ctx, p, S, op->t.ns_max);
    }
    return k1_launch(ctx, p, S, op->t.ns_max, op->k1_mc);
}

static void k1_fill_tables(const qmri_op* op, K1Params& p) {
    p.nf = op->N;
    p.tw = op->d_tw;
    p.frame_ptr = op->d_frame_ptr;
    p.samp = op->d_samp;
    p.p4tab = op->d_p4tab;
    p.p4_len = op->t.p4_len;
    p.tw2 = op->d_tw2;
    p.tw448 = op->d_tw448;
    p.itA = op->d_itA;
    p.itB = op->d_itB;
    p.ent = op->d_ent;
    p.rowmask = op->d_rowmask;
    p.n_ovf = op->t.n_ovf;
    p.C = op->C;
    p.nmeas = op->t.nmeas;
}

static int y_upload(qmri_op* op, const void* y, int y_dtype, int S) {
    qmri_ctx* ctx = op->ctx;
    if (!dtype_is_complex(y_dtype)) return qmri_fail(QMRI_EINVAL, "measurements y must be complex (QMRI_C64 / QMRI_C128)");
    size_t n = (size_t)S * op->t.nmeas;
    QCHECK(op->ybuf.ensure(std::max<size_t>(n, 1) * sizeof(float2)));
    QCHECK(op->stage.ensure(std::max<size_t>(n, 1) * dtype_size(y_dtype)));
    if (n == 0) return QMRI_OK;
    QCUDA(cudaMemcpyAsync(op->stage.p, y, n * dtype_size(y_dtype), cudaMemcpyHostToDevice, ctx->stream));
    if (y_dtype == QMRI_C64) cvt_c_in_kernel<float><<<nblk(n), 256, 0, ctx->stream>>>((const float*)op->stage.p, op->ybuf.as<float2>(), n);
    else cvt_c_in_kernel<double><<<nblk(n), 256, 0, ctx->stream>>>((const double*)op->stage.p, op->ybuf.as<float2>(), n);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

// H2D of a host N x M x C x S array into planar fp32 (re, im)
static int image_upload(qmri_op* op, const void* x, int dtype, int S, DevBuf& re, DevBuf& im) {
    qmri_ctx* ctx = op->ctx;
    size_t n = op->plane() * S;
    QCHECK(re.ensure(n * sizeof(float)));
    QCHECK(im.ensure(n * sizeof(float)));
    QCHECK(op->stage.ensure(n * dtype_size(dtype)));
    QCUDA(cudaMemcpyAsync(op->stage.p, x, n * dtype_size(dtype), cudaMemcpyHostToDevice, ctx->stream));
    return unpack_async(ctx, op->stage.p, dtype, re.as<float>(), im.as<float>(), n);
}
static int image_download(qmri_op* op, void* x, int dtype, int S, const float* re, const float* im) {
    qmri_ctx* ctx = op->ctx;
    size_t n = op->plane() * S;
    QCHECK(op->stage.ensure(n * dtype_size(dtype)));
    QCHECK(pack_async(ctx, op->stage.p, dtype, re, im, n));
    QCUDA(cudaMemcpyAsync(x, op->stage.p, n * dtype_size(dtype), cudaMemcpyDeviceToHost, ctx->stream));
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

extern "C" int qmri_forward(qmri_op* op, const void* x, int x_dtype, int S, void* y, int y_dtype) {
    if (!op || !x || !y) return qmri_fail(QMRI_EINVAL, "qmri_forward: null argument");
    if (S < 0 || !valid_dtype(x_dtype) || !dtype_is_complex(y_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_forward: bad S / dtype");
    if (S == 0) return QMRI_OK;
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    QCHECK(image_upload(op, x, x_dtype, S, op->a_re, op->a_im));
    size_t n = (size_t)S * op->t.nmeas;
    QCHECK(op->ybuf.ensure(std::max<size_t>(n, 1) * sizeof(float2)));
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_FORWARD;
    p.in_re = op->a_re.as<float>();
    p.in_im = dtype_is_complex(x_dtype) ? op->a_im.as<float>() : nullptr;
    p.y_out = op->ybuf.as<float2>();
    QCHECK(k1_dispatch(op, p, S));
    if (n) {
        QCHECK(op->stage.ensure(n * dtype_size(y_dtype)));
        if (y_dtype == QMRI_C64) cvt_c_out_kernel<float><<<nblk(n), 256, 0, ctx->stream>>>((float*)op->stage.p, op->ybuf.as<float2>(), n);
        else cvt_c_out_kernel<double><<<nblk(n), 256, 0, ctx->stream>>>((double*)op->stage.p, op->ybuf.as<float2>(), n);
        QLAUNCH_CHECK(ctx);
        QCUDA(cudaMemcpyAsync(y, op->stage.p, n * dtype_size(y_dtype), cudaMemcpyDeviceToHost, ctx->stream));
    }
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

extern "C" int qmri_adjoint(qmri_op* op, const void* y, int y_dtype, int S, void* x, int x_dtype) {
    if (!op || !y || !x) return qmri_fail(QMRI_EINVAL, "qmri_adjoint: null argument");
    if (S < 0 || !dtype_is_complex(x_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_adjoint: x must be complex");
    if (S == 0) return QMRI_OK;
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    QCHECK(y_upload(op, y, y_dtype, S));
    size_t n = op->plane() * S;
    QCHECK(op->a_re.ensure(n * sizeof(float)));
    QCHECK(op->a_im.ensure(n * sizeof(float)));
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_ADJOINT;
    p.y = op->ybuf.as<float2>();
    p.out_re = op->a_re.as<float>();
    p.out_im = op->a_im.as<float>();
    QCHECK(k1_dispatch(op, p, S));
    return image_download(op, x, x_dtype, S, op->a_re.as<float>(), op->a_im.as<float>());
}

extern "C" int qmri_xupdate(qmri_op* op, double rho, const void* y, int y_dtype, const void* v, int v_dtype, const void* u,
                            int u_dtype, int S, void* x, int x_dtype, void* w, int w_dtype, float* minmax) {
    if (!op || !y || !v || !x) return qmri_fail(QMRI_EINVAL, "qmri_xupdate: null argument");
    if (S < 0 || !valid_dtype(v_dtype) || !dtype_is_complex(x_dtype) || (u && !valid_dtype(u_dtype)) || (w && !dtype_is_complex(w_dtype)))
        return qmri_fail(QMRI_EINVAL, "qmri_xupdate: bad S / dtype");
    if (!(rho > 0.0)) return qmri_fail(QMRI_EINVAL, "qmri_xupdate: rho must be positive");
    if (S == 0) return QMRI_OK;
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    size_t n = op->plane() * S;
    QCHECK(y_upload(op, y, y_dtype, S));
    QCHECK(image_upload(op, v, v_dtype, S, op->a_re, op->a_im));                 // a = v
    if (u) QCHECK(image_upload(op, u, u_dtype, S, op->b_re, op->b_im));           // b = u
    QCHECK(op->c_re.ensure(n * sizeof(float)));
    QCHECK(op->c_im.ensure(n * sizeof(float)));
    float *ar = op->a_re.as<float>(), *ai = op->a_im.as<float>();
    float *br = u ? op->b_re.as<float>() : nullptr, *bi = u ? op->b_im.as<float>() : nullptr;
    float *cr = op->c_re.as<float>(), *ci = op->c_im.as<float>();
    sub_kernel<<<nblk(n), 256, 0, ctx->stream>>>(ar, ai, br, bi, cr, ci, n);     // c = z = v - u
    QLAUNCH_CHECK(ctx);
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_SOLVE;
    p.in_re = cr; p.in_im = ci;
    p.y = op->ybuf.as<float2>();
    p.out_re = ar; p.out_im = ai;                                                // a = x
    p.inv_1p_rho = (float)(1.0 / (1.0 + rho));
    p.rho = rho;
    QCHECK(k1_dispatch(op, p, S));
    QCHECK(image_download(op, x, x_dtype, S, ar, ai));
    if (w || minmax) {
        QCHECK(op->mm_ord.ensure(2 * S * sizeof(int)));
        QCHECK(op->mm_f.ensure(2 * S * sizeof(float)));
        QCHECK(k1_minmax_init(ctx, op->mm_ord.as<int>(), S));
        dim3 grid(std::min<unsigned>(nblk(op->plane()), 256), S);
        add_minmax_kernel<<<grid, 256, 0, ctx->stream>>>(ar, ai, br, bi, cr, ci, op->plane(), op->mm_ord.as<int>());  // c = w
        QLAUNCH_CHECK(ctx);
        minmax_finalize_kernel<<<nblk(S, 128), 128, 0, ctx->stream>>>(op->mm_ord.as<int>(), op->mm_f.as<float>(), S);
        QLAUNCH_CHECK(ctx);
        if (w) QCHECK(image_download(op, w, w_dtype, S, cr, ci));
        if (minmax) {
            QCUDA(cudaMemcpyAsync(minmax, op->mm_f.p, 2 * S * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
            QCUDA(cudaStreamSynchronize(ctx->stream));
        }
    }
    return QMRI_OK;
}

// ------------------------------------------------------------------------------------------
// denoiser entry points
// ------------------------------------------------------------------------------------------
extern "C" int qmri_unetres_load(qmri_ctx* ctx, int in_nc, const float* const* weights, int n_weights, qmri_net** out) {
    return unetres_create(ctx, in_nc, weights, n_weights, out);
}
extern "C" int qmri_unetres_destroy(qmri_net* net) {
    if (net) {
        DevSetter ds(net->ctx->device);
        cudaStreamSynchronize(net->ctx->stream);
    }
    unetres_free(net);
    return QMRI_OK;
}
extern "C" int qmri_unetres_set_precision(qmri_net* net, int mode) {
    if (!net) return qmri_fail(QMRI_EINVAL, "null net");
    if (mode != 0 && mode != 1) return qmri_fail(QMRI_EINVAL, "denoiser precision mode must be 0 (fp32) or 1 (tcgen05 split-bf16), got %d", mode);
    if (mode == 1 && !net->tc_available)
        return qmri_fail(QMRI_EUNSUPPORTED, "tensor mode unavailable: cuTensorMapEncodeTiled could not be resolved");
    net->precision = mode;
    return QMRI_OK;
}
extern "C" double qmri_unetres_flops(const qmri_net* net, int S, int H, int W) {
    return net ? unetres_flops(net->in_nc, S, H, W) : 0.0;
}
extern "C" int qmri_unetres_forward_dev(qmri_net* net, const float* in_dev, float* out_dev, const float* minmax_dev,
                                        const float* noise_map_dev, int S, int H, int W) {
    return unetres_forward_dev(net, in_dev, out_dev, minmax_dev, noise_map_dev, S, H, W, 1);
}

static int net_host_forward(qmri_net* net, const void* in, int in_dtype, void* out, int out_dtype, int S, int H, int W, int orient) {
    if (!net || !in || !out) return qmri_fail(QMRI_EINVAL, "denoiser: null argument");
    if (S < 0 || dtype_is_complex(in_dtype) || dtype_is_complex(out_dtype) || !valid_dtype(in_dtype) || !valid_dtype(out_dtype))
        return qmri_fail(QMRI_EINVAL, "denoiser: arrays must be real single or double");
    if (S == 0) return QMRI_OK;
    qmri_ctx* ctx = net->ctx;
    DevSetter ds(ctx->device);
    const size_t hw = (size_t)H * W;
    const size_t nin = hw * net->in_nc * S, nout = hw * 10 * S;
    const size_t raw = std::max(nin * dtype_size(in_dtype), nout * dtype_size(out_dtype));
    // io = [planar in | planar out | raw staging]
    size_t need = (nin + nout) * sizeof(float) + raw + 64;
    if (need > net->io_elems) {
        if (net->io) cudaFree(net->io);
        net->io = nullptr;
        net->io_elems = 0;
        cudaError_t e = cudaMalloc((void**)&net->io, need);
        if (e != cudaSuccess) return qmri_fail(QMRI_ENOMEM, "cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e));
        net->io_elems = need;
    }
    float* d_in = net->io;
    float* d_out = d_in + nin;
    void* d_raw = (void*)(d_out + nout + 4);
    d_raw = (void*)(((uintptr_t)d_raw + 15) & ~(uintptr_t)15);
    QCUDA(cudaMemcpyAsync(d_raw, in, nin * dtype_size(in_dtype), cudaMemcpyHostToDevice, ctx->stream));
    QCHECK(unpack_async(ctx, d_raw, in_dtype, d_in, nullptr, nin));
    // a multi-level (11-channel) host call carries the noise map as its 11th plane: split it off per slice
    if (net->in_nc == 11) {
        // planes of slice s: [11][hw]; the kernel wants [S][10][hw] + one shared map -> run slice by slice
        for (int s = 0; s < S; ++s) {
            const float* sl = d_in + (size_t)s * 11 * hw;
            QCHECK(unetres_forward_dev(net, sl, d_out + (size_t)s * 10 * hw, nullptr, sl + 10 * hw, 1, H, W, orient));
        }
    } else {
        QCHECK(unetres_forward_dev(net, d_in, d_out, nullptr, nullptr, S, H, W, orient));
    }
    QCHECK(pack_async(ctx, d_raw, out_dtype, d_out, nullptr, nout));
    QCUDA(cudaMemcpyAsync(out, d_raw, nout * dtype_size(out_dtype), cudaMemcpyDeviceToHost, ctx->stream));
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}
extern "C" int qmri_unetres_forward(qmri_net* net, const float* in, float* out, int S, int H, int W) {
    // PyTorch layout: planes [h][w], w fastest -> internal rows = h (H), fastest extent = W
    return net_host_forward(net, in, QMRI_F32, out, QMRI_F32, S, H, W, 0);
}
extern "C" int qmri_unetres_denoise(qmri_net* net, const void* in, int in_dtype, void* out, int out_dtype, int S, int H, int W) {
    // MATLAB layout H x W x C: planes [w][h], h fastest -> internal rows = w (W of them), fastest extent = H
    return net_host_forward(net, in, in_dtype, out, out_dtype, S, W, H, 1);
}

// ------------------------------------------------------------------------------------------
// ADMM loop
// ------------------------------------------------------------------------------------------
struct qmri_admm {
    qmri_op* op = nullptr;
    int S = 0;
    qmri_admm_params prm;
    DevBuf y, x0_re, x0_im, w_re, w_im, v, x_re, x_im, mm_ord, mm_f, noise, cb_in, cb_out;
    DevBuf k1_part, k1_cbuf;  // streaming x-update scratch (addresses are baked into the session's CUDA graph)
    // real-state loop (xupdate_real.cu): c_k and m_{k-1} on the sampled locations, and a second v buffer so that the last
    // x-update still finds v_{K-2}
    bool lean = false;
    int lean_group = 0;       // slices per forward / solve / adjoint triple (QMRI_K1R_GROUP; default: all)
    DevBuf v_alt, cstate, mprev;
    float *h_in = nullptr, *h_out = nullptr;  // pinned, host-callback path
    bool uploaded = false;
    // one steady-state ADMM iteration (x-update, min/max, 64-conv denoiser = ~130 launches) captured as a CUDA graph:
    // at small slice batches the loop is otherwise bound by the host's launch rate
    cudaGraphExec_t graph = nullptr;
    const void* graph_ws = nullptr;  // denoiser workspace / chunk / precision the graph was captured with
    int graph_chunk = 0, graph_prec = -1;
    int64_t graph_launches = 0;
    bool graph_failed = false;
    // convergence history (qmri_admm_monitor; PnP_ADMM.m:106-109): partial sums of the monitored x-update kernels, the slices'
    // |y|^2 and |gt|^2, and the history [rows][S] itself, written in the loop (and in its graph) at the row a device counter names
    int mon = 0;              // 0 off, 1 residual, 2 residual and ground-truth error
    bool gt_cplx = false;
    bool y2_stale = true;     // y was uploaded since |y|^2 was reduced
    int mon_G = 0;            // slab groups of the adjoint kernel (layout of mon_gt)
    DevBuf gt_re, gt_im, gt2, y2, mon_dc, mon_gt, hist_dc, hist_gt, hist_ctr;
    int hist_iters = 0;       // rows the last run recorded
    bool hist_has_gt = false;
    // monitor mode, and history buffers (address and capacity: the row limit is a kernel argument), the graph was captured with
    int graph_mon = -1;
    const void* graph_hist[2] = {nullptr, nullptr};
    size_t graph_hist_bytes[2] = {0, 0};
};

static bool admm_lean_eligible(const qmri_op* op, int S);

extern "C" int qmri_admm_create(qmri_op* op, int S, const qmri_admm_params* params, qmri_admm** out) {
    if (!op || !params || !out) return qmri_fail(QMRI_EINVAL, "qmri_admm_create: null argument");
    if (S < 1) return qmri_fail(QMRI_EINVAL, "qmri_admm_create: S must be >= 1");
    if (!(params->gamma > 0.0)) return qmri_fail(QMRI_EINVAL, "param.gamma must be positive");
    if (params->iters < 0) return qmri_fail(QMRI_EINVAL, "param.iter must be >= 0");
    if (!params->net && !params->fn) return qmri_fail(QMRI_EINVAL, "param.net missing: pass a qmri_net or a callback");
    if (params->multi_level && !params->noise_map) return qmri_fail(QMRI_EINVAL, "multi_level denoiser needs param.noise_map");
    if (params->net && params->net->in_nc != (params->multi_level ? 11 : 10))
        return qmri_fail(QMRI_EINVAL, "denoiser has %d input channels but denoiser_type wants %d", params->net->in_nc,
                         params->multi_level ? 11 : 10);
    if (op->C != 10) return qmri_fail(QMRI_EUNSUPPORTED, "PnP-ADMM needs C == 10 channels (denoiser output), got %d", op->C);
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    qmri_admm* st = new qmri_admm();
    st->op = op;
    st->S = S;
    st->prm = *params;
    const size_t n = op->plane() * S, hw = (size_t)op->N * op->M;
    int r = 0;
    r |= st->y.ensure(std::max<size_t>((size_t)S * op->t.nmeas, 1) * sizeof(float2));
    r |= st->x0_re.ensure(n * 4); r |= st->x0_im.ensure(n * 4);
    r |= st->w_re.ensure(n * 4);  r |= st->w_im.ensure(n * 4);
    r |= st->x_re.ensure(n * 4);  r |= st->x_im.ensure(n * 4);
    r |= st->v.ensure(n * 4);
    st->lean = admm_lean_eligible(op, S);
    if (getenv("QMRI_DEBUG"))
        fprintf(stderr, "libqmri_b200: admm session S = %d: %s-state x-update (general %d, stream_ok %d, real_ok %d, ns_max %d, r_n_ovf %d)\n", S,
                st->lean ? "real" : "complex", (int)op->general, (int)op->t.stream_ok, (int)op->t.real_ok, op->t.ns_max, op->t.r_n_ovf);
    if (st->lean) {
        const char* env = getenv("QMRI_K1R_GROUP");  // tuning knob: slices per kernel triple
        st->lean_group = std::max(1, std::min(S, env ? atoi(env) : S));  // one launch triple measured fastest (L2-sized groups: +33 %)
        const size_t ns = (size_t)op->t.ns_max;
        r |= st->v_alt.ensure(n * 4);
        r |= st->cstate.ensure(k1r_state_elems(S, op->C, (int)ns) * sizeof(float2));
        r |= st->mprev.ensure(k1r_state_elems(S, op->C, (int)ns) * sizeof(float2));
        // scratch of both kernel families, sized once (their addresses end up in the captured graph)
        const size_t part_c = k1_stream_part_elems(S, op->C, k1_stream_groups(S, op->C, ctx->sm_count), (int)ns);
        const size_t part_r = k1r_part_elems(st->lean_group, op->C, 8, (int)ns);
        r |= st->k1_part.ensure(std::max(part_c, part_r) * sizeof(float2));
        r |= st->k1_cbuf.ensure(k1_stream_cbuf_elems(S, op->C, (int)ns) * sizeof(float2));
    }
    r |= st->mm_ord.ensure(2 * S * sizeof(int));
    r |= st->mm_f.ensure(2 * S * sizeof(float));
    if (params->multi_level) r |= st->noise.ensure(hw * 4);
    if (!params->net) {
        const size_t cin = params->multi_level ? 11 : 10;
        r |= st->cb_in.ensure(hw * cin * S * 4);
        r |= st->cb_out.ensure(n * 4);
        if (params->fn_space == QMRI_HOST) {
            if (cudaMallocHost((void**)&st->h_in, hw * cin * S * 4) != cudaSuccess || cudaMallocHost((void**)&st->h_out, n * 4) != cudaSuccess) r |= 1;
        }
    }
    if (r) {
        qmri_admm_destroy(st);
        return qmri_fail(QMRI_ENOMEM, "qmri_admm_create: device allocation failed for S = %d", S);
    }
    if (params->multi_level) {
        cudaError_t e = cudaMemcpy(st->noise.p, params->noise_map, hw * 4, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            qmri_admm_destroy(st);
            return qmri_fail(QMRI_ECUDA, "noise map upload failed: %s", cudaGetErrorString(e));
        }
    }
    if (params->net) {
        int rr = unetres_reserve(params->net, S, op->M, op->N);
        if (rr) {
            qmri_admm_destroy(st);
            return rr;
        }
    }
    st->prm.noise_map = nullptr;  // host pointer is not retained
    *out = st;
    return QMRI_OK;
}

extern "C" int qmri_admm_destroy(qmri_admm* st) {
    if (!st) return QMRI_OK;
    DevSetter ds(st->op->ctx->device);
    cudaStreamSynchronize(st->op->ctx->stream);
    st->y.release(); st->x0_re.release(); st->x0_im.release(); st->w_re.release(); st->w_im.release();
    st->v.release(); st->x_re.release(); st->x_im.release(); st->mm_ord.release(); st->mm_f.release();
    st->noise.release(); st->cb_in.release(); st->cb_out.release(); st->k1_part.release(); st->k1_cbuf.release();
    st->v_alt.release(); st->cstate.release(); st->mprev.release();
    st->gt_re.release(); st->gt_im.release(); st->gt2.release(); st->y2.release(); st->mon_dc.release(); st->mon_gt.release();
    st->hist_dc.release(); st->hist_gt.release(); st->hist_ctr.release();
    if (st->h_in) cudaFreeHost(st->h_in);
    if (st->h_out) cudaFreeHost(st->h_out);
    if (st->graph) cudaGraphExecDestroy(st->graph);
    delete st;
    return QMRI_OK;
}

extern "C" int qmri_admm_upload(qmri_admm* st, const void* y, int y_dtype, const void* x0, int x0_dtype) {
    if (!st || !y || !x0) return qmri_fail(QMRI_EINVAL, "qmri_admm_upload: null argument");
    if (!dtype_is_complex(y_dtype) || !valid_dtype(x0_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_admm_upload: bad dtype");
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    const size_t ny = (size_t)st->S * op->t.nmeas, n = op->plane() * st->S;
    QCHECK(op->stage.ensure(std::max(ny * dtype_size(y_dtype), n * dtype_size(x0_dtype))));
    if (ny) {
        QCUDA(cudaMemcpyAsync(op->stage.p, y, ny * dtype_size(y_dtype), cudaMemcpyHostToDevice, ctx->stream));
        if (y_dtype == QMRI_C64) cvt_c_in_kernel<float><<<nblk(ny), 256, 0, ctx->stream>>>((const float*)op->stage.p, st->y.as<float2>(), ny);
        else cvt_c_in_kernel<double><<<nblk(ny), 256, 0, ctx->stream>>>((const double*)op->stage.p, st->y.as<float2>(), ny);
        QLAUNCH_CHECK(ctx);
    }
    QCUDA(cudaMemcpyAsync(op->stage.p, x0, n * dtype_size(x0_dtype), cudaMemcpyHostToDevice, ctx->stream));
    QCHECK(unpack_async(ctx, op->stage.p, x0_dtype, st->x0_re.as<float>(), st->x0_im.as<float>(), n));
    // w starts as X0 so that qmri_admm_xupdate_only (profiling) has a defined state before the first qmri_admm_run
    QCUDA(cudaMemcpyAsync(st->w_re.p, st->x0_re.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    QCUDA(cudaMemcpyAsync(st->w_im.p, st->x0_im.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    if (st->lean) {  // the same for the real-state loop: v = Re X0, c = m = 0
        QCUDA(cudaMemcpyAsync(st->v.p, st->x0_re.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        QCUDA(cudaMemsetAsync(st->cstate.p, 0, st->cstate.bytes, ctx->stream));
        QCUDA(cudaMemsetAsync(st->mprev.p, 0, st->mprev.bytes, ctx->stream));
    }
    st->uploaded = true;
    st->y2_stale = true;
    return QMRI_OK;
}

extern "C" int qmri_admm_monitor(qmri_admm* st, int enable, const void* gt, int gt_dtype) {
    if (!st) return qmri_fail(QMRI_EINVAL, "qmri_admm_monitor: null state");
    if (!enable) {
        st->mon = 0;
        return QMRI_OK;
    }
    if (gt && !valid_dtype(gt_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_admm_monitor: bad ground-truth dtype %d", gt_dtype);
    qmri_op* op = st->op;
    QCHECK(k1_monitor_supported(op));
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    const int S = st->S, C = op->C;
    const size_t n = op->plane() * S;
    st->mon_G = k1_stream_groups(S, C, ctx->sm_count);
    const int dc_n = op->general ? k1_general_residual_parts(op->g.nU) : C;
    QCHECK(st->mon_dc.ensure((size_t)S * dc_n * sizeof(double)));
    QCHECK(st->y2.ensure((size_t)S * sizeof(double)));
    QCHECK(st->hist_ctr.ensure(sizeof(int)));
    if (gt) {
        st->gt_cplx = dtype_is_complex(gt_dtype);
        QCHECK(st->gt_re.ensure(n * 4));
        if (st->gt_cplx) QCHECK(st->gt_im.ensure(n * 4));
        QCHECK(st->gt2.ensure((size_t)S * sizeof(double)));
        QCHECK(st->mon_gt.ensure((size_t)S * C * st->mon_G * sizeof(double)));
        QCHECK(op->stage.ensure(n * dtype_size(gt_dtype)));
        QCUDA(cudaMemcpyAsync(op->stage.p, gt, n * dtype_size(gt_dtype), cudaMemcpyHostToDevice, ctx->stream));
        QCHECK(unpack_async(ctx, op->stage.p, gt_dtype, st->gt_re.as<float>(), st->gt_cplx ? st->gt_im.as<float>() : nullptr, n));
        slice_sumsq_kernel<<<S, MON_THREADS, 0, ctx->stream>>>(st->gt_re.as<float>(), st->gt_cplx ? st->gt_im.as<float>() : nullptr,
                                                                op->plane(), st->gt2.as<double>());
        QLAUNCH_CHECK(ctx);
        QCUDA(cudaStreamSynchronize(ctx->stream));  // the host array may go away after this call
    }
    st->mon = gt ? 2 : 1;
    return QMRI_OK;
}

extern "C" int qmri_admm_history(qmri_admm* st, double* dc_res, double* gt_err, int* iters) {
    if (!st || !iters) return qmri_fail(QMRI_EINVAL, "qmri_admm_history: null argument");
    if (gt_err && !st->hist_has_gt)
        return qmri_fail(QMRI_EINVAL, "qmri_admm_history: gt_err asked for, but the last run had no ground truth (qmri_admm_monitor)");
    const int K = st->hist_iters, S = st->S;
    *iters = K;
    if (!K || (!dc_res && !gt_err)) return QMRI_OK;
    DevSetter ds(st->op->ctx->device);
    std::vector<double> h((size_t)K * S);
    for (int which = 0; which < 2; ++which) {
        double* out = which ? gt_err : dc_res;
        if (!out) continue;
        const DevBuf& b = which ? st->hist_gt : st->hist_dc;
        QCUDA(cudaMemcpyAsync(h.data(), b.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, st->op->ctx->stream));
        QCUDA(cudaStreamSynchronize(st->op->ctx->stream));
        for (int k = 0; k < K; ++k)  // device [k][s] -> MATLAB column-major iters x S
            for (int s = 0; s < S; ++s) out[k + (size_t)K * s] = h[(size_t)k * S + s];
    }
    return QMRI_OK;
}

// the monitor's arguments of one x-update (null when the session is not monitored)
static void admm_mon_params(const qmri_admm* st, K1Params& p) {
    if (!st->mon) return;
    p.mon_dc = st->mon_dc.as<double>();
    if (st->mon == 2) {
        p.mon_gt = st->mon_gt.as<double>();
        p.gt_re = st->gt_re.as<float>();
        p.gt_im = st->gt_cplx ? st->gt_im.as<float>() : nullptr;
    }
}

static int admm_mon_finalize(qmri_admm* st) {
    if (!st->mon) return QMRI_OK;
    qmri_op* op = st->op;
    // identity V: the solve kernel's partials are |y - A z|^2 and |y - A x| = rho / (1 + rho) |y - A z|; general V: |y - A x|^2
    const double f = op->general ? 1.0 : st->prm.gamma / (1.0 + st->prm.gamma);
    const int rows = (int)(st->hist_dc.bytes / (sizeof(double) * st->S));
    const int dc_n = op->general ? k1_general_residual_parts(op->g.nU) : op->C;
    monitor_finalize_kernel<<<1, MON_THREADS, 0, op->ctx->stream>>>(
        st->mon_dc.as<double>(), st->mon == 2 ? st->mon_gt.as<double>() : nullptr, st->y2.as<double>(), st->gt2.as<double>(),
        st->hist_ctr.as<int>(), st->hist_dc.as<double>(), st->mon == 2 ? st->hist_gt.as<double>() : nullptr, st->S, dc_n,
        op->C * st->mon_G, rows, f * f);
    QLAUNCH_CHECK(op->ctx);
    return QMRI_OK;
}

static int admm_k1(qmri_admm* st, bool write_x) {
    qmri_op* op = st->op;
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_ADMM;
    p.in_re = st->w_re.as<float>();
    p.in_im = st->w_im.as<float>();
    p.v = st->v.as<float>();
    p.out_re = st->w_re.as<float>();  // in place: every cluster reads its whole tile before it writes it
    p.out_im = st->w_im.as<float>();
    // general V with a ground truth: x is written on every iteration, and the launch that completes it sums |gt - x|^2
    write_x = write_x || (op->general && st->mon == 2);
    p.x_re = write_x ? st->x_re.as<float>() : nullptr;
    p.x_im = write_x ? st->x_im.as<float>() : nullptr;
    p.y = st->y.as<float2>();
    p.minmax = st->mm_ord.as<int>();
    p.inv_1p_rho = (float)(1.0 / (1.0 + st->prm.gamma));
    p.rho = st->prm.gamma;
    admm_mon_params(st, p);
    return k1_dispatch(op, p, st->S, &st->k1_part, &st->k1_cbuf);
}

// ---- real-state loop (xupdate_real.cu) ---------------------------------------------------------------------------------
// Opt-in (QMRI_K1_STATE=real) where the streaming kernels would run anyway (two slices or more), V is the identity and the mask
// fits the folded work-item tables.  Measured on B200 at 120 slices (profiles/r02_k1_real_vs_complex.md): the real kernels move 8
// (12 with the second read of v) instead of 24 bytes per pixel-channel and run half the FFT work, and take 3.20 instead of 4.13 us
// per slice-iteration - both families are bound by the sparse m-direction sums between two CTA barriers, not by bytes or FFT
// flops.  Counted against the 8 bytes it moves that is 0.19 of the HBM roofline (0.34 - 0.38 for the complex-state kernels at their
// 20), and the x-update is 0.6 % of the job: the complex-state kernels stay the default.
static bool admm_lean_eligible(const qmri_op* op, int S) {
    const char* env = getenv("QMRI_K1_STATE");
    if (!env || strcmp(env, "real")) return false;
    if (op->general || !op->t.stream_ok || !op->t.real_ok || op->k1_kernel == 1) return false;
    if (!k1r_fits(op->t.ns_max, op->t.r_n_ovf)) return false;
    return op->k1_kernel == 2 || (long long)S * op->C * K1_STREAM_MIN_IMAGES_DIV >= (long long)op->ctx->sm_count;
}

static void admm_lean_params(const qmri_admm* st, K1RealParams& p, int s0) {
    const qmri_op* op = st->op;
    const size_t ns = (size_t)op->t.ns_max, sc = (size_t)s0 * op->C * ns;
    p.y = st->y.as<float2>() + (size_t)s0 * op->t.nmeas;
    p.cstate = st->cstate.as<float2>() + sc;
    p.mprev = st->mprev.as<float2>() + sc;
    p.cbuf = st->k1_cbuf.as<float2>() + sc;
    p.part = st->k1_part.as<float2>();
    p.minmax = st->mm_ord.as<int>() + 2 * s0;
    p.frame_ptr = op->d_frame_ptr;
    p.tw2 = op->d_tw2;
    p.tw448 = op->d_tw448;
    p.itA = op->d_ritA;
    p.itB = op->d_ritB;
    p.ent = op->d_rent;
    p.rowmask = op->d_rrowmask;
    p.n_ovf = op->t.r_n_ovf;
    p.C = op->C;
    p.nmeas = op->t.nmeas;
    p.ns_max = op->t.ns_max;
    p.inv_1p_rho = (float)(1.0 / (1.0 + st->prm.gamma));
}

// steady state: out = v + Re(A^H c'), c' from the recurrence; slice groups keep v in L2 between the forward and adjoint kernels
static int admm_k1_lean(qmri_admm* st, const float* v, float* out) {
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    const size_t img = op->plane();
    const float half_inv_n = 0.5f / (float)op->N;
    for (int s0 = 0; s0 < st->S; s0 += st->lean_group) {
        const int sg = std::min(st->lean_group, st->S - s0);
        K1RealParams p = {};
        admm_lean_params(st, p, s0);
        p.v = v + (size_t)s0 * img;
        p.out = out + (size_t)s0 * img;
        p.G = k1r_groups(sg, op->C, ctx->sm_count);
        p.rec = 1;
        p.part_scale = half_inv_n;
        p.cbuf_scale = half_inv_n;
        QCHECK(k1r_forward(ctx, p, sg));
        QCHECK(k1r_solve(ctx, p, sg));
        QCHECK(k1r_adjoint(ctx, p, sg));
    }
    return QMRI_OK;
}

// first x-update (PnP_ADMM.m:102 with v = X0, u = 0): w_1 = X0 + A^H c_1, c_1 = (y - A X0) / (1 + rho); X0 is complex, so the
// complex streaming kernels do the transforms and the recurrence kernel keeps m_0 = A X0 and c_1
static int admm_k1_lean_first(qmri_admm* st) {
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_SOLVE;
    p.in_re = st->x0_re.as<float>();
    p.in_im = st->x0_im.as<float>();
    p.out_re = st->w_re.as<float>();
    p.out_im = st->w_im.as<float>();
    p.y = st->y.as<float2>();
    p.minmax = st->mm_ord.as<int>();
    p.inv_1p_rho = (float)(1.0 / (1.0 + st->prm.gamma));
    p.rho = st->prm.gamma;
    p.stage = K1_STAGE_FWD_ONLY | K1_STAGE_NO_SOLVE;
    QCHECK(k1_dispatch(op, p, st->S, &st->k1_part, &st->k1_cbuf));
    K1RealParams r = {};
    admm_lean_params(st, r, 0);
    r.G = k1_stream_groups(st->S, op->C, ctx->sm_count);  // the layout the complex forward kernel left in `part`
    r.rec = 0;
    r.part_scale = 1.0f / (float)op->N;
    r.cbuf_scale = 1.0f / (float)op->N;
    QCHECK(k1r_solve(ctx, r, st->S));
    p.stage = K1_STAGE_ADJ_ONLY;
    return k1_dispatch(op, p, st->S, &st->k1_part, &st->k1_cbuf);
}

// last x-update: the complex iterate x_K = 2 v_{K-1} - base + A^H (c_K - c_{K-1}), base = v_{K-2} (or X0 when K = 2)
static int admm_k1_lean_last(qmri_admm* st, const float* vcur, const float* base_re, const float* base_im) {
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    const size_t img = op->plane();
    for (int s0 = 0; s0 < st->S; s0 += st->lean_group) {
        const int sg = std::min(st->lean_group, st->S - s0);
        K1RealParams r = {};
        admm_lean_params(st, r, s0);
        r.v = vcur + (size_t)s0 * img;
        r.G = k1r_groups(sg, op->C, ctx->sm_count);
        r.rec = 2;
        r.part_scale = 0.5f / (float)op->N;
        r.cbuf_scale = 1.0f / (float)op->N;  // the complex inverse transform takes c as it is
        QCHECK(k1r_forward(ctx, r, sg));
        QCHECK(k1r_solve(ctx, r, sg));
    }
    QCHECK(k1r_last_base(ctx, vcur, base_re, base_im, st->x_re.as<float>(), st->x_im.as<float>(), img * st->S));
    K1Params p = {};
    k1_fill_tables(op, p);
    p.mode = K1_SOLVE;
    p.in_re = st->x_re.as<float>();
    p.in_im = st->x_im.as<float>();
    p.out_re = st->x_re.as<float>();  // in place: every thread reads the elements it writes
    p.out_im = st->x_im.as<float>();
    p.y = st->y.as<float2>();
    p.inv_1p_rho = (float)(1.0 / (1.0 + st->prm.gamma));
    p.rho = st->prm.gamma;
    p.stage = K1_STAGE_ADJ_ONLY;
    return k1_dispatch(op, p, st->S, &st->k1_part, &st->k1_cbuf);
}

static int admm_denoise(qmri_admm* st, float* v_out) {
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    const int S = st->S;
    const size_t hw = (size_t)op->N * op->M, n = op->plane() * S;
    const float* mm = st->mm_f.as<float>();
    if (st->prm.net) {
        // planes are MATLAB-ordered: rows = m (M of them), fastest extent = N
        return unetres_forward_dev(st->prm.net, st->w_re.as<float>(), v_out, mm,
                                   st->prm.multi_level ? st->noise.as<float>() : nullptr, S, op->M, op->N, 1);
    }
    // callback path: v_in = (Re w - min)/range [, noise map]; v = f(v_in) * range + min
    const int cin = st->prm.multi_level ? 11 : 10;
    float* vin = st->cb_in.as<float>();
    if (cin == 10) {
        QCHECK(normalize_planar(ctx, st->w_re.as<float>(), vin, mm, hw * 10, S, 0));
    } else {
        for (int s = 0; s < S; ++s) {
            QCHECK(normalize_planar(ctx, st->w_re.as<float>() + (size_t)s * hw * 10, vin + (size_t)s * hw * 11, mm + 2 * s, hw * 10, 1, 0));
            QCUDA(cudaMemcpyAsync(vin + (size_t)s * hw * 11 + hw * 10, st->noise.p, hw * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        }
    }
    int rc;
    if (st->prm.fn_space == QMRI_DEVICE) {
        rc = st->prm.fn(st->prm.user, vin, st->cb_out.as<float>(), op->N, op->M, cin, 10, S, QMRI_DEVICE, (void*)ctx->stream);
    } else {
        QCUDA(cudaMemcpyAsync(st->h_in, vin, hw * cin * S * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        rc = st->prm.fn(st->prm.user, st->h_in, st->h_out, op->N, op->M, cin, 10, S, QMRI_HOST, nullptr);
        if (rc == 0) QCUDA(cudaMemcpyAsync(st->cb_out.p, st->h_out, n * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (rc != 0) return qmri_fail(QMRI_ECALLBACK, "denoiser callback returned %d", rc);
    return normalize_planar(ctx, st->cb_out.as<float>(), v_out, mm, hw * 10, S, 1);
}

extern "C" int qmri_admm_run(qmri_admm* st, int iters) {
    if (!st) return qmri_fail(QMRI_EINVAL, "null state");
    if (!st->uploaded) return qmri_fail(QMRI_EINVAL, "qmri_admm_run: call qmri_admm_upload first");
    if (iters < 0) return qmri_fail(QMRI_EINVAL, "iters must be >= 0");
    qmri_op* op = st->op;
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    const int S = st->S;
    const size_t n = op->plane() * S;
    // x = v = X0, uold = 0 (PnP_ADMM.m:76-78); zero iterations return X0
    QCUDA(cudaMemcpyAsync(st->x_re.p, st->x0_re.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    QCUDA(cudaMemcpyAsync(st->x_im.p, st->x0_im.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    QCHECK(k1_minmax_init(ctx, st->mm_ord.as<int>(), S));
    st->hist_iters = st->mon ? iters : 0;
    st->hist_has_gt = st->mon == 2;
    if (st->mon) {  // history rows for this run, sized before any graph capture; row counter back to 0
        QCHECK(st->hist_dc.ensure((size_t)std::max(iters, 1) * S * sizeof(double)));
        if (st->mon == 2) QCHECK(st->hist_gt.ensure(st->hist_dc.bytes));
        if (st->y2_stale) {
            slice_sumsq_kernel<<<S, MON_THREADS, 0, ctx->stream>>>(reinterpret_cast<const float*>(st->y.p), nullptr,
                                                                    2 * (size_t)op->t.nmeas, st->y2.as<double>());
            QLAUNCH_CHECK(ctx);
            st->y2_stale = false;
        }
        QCUDA(cudaMemsetAsync(st->hist_ctr.p, 0, sizeof(int), ctx->stream));
    }
    // the real-state loop never forms x: a monitored session runs the complex-state loop
    const bool lean = st->lean && !st->mon;
    auto iteration = [&](int k) -> int {
        // real-state loop: the denoiser output of the second-to-last iteration goes to a second buffer, because the last
        // x-update needs v_{K-2} next to v_{K-1}
        float* v_out = (lean && k == iters - 2) ? st->v_alt.as<float>() : st->v.as<float>();
        if (k == 0 && lean) {
            QCHECK(admm_k1_lean_first(st));
            if (iters == 1) {  // x_1 is the result
                QCUDA(cudaMemcpyAsync(st->x_re.p, st->w_re.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
                QCUDA(cudaMemcpyAsync(st->x_im.p, st->w_im.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            }
        } else if (lean && k == iters - 1) {
            QCHECK(admm_k1_lean_last(st, st->v_alt.as<float>(), k == 1 ? st->x0_re.as<float>() : st->v.as<float>(),
                                     k == 1 ? st->x0_im.as<float>() : nullptr));
        } else if (lean) {
            QCHECK(admm_k1_lean(st, st->v.as<float>(), st->w_re.as<float>()));
        } else if (k == 0) {
            // Iteration 1 of PnP_ADMM.m:102 with v = X0, u = 0: x_1 = argmin |y - A x|^2 + rho |x - X0|^2, w_1 = x_1 + u_0 = x_1.
            // (For X0 = A^H y and A A^H = I this returns X0 itself - the reference driver's case - but param.X0 is the caller's.)
            K1Params p = {};
            k1_fill_tables(op, p);
            p.mode = K1_SOLVE;
            p.in_re = st->x0_re.as<float>();
            p.in_im = st->x0_im.as<float>();
            p.out_re = st->w_re.as<float>();
            p.out_im = st->w_im.as<float>();
            p.y = st->y.as<float2>();
            p.minmax = st->mm_ord.as<int>();
            p.inv_1p_rho = (float)(1.0 / (1.0 + st->prm.gamma));
            p.rho = st->prm.gamma;
            admm_mon_params(st, p);
            QCHECK(k1_dispatch(op, p, S, &st->k1_part, &st->k1_cbuf));
            if (iters == 1) {  // x_1 is the result
                QCUDA(cudaMemcpyAsync(st->x_re.p, st->w_re.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
                QCUDA(cudaMemcpyAsync(st->x_im.p, st->w_im.p, n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            }
        } else {
            QCHECK(admm_k1(st, k == iters - 1));
        }
        QCHECK(admm_mon_finalize(st));  // PnP_ADMM.m:106-109: row k of the history
        // PnP_ADMM.m:121-144 also denoise after the last x-update, but only x is returned (:148): v and u of the last iteration
        // are dead, so the final 64-layer forward is skipped
        if (k == iters - 1) return QMRI_OK;
        minmax_finalize_kernel<<<nblk(S, 128), 128, 0, ctx->stream>>>(st->mm_ord.as<int>(), st->mm_f.as<float>(), S);
        QLAUNCH_CHECK(ctx);
        return admm_denoise(st, v_out);
    };
    // Iterations 2 .. iters-2 launch the same kernels with the same arguments: capture one and replay it.  Iterations 0 and 1
    // run directly first, so every lazy initialisation (workspaces, tensor maps, function attributes) is done before capture.
    qmri_net* net = st->prm.net;
    const bool want_graph = net && !st->graph_failed && iters >= 6 && !getenv("QMRI_NO_GRAPH") && !getenv("QMRI_PROFILE") && !getenv("QMRI_TC_TRACE");
    for (int k = 0; k < iters; ++k) {
        if (!(want_graph && k >= 2 && k < iters - (lean ? 2 : 1))) {
            QCHECK(iteration(k));
            continue;
        }
        const int mon_key = st->mon | (st->mon == 2 && st->gt_cplx ? 4 : 0);
        if (st->graph && (st->graph_ws != net->ws || st->graph_chunk != net->chunk || st->graph_prec != net->precision ||
                          st->graph_mon != mon_key ||
                          (st->mon && (st->graph_hist[0] != st->hist_dc.p || st->graph_hist[1] != st->hist_gt.p ||
                                       st->graph_hist_bytes[0] != st->hist_dc.bytes || st->graph_hist_bytes[1] != st->hist_gt.bytes)))) {
            // the denoiser workspace moved or its mode changed since the capture, monitoring was switched, or the history moved
            cudaGraphExecDestroy(st->graph);
            st->graph = nullptr;
        }
        if (!st->graph) {
            const int64_t l0 = ctx->launches;
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
            int rc = QMRI_OK;
            if (e == cudaSuccess) {
                rc = iteration(k);
                e = cudaStreamEndCapture(ctx->stream, &g);
            }
            if (e == cudaSuccess && rc == QMRI_OK && g) e = cudaGraphInstantiate(&st->graph, g, 0);
            if (g) cudaGraphDestroy(g);
            if (e != cudaSuccess || rc != QMRI_OK || !st->graph) {
                cudaGetLastError();
                st->graph = nullptr;
                st->graph_failed = true;  // fall back to direct launches for the rest of this state's life
                fprintf(stderr, "libqmri_b200: warning: CUDA graph capture of the ADMM iteration failed (%s, rc %d); this session "
                                "continues with direct kernel launches (slower at small slice batches)\n",
                        e != cudaSuccess ? cudaGetErrorString(e) : "no error code", rc);
                ctx->launches = l0;
                QCHECK(iteration(k));
                for (++k; k < iters; ++k) QCHECK(iteration(k));
                return QMRI_OK;
            }
            st->graph_launches = ctx->launches - l0;
            ctx->launches = l0;
            st->graph_ws = net->ws;
            st->graph_chunk = net->chunk;
            st->graph_prec = net->precision;
            st->graph_mon = mon_key;
            st->graph_hist[0] = st->hist_dc.p;
            st->graph_hist[1] = st->hist_gt.p;
            st->graph_hist_bytes[0] = st->hist_dc.bytes;
            st->graph_hist_bytes[1] = st->hist_gt.bytes;
        }
        QCUDA(cudaGraphLaunch(st->graph, ctx->stream));
        ctx->launches += st->graph_launches;  // kernels inside the replayed graph
    }
    return QMRI_OK;
}

extern "C" int qmri_admm_xupdate_only(qmri_admm* st, int reps) {
    if (!st || !st->uploaded) return qmri_fail(QMRI_EINVAL, "qmri_admm_xupdate_only: state not ready");
    DevSetter ds(st->op->ctx->device);
    for (int i = 0; i < reps; ++i) {
        if (st->lean) QCHECK(admm_k1_lean(st, st->v.as<float>(), st->w_re.as<float>()));
        else QCHECK(admm_k1(st, false));
    }
    return QMRI_OK;
}

extern "C" int qmri_admm_xupdate_bytes(qmri_admm* st) { return st ? (st->lean ? 8 : 20) : 0; }

extern "C" int qmri_admm_download(qmri_admm* st, void* x_out, int x_dtype) {
    if (!st || !x_out) return qmri_fail(QMRI_EINVAL, "qmri_admm_download: null argument");
    if (!dtype_is_complex(x_dtype)) return qmri_fail(QMRI_EINVAL, "x must be complex");
    DevSetter ds(st->op->ctx->device);
    return image_download(st->op, x_out, x_dtype, st->S, st->x_re.as<float>(), st->x_im.as<float>());
}

extern "C" int qmri_admm_state_dev(qmri_admm* st, const float** x_re, const float** x_im) {
    if (!st) return qmri_fail(QMRI_EINVAL, "null state");
    if (x_re) *x_re = st->x_re.as<float>();
    if (x_im) *x_im = st->x_im.as<float>();
    return QMRI_OK;
}

extern "C" int qmri_pnp_admm(qmri_op* op, const void* y, int y_dtype, const void* x0, int x0_dtype, int S,
                             const qmri_admm_params* params, void* x_out, int x_dtype) {
    if (!params) return qmri_fail(QMRI_EINVAL, "qmri_pnp_admm: null params");
    qmri_admm* st = nullptr;
    QCHECK(qmri_admm_create(op, S, params, &st));
    int r = qmri_admm_upload(st, y, y_dtype, x0, x0_dtype);
    if (!r) r = qmri_admm_run(st, params->iters);
    if (!r) r = qmri_admm_download(st, x_out, x_dtype);
    qmri_admm_destroy(st);
    return r;
}

// ------------------------------------------------------------------------------------------
// dictionary matching
// ------------------------------------------------------------------------------------------
struct qmri_dict {
    qmri_ctx* ctx = nullptr;
    int64_t K = 0, a0 = 0, a1 = 0;
    int C = 0, CP = 0, Q = 0;
    float *Dp = nullptr, *normD = nullptr, *lut = nullptr;
    float* Dp_alloc = nullptr;  // what cudaMalloc returned; Dp = Dp_alloc - a0 * CP when only the shard's atoms are resident
    bool shard_only = false;    // D holds atoms [a0, a1) only: finish writes the pixels whose winner this handle owns, zeros elsewhere
    DevBuf stage, x_re, x_im, keys, qmap, pd, mt, dm;
    K2TcDict tc;          // tensor-pipe packing of the scored atoms (empty when C > 10 or the descriptor API is missing)
    bool tc_ok = false;
    DevBuf tc_stage;      // tf32-split pixel rows of the current call
};

static int dict_load(qmri_ctx* ctx, const float* D, const float* normD, const float* lut, int64_t K, int C, int Q,
                     int64_t shard_begin, int64_t shard_end, bool shard_only, qmri_dict** out) {
    if (!ctx || !D || !normD || !lut || !out) return qmri_fail(QMRI_EINVAL, "qmri_dict_load: null argument");
    if (K < 1 || K >= 0xFFFFFFFFll) return qmri_fail(QMRI_EINVAL, "dictionary size K = %lld out of range", (long long)K);
    if (C < 1 || C > 16) return qmri_fail(QMRI_EUNSUPPORTED, "dictionary matching supports 1..16 channels (got %d)", C);
    if (Q < 1) return qmri_fail(QMRI_EINVAL, "lut needs at least one column");
    if (shard_begin < 0 || shard_end > K || shard_begin >= shard_end) return qmri_fail(QMRI_EINVAL, "bad atom shard [%lld,%lld)", (long long)shard_begin, (long long)shard_end);
    DevSetter ds(ctx->device);
    qmri_dict* d = new qmri_dict();
    d->ctx = ctx;
    d->K = K; d->C = C; d->Q = Q; d->a0 = shard_begin; d->a1 = shard_end;
    d->CP = k2_padded_channels(C);
    d->shard_only = shard_only;
    // rows resident on this device: the whole dictionary, or atoms [a0, a1) only (D then holds just those rows)
    const int64_t R = shard_only ? shard_end - shard_begin : K;
    std::vector<float> Dp((size_t)R * d->CP, 0.f);
    for (int c = 0; c < C; ++c)
        for (int64_t k = 0; k < R; ++k) Dp[(size_t)k * d->CP + c] = D[(size_t)c * R + k];
    int r = dev_alloc(&d->Dp_alloc, Dp.size()) | dev_alloc(&d->normD, (size_t)K) | dev_alloc(&d->lut, (size_t)K * Q);
    if (r) {
        qmri_dict_destroy(d);
        return QMRI_ENOMEM;
    }
    // kernels index atoms globally: with a resident shard the base pointer is shifted so that row a0 is the first resident row
    // (rows outside [a0, a1) are never dereferenced: the scoring range is the shard and finish checks ownership)
    d->Dp = shard_only ? d->Dp_alloc - (ptrdiff_t)shard_begin * d->CP : d->Dp_alloc;
    cudaMemcpy(d->Dp_alloc, Dp.data(), Dp.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d->normD, normD, (size_t)K * 4, cudaMemcpyHostToDevice);
    cudaError_t e = cudaMemcpy(d->lut, lut, (size_t)K * Q * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        qmri_dict_destroy(d);
        return qmri_fail(QMRI_ECUDA, "dictionary upload failed: %s", cudaGetErrorString(e));
    }
    if (k2tc_supported(C)) {
        int rt = k2tc_dict_build(ctx, D, R, shard_only ? shard_begin : 0, C, shard_begin, shard_end, &d->tc);
        if (rt) {
            qmri_dict_destroy(d);
            return rt;
        }
        d->tc_ok = true;
    }
    *out = d;
    return QMRI_OK;
}
extern "C" int qmri_dict_load(qmri_ctx* ctx, const float* D, const float* normD, const float* lut, int64_t K, int C, int Q,
                              int64_t shard_begin, int64_t shard_end, qmri_dict** out) {
    return dict_load(ctx, D, normD, lut, K, C, Q, shard_begin, shard_end, false, out);
}
extern "C" int qmri_dict_load_shard(qmri_ctx* ctx, const float* D_shard, const float* normD, const float* lut, int64_t K, int C, int Q,
                                    int64_t shard_begin, int64_t shard_end, qmri_dict** out) {
    return dict_load(ctx, D_shard, normD, lut, K, C, Q, shard_begin, shard_end, true, out);
}
extern "C" int qmri_dict_destroy(qmri_dict* d) {
    if (!d) return QMRI_OK;
    DevSetter ds(d->ctx->device);
    cudaStreamSynchronize(d->ctx->stream);
    cudaFree(d->Dp_alloc); cudaFree(d->normD); cudaFree(d->lut);
    k2tc_dict_free(&d->tc);
    d->tc_stage.release();
    d->stage.release(); d->x_re.release(); d->x_im.release(); d->keys.release();
    d->qmap.release(); d->pd.release(); d->mt.release(); d->dm.release();
    delete d;
    return QMRI_OK;
}

extern "C" int qmri_match_keys_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, uint64_t* keys_dev) {
    if (!d || !x_re || !keys_dev) return qmri_fail(QMRI_EINVAL, "qmri_match_keys_dev: null argument");
    if (npix < 0) return qmri_fail(QMRI_EINVAL, "npix < 0");
    if (npix == 0) return QMRI_OK;
    DevSetter ds(d->ctx->device);
    QCUDA(cudaMemsetAsync(keys_dev, 0, (size_t)npix * 8, d->ctx->stream));
    K2Params p = {};
    p.x_re = x_re; p.x_im = x_im; p.npix = npix; p.Dp = d->Dp; p.a0 = d->a0; p.a1 = d->a1;
    p.keys = (unsigned long long*)keys_dev; p.C = d->C; p.CP = d->CP;
    // Pipe choice (profiles/r02_k2_pipes.md): the tcgen05 tf32 kernel from ~2000 atoms on, the FP32-FMA kernel for small
    // ranges and for C > 10; QMRI_K2_PIPE=fma|tensor forces one (tests, profiling).  Both produce the same keys.
    const char* pipe = getenv("QMRI_K2_PIPE");
    bool tensor = d->tc_ok && (d->a1 - d->a0) >= 2048;
    if (pipe && !strcmp(pipe, "fma")) tensor = false;
    if (pipe && !strcmp(pipe, "tensor")) {
        if (!d->tc_ok) return qmri_fail(QMRI_EUNSUPPORTED, "QMRI_K2_PIPE=tensor: this dictionary (C = %d) has no tensor-pipe packing", d->C);
        tensor = true;
    }
    if (tensor) {
        QCHECK(d->tc_stage.ensure(k2tc_stage_elems(npix) * sizeof(float)));
        return k2tc_launch_keys(d->ctx, d->tc, p, d->tc_stage.as<float>());
    }
    return k2_launch_keys(d->ctx, p);
}
extern "C" int qmri_match_finish_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, const uint64_t* keys_dev,
                                     float* qmap_dev, float* pd_dev, float* mt_dev, int32_t* dm_dev) {
    if (!d || !x_re || !keys_dev) return qmri_fail(QMRI_EINVAL, "qmri_match_finish_dev: null argument");
    if (npix <= 0) return npix == 0 ? QMRI_OK : qmri_fail(QMRI_EINVAL, "npix < 0");
    DevSetter ds(d->ctx->device);
    K2Finish f = {};
    f.x_re = x_re; f.x_im = x_im; f.npix = npix; f.Dp = d->Dp; f.normD = d->normD; f.lut = d->lut;
    f.K = d->K; f.C = d->C; f.CP = d->CP; f.Q = d->Q; f.keys = (const unsigned long long*)keys_dev;
    f.own0 = d->shard_only ? d->a0 : 0;
    f.own1 = d->shard_only ? d->a1 : d->K;
    f.qmap = qmap_dev; f.pd = pd_dev; f.mt = mt_dev; f.dm = dm_dev;
    return k2_launch_finish(d->ctx, f);
}
extern "C" int qmri_match_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, float* qmap_dev, float* pd_dev,
                              float* mt_dev, int32_t* dm_dev) {
    if (!d) return qmri_fail(QMRI_EINVAL, "null dict");
    if (npix <= 0) return npix == 0 ? QMRI_OK : qmri_fail(QMRI_EINVAL, "npix < 0");
    DevSetter ds(d->ctx->device);
    QCHECK(d->keys.ensure((size_t)npix * 8));
    QCHECK(qmri_match_keys_dev(d, x_re, x_im, npix, d->keys.as<uint64_t>()));
    return qmri_match_finish_dev(d, x_re, x_im, npix, d->keys.as<uint64_t>(), qmap_dev, pd_dev, mt_dev, dm_dev);
}
extern "C" int qmri_match(qmri_dict* d, const void* x, int x_dtype, int64_t npix, float* qmap, float* pd, float* mt, int32_t* dm) {
    if (!d || (!x && npix > 0)) return qmri_fail(QMRI_EINVAL, "qmri_match: null argument");
    if (npix < 0 || !valid_dtype(x_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_match: bad npix / dtype");
    if (npix == 0) return QMRI_OK;
    if (d->a0 != 0 || d->a1 != d->K || d->shard_only)
        return qmri_fail(QMRI_EINVAL, "qmri_match on an atom-sharded handle: use qmri_match_keys_dev + a max-reduction + qmri_match_finish_dev");
    qmri_ctx* ctx = d->ctx;
    DevSetter ds(ctx->device);
    const size_t n = (size_t)npix * d->C;
    const int cplx = dtype_is_complex(x_dtype);
    QCHECK(d->stage.ensure(n * dtype_size(x_dtype)));
    QCHECK(d->x_re.ensure(n * 4));
    if (cplx) QCHECK(d->x_im.ensure(n * 4));
    QCUDA(cudaMemcpyAsync(d->stage.p, x, n * dtype_size(x_dtype), cudaMemcpyHostToDevice, ctx->stream));
    QCHECK(unpack_async(ctx, d->stage.p, x_dtype, d->x_re.as<float>(), cplx ? d->x_im.as<float>() : nullptr, n));
    if (qmap) QCHECK(d->qmap.ensure((size_t)npix * d->Q * 4));
    if (pd) QCHECK(d->pd.ensure((size_t)npix * 8));
    if (mt) QCHECK(d->mt.ensure((size_t)npix * 4));
    if (dm) QCHECK(d->dm.ensure((size_t)npix * 4));
    QCHECK(qmri_match_dev(d, d->x_re.as<float>(), cplx ? d->x_im.as<float>() : nullptr, npix, qmap ? d->qmap.as<float>() : nullptr,
                          pd ? d->pd.as<float>() : nullptr, mt ? d->mt.as<float>() : nullptr, dm ? d->dm.as<int32_t>() : nullptr));
    if (qmap) QCUDA(cudaMemcpyAsync(qmap, d->qmap.p, (size_t)npix * d->Q * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (pd) QCUDA(cudaMemcpyAsync(pd, d->pd.p, (size_t)npix * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (mt) QCUDA(cudaMemcpyAsync(mt, d->mt.p, (size_t)npix * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (dm) QCUDA(cudaMemcpyAsync(dm, d->dm.p, (size_t)npix * 4, cudaMemcpyDeviceToHost, ctx->stream));
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

extern "C" int qmri_synthesize(qmri_dict* d, const float* qmap, int64_t npix, float* X, int32_t* atom_index) {
    if (!d || (npix > 0 && (!qmap || !X))) return qmri_fail(QMRI_EINVAL, "qmri_synthesize: null argument");
    if (npix < 0) return qmri_fail(QMRI_EINVAL, "npix < 0");
    if (d->Q < 2) return qmri_fail(QMRI_EINVAL, "qmri_synthesize needs dict.lut with (T1, T2) columns, got Q = %d", d->Q);
    if (d->shard_only) return qmri_fail(QMRI_EINVAL, "qmri_synthesize needs the whole dictionary resident (handle holds atoms [%lld,%lld) only)", (long long)d->a0, (long long)d->a1);
    if (npix == 0) return QMRI_OK;
    qmri_ctx* ctx = d->ctx;
    DevSetter ds(ctx->device);
    const size_t n = (size_t)npix;
    // stage: [T1 | T2 | PD] planes (the host array is npix x 3 column-major = exactly this), then X [C][npix]
    QCHECK(d->stage.ensure(n * 3 * 4));
    QCHECK(d->x_re.ensure(n * d->C * 4));
    QCHECK(d->keys.ensure(n * 8));
    QCHECK(d->dm.ensure(n * 4));
    QCUDA(cudaMemcpyAsync(d->stage.p, qmap, n * 3 * 4, cudaMemcpyHostToDevice, ctx->stream));
    K4Params p = {};
    p.t1 = d->stage.as<float>();
    p.t2 = p.t1 + n;
    p.pd = p.t1 + 2 * n;
    p.npix = npix;
    p.lut = d->lut; p.Dp = d->Dp; p.normD = d->normD;
    p.K = d->K; p.C = d->C; p.CP = d->CP;
    p.keys = d->keys.as<unsigned long long>();
    p.X = d->x_re.as<float>();
    p.index = atom_index ? d->dm.as<int32_t>() : nullptr;
    QCHECK(k4_launch(ctx, p));
    QCUDA(cudaMemcpyAsync(X, p.X, n * d->C * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (atom_index) QCUDA(cudaMemcpyAsync(atom_index, p.index, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

// ------------------------------------------------------------------------------------------
// the bare sampling matrix: P.for / P.adj (setup_subsampling_spiralgrided.m:36-42, setup_subsampling_epi.m:31-35)
// ------------------------------------------------------------------------------------------
static int p_matrix(qmri_op* op, PMatrix* P) {
    const size_t nm = std::max<size_t>((size_t)op->t.nmeas, 1);
    if (!op->p_idx.p) {
        QCHECK(op->p_idx.ensure(nm * sizeof(int32_t)));
        QCHECK(op->p_fp.ensure((size_t)(op->L + 1) * sizeof(int)));
        if (op->t.nmeas) QCUDA(cudaMemcpy(op->p_idx.p, op->t.idx.data(), (size_t)op->t.nmeas * sizeof(int32_t), cudaMemcpyHostToDevice));
        QCUDA(cudaMemcpy(op->p_fp.p, op->t.frame_ptr.data(), (size_t)(op->L + 1) * sizeof(int), cudaMemcpyHostToDevice));
        if (!op->hV.empty()) {
            QCHECK(op->p_V.ensure(op->hV.size() * sizeof(double)));
            QCUDA(cudaMemcpy(op->p_V.p, op->hV.data(), op->hV.size() * sizeof(double), cudaMemcpyHostToDevice));
        }
    }
    P->idx = op->p_idx.as<int32_t>();
    P->frame_ptr = op->p_fp.as<int>();
    P->V = op->hV.empty() ? nullptr : op->p_V.as<double>();
    P->L = op->L;
    P->C = op->C;
    P->NM = (int64_t)op->N * op->M;
    P->nmeas = op->t.nmeas;
    return QMRI_OK;
}

extern "C" int qmri_op_for(qmri_op* op, const void* kvec, int k_dtype, void* y, int y_dtype) {
    if (!op || !kvec || !y) return qmri_fail(QMRI_EINVAL, "qmri_op_for: null argument");
    if (!valid_dtype(k_dtype) || !dtype_is_complex(y_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_op_for: bad dtype (y must be complex)");
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    PMatrix P;
    QCHECK(p_matrix(op, &P));
    const size_t n = op->plane(), nm = (size_t)op->t.nmeas;
    QCHECK(op->p_k.ensure(2 * n * sizeof(double)));
    QCHECK(op->p_y.ensure(2 * std::max<size_t>(nm, 1) * sizeof(double)));
    QCHECK(op->p_stage.ensure(std::max(n * dtype_size(k_dtype), nm * dtype_size(y_dtype))));
    double *kr = op->p_k.as<double>(), *ki = kr + n, *yr = op->p_y.as<double>(), *yi = yr + std::max<size_t>(nm, 1);
    QCUDA(cudaMemcpyAsync(op->p_stage.p, kvec, n * dtype_size(k_dtype), cudaMemcpyHostToDevice, ctx->stream));
    QCHECK(aux_unpack_f64(ctx, op->p_stage.p, k_dtype, kr, ki, n));
    QCHECK(aux_p_for(ctx, P, kr, ki, yr, yi));
    if (nm) {
        QCHECK(aux_pack_f64(ctx, op->p_stage.p, y_dtype, yr, yi, nm));
        QCUDA(cudaMemcpyAsync(y, op->p_stage.p, nm * dtype_size(y_dtype), cudaMemcpyDeviceToHost, ctx->stream));
    }
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

extern "C" int qmri_op_adj(qmri_op* op, const void* y, int y_dtype, void* kvec, int k_dtype) {
    if (!op || !y || !kvec) return qmri_fail(QMRI_EINVAL, "qmri_op_adj: null argument");
    if (!valid_dtype(y_dtype) || !dtype_is_complex(k_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_op_adj: bad dtype (the k-space vector must be complex)");
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    PMatrix P;
    QCHECK(p_matrix(op, &P));
    const size_t n = op->plane(), nm = (size_t)op->t.nmeas;
    QCHECK(op->p_k.ensure(2 * n * sizeof(double)));
    QCHECK(op->p_y.ensure(2 * std::max<size_t>(nm, 1) * sizeof(double)));
    QCHECK(op->p_stage.ensure(std::max(n * dtype_size(k_dtype), nm * dtype_size(y_dtype))));
    double *kr = op->p_k.as<double>(), *ki = kr + n, *yr = op->p_y.as<double>(), *yi = yr + std::max<size_t>(nm, 1);
    if (nm) {
        QCUDA(cudaMemcpyAsync(op->p_stage.p, y, nm * dtype_size(y_dtype), cudaMemcpyHostToDevice, ctx->stream));
        QCHECK(aux_unpack_f64(ctx, op->p_stage.p, y_dtype, yr, yi, nm));
    }
    QCHECK(aux_p_adj(ctx, P, op->t.frame_ptr.data(), yr, yi, kr, ki));
    QCHECK(aux_pack_f64(ctx, op->p_stage.p, k_dtype, kr, ki, n));
    QCUDA(cudaMemcpyAsync(kvec, op->p_stage.p, n * dtype_size(k_dtype), cudaMemcpyDeviceToHost, ctx->stream));
    QCUDA(cudaStreamSynchronize(ctx->stream));
    return QMRI_OK;
}

// ------------------------------------------------------------------------------------------
// measurement noise (main_recon_tsmis_FFT.m:243)
// ------------------------------------------------------------------------------------------
extern "C" int qmri_awgn(qmri_ctx* ctx, void* y, int y_dtype, int64_t nmeas, int S, double snr_db, uint64_t seed) {
    if (!ctx || (!y && nmeas > 0 && S > 0)) return qmri_fail(QMRI_EINVAL, "qmri_awgn: null argument");
    if (!dtype_is_complex(y_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_awgn: measurements must be complex (QMRI_C64 / QMRI_C128)");
    if (nmeas < 0 || S < 0) return qmri_fail(QMRI_EINVAL, "qmri_awgn: negative size");
    if (nmeas == 0 || S == 0) return QMRI_OK;
    DevSetter ds(ctx->device);
    DevBuf raw, pw;
    const size_t bytes = (size_t)nmeas * S * dtype_size(y_dtype);
    int rc = raw.ensure(bytes);
    if (!rc) rc = pw.ensure((size_t)S * sizeof(double));
    auto body = [&]() -> int {
        QCUDA(cudaMemcpyAsync(raw.p, y, bytes, cudaMemcpyHostToDevice, ctx->stream));
        QCHECK(aux_awgn(ctx, raw.p, y_dtype, nmeas, S, snr_db, seed, pw.as<double>()));
        QCUDA(cudaMemcpyAsync(y, raw.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        return QMRI_OK;
    };
    if (!rc) rc = body();
    raw.release();
    pw.release();
    return rc;
}
extern "C" int qmri_awgn_dev(qmri_ctx* ctx, float* y_dev, int64_t nmeas, int S, double snr_db, uint64_t seed, double* power_dev) {
    if (!ctx || !y_dev || !power_dev) return qmri_fail(QMRI_EINVAL, "qmri_awgn_dev: null argument");
    if (nmeas < 0 || S < 0) return qmri_fail(QMRI_EINVAL, "qmri_awgn_dev: negative size");
    DevSetter ds(ctx->device);
    return aux_awgn(ctx, y_dev, QMRI_C64, nmeas, S, snr_db, seed, power_dev);
}

// ------------------------------------------------------------------------------------------
// foreground mask and metrics of the driver script (main_recon_tsmis_FFT.m:190-191, 328-384)
// ------------------------------------------------------------------------------------------
extern "C" int qmri_foreground_mask(qmri_ctx* ctx, const void* pd, int pd_dtype, int N, int M, double thresh, float* mask) {
    if (!ctx || !pd || !mask) return qmri_fail(QMRI_EINVAL, "qmri_foreground_mask: null argument");
    if (N < 1 || M < 1 || !valid_dtype(pd_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_foreground_mask: bad size / dtype");
    DevSetter ds(ctx->device);
    const size_t n = (size_t)N * M;
    DevBuf raw, pl, sc;
    int rc = raw.ensure(n * 16);
    if (!rc) rc = pl.ensure(4 * n * sizeof(double));  // re, im, |pd|, mask
    if (!rc) rc = sc.ensure(2 * n);
    auto body = [&]() -> int {
        double *re = pl.as<double>(), *im = re + n, *ab = im + n, *mk = ab + n;
        QCUDA(cudaMemcpyAsync(raw.p, pd, n * dtype_size(pd_dtype), cudaMemcpyHostToDevice, ctx->stream));
        QCHECK(aux_unpack_f64(ctx, raw.p, pd_dtype, re, im, n));
        QCHECK(aux_abs_scale(ctx, re, dtype_is_complex(pd_dtype) ? im : nullptr, nullptr, nullptr, ab, n));
        QCHECK(aux_foreground_mask(ctx, ab, N, M, thresh, mk, sc.as<unsigned char>()));
        QCHECK(aux_pack_f64(ctx, raw.p, QMRI_F32, mk, nullptr, n));
        QCUDA(cudaMemcpyAsync(mask, raw.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        return QMRI_OK;
    };
    if (!rc) rc = body();
    raw.release(); pl.release(); sc.release();
    return rc;
}

extern "C" int qmri_recon_metrics(qmri_ctx* ctx, int N, int M, int C, const void* qmap, int qmap_dtype, const void* qmap0, int qmap0_dtype,
                                  const float* mask, const void* X, int x_dtype, const void* X0, int x0_dtype, double* out) {
    if (!ctx || !qmap || !qmap0 || !out) return qmri_fail(QMRI_EINVAL, "qmri_recon_metrics: null argument");
    if ((X == nullptr) != (X0 == nullptr)) return qmri_fail(QMRI_EINVAL, "qmri_recon_metrics: pass both X and X0 or neither");
    if (N < 1 || M < 1 || C < 0 || C > 1000 || !valid_dtype(qmap_dtype) || !valid_dtype(qmap0_dtype) || (X && (!valid_dtype(x_dtype) || !valid_dtype(x0_dtype))))
        return qmri_fail(QMRI_EINVAL, "qmri_recon_metrics: bad size / dtype");
    DevSetter ds(ctx->device);
    const size_t n = (size_t)N * M;
    const int nch = X ? C : 0, npairs = 3 + nch;
    const size_t big = std::max<size_t>(3, (size_t)nch) * n;
    DevBuf raw, wk, pa, pb, part, res;
    int rc = raw.ensure(big * 16);
    if (!rc) rc = wk.ensure((2 * big + n + 2) * sizeof(double));  // re, im planes of the array being converted, mask, two maxima
    if (!rc) rc = pa.ensure((size_t)npairs * n * sizeof(double));
    if (!rc) rc = pb.ensure((size_t)npairs * n * sizeof(double));
    if (!rc) rc = part.ensure(aux_pair_metrics_partial_elems(npairs, N, M) * sizeof(double));
    if (!rc) rc = res.ensure((size_t)npairs * 3 * sizeof(double));
    auto body = [&]() -> int {
        double *re = wk.as<double>(), *im = re + big, *mk = im + big, *mx = mk + n;
        double *A = pa.as<double>(), *B = pb.as<double>();
        const double* mkp = nullptr;
        if (mask) {
            QCUDA(cudaMemcpyAsync(raw.p, mask, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
            QCHECK(aux_unpack_f64(ctx, raw.p, QMRI_F32, mk, nullptr, n));
            mkp = mk;
        }
        // side 0 = estimate (qmap, X), side 1 = reference (qmap0, X0)
        for (int side = 0; side < 2; ++side) {
            const void* q = side ? qmap0 : qmap;
            const int qd = side ? qmap0_dtype : qmap_dtype;
            double* dst = side ? B : A;
            QCUDA(cudaMemcpyAsync(raw.p, q, 3 * n * dtype_size(qd), cudaMemcpyHostToDevice, ctx->stream));
            QCHECK(aux_unpack_f64(ctx, raw.p, qd, re, im, 3 * n));
            // t1 = qmap(:,:,1) .* mask, t2 likewise (:330-333): MAE / PSNR / SSIM compare the real parts
            QCUDA(cudaMemcpyAsync(dst, re, 2 * n * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
            if (mkp) QCHECK(aux_mul_mask(ctx, dst, mkp, n, 2));
            // pd = |qmap(:,:,3) .* mask| / max(|.|)  (:334-337)
            QCHECK(aux_abs_scale(ctx, re + 2 * n, dtype_is_complex(qd) ? im + 2 * n : nullptr, mkp, nullptr, dst + 2 * n, n));
            QCHECK(aux_absmax(ctx, dst + 2 * n, n, mx + side));
            QCHECK(aux_abs_scale(ctx, dst + 2 * n, nullptr, nullptr, mx + side, dst + 2 * n, n));
            if (nch) {  // psnr / ssim of abs(X(:,:,c)) against abs(X0(:,:,c)), no mask (:355-369)
                const void* x = side ? X0 : X;
                const int xd = side ? x0_dtype : x_dtype;
                QCUDA(cudaMemcpyAsync(raw.p, x, (size_t)nch * n * dtype_size(xd), cudaMemcpyHostToDevice, ctx->stream));
                QCHECK(aux_unpack_f64(ctx, raw.p, xd, re, im, (size_t)nch * n));
                QCHECK(aux_abs_scale(ctx, re, dtype_is_complex(xd) ? im : nullptr, nullptr, nullptr, dst + 3 * n, (size_t)nch * n));
            }
        }
        QCHECK(aux_pair_metrics(ctx, A, B, mkp, npairs, N, M, part.as<double>(), res.as<double>()));
        std::vector<double> h((size_t)npairs * 3);
        QCUDA(cudaMemcpyAsync(h.data(), res.p, h.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        // out: tsmi_mean_psnr, tsmi_mean_ssim, t1_{mae,psnr,ssim}, t2_{...}, pd_{...}  (the script's print order, :372-379)
        double ps = 0.0, ss = 0.0;
        for (int c = 0; c < nch; ++c) {
            ps += h[(size_t)(3 + c) * 3 + 1];
            ss += h[(size_t)(3 + c) * 3 + 2];
        }
        out[0] = nch ? ps / nch : NAN;
        out[1] = nch ? ss / nch : NAN;
        for (int k = 0; k < 9; ++k) out[2 + k] = h[k];
        return QMRI_OK;
    };
    if (!rc) rc = body();
    raw.release(); wk.release(); pa.release(); pb.release(); part.release(); res.release();
    return rc;
}

// ------------------------------------------------------------------------------------------
// LRTV baseline: FISTA with a total-variation prox (main_files/algorithms/LRTV/FISTA_deep.m:31-103,
// unlocbox/prox/prox_tv.m:100-193; called at main_recon_tsmis_FFT.m:272-282)
// ------------------------------------------------------------------------------------------
namespace {
struct LrtvWork {
    qmri_op* op;
    qmri_ctx* ctx;
    size_t n;         // N M L
    size_t n2;        // stacked image: 2N x (M L)
    int R, Cc;
    DevBuf dbl, flt, ybuf, fx, part, sums;
    double *xr, *xi, *x2r, *x2i, *pr, *pi, *b, *r, *s, *po, *qo, *sol;
    float *fr, *fi, *gr, *gi;
    double h[4];
    int sync_sums() {
        QCUDA(cudaMemcpyAsync(h, sums.p, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        return QMRI_OK;
    }
    // fx = F.forward(planes)
    int forward(const float* re, const float* im) {
        K1Params p = {};
        k1_fill_tables(op, p);
        p.mode = K1_FORWARD;
        p.in_re = re; p.in_im = im;
        p.y_out = fx.as<float2>();
        return k1_dispatch(op, p, 1);
    }
    int adjoint(const float2* y, float* re, float* im) {
        K1Params p = {};
        k1_fill_tables(op, p);
        p.mode = K1_ADJOINT;
        p.y = y;
        p.out_re = re; p.out_im = im;
        return k1_dispatch(op, p, 1);
    }
    // prox_tv on x2 (in place); tv_tol / tv_maxit = the toolbox defaults the reference leaves untouched
    int prox_tv(double gamma, double tol, int maxit) {
        if (gamma == 0.0) return QMRI_OK;
        const int N = op->N;
        QCHECK(lrtv_stack(ctx, x2r, x2i, N, Cc, b));
        QCUDA(cudaMemsetAsync(r, 0, n2 * sizeof(double) * 4, ctx->stream));  // r, s, pold, qold are contiguous
        double told = 1.0, prev_obj = 0.0;
        for (int it = 1; it <= maxit; ++it) {
            const double t = (1.0 + sqrt(4.0 * told * told)) / 2.0;
            QCHECK(lrtv_tv_sol(ctx, b, r, s, gamma, R, Cc, sol, part.as<double>(), sums.as<double>()));
            QCHECK(lrtv_tv_update(ctx, sol, r, s, po, qo, gamma, (told - 1.0) / t, R, Cc, part.as<double>(), sums.as<double>()));
            QCHECK(sync_sums());
            const double obj = 0.5 * h[0] + gamma * h[1];
            const double rel = fabs(obj - prev_obj) / obj;
            prev_obj = obj;
            if (rel < tol) break;   // the dual update launched above is simply not used
            told = t;
        }
        return lrtv_unstack(ctx, sol, N, Cc, x2r, x2i);
    }
};
}  // namespace

extern "C" int qmri_lrtv(qmri_op* op, const void* y, int y_dtype, const qmri_lrtv_params* prm, void* x_out, int x_dtype, int* iters_done,
                         double* final_step) {
    if (!op || !y || !prm || !x_out) return qmri_fail(QMRI_EINVAL, "qmri_lrtv: null argument");
    if (!dtype_is_complex(y_dtype) || !dtype_is_complex(x_dtype)) return qmri_fail(QMRI_EINVAL, "qmri_lrtv: y and x must be complex");
    if (prm->iters < 0 || !(prm->step > 0.0) || prm->K < 0.0) return qmri_fail(QMRI_EINVAL, "qmri_lrtv: need iter >= 0, step > 0, K >= 0");
    qmri_ctx* ctx = op->ctx;
    DevSetter ds(ctx->device);
    LrtvWork w;
    w.op = op; w.ctx = ctx;
    w.n = op->plane();
    w.R = 2 * op->N;
    w.Cc = op->M * op->C;
    w.n2 = (size_t)w.R * w.Cc;
    const size_t nm = std::max<size_t>((size_t)op->t.nmeas, 1);
    int rc = w.dbl.ensure((6 * w.n + 6 * w.n2) * sizeof(double));
    if (!rc) rc = w.flt.ensure(4 * w.n * sizeof(float));
    if (!rc) rc = w.fx.ensure(nm * sizeof(float2));
    if (!rc) rc = w.part.ensure(lrtv_partial_elems(w.n2) * sizeof(double));
    if (!rc) rc = w.sums.ensure(4 * sizeof(double));
    auto body = [&]() -> int {
        double* d = w.dbl.as<double>();
        w.xr = d; w.xi = d + w.n; w.x2r = d + 2 * w.n; w.x2i = d + 3 * w.n; w.pr = d + 4 * w.n; w.pi = d + 5 * w.n;
        d += 6 * w.n;
        w.b = d; w.r = d + w.n2; w.s = d + 2 * w.n2; w.po = d + 3 * w.n2; w.qo = d + 4 * w.n2; w.sol = d + 5 * w.n2;
        float* f = w.flt.as<float>();
        w.fr = f; w.fi = f + w.n; w.gr = f + 2 * w.n; w.gi = f + 3 * w.n;
        QCHECK(y_upload(op, y, y_dtype, 1));
        const float2* yd = op->ybuf.as<float2>();
        QCUDA(cudaMemsetAsync(w.dbl.p, 0, 6 * w.n * sizeof(double), ctx->stream));   // x = 0, x2_prev = 0
        QCUDA(cudaMemsetAsync(w.flt.p, 0, 2 * w.n * sizeof(float), ctx->stream));
        QCUDA(cudaMemsetAsync(w.sums.p, 0, 4 * sizeof(double), ctx->stream));
        double step = prm->step, obj_prev = 0.0;
        const double tv_tol = prm->tv_tol > 0.0 ? prm->tv_tol : 10e-4;
        const int tv_maxit = prm->tv_maxit > 0 ? prm->tv_maxit : 200;
        int it = 0;
        for (it = 1; it <= prm->iters; ++it) {
            // err = F.forward(x) - y; grad1 = F.adjoint(err); cvxobj = |err|^2 / 2; val = |x|_TV          (FISTA_deep.m:55-62)
            QCHECK(w.forward(w.fr, w.fi));
            QCHECK(lrtv_residual(ctx, w.fx.as<float2>(), yd, (size_t)op->t.nmeas, w.part.as<double>(), w.sums.as<double>(), 2));
            QCHECK(w.adjoint(w.fx.as<float2>(), w.gr, w.gi));
            QCHECK(lrtv_stack(ctx, w.xr, w.xi, op->N, w.Cc, w.b));
            QCHECK(lrtv_norm_tv(ctx, w.b, w.R, w.Cc, w.part.as<double>(), w.sums.as<double>(), 3));
            QCHECK(w.sync_sums());
            const double cvxobj = 0.5 * w.h[2], val = w.h[3];
            for (;;) {                                                                                   // :66-88
                QCHECK(lrtv_grad_step(ctx, w.xr, w.xi, w.gr, w.gi, step, w.n, w.x2r, w.x2i));
                if (prm->K > 0.0) QCHECK(w.prox_tv(step * prm->K, tv_tol, tv_maxit));
                if (!prm->backtrack) break;
                // tmp = |F.forward(x2) - y|^2 / 2
                DevBuf& tmpf = op->a_re;  // scratch planes of the operator's host entry points
                QCHECK(tmpf.ensure(2 * w.n * sizeof(float)));
                float* tr = tmpf.as<float>();
                float* ti = tr + w.n;
                QCHECK(lrtv_to_float(ctx, w.x2r, w.x2i, w.n, tr, ti));
                QCHECK(w.forward(tr, ti));
                QCHECK(lrtv_residual(ctx, w.fx.as<float2>(), yd, (size_t)op->t.nmeas, w.part.as<double>(), w.sums.as<double>(), 2));
                QCHECK(lrtv_backtrack_terms(ctx, w.xr, w.xi, w.x2r, w.x2i, w.gr, w.gi, w.n, w.part.as<double>(), w.sums.as<double>()));
                QCHECK(w.sync_sums());
                const double tmp = 0.5 * w.h[2];
                if (tmp > cvxobj + w.h[0] + w.h[1] / (2.0 * step)) step *= 0.5;  // 'reducing stepsize...'
                else break;
            }
            // x = x2 + (t-1)/(t+2) (x2 - x2_prev)                                                       (:90-93)
            QCHECK(lrtv_momentum(ctx, w.xr, w.xi, w.x2r, w.x2i, w.pr, w.pi, (double)(it - 1) / (double)(it + 2), w.n, w.fr, w.fi));
            const double obj = cvxobj + prm->K * val;
            if (fabs(obj - obj_prev) / obj < prm->tol) break;                                            // :98
            obj_prev = obj;
        }
        if (iters_done) *iters_done = std::min(it, prm->iters);
        if (final_step) *final_step = step;
        // the loop's x (after the momentum step, :90) is what FISTA_deep returns
        QCHECK(op->stage.ensure(w.n * dtype_size(x_dtype)));
        QCHECK(aux_pack_f64(ctx, op->stage.p, x_dtype, w.xr, w.xi, w.n));
        QCUDA(cudaMemcpyAsync(x_out, op->stage.p, w.n * dtype_size(x_dtype), cudaMemcpyDeviceToHost, ctx->stream));
        QCUDA(cudaStreamSynchronize(ctx->stream));
        return QMRI_OK;
    };
    if (!rc) rc = body();
    w.dbl.release(); w.flt.release(); w.fx.release(); w.part.release(); w.sums.release();
    return rc;
}
