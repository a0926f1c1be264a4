// K1 "real" variant - the x-update of the PnP-ADMM loop with only REAL images crossing HBM (sm_100a).
//
// Reference being replaced: main_files/algorithms/PnP_ADMM/PnP_ADMM.m:102-103 (lsqr x-update), :115-118 (v = real(x + u)),
// :121 (global min / max), :144 (u += x - v), F of main_recon_tsmis_FFT.m:228-229 - for A A^H = I (V = eye).
//
// State reformulation (SURVEY.md 7.3-3, verified there to 4e-15 against the literal loop).  With w_k = x_k + u_{k-1}:
//   w_{k+1} = v_k + A^H c_{k+1},     c_{k+1} = (y - 2 m_k + m_{k-1} + c_k) / (1 + rho),     m_k = A v_k
// (A z_{k+1} = A (2 v_k - w_k) = 2 m_k - m_{k-1} - c_k because A A^H = I), started from m_0 = A X0, c_1 = (y - m_0) / (1 + rho).
// c and m live on the <= ~700 sampled k-space locations of a channel (5 KB); the only images the loop touches are the denoiser's
// output v_k (real) and its next input Re w_{k+1} = v_k + Re(A^H c_{k+1}): 8 bytes per pixel-channel per iteration instead of the 20
// of the complex-state form (read w 8 + v 4, write w' 8).  The complex iterate is materialised once, after the last iteration:
//   x_K = 2 v_{K-1} - v_{K-2} + A^H (c_K - c_{K-1})              (qmri_api.cu, through the complex streaming kernels).
// Real images also halve the transforms: two real columns ride through one complex length-224 FFT (xupdate_phases.cuh).
//
//   stream_fwdr_kernel   grid (G, C, S): 224 / G real columns of one image, 28 at a time: global -> registers (column pairs) ->
//                        FFT along n -> sampled DFT along m over folded rows; partial sample sums -> `part`
//   stream_solver_kernel grid (C, S): m_k from the G partials in a fixed order, the recurrence for c, m_{k-1} <- m_k, and the
//                        pre-scaled input of the inverse transform
//   stream_adjr_kernel   grid (G, C, S): sparse inverse DFT along m (Hermitian-packed) -> inverse FFT along n -> registers ->
//                        out = v + Re(corr) -> global; per-slice min / max by ordered-int atomics
// HBM traffic per pixel-channel: read v (4 B) in the forward kernel, read v again (4 B, from L2 when the caller runs the three
// kernels on slice groups that fit the L2) and write Re w' (4 B) in the adjoint kernel.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "xupdate_kernel.h"
#include "xupdate_phases.cuh"

using namespace k1;

namespace {

constexpr int PC = 14;                // packed (complex) columns per slab = 28 real columns
constexpr int THREADS = 16 * PC;      // 224
constexpr int SLABS = NF / (2 * PC);  // 8 slabs per image

__device__ __forceinline__ size_t late_offset(size_t off, float after) {
    size_t r;
    asm volatile("mov.u64 %0, %1;" : "=l"(r) : "l"(off), "f"(after));
    return r;
}

// ---------------- forward: partial sums of 2 A v over a group of slabs -------------------------------------
__global__ void __launch_bounds__(THREADS, 4) stream_fwdr_kernel(K1RealParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ws = reinterpret_cast<float2*>(smem_raw);                  // [PC][CS] slab workspace
    float2* tw2 = ws + PC * CS;                                        // [16][16]
    float2* tw448 = tw2 + 256;                                         // [448]
    float2* pc = tw448 + 2 * NF;                                       // [ns_max] sample accumulators
    uint32_t* s_ent = reinterpret_cast<uint32_t*>(pc + p.ns_max);      // [ns_max]

    const int tid = threadIdx.x;
    const int g = blockIdx.x, c = blockIdx.y, s = blockIdx.z;
    const int f0 = p.frame_ptr[c];
    const int ns = p.frame_ptr[c + 1] - f0;
    const size_t img = ((size_t)s * p.C + c) * (size_t)(NF * NF);

    for (int i = tid; i < 256; i += THREADS) tw2[i] = p.tw2[i];
    for (int i = tid; i < 2 * NF; i += THREADS) tw448[i] = p.tw448[i];
    for (int i = tid; i < ns; i += THREADS) {
        s_ent[i] = p.ent[f0 + i];
        pc[i] = make_float2(0.f, 0.f);
    }
    const uint32_t itA = p.itA[(size_t)c * NF + tid];
    const int l16 = tid & 15;
    const int col = tid >> 4;
    float2* colp = ws + col * CS;
    __syncthreads();

    const int slab0 = g * p.slabs_per_cta;
#pragma unroll 1
    for (int sl = 0; sl < p.slabs_per_cta; ++sl) {
        const int m0 = (slab0 + sl) * (2 * PC);
        {
            const size_t gi = img + (size_t)(m0 + 2 * col) * NF + l16;
            float2 a[16];
#pragma unroll
            for (int n1 = 0; n1 < 14; ++n1) a[n1] = make_float2(__ldg(p.v + gi + 16 * n1), __ldg(p.v + gi + NF + 16 * n1));
            fwd_s1_regs(a, l16, tw2);
            fft_s1_store(colp, l16, a);
            __syncwarp();
            if (l16 < 14) fft_s2_load(colp, l16, a);
            __syncwarp();
            if (l16 < 14) fft_s2_store<false>(colp, l16, a);
        }
        __syncthreads();
        p3r_item(ws, (int)(itA & 0xffu), s_ent + (itA >> 16), (int)((itA >> 8) & 0xffu), tw448, m0, pc);
        __syncthreads();
    }
    // every sample belongs to exactly one work item, i.e. to one thread: no race on pc above
    float2* part = p.part + (((size_t)s * p.C + c) * p.G + g) * (size_t)p.ns_max;
    for (int j = tid; j < ns; j += THREADS) part[j] = pc[j];
}

// ---------------- the recurrence on the samples ----------------------------------------------------------------
//   rec 0 (first x-update, from the complex forward transform of X0):  m = A X0,  c = (y - m) / (1 + rho)
//   rec 1 (steady state):                                              c = (y - 2 m + m_prev + c) / (1 + rho)
//   rec 2 (last x-update): as rec 1, but the inverse transform gets c_new - c_old (x_K = 2 v_{K-1} - v_{K-2} + A^H (c_K - c_{K-1}))
__global__ void __launch_bounds__(256) stream_solver_kernel(K1RealParams p) {
    const int c = blockIdx.x, s = blockIdx.y;
    const int f0 = p.frame_ptr[c];
    const int ns = p.frame_ptr[c + 1] - f0;
    const size_t sc = (size_t)s * p.C + c;
    const float2* part = p.part + sc * p.G * (size_t)p.ns_max;
    for (int j = threadIdx.x; j < ns; j += blockDim.x) {
        float sx = 0.f, sy = 0.f;
#pragma unroll 1
        for (int g0 = 0; g0 < p.G; g0 += 4) {  // fixed order: deterministic; four loads in flight
            float2 t[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] = g0 + i < p.G ? part[(size_t)(g0 + i) * p.ns_max + j] : make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                sx += t[i].x;
                sy += t[i].y;
            }
        }
        const float mx = sx * p.part_scale, my = sy * p.part_scale;
        const float2 y = p.y[(size_t)s * p.nmeas + f0 + j];
        const size_t si = sc * p.ns_max + j;
        float cx, cy, ox = 0.f, oy = 0.f;
        if (p.rec == 0) {
            cx = (y.x - mx) * p.inv_1p_rho;
            cy = (y.y - my) * p.inv_1p_rho;
        } else {
            const float2 mp = p.mprev[si], co = p.cstate[si];
            ox = co.x;
            oy = co.y;
            cx = (y.x - 2.f * mx + mp.x + co.x) * p.inv_1p_rho;
            cy = (y.y - 2.f * my + mp.y + co.y) * p.inv_1p_rho;
        }
        p.cstate[si] = make_float2(cx, cy);
        p.mprev[si] = make_float2(mx, my);
        if (p.rec == 2) p.cbuf[si] = make_float2((cx - ox) * p.cbuf_scale, (cy - oy) * p.cbuf_scale);
        else p.cbuf[si] = make_float2(cx * p.cbuf_scale, cy * p.cbuf_scale);
    }
}

// ---------------- adjoint: out = v + Re(A^H c), epilogue ----------------------------------------------------------
__global__ void __launch_bounds__(THREADS, 4) stream_adjr_kernel(K1RealParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ws = reinterpret_cast<float2*>(smem_raw);                  // [PC][CS]
    float2* tw2 = ws + PC * CS;                                        // [16][16]
    float2* tw448 = tw2 + 256;                                         // [448]
    float2* pc = tw448 + 2 * NF;                                       // [ns_max] c
    float2* ovf = pc + p.ns_max;                                       // [n_ovf][2 half slabs][OVF_STRIDE] overflow partials
    uint32_t* s_ent = reinterpret_cast<uint32_t*>(ovf + (size_t)p.n_ovf * 2 * OVF_STRIDE);  // [ns_max]
    __shared__ float red_min[THREADS / 32], red_max[THREADS / 32];

    const int tid = threadIdx.x;
    const int g = blockIdx.x, c = blockIdx.y, s = blockIdx.z;
    const int f0 = p.frame_ptr[c];
    const int ns = p.frame_ptr[c + 1] - f0;
    const size_t img = ((size_t)s * p.C + c) * (size_t)(NF * NF);

    for (int i = tid; i < 256; i += THREADS) tw2[i] = p.tw2[i];
    for (int i = tid; i < 2 * NF; i += THREADS) tw448[i] = p.tw448[i];
    for (int i = tid; i < ns; i += THREADS) {
        s_ent[i] = p.ent[f0 + i];
        pc[i] = p.cbuf[((size_t)s * p.C + c) * p.ns_max + i];
    }
    const uint32_t itA = p.itA[(size_t)c * NF + tid], itB = p.itB[(size_t)c * NF + tid];
    const int it_k1 = (int)(itA & 0xffu), it_cnt = (int)((itA >> 8) & 0xffu), it_start = (int)(itA >> 16);
    const int it_slot = (int)(itB & 0xffu), it_novf = (int)((itB >> 8) & 0xffu), it_ovf0 = (int)((itB >> 16) & 0xffu);
    const int l16 = tid & 15;
    const uint32_t rmask = p.rowmask[c * 16 + l16];
    const int col = tid >> 4;
    float2* colp = ws + col * CS;
    __syncthreads();

    float lmin = INFINITY, lmax = -INFINITY;
    const int slab0 = g * p.slabs_per_cta;
#pragma unroll 1
    for (int sl = 0; sl < p.slabs_per_cta; ++sl) {
        const int m0 = (slab0 + sl) * (2 * PC);
        const size_t gi = img + (size_t)(m0 + 2 * col) * NF + l16;
        if (it_cnt != 0) {
#pragma unroll 1
            for (int h = 0; h < 2; ++h) {
                float2 SP[NP_STREAM], SM[NP_STREAM];
                p4r_item_partial(SP, SM, s_ent + it_start, it_cnt, tw448, m0 + 14 * h, pc);
                if (it_slot == 0) p4r_store<false>(ws, it_k1, h, SP, SM);
                else p4_item_spill(ovf + ((size_t)(it_slot - 1) * 2 + h) * OVF_STRIDE, SP, SM);
            }
        }
        if (p.n_ovf) {
            __syncthreads();
            if (it_cnt != 0 && it_slot == 0 && it_novf) {
                // consecutive overflow slots of a row are 2 * OVF_STRIDE apart (the two half slabs interleave)
#pragma unroll 1
                for (int h = 0; h < 2; ++h) p4r_row_add_overflow(ws, it_k1, h, ovf + ((size_t)it_ovf0 * 2 + h) * OVF_STRIDE, it_novf, 2 * OVF_STRIDE);
            }
        }
        __syncthreads();
        {
            float2 a[16];
            if (l16 < 14) inv_s1_load(colp, l16, tw2, rmask, a);
            __syncwarp();
            if (l16 < 14) inv_s1_store(colp, l16, a);
            __syncwarp();
            inv_s2_regs(colp, l16, a);
            // a[d] = (column m0 + 2 col, column m0 + 2 col + 1) of Re(A^H c) at n = l16 + 16 d.  The offset of the v loads is
            // made to depend on the transform's last output so that they are not hoisted above it (held across it they spill).
            const size_t gl = late_offset(gi, a[13].y);
            float b[14];
#pragma unroll
            for (int d = 0; d < 14; ++d) b[d] = __ldg(p.v + gl + 16 * d);
#pragma unroll
            for (int d = 0; d < 14; ++d) {
                const float o = b[d] + a[d].x;
                p.out[gi + 16 * d] = o;
                lmin = fminf(lmin, o);
                lmax = fmaxf(lmax, o);
            }
#pragma unroll
            for (int d = 0; d < 14; ++d) b[d] = __ldg(p.v + gl + NF + 16 * d);
#pragma unroll
            for (int d = 0; d < 14; ++d) {
                const float o = b[d] + a[d].y;
                p.out[gi + NF + 16 * d] = o;
                lmin = fminf(lmin, o);
                lmax = fmaxf(lmax, o);
            }
        }
        __syncthreads();
    }
    if (p.minmax) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lmin = fminf(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
            lmax = fmaxf(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
        }
        if ((tid & 31) == 0) {
            red_min[tid >> 5] = lmin;
            red_max[tid >> 5] = lmax;
        }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < THREADS / 32; ++w) {
                lmin = fminf(lmin, red_min[w]);
                lmax = fmaxf(lmax, red_max[w]);
            }
            atomicMin(p.minmax + 2 * s, float_to_ordered(lmin));
            atomicMax(p.minmax + 2 * s + 1, float_to_ordered(lmax));
        }
    }
}

// x = 2 v - base (base complex or real): the image the last x-update's correction A^H (c_K - c_{K-1}) is added to
__global__ void last_base_kernel(const float* __restrict__ v, const float* __restrict__ base_re, const float* __restrict__ base_im,
                                 float* __restrict__ x_re, float* __restrict__ x_im, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        x_re[i] = 2.f * v[i] - base_re[i];
        x_im[i] = base_im ? -base_im[i] : 0.f;
    }
}

size_t fwdr_smem(const K1RealParams& p) { return (size_t)(PC * CS + 256 + 2 * NF + p.ns_max) * sizeof(float2) + (size_t)p.ns_max * 4 + 16; }
size_t adjr_smem(const K1RealParams& p) {
    return (size_t)(PC * CS + 256 + 2 * NF + p.ns_max + (size_t)p.n_ovf * 2 * OVF_STRIDE) * sizeof(float2) + (size_t)p.ns_max * 4 + 16;
}

}  // namespace

// Slab groups (CTAs) per image: the coarsest split that still gives four waves of CTAs (four resident per SM), at least 2.
int k1r_groups(int S, int C, int sm_count) {
    static const int forced = getenv("QMRI_K1R_G") ? atoi(getenv("QMRI_K1R_G")) : 0;  // tuning knob: 1, 2, 4 or 8
    if (forced == 1 || forced == 2 || forced == 4 || forced == 8) return forced;
    const double slots = 4.0 * sm_count;
    for (int G = 2; G < SLABS; G *= 2)
        if ((double)S * C * G / slots >= 4.0) return G;
    return SLABS;
}
size_t k1r_part_elems(int S, int C, int G, int ns_max) { return (size_t)S * C * G * ns_max; }
size_t k1r_state_elems(int S, int C, int ns_max) { return (size_t)S * C * ns_max; }
bool k1r_fits(int ns_max, int n_ovf) {
    K1RealParams p = {};
    p.ns_max = ns_max;
    p.n_ovf = n_ovf;
    return adjr_smem(p) <= 74 * 1024;  // three CTAs per SM at least (spiral masks: 48 KB, four; the EPI comb with its 81 overflow partials: 58 KB)
}

static int k1r_check(const K1RealParams& p, int S) {
    if (S > 65535) return qmri_fail(QMRI_EINVAL, "x-update: at most 65535 slices per launch (got %d)", S);
    if (p.G < 1 || SLABS % p.G) return qmri_fail(QMRI_EINVAL, "x-update (real streaming kernels): bad slab grouping %d", p.G);
    return QMRI_OK;
}

int k1r_forward(qmri_ctx* ctx, const K1RealParams& p_in, int S) {
    if (S <= 0) return QMRI_OK;
    QCHECK(k1r_check(p_in, S));
    K1RealParams p = p_in;
    p.slabs_per_cta = SLABS / p.G;
    static size_t conf_dev[QMRI_MAX_DEV] = {};
    size_t& conf = conf_dev[qmri_dev_slot(ctx)];
    const size_t sm = fwdr_smem(p);
    if (sm > conf) {
        QCUDA(cudaFuncSetAttribute(stream_fwdr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        conf = sm;
    }
    stream_fwdr_kernel<<<dim3(p.G, p.C, S), THREADS, sm, ctx->stream>>>(p);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

int k1r_solve(qmri_ctx* ctx, const K1RealParams& p, int S) {
    if (S <= 0) return QMRI_OK;
    stream_solver_kernel<<<dim3(p.C, S), 256, 0, ctx->stream>>>(p);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

int k1r_adjoint(qmri_ctx* ctx, const K1RealParams& p_in, int S) {
    if (S <= 0) return QMRI_OK;
    QCHECK(k1r_check(p_in, S));
    K1RealParams p = p_in;
    p.slabs_per_cta = SLABS / p.G;
    static size_t conf_dev[QMRI_MAX_DEV] = {};
    size_t& conf = conf_dev[qmri_dev_slot(ctx)];
    const size_t sm = adjr_smem(p);
    if (sm > 100 * 1024) return qmri_fail(QMRI_EUNSUPPORTED, "x-update (real streaming kernels): %zu bytes of shared memory needed", sm);
    if (sm > conf) {
        QCUDA(cudaFuncSetAttribute(stream_adjr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        conf = sm;
    }
    stream_adjr_kernel<<<dim3(p.G, p.C, S), THREADS, sm, ctx->stream>>>(p);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

int k1r_last_base(qmri_ctx* ctx, const float* v, const float* base_re, const float* base_im, float* x_re, float* x_im, size_t n) {
    if (!n) return QMRI_OK;
    const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, 148 * 16);
    last_base_kernel<<<blocks, 256, 0, ctx->stream>>>(v, base_re, base_im, x_re, x_im, n);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
