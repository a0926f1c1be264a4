// K1 "streaming" variant - the fused x-update for large slice batches (sm_100a).
//
// Reference being replaced: the same lines as xupdate_kernel.cu -
//   main_files/algorithms/PnP_ADMM/PnP_ADMM.m:102-103 (lsqr x-update), :115-118 (v = real(x+u)),
//   :121 (global min/max for the 0-1 normalisation), :144 (u += x - v),
// with F.forward / F.adjoint of main_recon_tsmis_FFT.m:228-229 - in the closed form
//   x = z + A^H (y - A z) / (1 + rho)          (A A^H = I, see xupdate_phases.cuh).
//
// The cluster kernel (xupdate_kernel.cu) keeps a whole (slice, channel) image on chip in the shared memory
// of eight CTAs; that is the right shape for a handful of slices, but it is bound by shared-memory traffic,
// cluster barriers and the sparse-DFT table walks.  For batches that fill the machine the update is split
// at its only global dependency - the <= ~700 sampled k-space values of a channel:
//   stream_fwd_kernel     grid (G, C, S): N / G columns of one image, R = N / 16 at a time:  global -> registers ->
//                         FFT along n -> sampled DFT along m;  partial sample sums -> `part` (5 KB per CTA)
//   stream_solve_kernel   grid (C, S): adds the G partials in a fixed order, c = (y - A z) / (1 + rho)
//   stream_adj_kernel     grid (G, C, S): sparse inverse DFT along m -> inverse FFT along n -> registers ->
//                         w' = v + corr (+ x on the last iteration) -> global; per-slice min / max
// Two instances of each kernel, by image side N == M: 224 (R = 14: CTAs of 224 threads, four per SM) and 256 (R = 16: CTAs of
// 256 threads, three per SM for the forward kernel and two for the adjoint kernel - see fwd_min_ctas / adj_min_ctas).
// No cluster, no DSMEM, work items small enough that the last wave is short.  The first / last FFT stage works on registers filled from / drained to global memory and the
// sparse sums run on per-row work items with rotating twiddles (xupdate_phases.cuh), so the shared-memory
// traffic is about a third of the cluster kernel's.  HBM traffic per pixel-channel: read w (8 B) + v (4 B)
// in the forward kernel, read v again (4 B) and write w' (8 B) in the adjoint kernel = 24 B against the
// 20 B of the single-pass formulation; `part` and `c` add < 2 %.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "xupdate_kernel.h"
#include "xupdate_phases.cuh"

using namespace k1;

namespace {

// Per image side N: R = N / 16 columns per slab, N threads = R column FFTs x 16 lanes (in the sparse passes one thread per work
// item, i.e. per k-space row), 16 slabs per image.
constexpr int SLABS = 16;
// CTAs per SM the register allocation is fitted to.  N = 256: the forward kernel fits three (80 registers); the adjoint kernel
// needs more than 80 (at three it spills the work-item fields it keeps across the slab loop), so it is fitted to two.
template <int N>
constexpr int fwd_min_ctas() { return N == 224 ? 4 : 3; }
template <int N>
constexpr int adj_min_ctas() { return N == 224 ? 4 : 2; }
// The monitored SOLVE instance (the first x-update of a monitored PnP-ADMM run, once per run) is fitted to one CTA less at 224:
// at four its ground-truth loads add spills.
template <int N, int MODE, bool MON>
constexpr int adj_min_ctas_mon() { return MON && MODE == K1_SOLVE && N == 224 ? 3 : adj_min_ctas<N>(); }

__device__ __forceinline__ size_t late_offset(size_t off, float after) {
    size_t r;
    asm volatile("mov.u64 %0, %1;" : "=l"(r) : "l"(off), "f"(after));
    return r;
}

template <int THREADS>
__device__ __forceinline__ double* mon_slot() {
    __shared__ double slot[THREADS];
    return slot + threadIdx.x;
}

struct Item {
    int k1, cnt, start, slot, novf, ovf0;
};
__device__ __forceinline__ Item decode_item(uint32_t A, uint32_t B) {
    Item it;
    it.k1 = (int)(A & 0xffu);
    it.cnt = (int)((A >> 8) & 0xffu);    // 0: no item
    it.start = (int)(A >> 16);
    it.slot = (int)(B & 0xffu);          // 0: primary item of its row
    it.novf = (int)((B >> 8) & 0xffu);
    it.ovf0 = (int)((B >> 16) & 0xffu);
    return it;
}

// ---------------- forward: partial sums of A z over a group of slabs -------------------------------------
template <int N, int MODE>
__global__ void __launch_bounds__(N, fwd_min_ctas<N>()) stream_fwd_kernel(K1Params p) {
    constexpr int MC = Side<N>::R, CS = Side<N>::CS, THREADS = N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ws = reinterpret_cast<float2*>(smem_raw);                  // [MC][CS] slab workspace
    float2* tw2 = ws + MC * CS;                                        // [16][16]
    float2* tw448 = tw2 + 256;                                         // [2N]
    float2* pc = tw448 + 2 * N;                                        // [ns_max] sample accumulators
    uint32_t* s_ent = reinterpret_cast<uint32_t*>(pc + p.ns_max);      // [ns_max]

    const int tid = threadIdx.x;
    const int g = blockIdx.x, c = blockIdx.y, s = blockIdx.z;
    const int ct = p.shared_mask ? 0 : c;  // table row: the channel's own frame, or the shared union mask (general V)
    const int f0 = p.frame_ptr[ct];
    const int ns = p.frame_ptr[ct + 1] - f0;
    const size_t img = ((size_t)s * p.C + c) * (size_t)(N * N);

    for (int i = tid; i < 256; i += THREADS) tw2[i] = p.tw2[i];
    for (int i = tid; i < 2 * N; i += THREADS) tw448[i] = p.tw448[i];
    for (int i = tid; i < ns; i += THREADS) {
        s_ent[i] = p.ent[f0 + i];
        pc[i] = make_float2(0.f, 0.f);
    }
    const uint32_t itA = p.itA[(size_t)ct * N + tid];
    const int l16 = tid & 15;
    const int col = tid >> 4;
    float2* colp = ws + col * CS;
    __syncthreads();

    const int slab0 = g * p.slabs_per_cta;
#pragma unroll 1
    for (int sl = 0; sl < p.slabs_per_cta; ++sl) {
        const int m0 = (slab0 + sl) * MC;
        {
            const size_t gi = img + (size_t)(m0 + col) * N + l16;
            float2 a[16];
            if (MODE == K1_ADMM) {  // z = 2 v - w
                float wr[MC], wi[MC], vv[MC];
#pragma unroll
                for (int n1 = 0; n1 < MC; ++n1) {
                    wr[n1] = __ldcs(p.in_re + gi + 16 * n1);
                    wi[n1] = __ldcs(p.in_im + gi + 16 * n1);
                    vv[n1] = __ldg(p.v + gi + 16 * n1);
                }
#pragma unroll
                for (int n1 = 0; n1 < MC; ++n1) a[n1] = make_float2(2.f * vv[n1] - wr[n1], -wi[n1]);
            } else {
#pragma unroll
                for (int n1 = 0; n1 < MC; ++n1)
                    a[n1] = make_float2(__ldcs(p.in_re + gi + 16 * n1), p.in_im ? __ldcs(p.in_im + gi + 16 * n1) : 0.f);
            }
            fwd_s1_regs<N>(a, l16, tw2);
            fft_s1_store<N>(colp, l16, a);
            __syncwarp();
            if (l16 < MC) fft_s2_load(colp, l16, a);
            __syncwarp();
            if (l16 < MC) fft_s2_store<false, N>(colp, l16, a);
        }
        __syncthreads();
        p3_item<N>(ws, (int)(itA & 0xffu), s_ent + (itA >> 16), (int)((itA >> 8) & 0xffu), tw448, m0, pc);
        __syncthreads();
    }
    // every sample belongs to exactly one work item, i.e. to one thread: no race on pc above
    float2* part = p.part + (((size_t)s * p.C + c) * p.G + g) * (size_t)p.slot_stride + p.slot_off;
    for (int j = tid; j < ns; j += THREADS) part[j] = pc[j];
}

// ---------------- solve on the samples ----------------------------------------------------------------------
// MON (monitored PnP-ADMM sessions, modes ADMM and SOLVE): also sum |y - A z|^2 over the channel's samples into mon_dc[s][c].  With
// x = z + A^H c, c = (y - A z) / (1 + rho) and A A^H = I, y - A x = (y - A z) - c = rho c, so |y - A x| = rho / (1 + rho) |y - A z|
// (the finalize kernel applies the factor): the data-consistency residual of PnP_ADMM.m:106-107 costs no transform.
constexpr int SOLVE_THREADS = 256;
template <int N, int MODE, bool MON>
__global__ void __launch_bounds__(SOLVE_THREADS) stream_solve_kernel(K1Params p) {
    const int c = blockIdx.x, s = blockIdx.y;
    const int f0 = p.frame_ptr[c];
    const int ns = p.frame_ptr[c + 1] - f0;
    const float inv_n = 1.0f / (float)N;  // unitary scaling 1/sqrt(N*M), once per transform direction
    const float2* part = p.part + ((size_t)s * p.C + c) * p.G * (size_t)p.slot_stride;
    double dc = 0.0;
    for (int j = threadIdx.x; j < ns; j += blockDim.x) {
        float sx = 0.f, sy = 0.f;
#pragma unroll 1
        for (int g0 = 0; g0 < p.G; g0 += 4) {  // fixed order: deterministic; four loads in flight (G is 4, 8 or 16; 2 only by hand)
            float2 t[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] = g0 + i < p.G ? part[(size_t)(g0 + i) * p.slot_stride + j] : make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                sx += t[i].x;
                sy += t[i].y;
            }
        }
        const float rx = sx, ry = sy;  // MON: the unscaled sums, so that the monitor adds no use of the scaled ones below (which
                                       // would stop the compiler from fusing their scaling into the subtraction: different bits)
        sx *= inv_n;
        sy *= inv_n;
        const size_t yi = (size_t)s * p.nmeas + f0 + j;
        if (MODE == K1_FORWARD) {
            p.y_out[yi] = make_float2(sx, sy);
        } else {
            const float2 y = p.y[yi];
            const float gsc = p.inv_1p_rho * inv_n;  // (y - A z)/(1 + rho), pre-scaled for the inverse transform
            p.cbuf[((size_t)s * p.C + c) * p.slot_stride + j] = make_float2((y.x - sx) * gsc, (y.y - sy) * gsc);
            if (MON) {
                const double dr = (double)y.x - (double)rx * inv_n, di = (double)y.y - (double)ry * inv_n;
                dc += dr * dr + di * di;
            }
        }
    }
    if (MON) {
        dc = block_sum_fixed<SOLVE_THREADS>(dc);
        if (threadIdx.x == 0) p.mon_dc[(size_t)s * p.C + c] = dc;
    }
}

// ---------------- adjoint: corr = A^H c, epilogue --------------------------------------------------------------
// MON (monitored PnP-ADMM sessions with a ground truth, modes ADMM and SOLVE): also sum |gt - x|^2 over the CTA's pixels into
// mon_gt[s][c][g] (PnP_ADMM.m:108-109).  ADMM mode forms x = 2 v - w + corr on every iteration, with the expression the
// last-iteration store uses, so the history of iteration k is the norm of what a k-iteration run returns.
template <int N, int MODE, bool MON>
__global__ void __launch_bounds__(N, adj_min_ctas_mon<N, MODE, MON>()) stream_adj_kernel(K1Params p) {
    constexpr int MC = Side<N>::R, CS = Side<N>::CS, OVF_STRIDE = Side<N>::OVF_STRIDE, THREADS = N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* ws = reinterpret_cast<float2*>(smem_raw);                  // [MC][CS]
    float2* tw2 = ws + MC * CS;                                        // [16][16]
    float2* tw448 = tw2 + 256;                                         // [2N]
    float2* pc = tw448 + 2 * N;                                        // [ns_max] c
    float2* ovf = pc + p.ns_max;                                       // [n_ovf][OVF_STRIDE] overflow partials
    uint32_t* s_ent = reinterpret_cast<uint32_t*>(ovf + (size_t)p.n_ovf * OVF_STRIDE);  // [ns_max]
    __shared__ float red_min[THREADS / 32], red_max[THREADS / 32];

    const int tid = threadIdx.x;
    const int g = blockIdx.x, c = blockIdx.y, s = blockIdx.z;
    const int ct = p.shared_mask ? 0 : c;
    const int f0 = p.frame_ptr[ct];
    const int ns = p.frame_ptr[ct + 1] - f0;
    const size_t img = ((size_t)s * p.C + c) * (size_t)(N * N);

    for (int i = tid; i < 256; i += THREADS) tw2[i] = p.tw2[i];
    for (int i = tid; i < 2 * N; i += THREADS) tw448[i] = p.tw448[i];
    for (int i = tid; i < ns; i += THREADS) {
        s_ent[i] = p.ent[f0 + i];
        if (MODE == K1_ADJOINT && !p.shared_mask) {
            const float2 y = p.y[(size_t)s * p.nmeas + f0 + i];
            pc[i] = make_float2(y.x * (1.0f / (float)N), y.y * (1.0f / (float)N));
        } else {
            pc[i] = p.cbuf[((size_t)s * p.C + c) * p.slot_stride + p.slot_off + i];
        }
    }
    const uint32_t itA = p.itA[(size_t)ct * N + tid], itB = p.itB[(size_t)ct * N + tid];
    const int l16 = tid & 15;
    const uint32_t rmask = p.rowmask[ct * 16 + l16];
    const int col = tid >> 4;
    float2* colp = ws + col * CS;
    __syncthreads();

    float lmin = INFINITY, lmax = -INFINITY;
    // MON: this thread's sum of |gt - x|^2, kept in shared memory rather than in the two registers a double takes (the kernel
    // is at its register limit)
    if (MON) *mon_slot<THREADS>() = 0.0;
    const int slab0 = g * p.slabs_per_cta;
#pragma unroll 1
    for (int sl = 0; sl < p.slabs_per_cta; ++sl) {
        const int m0 = (slab0 + sl) * MC;
        const size_t gi = img + (size_t)(m0 + col) * N + l16;
        {
            const Item it = decode_item(itA, itB);
            if (it.cnt != 0) {
                float2 SP[Side<N>::NP], SM[Side<N>::NP];
                p4_item_partial<N>(SP, SM, s_ent + it.start, it.cnt, tw448, m0, pc);
                if (it.slot == 0) p4_item_store<N>(ws, it.k1, SP, SM);
                else p4_item_spill<N>(ovf + (size_t)(it.slot - 1) * OVF_STRIDE, SP, SM);
            }
        }
        if (p.n_ovf) {
            __syncthreads();
            const Item it = decode_item(itA, itB);
            if (it.cnt != 0 && it.slot == 0 && it.novf) p4_row_add_overflow<N>(ws, it.k1, ovf + (size_t)it.ovf0 * OVF_STRIDE, it.novf);
        }
        __syncthreads();
        {
            float2 a[16];
            if (l16 < MC) inv_s1_load<N>(colp, l16, tw2, rmask, a);
            __syncwarp();
            if (l16 < MC) inv_s1_store(colp, l16, a);
            __syncwarp();
            inv_s2_regs<N>(colp, l16, a);
            // What the correction is added to (v in ADMM mode, z in SOLVE mode).  The offset is made to depend on the transform's
            // last output so that the R - 2R loads are not hoisted above it: held across the transform they spill.
            const size_t gl = late_offset(gi, a[MC - 1].y);
            float br[MC], bi[MC];
            if (MODE == K1_ADMM) {
#pragma unroll
                for (int d = 0; d < MC; ++d) br[d] = __ldg(p.v + gl + 16 * d);
            } else if (MODE == K1_SOLVE) {
#pragma unroll
                for (int d = 0; d < MC; ++d) {
                    br[d] = p.in_re[gl + 16 * d];  // plain loads: the general-V accumulation passes run this mode in place (in == out)
                    bi[d] = p.in_im ? p.in_im[gl + 16 * d] : 0.f;
                }
            }
            if (MODE == K1_ADMM && !MON && p.x_re) {  // last iteration: x = z + corr = 2 v - w + corr; w' may overwrite w in place, so x goes first
#pragma unroll
                for (int d = 0; d < MC; ++d) {
                    const float wr = __ldcs(p.in_re + gi + 16 * d), wi = __ldcs(p.in_im + gi + 16 * d);
                    p.x_re[gi + 16 * d] = 2.f * br[d] - wr + a[d].x;
                    p.x_im[gi + 16 * d] = a[d].y - wi;
                }
            }
            float ge = 0.f;
#pragma unroll
            for (int d = 0; d < MC; ++d) {
                float ore, oim;
                if (MODE == K1_ADMM) {  // w' = v + corr
                    ore = br[d] + a[d].x;
                    oim = a[d].y;
                } else if (MODE == K1_SOLVE) {  // x = z + corr
                    ore = br[d] + a[d].x;
                    oim = bi[d] + a[d].y;
                } else {  // adjoint
                    ore = a[d].x;
                    oim = a[d].y;
                }
                if (MON) {
                    float xr = ore, xi = oim;  // SOLVE: x is the output
                    if (MODE == K1_ADMM) {     // x = 2 v - w + corr, element by element ahead of the in-place store of w'
                        const float wr = __ldcs(p.in_re + gi + 16 * d), wi = __ldcs(p.in_im + gi + 16 * d);
                        xr = 2.f * br[d] - wr + a[d].x;
                        xi = a[d].y - wi;
                        if (p.x_re) {
                            p.x_re[gi + 16 * d] = xr;
                            p.x_im[gi + 16 * d] = xi;
                        }
                    }
                    const float er = __ldcs(p.gt_re + gi + 16 * d) - xr, ei = (p.gt_im ? __ldcs(p.gt_im + gi + 16 * d) : 0.f) - xi;
                    ge += er * er + ei * ei;
                }
                p.out_re[gi + 16 * d] = ore;
                p.out_im[gi + 16 * d] = oim;
                lmin = fminf(lmin, ore);
                lmax = fmaxf(lmax, ore);
            }
            if (MON) *mon_slot<THREADS>() += ge;
        }
        __syncthreads();
    }
    if (MON) {  // one partial per CTA, no atomics: graph replays and direct launches give the same bits
        const double t = block_sum_fixed<THREADS>(*mon_slot<THREADS>());
        if (tid == 0) p.mon_gt[((size_t)s * p.C + c) * p.G + g] = t;
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

template <int N>
size_t fwd_smem(const K1Params& p) {
    return (size_t)(Side<N>::R * Side<N>::CS + 256 + 2 * N + p.ns_max) * sizeof(float2) + (size_t)p.ns_max * 4 + 16;
}
template <int N>
size_t adj_smem(const K1Params& p) {
    return (size_t)(Side<N>::R * Side<N>::CS + 256 + 2 * N + p.ns_max + (size_t)p.n_ovf * Side<N>::OVF_STRIDE) * sizeof(float2) +
           (size_t)p.ns_max * 4 + 16;
}

template <int N, int MODE, bool MON>
int launch_adj(qmri_ctx* ctx, const K1Params& p, int S) {
    static size_t conf_dev[QMRI_MAX_DEV] = {};
    size_t& conf = conf_dev[qmri_dev_slot(ctx)];
    const size_t sa = adj_smem<N>(p);
    if (sa > conf) {
        QCUDA(cudaFuncSetAttribute(stream_adj_kernel<N, MODE, MON>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sa));
        conf = sa;
    }
    stream_adj_kernel<N, MODE, MON><<<dim3(p.G, p.C, S), N, sa, ctx->stream>>>(p);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

template <int N, int MODE>
int launch_mode(qmri_ctx* ctx, const K1Params& p, int S) {
    constexpr bool CAN_MON = MODE == K1_ADMM || MODE == K1_SOLVE;
    static size_t conf_f_dev[QMRI_MAX_DEV] = {};
    size_t& conf_f = conf_f_dev[qmri_dev_slot(ctx)];
    const size_t sf = fwd_smem<N>(p);
    if (sf > conf_f) {
        QCUDA(cudaFuncSetAttribute(stream_fwd_kernel<N, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sf));
        conf_f = sf;
    }
    if (MODE != K1_ADJOINT && !(p.stage & K1_STAGE_ADJ_ONLY)) {
        stream_fwd_kernel<N, MODE><<<dim3(p.G, p.C, S), N, sf, ctx->stream>>>(p);
        QLAUNCH_CHECK(ctx);
        if (!p.shared_mask && !(p.stage & K1_STAGE_NO_SOLVE)) {  // (the real-state loop runs its own recurrence on the partial sums)
            if (CAN_MON && p.mon_dc) stream_solve_kernel<N, MODE, CAN_MON><<<dim3(p.C, S), SOLVE_THREADS, 0, ctx->stream>>>(p);
            else stream_solve_kernel<N, MODE, false><<<dim3(p.C, S), SOLVE_THREADS, 0, ctx->stream>>>(p);
            QLAUNCH_CHECK(ctx);
        }
    }
    if (MODE != K1_FORWARD && !(p.stage & K1_STAGE_FWD_ONLY)) {
        if (CAN_MON && p.mon_gt) return launch_adj<N, MODE, CAN_MON>(ctx, p, S);
        return launch_adj<N, MODE, false>(ctx, p, S);
    }
    return QMRI_OK;
}

template <int N>
int launch_side(qmri_ctx* ctx, const K1Params& p, int S) {
    if (adj_smem<N>(p) > 100 * 1024)
        return qmri_fail(QMRI_EUNSUPPORTED, "x-update (streaming kernel): %zu bytes of shared memory needed", adj_smem<N>(p));
    switch (p.mode) {
        case K1_ADMM: return launch_mode<N, K1_ADMM>(ctx, p, S);
        case K1_SOLVE: return launch_mode<N, K1_SOLVE>(ctx, p, S);
        case K1_FORWARD: return launch_mode<N, K1_FORWARD>(ctx, p, S);
        default: return launch_mode<N, K1_ADJOINT>(ctx, p, S);
    }
}

}  // namespace

// Number of slab groups (CTAs) per image: the coarsest split that still gives four waves of CTAs (four CTAs per SM resident), but
// never coarser than 4.  Coarser groups stage the operator tables less often (13 KB per CTA against 37 KB of image data per
// slab); measured on B200, us per slice-iteration: S = 120: G = 2 / 4 / 8 / 16 -> 4.20 / 4.13 / 4.34 / 4.92; S = 60: G = 4 / 8 ->
// 4.50 / 4.58; S = 30: G = 8 / 16 -> 5.11 / 5.57.
int k1_stream_groups(int S, int C, int sm_count) {
    static const int forced = getenv("QMRI_K1_G") ? atoi(getenv("QMRI_K1_G")) : 0;  // tuning knob: 2, 4, 8 or 16
    if (forced == 2 || forced == 4 || forced == 8 || forced == 16) return forced;
    const double slots = 4.0 * sm_count;
    for (int G = 4; G < SLABS; G *= 2)
        if ((double)S * C * G / slots >= 4.0) return G;
    return SLABS;
}
size_t k1_stream_part_elems(int S, int C, int G, int ns_max) { return (size_t)S * C * G * ns_max; }
size_t k1_stream_cbuf_elems(int S, int C, int ns_max) { return (size_t)S * C * ns_max; }

int k1_stream_launch(qmri_ctx* ctx, const K1Params& p_in, int S, int ns_max) {
    if (S <= 0) return QMRI_OK;
    if (S > 65535) return qmri_fail(QMRI_EINVAL, "x-update: at most 65535 slices per launch (got %d)", S);
    K1Params p = p_in;
    p.ns_max = ns_max;
    if (p.G < 1 || SLABS % p.G || !p.part || !p.cbuf) return qmri_fail(QMRI_EINVAL, "x-update (streaming kernel): bad slab grouping / scratch");
    p.slabs_per_cta = SLABS / p.G;
    // monitoring: the residual partials need the solve kernel (identity V, whole x-update); the ground-truth partials an adjoint
    // launch that completes x (general V: the last adjoint-only pass)
    if ((p.mon_dc && (p.shared_mask || p.stage)) || ((p.mon_dc || p.mon_gt) && p.mode != K1_ADMM && p.mode != K1_SOLVE) ||
        (p.mon_gt && (!p.gt_re || (p.stage & K1_STAGE_FWD_ONLY))))
        return qmri_fail(QMRI_EINVAL, "x-update (streaming kernel): bad monitor arguments");
    if (!p.shared_mask) {
        p.slot_off = 0;
        p.slot_stride = ns_max;
    }
    if (p.nf == 224) return launch_side<224>(ctx, p, S);
    if (p.nf == 256) return launch_side<256>(ctx, p, S);
    return qmri_fail(QMRI_EUNSUPPORTED, "x-update (streaming kernel): image side %d (224 or 256)", p.nf);
}
