// General V (L x C, real): the per-k-space-location kernels around the streaming transforms.
//
// Reference: setup_subsampling_spiralgrided.m:36-37 / setup_subsampling_epi.m:31-32 build
//   P = [ S_1 kron(conj(V(1,:)), I) ; ... ; S_L kron(conj(V(L,:)), I) ],
// i.e. frame i samples  sum_c V(i,c) X^_c  on its own mask Omega_i (X^ = unitary 2-D FFT per channel).  With F = P fft2 / sqrt(NM)
// (main_recon_tsmis_FFT.m:228-229) the normal matrix of the x-update (PnP_ADMM.m:102, afun :153-171) is block diagonal in
// k-space: at location k the C x C block G_k = sum_{i: k in Omega_i} V(i,:)^T V(i,:), so the EXACT solve is
//   X^(k) = Z^(k) + (G_k + rho I)^{-1} sum_{i: k in Omega_i} V(i,:)^T ( y_i(k) - V(i,:) Z^(k) )      for k in the union U of the masks,
//   X^(k) = Z^(k) elsewhere.
// stream_fwd_kernel evaluates Z^_c on U for every channel (shared work-item table), the kernels below mix channels at each
// location, stream_adj_kernel transforms the sparse correction back.  (G_k + rho I)^{-1} is precomputed on the host per rho.
#include "common.cuh"
#include "xupdate_kernel.h"

namespace {

constexpr int CMAX = 16;

__device__ __forceinline__ float2 zhat(const GeneralMix& m, int s, int c, int u) {
    const float2* p = m.part + (((size_t)s * m.C + c) * m.G) * (size_t)m.nU + u;
    float sx = 0.f, sy = 0.f;
    for (int g = 0; g < m.G; ++g) {  // fixed order: deterministic
        const float2 t = p[(size_t)g * m.nU];
        sx += t.x;
        sy += t.y;
    }
    return make_float2(sx * m.inv_n, sy * m.inv_n);
}

__global__ void __launch_bounds__(128) mix_forward_kernel(GeneralMix m) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
    if (j >= m.nmeas) return;
    const int u = m.meas_u[j];
    const float* v = m.V + (size_t)m.meas_frame[j] * m.C;
    float ax = 0.f, ay = 0.f;
    for (int c = 0; c < m.C; ++c) {
        const float2 z = zhat(m, s, c, u);
        ax = fmaf(v[c], z.x, ax);
        ay = fmaf(v[c], z.y, ay);
    }
    m.y_out[(size_t)s * m.nmeas + j] = make_float2(ax, ay);
}

__global__ void __launch_bounds__(128) mix_adjoint_kernel(GeneralMix m) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
    if (u >= m.nU) return;
    float tx[CMAX], ty[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) tx[c] = ty[c] = 0.f;
    for (int e = m.memb_ptr[u]; e < m.memb_ptr[u + 1]; ++e) {
        const float2 y = m.y[(size_t)s * m.nmeas + m.memb_meas[e]];
        const float* v = m.V + (size_t)m.memb_frame[e] * m.C;
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < m.C) {
                tx[c] = fmaf(v[c], y.x, tx[c]);
                ty[c] = fmaf(v[c], y.y, ty[c]);
            }
    }
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
        if (c < m.C) m.cbuf[((size_t)s * m.C + c) * m.nU + u] = make_float2(tx[c] * m.inv_n, ty[c] * m.inv_n);
}

__global__ void __launch_bounds__(128) mix_solve_kernel(GeneralMix m) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
    if (u >= m.nU) return;
    float zx[CMAX], zy[CMAX], tx[CMAX], ty[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
        tx[c] = ty[c] = 0.f;
        if (c < m.C) {
            const float2 z = zhat(m, s, c, u);
            zx[c] = z.x;
            zy[c] = z.y;
        } else {
            zx[c] = zy[c] = 0.f;
        }
    }
    for (int e = m.memb_ptr[u]; e < m.memb_ptr[u + 1]; ++e) {
        const float2 y = m.y[(size_t)s * m.nmeas + m.memb_meas[e]];
        const float* v = m.V + (size_t)m.memb_frame[e] * m.C;
        float rx = y.x, ry = y.y;  // r = y_i(k) - V(i,:) Z^(k)
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < m.C) {
                rx = fmaf(-v[c], zx[c], rx);
                ry = fmaf(-v[c], zy[c], ry);
            }
#pragma unroll
        for (int c = 0; c < CMAX; ++c)
            if (c < m.C) {
                tx[c] = fmaf(v[c], rx, tx[c]);
                ty[c] = fmaf(v[c], ry, ty[c]);
            }
    }
    const float* Mi = m.Minv + (size_t)u * m.C * m.C;
#pragma unroll
    for (int r = 0; r < CMAX; ++r)
        if (r < m.C) {
            float dx = 0.f, dy = 0.f;
#pragma unroll
            for (int c = 0; c < CMAX; ++c)
                if (c < m.C) {
                    const float w = Mi[r * m.C + c];
                    dx = fmaf(w, tx[c], dx);
                    dy = fmaf(w, ty[c], dy);
                }
            m.cbuf[((size_t)s * m.C + r) * m.nU + u] = make_float2(dx * m.inv_n, dy * m.inv_n);  // pre-scaled for the inverse transform
        }
}

// PnP_ADMM.m:106-107 for general V (monitored sessions): the data-consistency residual of the solved x, per union location
// r_i(k) = y_i(k) - V(i,:) (Z^(k) + delta(k)) for every frame i sampling k, with delta = cbuf / inv_n (mix_solve_kernel pre-scales it
// for the inverse transform).  One double partial per block, reduced in a fixed order: no atomics.  A kernel of its own, so that
// mix_solve_kernel stays as it was for unmonitored sessions.
constexpr int RES_THREADS = 128;
__global__ void __launch_bounds__(RES_THREADS) mix_residual_kernel(GeneralMix m) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
    double acc = 0.0;
    if (u < m.nU) {
        float xx[CMAX], xy[CMAX];
        const float rs = 1.0f / m.inv_n;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
            xx[c] = xy[c] = 0.f;
            if (c < m.C) {
                const float2 z = zhat(m, s, c, u);
                const float2 d = m.cbuf[((size_t)s * m.C + c) * m.nU + u];
                xx[c] = z.x + d.x * rs;
                xy[c] = z.y + d.y * rs;
            }
        }
        for (int e = m.memb_ptr[u]; e < m.memb_ptr[u + 1]; ++e) {
            const float2 y = m.y[(size_t)s * m.nmeas + m.memb_meas[e]];
            const float* v = m.V + (size_t)m.memb_frame[e] * m.C;
            double rx = y.x, ry = y.y;
#pragma unroll
            for (int c = 0; c < CMAX; ++c)
                if (c < m.C) {
                    rx -= (double)v[c] * xx[c];
                    ry -= (double)v[c] * xy[c];
                }
            acc += rx * rx + ry * ry;
        }
    }
    acc = block_sum_fixed<RES_THREADS>(acc);
    if (threadIdx.x == 0) m.mon_dc[(size_t)s * gridDim.x + blockIdx.x] = acc;
}

}  // namespace

int k1_general_residual_parts(int nU) { return (nU + RES_THREADS - 1) / RES_THREADS; }
int k1_general_mix_residual(qmri_ctx* ctx, const GeneralMix& m) {
    if (m.S == 0) return QMRI_OK;
    if (m.nU == 0) return qmri_fail(QMRI_EINVAL, "general V: empty union mask");
    mix_residual_kernel<<<dim3(k1_general_residual_parts(m.nU), m.S), RES_THREADS, 0, ctx->stream>>>(m);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

int k1_general_mix_forward(qmri_ctx* ctx, const GeneralMix& m) {
    if (m.nmeas == 0 || m.S == 0) return QMRI_OK;
    mix_forward_kernel<<<dim3((m.nmeas + 127) / 128, m.S), 128, 0, ctx->stream>>>(m);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
int k1_general_mix_adjoint(qmri_ctx* ctx, const GeneralMix& m) {
    if (m.nU == 0 || m.S == 0) return QMRI_OK;
    mix_adjoint_kernel<<<dim3((m.nU + 127) / 128, m.S), 128, 0, ctx->stream>>>(m);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
int k1_general_mix_solve(qmri_ctx* ctx, const GeneralMix& m) {
    if (m.nU == 0 || m.S == 0) return QMRI_OK;
    mix_solve_kernel<<<dim3((m.nU + 127) / 128, m.S), 128, 0, ctx->stream>>>(m);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
