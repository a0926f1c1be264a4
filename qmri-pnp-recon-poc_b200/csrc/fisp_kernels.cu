// FISP-MRF dictionary on the device: the EPG simulation of each (T1, T2) atom and the temporal Gram matrix of the fingerprints
// (the inputs of the reference's dict.{D, normD, lut, V}, main_recon_tsmis_FFT.m:127-129).  Signal model: include/qmri.h.
//
// fisp_sim_kernel: one warp per atom.  With RF phase 0 every F state is purely imaginary and every Z state real, so F = i f turns
// Weigel's EPG into three real numbers per order; order k = 32 j + lane lives in registers fp[j], fm[j], z[j].  At pulse i only
// orders k <= max(min(i, T-1-i), min(i+1, T-2-i)) can still reach order 0 before the last readout, so only the slots j that hold
// such an order are updated (about T^2/4 order-updates per atom instead of T^2/2).  The gradient shift is one rotation by
// __shfl_sync per slot, with the value leaving lane 31 (lane 0) carried into the next (previous) slot.  Per pulse, one lane
// computes the relaxation of 32 consecutive pulses at a time and folds it into the rotation coefficients, kept per warp in
// shared memory; the flip-angle trigonometry is computed on the host in double and staged once per CTA.
//   COMPRESS = false: the raw fingerprint d_i goes to sig[i * ld + atom].
//   COMPRESS = true : d is projected on the fly onto V (T x C, shared memory) in double, and the unit-norm row D and its norm
//                     normD are written: no K x T array exists.
#include <math.h>

#include <algorithm>

#include "fisp_kernels.h"

// The kernels keep external linkage so that profiles show the same names from build to build.
constexpr int FISP_WARPS = 8;
constexpr int FISP_THREADS = 32 * FISP_WARPS;
constexpr unsigned FULL = 0xffffffffu;

static size_t fisp_smem_bytes(int T, int C) {
    return (size_t)T * sizeof(float4) + FISP_THREADS * (sizeof(float4) + sizeof(float2)) + (size_t)T * sizeof(float) +
           (size_t)T * C * sizeof(float);
}

template <int NJ, bool COMPRESS>
__global__ void __launch_bounds__(FISP_THREADS) fisp_sim_kernel(const FispParams p) {
    extern __shared__ float4 fisp_smem[];
    const int T = p.T;
    float4* s_pulse = fisp_smem;                                    // [T]
    float4* s_coef = s_pulse + T;                                   // [warp][32]: E2 cos^2(a/2), E2 sin^2(a/2), E2 sin a, E1 sin(a)/2
    float2* s_coef2 = reinterpret_cast<float2*>(s_coef + FISP_THREADS);  // [warp][32]: E1 cos a, 1 - E1
    float* s_tr = reinterpret_cast<float*>(s_coef2 + FISP_THREADS);      // [T]
    float* s_V = s_tr + T;                                          // [T][C]
    for (int i = threadIdx.x; i < T; i += FISP_THREADS) {
        s_pulse[i] = p.pulse[i];
        s_tr[i] = p.tr[i];
    }
    if (COMPRESS)
        for (int i = threadIdx.x; i < T * p.C; i += FISP_THREADS) s_V[i] = p.V[i];
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t k = p.a0 + (int64_t)blockIdx.x * FISP_WARPS + warp;
    if (k >= p.a1) return;  // whole warps only, after the block's last barrier
    const float T1 = p.lut[k], T2 = p.lut[p.K + k];
    const float r1 = 1.f / T1, r2 = 1.f / T2;
    const float ete = (float)exp(-p.te / (double)T2);

    float fp[NJ], fm[NJ], z[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) fp[j] = fm[j] = z[j] = 0.f;
    if (lane == 0) z[0] = p.inversion ? (float)(1.0 - 2.0 * exp(-p.ti / (double)T1)) : 1.f;
    float4* wc = s_coef + warp * 32;
    float2* wc2 = s_coef2 + warp * 32;
    double acc = 0.0;  // COMPRESS: lane c < C accumulates sum_i d_i V(i, c)

    for (int i = 0; i < T; ++i) {
        const int l = i & 31;
        if (l == 0) {
            __syncwarp();
            const int q = i + lane;
            if (q < T) {
                const float t = s_tr[q];
                const float4 a = s_pulse[q];
                // 1 - E1 from expm1f: the recovery term keeps its relative precision when E1 is close to 1 (long T1)
                const float E1 = expf(-t * r1), E2 = expf(-t * r2), om1 = -expm1f(-t * r1);
                wc[lane] = make_float4(E2 * a.x, E2 * a.y, E2 * a.z, 0.5f * E1 * a.z);
                wc2[lane] = make_float2(E1 * a.w, om1);
            }
            __syncwarp();
        }
        const float4 a = s_pulse[i];
        const float4 c = wc[l];
        const float2 c2 = wc2[l];
        // the sample i F+_0 e^{-te/T2} right after the pulse = -f+_0 e^{-te/T2} (meaningful in lane 0)
        const float d = -fmaf(a.x, fp[0], fmaf(a.y, fm[0], -a.z * z[0])) * ete;
        const int W = max(min(i, T - 1 - i), min(i + 1, T - 2 - i));
        const int J = W >> 5;
        // RF rotation T(a, 0) followed by relaxation over tr[i], folded into one 3 x 3 product per order
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            if (j <= J) {
                const float u = fp[j], v = fm[j], w = z[j];
                fp[j] = fmaf(c.x, u, fmaf(c.y, v, -c.z * w));
                fm[j] = fmaf(c.y, u, fmaf(c.x, v, c.z * w));
                z[j] = fmaf(c.w, u, fmaf(-c.w, v, c2.x * w));
            }
        }
        if (lane == 0) z[0] += c2.y;
        // dephasing by one order: f+_k <- f+_{k-1}, f-_k <- f-_{k+1}, then f+_0 = -f-_0 (F+_0 = conj F-_0)
        float carry = 0.f;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            if (j <= J) {
                const float r = __shfl_sync(FULL, fp[j], (lane + 31) & 31);
                fp[j] = lane == 0 ? carry : r;
                carry = r;
            }
        }
        carry = 0.f;  // order 32 (J + 1) is outside the live window: zero in the first half, irrelevant in the second
#pragma unroll
        for (int j = NJ - 1; j >= 0; --j) {
            if (j <= J) {
                const float r = __shfl_sync(FULL, fm[j], (lane + 1) & 31);
                fm[j] = lane == 31 ? carry : r;
                carry = r;
            }
        }
        if (lane == 0) fp[0] = -fm[0];
        if (COMPRESS) {
            const float dd = __shfl_sync(FULL, d, 0);
            if (lane < p.C) acc = fma((double)dd, (double)s_V[i * p.C + lane], acc);
        } else if (lane == 0) {
            p.sig[(int64_t)i * p.ld + (k - p.a0)] = d;
        }
    }
    if (COMPRESS) {
        double n2 = acc * acc;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(FULL, n2, o);
        const double nd = sqrt(__shfl_sync(FULL, n2, 0));  // one value for every channel of the row
        const int64_t n = p.a1 - p.a0, r = k - p.a0;
        if (lane < p.C) p.D[(int64_t)lane * n + r] = (float)(acc / nd);
        if (lane == 0) p.normD[r] = (float)nd;
    }
}

template <bool COMPRESS>
static int fisp_launch(qmri_ctx* ctx, const FispParams& p) {
    if (p.T < 1 || p.T > FISP_MAX_T) return qmri_fail(QMRI_EUNSUPPORTED, "FISP simulation: T = %d outside [1, %d]", p.T, FISP_MAX_T);
    const int64_t n = p.a1 - p.a0;
    if (n <= 0) return QMRI_OK;
    const size_t smem = fisp_smem_bytes(p.T, COMPRESS ? p.C : 0);
    const unsigned grid = (unsigned)((n + FISP_WARPS - 1) / FISP_WARPS);
    // slots needed: the highest live order is (T - 1) / 2
    const int slots = ((p.T - 1) / 2) / 32 + 1;
    auto run = [&](auto kernel) -> int {
        QCUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<grid, FISP_THREADS, smem, ctx->stream>>>(p);
        QLAUNCH_CHECK(ctx);
        return QMRI_OK;
    };
    if (slots <= 4) return run(fisp_sim_kernel<4, COMPRESS>);
    if (slots <= 8) return run(fisp_sim_kernel<8, COMPRESS>);
    return run(fisp_sim_kernel<16, COMPRESS>);
}

// ---- Gram matrix: 64 x 64 tiles of G on and above the diagonal, 16 x 16 threads with 4 x 4 outputs each, fp32 inputs widened
// to double in shared memory (an fp32 x fp32 product is exact in double), accumulated in double in a fixed order.
constexpr int GT = 64, GK = 16, GTHREADS = 256;
constexpr int GRAM_CTAS_TARGET = 592;  // 4 per SM of a B200; fixed so that G does not depend on the device

__global__ void __launch_bounds__(GTHREADS) fisp_gram_kernel(const float* __restrict__ X, int64_t ld, int64_t n, int T,
                                                             double* __restrict__ part, int parts) {
    __shared__ double As[GK][GT + 1], Bs[GK][GT + 1];
    const int nt = (T + GT - 1) / GT;
    int t = blockIdx.x, ti = 0;
    while (t >= nt - ti) {
        t -= nt - ti;
        ++ti;
    }
    const int tj = ti + t;
    const int pi = blockIdx.y;
    const int64_t k0 = n * pi / parts, k1 = n * (pi + 1) / parts;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i0 = ti * GT, j0 = tj * GT;
    double acc[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = 0.0;
    for (int64_t kb = k0; kb < k1; kb += GK) {
        for (int e = threadIdx.x; e < GK * GT; e += GTHREADS) {
            const int r = e / GK, kk = e % GK;
            const int64_t kg = kb + kk;
            const int ia = i0 + r, ib = j0 + r;
            As[kk][r] = (ia < T && kg < k1) ? (double)X[(int64_t)ia * ld + kg] : 0.0;
            Bs[kk][r] = (ib < T && kg < k1) ? (double)X[(int64_t)ib * ld + kg] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            double a[4], b[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                a[u] = As[kk][ty + 16 * u];
                b[u] = Bs[kk][tx + 16 * u];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int v = 0; v < 4; ++v) acc[u][v] = fma(a[u], b[v], acc[u][v]);
        }
        __syncthreads();
    }
    double* P = part + (size_t)pi * T * T;
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
            if (i < T && j < T) P[(size_t)i * T + j] += acc[u][v];
        }
}

// G(i, j) = G(j, i) = sum over parts, in order, of part[p](min(i,j), max(i,j)): exactly symmetric.
__global__ void fisp_gram_reduce_kernel(const double* __restrict__ part, int parts, int T, double* __restrict__ G) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)T * T) return;
    const int i = (int)(e / T), j = (int)(e % T);
    const size_t src = (size_t)min(i, j) * T + max(i, j);
    double s = 0.0;
    for (int q = 0; q < parts; ++q) s += part[(size_t)q * T * T + src];
    G[e] = s;
}

int fisp_launch_signals(qmri_ctx* ctx, const FispParams& p) { return fisp_launch<false>(ctx, p); }

int fisp_launch_compress(qmri_ctx* ctx, const FispParams& p) {
    if (p.C < 1 || p.C > FISP_MAX_C || p.C > p.T) return qmri_fail(QMRI_EINVAL, "FISP compression: C = %d outside [1, min(T, %d)]", p.C, FISP_MAX_C);
    return fisp_launch<true>(ctx, p);
}

int fisp_gram_parts(int T) {
    const int nt = (T + GT - 1) / GT, tiles = nt * (nt + 1) / 2;
    return std::max(1, std::min(64, (GRAM_CTAS_TARGET + tiles - 1) / tiles));
}

int fisp_launch_gram_accumulate(qmri_ctx* ctx, const float* X, int64_t ld, int64_t n, int T, double* part, int parts) {
    if (n <= 0) return QMRI_OK;
    const int nt = (T + GT - 1) / GT;
    fisp_gram_kernel<<<dim3(nt * (nt + 1) / 2, parts), GTHREADS, 0, ctx->stream>>>(X, ld, n, T, part, parts);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}

int fisp_launch_gram_reduce(qmri_ctx* ctx, const double* part, int parts, int T, double* G) {
    const size_t n = (size_t)T * T;
    fisp_gram_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(part, parts, T, G);
    QLAUNCH_CHECK(ctx);
    return QMRI_OK;
}
