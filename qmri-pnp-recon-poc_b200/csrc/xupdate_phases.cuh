// K1 - fused x-update: per-thread phase functions.
//
// One thread-block cluster owns one (slice, channel) 224 x 224 image; each CTA of
// the cluster owns a slab of MC consecutive columns m (MATLAB dim 2) kept in shared
// memory as interleaved complex fp32.  The data-consistency solve of
//   PnP_ADMM.m:102 (lsqr over afun :153-171) with F from main_recon_tsmis_FFT.m:228-229
// is evaluated in its exact closed form for A A^H = I (V = eye):
//   x = z + A^H (y - A z) / (1 + rho)
// A z is needed only at the <= ~700 sampled k-space locations of the channel and
// A^H c is the inverse transform of a sparse array, so the m-direction transforms
// are evaluated as sparse DFT sums, and only the n-direction (contiguous dim) uses
// full length-224 FFTs (224 = 14 x 16, two register-resident stages).  The streaming kernels
// (xupdate_stream.cu) also run N == M == 256 = 16 x 16: see Side below.
//
// The functions here are __host__ __device__ so that tests/test_k1_emulation.py can
// run the exact kernel arithmetic on the CPU (no GPU in the build container).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define QHD __host__ __device__ __forceinline__
#include <cuda_runtime.h>
#else
#define QHD inline
struct float2 { float x, y; };
struct float4 { float x, y, z, w; };
static inline float2 make_float2(float a, float b) { return float2{a, b}; }
#endif

namespace k1 {

constexpr int NF = 224;   // image side (N == M == 224) and FFT length of the cluster and real-image kernels
constexpr int CS = 225;   // shared-memory column stride in float2 (odd: conflict-free across columns)
constexpr int TWP = NF + NF / 16;  // padded twiddle table: entry t sits at t + (t >> 4), so strided lookups spread over banks

QHD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
QHD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
QHD float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
QHD float2 cswap(float2 a) { return make_float2(a.y, a.x); }
// multiply by -i
QHD float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }

// position of element (k1, n2) of the 14 x 16 intermediate inside a column; XOR swizzle keeps
// both the stage-1 stores (lanes = n2) and the stage-2 loads (lanes = k1) bank-conflict free
QHD int swz(int k1, int n2) { return 16 * k1 + (n2 ^ (k1 & 15)); }

// ---- 7-point DFT (forward, e^{-2 pi i/7}) ----------------------------------------
QHD void dft7(float2& x0, float2& x1, float2& x2, float2& x3, float2& x4, float2& x5, float2& x6) {
    const float C1 = 0.62348980185873353f, C2 = -0.22252093395631440f, C3 = -0.90096886790241913f;
    const float S1 = 0.78183148246802981f, S2 = 0.97492791218182361f, S3 = 0.43388373911755812f;
    float2 p1 = cadd(x1, x6), p2 = cadd(x2, x5), p3 = cadd(x3, x4);
    float2 q1 = csub(x1, x6), q2 = csub(x2, x5), q3 = csub(x3, x4);
    float2 a1 = make_float2(x0.x + C1 * p1.x + C2 * p2.x + C3 * p3.x, x0.y + C1 * p1.y + C2 * p2.y + C3 * p3.y);
    float2 a2 = make_float2(x0.x + C2 * p1.x + C3 * p2.x + C1 * p3.x, x0.y + C2 * p1.y + C3 * p2.y + C1 * p3.y);
    float2 a3 = make_float2(x0.x + C3 * p1.x + C1 * p2.x + C2 * p3.x, x0.y + C3 * p1.y + C1 * p2.y + C2 * p3.y);
    float2 b1 = make_float2(S1 * q1.x + S2 * q2.x + S3 * q3.x, S1 * q1.y + S2 * q2.y + S3 * q3.y);
    float2 b2 = make_float2(S2 * q1.x - S3 * q2.x - S1 * q3.x, S2 * q1.y - S3 * q2.y - S1 * q3.y);
    float2 b3 = make_float2(S3 * q1.x - S1 * q2.x + S2 * q3.x, S3 * q1.y - S1 * q2.y + S2 * q3.y);
    x0 = make_float2(x0.x + p1.x + p2.x + p3.x, x0.y + p1.y + p2.y + p3.y);
    // X_k = A_k - i B_k ; X_{7-k} = A_k + i B_k
    x1 = make_float2(a1.x + b1.y, a1.y - b1.x);
    x6 = make_float2(a1.x - b1.y, a1.y + b1.x);
    x2 = make_float2(a2.x + b2.y, a2.y - b2.x);
    x5 = make_float2(a2.x - b2.y, a2.y + b2.x);
    x3 = make_float2(a3.x + b3.y, a3.y - b3.x);
    x4 = make_float2(a3.x - b3.y, a3.y + b3.x);
}

// e^{-2 pi i k / 14}, k = 0..6
QHD float2 w14(int k) {
    switch (k) {
        case 0: return make_float2(1.0f, 0.0f);
        case 1: return make_float2(0.90096886790241913f, -0.43388373911755812f);
        case 2: return make_float2(0.62348980185873353f, -0.78183148246802981f);
        case 3: return make_float2(0.22252093395631440f, -0.97492791218182361f);
        case 4: return make_float2(-0.22252093395631440f, -0.97492791218182361f);
        case 5: return make_float2(-0.62348980185873353f, -0.78183148246802981f);
        default: return make_float2(-0.90096886790241913f, -0.43388373911755812f);
    }
}

// 14-point DFT, natural order in and out (radix-2 DIT over two 7-point DFTs)
QHD void dft14(float2 (&x)[16]) {
    float2 e0 = x[0], e1 = x[2], e2 = x[4], e3 = x[6], e4 = x[8], e5 = x[10], e6 = x[12];
    float2 o0 = x[1], o1 = x[3], o2 = x[5], o3 = x[7], o4 = x[9], o5 = x[11], o6 = x[13];
    dft7(e0, e1, e2, e3, e4, e5, e6);
    dft7(o0, o1, o2, o3, o4, o5, o6);
    float2 t;
    x[0] = cadd(e0, o0); x[7] = csub(e0, o0);
    t = cmul(o1, w14(1)); x[1] = cadd(e1, t); x[8] = csub(e1, t);
    t = cmul(o2, w14(2)); x[2] = cadd(e2, t); x[9] = csub(e2, t);
    t = cmul(o3, w14(3)); x[3] = cadd(e3, t); x[10] = csub(e3, t);
    t = cmul(o4, w14(4)); x[4] = cadd(e4, t); x[11] = csub(e4, t);
    t = cmul(o5, w14(5)); x[5] = cadd(e5, t); x[12] = csub(e5, t);
    t = cmul(o6, w14(6)); x[6] = cadd(e6, t); x[13] = csub(e6, t);
}

QHD void dft4(float2& a, float2& b, float2& c, float2& d) {
    float2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = mul_mi(csub(b, d));
    a = cadd(s0, s2);
    c = csub(s0, s2);
    b = cadd(s1, s3);
    d = csub(s1, s3);
}

// e^{-2 pi i k / 16}, k = 0..9 (all that 4x4 needs)
QHD float2 w16(int k) {
    const float c1 = 0.92387953251128674f, s1 = 0.38268343236508977f, r = 0.70710678118654752f;
    switch (k) {
        case 0: return make_float2(1.0f, 0.0f);
        case 1: return make_float2(c1, -s1);
        case 2: return make_float2(r, -r);
        case 3: return make_float2(s1, -c1);
        case 4: return make_float2(0.0f, -1.0f);
        case 6: return make_float2(-r, -r);
        default: return make_float2(-c1, s1);  // k == 9
    }
}

// 16-point DFT, natural order in and out: n = 4a + b, k = ka + 4 kb
QHD void dft16(float2 (&x)[16]) {
#pragma unroll
    for (int b = 0; b < 4; ++b) dft4(x[b], x[4 + b], x[8 + b], x[12 + b]);  // over a; result index ka at x[4 ka + b]
#pragma unroll
    for (int ka = 1; ka < 4; ++ka)
#pragma unroll
        for (int b = 1; b < 4; ++b) x[4 * ka + b] = cmul(x[4 * ka + b], w16(ka * b));
#pragma unroll
    for (int ka = 0; ka < 4; ++ka) dft4(x[4 * ka + 0], x[4 * ka + 1], x[4 * ka + 2], x[4 * ka + 3]);  // over b; kb at x[4 ka + kb]
    // x[4 ka + kb] holds X[ka + 4 kb] -> transpose to natural order
#pragma unroll
    for (int ka = 0; ka < 4; ++ka)
#pragma unroll
        for (int kb = ka + 1; kb < 4; ++kb) {
            float2 t = x[4 * ka + kb];
            x[4 * ka + kb] = x[4 * kb + ka];
            x[4 * kb + ka] = t;
        }
}

// ---- length-224 FFT along a shared-memory column, 16 threads per column -----------
// X[k1 + 14 k2] = sum_{n2} w16^{n2 k2} [ w224^{n2 k1} sum_{n1} x[16 n1 + n2] w14^{n1 k1} ]
// The inverse transform is the forward one with re/im swapped on the way in and out.
template <bool INV>
QHD void fft_s1_load(const float2* col, int n2, const float2* tw, float2 (&a)[16]) {
#pragma unroll
    for (int n1 = 0; n1 < 14; ++n1) {
        float2 v = col[16 * n1 + n2];
        a[n1] = INV ? cswap(v) : v;
    }
    dft14(a);
#pragma unroll
    for (int k1 = 1; k1 < 14; ++k1) a[k1] = cmul(a[k1], tw[n2 * k1]);
}
// (the stage-1 store and the stage-2 store / loads below are shared with the streaming kernels, which also run N = 256: R = N / 16)
template <int N = NF>
QHD void fft_s1_store(float2* col, int n2, const float2 (&a)[16]) {
#pragma unroll
    for (int k1 = 0; k1 < N / 16; ++k1) col[swz(k1, n2)] = a[k1];
}
QHD void fft_s2_load(const float2* col, int k1, float2 (&b)[16]) {
#pragma unroll
    for (int n2 = 0; n2 < 16; ++n2) b[n2] = col[swz(k1, n2)];
    dft16(b);
}
template <bool INV, int N = NF>
QHD void fft_s2_store(float2* col, int k1, const float2 (&b)[16]) {
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) col[k1 + (N / 16) * k2] = INV ? cswap(b[k2]) : b[k2];
}

// ---- sparse m-direction transforms -------------------------------------------------
// forward: partial sum over this CTA's columns of  T[m][k1] * e^{-2 pi i k2 m / 224}
template <int MC>
QHD float2 sampled_dft_partial(const float2* cols, const float2* twp, int m0, int k1, int k2) {
    int idx = (k2 * m0) % NF;
    float ax = 0.f, ay = 0.f;
#pragma unroll 4
    for (int mm = 0; mm < MC; ++mm) {
        float2 t = twp[idx + (idx >> 4)];
        float2 v = cols[mm * CS + k1];
        ax = fmaf(v.x, t.x, ax);
        ax = fmaf(-v.y, t.y, ax);
        ay = fmaf(v.x, t.y, ay);
        ay = fmaf(v.y, t.x, ay);
        idx += k2;
        if (idx >= NF) idx -= NF;
    }
    return make_float2(ax, ay);
}

// inverse: column m of the sparse k-space array,  T'[m][k1] = sum_{j in row k1} c_j e^{+2 pi i k2_j m / 224}.
// `tab` is one of the 8 flat work lists of the frame (op_tables.h): entries k2 | k1 << 8 | j << 16 | last << 31, padded to a
// common length, so the thread (one column m, one list) runs a single branch-free loop and stores a row at its last entry;
// rows without samples appear as one entry with the zero coefficient c[ns_max].  twp: padded twiddles.
QHD void sparse_idft_flat(float2* col, const float2* c, const float2* twp, const uint32_t* tab, int len, int m) {
    float ax = 0.f, ay = 0.f;
#pragma unroll 4
    for (int i = 0; i < len; ++i) {
        const uint32_t en = tab[i];
        const float2 cj = c[(en >> 16) & 0x7fff];
        const uint32_t idx = ((en & 0xff) * (uint32_t)m) % NF;
        const float2 t = twp[idx + (idx >> 4)];  // conj(t) = e^{+...}
        ax = fmaf(cj.x, t.x, ax);
        ax = fmaf(cj.y, t.y, ax);
        ay = fmaf(cj.y, t.x, ay);
        ay = fmaf(-cj.x, t.y, ay);
        if (en & 0x80000000u) {
            col[(en >> 8) & 0xff] = make_float2(ax, ay);
            ax = 0.f;
            ay = 0.f;
        }
    }
}


// =====================================================================================
// Streaming variant (xupdate_stream.cu): one CTA walks the sixteen R-column slabs of a
// (slice, channel) image one after the other, so no cluster exchange is needed.
// Image sides N = 16 R: 224 (R = 14) and 256 (R = 16); the functions below take N as a template
// argument, and the 224 instance is the arithmetic of the original 224-only kernels.
//  * the first forward stage takes its R inputs from registers (loaded straight from
//    global memory), the last inverse stage leaves its R outputs in registers (stored
//    straight to global memory): two shared-memory passes fewer per transform;
//  * the inverse transform runs radix 16 first, radix R last, so that a half-warp's
//    outputs n = c + 16 d are 16 consecutive floats in global memory;
//  * the sparse m-direction sums are evaluated per k-space ROW k1: the thread keeps the
//    R slab values of its row in registers and walks the row's samples with a rotating
//    twiddle (t <- t * e^{-+2 pi i k2 / N}), so the inner loops touch no shared memory.
// tw2[i][j] = e^{-2 pi i (i j) / N}, i, j < 16: stage twiddles, lanes contiguous in j.
// =====================================================================================
template <int N>
struct Side {
    static_assert(N == 224 || N == 256, "streaming kernels: N == M == 224 or 256");
    static constexpr int R = N / 16;            // radix of the first forward / last inverse stage = columns per slab
    static constexpr int CS = N + 1;            // shared-memory column stride in float2 (odd: conflict-free across columns)
    static constexpr int NP = R / 2;            // column pairs per slab in the sparse sums
    static constexpr int OVF_STRIDE = R + 1;    // float2 per overflow partial (R used; odd stride keeps the lanes on different banks)
};
template <int R>
QHD void dft_r(float2 (&x)[16]) {
    if constexpr (R == 14) dft14(x);
    else dft16(x);
}

constexpr int QMAX_STREAM = 64;      // most samples one work item may carry
constexpr int OVF_MAX_STREAM = 96;   // most overflow partials (row chunks beyond the first) per frame

// A shared-memory load the compiler keeps in program order (device code): 15 twiddles fetched ahead of their use on top of
// the 16 complex values of the transform do not fit the 72-register budget of four CTAs per SM.
QHD float2 ld_ordered(const float2* p) {
#if defined(__CUDA_ARCH__)
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"((unsigned)__cvta_generic_to_shared(p)));
    return v;
#else
    return *p;
#endif
}

// forward stage 1 on register inputs: a[n1] = x[16 n1 + n2], n1 < R
template <int N = NF>
QHD void fwd_s1_regs(float2 (&a)[16], int n2, const float2* tw2) {
    constexpr int R = Side<N>::R;
    dft_r<R>(a);
#pragma unroll
    for (int k1 = 1; k1 < R; ++k1) a[k1] = cmul(a[k1], tw2[16 * k1 + n2]);
}

// inverse transform of one column via the swap identity  ifft(U) = swap(fft(swap(U))) (unnormalised):
// input index k = R a + b, output index n = c + 16 d
//   X[c + 16 d] = sum_b wR^{b d} [ wN^{b c} sum_a U[R a + b] w16^{a c} ]
// mask: bit a set = row R a + b holds samples; the other rows of the sparse k-space array are zero and are not read
template <int N = NF>
QHD void inv_s1_load(const float2* col, int b, const float2* tw2, uint32_t mask, float2 (&x)[16]) {
#pragma unroll
    for (int a = 0; a < 16; ++a) x[a] = ((mask >> a) & 1u) ? cswap(col[Side<N>::R * a + b]) : make_float2(0.f, 0.f);
    dft16(x);
#pragma unroll
    for (int c = 1; c < 16; ++c) x[c] = cmul(x[c], ld_ordered(tw2 + 16 * c + b));
}
QHD void inv_s1_store(float2* col, int b, const float2 (&x)[16]) {
#pragma unroll
    for (int c = 0; c < 16; ++c) col[swz(b, c)] = x[c];
}
// leaves x[d] = (inverse transform)[c + 16 d], d < R
template <int N = NF>
QHD void inv_s2_regs(const float2* col, int c, float2 (&x)[16]) {
    constexpr int R = Side<N>::R;
#pragma unroll
    for (int b = 0; b < R; ++b) x[b] = col[swz(b, c)];
    dft_r<R>(x);
#pragma unroll
    for (int d = 0; d < R; ++d) x[d] = cswap(x[d]);
}

// ---- sparse m-direction sums of the streaming kernel -------------------------------------------------
// Work item = (k-space row k1, up to Q of the row's samples, one slab of R columns); ent[q] = j | k2 << 16.
// The R columns are taken in NP = R / 2 pairs mirrored about the centre of the slab, columns NP - 1 - d' and NP + d'
// (d = d' + 1/2):
//   e^{-i phi (base +- d)} = tc * r_d^{+-1},   tc = e^{-i phi base} (base = m0 + NP - 1/2),   r_d = e^{-i phi d},   phi = 2 pi k2 / N
// so with P_d = T[NP+d'] + T[NP-1-d'], M_d = T[NP+d'] - T[NP-1-d'] (formed once per item) a sample costs 4 FMAs and one twiddle
// rotation per column PAIR.  tw2n[x] = e^{-2 pi i x / (2N)} (448 or 512 entries; K1Params::tw448) supplies the half-integer phases.
constexpr int HC_STREAM = Side<NF>::R;
constexpr int NP_STREAM = Side<NF>::NP;          // column pairs per half slab of the real-image kernels
constexpr int OVF_STRIDE = Side<NF>::OVF_STRIDE;

// forward: pc[j] += sum_mm T[mm][k1] e^{-2 pi i k2 (m0 + mm) / N} over the R columns starting at ws (m0 = first column)
template <int N = NF>
QHD void p3_item(const float2* ws, int k1, const uint32_t* ent, int cnt, const float2* tw2n, int m0, float2* pc) {
    constexpr int CS = Side<N>::CS, NP = Side<N>::NP;
    if (cnt == 0) return;
    float2 Pp[NP], Mm[NP];
#pragma unroll
    for (int d = 0; d < NP; ++d) {
        const float2 tp = ws[(NP + d) * CS + k1], tm = ws[(NP - 1 - d) * CS + k1];
        Pp[d] = cadd(tp, tm);
        Mm[d] = csub(tp, tm);
    }
    for (int q = 0; q < cnt; ++q) {
        const uint32_t en = ent[q];
        const int k2 = (int)(en >> 16), j = (int)(en & 0xffffu);
        float2 r = tw2n[k2];          // r_{1/2}
        const float2 st = cmul(r, r);     // e^{-i phi}
        const float2 tc = tw2n[(k2 * (2 * m0 + 2 * NP - 1)) % (2 * N)];
        float ax = 0.f, ay = 0.f;
#pragma unroll
        for (int d = 0; d < NP; ++d) {
            ax = fmaf(r.x, Pp[d].x, ax);
            ax = fmaf(-r.y, Mm[d].y, ax);
            ay = fmaf(r.x, Pp[d].y, ay);
            ay = fmaf(r.y, Mm[d].x, ay);
            r = cmul(r, st);
        }
        const float2 a = cmul(make_float2(ax, ay), tc);
        const float2 o = pc[j];
        pc[j] = make_float2(o.x + a.x, o.y + a.y);
    }
}

// inverse, step 1: partial sums of  U[mm] = sum_j c_j e^{+2 pi i k2_j (m0 + mm) / N}  in the (P, M) basis:
//   SP_d = sum_j u_j Re r_d,  SM_d = sum_j u_j Im r_d,  u_j = c_j conj(tc_j)
template <int N = NF>
QHD void p4_item_partial(float2 (&SP)[Side<N>::NP], float2 (&SM)[Side<N>::NP], const uint32_t* ent, int cnt, const float2* tw2n, int m0,
                         const float2* pc) {
    constexpr int NP = Side<N>::NP;
#pragma unroll
    for (int d = 0; d < NP; ++d) {
        SP[d] = make_float2(0.f, 0.f);
        SM[d] = make_float2(0.f, 0.f);
    }
    for (int q = 0; q < cnt; ++q) {
        const uint32_t en = ent[q];
        const int k2 = (int)(en >> 16), j = (int)(en & 0xffffu);
        float2 r = tw2n[k2];
        const float2 st = cmul(r, r);
        const float2 tc = tw2n[(k2 * (2 * m0 + 2 * NP - 1)) % (2 * N)];
        const float2 u = cmul(pc[j], make_float2(tc.x, -tc.y));
#pragma unroll
        for (int d = 0; d < NP; ++d) {
            SP[d].x = fmaf(u.x, r.x, SP[d].x);
            SP[d].y = fmaf(u.y, r.x, SP[d].y);
            SM[d].x = fmaf(u.x, r.y, SM[d].x);
            SM[d].y = fmaf(u.y, r.y, SM[d].y);
            r = cmul(r, st);
        }
    }
}
// inverse, step 2: a primary item leaves the (P, M) basis and writes its row ...
template <int N = NF>
QHD void p4_item_store(float2* ws, int k1, const float2 (&SP)[Side<N>::NP], const float2 (&SM)[Side<N>::NP]) {
    constexpr int CS = Side<N>::CS, NP = Side<N>::NP;
#pragma unroll
    for (int d = 0; d < NP; ++d) {
        ws[(NP + d) * CS + k1] = make_float2(SP[d].x + SM[d].y, SP[d].y - SM[d].x);       // u conj(r)
        ws[(NP - 1 - d) * CS + k1] = make_float2(SP[d].x - SM[d].y, SP[d].y + SM[d].x);   // u r
    }
}
// ... and, after a barrier, adds the row's overflow partials in slot order (consecutive slots are OVF_STRIDE apart)
template <int N = NF>
QHD void p4_row_add_overflow(float2* ws, int k1, const float2* ovf, int novf) {
    constexpr int CS = Side<N>::CS, NP = Side<N>::NP;
    float2 SP[NP], SM[NP];
#pragma unroll
    for (int d = 0; d < NP; ++d) {
        SP[d] = ovf[d];
        SM[d] = ovf[NP + d];
    }
    for (int i = 1; i < novf; ++i) {
        const float2* o = ovf + (size_t)i * Side<N>::OVF_STRIDE;
#pragma unroll
        for (int d = 0; d < NP; ++d) {
            const float2 a = o[d], b = o[NP + d];
            SP[d].x += a.x; SP[d].y += a.y;
            SM[d].x += b.x; SM[d].y += b.y;
        }
    }
#pragma unroll
    for (int d = 0; d < NP; ++d) {
        float2 up = ws[(NP + d) * CS + k1], um = ws[(NP - 1 - d) * CS + k1];
        ws[(NP + d) * CS + k1] = make_float2(up.x + (SP[d].x + SM[d].y), up.y + (SP[d].y - SM[d].x));
        ws[(NP - 1 - d) * CS + k1] = make_float2(um.x + (SP[d].x - SM[d].y), um.y + (SP[d].y + SM[d].x));
    }
}
template <int N = NF>
QHD void p4_item_spill(float2* o, const float2 (&SP)[Side<N>::NP], const float2 (&SM)[Side<N>::NP]) {
#pragma unroll
    for (int d = 0; d < Side<N>::NP; ++d) {
        o[d] = SP[d];
        o[Side<N>::NP + d] = SM[d];
    }
}

// =====================================================================================
// Real-image variant (xupdate_real.cu): in the loop the transforms only ever see REAL images -
//   forward   m = A v            (v = denoiser output, real)
//   inverse   Re(A^H c)          (only the real part of w = v + A^H c feeds the denoiser)
// so two real columns (m, m+1) ride through one complex length-224 FFT:
//   forward: Z = FFT_n(v[:, m] + i v[:, m+1]);  T_m(k1) = (Z(k1) + conj Z(-k1)) / 2,  T_{m+1}(k1) = (Z(k1) - conj Z(-k1)) / (2i)
//   inverse: Re IFFT2(C) = IFFT2(C_h), C_h(k) = (C(k) + conj C(-k)) / 2 Hermitian, so U_h(k1, m) is Hermitian in k1 for every m
//            and IFFT_n(U_h(., m) + i U_h(., m+1)) = column m + i column m+1.
// A slab is 14 packed columns = 28 real columns; the sparse sums take it as two half slabs of 7 packed = 14 real columns.
// Work items cover FOLDED rows k1 <= 112 (op_tables.h): a sample of row 224 - k1 enters row k1 as (224 - k2) mod 224 with its
// value conjugated - T(224 - k1, m) = conj T(k1, m) - so one item serves both rows from the same registers.
// Entry word: j | k2' << 16 | conj << 31.  Scaling: the forward sums come out 2 x too large (the 1/2 of T is left to the solve
// kernel) and the inverse expects c already multiplied by 1/2 (the 1/2 of C_h).
// =====================================================================================
constexpr int HP_REAL = 7;        // packed columns per half slab

// forward: pc[j] += sum over the 28 real columns of the slab starting at real column m0 of  2 T_m(k1) e^{-2 pi i k2 m / 224}
QHD void p3r_item(const float2* ws, int k1, const uint32_t* ent, int cnt, const float2* tw448, int m0, float2* pc) {
    if (cnt == 0) return;
    const int k1n = k1 ? NF - k1 : 0;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
        // 2 T_a = Z(k1) + conj Z(-k1),  2 T_b = (Z(k1) - conj Z(-k1)) / i;  mirrored about packed column 3 of the half slab
        float2 Ea[4], Em[4], Oa[4], Om[4];  // [0]: centre value in Ea / Oa; [d]: sums (a) and differences (m) of columns 3 + d, 3 - d
        {
            float2 ta[HP_REAL], tb[HP_REAL];
#pragma unroll
            for (int j = 0; j < HP_REAL; ++j) {
                const float2 zp = ws[(HP_REAL * h + j) * CS + k1], zn = ws[(HP_REAL * h + j) * CS + k1n];
                ta[j] = make_float2(zp.x + zn.x, zp.y - zn.y);
                tb[j] = make_float2(zp.y + zn.y, zn.x - zp.x);
            }
            Ea[0] = ta[3];
            Oa[0] = tb[3];
            Em[0] = Om[0] = make_float2(0.f, 0.f);
#pragma unroll
            for (int d = 1; d < 4; ++d) {
                Ea[d] = cadd(ta[3 + d], ta[3 - d]);
                Em[d] = csub(ta[3 + d], ta[3 - d]);
                Oa[d] = cadd(tb[3 + d], tb[3 - d]);
                Om[d] = csub(tb[3 + d], tb[3 - d]);
            }
        }
        const int mh = m0 + 14 * h;
        for (int q = 0; q < cnt; ++q) {
            const uint32_t en = ent[q];
            const int k2 = (int)((en >> 16) & 0xffu), j = (int)(en & 0xffffu);
            const float2 wk = tw448[2 * k2];                           // e^{-i phi}, phi = 2 pi k2 / 224
            const float2 r1 = cmul(wk, wk);                            // e^{-2 i phi}: one packed column
            const float2 tc = tw448[(2 * k2 * (mh + 6)) % (2 * NF)];   // e^{-i phi (mh + 6)}: packed column 3 = real column mh + 6
            float2 r = r1;
            float ex = Ea[0].x, ey = Ea[0].y, ox = Oa[0].x, oy = Oa[0].y;
#pragma unroll
            for (int d = 1; d < 4; ++d) {
                ex = fmaf(r.x, Ea[d].x, ex);
                ex = fmaf(-r.y, Em[d].y, ex);
                ey = fmaf(r.x, Ea[d].y, ey);
                ey = fmaf(r.y, Em[d].x, ey);
                ox = fmaf(r.x, Oa[d].x, ox);
                ox = fmaf(-r.y, Om[d].y, ox);
                oy = fmaf(r.x, Oa[d].y, oy);
                oy = fmaf(r.y, Om[d].x, oy);
                if (d < 3) r = cmul(r, r1);
            }
            const float2 o = cmul(make_float2(ox, oy), wk);            // the odd real column of a pair sits one column further
            float2 a = cmul(make_float2(ex + o.x, ey + o.y), tc);
            if (en & 0x80000000u) a.y = -a.y;                          // sample of row 224 - k1: conj of the sum for (k1, -k2)
            const float2 pv = pc[j];
            pc[j] = make_float2(pv.x + a.x, pv.y + a.y);
        }
    }
}

// inverse, step 1 (one half slab of 14 real columns starting at mh): like p4_item_partial with the folded entries
QHD void p4r_item_partial(float2 (&SP)[NP_STREAM], float2 (&SM)[NP_STREAM], const uint32_t* ent, int cnt, const float2* tw448, int mh,
                          const float2* pc) {
#pragma unroll
    for (int d = 0; d < NP_STREAM; ++d) {
        SP[d] = make_float2(0.f, 0.f);
        SM[d] = make_float2(0.f, 0.f);
    }
    for (int q = 0; q < cnt; ++q) {
        const uint32_t en = ent[q];
        const int k2 = (int)((en >> 16) & 0xffu), j = (int)(en & 0xffffu);
        float2 r = tw448[k2];
        const float2 st = cmul(r, r);
        const float2 tc = tw448[(k2 * (2 * mh + 13)) % (2 * NF)];
        float2 cv = pc[j];
        if (en & 0x80000000u) cv.y = -cv.y;
        const float2 u = cmul(cv, make_float2(tc.x, -tc.y));
#pragma unroll
        for (int d = 0; d < NP_STREAM; ++d) {
            SP[d].x = fmaf(u.x, r.x, SP[d].x);
            SP[d].y = fmaf(u.y, r.x, SP[d].y);
            SM[d].x = fmaf(u.x, r.y, SM[d].x);
            SM[d].y = fmaf(u.y, r.y, SM[d].y);
            r = cmul(r, st);
        }
    }
}
// inverse, step 2: leave the (P, M) basis, pack real column pairs (a, b) = (2 j, 2 j + 1) of the half slab as
//   Zp_j(k1) = G_a + i G_b,   Zp_j(-k1) = conj G_a + i conj G_b      (G = the folded row's partial U_h)
// and store (ACC = false: primary item) or add (ACC = true: overflow partials) rows k1 and 224 - k1 of packed columns 7 h + j.
// Rows 0 and 112 are their own mirror: both contributions land on the same element.
template <bool ACC>
QHD void p4r_store(float2* ws, int k1, int h, const float2 (&SP)[NP_STREAM], const float2 (&SM)[NP_STREAM]) {
    const int k1n = k1 ? NF - k1 : 0;
    float2 G[2 * NP_STREAM];
#pragma unroll
    for (int d = 0; d < NP_STREAM; ++d) {
        G[7 + d] = make_float2(SP[d].x + SM[d].y, SP[d].y - SM[d].x);   // u conj(r)
        G[6 - d] = make_float2(SP[d].x - SM[d].y, SP[d].y + SM[d].x);   // u r
    }
#pragma unroll
    for (int j = 0; j < HP_REAL; ++j) {
        const float2 a = G[2 * j], b = G[2 * j + 1];
        float2 zp = make_float2(a.x - b.y, a.y + b.x);
        const float2 zn = make_float2(a.x + b.y, b.x - a.y);
        float2* colp = ws + (HP_REAL * h + j) * CS;
        if (k1n == k1) {
            zp = make_float2(zp.x + zn.x, zp.y + zn.y);
            if (ACC) {
                const float2 o = colp[k1];
                zp = make_float2(o.x + zp.x, o.y + zp.y);
            }
            colp[k1] = zp;
        } else {
            if (ACC) {
                const float2 o = colp[k1], on = colp[k1n];
                colp[k1] = make_float2(o.x + zp.x, o.y + zp.y);
                colp[k1n] = make_float2(on.x + zn.x, on.y + zn.y);
            } else {
                colp[k1] = zp;
                colp[k1n] = zn;
            }
        }
    }
}
// the row's overflow partials, summed in slot order, then added through the same packing
QHD void p4r_row_add_overflow(float2* ws, int k1, int h, const float2* ovf, int novf, int stride) {
    float2 SP[NP_STREAM], SM[NP_STREAM];
#pragma unroll
    for (int d = 0; d < NP_STREAM; ++d) {
        SP[d] = ovf[d];
        SM[d] = ovf[NP_STREAM + d];
    }
    for (int i = 1; i < novf; ++i) {
        const float2* o = ovf + (size_t)i * stride;
#pragma unroll
        for (int d = 0; d < NP_STREAM; ++d) {
            const float2 a = o[d], b = o[NP_STREAM + d];
            SP[d].x += a.x; SP[d].y += a.y;
            SM[d].x += b.x; SM[d].y += b.y;
        }
    }
    p4r_store<true>(ws, k1, h, SP, SM);
}

// item table words (op_tables.h): A = k1 | cnt << 8 | start << 16 (cnt == 0: no item - every item carries a sample, and k1 == 255
//                                     is a real row at N = 256; the no-item word is 255);
//                                 B = slot | novf << 8 | ovf0 << 16 (slot 0: primary; bits 24-31 unused: rows without samples are
//                                     skipped by the inverse FFT through the row mask)

}  // namespace k1
