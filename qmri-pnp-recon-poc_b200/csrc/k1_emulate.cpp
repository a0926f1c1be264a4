// CPU emulation of the K1 kernel's control flow, thread by thread, using the very same
// phase functions (xupdate_phases.cuh) and tables (op_tables.h) as the CUDA kernel.
// TEST INFRASTRUCTURE: built into libk1emu.so by __graft_entry__.build() and driven by
// tests/test_k1_emulation.py, because the build container has no GPU.  Never shipped in,
// nor called by, libqmri_b200.so.
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "op_tables.h"
#include "xupdate_phases.cuh"

using namespace k1;

template <int MC>
static void emulate(int mode, int C, int S, const optab::K1Tables& t, const float* in_re, const float* in_im,
                    const float* v, const float* y, float rho, float* out_re, float* out_im, float* y_out,
                    float* minmax) {
    constexpr int THREADS = 8 * MC, CL = NF / MC, GROUPS = THREADS / 16, ROUNDS = MC / GROUPS;
    const float2* tw = reinterpret_cast<const float2*>(t.tw.data());
    std::vector<float2> twp(TWP, float2{0, 0});  // padded copy, as the kernel builds it in shared memory
    for (int i = 0; i < NF; ++i) twp[i + (i >> 4)] = tw[i];
    const size_t plane = (size_t)NF * NF;
    for (int s = 0; s < S; ++s) {
        float lmin = INFINITY, lmax = -INFINITY;
        for (int c = 0; c < C; ++c) {
            const int f0 = t.frame_ptr[c], ns = t.frame_ptr[c + 1] - f0;
            std::vector<std::vector<float2>> cols(CL, std::vector<float2>((size_t)MC * CS, float2{0, 0}));
            std::vector<std::vector<float2>> pc(CL, std::vector<float2>(t.ns_max + 1, float2{0, 0}));  // [ns_max] stays zero
            const size_t base = ((size_t)(s * C + c)) * plane;
            auto run_fft = [&](int r, bool inv) {
                for (int rd = 0; rd < ROUNDS; ++rd) {
                    std::vector<float2> regs((size_t)THREADS * 16);
                    for (int tid = 0; tid < THREADS; ++tid) {
                        float2* col = cols[r].data() + (rd * GROUPS + (tid >> 4)) * CS;
                        float2(&a)[16] = *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]);
                        if (inv) fft_s1_load<true>(col, tid & 15, tw, a);
                        else fft_s1_load<false>(col, tid & 15, tw, a);
                    }
                    for (int tid = 0; tid < THREADS; ++tid) {
                        float2* col = cols[r].data() + (rd * GROUPS + (tid >> 4)) * CS;
                        fft_s1_store(col, tid & 15, *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]));
                    }
                    for (int tid = 0; tid < THREADS; ++tid) {
                        float2* col = cols[r].data() + (rd * GROUPS + (tid >> 4)) * CS;
                        if ((tid & 15) < 14) fft_s2_load(col, tid & 15, *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]));
                    }
                    for (int tid = 0; tid < THREADS; ++tid) {
                        float2* col = cols[r].data() + (rd * GROUPS + (tid >> 4)) * CS;
                        if ((tid & 15) < 14) {
                            if (inv) fft_s2_store<true>(col, tid & 15, *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]));
                            else fft_s2_store<false>(col, tid & 15, *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]));
                        }
                    }
                }
            };
            if (mode != 3) {
                for (int r = 0; r < CL; ++r) {
                    const size_t slab = base + (size_t)r * MC * NF;
                    for (int e = 0; e < MC * NF; ++e) {
                        int mm = e / NF, n = e % NF;
                        float re = in_re[slab + e], im = in_im ? in_im[slab + e] : 0.f;
                        if (mode == 0) {
                            re = 2.f * v[slab + e] - re;
                            im = -im;
                        }
                        cols[r][mm * CS + n] = float2{re, im};
                    }
                    run_fft(r, false);
                    for (int j = 0; j < ns; ++j) {
                        uint16_t kk = t.samp[f0 + j];
                        pc[r][j] = sampled_dft_partial<MC>(cols[r].data(), twp.data(), r * MC, kk & 0xff, kk >> 8);
                    }
                }
                const float inv_n = 1.0f / (float)NF;
                std::vector<float2> cfull(t.ns_max + 1, float2{0, 0});
                for (int j = 0; j < ns; ++j) {
                    float sx = 0.f, sy = 0.f;
                    for (int r = 0; r < CL; ++r) {
                        sx += pc[r][j].x;
                        sy += pc[r][j].y;
                    }
                    sx *= inv_n;
                    sy *= inv_n;
                    size_t yi = (size_t)s * t.nmeas + f0 + j;
                    if (mode == 2) {
                        y_out[2 * yi] = sx;
                        y_out[2 * yi + 1] = sy;
                    } else {
                        float g = (1.0f / (1.0f + rho)) * inv_n;
                        cfull[j] = float2{(y[2 * yi] - sx) * g, (y[2 * yi + 1] - sy) * g};
                    }
                }
                if (mode == 2) continue;
                for (int r = 0; r < CL; ++r) pc[r] = cfull;
            } else {
                const float inv_n = 1.0f / (float)NF;
                for (int r = 0; r < CL; ++r)
                    for (int j = 0; j < ns; ++j) {
                        size_t yi = (size_t)s * t.nmeas + f0 + j;
                        pc[r][j] = float2{y[2 * yi] * inv_n, y[2 * yi + 1] * inv_n};
                    }
            }
            for (int r = 0; r < CL; ++r) {
                for (int tid = 0; tid < THREADS; ++tid) {
                    const int mm = tid % MC, ph = tid / MC;
                    sparse_idft_flat(cols[r].data() + mm * CS, pc[r].data(), twp.data(),
                                     t.p4tab.data() + ((size_t)c * optab::K1_PHASES + ph) * t.p4_len, t.p4_len, r * MC + mm);
                }
                run_fft(r, true);
                const size_t slab = base + (size_t)r * MC * NF;
                for (int e = 0; e < MC * NF; ++e) {
                    int mm = e / NF, n = e % NF;
                    float2 cr = cols[r][mm * CS + n];
                    float ore, oim;
                    if (mode == 0) {
                        ore = v[slab + e] + cr.x;
                        oim = cr.y;
                    } else if (mode == 1) {
                        ore = in_re[slab + e] + cr.x;
                        oim = (in_im ? in_im[slab + e] : 0.f) + cr.y;
                    } else {
                        ore = cr.x;
                        oim = cr.y;
                    }
                    out_re[slab + e] = ore;
                    out_im[slab + e] = oim;
                    lmin = fminf(lmin, ore);
                    lmax = fmaxf(lmax, ore);
                }
            }
        }
        if (minmax) {
            minmax[2 * s] = lmin;
            minmax[2 * s + 1] = lmax;
        }
    }
}

// Streaming kernels (xupdate_stream.cu): forward kernel per slab group (G CTAs per image, N threads each), solve kernel,
// adjoint kernel - same control flow, thread by thread.
template <int N>
static void emulate_stream(int mode, int C, int S, const optab::K1Tables& t, const float* in_re, const float* in_im,
                           const float* v, const float* y, float rho, float* out_re, float* out_im, float* y_out,
                           float* minmax) {
    constexpr int MC = Side<N>::R, CS = Side<N>::CS, NP = Side<N>::NP, OVF_STRIDE = Side<N>::OVF_STRIDE;
    constexpr int THREADS = 16 * MC, SLABS = N / MC, G = 4, SPC = SLABS / G;
    const float2* tw2 = reinterpret_cast<const float2*>(t.tw2.data());
    const float2* tw448 = reinterpret_cast<const float2*>(t.tw448.data());
    const size_t plane = (size_t)N * N;
    const float inv_n = 1.0f / (float)N;
    for (int s = 0; s < S; ++s) {
        float lmin = INFINITY, lmax = -INFINITY;
        for (int c = 0; c < C; ++c) {
            const int f0 = t.frame_ptr[c], ns = t.frame_ptr[c + 1] - f0;
            const size_t img = ((size_t)(s * C + c)) * plane;
            const uint32_t* ent = t.ent.data() + f0;
            const uint32_t* itA = t.itA.data() + (size_t)c * N;
            const uint32_t* itB = t.itB.data() + (size_t)c * N;
            std::vector<float2> regs((size_t)THREADS * 16);
            auto A = [&](int tid) -> float2(&)[16] { return *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]); };
            std::vector<float2> cvec((size_t)t.ns_max + 1, float2{0, 0});
            if (mode == 3) {
                for (int j = 0; j < ns; ++j) {
                    size_t yi = (size_t)s * t.nmeas + f0 + j;
                    cvec[j] = float2{y[2 * yi] * inv_n, y[2 * yi + 1] * inv_n};
                }
            } else {
                std::vector<std::vector<float2>> part(G, std::vector<float2>((size_t)t.ns_max + 1, float2{0, 0}));
                for (int g = 0; g < G; ++g) {  // one forward CTA
                    std::vector<float2> ws((size_t)MC * CS, float2{0, 0});
                    std::vector<float2>& pc = part[g];
                    for (int sl = 0; sl < SPC; ++sl) {
                        const int m0 = (g * SPC + sl) * MC;
                        for (int tid = 0; tid < THREADS; ++tid) {
                            const int l16 = tid & 15, col = tid >> 4;
                            const size_t gi = img + (size_t)(m0 + col) * N + l16;
                            float2(&a)[16] = A(tid);
                            for (int n1 = 0; n1 < MC; ++n1) {
                                float re = in_re[gi + 16 * n1], im = in_im ? in_im[gi + 16 * n1] : 0.f;
                                if (mode == 0) {
                                    re = 2.f * v[gi + 16 * n1] - re;
                                    im = -im;
                                }
                                a[n1] = float2{re, im};
                            }
                            fwd_s1_regs<N>(a, l16, tw2);
                        }
                        for (int tid = 0; tid < THREADS; ++tid) fft_s1_store<N>(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            if ((tid & 15) < MC) fft_s2_load(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            if ((tid & 15) < MC) fft_s2_store<false, N>(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            p3_item<N>(ws.data(), (int)(itA[tid] & 0xffu), ent + (itA[tid] >> 16), (int)((itA[tid] >> 8) & 0xffu), tw448, m0, pc.data());
                    }
                }
                for (int j = 0; j < ns; ++j) {  // solve kernel
                    size_t yi = (size_t)s * t.nmeas + f0 + j;
                    float sx = 0.f, sy = 0.f;
                    for (int g = 0; g < G; ++g) {
                        sx += part[g][j].x;
                        sy += part[g][j].y;
                    }
                    sx *= inv_n;
                    sy *= inv_n;
                    if (mode == 2) {
                        y_out[2 * yi] = sx;
                        y_out[2 * yi + 1] = sy;
                    } else {
                        float gsc = (1.0f / (1.0f + rho)) * inv_n;
                        cvec[j] = float2{(y[2 * yi] - sx) * gsc, (y[2 * yi + 1] - sy) * gsc};
                    }
                }
                if (mode == 2) continue;
            }
            for (int g = 0; g < G; ++g) {  // one adjoint CTA
                std::vector<float2> ws((size_t)MC * CS, float2{0, 0});
                std::vector<float2> ovf((size_t)std::max(t.n_ovf, 1) * OVF_STRIDE, float2{0, 0});
                for (int sl = 0; sl < SPC; ++sl) {
                    const int m0 = (g * SPC + sl) * MC;
                    for (auto& e : ws) e = float2{NAN, NAN};  // rows without samples are never written: they must never be read either
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int k1row = (int)(itA[tid] & 0xffu), cnt = (int)((itA[tid] >> 8) & 0xffu), slot = (int)(itB[tid] & 0xffu);
                        if (cnt != 0) {
                            float2 SP[NP], SM[NP];
                            p4_item_partial<N>(SP, SM, ent + (itA[tid] >> 16), cnt, tw448, m0, cvec.data());
                            if (slot == 0) p4_item_store<N>(ws.data(), k1row, SP, SM);
                            else p4_item_spill<N>(ovf.data() + (size_t)(slot - 1) * OVF_STRIDE, SP, SM);
                        }
                    }
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int k1row = (int)(itA[tid] & 0xffu), cnt = (int)((itA[tid] >> 8) & 0xffu), slot = (int)(itB[tid] & 0xffu);
                        const int novf = (int)((itB[tid] >> 8) & 0xffu), ovf0 = (int)((itB[tid] >> 16) & 0xffu);
                        if (cnt != 0 && slot == 0 && novf) p4_row_add_overflow<N>(ws.data(), k1row, ovf.data() + (size_t)ovf0 * OVF_STRIDE, novf);
                    }
                    for (int tid = 0; tid < THREADS; ++tid)
                        if ((tid & 15) < MC) inv_s1_load<N>(ws.data() + (tid >> 4) * CS, tid & 15, tw2, t.rowmask[(size_t)c * 16 + (tid & 15)], A(tid));
                    for (int tid = 0; tid < THREADS; ++tid)
                        if ((tid & 15) < MC) inv_s1_store(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int l16 = tid & 15, col = tid >> 4;
                        const size_t gi = img + (size_t)(m0 + col) * N + l16;
                        float2(&a)[16] = A(tid);
                        inv_s2_regs<N>(ws.data() + col * CS, l16, a);
                        for (int d = 0; d < MC; ++d) {
                            float ore, oim;
                            if (mode == 0) {
                                ore = v[gi + 16 * d] + a[d].x;
                                oim = a[d].y;
                            } else if (mode == 1) {
                                ore = in_re[gi + 16 * d] + a[d].x;
                                oim = (in_im ? in_im[gi + 16 * d] : 0.f) + a[d].y;
                            } else {
                                ore = a[d].x;
                                oim = a[d].y;
                            }
                            out_re[gi + 16 * d] = ore;
                            out_im[gi + 16 * d] = oim;
                            lmin = fminf(lmin, ore);
                            lmax = fmaxf(lmax, ore);
                        }
                    }
                }
            }
        }
        if (minmax) {
            minmax[2 * s] = lmin;
            minmax[2 * s + 1] = lmax;
        }
    }
}

// Real-image streaming kernels (xupdate_real.cu), thread by thread: op 0 = forward (y_out = A v), op 1 = adjoint
// (out = v + Re(A^H c), c handed over in `y`).  Same phase functions, folded-row tables and scalings as the CUDA kernels.
static void emulate_real(int op, int C, int S, const optab::K1Tables& t, const float* v, const float* y, float* out, float* y_out,
                         float* minmax) {
    constexpr int PC = 14, THREADS = 16 * PC, SLABS = NF / (2 * PC), G = 2, SPC = SLABS / G;
    const float2* tw2 = reinterpret_cast<const float2*>(t.tw2.data());
    const float2* tw448 = reinterpret_cast<const float2*>(t.tw448.data());
    const size_t plane = (size_t)NF * NF;
    const float inv_n = 1.0f / (float)NF;
    for (int s = 0; s < S; ++s) {
        float lmin = INFINITY, lmax = -INFINITY;
        for (int c = 0; c < C; ++c) {
            const int f0 = t.frame_ptr[c], ns = t.frame_ptr[c + 1] - f0;
            const size_t img = ((size_t)(s * C + c)) * plane;
            const uint32_t* ent = t.r_ent.data() + f0;
            const uint32_t* itA = t.r_itA.data() + (size_t)c * NF;
            const uint32_t* itB = t.r_itB.data() + (size_t)c * NF;
            std::vector<float2> regs((size_t)THREADS * 16);
            auto A = [&](int tid) -> float2(&)[16] { return *reinterpret_cast<float2(*)[16]>(&regs[(size_t)tid * 16]); };
            if (op == 0) {
                std::vector<std::vector<float2>> part(G, std::vector<float2>((size_t)t.ns_max + 1, float2{0, 0}));
                for (int g = 0; g < G; ++g) {
                    std::vector<float2> ws((size_t)PC * CS, float2{0, 0});
                    for (int sl = 0; sl < SPC; ++sl) {
                        const int m0 = (g * SPC + sl) * 2 * PC;
                        for (int tid = 0; tid < THREADS; ++tid) {
                            const int l16 = tid & 15, col = tid >> 4;
                            const size_t gi = img + (size_t)(m0 + 2 * col) * NF + l16;
                            float2(&a)[16] = A(tid);
                            for (int n1 = 0; n1 < 14; ++n1) a[n1] = float2{v[gi + 16 * n1], v[gi + NF + 16 * n1]};
                            fwd_s1_regs(a, l16, tw2);
                        }
                        for (int tid = 0; tid < THREADS; ++tid) fft_s1_store(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            if ((tid & 15) < 14) fft_s2_load(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            if ((tid & 15) < 14) fft_s2_store<false>(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                        for (int tid = 0; tid < THREADS; ++tid)
                            p3r_item(ws.data(), (int)(itA[tid] & 0xffu), ent + (itA[tid] >> 16), (int)((itA[tid] >> 8) & 0xffu), tw448, m0, part[g].data());
                    }
                }
                for (int j = 0; j < ns; ++j) {
                    const size_t yi = (size_t)s * t.nmeas + f0 + j;
                    float sx = 0.f, sy = 0.f;
                    for (int g = 0; g < G; ++g) {
                        sx += part[g][j].x;
                        sy += part[g][j].y;
                    }
                    y_out[2 * yi] = sx * (0.5f * inv_n);
                    y_out[2 * yi + 1] = sy * (0.5f * inv_n);
                }
                continue;
            }
            std::vector<float2> cvec((size_t)t.ns_max + 1, float2{0, 0});
            for (int j = 0; j < ns; ++j) {
                const size_t yi = (size_t)s * t.nmeas + f0 + j;
                cvec[j] = float2{y[2 * yi] * (0.5f * inv_n), y[2 * yi + 1] * (0.5f * inv_n)};
            }
            for (int g = 0; g < G; ++g) {
                std::vector<float2> ws((size_t)PC * CS, float2{0, 0});
                std::vector<float2> ovf((size_t)std::max(t.r_n_ovf, 1) * 2 * OVF_STRIDE, float2{0, 0});
                for (int sl = 0; sl < SPC; ++sl) {
                    const int m0 = (g * SPC + sl) * 2 * PC;
                    for (auto& e : ws) e = float2{NAN, NAN};  // rows outside the symmetric row mask are never written nor read
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int k1row = (int)(itA[tid] & 0xffu), cnt = (int)((itA[tid] >> 8) & 0xffu), slot = (int)(itB[tid] & 0xffu);
                        if (cnt == 0) continue;
                        for (int h = 0; h < 2; ++h) {
                            float2 SP[NP_STREAM], SM[NP_STREAM];
                            p4r_item_partial(SP, SM, ent + (itA[tid] >> 16), cnt, tw448, m0 + 14 * h, cvec.data());
                            if (slot == 0) p4r_store<false>(ws.data(), k1row, h, SP, SM);
                            else p4_item_spill(ovf.data() + ((size_t)(slot - 1) * 2 + h) * OVF_STRIDE, SP, SM);
                        }
                    }
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int k1row = (int)(itA[tid] & 0xffu), cnt = (int)((itA[tid] >> 8) & 0xffu), slot = (int)(itB[tid] & 0xffu);
                        const int novf = (int)((itB[tid] >> 8) & 0xffu), ovf0 = (int)((itB[tid] >> 16) & 0xffu);
                        if (cnt != 0 && slot == 0 && novf)
                            for (int h = 0; h < 2; ++h)
                                p4r_row_add_overflow(ws.data(), k1row, h, ovf.data() + ((size_t)ovf0 * 2 + h) * OVF_STRIDE, novf, 2 * OVF_STRIDE);
                    }
                    for (int tid = 0; tid < THREADS; ++tid)
                        if ((tid & 15) < 14) inv_s1_load(ws.data() + (tid >> 4) * CS, tid & 15, tw2, t.r_rowmask[(size_t)c * 16 + (tid & 15)], A(tid));
                    for (int tid = 0; tid < THREADS; ++tid)
                        if ((tid & 15) < 14) inv_s1_store(ws.data() + (tid >> 4) * CS, tid & 15, A(tid));
                    for (int tid = 0; tid < THREADS; ++tid) {
                        const int l16 = tid & 15, col = tid >> 4;
                        const size_t gi = img + (size_t)(m0 + 2 * col) * NF + l16;
                        float2(&a)[16] = A(tid);
                        inv_s2_regs(ws.data() + col * CS, l16, a);
                        for (int d = 0; d < 14; ++d) {
                            const float oa = v[gi + 16 * d] + a[d].x, ob = v[gi + NF + 16 * d] + a[d].y;
                            out[gi + 16 * d] = oa;
                            out[gi + NF + 16 * d] = ob;
                            lmin = fminf(lmin, fminf(oa, ob));
                            lmax = fmaxf(lmax, fmaxf(oa, ob));
                        }
                    }
                }
            }
        }
        if (minmax) {
            minmax[2 * s] = lmin;
            minmax[2 * s + 1] = lmax;
        }
    }
}

extern "C" {

// pattern: 0 = spiral(S_curve = (int)arg), 1 = epi(percentage = arg).  Returns nmeas; fills idx/frame_ptr when non-null.
int k1emu_masks(int pattern, int N, double arg, int L, int32_t* idx, int64_t* frame_ptr) {
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(N, (int)arg, L, frames);
    else optab::epi_frames(N, N, arg, L, frames);
    int64_t n = 0;
    for (int f = 0; f < L; ++f) {
        if (frame_ptr) frame_ptr[f] = n;
        for (int32_t k : frames[f]) {
            if (idx) idx[n] = k;
            ++n;
        }
    }
    if (frame_ptr) frame_ptr[L] = n;
    return (int)n;
}

// mode: 0 ADMM (in = w, v given, out = w'), 1 SOLVE (in = z, out = x), 2 FORWARD (in = x, y_out), 3 ADJOINT (y, out)
int k1emu_run(int mode, int mc, int pattern, double arg, int C, int S, const float* in_re, const float* in_im,
              const float* v, const float* y, float rho, float* out_re, float* out_im, float* y_out, float* minmax) {
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(NF, (int)arg, C, frames);
    else optab::epi_frames(NF, NF, arg, C, frames);
    optab::K1Tables t;
    const char* env = getenv("QMRI_K1_QMIN");  // same knob and default as the library (qmri_api.cu)
    optab::build_k1_tables(NF, frames, t, env ? atoi(env) : 8);
    if (mc == 0) {  // streaming kernel
        if (!t.stream_ok) return -1;
        emulate_stream<NF>(mode, C, S, t, in_re, in_im, v, y, rho, out_re, out_im, y_out, minmax);
        return t.nmeas;
    }
    if (mc == 56) emulate<56>(mode, C, S, t, in_re, in_im, v, y, rho, out_re, out_im, y_out, minmax);
    else emulate<28>(mode, C, S, t, in_re, in_im, v, y, rho, out_re, out_im, y_out, minmax);
    return t.nmeas;
}

// The streaming kernels at image side n (224 or 256; N == M), same modes and arguments as k1emu_run.  Returns nmeas, -1 if the
// mask does not fit the work-item tables, -2 for another side.
int k1emu_run_n(int n, int mode, int pattern, double arg, int C, int S, const float* in_re, const float* in_im, const float* v,
                const float* y, float rho, float* out_re, float* out_im, float* y_out, float* minmax) {
    if (n != 224 && n != 256) return -2;
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(n, (int)arg, C, frames);
    else optab::epi_frames(n, n, arg, C, frames);
    optab::K1Tables t;
    const char* env = getenv("QMRI_K1_QMIN");
    optab::build_k1_tables(n, frames, t, env ? atoi(env) : 8);
    if (!t.stream_ok) return -1;
    if (n == 224) emulate_stream<224>(mode, C, S, t, in_re, in_im, v, y, rho, out_re, out_im, y_out, minmax);
    else emulate_stream<256>(mode, C, S, t, in_re, in_im, v, y, rho, out_re, out_im, y_out, minmax);
    return t.nmeas;
}

// The streaming kernels' work-item tables (op_tables.h) at image side n for C frames of a mask: itA / itB [C][n], ent [nmeas],
// rowmask [C][16] (each may be null).  Returns nmeas, -1 if the mask does not fit the tables.
int k1emu_stream_tables(int n, int pattern, double arg, int C, uint32_t* itA, uint32_t* itB, uint32_t* ent, uint16_t* rowmask) {
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(n, (int)arg, C, frames);
    else optab::epi_frames(n, n, arg, C, frames);
    optab::K1Tables t;
    const char* env = getenv("QMRI_K1_QMIN");
    optab::build_k1_tables(n, frames, t, env ? atoi(env) : 8);
    if (!t.stream_ok) return -1;
    if (itA) memcpy(itA, t.itA.data(), sizeof(uint32_t) * t.itA.size());
    if (itB) memcpy(itB, t.itB.data(), sizeof(uint32_t) * t.itB.size());
    if (ent) memcpy(ent, t.ent.data(), sizeof(uint32_t) * t.nmeas);
    if (rowmask) memcpy(rowmask, t.rowmask.data(), sizeof(uint16_t) * t.rowmask.size());
    return t.nmeas;
}

// real-image kernels: op 0 forward (v -> y_out), op 1 adjoint (c in y, out = v + Re(A^H c)).  Returns nmeas, -1 if the mask does
// not fit the folded work-item tables; *n_ovf receives the overflow-slot count (what sizes the kernels' shared memory).
int k1emu_run_real(int op, int pattern, double arg, int C, int S, const float* v, const float* y, float* out, float* y_out, float* minmax,
                   int* n_ovf) {
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(NF, (int)arg, C, frames);
    else optab::epi_frames(NF, NF, arg, C, frames);
    optab::K1Tables t;
    const char* env = getenv("QMRI_K1_QMIN");
    optab::build_k1_tables(NF, frames, t, env ? atoi(env) : 8);
    if (!t.real_ok) return -1;
    if (n_ovf) *n_ovf = t.r_n_ovf;
    emulate_real(op, C, S, t, v, y, out, y_out, minmax);
    return t.nmeas;
}

// General V host logic (op_tables.h): union / membership tables and the per-location inverses (G_u + rho I)^{-1}.
// Returns nU; fills ulist [nU], nparts, and Minv [nU][C][C] when non-null.
int k1emu_general(int pattern, double arg, int L, int C, const double* V, double rho, int32_t* ulist, int* nparts, float* Minv) {
    std::vector<std::vector<int32_t>> frames;
    if (pattern == 0) optab::spiral_frames(NF, (int)arg, L, frames);
    else optab::epi_frames(NF, NF, arg, L, frames);
    optab::GeneralTables g;
    const char* env = getenv("QMRI_K1_QMIN");
    optab::build_general_tables(NF, frames, V, L, C, g, env ? atoi(env) : 8);
    if (!g.ok) return -1;
    if (ulist) memcpy(ulist, g.ulist.data(), sizeof(int32_t) * g.nU);
    if (nparts) *nparts = (int)g.parts.size();
    if (Minv) {
        std::vector<float> m;
        optab::general_inverses(g, rho, m);
        memcpy(Minv, m.data(), sizeof(float) * m.size());
    }
    // every measurement must be reachable from its union slot and the parts must tile the union
    int64_t covered = 0;
    for (size_t p = 0; p < g.parts.size(); ++p) covered += g.parts[p].nmeas;
    if (covered != g.nU || (int)g.memb_meas.size() != (int)g.meas_u.size()) return -2;
    for (int u = 0; u < g.nU; ++u)
        for (int e = g.memb_ptr[u]; e < g.memb_ptr[u + 1]; ++e)
            if (g.meas_u[g.memb_meas[e]] != u || g.meas_frame[g.memb_meas[e]] != g.memb_frame[e]) return -3;
    return g.nU;
}
}
