// FISP-MRF dictionary simulation (EPG) and its temporal Gram matrix - host interface of csrc/fisp_kernels.cu.
#pragma once
#include "common.cuh"

// Longest schedule the simulation kernel holds in registers: orders k = 32 j + lane, j < 16, and at most (T - 1) / 2 + 1 orders are
// ever live (DESIGN.md §4, FISP dictionary).
constexpr int FISP_MAX_T = 1024;
constexpr int FISP_MAX_C = 16;

struct FispParams {
    int T = 0;
    const float4* pulse = nullptr;  // [T] (cos^2(a/2), sin^2(a/2), sin a, cos a) of each flip angle a
    const float* tr = nullptr;      // [T] repetition times, seconds
    const float* lut = nullptr;     // K x 2 column-major (T1, T2), seconds
    int64_t K = 0;
    int64_t a0 = 0, a1 = 0;         // atoms simulated by this launch
    double te = 0.0, ti = 0.0;
    int inversion = 0;
    // signals: sig[i * ld + (k - a0)]
    float* sig = nullptr;
    int64_t ld = 0;
    // compress: V [T][C] (pulse-major), D [C][a1 - a0] (column-major rows = atoms), normD [a1 - a0]
    const float* V = nullptr;
    int C = 0;
    float* D = nullptr;
    float* normD = nullptr;
};

int fisp_launch_signals(qmri_ctx* ctx, const FispParams& p);
int fisp_launch_compress(qmri_ctx* ctx, const FispParams& p);

// Gram matrix of fingerprints held as X[i * ld + k], i < T, k < n.  The n atoms are split into `parts` contiguous ranges; range p
// adds its products to part[p] (T x T doubles, upper tiles only), so every element has exactly one writer: no atomics, and the
// same inputs give the same bits.  fisp_gram_parts picks `parts` for T; fisp_gram_reduce sums the parts in order into the
// symmetric G (T x T).
int fisp_gram_parts(int T);
int fisp_launch_gram_accumulate(qmri_ctx* ctx, const float* X, int64_t ld, int64_t n, int T, double* part, int parts);
int fisp_launch_gram_reduce(qmri_ctx* ctx, const double* part, int parts, int T, double* G);
