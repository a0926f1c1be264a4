// Host-visible interface of the K1 kernel (see xupdate_kernel.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct qmri_ctx;

constexpr int K1_PHASES = 8;  // == optab::K1_PHASES

enum { K1_ADMM = 0, K1_SOLVE = 1, K1_FORWARD = 2, K1_ADJOINT = 3 };
enum { K1_STAGE_FWD_ONLY = 1, K1_STAGE_ADJ_ONLY = 2, K1_STAGE_NO_SOLVE = 4 };

struct K1Params {
    // planar fp32 images [S][C][M][N] (n fastest - the MATLAB layout of an N x M x C x S array)
    const float* in_re;   // ADMM: Re w       SOLVE/FORWARD: Re z
    const float* in_im;   // ADMM: Im w       SOLVE/FORWARD: Im z (may be null = real input)
    const float* v;       // ADMM: denoised v (real)
    float* out_re;        // ADMM: Re w'      SOLVE: Re x      ADJOINT: Re A^H y
    float* out_im;
    float* x_re;          // ADMM only, optional: x of this iteration (written on the last one)
    float* x_im;
    const float2* y;      // [S][nmeas] measurements
    float2* y_out;        // FORWARD: [S][nmeas]
    int* minmax;          // optional [S][2] ordered-int min / max of out_re
    // per-operator tables (device)
    const float2* tw;        // [N] e^{-2 pi i t / N}
    const int* frame_ptr;    // [C+1]
    const uint16_t* samp;    // [nmeas] k1 | k2 << 8, frame-major, ascending k = k1 + N k2
    const uint32_t* p4tab;   // [C][8][p4_len] flat work lists of the sparse inverse pass (op_tables.h)
    int p4_len;
    // streaming kernel tables (xupdate_stream.cu; op_tables.h)
    const float2* tw2;       // [16][16] e^{-2 pi i (i j) / N}
    const float2* tw448;     // [2N] e^{-2 pi i t / (2N)} (2N entries)
    const uint32_t* itA;     // [C][N] work item of thread tid: k1 | cnt << 8 | start << 16 (cnt == 0: no item)
    const uint32_t* itB;     // [C][N] slot | novf << 8 | ovf0 << 16
    const uint32_t* ent;     // [nmeas] j | k2 << 16, frame-major, grouped by item
    const uint16_t* rowmask; // [C][16] non-empty rows, by inverse-FFT lane
    int n_ovf;               // overflow partials per frame (sizes the shared-memory slots)
    float2* part;            // scratch [S][C][G][ns_max] partial sample sums of the forward kernel
    float2* cbuf;            // scratch [S][C][ns_max]    c = (y - A z) / (1 + rho)
    int slot_off;            // general V: first union slot of the part these tables cover (0 otherwise)
    int slot_stride;         // samples per image in part / cbuf (general V: the whole union; otherwise ns_max; set by k1_stream_launch)
    int stage;               // general V: K1_STAGE_FWD_ONLY / K1_STAGE_ADJ_ONLY run one half of the streaming path (0 = both)
    int shared_mask;         // general V: every channel is transformed on the same (union) mask - tables of "frame" 0, cbuf in all modes
    int G;                   // slab groups (CTAs) per image: 2, 4, 8 or 16
    int slabs_per_cta;       // 16 / G (set by k1_stream_launch)
    int C;
    int nmeas;
    int ns_max;              // largest per-frame sample count (sizes the shared-memory tables; set by k1_launch)
    int mode;
    float inv_1p_rho;
    double rho;              // host side only (general V: selects the precomputed (G_k + rho I)^{-1})
    int nf;                  // image side N == M: 224 (every kernel) or 160, 192, 256 (streaming kernels only)
    // PnP-ADMM progress monitor (qmri_admm_monitor; streaming kernels, modes ADMM and SOLVE): the monitored kernel instances write
    // double partial sums, each reduced in a fixed order.  Null: the unmonitored instances run.
    double* mon_dc;          // [S][C] sum over the channel's samples of |y - A z|^2 (stream_solve_kernel; general V: GeneralMix)
    double* mon_gt;          // [S][C][G] sum over the CTA's pixels of |gt - x|^2 (stream_adj_kernel; needs gt_re)
    const float* gt_re;      // [S][C][M][N] ground truth
    const float* gt_im;      // optional imaginary plane (null: real ground truth)
};

int k1_launch(qmri_ctx* ctx, const K1Params& p, int S, int ns_max, int mc);  // cluster kernel: N == M == 224 only
constexpr int K1_STREAM_MIN_IMAGES_DIV = 8;  // streaming kernels from S * C >= SM count / 8 images on (two 10-channel slices on B200)
// streaming variant: G CTAs per (slice, channel); needs K1Tables::stream_ok.  The only x-update kernels for N != 224.
int k1_stream_groups(int S, int C, int sm_count);
size_t k1_stream_part_elems(int S, int C, int G, int ns_max);
size_t k1_stream_cbuf_elems(int S, int C, int ns_max);
int k1_stream_launch(qmri_ctx* ctx, const K1Params& p, int S, int ns_max);
int k1_minmax_init(qmri_ctx* ctx, int* minmax, int S);

// real-image variant of the streaming kernels (xupdate_real.cu): the PnP-ADMM loop with only real images crossing HBM
struct K1RealParams {
    const float* v;          // [S][C][M][N] real image: transformed by the forward kernel, added to by the adjoint kernel
    float* out;              // [S][C][M][N] v + Re(A^H c)
    const float2* y;         // [S][nmeas]
    float2* cstate;          // [S][C][ns_max] c_k (unscaled), updated in place
    float2* mprev;           // [S][C][ns_max] m_{k-1} = A v_{k-1}, updated in place
    float2* part;            // [S][C][G][ns_max] partial sample sums of the forward kernel
    float2* cbuf;            // [S][C][ns_max] input of the inverse transform (pre-scaled)
    int* minmax;             // optional [S][2] ordered-int min / max of out
    const int* frame_ptr;    // [C+1]
    const float2* tw2;       // [16][16]
    const float2* tw448;     // [448]
    const uint32_t* itA;     // [C][224] folded-row work items (K1Tables::r_itA)
    const uint32_t* itB;
    const uint32_t* ent;     // [nmeas] j | k2' << 16 | conj << 31
    const uint16_t* rowmask; // [C][16] symmetric row mask
    int n_ovf;
    int G;                   // slab groups (CTAs) per image of `part`: 1, 2, 4 or 8 (8 slabs of 28 real columns)
    int slabs_per_cta;       // set by the launchers
    int C, nmeas, ns_max;
    int rec;                 // stream_solver_kernel: 0 first x-update, 1 steady state, 2 last x-update
    float part_scale;        // what the summed partials are multiplied by to give m = A v
    float cbuf_scale;        // what c is multiplied by on its way into the inverse transform
    float inv_1p_rho;
};
int k1r_groups(int S, int C, int sm_count);
size_t k1r_part_elems(int S, int C, int G, int ns_max);
size_t k1r_state_elems(int S, int C, int ns_max);
bool k1r_fits(int ns_max, int n_ovf);
int k1r_forward(qmri_ctx* ctx, const K1RealParams& p, int S);
int k1r_solve(qmri_ctx* ctx, const K1RealParams& p, int S);
int k1r_adjoint(qmri_ctx* ctx, const K1RealParams& p, int S);
int k1r_last_base(qmri_ctx* ctx, const float* v, const float* base_re, const float* base_im, float* x_re, float* x_im, size_t n);

// general V: the per-location kernels that mix channels around the streaming transforms (xupdate_general.cu)
struct GeneralMix {
    const float2* part;      // [S][C][G][nU] partial sums of the forward transform on the union (stream_fwd_kernel)
    float2* cbuf;            // [S][C][nU]    input of the adjoint transform (stream_adj_kernel)
    const float2* y;         // [S][nmeas]
    float2* y_out;           // [S][nmeas]
    const float* V;          // [L][C]
    const float* Minv;       // [nU][C][C]  (G_u + rho I)^{-1}
    const int* memb_ptr;     // [nU + 1]
    const int* memb_frame;   // [nmeas]
    const int* memb_meas;    // [nmeas]
    const int* meas_u;       // [nmeas]
    const int* meas_frame;   // [nmeas]
    int S, C, L, G, nU, nmeas;
    float inv_n;             // 1 / N: unitary scaling 1/sqrt(N*M), once per transform direction
    double* mon_dc;          // monitored PnP-ADMM sessions: [S][k1_general_residual_parts(nU)] partial sums of |y - A x|^2
};
int k1_general_mix_forward(qmri_ctx* ctx, const GeneralMix& m);   // y_i(k) = sum_c V(i,c) Z^_c(k)
int k1_general_mix_adjoint(qmri_ctx* ctx, const GeneralMix& m);   // cbuf_c(k) = sum_{i: k in Omega_i} V(i,c) y_i(k)
int k1_general_mix_solve(qmri_ctx* ctx, const GeneralMix& m);     // cbuf(k) = (G_k + rho I)^{-1} sum_i V(i,:)^T (y_i(k) - V(i,:) Z^(k))
// after mix_solve: sum over the union locations of a block of sum_i |y_i(k) - V(i,:) X^(k)|^2, X^ = Z^ + delta -> m.mon_dc
int k1_general_mix_residual(qmri_ctx* ctx, const GeneralMix& m);
int k1_general_residual_parts(int nU);
