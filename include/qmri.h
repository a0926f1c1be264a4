/*
 * qmri.h - C ABI of libqmri_b200.so: the B200 (sm_100a) implementation of the
 * PnP-ADMM MRF reconstruction hot path of ketanfatania/QMRI-PnP-Recon-POC.
 *
 * This is the drop-in boundary.  The reference is MATLAB (+ PyTorch for the
 * denoiser definition); a MATLAB maintainer binds these entry points through one
 * MEX gateway (qmri-pnp-recon-poc_b200/mex/qmri_b200_mex.cpp, see INTEGRATION.md),
 * the test-suite and bench bind them through ctypes (qmri_b200/_capi.py).  Plain
 * pointers and sizes only - no torch / MATLAB types cross this boundary.
 *
 * Every entry point cites the reference interface it replaces (paths relative to
 * the reference checkout).
 *
 * Conventions
 *  - return 0 on success, a negative QMRI_E* code otherwise; never throws.
 *    qmri_last_error() returns the message of the last failure on this thread.
 *  - opaque handles own all device memory; host pointers are borrowed for the
 *    duration of the call and inputs are never written.
 *  - host arrays use the MATLAB layout: column-major, N x M x C (x S slices as a
 *    trailing dimension), complex numbers interleaved (re,im).  Split-complex
 *    MATLAB arrays (pre-R2018a MEX API, Octave) are interleaved by the gateway.
 *  - all device arithmetic is single precision (the reference computes the
 *    x-update in double and denoiser/matching in single); parity tolerances are
 *    stated in tests/.
 *  - one qmri_ctx per process and GPU; a ctx is not thread-safe (MATLAB is single
 *    threaded), distinct ctxs are independent.
 *  - entry points with the _dev suffix take DEVICE pointers in the library's
 *    planar fp32 layout and enqueue on the ctx stream without synchronising;
 *    they exist so that callers that already hold data in HBM (bench.py's
 *    kernel-only timing, the multi-GPU atom-sharded matcher) avoid the copies.
 */
#ifndef QMRI_B200_H
#define QMRI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QMRI_VERSION 100

/* ---- error codes ---------------------------------------------------------- */
enum {
    QMRI_OK = 0,
    QMRI_EINVAL = -1,       /* bad argument (null pointer, bad size, bad dtype)          */
    QMRI_EUNSUPPORTED = -2, /* valid in the reference but outside this build's scope     */
    QMRI_ECUDA = -3,        /* CUDA runtime / launch failure                             */
    QMRI_ENOMEM = -4,       /* host or device allocation failed                          */
    QMRI_ECALLBACK = -5     /* the denoiser callback returned non-zero                   */
};

/* ---- element types of host arrays ------------------------------------------ */
enum {
    QMRI_F32 = 0,  /* real single                */
    QMRI_F64 = 1,  /* real double                */
    QMRI_C64 = 2,  /* complex single, interleaved */
    QMRI_C128 = 3  /* complex double, interleaved */
};

enum { QMRI_HOST = 0, QMRI_DEVICE = 1 };

typedef struct qmri_ctx qmri_ctx;
typedef struct qmri_op qmri_op;
typedef struct qmri_net qmri_net;
typedef struct qmri_dict qmri_dict;
typedef struct qmri_admm qmri_admm;

/* ---- context ---------------------------------------------------------------- */
int qmri_version(void);
/* Binds to CUDA device `device_id` (must be compute capability 10.x). */
int qmri_ctx_create(qmri_ctx** out, int device_id);
int qmri_ctx_destroy(qmri_ctx* ctx);
/* Use an externally owned cudaStream_t for all work of this ctx (NULL = own stream). */
int qmri_ctx_set_stream(qmri_ctx* ctx, void* cuda_stream);
int qmri_ctx_synchronize(qmri_ctx* ctx);
/* Number of kernels this ctx has launched since creation (bench.py's gpu_launches). */
int64_t qmri_ctx_launch_count(qmri_ctx* ctx);
const char* qmri_last_error(void);

/* ---- acquisition operator ---------------------------------------------------
 * Replaces the struct of handles P.for / P.adj returned by
 *   setup_subsampling_spiralgrided(N,M,S,V)  main_files/subsampling_patterns/setup_subsampling_spiralgrided.m:1-43
 *   setup_subsampling_epi(N,M,percentage,V)  main_files/subsampling_patterns/setup_subsampling_epi.m:1-37
 * and the closures F.forward / F.adjoint of main_recon_tsmis_FFT.m:228-229.
 * V is L x C column-major, real (the reference passes real(dict.V)).
 * Scope of this build: N == M == 224 or N == M == 256 (other sizes: QMRI_EUNSUPPORTED).  At 256 the x-update runs on the
 * streaming kernels at every batch size (QMRI_K1_KERNEL=cluster is refused; QMRI_K1_STATE=real runs the complex loop).  V == eye(C) (the BASELINE configuration) takes the diagonal data-consistency
 * path; any other real L x C V (C <= 16) takes the exact per-location block solve on the union of the L masks
 * (SURVEY.md 8f-2; the union is processed in parts of <= 3400 k-space locations, e.g. 4 parts for 200 spiral frames).
 */
int qmri_op_spiral(qmri_ctx* ctx, int N, int M, int S_curve, const double* V, int L, int C, qmri_op** out);
int qmri_op_epi(qmri_ctx* ctx, int N, int M, double percentage, const double* V, int L, int C, qmri_op** out);
/* Operator from explicit masks: idx = 0-based column-major k indices, frame-major,
 * ascending inside a frame; frame_ptr has L+1 entries. */
int qmri_op_create(qmri_ctx* ctx, int N, int M, int C, int L, const int32_t* idx, const int64_t* frame_ptr,
                   const double* V, qmri_op** out);
int qmri_op_destroy(qmri_op* op);
/* Number of measurements per slice (rows of P). */
int64_t qmri_op_nmeas(const qmri_op* op);
/* Copies the sampled locations out (idx: nmeas int32, frame_ptr: L+1 int64) - lets
 * callers pin the mask constructors against the reference's `find` output. */
int qmri_op_indices(const qmri_op* op, int32_t* idx, int64_t* frame_ptr);

/* The bare sampling matrix the constructors return as handles (setup_subsampling_spiralgrided.m:36-42,
 * setup_subsampling_epi.m:31-35): P = vertical stack of S_i * kron(conj(V(i,:)), I).
 *   y = P.for(vec):  vec = N*M*C k-space column (reshape(fft2(x),[],1)), y = nmeas complex
 *   vec = P.adj(y):  P' * y
 * Both run on the device in double precision (a gather / scatter; exact for V = eye(C)). */
int qmri_op_for(qmri_op* op, const void* kvec, int k_dtype, void* y, int y_dtype);
int qmri_op_adj(qmri_op* op, const void* y, int y_dtype, void* kvec, int k_dtype);

/* Y = awgn(Y, snr, 'measured')   main_recon_tsmis_FFT.m:243
 * In place on an nmeas x S interleaved complex array: complex white Gaussian noise of power
 * mean(|Y(:,s)|^2) / 10^(snr_db/10) per slice, Philox-4x32-10 counter (sample, slice) keyed by `seed`, Box-Muller in double:
 * the same seed gives the same noise whatever the batch size.  (MATLAB's generator is not reproduced: statistical equality only.) */
int qmri_awgn(qmri_ctx* ctx, void* y, int y_dtype, int64_t nmeas, int S, double snr_db, uint64_t seed);
/* Device-resident variant: y_dev = float2 [S][nmeas]; power_dev = S doubles of scratch (receives mean |y|^2 per slice). */
int qmri_awgn_dev(qmri_ctx* ctx, float* y_dev, int64_t nmeas, int S, double snr_db, uint64_t seed, double* power_dev);

/* y = F.forward(x)   main_recon_tsmis_FFT.m:228   x: N x M x C x S (real or complex), y: nmeas x S complex */
int qmri_forward(qmri_op* op, const void* x, int x_dtype, int S, void* y, int y_dtype);
/* x = F.adjoint(y)   main_recon_tsmis_FFT.m:229   y: nmeas x S complex, x: N x M x C x S complex */
int qmri_adjoint(qmri_op* op, const void* y, int y_dtype, int S, void* x, int x_dtype);

/* One least-squares step, PnP_ADMM.m:102 (lsqr over afun, :153-171), solved exactly:
 *   x = argmin ||y - A x||^2 + rho ||x - (v - u)||^2
 * plus what the loop derives from it: w = x + u (:115) and per-slice min / max of
 * real(w) (:121,:177-178).  u may be NULL (the scalar 0 of :78).  w and minmax
 * (2 floats per slice: min, max) may be NULL.  v: real or complex; u, x, w complex. */
int qmri_xupdate(qmri_op* op, double rho, const void* y, int y_dtype, const void* v, int v_dtype,
                 const void* u, int u_dtype, int S, void* x, int x_dtype, void* w, int w_dtype, float* minmax);

/* ---- denoiser -----------------------------------------------------------------
 * Replaces param.net = @(x) denoiseImage_PnP_ADMM(x, Net, true, false)
 * (main_recon_tsmis_FFT.m:164, main_files/utils/denoiseImage_PnP_ADMM.m:73-114) evaluating
 * UNetRes(in_nc, 10, nc=[64,128,256,512], nb=4, 'R', 'strideconv', 'convtranspose'), bias-free
 * (PyTorch_Denoiser/zhang_dpir_testing_code/network_unet.py:68-117, main_train.py:247).
 * weights: the 64 tensors of state_dict() in its key order, PyTorch layouts
 * (Conv2d [Cout,Cin,kh,kw], ConvTranspose2d [Cin,Cout,kh,kw]), float32, host. */
int qmri_unetres_load(qmri_ctx* ctx, int in_nc, const float* const* weights, int n_weights, qmri_net** out);
int qmri_unetres_destroy(qmri_net* net);
/* precision: 0 = fp32 CUDA-core path (exact mode), 1 = tcgen05 split-bf16 tensor path. */
int qmri_unetres_set_precision(qmri_net* net, int mode);
/* Plain forward, PyTorch layout: in S x in_nc x H x W, out S x 10 x H x W (host float32). H, W multiples of 8. */
int qmri_unetres_forward(qmri_net* net, const float* in, float* out, int S, int H, int W);
/* MATLAB layout (what param.net receives): in H x W x in_nc (x S), out H x W x 10 (x S), column-major. */
int qmri_unetres_denoise(qmri_net* net, const void* in, int in_dtype, void* out, int out_dtype, int S, int H, int W);
/* Device-resident: planar [S][in_nc][W][H] fp32 in, [S][10][W][H] out; optional per-slice affine
 * (minmax: 2 floats per slice on device; NULL = identity) folded into the head load / tail store. */
int qmri_unetres_forward_dev(qmri_net* net, const float* in_dev, float* out_dev, const float* minmax_dev,
                             const float* noise_map_dev, int S, int H, int W);
/* FLOPs (2*MAC) of one forward at S x H x W. */
double qmri_unetres_flops(const qmri_net* net, int S, int H, int W);

/* A pluggable proximal step: v_out = f(v_in), v_in S slices of H x W x Cin in [0,1] (MATLAB
 * layout, float32), v_out S slices of H x W x Cout.  `space` tells where the pointers live. */
typedef int (*qmri_denoise_fn)(void* user, const float* v_in, float* v_out, int H, int W, int Cin, int Cout,
                               int S, int space, void* cuda_stream);

/* ---- the ADMM loop -------------------------------------------------------------
 * Replaces x = PnP_ADMM(y, param)   main_files/algorithms/PnP_ADMM/PnP_ADMM.m:1-148
 * with the param struct of main_recon_tsmis_FFT.m:164-170,285-292. */
typedef struct qmri_admm_params {
    int iters;              /* param.iter                                            */
    double gamma;           /* param.gamma (rho)                                     */
    double cg_tol;          /* param.cg_tol - accepted, unused: the solve is exact   */
    int multi_level;        /* param.denoiser_type == 'multi_level'                  */
    const float* noise_map; /* param.noise_map, N x M column-major host float32       */
    qmri_net* net;          /* built-in denoiser, or NULL to use fn                   */
    qmri_denoise_fn fn;     /* param.net as a callback (used when net == NULL)        */
    void* user;
    int fn_space;           /* QMRI_HOST or QMRI_DEVICE pointers for fn               */
} qmri_admm_params;

/* Whole call: H2D of y and X0, `iters` iterations on the device, D2H of x. */
int qmri_pnp_admm(qmri_op* op, const void* y, int y_dtype, const void* x0, int x0_dtype, int S,
                  const qmri_admm_params* params, void* x_out, int x_dtype);
/* The same, split so that the loop can be timed with inputs resident in HBM. */
int qmri_admm_create(qmri_op* op, int S, const qmri_admm_params* params, qmri_admm** out);
int qmri_admm_upload(qmri_admm* st, const void* y, int y_dtype, const void* x0, int x0_dtype);
int qmri_admm_run(qmri_admm* st, int iters);   /* restarts from X0 every call */
int qmri_admm_download(qmri_admm* st, void* x_out, int x_dtype);
/* Device views of the state after a run: planar fp32 [S][C][M][N]. */
int qmri_admm_state_dev(qmri_admm* st, const float** x_re, const float** x_im);
int qmri_admm_destroy(qmri_admm* st);
/* Kernel-only x-update step on a resident state (w, v) -> w' ; used by bench.py for the K1 roofline.  With a monitor attached
 * (qmri_admm_monitor) a complex-state session runs the monitored kernel instances, which write their partial sums but no history
 * row; a real-state session (QMRI_K1_STATE=real) runs its real-state kernels, which are never monitored. */
int qmri_admm_xupdate_only(qmri_admm* st, int reps);
/* Algorithmic HBM bytes per pixel-channel of one x-update in the state formulation this session runs: 8 for the real-state
 * loop (read v, write Re w'; two slices or more, V = eye: csrc/xupdate_real.cu), 20 for the complex-state kernels (read w and v,
 * write w').  bench.py reports the x-update roofline against this figure, never against bytes that do not move. */
int qmri_admm_xupdate_bytes(qmri_admm* st);
/* Convergence history, PnP_ADMM.m:106-109: after the x-update of iteration k = 1..iters, per slice s,
 *   dc_res(k, s) = |y_s - F.forward(x_k,s)| / |y_s|        gt_err(k, s) = |gt_s - x_k,s| / |gt_s|
 * over all N*M*C entries of the slice (x_k before the denoiser; k = 1 is the solve from X0; a zero denominator gives NaN).
 * Recorded on the device inside the loop (and its CUDA graph), downloaded once by qmri_admm_history.  Call qmri_admm_monitor
 * after qmri_admm_create; it holds for every later run until it is called again.  gt: N x M x C x S host array (param.gt_tsmi),
 * real or complex, any of the four dtypes, or NULL for the residual only; enable = 0 switches monitoring off (the unmonitored
 * kernels run, unchanged).  A monitored session runs the complex-state streaming x-update at every batch size (general V included):
 * QMRI_EUNSUPPORTED with QMRI_K1_KERNEL=cluster; QMRI_K1_STATE=real sessions run the complex-state loop while monitored. */
int qmri_admm_monitor(qmri_admm* st, int enable, const void* gt, int gt_dtype);
/* History of the last run, MATLAB column-major iters x S doubles.  *iters receives the rows (0 when the last run was not
 * monitored or ran no iteration); dc_res / gt_err may be NULL (query the size first).  QMRI_EINVAL if gt_err is asked for and the
 * last run had no ground truth. */
int qmri_admm_history(qmri_admm* st, double* dc_res, double* gt_err, int* iters);

/* ---- dictionary matching ---------------------------------------------------------
 * Replaces out = mrf_dtm_cpu(dict, data, par)   main_files/dictionary_matching/mrf_dtm_cpu.m:1-166
 * dict.D [K x C] column-major float32 (unit-norm atoms), dict.normD [K], dict.lut [K x Q]
 * column-major (mrf_dtm_cpu.m:8-12).  Atoms [shard_begin, shard_end) are scored by this
 * handle (the whole dictionary when 0,K); D/normD/lut are kept whole for the gathers. */
int qmri_dict_load(qmri_ctx* ctx, const float* D, const float* normD, const float* lut, int64_t K, int C, int Q,
                   int64_t shard_begin, int64_t shard_end, qmri_dict** out);
/* Atom-sharded residency (BASELINE config 5: a dictionary too large for one GPU): D_shard holds ONLY the rows
 * [shard_begin, shard_end) ((shard_end - shard_begin) x C column-major); normD / lut stay whole (12 B per atom).
 * qmri_match_finish_dev on such a handle writes the pixels whose winning atom it owns and zeros elsewhere, so the
 * per-rank outputs combine with a sum all-reduce (every pixel has exactly one owner). */
int qmri_dict_load_shard(qmri_ctx* ctx, const float* D_shard, const float* normD, const float* lut, int64_t K, int C, int Q,
                         int64_t shard_begin, int64_t shard_end, qmri_dict** out);
int qmri_dict_destroy(qmri_dict* d);
/* x: npix x C column-major, real or complex.  Outputs (any may be NULL, cf. par.f.*):
 * qmap npix x Q float (NaN -> 0, :139), pd npix complex float interleaved (:96), mt npix float
 * (max |<d,x>|, :92), dm npix int32 1-based (:92). */
int qmri_match(qmri_dict* d, const void* x, int x_dtype, int64_t npix, float* qmap, float* pd, float* mt, int32_t* dm);
/* Device-resident planar input x_re/x_im [C][npix] (x_im may be NULL for real data). */
int qmri_match_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, float* qmap_dev, float* pd_dev,
                   float* mt_dev, int32_t* dm_dev);
/* Atom-sharded matching (BASELINE config 5): local packed keys
 *   key = float_bits(|<d, x s>|^2) << 32 | (0xFFFFFFFF - global_atom_index)
 * (max over ranks of the key = max score, lowest index on ties = MATLAB's first-index rule; s = a power of two that depends on
 * the pixel's data alone and keeps the squared score inside the fp32 range - the same on every rank, atom range and kernel),
 * reduced by the caller (NCCL max over uint64 / int64), then finished from the reduced keys. */
int qmri_match_keys_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, uint64_t* keys_dev);
int qmri_match_finish_dev(qmri_dict* d, const float* x_re, const float* x_im, int64_t npix, const uint64_t* keys_dev,
                          float* qmap_dev, float* pd_dev, float* mt_dev, int32_t* dm_dev);

/* ---- TSMI synthesis (SURVEY.md 8f-1) ------------------------------------------------
 * main_synthesize_tsmis.m:84-98: I = knnsearch(KDTreeSearcher(dict.lut), qm(:,1:2)) as an exhaustive fused
 * nearest-(T1,T2) scan on the GPU, X = D(I,:) .* normD(I) .* |PD|, sign-aligned to channel 1.
 * qmap: npix x 3 column-major (T1,T2,PD) host float32 -> X npix x C column-major float32;
 * atom_index (optional): 1-based I.  Exact distance ties resolve to the lowest atom index. */
int qmri_synthesize(qmri_dict* d, const float* qmap, int64_t npix, float* X, int32_t* atom_index);

/* ---- foreground mask and quality metrics (SURVEY.md 8f-4) ------------------------------
 * mask = getmask_fromPD(PD, thresh)   main_files/utils/getmask_fromPD.m:1-15 (called at main_recon_tsmis_FFT.m:190):
 * |PD| / max, values below thresh zeroed, holes filled (8-connected background), binarised.  pd: N x M column-major,
 * real or complex; mask: N x M float 0/1. */
int qmri_foreground_mask(qmri_ctx* ctx, const void* pd, int pd_dtype, int N, int M, double thresh, float* mask);
/* The metrics block of main_recon_tsmis_FFT.m:328-384, computed on the device in double:
 *   qmap  N x M x 3 = cat(3, out.qmap, out.pd) (T1, T2, PD; real or complex), qmap0 the ground truth, mask from
 *   qmri_foreground_mask (NULL = all ones); X, X0: N x M x C reconstructed / ground-truth TSMIs (both NULL to skip).
 *   out[11] = tsmi_mean_psnr, tsmi_mean_ssim, t1_mae, t1_psnr, t1_ssim, t2_mae, t2_psnr, t2_ssim, pd_mae, pd_psnr, pd_ssim
 * with MATLAB's psnr (peak 1 for double images) and ssim defaults (11 x 11 Gaussian window, sigma 1.5, replicate
 * padding, dynamic range 1). */
int qmri_recon_metrics(qmri_ctx* ctx, int N, int M, int C, const void* qmap, int qmap_dtype, const void* qmap0, int qmap0_dtype,
                       const float* mask, const void* X, int x_dtype, const void* X0, int x0_dtype, double* out);

/* ---- LRTV comparison baseline (SURVEY.md 8f-4) ------------------------------------------
 * x = FISTA_deep(data, param)   main_files/algorithms/LRTV/FISTA_deep.m:1-115 with the TV prox of
 * unlocbox/prox/prox_tv.m (called at main_recon_tsmis_FFT.m:272-282: K = 4e-5, iter = 200, step = numel(X0)/numel(Y),
 * tol = 1e-4, backtrack = 1).  One slice; y nmeas complex -> x N x M x C complex.  The TV prox keeps the toolbox defaults
 * (tv_tol = 10e-4, tv_maxit = 200) unless set.  Double-precision state on the device, the operator in single. */
typedef struct qmri_lrtv_params {
    double K;        /* param.K: TV weight                               */
    int iters;       /* param.iter                                       */
    double step;     /* param.step: initial FISTA step                   */
    double tol;      /* param.tol: relative objective change that stops  */
    int backtrack;   /* param.backtrack                                  */
    double tv_tol;   /* 0 = toolbox default 10e-4                        */
    int tv_maxit;    /* 0 = toolbox default 200                          */
} qmri_lrtv_params;
int qmri_lrtv(qmri_op* op, const void* y, int y_dtype, const qmri_lrtv_params* params, void* x_out, int x_dtype, int* iters_done,
              double* final_step);

#ifdef __cplusplus
}
#endif
#endif /* QMRI_B200_H */
