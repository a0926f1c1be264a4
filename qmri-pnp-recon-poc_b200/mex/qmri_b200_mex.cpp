// qmri_b200_mex.cpp - single MEX gateway between MATLAB and libqmri_b200.so (include/qmri.h).
//
//   out = qmri_b200_mex(command, args...)
//
// Build on a MATLAB host:
//   mex -R2018a qmri_b200_mex.cpp -I../../include -L../lib -lqmri_b200        (interleaved complex: zero-copy)
//   mex         qmri_b200_mex.cpp -I../../include -L../lib -lqmri_b200        (legacy split complex / GNU Octave's mkoctfile --mex)
// The C ABI takes interleaved complex only.  With the split-complex API (MX_HAS_INTERLEAVED_COMPLEX == 0) the gateway
// interleaves complex inputs into a temporary before the call and splits complex outputs after it (CplxIn / CplxOut below).
// In this repository's build container there is no MATLAB: the file is compiled against mex/mock_mex.h - a functional
// mock - in both complex models and EXECUTED by tests/test_mex_gateway.py against the ctypes path.
//
// Handles (ctx / op / net / dict) are returned to MATLAB as uint64 scalars and kept alive across calls (mexLock); everything
// is released by `qmri_b200_mex('shutdown')` or at mexAtExit.  prhs arrays are never written.  Errors from the library become
// MATLAB exceptions `qmri:<code>`.
#ifdef QMRI_MOCK_MEX
#include "mock_mex.h"
#else
#include <mex.h>
#endif
#ifndef MX_HAS_INTERLEAVED_COMPLEX
#define MX_HAS_INTERLEAVED_COMPLEX 0
#endif
#include <stdint.h>
#include <string.h>

#include <string>
#include <vector>

#include "qmri.h"

namespace {

std::vector<qmri_op*> g_ops;
std::vector<qmri_net*> g_nets;
std::vector<qmri_dict*> g_dicts;
qmri_ctx* g_ctx = nullptr;
qmri_op* g_last_op = nullptr;
bool g_locked = false;

void shutdown() {
    for (auto* o : g_ops) qmri_op_destroy(o);
    for (auto* n : g_nets) qmri_unetres_destroy(n);
    for (auto* d : g_dicts) qmri_dict_destroy(d);
    g_ops.clear(); g_nets.clear(); g_dicts.clear();
    g_last_op = nullptr;
    if (g_ctx) qmri_ctx_destroy(g_ctx);
    g_ctx = nullptr;
}

void check(int rc) {
    if (rc != QMRI_OK) mexErrMsgIdAndTxt("qmri:error", "libqmri_b200 error %d: %s", rc, qmri_last_error());
}

qmri_ctx* ctx() {
    if (!g_ctx) {
        check(qmri_ctx_create(&g_ctx, 0));
        if (!g_locked) { mexLock(); mexAtExit(shutdown); g_locked = true; }
    }
    return g_ctx;
}

int dtype_of(const mxArray* a) {
    const bool c = mxIsComplex(a) != 0;
    if (mxIsDouble(a)) return c ? QMRI_C128 : QMRI_F64;
    if (mxIsSingle(a)) return c ? QMRI_C64 : QMRI_F32;
    mexErrMsgIdAndTxt("qmri:type", "arrays must be single or double");
    return -1;
}

// An input array as the ABI wants it: for real arrays and for the interleaved-complex API this is the MATLAB buffer itself;
// with the split-complex API a complex array is interleaved into `tmp` first.
struct CplxIn {
    const void* p = nullptr;
    int dtype = 0;
    std::vector<unsigned char> tmp;
    explicit CplxIn(const mxArray* a) {
        dtype = dtype_of(a);
        p = mxGetData(a);
#if !MX_HAS_INTERLEAVED_COMPLEX
        if (mxIsComplex(a)) {
            const size_t n = mxGetNumberOfElements(a), es = mxIsDouble(a) ? 8 : 4;
            tmp.resize(2 * n * es);
            const unsigned char* re = (const unsigned char*)mxGetData(a);
            const unsigned char* im = (const unsigned char*)mxGetImagData(a);
            for (size_t i = 0; i < n; ++i) {
                memcpy(&tmp[(2 * i) * es], re + i * es, es);
                memcpy(&tmp[(2 * i + 1) * es], im + i * es, es);
            }
            p = tmp.data();
        }
#endif
    }
};
// A complex output array: the ABI writes interleaved values either straight into the MATLAB buffer (interleaved API) or into
// `tmp`, which finish() splits into the real / imaginary planes.
struct CplxOut {
    mxArray* a = nullptr;
    void* p = nullptr;
    std::vector<unsigned char> tmp;
    CplxOut(mwSize ndim, const mwSize* dims, mxClassID cls) {
        a = mxCreateNumericArray(ndim, dims, cls, mxCOMPLEX);
        p = mxGetData(a);
#if !MX_HAS_INTERLEAVED_COMPLEX
        tmp.resize(2 * mxGetNumberOfElements(a) * (cls == mxDOUBLE_CLASS ? 8 : 4));
        p = tmp.data();
#endif
    }
    mxArray* finish() {
#if !MX_HAS_INTERLEAVED_COMPLEX
        const size_t n = mxGetNumberOfElements(a), es = mxIsDouble(a) ? 8 : 4;
        unsigned char* re = (unsigned char*)mxGetData(a);
        unsigned char* im = (unsigned char*)mxGetImagData(a);
        for (size_t i = 0; i < n; ++i) {
            memcpy(re + i * es, &tmp[(2 * i) * es], es);
            memcpy(im + i * es, &tmp[(2 * i + 1) * es], es);
        }
#endif
        return a;
    }
};

mxArray* handle_out(void* p) {
    mxArray* a = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
    *(uint64_t*)mxGetData(a) = (uint64_t)(uintptr_t)p;
    return a;
}
template <typename T>
T* handle_in(const mxArray* a) { return (T*)(uintptr_t)(*(const uint64_t*)mxGetData(a)); }

int slices_of(const mxArray* a, int base_dims) {
    return mxGetNumberOfDimensions(a) > (mwSize)base_dims ? (int)mxGetDimensions(a)[base_dims] : 1;
}
int dim_of(const mxArray* a, int i) { return mxGetNumberOfDimensions(a) > (mwSize)i ? (int)mxGetDimensions(a)[i] : 1; }

// param.net as a MATLAB function handle: D2H hop per iteration (slow path, same results)
struct FevalCtx { const mxArray* fn; };
int feval_denoiser(void* user, const float* v_in, float* v_out, int H, int W, int Cin, int Cout, int S, int space, void*) {
    if (space != QMRI_HOST) return 2;
    FevalCtx* fc = (FevalCtx*)user;
    for (int s = 0; s < S; ++s) {
        mwSize dims[3] = {(mwSize)H, (mwSize)W, (mwSize)Cin};
        mxArray* in = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);  // PnP_ADMM hands the net a double array
        double* d = (double*)mxGetData(in);
        const float* src = v_in + (size_t)s * H * W * Cin;
        for (size_t i = 0; i < (size_t)H * W * Cin; ++i) d[i] = src[i];
        mxArray* rhs[2] = {const_cast<mxArray*>(fc->fn), in};
        mxArray* lhs[1] = {nullptr};
        if (mexCallMATLAB(1, lhs, 2, rhs, "feval") != 0 || !lhs[0]) { mxDestroyArray(in); return 1; }
        if (mxGetNumberOfElements(lhs[0]) != (size_t)H * W * Cout || mxIsComplex(lhs[0])) { mxDestroyArray(in); mxDestroyArray(lhs[0]); return 3; }
        float* dst = v_out + (size_t)s * H * W * Cout;
        if (mxIsDouble(lhs[0])) { const double* o = (const double*)mxGetData(lhs[0]); for (size_t i = 0; i < (size_t)H * W * Cout; ++i) dst[i] = (float)o[i]; }
        else if (mxIsSingle(lhs[0])) { const float* o = (const float*)mxGetData(lhs[0]); for (size_t i = 0; i < (size_t)H * W * Cout; ++i) dst[i] = o[i]; }
        else { mxDestroyArray(in); mxDestroyArray(lhs[0]); return 4; }
        mxDestroyArray(in);
        mxDestroyArray(lhs[0]);
    }
    return 0;
}

}  // namespace

extern "C" void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    if (nrhs < 1) mexErrMsgIdAndTxt("qmri:usage", "qmri_b200_mex(command, ...)");
    char* c = mxArrayToString(prhs[0]);
    std::string cmd = c ? c : "";
    mxFree(c);
    auto need = [&](int n) { if (nrhs < n) mexErrMsgIdAndTxt("qmri:usage", "%s: expected %d arguments, got %d", cmd.c_str(), n - 1, nrhs - 1); };

    if (cmd == "op_spiral" || cmd == "op_epi") {            // (N, M, S|percentage, V) -> op handle
        need(5);
        const int N = (int)mxGetScalar(prhs[1]), M = (int)mxGetScalar(prhs[2]);
        const mxArray* V = prhs[4];
        const int L = dim_of(V, 0), C = dim_of(V, 1);
        if (!mxIsDouble(V) || mxIsComplex(V)) mexErrMsgIdAndTxt("qmri:type", "V must be real double (real(dict.V))");
        qmri_op* op = nullptr;
        if (cmd == "op_spiral") check(qmri_op_spiral(ctx(), N, M, (int)mxGetScalar(prhs[3]), (const double*)mxGetData(V), L, C, &op));
        else check(qmri_op_epi(ctx(), N, M, mxGetScalar(prhs[3]), (const double*)mxGetData(V), L, C, &op));
        g_ops.push_back(op);
        g_last_op = op;
        plhs[0] = handle_out(op);
    } else if (cmd == "last_op") {                           // () -> the operator built most recently (0 if none)
        plhs[0] = handle_out(g_last_op);
    } else if (cmd == "nmeas") {                             // (op) -> rows of P
        need(2);
        plhs[0] = mxCreateDoubleScalar((double)qmri_op_nmeas(handle_in<qmri_op>(prhs[1])));
    } else if (cmd == "forward") {                           // (op, x[N M C (S)]) -> y[nmeas (S)]
        need(3);
        qmri_op* op = handle_in<qmri_op>(prhs[1]);
        const int S = slices_of(prhs[2], 3);
        mwSize dims[2] = {(mwSize)qmri_op_nmeas(op), (mwSize)S};
        CplxIn x(prhs[2]);
        CplxOut y(2, dims, mxDOUBLE_CLASS);
        check(qmri_forward(op, x.p, x.dtype, S, y.p, QMRI_C128));
        plhs[0] = y.finish();
    } else if (cmd == "adjoint") {                           // (op, y, [N M C]) -> x
        need(4);
        qmri_op* op = handle_in<qmri_op>(prhs[1]);
        const int S = slices_of(prhs[2], 1);
        const double* sz = (const double*)mxGetData(prhs[3]);
        mwSize dims[4] = {(mwSize)sz[0], (mwSize)sz[1], (mwSize)sz[2], (mwSize)S};
        CplxIn y(prhs[2]);
        CplxOut x(4, dims, mxDOUBLE_CLASS);
        check(qmri_adjoint(op, y.p, y.dtype, S, x.p, QMRI_C128));
        plhs[0] = x.finish();
    } else if (cmd == "p_for") {                             // (op, vec[N*M*C]) -> P*vec    K.for of setup_subsampling_*.m
        need(3);
        qmri_op* op = handle_in<qmri_op>(prhs[1]);
        mwSize dims[2] = {(mwSize)qmri_op_nmeas(op), 1};
        CplxIn v(prhs[2]);
        CplxOut y(2, dims, mxDOUBLE_CLASS);
        check(qmri_op_for(op, v.p, v.dtype, y.p, QMRI_C128));
        plhs[0] = y.finish();
    } else if (cmd == "p_adj") {                             // (op, y[nmeas], numel) -> P'*y    K.adj
        need(4);
        qmri_op* op = handle_in<qmri_op>(prhs[1]);
        mwSize dims[2] = {(mwSize)mxGetScalar(prhs[3]), 1};
        CplxIn y(prhs[2]);
        CplxOut v(2, dims, mxDOUBLE_CLASS);
        check(qmri_op_adj(op, y.p, y.dtype, v.p, QMRI_C128));
        plhs[0] = v.finish();
    } else if (cmd == "awgn") {                              // (Y, snr, seed) -> Y + noise      awgn(Y, snr, 'measured')
        need(4);
        if (!mxIsComplex(prhs[1])) mexErrMsgIdAndTxt("qmri:type", "awgn: Y must be complex");
        const mwSize* d = mxGetDimensions(prhs[1]);
        const mwSize nd = mxGetNumberOfDimensions(prhs[1]);
        CplxIn yin(prhs[1]);
        CplxOut y(nd, d, mxIsDouble(prhs[1]) ? mxDOUBLE_CLASS : mxSINGLE_CLASS);
        const size_t es = mxIsDouble(prhs[1]) ? 16 : 8;
        memcpy(y.p, yin.p, mxGetNumberOfElements(prhs[1]) * es);
        const int64_t nmeas = (int64_t)d[0];
        const int S = (int)(mxGetNumberOfElements(prhs[1]) / (nmeas ? nmeas : 1));
        check(qmri_awgn(ctx(), y.p, yin.dtype, nmeas, S, mxGetScalar(prhs[2]), (uint64_t)mxGetScalar(prhs[3])));
        plhs[0] = y.finish();
    } else if (cmd == "mask") {                              // (PD[N M], thresh) -> mask   getmask_fromPD
        need(3);
        const int N = dim_of(prhs[1], 0), M = dim_of(prhs[1], 1);
        CplxIn pd(prhs[1]);
        std::vector<float> m((size_t)N * M);
        check(qmri_foreground_mask(ctx(), pd.p, pd.dtype, N, M, mxGetScalar(prhs[2]), m.data()));
        plhs[0] = mxCreateNumericMatrix((mwSize)N, (mwSize)M, mxDOUBLE_CLASS, mxREAL);
        double* o = (double*)mxGetData(plhs[0]);
        for (size_t i = 0; i < m.size(); ++i) o[i] = m[i];
    } else if (cmd == "metrics") {                           // (qmap[N M 3], qmap0[N M 3], mask[N M] double, X, X0) -> 11 x 1
        need(6);
        const int N = dim_of(prhs[1], 0), M = dim_of(prhs[1], 1), C = dim_of(prhs[4], 2);
        CplxIn q(prhs[1]), q0(prhs[2]), X(prhs[4]), X0(prhs[5]);
        std::vector<float> m(mxGetNumberOfElements(prhs[3]));
        const double* ms = (const double*)mxGetData(prhs[3]);
        for (size_t i = 0; i < m.size(); ++i) m[i] = (float)ms[i];
        plhs[0] = mxCreateNumericMatrix(11, 1, mxDOUBLE_CLASS, mxREAL);
        check(qmri_recon_metrics(ctx(), N, M, C, q.p, q.dtype, q0.p, q0.dtype, m.empty() ? nullptr : m.data(), X.p, X.dtype, X0.p, X0.dtype,
                                 (double*)mxGetData(plhs[0])));
    } else if (cmd == "net_load") {                          // (in_nc, cell{64} of single weight tensors) -> net handle
        need(3);
        std::vector<const float*> w(64);
        for (int i = 0; i < 64; ++i) {
            const mxArray* t = mxGetCell(prhs[2], i);
            if (!t || !mxIsSingle(t) || mxIsComplex(t)) mexErrMsgIdAndTxt("qmri:type", "weights must be a cell of 64 real single arrays (PyTorch memory order)");
            w[i] = (const float*)mxGetData(t);
        }
        qmri_net* net = nullptr;
        check(qmri_unetres_load(ctx(), (int)mxGetScalar(prhs[1]), w.data(), 64, &net));
        g_nets.push_back(net);
        plhs[0] = handle_out(net);
    } else if (cmd == "net_precision") {                     // (net, 0 | 1)
        need(3);
        check(qmri_unetres_set_precision(handle_in<qmri_net>(prhs[1]), (int)mxGetScalar(prhs[2])));
    } else if (cmd == "denoise") {                           // (net, A[H W Cin (S)]) -> [H W 10 (S)], class of A
        need(3);
        qmri_net* net = handle_in<qmri_net>(prhs[1]);
        if (mxIsComplex(prhs[2])) mexErrMsgIdAndTxt("qmri:type", "denoiser input must be real");
        const mwSize* d = mxGetDimensions(prhs[2]);
        const int S = slices_of(prhs[2], 3);
        mwSize od[4] = {d[0], d[1], 10, (mwSize)S};
        plhs[0] = mxCreateNumericArray(4, od, mxIsDouble(prhs[2]) ? mxDOUBLE_CLASS : mxSINGLE_CLASS, mxREAL);
        check(qmri_unetres_denoise(net, mxGetData(prhs[2]), dtype_of(prhs[2]), mxGetData(plhs[0]), dtype_of(plhs[0]), S, (int)d[0], (int)d[1]));
    } else if (cmd == "pnp_admm") {                          // (op, y, param struct) -> x [, info] ; param.net = net handle or function handle
        need(4);
        qmri_op* op = handle_in<qmri_op>(prhs[1]);
        const mxArray* prm = prhs[3];
        const mxArray* X0 = mxGetField(prm, 0, "X0");
        const mxArray* net = mxGetField(prm, 0, "net");
        const mxArray* it = mxGetField(prm, 0, "iter");
        const mxArray* gm = mxGetField(prm, 0, "gamma");
        if (!X0 || !net || !it || !gm) mexErrMsgIdAndTxt("qmri:param", "param.X0, param.net, param.iter and param.gamma are required");
        qmri_admm_params p;
        memset(&p, 0, sizeof(p));
        p.iters = (int)mxGetScalar(it);
        p.gamma = mxGetScalar(gm);
        const mxArray* tol = mxGetField(prm, 0, "cg_tol");
        p.cg_tol = tol ? mxGetScalar(tol) : 1e-4;
        const mxArray* dt = mxGetField(prm, 0, "denoiser_type");
        char* dts = dt ? mxArrayToString(dt) : nullptr;
        p.multi_level = dts && strcmp(dts, "multi_level") == 0;
        mxFree(dts);
        std::vector<float> nm;
        if (p.multi_level) {
            const mxArray* m = mxGetField(prm, 0, "noise_map");
            if (!m) mexErrMsgIdAndTxt("qmri:param", "param.noise_map is required for multi_level");
            nm.resize(mxGetNumberOfElements(m));
            if (mxIsDouble(m)) { const double* s = (const double*)mxGetData(m); for (size_t i = 0; i < nm.size(); ++i) nm[i] = (float)s[i]; }
            else memcpy(nm.data(), mxGetData(m), nm.size() * 4);
            p.noise_map = nm.data();
        }
        FevalCtx fc = {net};
        if (mxIsClass(net, "function_handle")) { p.fn = feval_denoiser; p.user = &fc; p.fn_space = QMRI_HOST; }
        else p.net = handle_in<qmri_net>(net);
        const int S = slices_of(X0, 3);
        const mwSize* d = mxGetDimensions(X0);
        mwSize od[4] = {d[0], d[1], (mwSize)dim_of(X0, 2), (mwSize)S};
        CplxIn y(prhs[2]), x0(X0);
        CplxOut x(4, od, mxDOUBLE_CLASS);
        if (nlhs < 2) {
            check(qmri_pnp_admm(op, y.p, y.dtype, x0.p, x0.dtype, S, &p, x.p, QMRI_C128));
            plhs[0] = x.finish();
        } else {  // [x, info]: the session API with the convergence history of PnP_ADMM.m:106-109 (info.dc_res, info.gt_err: iter x S)
            const mxArray* gt = mxGetField(prm, 0, "gt_tsmi");
            if (gt && mxGetNumberOfElements(gt) == 0) gt = nullptr;
            if (gt && mxGetNumberOfElements(gt) != mxGetNumberOfElements(X0))
                mexErrMsgIdAndTxt("qmri:param", "param.gt_tsmi must have the size of param.X0");
            std::vector<CplxIn> g;
            if (gt) g.emplace_back(gt);
            qmri_admm* st = nullptr;
            check(qmri_admm_create(op, S, &p, &st));
            int K = 0;
            int r = qmri_admm_monitor(st, 1, gt ? g[0].p : nullptr, gt ? g[0].dtype : QMRI_F64);
            if (!r) r = qmri_admm_upload(st, y.p, y.dtype, x0.p, x0.dtype);
            if (!r) r = qmri_admm_run(st, p.iters);
            if (!r) r = qmri_admm_download(st, x.p, QMRI_C128);
            if (!r) r = qmri_admm_history(st, nullptr, nullptr, &K);
            mxArray* dc = mxCreateNumericMatrix((mwSize)K, (mwSize)S, mxDOUBLE_CLASS, mxREAL);
            mxArray* ge = gt ? mxCreateNumericMatrix((mwSize)K, (mwSize)S, mxDOUBLE_CLASS, mxREAL) : mxCreateNumericMatrix(0, 0, mxDOUBLE_CLASS, mxREAL);
            if (!r && K) r = qmri_admm_history(st, (double*)mxGetData(dc), gt ? (double*)mxGetData(ge) : nullptr, &K);
            qmri_admm_destroy(st);
            if (r) {
                mxDestroyArray(dc);
                mxDestroyArray(ge);
            }
            check(r);
            plhs[0] = x.finish();
            const char* names[2] = {"dc_res", "gt_err"};
            plhs[1] = mxCreateStructMatrix(1, 1, 2, names);
            mxSetField(plhs[1], 0, "dc_res", dc);
            mxSetField(plhs[1], 0, "gt_err", ge);
        }
    } else if (cmd == "dict_load") {                         // (D single KxC, normD single, lut single KxQ) -> dict handle
        need(4);
        const mwSize* d = mxGetDimensions(prhs[1]);
        const int Q = dim_of(prhs[3], 1);
        if (!mxIsSingle(prhs[1]) || !mxIsSingle(prhs[2]) || !mxIsSingle(prhs[3]) || mxIsComplex(prhs[1]))
            mexErrMsgIdAndTxt("qmri:type", "pass single(real(dict.D)), single(dict.normD), single(dict.lut)");
        qmri_dict* dd = nullptr;
        check(qmri_dict_load(ctx(), (const float*)mxGetData(prhs[1]), (const float*)mxGetData(prhs[2]), (const float*)mxGetData(prhs[3]),
                             (int64_t)d[0], (int)d[1], Q, 0, (int64_t)d[0], &dd));
        g_dicts.push_back(dd);
        plhs[0] = handle_out(dd);
    } else if (cmd == "match") {                             // (dict, x[npix x C], Q) -> qmap, pd, mt, dm
        need(4);
        qmri_dict* dd = handle_in<qmri_dict>(prhs[1]);
        const int64_t npix = (int64_t)mxGetDimensions(prhs[2])[0];
        const int Q = (int)mxGetScalar(prhs[3]);
        CplxIn x(prhs[2]);
        mwSize pdims[2] = {(mwSize)npix, 1};
        CplxOut pd(2, pdims, mxSINGLE_CLASS);
        plhs[0] = mxCreateNumericMatrix((mwSize)npix, (mwSize)Q, mxSINGLE_CLASS, mxREAL);
        plhs[2] = mxCreateNumericMatrix((mwSize)npix, 1, mxSINGLE_CLASS, mxREAL);
        plhs[3] = mxCreateNumericMatrix((mwSize)npix, 1, mxINT32_CLASS, mxREAL);
        check(qmri_match(dd, x.p, x.dtype, npix, (float*)mxGetData(plhs[0]), (float*)pd.p, (float*)mxGetData(plhs[2]), (int32_t*)mxGetData(plhs[3])));
        plhs[1] = pd.finish();
    } else if (cmd == "fisp_signals" || cmd == "fisp_gram" || cmd == "fisp_compress") {
        // fisp_signals  (lut single K x 2, seq)                     -> sig single K x T
        // fisp_gram     (lut, seq)                                  -> G double T x T
        // fisp_compress (lut, seq, V double T x C [, a0, a1])       -> [D single (a1-a0) x C, normD single (a1-a0) x 1]
        // seq: struct with flip_deg, tr (T doubles), te, ti ([] = no inversion); a0, a1: 0-based atom range [a0, a1)
        need(3);
        const mxArray* lut = prhs[1];
        const mxArray* s = prhs[2];
        if (!mxIsSingle(lut) || mxIsComplex(lut) || dim_of(lut, 1) != 2) mexErrMsgIdAndTxt("qmri:type", "lut must be real single K x 2 (T1, T2)");
        const mxArray* flip = mxGetField(s, 0, "flip_deg");
        const mxArray* tr = mxGetField(s, 0, "tr");
        const mxArray* te = mxGetField(s, 0, "te");
        const mxArray* ti = mxGetField(s, 0, "ti");
        if (!flip || !tr || !te) mexErrMsgIdAndTxt("qmri:param", "seq.flip_deg, seq.tr and seq.te are required");
        if (!mxIsDouble(flip) || !mxIsDouble(tr) || mxIsComplex(flip) || mxIsComplex(tr))
            mexErrMsgIdAndTxt("qmri:type", "seq.flip_deg and seq.tr must be real double");
        if (mxGetNumberOfElements(flip) != mxGetNumberOfElements(tr)) mexErrMsgIdAndTxt("qmri:param", "seq.flip_deg and seq.tr differ in length");
        qmri_fisp_seq q;
        memset(&q, 0, sizeof(q));
        q.T = (int)mxGetNumberOfElements(flip);
        q.flip_deg = (const double*)mxGetData(flip);
        q.tr = (const double*)mxGetData(tr);
        q.te = mxGetScalar(te);
        q.inversion = ti && mxGetNumberOfElements(ti) > 0;
        q.ti = q.inversion ? mxGetScalar(ti) : 0.0;
        const int64_t K = (int64_t)dim_of(lut, 0);
        const float* L = (const float*)mxGetData(lut);
        if (cmd == "fisp_signals") {
            plhs[0] = mxCreateNumericMatrix((mwSize)K, (mwSize)q.T, mxSINGLE_CLASS, mxREAL);
            check(qmri_fisp_signals(ctx(), &q, L, K, (float*)mxGetData(plhs[0])));
        } else if (cmd == "fisp_gram") {
            plhs[0] = mxCreateNumericMatrix((mwSize)q.T, (mwSize)q.T, mxDOUBLE_CLASS, mxREAL);
            check(qmri_fisp_gram(ctx(), &q, L, K, (double*)mxGetData(plhs[0])));
        } else {
            need(4);
            const mxArray* V = prhs[3];
            if (!mxIsDouble(V) || mxIsComplex(V)) mexErrMsgIdAndTxt("qmri:type", "V must be real double T x C");
            const int64_t a0 = nrhs > 5 ? (int64_t)mxGetScalar(prhs[4]) : 0, a1 = nrhs > 5 ? (int64_t)mxGetScalar(prhs[5]) : K;
            if (dim_of(V, 0) != q.T) mexErrMsgIdAndTxt("qmri:param", "V must have T = %d rows", q.T);
            const int C = dim_of(V, 1);
            const mwSize n = a1 > a0 ? (mwSize)(a1 - a0) : 0;
            plhs[0] = mxCreateNumericMatrix(n, (mwSize)C, mxSINGLE_CLASS, mxREAL);
            plhs[1] = mxCreateNumericMatrix(n, 1, mxSINGLE_CLASS, mxREAL);
            check(qmri_fisp_compress(ctx(), &q, L, K, (const double*)mxGetData(V), C, a0, a1, (float*)mxGetData(plhs[0]),
                                     (float*)mxGetData(plhs[1])));
        }
    } else if (cmd == "shutdown") {
        shutdown();
    } else {
        mexErrMsgIdAndTxt("qmri:usage", "unknown command '%s'", cmd.c_str());
    }
}
