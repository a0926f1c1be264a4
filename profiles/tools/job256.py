"""The benchmark job at N x N (--side, default 256): 8 volunteers x 15 slices from benchdata.make_qmaps(N=N, M=N), TSMIs synthesised on the
device, 30 dB AWGN, spiral mask (S = 771), rho = 0.05, 100 PnP-ADMM iterations with the random-init UNetRes (tensor mode), then
matching against 100 000 atoms - timed like bench.py (DESIGN.md section 5: CUDA events on the library's stream, warm-up first,
a 256 MiB buffer written between steps so the 1.6 GB of loop state is not served from L2).

Prints one JSON line (and writes it to --out): slice-iterations/s of the job, the x-update alone (us per slice-iteration and its
fraction of HBM counted at 20 B per pixel-channel), ms per denoiser forward, single-slice reconstruction latency, and the GPU's
name and power limit read in the same run.
Usage (GPU box): python profiles/tools/job256.py [--side 256] [--steps 2] [--warmup 1] [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "qmri-pnp-recon-poc_b200")]
import numpy as np  # noqa: E402

N, C_CH, HW = 256, 10, 256 * 256
VOLUNTEERS, PER_VOLUNTEER = 8, 15
HBM_DATASHEET_GBS = 7700.0   # HGX B200 data sheet, per GPU


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    f = [s.strip() for s in out.stdout.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_max_clock": f[2]} if len(f) == 3 else {"nvidia_smi": out.stdout + out.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--atoms", type=int, default=100000)
    ap.add_argument("--side", type=int, default=256, help="image side N == M (160, 192, 224 or 256)")
    ap.add_argument("--out")
    args = ap.parse_args()
    global N, HW
    N, HW = args.side, args.side * args.side
    import torch
    import bench
    import benchdata
    import qmri_b200 as q

    info = gpu_info()
    ctx = q.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    lib, vp = ctx.lib, C.c_void_p
    S, iters = VOLUNTEERS * PER_VOLUNTEER, args.iters

    t0 = time.time()
    dct = benchdata.make_dictionary(K_target=args.atoms, cut=3, seed=0)
    d = q.Dictionary(dct, ctx=ctx)
    X = np.empty((N, N, C_CH, S), np.float64, order="F")
    for vol in range(VOLUNTEERS):
        qm = benchdata.make_qmaps(seed=vol, S=PER_VOLUNTEER, N=N, M=N)              # [15 x 3 x N x N]
        for sl in range(PER_VOLUNTEER):
            X[..., vol * PER_VOLUNTEER + sl] = q.synthesize_tsmis(d, qm[sl])          # on the GPU
    P = q.setup_subsampling_spiralgrided(N, N, bench.SPIRAL_S, np.eye(C_CH), ctx=ctx)
    F = q.fft_operator(P)
    Y = np.empty((P.nmeas, S), np.complex128, order="F")
    X0 = np.empty((N, N, C_CH, S), np.complex128, order="F")
    for s0 in range(0, S, 16):
        s1 = min(S, s0 + 16)
        y = q.awgn(F.forward(X[..., s0:s1]), bench.SNR_DB, "measured", seed=1000 + s0, ctx=ctx)
        Y[:, s0:s1] = y
        X0[..., s0:s1] = F.adjoint(y)
    del X
    net = q.UNetRes(bench.make_weights(), in_nc=10, ctx=ctx)
    net.set_precision("tc")
    param = {"iter": iters, "gamma": bench.RHO, "cg_tol": 1e-4, "F": F, "X0": X0, "net": net, "denoiser_type": "single_level"}
    sess = q.AdmmSession(param, S)
    sess.upload(Y, X0)
    xr, xi = sess.state_dev()
    qmap_d = torch.empty(S * HW * 2, dtype=torch.float32, device="cuda")
    pd_d = torch.empty(S * HW * 2, dtype=torch.float32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    sys.stderr.write(f"[job256] setup {time.time() - t0:.1f} s: {S} slices, K = {d.K} atoms, nmeas = {P.nmeas}\n")

    def timed(fn, steps, warmup, do_flush=True):
        for _ in range(warmup):
            if do_flush:
                flush.zero_()
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            if do_flush:
                flush.zero_()
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def match(xr_, xi_, n):
        for s in range(n):
            off = s * C_CH * HW * 4
            q._capi.check(lib.qmri_match_dev(d.handle, vp(xr_ + off), vp(xi_ + off), HW, vp(qmap_d.data_ptr() + s * HW * 8),
                                            vp(pd_d.data_ptr() + s * HW * 8), None, None))

    def job():
        sess.run(iters)
        match(xr, xi, S)

    ms_job = timed(job, args.steps, args.warmup)
    ms_match = timed(lambda: match(xr, xi, S), 2, 1, do_flush=False)

    # x-update alone on the resident 120-slice state (1.6 GB: larger than L2)
    reps = 20
    ms_k1 = timed(lambda: sess.xupdate_only(reps), 3, 2, do_flush=False)
    t_k1 = ms_k1 * 1e-3 / (3 * reps)
    bpp = sess.xupdate_bytes()
    gbs_20 = 20.0 * HW * C_CH * S / t_k1 / 1e9
    peaks = bench.load_peaks()

    # denoiser forward on 120 slices
    vin = torch.rand(S * C_CH * HW, device="cuda")
    vout = torch.empty_like(vin)

    def fwd():
        q._capi.check(lib.qmri_unetres_forward_dev(net.handle, vp(vin.data_ptr()), vp(vout.data_ptr()), None, None, S, N, N))
    ms_fwd = timed(lambda: [fwd() for _ in range(6)], 2, 1, do_flush=False) / 12
    fwd_flops = net.flops(S, N, N)
    del vin, vout
    sess.close()

    # single-slice reconstruction latency: 100 iterations + matching of the slice, state resident
    sess1 = q.AdmmSession(dict(param, X0=X0[..., :1]), 1)
    sess1.upload(Y[:, :1], X0[..., :1])
    xr1, xi1 = sess1.state_dev()

    def one():
        sess1.run(iters)
        match(xr1, xi1, 1)
    ms_one = timed(one, 3, 1, do_flush=False) / 3
    sess1.close()

    line = {
        "what": f"{N} x {N} job: {S}-slice PnP-ADMM recon (spiral S = {bench.SPIRAL_S}, {P.nmeas // C_CH} samples per frame, rho {bench.RHO}, "
                f"{iters} iterations, random-init UNetRes 10->10 in tensor mode) + matching ({d.K} atoms, cut3)",
        "gpu": info,
        "slice_iterations_per_s": S * iters * args.steps / (ms_job * 1e-3),
        "ms_per_step": ms_job / args.steps, "steps": args.steps, "warmup": args.warmup,
        "matching_ms_per_step": ms_match / 2,
        "xupdate": {"us_per_slice_iteration": 1e6 * t_k1 / S, "state_bytes_per_pixel_channel": bpp,
                    "gbs_counted_at_20B": gbs_20,
                    "frac_of_hbm_datasheet_at_20B": gbs_20 / HBM_DATASHEET_GBS,
                    "frac_of_bench_peak_at_20B": gbs_20 / peaks["hbm_gbs"], "bench_peak_gbs": peaks["hbm_gbs"], "bench_peak_src": peaks["src"],
                    "timed": f"2 warm-up + 3 timed batches of {reps} x-updates on the resident {S}-slice state"},
        "denoiser": {"ms_per_forward": ms_fwd, "slices": S, "tflops": fwd_flops / (ms_fwd * 1e-3) / 1e12},
        "single_slice": {"ms_per_reconstruction": ms_one, "what": f"{iters} iterations + matching of one slice, state resident"},
    }
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
