"""What the PnP-ADMM convergence history (AdmmSession.monitor, PnP_ADMM.m:106-109) costs at the benchmark job's shape: 120 slices,
spiral mask (S = 771), rho = 0.05, the random-init built-in UNetRes in tensor mode, at 224 x 224 and at 256 x 256.

For each image size one session is run in three modes - unmonitored, residual only, residual + ground-truth error - alternated
round by round in the same process, so clock and power drift fall on all three alike.  Per mode it reports the time of a
--iters-iteration run (CUDA events on the library's stream, a 256 MiB buffer written before each run so that the 1.6 / 2.1 GB
of loop state is not served from L2) and the x-update alone (AdmmSession.xupdate_only: the monitored kernel instances when
monitoring is on, without the once-per-iteration finalize), in us per slice-iteration.  The GPU's name and power limit are
read in the same run.  Inputs are a seeded smooth TSMI, not the benchmark's synthesised one: only the shapes matter here.

Usage (GPU box): python profiles/tools/monitor_cost.py [--rounds 3] [--iters 20] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "qmri-pnp-recon-poc_b200")]
import numpy as np  # noqa: E402

S, C_CH = 120, 10
MODES = ("off", "residual", "residual+gt")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    f = [s.strip() for s in out.stdout.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_max_clock": f[2]} if len(f) == 3 else {"nvidia_smi": out.stdout + out.stderr}


def tsmi(N, seed):
    rng = np.random.default_rng(seed)
    n = np.arange(N, dtype=np.float32)[:, None, None] / N
    m = np.arange(N, dtype=np.float32)[None, :, None] / N
    c = np.arange(C_CH, dtype=np.float32)[None, None, :]
    base = np.exp(-((n - 0.5) ** 2 + (m - 0.45) ** 2) * 8) * np.cos(0.3 * c) + 0.2 * np.sin(7 * n + c) * np.cos(5 * m)
    X = np.empty((N, N, C_CH, S), np.float32, order="F")
    for s in range(S):
        X[..., s] = base * (1.0 + 0.01 * s) + 0.05 * rng.standard_normal(base.shape, dtype=np.float32)
    return X


def measure(q, torch, bench, ctx, stream, net, N, args):
    P = q.setup_subsampling_spiralgrided(N, N, bench.SPIRAL_S, np.eye(C_CH), ctx=ctx)
    F = q.fft_operator(P)
    X = tsmi(N, N)
    Y = np.empty((P.nmeas, S), np.complex64, order="F")
    X0 = np.empty((N, N, C_CH, S), np.complex64, order="F")
    for s0 in range(0, S, 16):
        s1 = min(S, s0 + 16)
        y = q.awgn(F.forward(X[..., s0:s1]), bench.SNR_DB, "measured", seed=1000 + s0, ctx=ctx)
        Y[:, s0:s1] = y
        X0[..., s0:s1] = F.adjoint(y)
    param = {"iter": args.iters, "gamma": bench.RHO, "F": F, "X0": X0, "net": net, "denoiser_type": "single_level"}
    sess = q.AdmmSession(param, S)
    sess.upload(Y, X0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def set_mode(mode):
        if mode == "off":
            sess.monitor(enable=False)
        else:
            sess.monitor(X if mode == "residual+gt" else None)

    def timed(fn, reps, do_flush):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if do_flush:
            flush.zero_()
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    for mode in MODES:  # warm-up: graph capture and lazy initialisation of every mode
        set_mode(mode)
        sess.run(args.iters)
        sess.xupdate_only(2)
    torch.cuda.synchronize()
    run_ms = {m: [] for m in MODES}
    k1_us = {m: [] for m in MODES}
    reps = 20
    for _ in range(args.rounds):
        for mode in MODES:
            set_mode(mode)
            run_ms[mode].append(timed(lambda: sess.run(args.iters), 1, True))
            k1_us[mode].append(timed(lambda: sess.xupdate_only(reps), 1, False) * 1e3 / (reps * S))
    set_mode("residual+gt")
    sess.run(args.iters)
    h = sess.history()
    sess.close()
    out = {"image": f"{N} x {N}", "nmeas_per_slice": P.nmeas, "slices": S, "iters": args.iters, "rounds": args.rounds}
    for mode in MODES:
        out[mode] = {"run_ms": run_ms[mode], "run_ms_median": float(np.median(run_ms[mode])),
                     "slice_iterations_per_s": S * args.iters / (float(np.median(run_ms[mode])) * 1e-3),
                     "xupdate_us_per_slice_iteration": k1_us[mode], "xupdate_us_median": float(np.median(k1_us[mode]))}
    base_run, base_k1 = out["off"]["run_ms_median"], out["off"]["xupdate_us_median"]
    for mode in MODES[1:]:
        out[mode]["run_vs_off"] = out[mode]["run_ms_median"] / base_run
        out[mode]["xupdate_vs_off"] = out[mode]["xupdate_us_median"] / base_k1
    out["off"]["run_spread"] = (max(run_ms["off"]) - min(run_ms["off"])) / base_run
    out["last_history_row"] = {"dc_residual_slice0": float(h["dc_residual"][-1, 0]), "gt_error_slice0": float(h["gt_error"][-1, 0])}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--sizes", default="224,256")
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    import bench
    import qmri_b200 as q

    info = gpu_info()
    ctx = q.Context(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    net = q.UNetRes(bench.make_weights(), in_nc=10, ctx=ctx)
    net.set_precision("tc")
    res = {"what": "PnP-ADMM convergence history: unmonitored / residual only / residual + ground-truth error, alternated in one "
                   "process (profiles/tools/monitor_cost.py)", "gpu": info,
           "shapes": [measure(q, torch, bench, ctx, stream, net, int(n), args) for n in args.sizes.split(",")]}
    s = json.dumps(res)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
