"""Cost of simulating FISP-MRF dictionaries on the GPU (qmri_b200.fisp_gram / fisp_dictionary): K in {100 000, 1 048 576} atoms,
T in {1000, 200} pulses (cut0, cut3), C = 10.

Per shape: one warm-up call of each entry point, then --reps timed calls, each timed with CUDA events on the library's stream
(the whole call: the upload of the schedule and of the K x 2 look-up table, the kernels, the download of G or of D / normD).
  - fisp_gram: the EPG simulation of all K atoms in chunks of 32 768 plus the double-precision Gram accumulation.
  - fisp_compress (fisp_dictionary with a given V): the EPG simulation of all K atoms with the projection onto V fused in.
Rates:
  - EPG: live order-updates sum_i w_i per atom, w_i = live_orders(i, T) + 1 (oracle/epg.py), times 15 FP32 flops per update
    (the rotation with the relaxation folded in: three rows of one multiply and two fused multiply-adds), over the compress time.
  - Gram: K T (T + 1) / 2 double multiply-adds (the upper triangle) = K T (T + 1) flops, over (gram time - compress time).
The CPU oracle (oracle/epg.py epg_fisp_real, numpy float64, vectorised over 64 atoms) is timed on 64 atoms and extrapolated to K.
The GPU's name and power limit are read in the same run.

Usage (GPU box): python profiles/tools/fisp_dict.py [--reps 3] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "qmri-pnp-recon-poc_b200"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402

FLOPS_PER_UPDATE = 15


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    f = [s.strip() for s in out.stdout.strip().split(",")]
    return {"name": f[0], "power_limit": f[1], "sm_max_clock": f[2]} if len(f) == 3 else {"nvidia_smi": out.stdout + out.stderr}


def timed(torch, fn, reps):
    fn()  # warm-up
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="directory to write r06_fisp.json and r06_fisp_table.md to (without it the results are only printed)")
    args = ap.parse_args()
    import torch
    import qmri_b200 as q
    from oracle import epg
    from test_oracle_epg import schedule
    ctx = q.Context.default(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    res = {"what": "FISP-MRF dictionary simulation on the GPU (profiles/tools/fisp_dict.py)", "gpu": gpu_info(), "shapes": []}
    for T in (1000, 200):
        seq = dict(schedule(T, seed=0), ti=0.02)
        updates = sum(epg.live_orders(i, T) + 1 for i in range(T))
        rng = np.random.default_rng(0)
        l64 = np.stack([rng.uniform(0.1, 4.0, 64), rng.uniform(0.01, 0.6, 64)], axis=1)
        t0 = time.perf_counter()
        epg.epg_fisp_real(l64[:, 0], l64[:, 1], seq)
        cpu_per_atom = (time.perf_counter() - t0) / 64
        for K in (100_000, 1_048_576):
            lut = np.stack([rng.uniform(0.1, 4.0, K), rng.uniform(0.01, 0.6, K)], axis=1).astype(np.float32)
            G = q.fisp_gram(lut, seq, ctx)
            V = q.temporal_basis(G, 10)
            g_ms = timed(torch, lambda: q.fisp_gram(lut, seq, ctx), args.reps)
            c_ms = timed(torch, lambda: q.fisp_dictionary(lut, seq, V=V, ctx=ctx), args.reps)
            g, c = float(np.median(g_ms)), float(np.median(c_ms))
            row = {"T": T, "K": K, "live_order_updates_per_atom": updates, "gram_ms": g_ms, "compress_ms": c_ms,
                   "gram_ms_median": g, "compress_ms_median": c,
                   "epg_fp32_tflops_from_compress": K * updates * FLOPS_PER_UPDATE / (c * 1e-3) / 1e12,
                   "gram_fp64_tflops_from_difference": (K * T * (T + 1) / ((g - c) * 1e-3) / 1e12) if g > c else None,
                   "cpu_oracle_s_per_atom": cpu_per_atom, "cpu_oracle_s_extrapolated_to_K": cpu_per_atom * K}
            print(json.dumps(row), flush=True)
            res["shapes"].append(row)
    res["gpu_after"] = gpu_info()
    lines = [f"GPU: {res['gpu']}", "", "| T | K | fisp_gram ms | fisp_compress ms | EPG FP32 TFLOP/s | Gram FP64 TFLOP/s | CPU oracle s (extrapolated) |",
             "|---|---|---|---|---|---|---|"]
    for r in res["shapes"]:
        gt = "—" if r["gram_fp64_tflops_from_difference"] is None else f"{r['gram_fp64_tflops_from_difference']:.2f}"
        lines.append(f"| {r['T']} | {r['K']} | {r['gram_ms_median']:.1f} | {r['compress_ms_median']:.1f} | "
                     f"{r['epg_fp32_tflops_from_compress']:.2f} | {gt} | {r['cpu_oracle_s_extrapolated_to_K']:.0f} |")
    print("\n".join(lines))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r06_fisp.json"), "w") as f:
            json.dump(res, f)
        with open(os.path.join(args.out, "r06_fisp_table.md"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
