#!/usr/bin/env python
"""bench.py - PnP-ADMM MRF reconstruction + dictionary matching on B200 (contract: the task's bench section).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--mask spiral|epi] [--slices 120] [--iters 100]
                    [--dump-outputs DIR]

Metric (BASELINE.json): ADMM slice-iterations/s on 224 x 224 x 10 slices, whole job over all N GPUs.
Workload (north star, BASELINE configs[3]): the 120-slice job (8 synthetic volunteers x 15 slices, QMaps rendered through the
`main_synthesize_tsmis` path on the GPU, 30 dB AWGN), cut3 dictionary, spiral mask (771-sample curve, 6184 measurements per
slice; `--mask epi` = the 1/65 EPI comb of configs[2]), rho = 0.05, 100 PnP-ADMM iterations with the random-init DRUNet
(UNetRes 10->10), then T1/T2/PD dictionary matching of every pixel of every slice against K = 100 000 atoms.
One "step" = the whole job: x = PnP_ADMM(y, param) for every slice + out = mrf_dtm_cpu(dict, out, par).
`--gpus N` runs the SAME 120-slice job slice-sharded over N ranks (15 per GPU at N = 8, no collective on the path): strong
scaling - `value` = 120 * 100 * K / t (slice-iterations/s), t = max over ranks of the device time of K steps.

  value    : inputs (y, X0, dictionary, weights) resident in HBM; loop + matching only, device-timed
  e2e      : the reference-facing calls with HOST buffers: H2D of y and X0, the loop, D2H of x, then mrf_dtm_cpu on the host
             array (H2D of x, D2H of qmap and pd) - every copy inside the timed region
  roofline : the dominant kernel group = the denoiser's conv kernels (tensor pipe), timed back to back at the workload's
             slice count (working set >> L2, no flush needed); `frac_bound_from_step` = all denoiser flops of a step / the
             step's own time (an upper bound that needs no separate timing)
  roofline_k1 / roofline_k2 : x-update (HBM, 20 B per pixel-channel) and matching (its pipe), timed live on the same data
  extras   : single_slice (BASELINE configs[1]), epi_15 (configs[2] per-GPU shape), match_1M (configs[4], atom-sharded,
             NCCL (max, idx) + owner-computes outputs) - short legs, reported beside the headline
  cpu_baseline / `--impl reference`: the reference's CPU path restated by oracle/ (NumPy/SciPy x-update + PyTorch-CPU UNetRes +
             blocked-sgemm matching) on the host cores - MATLAB / Octave are absent from the image (kind "port").
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree and leaves nothing in it
ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "qmri-pnp-recon-poc_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_IMG, C_CH = 224, 10
HW = N_IMG * N_IMG
SPIRAL_S = 771
EPI_PCT = 1.0 / 65.0
RHO = 0.05
SNR_DB = 30.0
METRIC = "ADMM slice-iterations/s (224x224x10 slices; step = 120-slice PnP-ADMM recon + T1/T2/PD matching)"


def workload_config(args, world):
    """The `config` both arms print (the driver compares them)."""
    return {"workload": f"BASELINE configs[3]: {args.slices}-slice PnP-ADMM recon (cut{args.cut}, {args.mask} mask, rho {RHO}, "
                        f"{args.iters} iterations, random-init UNetRes 10->10) + dictionary matching ({args.atoms} atoms)",
            "slices": args.slices, "iters_per_step": args.iters, "mask": args.mask, "atoms": args.atoms, "cut": args.cut,
            "l2": "inputs larger than L2 (120 slices = 1.2 GB of state); 256 MiB buffer written between steps as well",
            "parallelism": f"slice-sharded x{world} (strong scaling of one job), no collective on the path"}


def load_traffic():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def synthetic_slices(S, seed):
    """Seeded smooth brain-like 10-channel real TSMIs (N x M x C x S) - the analytic stand-in used by tests and the CPU arm
    (the GPU arm renders its slices from QMaps through the dictionary; throughput does not depend on content)."""
    rng = np.random.default_rng(seed)
    n = np.arange(N_IMG)[:, None, None, None] / N_IMG - 0.5
    m = np.arange(N_IMG)[None, :, None, None] / N_IMG - 0.5
    c = np.arange(C_CH)[None, None, :, None]
    s = rng.uniform(0.8, 1.2, size=(1, 1, 1, S))
    brain = ((n / 0.42) ** 2 + (m / 0.36) ** 2 <= 1.0) * 1.0
    X = brain * (np.cos(0.35 * c) * np.exp(-4 * (n ** 2 + m ** 2)) * s + 0.15 * np.sin(9 * n * s + c) * np.cos(7 * m))
    X = X + 0.01 * rng.standard_normal(X.shape) * brain
    X *= np.sign(X[:, :, 0:1, :] + 1e-30)  # channel 1 non-negative, like main_synthesize_tsmis.m:97-98
    return np.asfortranarray(X)


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region through NVML (fallback: one nvidia-smi query per sample).
    Samples are taken by the timing loop once the timed steps are enqueued, sparsely (default every 2 s): a query can stall
    this process's launches for tens of ms, which is < 1 % at this period and is part of the reported time."""

    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.reasons, self.mx = [], set(), None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.idx
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                phys = int(vis.split(",")[self.idx])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None
        self.sample()              # first query outside the timed region (lazy NVML initialisation takes ~0.5 s)
        self.sm, self.reasons = [], set()

    def sample(self):
        try:
            self._sample()
        except Exception:
            pass

    def _sample(self):
        if self.nvml is not None:
            self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)))
            mask = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            for nm, bit in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(nm)
            return
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout
        f = [x.strip() for x in out.strip().split(",")]
        self.sm.append(float(f[0]))
        self.mx = float(f[1])
        for nm, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
            if val.lower().startswith("active"):
                self.reasons.add(nm)

    def stop(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["clock sampling unavailable"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.mx, "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# =====================================================================================================================
# reference arm / cpu_baseline: the reference's CPU path (oracle/ restatement) on the host cores
# =====================================================================================================================
class CpuReference:
    """One slice of the job on the CPU: x = PnP_ADMM(y, param) restated (oracle.admm: NumPy x-update with scipy.fft workers +
    the PyTorch-CPU UNetRes the reference defines) and mrf_dtm_cpu restated as the reference computes it (single-precision
    D * x' in blocks of pixels, abs, max - oracle.matching precision 'f32').  Thread settings: intra-op threads for torch and
    scipy.fft workers are tuned once (all hardware threads vs physical cores) during warm-up, BLAS left alone."""

    def __init__(self, args):
        import torch
        import benchdata
        from oracle import sampling, unetres
        self.args = args
        self.ncpu = os.cpu_count() or 1
        self.torch = torch
        V = np.eye(C_CH)
        P = (sampling.setup_subsampling_spiralgrided(N_IMG, N_IMG, SPIRAL_S, V) if args.mask == "spiral"
             else sampling.setup_subsampling_epi(N_IMG, N_IMG, EPI_PCT, V))
        self.F = FastFOperator(P, workers=self.ncpu)
        X = synthetic_slices(1, 1000)[..., 0]
        Y = self.F.forward(X)
        rng = np.random.default_rng(0)
        self.Y = Y + (rng.standard_normal(Y.shape) + 1j * rng.standard_normal(Y.shape)) * np.sqrt(np.mean(np.abs(Y) ** 2) / 10 ** (SNR_DB / 10) / 2)
        self.X0 = self.F.adjoint(self.Y)
        self.sd = unetres.make_state_dict(10, seed=0)
        self.unetres = unetres
        self.dict = benchdata.make_dictionary(K_target=args.atoms, cut=args.cut, seed=0)
        self.threads = self.ncpu
        self.x_last = self.X0

    def set_threads(self, t):
        self.threads = t
        self.torch.set_num_threads(t)
        self.F.workers = t

    def tune(self):
        """Pick the faster of {all hardware threads, half of them (= physical cores with SMT)} on two iterations."""
        best, best_t = None, self.ncpu
        for t in sorted({self.ncpu, max(1, self.ncpu // 2)}, reverse=True):
            self.set_threads(t)
            self.iterations(1)
            dt = self.iterations(2)
            if best is None or dt < best:
                best, best_t = dt, t
        self.set_threads(best_t)
        return best_t

    def iterations(self, n):
        from oracle.admm import pnp_admm
        param = {"iter": n, "gamma": RHO, "F": self.F, "X0": self.X0,
                 "net": lambda v: self.unetres.denoise_matlab_layout(self.sd, v)}
        t0 = time.perf_counter()
        self.x_last = pnp_admm(self.Y, param, solver="closed")
        return time.perf_counter() - t0

    def match(self, npix):
        """mrf_dtm_cpu.m:84-98,136-148 on the first npix pixels of the last reconstruction, all K atoms, the way a tuned CPU
        build computes it: single precision, D * x' as two multi-threaded sgemms (real and imaginary part of x; D is real),
        |ip|^2, max over atoms, gather of pd and the LUT rows (the same result as oracle.matching, precision 'f32')."""
        torch = self.torch
        x = self.x_last.reshape((HW, C_CH), order="F")[:npix]
        t0 = time.perf_counter()
        D = torch.from_numpy(self.dict["D"])                              # K x C float32
        xr = torch.from_numpy(np.ascontiguousarray(x.real, dtype=np.float32))
        xi = torch.from_numpy(np.ascontiguousarray(x.imag, dtype=np.float32))
        K = D.shape[0]
        bs = max(1, min(npix, int(1e9 // K)))                             # par.fp.blockSize = 1e9 (main_recon_tsmis_FFT.m:309)
        for c0 in range(0, npix, bs):
            ipr = D @ xr[c0:c0 + bs].T                                    # K x B
            ipi = D @ xi[c0:c0 + bs].T
            dm = torch.argmax(ipr * ipr + ipi * ipi, dim=0)
            cols = torch.arange(dm.numel())
            nd = torch.from_numpy(self.dict["normD"])[dm]
            pd = torch.complex(ipr[dm, cols], -ipi[dm, cols]) / nd          # ip = D * ctranspose(x)
            qmap = torch.from_numpy(self.dict["lut"])[dm]
            del pd, qmap
        return time.perf_counter() - t0

    def sample(self, n_iters, match_px):
        """Seconds per slice-iteration of the whole job, extrapolated from a bounded sample: n_iters ADMM iterations of one
        slice + matching of match_px pixels; job cost per slice = iters * t_iter + t_match(224^2 pixels)."""
        t_it = self.iterations(n_iters) / n_iters
        t_px = self.match(match_px) / match_px
        per_slice = self.args.iters * t_it + HW * t_px
        return per_slice / self.args.iters, t_it, t_px


class FastFOperator:
    """oracle.sampling.FOperator with scipy.fft (multi-threaded pocketfft) instead of numpy.fft - same arithmetic, the
    faster CPU library BASELINE.md section 2 names."""

    def __init__(self, P, workers):
        self.P = P
        self.N, self.M, self.C = P.N, P.M, P.C
        self.workers = workers

    def forward(self, x):
        import scipy.fft as sfft
        xh = sfft.fft2(np.asarray(x).reshape(self.N, self.M, self.C), axes=(0, 1), workers=self.workers)
        return self.P.for_(xh.reshape(-1, order="F")) / np.sqrt(self.N * self.M)

    def adjoint(self, y):
        import scipy.fft as sfft
        k = self.P.adj(np.asarray(y)).reshape((self.N, self.M, self.C), order="F")
        return sfft.ifft2(k, axes=(0, 1), workers=self.workers) * np.sqrt(self.N * self.M)


REF_ENVS = {"inherited": {}, "omp1": {"OMP_NUM_THREADS": "1"}, "omp1_passive": {"OMP_NUM_THREADS": "1", "OMP_WAIT_POLICY": "PASSIVE"}}


def pick_reference_env(args):
    """The CPU arm's speed depends on how the OpenMP runtimes of NumPy / SciPy / PyTorch share the cores (measured on the B200
    hosts: the same code ran 4.2 it/s with the inherited environment and 8 it/s under torchrun's OMP_NUM_THREADS=1, which stops
    the second runtime's spinning pool from oversubscribing; on other hosts it is the other way round).  Environment variables
    must be set before the libraries load, so each candidate is probed in a child process (two iterations) and the fastest is
    used for the measurement - the reference arm gets the best configuration the box offers."""
    best, best_name = None, "inherited"
    for name, env in REF_ENVS.items():
        e = dict(os.environ, QMRI_REF_CHILD=name, **env)
        if name == "inherited":
            e = dict(os.environ, QMRI_REF_CHILD=name)
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-probe", "--mask", args.mask, "--atoms", "2000", "--cut", str(args.cut)]
        try:
            out = subprocess.run(cmd, env=e, capture_output=True, text=True, timeout=600)
            t = float(out.stdout.strip().splitlines()[-1])
        except Exception:
            continue
        sys.stderr.write(f"[bench] reference environment {name}: {1e3 * t:.1f} ms per ADMM iteration\n")
        if best is None or t < best:
            best, best_name = t, name
    return best_name


def run_reference(args, rank, world):
    if rank != 0:
        return  # the other ranks exit 0 without work
    if args.ref_probe:   # child of pick_reference_env: seconds per ADMM iteration with tuned thread counts
        ref = CpuReference(args)
        ref.tune()
        print(ref.iterations(2) / 2)
        return
    if "QMRI_REF_CHILD" not in os.environ:
        name = pick_reference_env(args)
        env = dict(os.environ, QMRI_REF_CHILD=name, **REF_ENVS[name])
        sys.stdout.flush()
        os.execve(sys.executable, [sys.executable, os.path.abspath(__file__)] + sys.argv[1:], env)
    ref = CpuReference(args)
    threads = ref.tune()   # untimed: also warms oneDNN primitives / FFT plans
    for _ in range(max(0, args.warmup - 1)):
        ref.sample(1, 256)
    times = []
    t_total = 0.0
    for _ in range(args.steps):
        t0 = time.perf_counter()
        per_it, t_it, t_px = ref.sample(args.ref_iters, args.ref_match_px)
        t_total += time.perf_counter() - t0
        times.append((per_it, t_it, t_px))
    per_it = float(np.mean([t[0] for t in times]))
    value = 1.0 / per_it
    sample = (f"each step = {args.ref_iters} ADMM iterations of one slice + matching of {args.ref_match_px} pixels against all "
              f"{args.atoms} atoms, extrapolated to the job (per slice: {args.iters} iterations + {HW} pixels); measured "
              f"{1e3 * np.mean([t[1] for t in times]):.1f} ms per iteration, {1e9 * np.mean([t[2] for t in times]) / args.atoms:.3f} ns per px-atom; "
              f"oracle/ restatement (scipy.fft x-update + PyTorch-CPU UNetRes + sgemm matching), {threads} threads of {ref.ncpu} "
              f"(tuned), OpenMP environment '{os.environ.get('QMRI_REF_CHILD', 'inherited')}' (fastest of {list(REF_ENVS)}); MATLAB / Octave absent "
              f"from the image; N > 1: rank 0 alone runs this CPU job")
    line = {
        "metric": METRIC, "value": value, "unit": "slice-iterations/s", "impl": "reference", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64 x-update / f32 denoiser and matching", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "slice-iterations/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "slice-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# =====================================================================================================================
# our arm
# =====================================================================================================================
def make_weights():
    """torch.manual_seed(0) default-init UNetRes weights in the reference's construction order (main_train.py:247,264-266)."""
    import torch
    import torch.nn as nn
    import qmri_b200 as q
    torch.manual_seed(0)
    sd = {}
    for key, shape in q.state_dict_keys(10):
        if re.fullmatch(r"m_up\d\.0\.weight", key):
            m = nn.ConvTranspose2d(shape[0], shape[1], 2, 2, 0, bias=False)
        elif shape[2] == 2:
            m = nn.Conv2d(shape[1], shape[0], 2, 2, 0, bias=False)
        else:
            m = nn.Conv2d(shape[1], shape[0], 3, 1, 1, bias=False)
        sd[key] = m.weight.detach()
    return sd


def run_ours(args, rank, world, local_rank):
    import torch
    import benchdata
    import qmri_b200 as q
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = q.Context(local_rank)
    # a dedicated torch stream shared with the library: CUDA events recorded on it see the library's kernels, and NCCL
    # collectives issued by torch are ordered against them without host synchronisation
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    peaks = load_peaks()
    iters = args.iters
    g0, g1 = q.slice_shard(args.slices, world, rank)
    S = g1 - g0
    if S < 1:
        raise SystemExit(f"rank {rank}: no slices to reconstruct ({args.slices} slices over {world} ranks)")
    lib = ctx.lib
    vp = C.c_void_p

    def log(msg):
        if rank == 0:
            sys.stderr.write(f"[bench] {msg}\n")
            sys.stderr.flush()

    # ---- problem: dictionary -> QMaps -> TSMIs (on the GPU) -> k-space + noise (on the GPU) -------------------------
    t_setup = time.time()
    dct = benchdata.make_dictionary(K_target=args.atoms, cut=args.cut, seed=0)
    d = q.Dictionary(dct, ctx=ctx)
    K = d.K
    qmaps = benchdata.volunteer_slices(g0, g1)                                  # [S x 3 x 224 x 224]
    X = np.empty((N_IMG, N_IMG, C_CH, S), np.float64, order="F")
    for s in range(S):
        X[..., s] = q.synthesize_tsmis(d, qmaps[s])                               # main_synthesize_tsmis.m:84-98 on the GPU
    V = np.eye(C_CH)
    if args.mask == "spiral":
        P = q.setup_subsampling_spiralgrided(N_IMG, N_IMG, SPIRAL_S, V, ctx=ctx)
    else:
        P = q.setup_subsampling_epi(N_IMG, N_IMG, EPI_PCT, V, ctx=ctx)
    F = q.fft_operator(P)
    Y = np.empty((P.nmeas, S), np.complex128, order="F")
    X0 = np.empty((N_IMG, N_IMG, C_CH, S), np.complex128, order="F")
    for s0 in range(0, S, 16):                                                    # bounded host temporaries
        s1 = min(S, s0 + 16)
        y = q.awgn(F.forward(X[..., s0:s1]), SNR_DB, "measured", seed=1000 + g0 + s0, ctx=ctx)   # main_recon_tsmis_FFT.m:237-243
        Y[:, s0:s1] = y
        X0[..., s0:s1] = F.adjoint(y)                                             # param.X0 = F.adjoint(Y), :292
    net = q.UNetRes(make_weights(), in_nc=10, ctx=ctx)
    net.set_precision(args.precision)
    param = {"iter": iters, "gamma": RHO, "cg_tol": 1e-4, "F": F, "X0": X0, "net": net, "denoiser_type": "single_level"}
    sess = q.AdmmSession(param, S)
    log(f"setup {time.time() - t_setup:.1f} s: {S} slices on this rank, K = {K} atoms, nmeas = {P.nmeas}")

    def pinned(a):
        t = torch.empty(a.size * (2 if np.iscomplexobj(a) else 1), dtype=torch.float64).pin_memory()
        v = t.numpy().view(a.dtype).reshape(a.shape, order="F")
        v[...] = a
        return t, v
    _ty, Yp = pinned(Y)
    _tx, X0p = pinned(X0)
    _to, Xout = pinned(np.zeros((N_IMG, N_IMG, C_CH, S), np.complex128, order="F"))
    del X, Y, X0
    qmap_h = torch.empty(S * HW * 2, dtype=torch.float32).pin_memory()
    pd_h = torch.empty(S * HW * 2, dtype=torch.float32).pin_memory()
    qmap_d = torch.empty(S * HW * 2, dtype=torch.float32, device="cuda")
    pd_d = torch.empty(S * HW * 2, dtype=torch.float32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup, sampler=None, collective=True, label=None, do_flush=True):
        """collective=False: a leg only this rank runs (no barrier / all-reduce)."""
        sync = barrier if collective else torch.cuda.synchronize
        for _ in range(warmup):
            if do_flush:
                flush.zero_()
            fn()
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        l0 = ctx.launch_count
        e0.record(stream)
        for i in range(steps):
            if do_flush:
                flush.zero_()      # evict L2 between steps (256 MiB > 126 MB L2)
            fn()
            marks[i].record(stream)
        e1.record(stream)
        if sampler is not None:    # sample clocks while the GPU works through the enqueued steps
            sampler.sample()
            while not e1.query():
                time.sleep(args.clock_period)
                sampler.sample()
        sync()
        ms = e0.elapsed_time(e1)
        if rank == 0 and label:
            per = [round(([e0] + marks)[i].elapsed_time(marks[i]), 2) for i in range(steps)]
            log(f"{label}: per-step ms {per}")
        return (max_over_ranks(ms) if collective else ms), ctx.launch_count - l0

    xr_p, xi_p = None, None

    def match_resident():
        """out = mrf_dtm_cpu(dict, out, par) on the reconstructed slices where they lie (planar [S][C][M][N] in HBM)."""
        for s in range(S):
            off = s * C_CH * HW * 4
            q._capi.check(lib.qmri_match_dev(d.handle, vp(xr_p + off), vp(xi_p + off), HW, vp(qmap_d.data_ptr() + s * HW * 8),
                                            vp(pd_d.data_ptr() + s * HW * 8), None, None))

    def job_resident():
        sess.run(iters)
        match_resident()

    # ---- value: loop + matching, inputs resident in HBM ----------------------------------------------------------------
    sess.upload_raw(Yp, X0p)
    xr_p, xi_p = sess.state_dev()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, launches = timed(job_resident, args.steps, args.warmup, sampler if rank == 0 else None, label="value pass")
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["how"] = f"NVML queries every {args.clock_period} s during the timed pass `value` is taken from"
    value = args.slices * iters * args.steps / (ms_dev * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, args.slices, g0, sess, Xout, qmap_d, pd_d, dist, rank)
    # share of matching inside the step (same data, same stream)
    ms_match, _ = timed(match_resident, 2, 1, label="matching only", do_flush=False)

    # ---- e2e: the reference-facing calls with host buffers ---------------------------------------------------------------
    def e2e_step():
        sess.upload_raw(Yp, X0p)                      # H2D y, X0
        sess.run(iters)
        sess.download(Xout)                           # D2H x (synchronises)
        for s in range(S):                            # out = mrf_dtm_cpu(dict, out, par) per slice, host arrays in and out
            xs = Xout[..., s]
            q._capi.check(lib.qmri_match(d.handle, vp(xs.ctypes.data), q.QMRI_C128, HW, vp(qmap_h.data_ptr() + s * HW * 8),
                                        vp(pd_h.data_ptr() + s * HW * 8), None, None))
    ms_e2e, _ = timed(e2e_step, args.steps, 1, label="e2e pass")
    e2e_value = args.slices * iters * args.steps / (ms_e2e * 1e-3)
    h2d = int(Yp.nbytes + X0p.nbytes + Xout.nbytes)            # y, X0, and x again for the matching call
    d2h = int(Xout.nbytes + qmap_h.numel() * 4 + pd_h.numel() * 4)

    # ---- roofline legs ---------------------------------------------------------------------------------------------------
    tensor_peak = peaks["bf16_tflops_sustained"]
    traffic = load_traffic()
    vin = torch.rand(S * 10 * HW, device="cuda")
    vout = torch.empty_like(vin)

    def fwd():
        q._capi.check(lib.qmri_unetres_forward_dev(net.handle, vp(vin.data_ptr()), vp(vout.data_ptr()), None, None, S, N_IMG, N_IMG))
    reps_f = 6 if S >= 8 else 30
    ms_fwd, _ = timed(lambda: [fwd() for _ in range(reps_f)], 2, 1, label="denoiser forwards", do_flush=False)
    ms_per_fwd = ms_fwd / (2 * reps_f)
    fwd_flops = net.flops(S, N_IMG, N_IMG)
    fwd_tflops = fwd_flops / (ms_per_fwd * 1e-3) / 1e12
    step_ms = ms_dev / args.steps
    t_fwd = traffic.get(f"unetres_forward_S{S}") or traffic.get(f"unetres_forward_S{min(S, 15) if S >= 15 else S}")   # exact slice count first
    max_chunk = int(os.environ.get("QMRI_NET_CHUNK", "128"))   # unetres.h max_chunk: slices per pass through the network
    chunks = -(-S // max_chunk)
    per_chunk = -(-S // chunks)
    roofline = {"bound": "tensor", "kernel": f"UNetRes forward = 66 launches per pass of <= {max_chunk} slices (tc_conv3x3_pair_kernel: 58 3x3 convs = 97% of the algorithmic flops, + head and tail as zero-padded 64 -> 64 convs)",
                "achieved": fwd_tflops, "peak": tensor_peak, "unit": "TFLOP/s", "frac": fwd_tflops / tensor_peak,
                "frac_of_3_product_ceiling": 3 * fwd_tflops / tensor_peak,
                "frac_bound_from_step": fwd_flops * (iters - 1) / (step_ms * 1e-3) / 1e12 / tensor_peak,
                "traffic": ((t_fwd["dram_read_bytes"] + t_fwd["dram_write_bytes"]) * (S / t_fwd.get("slices", 15))) if t_fwd else None,
                "traffic_note": (t_fwd or {}).get("how", "no committed ncu capture for this slice count"),
                "peak_source": f"{peaks['src']} dense bf16 (sustained); split-bf16 operands need 3 bf16 products per fp32 product (1e-4 parity bar), so the ceiling for algorithmic flops is peak / 3",
                "ms_per_forward": ms_per_fwd, "slices": S, "chunks": f"{chunks} x {per_chunk}", "precision_mode": args.precision,
                "algorithmic_flops_per_forward": fwd_flops,
                "consistency": f"{iters - 1} forwards x {ms_per_fwd:.3f} ms = {(iters - 1) * ms_per_fwd:.1f} ms of the {step_ms:.1f} ms step"}
    del vin, vout
    # K1 on the resident state (S slices; >> L2 from ~13 slices on), timed twice: (b) straight after the denoiser legs, i.e. in the
    # power-capped clock state the job leaves behind, and (a) alone, after an idle period that lets the power cap release -
    # MEASURED_PEAKS.json's HBM figure is a burst number for a kernel timed alone, and this kernel's speed follows the SM clock.
    reps = 20

    def k1_leg(label):
        smp = ClockSampler(local_rank)
        if rank == 0:
            smp.start()
        ms, _ = timed(lambda: sess.xupdate_only(reps), 3, 2, label=label, do_flush=False)
        if rank == 0:
            smp.sample()
        return ms, (smp.stop() if rank == 0 else None)
    ms_k1_hot, clk_hot = k1_leg("x-update only (straight after the denoiser legs)")
    barrier()
    time.sleep(args.k1_idle)
    ms_k1, clk_alone = k1_leg("x-update only (alone, after %.0f s idle)" % args.k1_idle)
    t_launch = ms_k1 * 1e-3 / (3 * reps)
    t_launch_hot = ms_k1_hot * 1e-3 / (3 * reps)
    bpp = sess.xupdate_bytes()                     # 8: real-state loop (read v, write Re w'); 20: complex-state kernels
    gbs = float(bpp) * HW * C_CH * S / t_launch / 1e9
    t_k1 = traffic.get(f"k1_xupdate_S{S}_{bpp}B") or (traffic.get(f"k1_xupdate_S{S}") if bpp == 20 else None)
    us_it = 1e6 * t_launch / S
    roof_k1 = {"bound": "hbm", "kernel": ("x-update, real-state loop: stream_fwdr + stream_solver + stream_adjr (PnP_ADMM.m:102,115-118,144 fused)" if bpp == 8
                                          else "x-update, complex-state kernels (PnP_ADMM.m:102,115-118,144 fused)"),
               "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
               "frac": gbs / peaks["hbm_gbs"], "traffic": (t_k1["dram_read_bytes"] + t_k1["dram_write_bytes"]) if t_k1 else None,
               "traffic_note": (t_k1 or {}).get("how", "no committed ncu capture for this slice count"),
               "slices": S, "us_per_slice_iteration": us_it, "algorithmic_bytes_per_pixel_channel": bpp,
               "algorithmic_bytes_per_launch": bpp * HW * C_CH * S,
               "vs_complex_state_target": {"what": "the north-star target was written for the 20 B/px-ch complex-state form: 70 % of HBM there = "
                                                   f"{20.0 * HW * C_CH / (0.7 * peaks['hbm_gbs'] * 1e9) * 1e6:.2f} us per slice-iteration",
                                           "us_per_slice_iteration": us_it,
                                           "frac_if_counted_at_20B": 20.0 * HW * C_CH * S / t_launch / 1e9 / peaks["hbm_gbs"]},
               "timed": f"alone: {args.k1_idle:.0f} s idle after the denoiser legs, 2 warm-up + 3 timed batches of {reps} x-updates; SM clock right after: "
                        f"{(clk_alone or {}).get('sm_mhz')} MHz",
               "in_job_power_state": {"what": "the same leg straight after the denoiser legs (power-capped clocks, as inside the job)",
                                      "us_per_slice_iteration": 1e6 * t_launch_hot / S,
                                      "achieved": float(bpp) * HW * C_CH * S / t_launch_hot / 1e9,
                                      "frac": float(bpp) * HW * C_CH * S / t_launch_hot / 1e9 / peaks["hbm_gbs"],
                                      "sm_mhz": (clk_hot or {}).get("sm_mhz")},
               "l2_note": None if S * bpp * HW * C_CH > 2 * (126 << 20) else "working set fits L2: not an HBM measurement"}
    # K2 from the matching-only leg above (complex data: 40 flop per px-atom).  Pipe choice (profiles/r02_k2_pipes.md, from ncu
    # counters): the tcgen05 tf32 kernel from 2048 atoms on, the FP32-FMA kernel below and for C > 10.
    pxa = S * HW * K * 2 / (ms_match * 1e-3)
    sm_mhz = ((clocks or {}).get("sm_max_mhz") or 1965.0)
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    pipe = "fma" if (os.environ.get("QMRI_K2_PIPE") == "fma" or K < 2048) else "tensor"
    if pipe == "tensor":
        tf32_peak = peaks["bf16_tflops_sustained"] / 2.0
        roof_k2 = {"bound": "tensor", "kernel": "match_tc_kernel (tcgen05 kind::tf32, split operands, group-maximum epilogue, FP32 rescore)",
                   "achieved": pxa * 40 / 1e12, "peak": tf32_peak, "unit": "TFLOP/s", "frac": pxa * 40 / 1e12 / tf32_peak,
                   "peak_source": f"{peaks['src']} dense bf16 (sustained) / 2 = tf32 rate",
                   "issued_tflops": pxa * 128 / 1e12, "frac_issued": pxa * 128 / 1e12 / tf32_peak,
                   "issued_note": "the split a = hi + lo lays 3 x 10 channels along K = 32 and complex pixels take two accumulators: 128 tensor "
                                  "flops are issued per 40 algorithmic ones",
                   "limiter": "the epilogue, not the MMA: every score is read back from TMEM and costs 3 FP32 instructions on 8 warps "
                              "(profiles/r02_k2_pipes.md: tensor pipe 41 % active before the 8-warp epilogue; TMEM-read + FP32 microbenchmark "
                              "profiles/r02_ldtm_bench.txt: 22.8 scores/clk/SM with 4 warps, 30.9 with 8)",
                   "scores_per_clk_per_sm": pxa / (148 * sm_mhz * 1e6),
                   "vs_fp32_fma_kernel": {"px_atoms_per_s": 1.26e12, "what": "match_kernel on the same data (profiles/r02_k2_pipes.md): 76 % FMA-pipe active, 0.67 of the FP32 peak"},
                   "px_atoms_per_s": pxa, "atoms": K, "pixels": S * HW,
                   "ms_per_slice": ms_match / (2 * S), "share_of_step": (ms_match / 2) / step_ms}
    else:
        roof_k2 = {"bound": "fp32", "kernel": "match_kernel", "achieved": pxa * 40 / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                   "frac": pxa * 40 / 1e12 / fp32_peak, "px_atoms_per_s": pxa, "atoms": K, "pixels": S * HW,
                   "ms_per_slice": ms_match / (2 * S), "share_of_step": (ms_match / 2) / step_ms}

    # ---- extras: the other BASELINE configs, short legs ---------------------------------------------------------------------
    extras = {}
    if not args.skip_extra:
        extras = run_extras(args, q, ctx, net, F, d, dct, Yp, X0p, timed, log, rank, world, dist, stream, peaks)

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        # the reference arm as a child process (it picks its own OpenMP environment): one step of its bounded sample
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1", "--mask", args.mask, "--cut", str(args.cut),
               "--atoms", str(args.atoms), "--slices", str(args.slices), "--iters", str(args.iters), "--ref-iters", str(args.cpu_iters),
               "--ref-match-px", str(args.ref_match_px)]
        try:
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
            out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1200)
            cpu = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:  # the GPU numbers stand on their own
            cpu = {"value": None, "unit": "slice-iterations/s", "cores": os.cpu_count(), "kind": "port", "sample": f"reference arm failed: {e}"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "slice-iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 (x-update fp32 FFT; denoiser " + ("split-bf16 tcgen05, fp32 accumulate" if args.precision == "tc" else "fp32 CUDA cores") + "; matching fp32)",
            "data": "synthetic",
            "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": "slice-iterations/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d * world if world > 1 else h2d, "d2h_bytes_per_step": d2h * world if world > 1 else d2h,
                    "bytes_note": "rank 0's bytes x ranks" if world > 1 else "y, X0 up; x down; x up again for mrf_dtm_cpu; qmap, pd down"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_k1": roof_k1,
            "roofline_k2": roof_k2,
            "slices_per_gpu": S,
            "cpu_baseline": cpu,
        }
        line.update(extras)
        print(json.dumps(line))
    sess.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


DUMP_PIXELS = 1 << 19   # 96 B per pixel (x: C complex channels, qmap: T1 and T2, pd: complex) -> 48 MiB of files at most


def dump_outputs(path, slices, g0, sess, x_host, qmap_d, pd_d, dist, rank):
    """What the timed step hands its caller, taken from its last step: x = PnP_ADMM(y, param) and out.qmap / out.pd of
    mrf_dtm_cpu, at the same pixels of the job - all of them when the job has at most DUMP_PIXELS, else a sorted sample drawn
    with a fixed seed (independent of the number of ranks).  Written as float32 to path/x.npy [P x C x 2] (re, im of every
    channel), path/qmap.npy [P x 2] (T1, T2) and path/pd.npy [P x 2] (re, im); pixel g is slice g // (N M), column-major
    pixel g % (N M) of that slice."""
    import torch
    S = x_host.shape[3]
    total = slices * HW
    pick = np.arange(total) if total <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(total, DUMP_PIXELS, replace=False))
    mine = (pick >= g0 * HW) & (pick < (g0 + S) * HW)
    s, p = np.divmod(pick[mine] - g0 * HW, HW)
    sess.download(x_host)
    x = x_host.reshape((HW, C_CH, S), order="F")[p, :, s]                       # P_mine x C complex
    rows = np.zeros((pick.size, 2 * C_CH + 4), np.float32)
    rows[mine, :2 * C_CH] = np.stack([x.real, x.imag], axis=2).reshape(-1, 2 * C_CH)
    rows[mine, 2 * C_CH:2 * C_CH + 2] = qmap_d.view(S, 2, HW).cpu().numpy()[s, :, p]   # per slice: npix x 2 column-major
    rows[mine, 2 * C_CH + 2:] = pd_d.view(S, HW, 2).cpu().numpy()[s, p]              # per slice: npix complex interleaved
    if dist is not None:   # every rank fills the rows of its own slices
        t = torch.from_numpy(rows).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        rows = t.cpu().numpy()
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "x.npy"), rows[:, :2 * C_CH].reshape(-1, C_CH, 2))
        np.save(os.path.join(path, "qmap.npy"), rows[:, 2 * C_CH:2 * C_CH + 2])
        np.save(os.path.join(path, "pd.npy"), rows[:, 2 * C_CH + 2:])
        sys.stderr.write(f"[bench] outputs of the last timed step ({pick.size} of {total} pixels) written to {path}\n")


def run_extras(args, q, ctx, net, F, d, dct, Yp, X0p, timed, log, rank, world, dist, stream, peaks):
    """Short legs for the other BASELINE configs (reported beside the headline, never part of `value`)."""
    import torch
    import benchdata
    lib = ctx.lib
    vp = C.c_void_p
    out = {}
    iters = args.iters
    S_have = X0p.shape[3]
    # configs[1]: one slice, spiral (latency-bound: 64 dependent layers per iteration) - rank 0 only
    if rank == 0:
        y1 = np.asfortranarray(Yp[:, :1])
        x1 = np.asfortranarray(X0p[..., :1])
        prm = {"iter": iters, "gamma": RHO, "F": F, "X0": x1, "net": net, "denoiser_type": "single_level"}
        s1 = q.AdmmSession(prm, 1)
        s1.upload_raw(y1, x1)
        ms1, _ = timed(lambda: s1.run(iters), 3, 2, collective=False, label="single slice")
        out["single_slice"] = {"config": f"BASELINE configs[1]: one slice, {args.mask}, {iters} iterations", "ms_per_reconstruction": ms1 / 3,
                               "slice_iterations_per_s": iters * 3 / (ms1 * 1e-3)}
        s1.close()
    # configs[2]: 15-slice batch on the EPI mask (per-GPU shape of the 120-slice job at 8 GPUs) - rank 0 only
    if rank == 0 and S_have >= 1:
        n15 = min(15, S_have)
        Pe = q.setup_subsampling_epi(N_IMG, N_IMG, EPI_PCT, np.eye(C_CH), ctx=ctx)
        Fe = q.fft_operator(Pe)
        xe = np.real(np.asfortranarray(X0p[..., :n15]))
        ye = q.awgn(Fe.forward(xe), SNR_DB, "measured", seed=7, ctx=ctx)
        x0e = Fe.adjoint(ye)
        se = q.AdmmSession({"iter": iters, "gamma": RHO, "F": Fe, "X0": x0e, "net": net, "denoiser_type": "single_level"}, n15)
        se.upload(ye, x0e)
        mse, _ = timed(lambda: se.run(iters), 2, 1, collective=False, label=f"EPI x{n15}")
        out["epi_15"] = {"config": f"BASELINE configs[2]: {n15}-slice batch, EPI 1/65 ({Pe.nmeas} meas/slice), {iters} iterations, one GPU's shard",
                         "ms_per_reconstruction": mse / 2, "slice_iterations_per_s": n15 * iters * 2 / (mse * 1e-3)}
        se.close()
        Pe.close()
    # configs[4]: 1M-atom dictionary, atom-sharded over the ranks; NCCL max-reduction of the packed (score, index) keys and a sum
    # all-reduce of the owner-computed outputs.  Every rank renders and uploads ONLY its shard of atoms.
    if args.big_atoms > 0:
        lutK = benchdata.dictionary_grid(args.big_atoms).shape[0]
        a0, a1 = q.atom_shard(lutK, world, rank)
        big = benchdata.make_dictionary(K_target=args.big_atoms, cut=args.cut, seed=0, atoms=(a0, a1))
        big["normD"] = np.nan_to_num(big["normD"], nan=1.0)
        if dist is not None:  # normD of the other shards: one all-gather-free trick - every rank fills its range, sum-reduce
            nd = torch.zeros(lutK, dtype=torch.float32, device="cuda")
            nd[a0:a1] = torch.from_numpy(big["normD"][a0:a1]).cuda()
            dist.all_reduce(nd, op=dist.ReduceOp.SUM)
            big["normD"] = nd.cpu().numpy()
        db = q.Dictionary(big, ctx=ctx, shard=(a0, a1), shard_only=True)
        npix = HW
        g = torch.Generator(device="cuda")
        g.manual_seed(5)  # same pixels on every rank
        xr = torch.randn(C_CH * npix, device="cuda", generator=g)
        xi = torch.randn(C_CH * npix, device="cuda", generator=g)

        def big_match():
            q.mrf_dtm_sharded(db, xr, xi, npix, shared_stream=True)
        msb, _ = timed(big_match, 3, 2, label="1M-atom sharded matching")
        out["match_1M"] = {"config": f"BASELINE configs[4]: one slice against {lutK} atoms, atom-sharded x{world}"
                                     + (", NCCL max all-reduce of packed (score, index) keys (8 B/px) + sum all-reduce of owner-computed outputs (32 B/px)" if world > 1 else ""),
                           "ms_per_slice": msb / 3, "px_atoms_per_s": npix * lutK * 3 / (msb * 1e-3), "atoms_per_rank": a1 - a0,
                           "collective": "ncclAllReduce(max, int64 keys) + ncclAllReduce(sum, fp32 outputs)" if world > 1 else None}
        db.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--slices", type=int, default=120, help="slices of the whole job (sharded over the ranks); 120 = 8 volunteers x 15")
    ap.add_argument("--iters", type=int, default=100, help="ADMM iterations per reconstruction (param.iter)")
    ap.add_argument("--mask", default="spiral", choices=["spiral", "epi"])
    ap.add_argument("--cut", type=int, default=3, choices=[0, 1, 2, 3, 4])
    ap.add_argument("--atoms", type=int, default=100000, help="dictionary size of the job's matching step")
    ap.add_argument("--big-atoms", type=int, default=1048576, help="dictionary size of the atom-sharded configs[4] leg (0 = skip)")
    ap.add_argument("--precision", default="tc", choices=["tc", "fp32"], help="denoiser precision mode: tc (tcgen05 split-bf16, default) / fp32 (CUDA cores)")
    ap.add_argument("--cpu-iters", type=int, default=8)
    ap.add_argument("--ref-iters", type=int, default=3)
    ap.add_argument("--ref-match-px", type=int, default=2048)
    ap.add_argument("--ref-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--clock-period", type=float, default=2.0)
    ap.add_argument("--k1-idle", type=float, default=4.0, help="idle seconds before the x-update-alone roofline leg (lets the power cap release)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write x, qmap and pd of the last timed step to DIR/<name>.npy (float32; "
                                                          f"a fixed, seeded sample of {DUMP_PIXELS} pixels when the job has more)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # launched by hand without torchrun: start one rank per GPU the way the driver does
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
