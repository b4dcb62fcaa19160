#!/usr/bin/env python
"""Benchmark of the ASVGP hot path on B200: ELBO + gradient datapoints/s at N = 1e8, M = 1e4 (BASELINE.json configs[2]).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload 1d|1d-random|...] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic points:
    accumulate (asvgp_accum_1d, O(N))  ->  [N>1: one NCCL all-reduce of the packed band]  ->  Kuu assembly +
    ELBO + 3 hyper-parameter gradients (asvgp_elbo_grad_1d, O(M k^2), replicated per rank).
`value` is whole-job datapoints/s with inputs resident in HBM; `e2e` is the same metric through the public API
(`GPR_1d((X, y), kernel, basis)` + `training_loss_and_gradients()`) with HOST buffers, host->device copies inside the
timed region.  Weak scaling: every rank owns N points.  `--impl reference` times the CPU port of the reference's own
algorithm (oracle/asvgp_oracle.py: the same SciPy sparse calls as reference gpr.py:39-44 + LAPACK band routines) on
all host cores over a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the source tree may be read-only; the benchmark writes nothing into it
# stdout carries exactly ONE JSON line: library chatter (NCCL's version banner, torchrun notices) goes to stderr instead
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()

WORKLOADS = {
    # name: (N per rank, M, spline order, kernel, sorted?)
    "1d": (100_000_000, 10_000, 3, "Matern52", True),
    "1d-m32": (100_000_000, 10_000, 3, "Matern32", True),
    "1d-random": (100_000_000, 10_000, 3, "Matern52", False),
    "1d-c2": (1_000_000, 1_000, 3, "Matern32", True),
}
WORKLOADS_2D = {
    # name: (raster n1 x n2 per rank, m per dimension, spline order)   — BASELINE.json configs[3] (eNATL60-shaped)
    "2d": (10_000, 10_000, 200, 3),
    "2d-k4": (10_000, 10_000, 100, 4),          # what experiments/eNATL60/eNATL60.py:84 itself uses (B4, m = 100)
    "2d-small": (2_000, 2_000, 60, 3),
}
HYPERS_2D = ((1.0, 5.0), (1.0, 4.0), 0.01)      # (v1, l1), (v2, l2), sigma^2: lengthscales ~ 18 knot spacings
BYTES_PER_POINT_ACCUM_2D = 24                   # X[n,2] and y read once (SURVEY §8(d))
HYPERS = (1.0, 1.0, 0.1)          # variance, lengthscale, sigma^2 (SURVEY §8(d) C2/C3)
BYTES_PER_POINT_ACCUM = 16         # x and y read once (SURVEY §8(d))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="1d", choices=sorted(WORKLOADS) + sorted(WORKLOADS_2D))
    ap.add_argument("--no-2d", action="store_true", help="skip the 2-D Kronecker summary appended to the 1-D line")
    ap.add_argument("--n", type=float, default=None, help="override points per rank (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float64), to compare two builds")
    return ap.parse_args()


def launch_count():
    """Kernels launched by libasvgp_sm100a so far in this process (the library counts every launch it makes)."""
    from asvgp_b200 import _lib

    return int(_lib.load().asvgp_launch_count())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Writes every tensor of `arrays` as dirname/<name>.npy in float64.  The inputs are seeded, so two builds run with
    the same arguments can be compared output for output."""
    import numpy as np

    host = {name: np.asarray(t.detach().cpu().numpy(), dtype=np.float64) for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of %d bytes exceed the dump limit" % total
    os.makedirs(dirname, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, in the background, during the timed region)
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clocks and throttle reasons of GPU `index` DURING the timed region: NVML (pynvml) every 2 ms when it
    is importable, else `nvidia-smi` as fast as it answers."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], threading.Event(), None
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        nv = self.nvml
        while not self.stop_flag.is_set():
            try:
                if nv is not None:
                    sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(
                        nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                    bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                            nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
                    self.samples.append([sm, self.max_sm] + ["Active" if r & b else "Not Active" for b in bits])
                    self.stop_flag.wait(float(os.environ.get("ASVGP_BENCH_CLOCK_PERIOD", "0.002")))
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.02)

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop_flag.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples (NVML and nvidia-smi unavailable)"]}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES)
                   if any(str(s[2 + i]).lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------------------------
# synthetic data (SURVEY §8(d)): x ~ U(0, M) on domain (-1, M+1) so delta ~ 1; smooth signal + noise, standardised
# ---------------------------------------------------------------------------------------------------------------------
def make_data(torch, n, m, rank, world, is_sorted, seed=1997):
    gen = torch.Generator(device="cuda").manual_seed(seed + rank)
    lo, hi = (m * rank / world, m * (rank + 1) / world) if is_sorted else (0.0, float(m))
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen) * (hi - lo) + lo
    x.clamp_(1e-9, m - 1e-9)
    if is_sorted:
        x = torch.sort(x).values
    y = torch.sin(x * (2 * 3.141592653589793 / 37.0)) + 0.5 * torch.sin(x * (2 * 3.141592653589793 / 3.1))
    y += 0.3 * torch.randn(n, dtype=torch.float64, device="cuda", generator=gen)
    y = (y - y.mean()) / y.std()
    return x, y


def cpu_sample(n, m, seed=1997):
    import numpy as np

    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(1e-9, m - 1e-9, n))
    y = np.sin(x * (2 * np.pi / 37.0)) + 0.5 * np.sin(x * (2 * np.pi / 3.1)) + 0.3 * rng.standard_normal(n)
    return x, (y - y.mean()) / y.std()


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's algorithm
# ---------------------------------------------------------------------------------------------------------------------
_CPU_SHARED = {}


def _cpu_chunk(span):
    from oracle import asvgp_oracle as O

    d = _CPU_SHARED          # inherited by fork: no pickling of the point arrays
    return O.precompute_1d(d["mesh"], d["delta"], d["k"], d["m"], d["x"][span[0]:span[1]], d["y"][span[0]:span[1]])


def cpu_step(pool, cores, mesh, delta, k, m, kind, tables, x, y):
    """One reference-style step on the CPU: S1 precompute (gpr.py:39-44) over `cores` processes, then the ELBO
    (gpr.py:49-89) and its three derivatives by central differences of the banded ELBO (the reference gets them from
    TF reverse mode, which costs about two more banded passes — 6 extra O(M) evaluations are the same order)."""
    import numpy as np

    from oracle import asvgp_oracle as O

    n = x.shape[0]
    if pool is None:
        parts = [O.precompute_1d(mesh, delta, k, m, x, y)]
    else:
        cuts = np.linspace(0, n, cores + 1).astype(np.int64)
        parts = pool.map(_cpu_chunk, [(int(a), int(b)) for a, b in zip(cuts, cuts[1:])])
    G = sum(p[0] for p in parts)
    b = sum(p[1] for p in parts)
    yy = sum(p[2] for p in parts)
    v, l, s2 = HYPERS

    def f(v, l, s2):
        return O.elbo_1d(O.make_Kuu(kind, l, v, tables), G, b, yy, n, v, s2)

    e = f(v, l, s2)
    h = 1e-5
    grad = [(f(v + h, l, s2) - f(v - h, l, s2)) / (2 * h), (f(v, l + h, s2) - f(v, l - h, s2)) / (2 * h),
            (f(v, l, s2 + h) - f(v, l, s2 - h)) / (2 * h)]
    return e, grad


def run_cpu(n_sample, m, k, kind, steps, warmup, cores):
    import multiprocessing as mp

    from oracle import asvgp_oracle as O

    mesh, delta = O.make_mesh(-1, m + 1, m, k)
    tables = O.static_bands(k, m, delta)
    x, y = cpu_sample(n_sample, m)
    _CPU_SHARED.update(mesh=mesh, delta=delta, k=k, m=m, x=x, y=y)
    pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
    try:
        for _ in range(warmup):
            cpu_step(pool, cores, mesh, delta, k, m, kind, tables, x, y)
        t0 = time.perf_counter()
        for _ in range(steps):
            cpu_step(pool, cores, mesh, delta, k, m, kind, tables, x, y)
        dt = (time.perf_counter() - t0) / steps
    finally:
        if pool is not None:
            pool.close()
    return n_sample / dt, dt


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    if args.workload in WORKLOADS_2D:
        n1, n2, m, k = WORKLOADS_2D[args.workload]
        value, dt, n_sample, t_acc, t_fac = run_cpu_2d(args.workload, max(1, min(args.steps, 3)), 0, cores)
        sample = ("O(N) precompute timed on the first %d raster points over %d processes (%.2f s) and extrapolated "
                  "linearly to N=%d, plus one LAPACK banded ELBO evaluation at full M (%.2f s); no gradients"
                  % (n_sample, cores, t_acc, n1 * n2, t_fac))
        emit(({
            "impl": "reference", "metric": "elbo_grad_datapoints_per_s", "value": value, "unit": "datapoints/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config_2d(args.workload, n1, n2, m, k),
            "cpu_baseline": {"value": value, "unit": "datapoints/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "datapoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return
    n, m, k, kind, is_sorted = WORKLOADS[args.workload]
    n_sample = int(min(n, 2_000_000 * cores))            # ~1 s of work per core per step
    value, dt = run_cpu(n_sample, m, k, kind, args.steps, max(args.warmup, 1), cores)
    sample = "first %d of the %d points per step, %d processes (SciPy sparsetools/LAPACK are single-threaded)" % (
        n_sample, n, cores)
    emit(({
        "impl": "reference", "metric": "elbo_grad_datapoints_per_s", "value": value, "unit": "datapoints/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, n, m, k, kind, is_sorted),
        "cpu_baseline": {"value": value, "unit": "datapoints/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "datapoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(name, n, m, k, kind, is_sorted):
    return {"workload": "1-D collapsed ELBO + (variance, lengthscale, sigma2) gradients, N=%d points per GPU, M=%d "
                        "B%d-spline features, %s, x %s" % (n, m, k, kind, "sorted ascending" if is_sorted else "in random order"),
            "name": name, "n_per_gpu": n, "m": m, "order": k, "kernel": kind, "hypers": list(HYPERS),
            "l2_policy": "inputs (16 B/pt x N = %.1f GB) are larger than the 126 MB L2" % (16 * n / 1e9)}



# ---------------------------------------------------------------------------------------------------------------------
# 2-D Kronecker workload (BASELINE.json configs[3]): eNATL60-shaped raster, x1 slow, flat X[N, 2]
# ---------------------------------------------------------------------------------------------------------------------
DOM_2D = ((-80, -25), (15, 55))            # basis domains (experiments/eNATL60/eNATL60.py:84)
INNER_2D = ((-75.0, -30.0), (20.0, 50.0))  # data extent (eNATL60.py:43-46)


def make_data_2d(torch, n1, n2, rank, world, seed=1997):
    lo = INNER_2D[0][0] + (INNER_2D[0][1] - INNER_2D[0][0]) * rank / world
    hi = INNER_2D[0][0] + (INNER_2D[0][1] - INNER_2D[0][0]) * (rank + 1) / world
    x1 = torch.linspace(lo, hi, n1 + 2, dtype=torch.float64, device="cuda")[1:-1]
    x2 = torch.linspace(INNER_2D[1][0], INNER_2D[1][1], n2, dtype=torch.float64, device="cuda")
    X = torch.stack([x1[:, None].expand(n1, n2), x2[None, :].expand(n1, n2)], -1).reshape(-1, 2).contiguous()
    gen = torch.Generator(device="cpu").manual_seed(seed)
    y = torch.zeros(n1 * n2, dtype=torch.float64, device="cuda")
    for _ in range(8):                                    # smooth field: 8 random 2-D sinusoids (SURVEY §8(d) C4)
        f1, f2, ph = (torch.rand(3, generator=gen, dtype=torch.float64) * torch.tensor([0.6, 0.8, 6.28])).tolist()
        y += torch.sin(X[:, 0] * f1 + X[:, 1] * f2 + ph)
    g2 = torch.Generator(device="cuda").manual_seed(seed + 17 + rank)
    y += 0.05 * torch.randn(n1 * n2, dtype=torch.float64, device="cuda", generator=g2)
    y = (y - 0.0) / 2.0
    return X, y


def workload_config_2d(name, n1, n2, m, k):
    n = n1 * n2
    return {"workload": "2-D Kronecker collapsed ELBO + (v1, l1, v2, l2, sigma2) gradients, N=%d raster points "
                        "(%d x %d, x1 slow) per GPU, M=%d x %d B%d-spline features, Matern32 x Matern32"
                        % (n, n1, n2, m, m, k),
            "name": name, "n_per_gpu": n, "m": [m, m], "order": k, "kernel": "Matern32xMatern32",
            "hypers": [list(HYPERS_2D[0]), list(HYPERS_2D[1]), HYPERS_2D[2]],
            "l2_policy": "inputs (24 B/pt x N = %.1f GB) are larger than the 126 MB L2; a 512 MB write flushes it before every "
                         "step (inside the timed region)" % (24 * n / 1e9),
            "input_layout": "the caller states the raster shape (GPR_kron(..., raster_shape=(n1, n2)) / asvgp_accum_2d_raster): "
                            "no on-device classification pass; every point is still verified against the statement"}


def run_2d(args, name, torch, dist, world, rank, steps, warmup, with_e2e=True, dump=None):
    """Times the 2-D path; returns the summary dict (rank 0) — used as the main line for --workload 2d* and as the
    `kron_2d` appendix of the default 1-D line.  dump: directory for the outputs of the last timed step (rank 0)."""
    import numpy as np

    from asvgp_b200 import basis as B, kernels as Kn, ops
    from asvgp_b200.gpr import GPR_kron
    from asvgp_b200.inducing_features import SplineFeatures1D

    n1, n2, m, k = WORKLOADS_2D[name]
    if args.n:
        n1 = n2 = int(round(float(args.n) ** 0.5))
    n = n1 * n2
    cls = getattr(B, "B%dSpline" % k)
    bases = [cls(DOM_2D[0][0], DOM_2D[0][1], m), cls(DOM_2D[1][0], DOM_2D[1][1], m)]
    kerns = [Kn.Matern32(variance=HYPERS_2D[0][0], lengthscales=HYPERS_2D[0][1]),
             Kn.Matern32(variance=HYPERS_2D[1][0], lengthscales=HYPERS_2D[1][1])]
    X, y = make_data_2d(torch, n1, n2, rank, world)

    # the model object without its constructor's accumulate pass: the timed step does that pass itself
    model = GPR_kron.__new__(GPR_kron)
    model.kernels, model.bases, model.order, model.d = kerns, bases, k, 2
    model.likelihood = Kn.Gaussian(HYPERS_2D[2])
    model.inducing_features = [SplineFeatures1D(kerns[i], bases[i]) for i in range(2)]
    model._acc = torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda")
    model._Gs, model._b, model._scal = ops.split_accum_2d(model._acc, bases)
    cellmom = ops.moment_table_2d(bases)
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    result = {}

    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float64, device="cuda")      # 512 MB > the 126 MB L2

    def step(timers=None):
        # every step ends with a host read of the bound, so the host is never ahead of the GPU here; the L2 flush (the
        # timing rules' "write a buffer larger than L2", ~80 us) also gives the host the time it needs to enqueue the
        # accumulate kernel behind it, so that the accumulate phase below times the kernel and not the launch latency
        model._acc.zero_(); cellmom.zero_()
        flush.fill_(0.0)
        if timers: timers[0].record()
        # the workload IS a raster (BASELINE.json configs[3]: "gridded points") and says so: no on-device classification pass
        ops.accum_2d(X, y, bases, cellmom, model._scal, raster_row_len=n2)
        if timers: timers[1].record()
        ops.expand_moments_2d(cellmom, bases, model._acc)
        if world > 1:
            dist.all_reduce(model._acc)
        if timers: timers[2].record()
        result["elbo"], result["grads"] = model.elbo_and_grad()        # factor + selected inverse + one D2H read
        if timers: timers[3].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        step()
    barrier()
    elbo0 = result["elbo"]
    grad0 = [float(result["grads"][id(p)]) for p in model.trainable_variables]
    assert np.isfinite(elbo0) and np.isfinite(grad0).all()

    # gradient sanity, outside the timed region: central difference of the bound itself in one hyper-parameter
    # (two extra factorisations).  r01's selected inverse returned 1e52-sized noise here and nothing noticed.
    lpar = kerns[0].lengthscales
    l0, h = HYPERS_2D[0][1], 1e-4 * HYPERS_2D[0][1]
    lpar.assign(l0 + h); e_plus = float(model.elbo())
    lpar.assign(l0 - h); e_minus = float(model.elbo())
    lpar.assign(l0)
    fd = (e_plus - e_minus) / (2 * h)
    grad_check = {"param": "lengthscale of dimension 1", "central_difference": fd, "analytic": grad0[1],
                  "rel_err": abs(fd - grad0[1]) / max(abs(fd), 1e-300)}
    assert grad_check["rel_err"] < 1e-5, "2-D gradient fails its finite-difference check: %r" % (grad_check,)

    phase_ev = [[ev() for _ in range(4)] for _ in range(steps)]
    t0, t1 = ev(), ev()
    with ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) as clocks:
        for _ in range(max(warmup, 3)):       # warm-up immediately before the timed steps (see the 1-D arm)
            step()
        barrier()
        clocks.samples.clear()
        launches0 = launch_count()
        t0.record()
        for i in range(steps):
            step(phase_ev[i])
        t1.record()
        barrier()
        launches = launch_count() - launches0
    if dump and rank == 0:
        dump_outputs(dump, {
            "elbo": torch.tensor([result["elbo"]], dtype=torch.float64),
            "grad": torch.tensor([float(result["grads"][id(p)]) for p in model.trainable_variables], dtype=torch.float64),
            "KufKfu_stencil": model._Gs, "Kuf_y": model._b, "tr_yTy_count": model._scal})
    total_ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = total_ms.item() / steps
    accum_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in phase_ev]))
    red_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in phase_ev]))
    fact_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in phase_ev]))
    assert abs(result["elbo"] - elbo0) <= 1e-12 * abs(elbo0), "2-D ELBO is not reproducible from step to step"

    e2e = None
    if with_e2e:
        Xh = torch.empty((n, 2), dtype=torch.float64).pin_memory(); Xh.copy_(X)
        yh = torch.empty(n, dtype=torch.float64).pin_memory(); yh.copy_(y)

        def e2e_step():
            mdl = GPR_kron((Xh, yh.view(-1, 1)), kerns, bases, check_inputs=False, raster_shape=(n1, n2))
            mdl.likelihood.variance.assign(HYPERS_2D[2])
            return mdl.training_loss_and_gradients()

        e2e_step()
        barrier()
        k_e2e = max(2, min(steps, 5))
        w0 = time.perf_counter()
        for _ in range(k_e2e):
            loss, _g = e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - w0) / k_e2e], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        assert abs(-loss - elbo0) <= 1e-9 * abs(elbo0), "e2e ELBO differs from the device-resident one"
        e2e = {"value": world * n / dt.item(), "unit": "datapoints/s", "h2d_bytes_per_step": 24 * n,
               "d2h_bytes_per_step": 24 * 8, "ms_per_step": dt.item() * 1e3, "steps": k_e2e,
               "host_buffers": "pinned",
               "api": "GPR_kron((X_host, y_host), kernels, bases).training_loss_and_gradients()"}
        if world == 1:
            # the same call with ordinary (pageable) numpy arrays: the library stages them through its own pinned buffers
            Xn, yn = Xh.numpy().copy(), yh.numpy().copy()
            del Xh, yh

            def e2e_np():
                mdl = GPR_kron((Xn, yn.reshape(-1, 1)), kerns, bases, check_inputs=False, raster_shape=(n1, n2))
                mdl.likelihood.variance.assign(HYPERS_2D[2])
                return mdl.training_loss_and_gradients()

            e2e_np()
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            for _ in range(2):
                e2e_np()
            torch.cuda.synchronize()
            dtp = (time.perf_counter() - w0) / 2
            e2e["pageable"] = {"value": n / dtp, "ms_per_step": dtp * 1e3, "host_buffers": "pageable numpy arrays"}
            del Xn, yn
        else:
            del Xh, yh

    # predictor on the same raster (BASELINE.json configs[4]): sharded over ranks, no collective
    # (the posterior — factorisation, selected inverse, per-cell polynomial table — is computed once per model; every batch
    # of test points then streams through the table, as the reference's 10 000-point prediction chunks reuse its factors)
    alpha, SigP, S1, S2, _info = model.posterior_weights()
    prior = HYPERS_2D[0][0] * HYPERS_2D[1][0]
    table = ops.predict_2d_prepare(bases, alpha, SigP, S1, S2)
    pm, pv = torch.empty(n, dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    q0, q1 = ev(), ev()
    q0.record()
    for _ in range(3):
        ops.predict_2d_prepare(bases, alpha, SigP, S1, S2, work=table)
    q1.record()
    for _ in range(2):
        ops.predict_2d_apply(X, bases, table, prior, raster_row_len=n2, mean=pm, var=pv)
    p0, p1 = ev(), ev()
    barrier()
    prep_ms = q0.elapsed_time(q1) / 3
    p0.record()
    for _ in range(3):
        ops.predict_2d_apply(X, bases, table, prior, raster_row_len=n2, mean=pm, var=pv)
    p1.record()
    barrier()
    del pm, pv
    pred_ms = torch.tensor([p0.elapsed_time(p1) / 3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(pred_ms, op=dist.ReduceOp.MAX)
    pred_ms = pred_ms.item()

    peaks, peak_kind = measured_peaks()
    achieved = BYTES_PER_POINT_ACCUM_2D * n / (accum_ms * 1e-3) / 1e9
    M, w = m * m, k * (m + 1)
    flops = float(M) * w * w                       # Cholesky of the band; the selected inverse is ~2x that again
    n_blk = -(-M // 64)
    return {
        "metric": "elbo_grad_datapoints_per_s", "value": world * n / (ms_per_step * 1e-3), "unit": "datapoints/s",
        "n_gpus": world, "steps": steps, "warmup": max(warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config_2d(name, n1, n2, m, k),
        "phases_ms": {"accumulate": accum_ms, "expand_allreduce": red_ms, "factor_selinv_grad": fact_ms,
                      "predict_same_raster": pred_ms, "predict_table_once_per_model": prep_ms},
        "predict_points_per_s": world * n / (pred_ms * 1e-3),
        "elbo": elbo0, "grad": grad0, "grad_check": grad_check, "parity_checked": True,
        "roofline": {"kernel": "accum_2d_cols_kernel<%d> (separable raster, chosen by the device-side probe of asvgp_accum_2d)" % k,
                     "bound": "hbm", "achieved": achieved,
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                     "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == "measured" else "fallback",
                     "algorithmic_bytes_per_launch": BYTES_PER_POINT_ACCUM_2D * n, "launch_ms": accum_ms,
                     "traffic": _traffic("accum_2d")},
        "fp64_phase": {"what": "block-band Cholesky of P (bandwidth %d) + selected inverse + contractions" % w,
                       "cholesky_flop": flops, "ms": fact_ms,
                       "note": "latency-bound chain of %d block columns; flop rate vs the ~37 TF/s fp64 pipe is "
                               "reported for orientation only" % n_blk,
                       "cholesky_equiv_tflops": 3 * flops / (fact_ms * 1e-3) / 1e12},
        "clocks": clocks.summary(),
        # counted by the library itself (asvgp_launch_count) over the timed region
        "gpu_launches": launches,
        "e2e": e2e,
    }


def _traffic(kernel):
    tpath = os.path.join(ROOT, "profiles", "%s_traffic.json" % kernel)
    if os.path.exists(tpath):
        return json.load(open(tpath)).get("dram_bytes_per_launch")
    return None


def run_cpu_2d(name, steps, warmup, cores):
    """CPU arm of the 2-D workload: the port's O(N) precompute (same SciPy sparse calls as reference gpr.py:268-271)
    on a bounded sample over `cores` processes + ONE banded ELBO evaluation at full M (LAPACK dpbtrf; the reference's
    dense tf.linalg.cholesky of the M x M matrix is infeasible at 200 x 200).  Gradients are NOT included, which
    favours this arm."""
    import multiprocessing as mp

    import numpy as np

    from oracle import asvgp_oracle as O

    n1, n2, m, k = WORKLOADS_2D[name]
    n = n1 * n2
    meshes, deltas = zip(*[O.make_mesh(DOM_2D[i][0], DOM_2D[i][1], m, k) for i in range(2)])
    n_sample = int(min(n, 400_000 * cores))
    rows = max(1, n_sample // n2)
    x1 = np.linspace(INNER_2D[0][0], INNER_2D[0][1], n1 + 2)[1:-1][:rows]
    x2 = np.linspace(INNER_2D[1][0], INNER_2D[1][1], n2)
    X = np.stack(np.meshgrid(x1, x2, indexing="ij"), -1).reshape(-1, 2)
    rng = np.random.default_rng(0)
    y = np.sin(X[:, 0] / 4) * np.cos(X[:, 1] / 3) + 0.05 * rng.standard_normal(X.shape[0])
    n_sample = X.shape[0]
    _CPU_SHARED.update(meshes=meshes, deltas=deltas, k=k, ms=[m, m], X=X, y=y)
    T = [O.static_bands(k, m, d) for d in deltas]
    Ks = [O.make_Kuu("Matern32", HYPERS_2D[i][1], HYPERS_2D[i][0], T[i]) for i in range(2)]
    pool = mp.get_context("fork").Pool(cores) if cores > 1 else None
    cuts = np.linspace(0, n_sample, cores + 1).astype(np.int64)
    spans = [(int(a), int(b)) for a, b in zip(cuts, cuts[1:])]

    def one():
        t0 = time.perf_counter()
        parts = pool.map(_cpu_chunk_2d, spans) if pool else [_cpu_chunk_2d(spans[0])]
        G = sum(p[0] for p in parts); b = sum(p[1] for p in parts); yy = sum(p[2] for p in parts)
        t1 = time.perf_counter()
        # regularise the sample's Gram as the full data set would (every cell populated): scale to N
        e = O.elbo_kron_banded(Ks, G * (n / n_sample), b * (n / n_sample), yy * (n / n_sample), n,
                               [HYPERS_2D[0][0], HYPERS_2D[1][0]], HYPERS_2D[2], k, [m, m])
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1, e

    try:
        for _ in range(warmup):
            one()
        ta, tf = [], []
        for _ in range(steps):
            a, f, _e = one()
            ta.append(a); tf.append(f)
    finally:
        if pool is not None:
            pool.close()
    t_acc, t_fac = float(np.mean(ta)), float(np.mean(tf))
    full_step = n / (n_sample / t_acc) + t_fac
    return n / full_step, full_step, n_sample, t_acc, t_fac


def _cpu_chunk_2d(span):
    from oracle import asvgp_oracle as O

    d = _CPU_SHARED
    return O.precompute_kron(d["meshes"], d["deltas"], d["k"], d["ms"], d["X"][span[0]:span[1]], d["y"][span[0]:span[1]])

# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
def run_unordered(torch):
    """Accumulate times for the secondary orderings of SURVEY 8(d): C3-ii (1-D, x in random order) and C4 shuffled,
    through the bucket-partition entry points (partition passes included), next to the streaming kernels on the same data."""
    from asvgp_b200 import basis as B, ops

    def timeit(fn, reps):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    out = {}
    n, m, k = WORKLOADS["1d"][:3]
    g = torch.Generator(device="cuda"); g.manual_seed(1997)
    basis = getattr(B, "B%dSpline" % k)(-1, m + 1, m)
    x = torch.rand(n, dtype=torch.float64, device="cuda", generator=g) * m
    y = torch.sin(x / 37)
    acc = torch.zeros(ops.accum_size_1d(basis), dtype=torch.float64, device="cuda")
    out["accum_1d_random_order_ms"] = {"binned": timeit(lambda: ops.accum_1d(x, y, basis, acc, binned=True), 5),
                                       "streaming": timeit(lambda: ops.accum_1d(x, y, basis, acc), 2), "points": n}
    del x, y
    n1, n2, m2, k2 = WORKLOADS_2D["2d"]
    cls = getattr(B, "B%dSpline" % k2)
    bases = [cls(-80, -25, m2), cls(15, 55, m2)]
    x1 = torch.linspace(-75, -30, n1, dtype=torch.float64, device="cuda")
    x2 = torch.linspace(20, 50, n2, dtype=torch.float64, device="cuda")
    X = torch.stack([x1[:, None].expand(n1, n2), x2[None, :].expand(n1, n2)], -1).reshape(-1, 2)
    X = X[torch.randperm(n1 * n2, device="cuda", generator=g)].contiguous()
    yy = torch.sin(X[:, 0] / 4) * torch.cos(X[:, 1] / 3)
    acc2 = torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda")
    cm = ops.moment_table_2d(bases)
    scal = ops.split_accum_2d(acc2, bases)[2]
    out["accum_2d_shuffled_ms"] = {"binned": timeit(lambda: ops.accum_2d(X, yy, bases, cm, scal, binned=True), 3),
                                   "streaming": timeit(lambda: ops.accum_2d(X, yy, bases, cm, scal), 1), "points": n1 * n2}
    del X, yy
    torch.cuda.empty_cache()
    return out


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from asvgp_b200 import basis as B, kernels as Kn, ops
    from asvgp_b200.gpr import GPR_1d

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.workload in WORKLOADS_2D:
        line = run_2d(args, args.workload, torch, dist, world, rank, args.steps, args.warmup, with_e2e=not args.no_e2e,
                      dump=args.dump_outputs)
        if rank == 0:
            if world == 1 and not args.no_cpu_baseline:
                v, dt, n_sample, t_acc, t_fac = run_cpu_2d(args.workload, 1, 0, 1)
                line["cpu_baseline"] = {
                    "value": v, "unit": "datapoints/s", "cores": 1, "kind": "port",
                    "sample": "precompute on the first %d raster points (%.1f s, extrapolated linearly to N) + one "
                              "LAPACK banded ELBO at full M (%.1f s), no gradients, single thread" % (n_sample, t_acc, t_fac)}
            emit(line)
        if world > 1:
            dist.destroy_process_group()
        return
    n, m, k, kind, is_sorted = WORKLOADS[args.workload]
    if args.n:
        n = int(args.n)
    basis = getattr(B, "B%dSpline" % k)(-1, m + 1, m)
    kern = getattr(Kn, kind)(variance=HYPERS[0], lengthscales=HYPERS[1])
    x, y = make_data(torch, n, m, rank, world, is_sorted)

    from asvgp_b200.inducing_features import SplineFeatures1D

    feats = SplineFeatures1D(kern, basis)
    acc = torch.zeros(ops.accum_size_1d(basis), dtype=torch.float64, device="cuda")
    out = torch.empty(16, dtype=torch.float64, device="cuda")
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731

    binned = not is_sorted            # random order: bucket-partition path, the binning passes are inside the timed accumulate

    # the one collective of the step: a one-shot all-reduce over NVLink peer memory (asvgp_allreduce_oneshot, the ranks
    # accumulate straight into symmetric buffers); NCCL all_reduce when symmetric memory is unavailable
    red = None
    if world > 1 and os.environ.get("ASVGP_NCCL_ALLREDUCE") is None:
        from asvgp_b200 import dist as adist

        red = adist.oneshot_reducer(acc.numel())

    KUU_GATE = os.environ.get("ASVGP_BENCH_KUU_GATE", "1") != "0"

    def step(timers=None, xs=None, ys=None):
        # The Kuu chain (log|Kuu|, band(Kuu^-1), tangents: hyper-parameters only) goes to a side stream FIRST, so that the
        # O(N) accumulate hides it; the P chains + bound follow the accumulate and its all-reduce (ops.kuu_chain_1d).
        tgt = red.buffer() if red is not None else acc
        tgt.zero_()
        if timers: timers[0].record()
        Kuu, dKuu = feats.make_Kuu_device(kern, want_grad=True)
        kuu = ops.kuu_chain_1d(Kuu, dKuu, basis, gate=KUU_GATE, timing=timers is not None)
        if timers: timers[1].record(); timers.append(kuu.event)
        ops.accum_1d(x if xs is None else xs, y if ys is None else ys, basis, acc=tgt, binned=binned)
        if timers: timers[2].record()
        if red is not None:
            red.reduce(acc)
        elif world > 1:
            dist.all_reduce(acc)
        if timers: timers[3].record()
        ops.elbo_grad_1d(Kuu, dKuu, acc, basis, HYPERS[0], HYPERS[2], out=out, kuu=kuu)
        if timers: timers[4].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    res0 = out.cpu().numpy().copy()
    assert res0[8] == 0 and np.isfinite(res0[:4]).all(), "ELBO evaluation failed: %r" % (res0,)
    # gradient sanity, outside the timed region: central difference of the bound itself in the lengthscale
    outp, outm = torch.empty_like(out), torch.empty_like(out)
    h = 1e-4 * HYPERS[1]
    for sign, o in ((1.0, outp), (-1.0, outm)):
        kern.lengthscales.assign(HYPERS[1] + sign * h)
        Kuu, dKuu = feats.make_Kuu_device(kern, want_grad=True)
        ops.elbo_grad_1d(Kuu, dKuu, acc, basis, HYPERS[0], HYPERS[2], out=o)
    kern.lengthscales.assign(HYPERS[1])
    fd = (outp[0].item() - outm[0].item()) / (2 * h)
    grad_check = {"param": "lengthscale", "central_difference": fd, "analytic": float(res0[2]),
                  "rel_err": abs(fd - res0[2]) / max(abs(fd), 1e-300)}
    assert grad_check["rel_err"] < 1e-5, "1-D gradient fails its finite-difference check: %r" % (grad_check,)

    # ---- timed region: exactly K steps, CUDA events, max over ranks ------------------------------------------------
    phase_ev = [[ev() for _ in range(5)] for _ in range(args.steps)]
    t0, t1 = ev(), ev()
    with ClockSampler(local) as clocks:
        # the W warm-up steps run IMMEDIATELY before the timed ones (the steps further up only produced the result that the gradient
        # check above compares with): the checks and the sampler's NVML start-up leave the device idle for tens of milliseconds, and
        # the first ~20 steps after such a pause run 4 % slower (the driver times K = 20)
        for _ in range(max(args.warmup, 3)):
            step()
        barrier()
        clocks.samples.clear()               # clock samples of the timed region only
        launches0 = launch_count()
        t0.record()
        h0 = time.perf_counter()
        for i in range(args.steps):
            step(phase_ev[i])
        t1.record()
        host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / args.steps      # must stay below ms_per_step, else the host is the bound
        barrier()
        launches = launch_count() - launches0
    if args.dump_outputs and rank == 0:
        # out[9:15] holds clock counters, not results; acc holds the all-reduced statistics the bound was evaluated on
        G_band, Kuf_y, scal = ops.split_accum_1d(acc, basis)
        dump_outputs(args.dump_outputs, {"elbo": out[0:1], "grad": out[1:4], "bound_terms": torch.cat([out[4:9], out[15:16]]),
                                         "KufKfu_band": G_band, "Kuf_y": Kuf_y, "tr_yTy_count": scal})
    total_ms = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device="cuda")
    kuu_asm_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in phase_ev]))
    accum_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in phase_ev]))
    allred_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in phase_ev]))
    elbo_ms = float(np.mean([e[3].elapsed_time(e[4]) for e in phase_ev]))
    kuu_done_ms = float(np.mean([e[1].elapsed_time(e[5]) for e in phase_ev]))     # side stream: Kuu chain complete, after the accumulate's start
    # the pieces the accumulate hides, and the latency of a bound evaluation on its own (what one optimiser iteration costs
    # once G is accumulated: example.py:31-32), each timed alone outside the timed region
    Kuu_, dKuu_ = feats.make_Kuu_device(kern, want_grad=True)
    a0, a1, a2 = ev(), ev(), ev()
    reps = 20
    torch.cuda.synchronize()
    a0.record()
    for _ in range(reps):
        h_ = ops.kuu_chain_1d(Kuu_, dKuu_, basis)
        torch.cuda.current_stream().wait_event(h_.event)
    a1.record()
    for _ in range(reps):
        ops.elbo_grad_1d(Kuu_, dKuu_, acc, basis, HYPERS[0], HYPERS[2], out=outp)
    a2.record()
    torch.cuda.synchronize()
    kuu_chain_alone_ms, elbo_call_alone_ms = a0.elapsed_time(a1) / reps, a1.elapsed_time(a2) / reps
    # the accumulate kernel with nothing beside it (in the step the Kuu chain's cluster holds 8 SMs and reads its tables next to it)
    scratch_acc = torch.zeros_like(acc)
    b0, b1 = ev(), ev()
    ops.accum_1d(x, y, basis, acc=scratch_acc, binned=binned)
    torch.cuda.synchronize()
    b0.record()
    for _ in range(10):
        ops.accum_1d(x, y, basis, acc=scratch_acc, binned=binned)
    b1.record()
    torch.cuda.synchronize()
    accum_alone_ms = b0.elapsed_time(b1) / 10
    del scratch_acc
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = total_ms.item() / args.steps
    value = world * n / (ms_per_step * 1e-3)

    # ---- strong scaling (SURVEY 8(e) "report both"): the SAME global N split over the ranks ---------------------------------
    strong = None
    if world > 1:
        n_s = n // world
        xs_, ys_ = x[:n_s], y[:n_s]
        sev = [[ev() for _ in range(5)] for _ in range(args.steps)]

        def strong_step(t):
            step(t, xs_, ys_)

        for _ in range(3):
            strong_step(sev[0])
        s0, s1 = ev(), ev()
        barrier()
        s0.record()
        for i in range(args.steps):
            strong_step(sev[i])
        s1.record()
        barrier()
        sms = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(sms, op=dist.ReduceOp.MAX)
        sms = sms.item() / args.steps
        strong = {"scaling": "strong", "n_global": n_s * world, "n_per_gpu": n_s, "ms_per_step": sms,
                  "value": n_s * world / (sms * 1e-3), "unit": "datapoints/s",
                  "phases_ms": {"kuu_assemble_and_fork": float(np.mean([e[0].elapsed_time(e[1]) for e in sev])),
                                "accumulate": float(np.mean([e[1].elapsed_time(e[2]) for e in sev])),
                                "allreduce": float(np.mean([e[2].elapsed_time(e[3]) for e in sev])),
                                "join_p_chains_bound": float(np.mean([e[3].elapsed_time(e[4]) for e in sev]))},
                  "note": "global N fixed at the 1-GPU workload's N; only the accumulate phase shrinks with the number of "
                          "ranks, the banded chains are replicated (the Kuu chain hidden behind accumulate + all-reduce as "
                          "far as they last)"}
        step()          # leave `acc` / `out` as the weak-scaling step left them (the predictor below reuses acc)
        barrier()

    # ---- end to end through the public API with host buffers ---------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        xh = torch.empty(n, dtype=torch.float64).pin_memory(); xh.copy_(x)
        yh = torch.empty(n, dtype=torch.float64).pin_memory(); yh.copy_(y)

        def e2e_step():
            model = GPR_1d((xh.view(-1, 1), yh.view(-1, 1)), kern, basis, check_inputs=False)
            model.likelihood.variance.assign(HYPERS[2])
            return model.training_loss_and_gradients()        # reads loss + gradient back to the host

        for _ in range(2):
            e2e_step()
        barrier()
        k_e2e = max(3, min(args.steps, 10))
        w0 = time.perf_counter()
        for _ in range(k_e2e):
            loss, grad = e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - w0) / k_e2e], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        assert abs(-loss - res0[0]) <= 1e-9 * abs(res0[0]), "e2e ELBO differs from the device-resident one"
        e2e = {"value": world * n / dt.item(), "unit": "datapoints/s", "h2d_bytes_per_step": 16 * n,
               "d2h_bytes_per_step": 16 * 8, "ms_per_step": dt.item() * 1e3, "steps": k_e2e,
               "host_buffers": "pinned", "pcie_gb_per_s_per_rank": 16 * n / dt.item() / 1e9,
               # all ranks read pinned host memory at once: the aggregate is what the box's host DRAM / PCIe root complexes give
               "aggregate_h2d_gb_per_s": world * 16 * n / dt.item() / 1e9,
               "host": {"cpus_visible": len(os.sched_getaffinity(0)),
                        "numa_nodes": len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
                        if os.path.isdir("/sys/devices/system/node") else None},
               "api": "GPR_1d((X_host, y_host), kernel, basis).training_loss_and_gradients()"}
        if world == 1:
            # the same call with ordinary (pageable) numpy arrays: staged through the library's pinned buffers
            xn, yn = xh.numpy().copy(), yh.numpy().copy()
            del xh, yh

            def e2e_np():
                mdl = GPR_1d((xn.reshape(-1, 1), yn.reshape(-1, 1)), kern, basis, check_inputs=False)
                mdl.likelihood.variance.assign(HYPERS[2])
                return mdl.training_loss_and_gradients()

            e2e_np()
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            for _ in range(3):
                e2e_np()
            torch.cuda.synchronize()
            dtp = (time.perf_counter() - w0) / 3
            e2e["pageable"] = {"value": n / dtp, "ms_per_step": dtp * 1e3, "host_buffers": "pageable numpy arrays"}
            del xn, yn
        else:
            del xh, yh

    # 1-D predictor on the same points (sharded over ranks, no collective): posterior weights once, then mean/variance
    from asvgp_b200.gpr import GPR_1d as _G1

    pm = _G1.__new__(_G1)
    pm.kernel, pm.basis, pm.inducing_features, pm._acc, pm._accs, pm._chunks = kern, basis, feats, acc, [acc], 0
    pm.likelihood = Kn.Gaussian(HYPERS[2])
    alpha, S_band, _info = pm.posterior_weights()
    for _ in range(2):
        ops.predict_1d(x, basis, alpha, S_band, HYPERS[0])
    q0, q1 = ev(), ev()
    barrier()
    q0.record()
    for _ in range(5):
        ops.predict_1d(x, basis, alpha, S_band, HYPERS[0])
    q1.record()
    barrier()
    pred_ms = torch.tensor([q0.elapsed_time(q1) / 5], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(pred_ms, op=dist.ReduceOp.MAX)
    pred_ms = pred_ms.item()

    kron = None
    if args.workload == "1d" and not args.no_2d and not args.n:
        del x, y
        torch.cuda.empty_cache()
        try:
            kron = run_2d(args, "2d", torch, dist, world, rank, max(3, min(args.steps, 5)), 3, with_e2e=not args.no_e2e)
        except Exception as exc:            # the appendix must never take the headline line down with it
            kron = {"error": repr(exc)}
        if world == 1 and isinstance(kron, dict) and "error" not in kron:
            torch.cuda.empty_cache()
            try:        # the shape experiments/eNATL60/eNATL60.py:84 itself uses (B4 splines, m = 100 per dimension)
                k4 = run_2d(args, "2d-k4", torch, dist, world, rank, 3, 3, with_e2e=False)
                kron["enatl60_k4_m100"] = {key: k4[key] for key in ("ms_per_step", "value", "phases_ms", "elbo", "grad",
                                                                     "grad_check", "roofline", "config", "gpu_launches")}
            except Exception as exc:
                kron["enatl60_k4_m100"] = {"error": repr(exc)}

    unordered = None
    if args.workload == "1d" and world == 1 and not args.no_2d and not args.n:
        torch.cuda.empty_cache()
        try:
            unordered = run_unordered(torch)
        except Exception as exc:
            unordered = {"error": repr(exc)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_kind = measured_peaks()
    achieved = BYTES_PER_POINT_ACCUM * n / (accum_ms * 1e-3) / 1e9
    traffic = _traffic("accum_1d")
    line = {
        "metric": "elbo_grad_datapoints_per_s", "value": value, "unit": "datapoints/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, n, m, k, kind, is_sorted),
        "phases_ms": {"kuu_assemble_and_fork": kuu_asm_ms, "accumulate": accum_ms, "allreduce": allred_ms,
                      "join_p_chains_bound": elbo_ms, "predict_same_points": pred_ms,
                      "kuu_chain_done_after_accumulate_start": kuu_done_ms, "kuu_chain_alone_side_stream": kuu_chain_alone_ms, "bound_evaluation_alone": elbo_call_alone_ms},
        "host_enqueue_ms_per_step": host_enqueue_ms,
        "overlap": "the Kuu chain (log|Kuu|, band(Kuu^-1), lengthscale tangents: depends on the hyper-parameters only) runs on a "
                   "side stream while the accumulate streams the data; the two P chains and the bound follow the all-reduce",
        "predict_points_per_s": world * n / (pred_ms * 1e-3),
        "elbo": float(res0[0]), "grad": [float(v) for v in res0[1:4]], "grad_check": grad_check, "parity_checked": True,
        "roofline": {"kernel": ("accum_1d_kernel<%d,2>" % k) if not binned else
                     "asvgp_accum_1d_binned (part_hist + part_scan + part_scatter + accum_1d_units_kernel<%d>)" % k,
                     "bound": "hbm", "achieved": achieved,
                     "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                     "peak_source": peak_kind + " (MEASURED_PEAKS.json hbm_gbs)" if peak_kind == "measured" else "fallback",
                     "algorithmic_bytes_per_launch": BYTES_PER_POINT_ACCUM * n, "launch_ms": accum_ms, "traffic": traffic,
                     "launch_ms_alone": accum_alone_ms, "frac_alone": BYTES_PER_POINT_ACCUM * n / (accum_alone_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                     "note": "launch_ms / frac: inside the timed steps, where the Kuu chain runs beside the kernel on a side stream (a "
                             "cluster of 8 CTAs holds 8 SMs); *_alone: the same launch with nothing beside it"},
        "clocks": clocks.summary(),
        # counted by the library itself (asvgp_launch_count) over the timed region
        "gpu_launches": launches,
    }
    if strong is not None:
        line["strong_scaling"] = strong
    if world > 1:
        line["collective"] = ("asvgp_allreduce_oneshot: one kernel per rank over NVLink peer memory (symmetric buffers), sums in rank "
                              "order" if red is not None else "torch.distributed.all_reduce (NCCL)")
        if red is not None:
            red.check()
    if e2e is not None:
        line["e2e"] = e2e
    if kron is not None:
        line["kron_2d"] = kron
    if unordered is not None:
        line["unordered_inputs"] = unordered
    if world == 1 and not args.no_cpu_baseline:
        n_sample = min(n, 20_000_000)
        v1, dt1 = run_cpu(n_sample, m, k, kind, 1, 0, 1)
        line["cpu_baseline"] = {"value": v1, "unit": "datapoints/s", "cores": 1, "kind": "port",
                                "sample": "one step on the first %d sorted points of the workload (%.1f s), single "
                                          "thread like the reference's SciPy/LAPACK path" % (n_sample, dt1)}
    if world == 1 and not args.no_cpu_baseline and isinstance(kron, dict) and "error" not in kron:
        v2, dt2, n_sample2, t_acc2, t_fac2 = run_cpu_2d("2d", 1, 0, 1)
        kron["cpu_baseline"] = {
            "value": v2, "unit": "datapoints/s", "cores": 1, "kind": "port",
            "sample": "precompute on the first %d raster points (%.1f s, extrapolated linearly to N) + one LAPACK banded "
                      "ELBO at full M (%.1f s), no gradients, single thread" % (n_sample2, t_acc2, t_fac2)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
