"""float32 training data against float64: kernel, step and end-to-end times of the accumulate paths, in one call.

    python tools/float32_inputs_bench.py [--out profiles/float32_inputs.json] [--reps 20]

Every arm reads the same seeded values (the float64 arm gets the float32 values cast up), the arms are alternated, times are
CUDA events (kernel / step) or a host clock around work ending in a synchronise (host path), medians over --reps.  The outputs
of the arms are asserted to agree as in tests/test_gpu_float32_inputs.py.  The card name and power limit (read-only
nvidia-smi query) and the HBM peak used for the shares (MEASURED_PEAKS.json, else a device copy measured here) are recorded."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from asvgp_b200 import basis as B, kernels as Kn, ops  # noqa: E402
from asvgp_b200.inducing_features import SplineFeatures1D  # noqa: E402

ARMS_1D = [("f64", "f64"), ("f64", "f32"), ("f32", "f32")]
DT = {"f64": torch.float64, "f32": torch.float32}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                       # recorded, not fatal: the numbers still carry torch's device name
        return {"name": torch.cuda.get_device_name(), "query_error": str(exc)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        pass
    a = torch.empty(1 << 28, dtype=torch.float64, device="cuda")     # 2 GiB, far larger than L2
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    ts = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    gbs = 2 * a.numel() * 8 / (np.median(ts) * 1e6)
    del a, b
    return gbs, "device copy measured in this call (read + write bytes / time)"


def timed(fn, reps, arms):
    """fn(arm) -> None, enqueues the work; alternates the arms; median CUDA-event ms per arm."""
    ts = {a: [] for a in arms}
    for a in arms:
        fn(a)
    torch.cuda.synchronize()
    for _ in range(reps):
        for a in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(a); e1.record(); torch.cuda.synchronize()
            ts[a].append(e0.elapsed_time(e1))
    return {a: {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))} for a, v in ts.items()}


def agree(outs, tol=1e-11):
    ref = outs[0].double()
    scale = float(ref.abs().max())
    for o in outs[1:]:
        err = float((o.double() - ref).abs().max())
        assert err <= tol * scale, "arms disagree: %g > %g" % (err, tol * scale)
    return True


def key(a):
    return "x_%s_y_%s" % a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "float32_inputs.json"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card()}
    peak, src = hbm_peak()
    res["hbm_peak_gbs"], res["hbm_peak_source"] = peak, src
    g = torch.Generator(device="cuda").manual_seed(1997)

    # ---- 1-D accumulate, N = 1e8 sorted, M = 1e4, k = 3 -------------------------------------------------------------
    n, m = 100_000_000, 10_000
    basis = B.B3Spline(-1, m + 1, m)
    x32 = torch.sort(torch.rand(n, device="cuda", generator=g) * m)[0]
    y32 = torch.sin(x32 / 37.0) + 0.3 * torch.randn(n, device="cuda", generator=g)
    data = {"f32": (x32, y32), "f64": (x32.double(), y32.double())}
    acc = {a: torch.zeros(ops.accum_size_1d(basis), dtype=torch.float64, device="cuda") for a in ARMS_1D}

    def run_acc(a):
        acc[a].zero_()
        ops.accum_1d(data[a[0]][0], data[a[1]][1], basis, acc=acc[a])

    t = timed(run_acc, args.reps, ARMS_1D)
    agree([acc[a] for a in ARMS_1D])
    one = {}
    for a in ARMS_1D:
        bpp = DT[a[0]].itemsize + DT[a[1]].itemsize
        ms = t[a]["median_ms"]
        one[key(a)] = dict(t[a], bytes_per_point=bpp, achieved_gbs=n * bpp / (ms * 1e6),
                           share_of_hbm_peak=n * bpp / (ms * 1e6) / peak, points_per_s=n / (ms * 1e-3))
    res["accum_1d_sorted_1e8"] = dict(n=n, m=m, order=3, arms=one)

    # ---- the bench-shaped step: Kuu assembly + chain on the side stream, accumulate, P chains and bound ---------------
    kern = Kn.Matern32(variance=1.0, lengthscales=1.0)
    feats = SplineFeatures1D(kern, basis)
    out = {a: torch.empty(16, dtype=torch.float64, device="cuda") for a in ARMS_1D}

    def run_step(a):
        acc[a].zero_()
        Kuu, dKuu = feats.make_Kuu_device(kern, want_grad=True)
        kuu = ops.kuu_chain_1d(Kuu, dKuu, basis, gate=True)
        ops.accum_1d(data[a[0]][0], data[a[1]][1], basis, acc=acc[a])
        ops.elbo_grad_1d(Kuu, dKuu, acc[a], basis, 1.0, 0.1, out=out[a], kuu=kuu)

    t = timed(run_step, args.reps, ARMS_1D)
    agree([out[a][:4] for a in ARMS_1D], tol=1e-9)
    res["step_1d_sorted_1e8"] = {key(a): t[a] for a in ARMS_1D}

    # ---- end to end from pinned host arrays ------------------------------------------------------------------------------
    host = {"f32": (x32.cpu().pin_memory(), y32.cpu().pin_memory())}
    host["f64"] = (host["f32"][0].double().pin_memory(), host["f32"][1].double().pin_memory())
    del data
    torch.cuda.empty_cache()
    e2e = {a: [] for a in ARMS_1D}
    for r in range(1 + max(3, args.reps // 4)):
        for a in ARMS_1D:
            acc[a].zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ops.accum_1d_host(host[a[0]][0], host[a[1]][1], basis, acc=acc[a])
            torch.cuda.synchronize()
            if r:
                e2e[a].append((time.perf_counter() - t0) * 1e3)
    agree([acc[a] for a in ARMS_1D])
    res["host_pinned_1d_sorted_1e8"] = {key(a): {"median_ms": float(np.median(v)), "points_per_s": n / (np.median(v) * 1e-3),
                                                 "pcie_bytes_per_point": DT[a[0]].itemsize + DT[a[1]].itemsize}
                                        for a, v in e2e.items()}
    del host
    torch.cuda.empty_cache()

    # ---- shuffled 1-D, binned ------------------------------------------------------------------------------------------
    nb = 20_000_000
    xs32 = torch.rand(nb, device="cuda", generator=g) * m
    ys32 = torch.sin(xs32 / 37.0) + 0.25
    sdata = {"f32": (xs32, ys32), "f64": (xs32.double(), ys32.double())}
    arms2 = [("f64", "f64"), ("f32", "f32")]

    def run_binned(a):
        acc[a].zero_()
        ops.accum_1d(sdata[a[0]][0], sdata[a[1]][1], basis, acc=acc[a], binned=True)

    t = timed(run_binned, max(5, args.reps // 2), arms2)
    agree([acc[a] for a in arms2])
    res["accum_1d_binned_shuffled_2e7"] = {key(a): t[a] for a in arms2}
    del sdata, xs32, ys32
    torch.cuda.empty_cache()

    # ---- 2-D raster 1e8 points (10^4 x 10^4), 200 x 200 knots, k = 3; and shuffled binned -------------------------------
    n1 = n2 = 10_000
    bases = [B.B3Spline(-80, -25, 200), B.B3Spline(15, 55, 200)]
    g1 = torch.linspace(-79.9, -25.1, n1, device="cuda", dtype=torch.float32)
    g2 = torch.linspace(15.1, 54.9, n2, device="cuda", dtype=torch.float32)
    X32 = torch.stack(torch.meshgrid(g1, g2, indexing="ij"), -1).reshape(-1, 2).contiguous()
    Y32 = (torch.sin(X32[:, 0] / 4.0) * torch.cos(X32[:, 1] / 3.0)).contiguous()
    del g1, g2
    d2 = {"f32": (X32, Y32), "f64": (X32.double(), Y32.double())}
    acc2 = {a: torch.zeros(ops.accum_size_2d(bases), dtype=torch.float64, device="cuda") for a in arms2}
    cm = {a: ops.moment_table_2d(bases) for a in arms2}

    def run_2d(a, **kw):
        cm[a].zero_()
        scal = ops.split_accum_2d(acc2[a], bases)[2]
        scal.zero_()
        ops.accum_2d(d2[a[0]][0], d2[a[1]][1], bases, cm[a], scal, **kw)

    t = timed(run_2d, args.reps, arms2)
    sel = {key(a): int(cm[a][-1:].view(torch.int32)[0].item()) for a in arms2}
    agree([cm[a][:-1] for a in arms2])
    n2d = n1 * n2
    res["accum_2d_raster_1e8"] = {key(a): dict(t[a], probe_select=sel[key(a)],
                                               bytes_per_point=2 * DT[a[0]].itemsize + DT[a[1]].itemsize,
                                               achieved_gbs=n2d * (2 * DT[a[0]].itemsize + DT[a[1]].itemsize) / (t[a]["median_ms"] * 1e6))
                                  for a in arms2}
    perm = torch.randperm(n2d // 4, device="cuda", generator=g)
    d2 = {"f32": (X32[perm].contiguous(), Y32[perm].contiguous())}
    d2["f64"] = (d2["f32"][0].double(), d2["f32"][1].double())
    del X32, Y32, perm
    t = timed(lambda a: run_2d(a, binned=True), max(5, args.reps // 2), arms2)
    agree([cm[a][:-1] for a in arms2])
    res["accum_2d_binned_shuffled_2.5e7"] = {key(a): t[a] for a in arms2}

    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
