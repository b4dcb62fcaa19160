"""Cost of multi-output targets in GPR_kron on one GPU: for D output columns on one 10^8-point raster, the per-step time of
elbo_and_grad (one factorisation + selected inverse with D right-hand sides + D x kron_terms; CUDA events) next to D separate
single-column models, the construction time and the predict_f time per 10^8 points.  With --parent-lib (the library of the
parent commit) the D = 1 step is also timed on that library, the two alternated in the same process.

    python tools/multi_output_bench.py [--out profiles/multi_output.json] [--parent-lib PATH] [--n 1e8] [--steps 20]

Writes one JSON with the GPU name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

WORKLOADS = {"2d": (200, 3), "2d-k4": (100, 4)}          # m per dimension, order
DOM = ((-80.0, -25.0), (15.0, 55.0))
HYP, S2 = [(1.0, 6.0), (0.8, 5.0)], 0.01


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                      # noqa: BLE001
        return {"error": repr(exc)}


def load_parent(path):
    """The parent commit's library as a second ctypes handle, with the signatures of the functions it exports."""
    import ctypes

    from asvgp_b200 import _lib

    lib = ctypes.CDLL(os.path.abspath(path))
    lib.asvgp_last_error.restype = ctypes.c_char_p
    lib.asvgp_last_error.argtypes = []
    table = {name: (ctypes.c_int, args) for name, args in _lib.SIGNATURES.items()}
    table.update(_lib.VALUE_FUNCTIONS)
    for name, (restype, argtypes) in table.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = restype, argtypes
    return lib


def main():
    import numpy as np
    import torch

    from asvgp_b200 import _lib, basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "multi_output.json"))
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--n", type=float, default=1e8)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--ds", default="1,4,16")
    ap.add_argument("--workloads", default="2d,2d-k4")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    new_lib = _lib.load()
    parent = load_parent(args.parent_lib) if args.parent_lib else None
    n1 = n2 = int(round(args.n ** 0.5))
    n = n1 * n2
    x1 = torch.linspace(-75.0, -30.0, n1, dtype=torch.float64, device="cuda")
    x2 = torch.linspace(20.0, 50.0, n2, dtype=torch.float64, device="cuda")
    X = torch.stack(torch.meshgrid(x1, x2, indexing="ij"), -1).reshape(-1, 2).contiguous()
    ds = [int(v) for v in args.ds.split(",")]
    gen = torch.Generator(device="cuda").manual_seed(0)
    Y = torch.empty((n, max(ds)), dtype=torch.float64, device="cuda")
    for d in range(max(ds)):                       # seeded smooth fields + noise, one per column
        Y[:, d] = torch.sin(X[:, 0] / (3.0 + 0.3 * d)) * torch.cos(X[:, 1] / (2.5 + 0.2 * d))
        Y[:, d] += 0.05 * torch.randn(n, dtype=torch.float64, device="cuda", generator=gen)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float64, device="cuda")      # 512 MB > L2, between timed calls

    def build(wl, y):
        m, k = WORKLOADS[wl]
        cls = getattr(B, "B%dSpline" % k)
        bases = [cls(DOM[0][0], DOM[0][1], m), cls(DOM[1][0], DOM[1][1], m)]
        kerns = [Kn.Matern32(variance=v, lengthscales=l) for v, l in HYP]
        model = GPR_kron((X, y), kerns, bases, raster_shape=(n1, n2), check_inputs=False)
        model.likelihood.variance.assign(S2)
        return model

    def time_steps(fn, steps):
        t = []
        for _ in range(steps):
            flush.fill_(0.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            t.append(a.elapsed_time(b))
        return float(np.median(t)), float(np.min(t)), float(np.max(t))

    results = []
    for wl in args.workloads.split(","):
        for D in ds:
            y = Y[:, 0].contiguous() if D == 1 else Y[:, :D]
            torch.cuda.synchronize(); t0 = time.perf_counter()
            model = build(wl, y)
            torch.cuda.synchronize(); t_build = (time.perf_counter() - t0) * 1e3
            for _ in range(3):
                model.elbo_and_grad()
            step = time_steps(model.elbo_and_grad, args.steps)
            singles = [model] if D == 1 else [build(wl, Y[:, d].contiguous()) for d in range(D)]
            for s in singles:
                s.elbo_and_grad()
            sep = time_steps(lambda: [s.elbo_and_grad() for s in singles], args.steps)
            Xp = X
            model.predict_f(Xp[:1000])                 # table prepared (and warmed) once per hyper-parameter set
            pred = time_steps(lambda: model.predict_f(Xp, raster_shape=(n1, n2)), 5)
            row = {"workload": wl, "m": WORKLOADS[wl][0], "order": WORKLOADS[wl][1], "n_points": n, "D": D,
                   "step_ms_median_min_max": step, "separate_models_step_ms_median_min_max": sep,
                   "construction_ms": t_build, "predict_f_ms_per_1e8_points": pred[0] * 1e8 / n,
                   "elbo": float(model.elbo())}
            if D == 1 and parent is not None:
                # the same model object, its whole step on the parent's kernels and on this build's, alternated
                arms = {"new": [], "parent": []}
                for _ in range(args.steps):
                    for arm, lib in (("new", new_lib), ("parent", parent)):
                        _lib._lib = lib
                        model.elbo_and_grad()
                        arms[arm].append(time_steps(model.elbo_and_grad, 1)[0])
                _lib._lib = new_lib
                _lib._lib = parent; e_parent = model.elbo_and_grad()[0]; _lib._lib = new_lib
                row["d1_alternated_ms_median"] = {a: float(np.median(v)) for a, v in arms.items()}
                row["d1_alternated_ms_min"] = {a: float(np.min(v)) for a, v in arms.items()}
                row["d1_elbo_parent_minus_new"] = float(e_parent - model.elbo_and_grad()[0])
            print(json.dumps(row), flush=True)
            results.append(row)
            del model, singles
            torch.cuda.empty_cache()
    out = {"gpu": info, "timing": "CUDA events around each call, median over --steps calls, a 512 MB buffer written "
                                  "between calls (L2 flushed)", "steps": args.steps, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
