"""Many independent 1-D series on one GPU: GPR_1d_many against a Python loop over GPR_1d models, one per series.

Workloads (S series of N_s sorted points each, M cubic B-splines, Matern32): (1024, 1e5, 1000), (64, 1e6, 1e4) and
(1e4, 1e4, 1000) hold 1e8 points each (1.6 GB of float64 data, far more than L2), and (4096, 100, 100) shows what short
series cost.  For each workload and arm, the arms alternated, median of --reps:
  * accumulate: building the model(s) on device-resident data (GB/s at 16 B per point);
  * bound: one -ELBO and gradient of all S series (training_loss_and_gradients);
  * predict: posterior plus predict_f of 1e3 test points per series.
Then a full L-BFGS-B fit of 256 series of 1e5 points (M = 1000): GPR_1d_many.optimize() against 256 serial Scipy().minimize.
Times are host wall clock around work that ends in a device synchronise.

    python tools/many_series_bench.py [--out profiles/many_series.json] [--reps 3]

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

WORKLOADS = ((1024, 100_000, 1000), (64, 1_000_000, 10_000), (10_000, 10_000, 1000), (4096, 100, 100))
N_TEST = 1000


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                      # noqa: BLE001
        return {"error": repr(exc)}


def _data(S, n, m, seed):
    import torch

    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.sort(torch.rand((S, n), generator=g, device="cuda", dtype=torch.float64) * (m - 0.02) + 0.01, dim=1).values
    y = torch.sin(x / 7.0) + 0.3 * torch.randn((S, n), generator=g, device="cuda", dtype=torch.float64)
    return x.reshape(-1, 1), y.reshape(-1)


def _timed(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    import numpy as np
    import torch

    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_1d, GPR_1d_many
    from asvgp_b200.optimizers import Scipy

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "many_series.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--fit-series", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info(), "kernel": "Matern32", "order": 3, "reps": args.reps, "workloads": []}

    for S, n, m in WORKLOADS:
        basis = B.B3Spline(0, m, m)
        X, y = _data(S, n, m, seed=S)
        offsets = np.arange(S + 1, dtype=np.int64) * n
        xt = torch.linspace(0.005, m - 0.005, N_TEST, device="cuda", dtype=torch.float64).repeat(S).reshape(-1, 1)
        off_t = np.arange(S + 1, dtype=np.int64) * N_TEST

        def build_many():
            return GPR_1d_many((X, y), offsets, Kn.Matern32(), basis, check_inputs=False)

        def build_loop():
            return [GPR_1d((X[i * n:(i + 1) * n], y[i * n:(i + 1) * n]), Kn.Matern32(), basis, check_inputs=False)
                    for i in range(S)]

        many, loop = build_many(), build_loop()                       # warm-up of every shape the timed runs use
        many.training_loss_and_gradients(), [md.training_loss_and_gradients() for md in loop]
        many.predict_f(xt, off_t), [md.predict_f(xt[:N_TEST]) for md in loop]
        # the two arms agree
        lm = many.training_loss_and_gradients()[0]
        ll = np.array([md.training_loss_and_gradients()[0] for md in loop])
        max_rel = float(np.max(np.abs(lm - ll) / np.abs(ll)))
        t = {k: {"many": [], "loop": []} for k in ("accumulate", "bound", "predict")}
        for _ in range(args.reps):
            for arm in ("many", "loop"):
                dt, model = _timed(build_many if arm == "many" else build_loop)
                t["accumulate"][arm].append(dt)
                if arm == "many":
                    t["bound"][arm].append(_timed(model.training_loss_and_gradients)[0])
                    t["predict"][arm].append(_timed(lambda: model.predict_f(xt, off_t))[0])
                else:
                    t["bound"][arm].append(_timed(lambda: [md.training_loss_and_gradients() for md in model])[0])
                    t["predict"][arm].append(_timed(lambda: [md.predict_f(xt[:N_TEST]) for md in model])[0])
                del model
        med = {k: {a: float(np.median(v[a])) for a in v} for k, v in t.items()}
        row = {"S": S, "N_s": n, "M": m, "points": S * n, "bytes_per_point": 16, "max_rel_loss_difference": max_rel,
               "ms": {k: {a: 1e3 * v for a, v in d.items()} for k, d in med.items()},
               "accumulate_GBps": {a: 16 * S * n / med["accumulate"][a] / 1e9 for a in ("many", "loop")},
               "bounds_per_s": {a: S / med["bound"][a] for a in ("many", "loop")},
               "speedup": {k: med[k]["loop"] / med[k]["many"] for k in med}}
        print(json.dumps(row), flush=True)
        result["workloads"].append(row)
        del many, loop, X, y, xt
        torch.cuda.empty_cache()

    # full fit
    S, n, m = args.fit_series, 100_000, 1000
    basis = B.B3Spline(0, m, m)
    X, y = _data(S, n, m, seed=99)
    offsets = np.arange(S + 1, dtype=np.int64) * n
    many = GPR_1d_many((X, y), offsets, Kn.Matern32(), basis, check_inputs=False)
    loop = [GPR_1d((X[i * n:(i + 1) * n], y[i * n:(i + 1) * n]), Kn.Matern32(), basis, check_inputs=False) for i in range(S)]

    def fit_loop():
        return [Scipy().minimize(md.training_loss, md.trainable_variables) for md in loop]

    U0 = many.U.copy()
    dt_many, res_many = _timed(many.optimize)
    dt_loop, res_loop = _timed(fit_loop)
    same = sum(bool(np.array_equal(a.x, b.x)) for a, b in zip(res_many, res_loop))
    result["fit"] = {"S": S, "N_s": n, "M": m, "s": {"many": dt_many, "loop": dt_loop}, "speedup": dt_loop / dt_many,
                     "iterations": {"many": int(sum(r.nit for r in res_many)), "loop": int(sum(r.nit for r in res_loop))},
                     "runs_with_identical_iterates": same, "start": U0[0].tolist()}
    print(json.dumps(result["fit"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
