"""Throughput of batched hyper-parameter evaluation of the 2-D Kronecker bound on one GPU.

For each shape (200 x 200 order 3 at bench.py's hypers, 100 x 100 order 4 = the eNATL60 shape, 40 x 40 order 3) and B in
1, 2, 4, ..., 64 settings (as memory allows): CUDA-event time of one GPR_kron.training_loss_and_gradients_batch(U) against B
calls of training_loss_and_gradients(), the two arms alternated (5 repeats, median); evaluations per second of each.  The
factorisation does not depend on N, so the shapes use a modest raster.
Then the wall time of a 16-start L-BFGS-B optimisation (Scipy.minimize(starts=...)) against the 16 serial runs on an
eNATL-shaped problem (N ~ 2e6 raster points, 100 x 100 B4 features), and, with --parent DIR (a built checkout of the parent
commit), bench.py's 2-D step in that checkout and in this one, alternated.

    python tools/kron_batched_bench.py [--out profiles/kron_batched.json] [--parent DIR]

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

BATCHES = (1, 2, 4, 8, 16, 32, 64)
DOM = ((-80, -25), (15, 55))                 # bench.py's 2-D basis domains and data extent
INNER = ((-75.0, -30.0), (20.0, 50.0))
HYPERS = ((1.0, 5.0), (1.0, 4.0), 0.01)      # bench.py's HYPERS_2D
SHAPES = (("200x200 k3 (bench)", 200, 3, 1000), ("100x100 k4 (eNATL60)", 100, 4, 1000), ("40x40 k3", 40, 3, 400))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                      # noqa: BLE001
        return {"error": repr(exc)}


def raster(torch, n1, seed=1997):
    """bench.py-style smooth field on an n1 x n1 raster over the eNATL60 extent."""
    x1 = torch.linspace(INNER[0][0], INNER[0][1], n1 + 2, dtype=torch.float64, device="cuda")[1:-1]
    x2 = torch.linspace(INNER[1][0], INNER[1][1], n1, dtype=torch.float64, device="cuda")
    X = torch.stack([x1[:, None].expand(n1, n1), x2[None, :].expand(n1, n1)], -1).reshape(-1, 2).contiguous()
    gen = torch.Generator(device="cpu").manual_seed(seed)
    y = torch.zeros(n1 * n1, dtype=torch.float64, device="cuda")
    for _ in range(8):
        f1, f2, ph = (torch.rand(3, generator=gen, dtype=torch.float64) * torch.tensor([0.6, 0.8, 6.28])).tolist()
        y += torch.sin(X[:, 0] * f1 + X[:, 1] * f2 + ph)
    y += 0.05 * torch.randn(n1 * n1, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    return X, y / 2.0


def model_for(torch, m, k, n1):
    from asvgp_b200 import basis as B, kernels as Kn
    from asvgp_b200.gpr import GPR_kron

    cls = getattr(B, "B%dSpline" % k)
    bases = [cls(DOM[0][0], DOM[0][1], m), cls(DOM[1][0], DOM[1][1], m)]
    kerns = [Kn.Matern32(variance=HYPERS[0][0], lengthscales=HYPERS[0][1]),
             Kn.Matern32(variance=HYPERS[1][0], lengthscales=HYPERS[1][1])]
    X, y = raster(torch, n1)
    model = GPR_kron((X, y.view(-1, 1)), kerns, bases, check_inputs=False, raster_shape=(n1, n1))
    model.likelihood.variance.assign(HYPERS[2])
    return model


def settings(model, B, rng):
    """B settings around the bench hypers (each value times 0.7 ... 1.4), unconstrained."""
    from asvgp_b200.kernels import _inv_softplus

    base = [p.value for p in model.trainable_variables]
    return [[_inv_softplus(v * f - p.lower) for v, f, p in zip(base, row, model.trainable_variables)]
            for row in rng.uniform(0.7, 1.4, (B, len(base)))]


def main():
    import numpy as np
    import torch

    from asvgp_b200 import _lib, ops
    from asvgp_b200.optimizers import Scipy

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kron_batched.json"))
    ap.add_argument("--parent", default=None, help="a built checkout of the parent commit: compare bench.py's 2-D step")
    ap.add_argument("--starts", type=int, default=16)
    ap.add_argument("--bench-steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    _lib.load()
    rng = np.random.default_rng(2026)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def gpu_ms(fn, reps):
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    shapes = []
    for label, m, k, n1 in SHAPES:
        model = model_for(torch, m, k, n1)
        params = model.trainable_variables
        slot_bytes = ops.kron_batch_slot_bytes(m, m, k, 1)
        rows = []
        for nb in BATCHES:
            free = ops.kron_batch_free_bytes(m, m, k, 1)
            if nb > 1 and nb * slot_bytes > 0.8 * free:
                rows.append(dict(B=nb, skipped="%d slots of %.2f GB do not fit in 0.8 of %.1f GB free" % (nb, slot_bytes / 1e9, free / 1e9)))
                continue
            U = np.array(settings(model, nb, rng))

            def batched():
                model.training_loss_and_gradients_batch(U)

            def serial():
                saved = [p.unconstrained for p in params]
                for row in U:
                    for p, u in zip(params, row):
                        p.unconstrained = float(u)
                    model.training_loss_and_gradients()
                for p, u in zip(params, saved):
                    p.unconstrained = u

            batched(); serial(); torch.cuda.synchronize()          # warm-up (plans, workspaces, modules)
            reps = max(2, 16 // nb)
            t_b, t_s = [], []
            for _ in range(5):                    # arms alternated
                t_b.append(gpu_ms(batched, reps))
                t_s.append(gpu_ms(serial, reps))
            med = lambda a: float(np.median(a))   # noqa: E731
            row = dict(B=nb, batched_ms=med(t_b), serial_ms=med(t_s), batched_evals_per_s=nb / med(t_b) * 1e3,
                       serial_evals_per_s=nb / med(t_s) * 1e3, speedup=med(t_s) / med(t_b),
                       spread_batched_ms=[min(t_b), max(t_b)], spread_serial_ms=[min(t_s), max(t_s)])
            print(label, json.dumps(row), flush=True)
            rows.append(row)
        shapes.append(dict(shape=label, m=[m, m], order=k, n=n1 * n1, slot_gb=slot_bytes / 1e9,
                           plan=ops.kron_plan_info(m, m, k), batches=rows))
        del model
        ops._KRON_BATCH_WS.clear()
        ops._KRON_WS.clear()
        torch.cuda.empty_cache()

    # multi-start L-BFGS-B on the eNATL60 shape: S starts in lockstep against S serial runs from the same starts
    n1 = 1414
    model = model_for(torch, 100, 4, n1)
    params = model.trainable_variables
    S = args.starts
    starts = np.array(settings(model, S, rng))
    saved = [p.unconstrained for p in params]
    opts = dict(options={"maxiter": 100})
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = Scipy().minimize(model.training_loss, params, starts=starts, **opts)
    t_multi = time.perf_counter() - t0
    t0 = time.perf_counter()
    serial_res = []
    for u0 in starts:
        for p, u in zip(params, u0):
            p.unconstrained = float(u)
        try:
            serial_res.append(Scipy().minimize(model.training_loss, params, **opts))
        except np.linalg.LinAlgError:
            serial_res.append(None)
    t_serial = time.perf_counter() - t0
    for p, u in zip(params, saved):
        p.unconstrained = u
    dx = max(float(np.abs(s.x - r.x).max()) for s, r in zip(serial_res, res.results) if s is not None and np.isfinite(r.fun))
    multi = dict(shape="100x100 k4", n=n1 * n1, starts=S, maxiter=100, wall_s_multi_start=t_multi, wall_s_serial=t_serial,
                 speedup=t_serial / t_multi, total_evaluations=int(sum(r.nfev for r in res.results if np.isfinite(r.fun))),
                 best_loss=float(res.fun), max_abs_x_difference_to_serial=dx)
    print(json.dumps(multi), flush=True)
    del model
    ops._KRON_BATCH_WS.clear()
    torch.cuda.empty_cache()

    bench = None
    if args.parent:
        cmd = [sys.executable, "bench.py", "--gpus", "1", "--workload", "2d", "--steps", str(args.bench_steps), "--warmup", "3",
               "--no-cpu-baseline", "--no-e2e"]
        bench = {"command": " ".join(cmd[1:]), "parent": [], "change": []}
        for _ in range(2):                        # alternated
            for arm, cwd in (("parent", os.path.abspath(args.parent)), ("change", ROOT)):
                out = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
                line = next((ln for ln in reversed(out.stdout.splitlines()) if ln.startswith("{")), None)
                if line is None:
                    bench[arm].append({"error": out.stderr[-2000:]})
                    continue
                d = json.loads(line)
                bench[arm].append({key: d.get(key) for key in ("ms_per_step", "phases_ms", "gpu_launches", "elbo")})
                print(arm, json.dumps(bench[arm][-1])[:400], flush=True)
    out = dict(gpu=gpu_info(), torch=torch.__version__,
               note="CUDA events over `reps` back-to-back calls, median of 5 alternated repeats; every call ends with its "
                    "device-to-host read.  Serial = training_loss_and_gradients() per setting (method 'nd').",
               shapes=shapes, multi_start=multi, bench_2d=bench)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
