"""Throughput of batched hyper-parameter evaluation of the 1-D bound on one GPU (M = 10^4 cubic B-splines, Matern52, the
C3 shape of tests/scale_cases.py with fewer points: the bound's cost does not depend on N).

For B in 1, 2, 4, ..., 64 settings:
  * GPU time of one batched evaluation (asvgp_kuu_assemble_batched + asvgp_elbo_grad_1d_batched), CUDA events, against B
    single evaluations as GPR_1d runs them (asvgp_kuu_assemble, the Kuu chain on its side stream, the P chains), the two
    arms alternated; evaluations per second of each;
  * host wall time of one L-BFGS round: GPR_1d.training_loss_and_gradients_batch (launches, the one D2H read, combining)
    against B calls of training_loss_and_gradients;
  * the same batched evaluation with chunks = 256 (2-CTA clusters instead of 8): more chains resident at once, another
    chunking (its bits differ from the default's in the last places).
Then the wall time of a 16-start L-BFGS-B optimisation (Scipy.minimize(starts=...)) against the 16 serial runs.

    python tools/batched_bound_bench.py [--out profiles/batched_bound.json] [--reps 30]

Writes one JSON with the GPU name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

BATCHES = (1, 2, 4, 8, 16, 32, 64)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:                      # noqa: BLE001
        return {"error": repr(exc)}


def main():
    import numpy as np
    import torch

    import scale_cases as SC
    from asvgp_b200 import _lib, basis as B, kernels as Kn, ops
    from asvgp_b200.gpr import GPR_1d
    from asvgp_b200.optimizers import Scipy

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batched_bound.json"))
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--n", type=float, default=2e6)
    ap.add_argument("--starts", type=int, default=16)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    _lib.load()
    m, k = SC.C3_M, SC.C3_ORDER
    x, y, _ = SC.case_1d(n=int(args.n), m=m, seed=31, n_test=1)
    basis = B.B3Spline(-1, m + 1, m)
    model = GPR_1d((torch.from_numpy(x).cuda().view(-1, 1), torch.from_numpy(y).cuda().view(-1, 1)), Kn.Matern52(), basis)
    acc = model._acc
    params = model.trainable_variables
    rng = np.random.default_rng(2026)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def gpu_ms(fn, reps):
        fn()
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / reps

    rows = []
    for nb in BATCHES:
        U = np.column_stack([rng.uniform(-0.5, 1.5, nb), rng.uniform(0.0, 2.5, nb), rng.uniform(-3.0, -1.0, nb)])
        vals = np.array([[p.value_at(u) for p, u in zip(params, row)] for row in U])
        v, l, s2 = vals[:, 0], vals[:, 1], vals[:, 2]

        def batched(chunks=0):
            Kuu, dKuu = model.inducing_features.make_Kuu_device_batched(model.kernel, l, v)
            ops.elbo_grad_1d_batched(Kuu, dKuu, acc.view(1, -1), basis, v, s2, chunks=chunks)

        def serial():
            for b in range(nb):
                terms = model.inducing_features._terms(model.kernel, l[b], v[b])
                Kuu, dKuu = ops.kuu_assemble(basis, [t[0] for t in terms], [t[1] for t in terms], [t[2] for t in terms])
                ops.elbo_grad_1d(Kuu, dKuu, acc, basis, v[b], s2[b])

        reps = max(3, args.reps // nb)
        t_b, t_s, t_256 = [], [], []
        for _ in range(5):                        # arms alternated
            t_b.append(gpu_ms(batched, reps))
            t_s.append(gpu_ms(serial, reps))
            t_256.append(gpu_ms(lambda: batched(256), reps))
        # host wall time of one optimiser round (launches + one D2H read + combining), arms alternated
        w_b, w_s = [], []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                model.training_loss_and_gradients_batch(U)
            w_b.append((time.perf_counter() - t0) * 1e3 / reps)
            saved = [p.unconstrained for p in params]
            t0 = time.perf_counter()
            for _ in range(reps):
                for row in U:
                    for p, u in zip(params, row):
                        p.unconstrained = float(u)
                    model.training_loss_and_gradients()
            w_s.append((time.perf_counter() - t0) * 1e3 / reps)
            for p, u in zip(params, saved):
                p.unconstrained = u
        med = lambda a: float(np.median(a))
        row = dict(B=nb, batched_gpu_ms=med(t_b), serial_gpu_ms=med(t_s), batched_chunks256_gpu_ms=med(t_256),
                   batched_evals_per_s=nb / med(t_b) * 1e3, serial_evals_per_s=nb / med(t_s) * 1e3,
                   chunks256_evals_per_s=nb / med(t_256) * 1e3, gpu_speedup=med(t_s) / med(t_b),
                   round_wall_ms_batched=med(w_b), round_wall_ms_serial=med(w_s),
                   spread_batched_gpu_ms=[min(t_b), max(t_b)], spread_serial_gpu_ms=[min(t_s), max(t_s)])
        print(json.dumps(row), flush=True)
        rows.append(row)

    # multi-start L-BFGS-B: S starts in lockstep against S serial runs from the same starts
    S = args.starts
    starts = np.column_stack([rng.uniform(-0.5, 1.5, S), rng.uniform(0.0, 2.5, S), rng.uniform(-3.0, -1.0, S)])
    saved = [p.unconstrained for p in params]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = Scipy().minimize(model.training_loss, params, starts=starts)
    t_multi = time.perf_counter() - t0
    t0 = time.perf_counter()
    serial_res = []
    for u0 in starts:
        for p, u in zip(params, u0):
            p.unconstrained = float(u)
        try:
            serial_res.append(Scipy().minimize(model.training_loss, params))
        except np.linalg.LinAlgError:
            serial_res.append(None)
    t_serial = time.perf_counter() - t0
    for p, u in zip(params, saved):
        p.unconstrained = u
    same = all(s is None and r.fun == np.inf or s is not None and np.array_equal(s.x, r.x) and s.nit == r.nit
               for s, r in zip(serial_res, res.results))
    multi = dict(starts=S, wall_s_multi_start=t_multi, wall_s_serial=t_serial, speedup=t_serial / t_multi,
                 rounds_evaluations=int(max(r.nfev for r in res.results if np.isfinite(r.fun))),
                 total_evaluations=int(sum(r.nfev for r in res.results if np.isfinite(r.fun))),
                 best_loss=float(res.fun), iterates_equal_serial=bool(same))
    print(json.dumps(multi), flush=True)
    out = dict(gpu=gpu_info(), torch=torch.__version__, m=m, order=k, kernel="Matern52", n=int(args.n),
               note="GPU times: CUDA events over `reps` back-to-back calls, median of 5 alternated repeats; the working set "
                    "(bands, row tables) stays in L2, as it does inside an optimiser loop.",
               batches=rows, multi_start=multi)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
