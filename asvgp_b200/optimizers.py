"""`Scipy` — the slice of `gpflow.optimizers.Scipy` the reference uses (experiments/snelson/example.py:31-32):
L-BFGS-B over the unconstrained (softplus-transformed) variables, loss and gradient from one GPU evaluation."""
import threading

import numpy as np
import scipy.optimize


def _same_on_every_rank(u):
    """Data-parallel runs: every rank drives its own L-BFGS on (up to rounding) the same loss and gradient; rank 0's iterate
    is broadcast before each evaluation so that the replicas can never drift apart by an ulp and take different line-search
    branches (the factorisation uses fp64 REDs, whose summation order is not fixed)."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return u
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.as_tensor(np.asarray(u, dtype=np.float64)).to(dev)
    dist.broadcast(t, src=0)
    return t.cpu().numpy()


def lockstep_minimize(fun_batch, starts, method="L-BFGS-B", pass_ids=False, **scipy_kwargs):
    """One scipy.optimize.minimize per row of starts[B, n], advanced in lockstep: each run lives in a worker thread whose
    objective posts its point and blocks; once every run still going has posted, fun_batch(U[b', n]) evaluates them all
    at once and returns (loss[b'], grad[b', n], info[b']).  A run sees exactly the values a serial run would, so its iterates
    are those of the serial run from the same start.  Line-search evaluations are simply more rounds; a finished run leaves
    the rounds.  A row with info != 0 raises numpy.linalg.LinAlgError inside that run's objective (as a failing serial
    evaluation does); the run ends with success=False and fun=+inf while the others go on.  Returns the B results.
    pass_ids=True: fun_batch(U, ids) also receives the run indices (rows of starts) of the rows of U, for objectives that
    differ from run to run (one model per run)."""
    starts = np.array(starts, dtype=np.float64, ndmin=2)
    B = starts.shape[0]
    cv = threading.Condition()
    running, posted, replies, results = set(range(B)), {}, {}, [None] * B

    def run(b):
        last = [starts[b]]

        def fun(u):
            last[0] = np.array(u, dtype=np.float64)
            with cv:
                posted[b] = last[0]
                cv.notify_all()
                cv.wait_for(lambda: b in replies)
                reply = replies.pop(b)
            if isinstance(reply, BaseException):
                raise reply
            loss, grad, info = reply
            if info != 0:
                raise np.linalg.LinAlgError("banded Cholesky failed: non-positive pivot %d" % int(info))
            return loss, grad

        try:
            res = scipy.optimize.minimize(fun, starts[b], jac=True, method=method, **scipy_kwargs)
        except np.linalg.LinAlgError as e:
            res = scipy.optimize.OptimizeResult(x=last[0], fun=np.inf, success=False, status=-1,
                                                message=str(e), nit=-1)
        except BaseException as e:      # an error of the evaluation itself: the caller re-raises it
            res = e
        with cv:
            results[b] = res
            running.discard(b)
            cv.notify_all()

    threads = [threading.Thread(target=run, args=(b,), daemon=True) for b in range(B)]
    for t in threads:
        t.start()
    error = None
    while True:
        with cv:
            cv.wait_for(lambda: all(b in posted for b in running))
            if not running:
                break
            ids = sorted(running)
            U = np.stack([posted.pop(b) for b in ids])
        try:
            if error is not None:
                raise error
            loss, grad, info = fun_batch(U, np.array(ids)) if pass_ids else fun_batch(U)
            reply = {b: (float(loss[i]), np.array(grad[i], dtype=np.float64), int(info[i])) for i, b in enumerate(ids)}
        except BaseException as e:      # stop every run, then re-raise
            error = e
            reply = {b: e for b in ids}
        with cv:
            replies.update(reply)
            cv.notify_all()
    for t in threads:
        t.join()
    if error is not None:
        raise error
    for r in results:
        if isinstance(r, BaseException):
            raise r
    return results


class Scipy:
    def minimize(self, closure, variables, method="L-BFGS-B", starts=None, **scipy_kwargs):
        """L-BFGS-B (by default) over the unconstrained values of `variables`; the model ends at the result.

        starts[B, len(variables)]: multi-start — B runs from these unconstrained points, advanced in lockstep with one
        batched evaluation (the model's training_loss_and_gradients_batch) per round; every run takes the iterates a
        serial run from its start would.  The model is set to the run with the lowest loss, whose result is returned
        with `results` (all B results, in the order of starts) and `best` (its index) added."""
        model = getattr(closure, "__self__", None)
        if model is None or not hasattr(model, "training_loss_and_gradients"):
            raise TypeError("closure must be the bound `training_loss` of an asvgp_b200 model")
        variables = list(variables)
        model_vars = model.trainable_variables
        index = [next(i for i, p in enumerate(model_vars) if p is v) for v in variables]
        if starts is not None:
            return self._minimize_multi(model, variables, index, starts, method, scipy_kwargs)

        def fun(u):
            u = _same_on_every_rank(u)
            for v, ui in zip(variables, u):
                v.unconstrained = float(ui)
            loss, grad = model.training_loss_and_gradients()
            return loss, grad[index]

        u0 = np.array([v.unconstrained for v in variables], dtype=np.float64)
        res = scipy.optimize.minimize(fun, u0, jac=True, method=method, **scipy_kwargs)
        for v, ui in zip(variables, res.x):
            v.unconstrained = float(ui)
        return res

    @staticmethod
    def _minimize_multi(model, variables, index, starts, method, scipy_kwargs):
        batch = getattr(model, "training_loss_and_gradients_batch", None)
        if batch is None:
            raise NotImplementedError("%s has no batched evaluation (training_loss_and_gradients_batch)"
                                      % type(model).__name__)
        starts = np.asarray(starts, dtype=np.float64)
        if starts.ndim != 2 or starts.shape[1] != len(variables) or starts.shape[0] < 1:
            raise ValueError("starts must be [B, %d] (B >= 1), got shape %s" % (len(variables), starts.shape))
        if not np.isfinite(starts).all():
            raise ValueError("starts must be finite")
        fixed = np.array([p.unconstrained for p in model.trainable_variables], dtype=np.float64)

        def fun_batch(U):
            U = _same_on_every_rank(U)          # rank 0's points, once per round
            full = np.repeat(fixed[None, :], U.shape[0], axis=0)
            full[:, index] = U
            loss, grad, info = batch(full)
            return loss, grad[:, index], info

        results = lockstep_minimize(fun_batch, starts, method=method, **scipy_kwargs)
        finite = [b for b, r in enumerate(results) if np.isfinite(r.fun)]
        if not finite:
            raise np.linalg.LinAlgError("every start failed: %s" % results[0].message)
        best = min(finite, key=lambda b: results[b].fun)
        for v, ui in zip(variables, results[best].x):
            v.unconstrained = float(ui)
        out = scipy.optimize.OptimizeResult(results[best])
        out.results, out.best = results, best
        return out
