"""Models `GPR_1d` and `GPR_kron` — same constructor, attributes and methods as reference asvgp/gpr.py:18-136 and
:239-359, computed by the sm_100a kernels of libasvgp_sm100a (no CPU fallback).

What differs from the reference is only *how*:
  * the O(N) precompute never materialises Kuf (fused accumulate kernel, asvgp_accum_1d);
  * the per-step banded algebra (2 Choleskys, Takahashi inverse, triangular solve, gpr.py:55-75) runs as partitioned
    sweeps on the GPU and returns the hyper-parameter gradients with the ELBO (the reference gets them from TF
    reverse mode when `gpflow.optimizers.Scipy` asks, example.py:31-32);
  * prediction is O(n*) instead of O(n* M): only the (k+1) window entries of alpha and of
    band(P^-1) - band(Kuu^-1) matter (gpr.py:103-118);
  * with torch.distributed initialised the data passed in are this rank's shard and the packed accumulator is
    all-reduced once (SURVEY §8(e)).
"""
import numpy as np
import torch

from . import _lib
from . import dist as _dist
from . import ops
from .inducing_features import SplineFeatures1D
from .ops import Bound1D
from .kernels import Gaussian, Parameter, hyper_value, kernel_kind


class _ModelBase:
    """The slice of gpflow.models.GPModel + InternalDataTrainingLossMixin the reference's scripts use."""

    _host = None

    def _device_stats(self):
        """(G, Kuf_y [D, M], sum(y_d^2) [D], N) of the D output columns as device tensors; G is the model's own form of KufKfu."""
        raise NotImplementedError

    # -- the reference's cached attributes (host copies, fetched lazily) --------------------------------------
    def _host_stats(self):
        if self._host is None:
            G, B, yy, n = (t.cpu().numpy() for t in self._device_stats())
            self._host = (G, np.ascontiguousarray(B.T), float(yy.sum()), int(n))
        return self._host

    @property
    def Kuf_y(self):
        """(M, D): one column per output column."""
        return self._host_stats()[1]

    @property
    def tr_yTy(self):
        """sum(y^2) over all output columns (reference gpr.py:78-79)."""
        return self._host_stats()[2]

    @property
    def num_data(self):
        """Global number of datapoints (all shards)."""
        return self._host_stats()[3]

    def maximum_log_likelihood_objective(self):
        return self.elbo()

    def training_loss(self):
        return -self.maximum_log_likelihood_objective()

    def training_loss_and_gradients(self):
        """(-ELBO, d(-ELBO)/d unconstrained variables) in the order of `trainable_variables`."""
        elbo, grads = self.elbo_and_grad()
        g = [-(grads[id(p)] * p.dvalue_dunconstrained()) for p in self.trainable_variables]
        return -elbo, np.array(g, dtype=np.float64)

    def predict_log_density(self, data):
        """log N(y | mean, var + sigma2) per test point (used by reference electricity.py:138)."""
        X, y = data
        mean, var = self.predict_f(X)
        mean, var = np.asarray(_to_numpy(mean)), np.asarray(_to_numpy(var))
        s2 = var + hyper_value(self.likelihood.variance)
        y = np.asarray(_to_numpy(y)).reshape(mean.shape)
        return (-0.5 * np.log(2 * np.pi * s2) - 0.5 * (y - mean) ** 2 / s2).sum(-1)


def _grad_dict(pairs):
    """{id(param): derivative}, summed when the same parameter object appears more than once (e.g. one kernel object
    shared by both dimensions of a Kronecker model)."""
    out = {}
    for p, v in pairs:
        out[id(p)] = out.get(id(p), 0.0) + v
    return out


def _unique(params):
    seen, out = set(), []
    for p in params:
        if id(p) not in seen:
            seen.add(id(p))
            out.append(p)
    return out


def _to_numpy(a):
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a


def _like_input(Xnew, mean, var):
    """(mean, var) as they are for a CUDA tensor Xnew, else as numpy arrays."""
    if isinstance(Xnew, torch.Tensor) and Xnew.is_cuda:
        return mean, var
    return mean.cpu().numpy(), var.cpu().numpy()


def _check_domain(X, bases):
    """Every column i of X[n, d] lies strictly inside the domain of bases[i] (reference gpr.py:22-26); AssertionError if not."""
    for i, basis in enumerate(bases):
        col = X[:, i]
        lo, hi = (torch.aminmax(col) if isinstance(col, torch.Tensor) else (col.min(), col.max()))
        assert float(lo) > basis.a and float(hi) < basis.b, "inputs must lie strictly inside the basis domain"


def _output_columns(y, model, most, error=ValueError):
    """y[n] or y[n, D] as (y[n, D], D); D outside 1 ... most raises `error`."""
    if y.ndim == 1:
        y = y.reshape(-1, 1)
    D = int(y.shape[1])
    if not 1 <= D <= most:
        raise error("%s takes 1 ... %d output columns, got %d" % (model, most, D))
    return y, D


def _combine_columns(values, infos, shared):
    """The bound of D output columns from their single-column bounds: row values[d] (1 + G entries) holds column d's ELBO and,
    if G > 0, its G derivatives.  The reference scales the log-dets by D and sums the data-fit terms over the columns, but counts the
    prior and trace terms T = (-N prior + trace) / (2 sigma2) once, not D times (gpr.py:81-87), so D - 1 copies of T are taken
    out of the column sums again.  shared() returns [T, dT] (model-specific; read only for D > 1; its first 1 + G entries are
    used).  The columns are added in order.  Returns (elbo, grad[G], info), info = the first non-zero of `infos` (0.0 if none)."""
    total = values[0]
    for row in values[1:]:
        total = total + row
    if len(values) > 1:
        total = total - (len(values) - 1) * shared()[: total.size]
    info = next((i for i in infos if i != 0), 0.0)
    return total[0], total[1:], info


def _losses(bounds, params, U):
    """(loss[n], grad[n, G], info[n]) from n combined bounds (elbo, grad[G], info) at the unconstrained points U[n, G] of
    `params`: loss = -ELBO and its gradient in U.  A failed bound (info != 0) gives loss +inf, NaN gradients and its pivot."""
    n = len(U)
    loss, grad, info = np.empty(n), np.empty((n, len(params))), np.zeros(n, dtype=np.int64)
    for b, ((elbo, g, inf), u) in enumerate(zip(bounds, U)):
        if inf != 0:
            loss[b], grad[b], info[b] = np.inf, np.nan, int(inf)
            continue
        loss[b] = -float(elbo)
        grad[b] = [-(g_j * p.dvalue_dunconstrained_at(float(u_j))) for g_j, p, u_j in zip(g, params, u)]
    return loss, grad, info


def _values_at(params, U):
    """Constrained values [n, len(params)] of params at the unconstrained rows U[n, len(params)]."""
    return np.array([[p.value_at(float(u)) for p, u in zip(params, row)] for row in U]).reshape(-1, len(params))


class GPR_1d(_ModelBase):
    """Collapsed-bound sparse GP regression in 1-D with B-spline inducing features (reference gpr.py:18-136).

    data = (X[n, 1], y[n] or y[n, D]) as CUDA tensors or host arrays; X and y may each be float32 or float64 and are read
    as they are (the accumulate converts every value to float64 in registers, so the model equals the one built from the
    float64-converted data up to summation order).  Everything after the O(N) pass is float64."""

    _acc_batch = None       # the accumulators as one [D, L] tensor (training_loss_and_gradients_batch), built on first use
    _n_host = None

    def __init__(self, data, kernel, basis, distributed="auto", check_inputs=True, chunks=0):
        # Check inputs (reference gpr.py:22-26)
        self._kind = kernel_kind(kernel)
        X, y = data
        assert X.shape[1] == 1
        if y.ndim == 1:
            y = y.reshape(-1, 1)
        self.X, self.y = X, y
        n_out = int(y.shape[1])
        on_device = isinstance(X, torch.Tensor) and X.is_cuda
        if check_inputs and X.shape[0]:
            _check_domain(X, [basis])

        # Init model (reference gpr.py:29-34)
        self.kernel = kernel
        self.likelihood = Gaussian()
        self.mean_function = None
        self.num_latent_gps = 1
        self.basis = basis
        self.inducing_features = SplineFeatures1D(kernel, basis)
        self.bandwidth = self.basis.order
        self._chunks = chunks

        # Precompute static quantities (reference gpr.py:39-44): one fused pass over this rank's points,
        # then (multi-GPU) one all-reduce of the packed buffer.
        # Multi-output y (D columns, gpr.py:40,78-79) keeps one packed accumulator per column: G and N are
        # shared, Kuf_y and sum(y^2) are per column.
        self._accs = []
        for d in range(n_out):
            yd = y[:, d] if n_out > 1 else y.reshape(-1)
            if on_device:
                self._accs.append(ops.accum_1d(X.reshape(-1), yd.contiguous(), basis, binned="auto"))
            else:                   # host data: streamed through pinned staging buffers, never fully resident
                self._accs.append(ops.accum_1d_host(X, np.ascontiguousarray(yd), basis))
        self._distributed = _dist.is_distributed(distributed)
        if self._distributed:
            red = _dist.oneshot_reducer(self._accs[0].numel()) if (len(self._accs) == 1 and self._accs[0].is_cuda) else None
            if red is not None:          # one kernel over NVLink peer memory (asvgp_allreduce_oneshot); else NCCL
                red.buffer().copy_(self._accs[0])
                red.reduce(self._accs[0])
            elif len(self._accs) == 1:
                _dist.allreduce_packed(self._accs[0])
            else:                   # D output columns: still ONE collective, over the stacked packed buffers
                stacked = torch.stack(self._accs)
                _dist.allreduce_packed(stacked)
                self._accs = list(stacked.unbind(0))
        self._acc = self._accs[0]
        self._G, self._b, self._scal = ops.split_accum_1d(self._acc, basis)
        self._outs = [torch.empty(16, dtype=torch.float64, device=self._acc.device) for _ in self._accs]
        self._out = self._outs[0]

    def _device_stats(self):
        parts = [ops.split_accum_1d(acc, self.basis) for acc in self._accs]
        return self._G, torch.stack([p[1] for p in parts]), torch.stack([p[2][0] for p in parts]), self._scal[1]

    @property
    def KufKfu(self):
        return self._host_stats()[0]

    @property
    def KufKfu_sparse(self):
        from . import utils

        full = utils.band_to_sparse(self.KufKfu)
        return full + full.T - __import__("scipy.sparse", fromlist=["diags"]).diags(self.KufKfu[0])

    @property
    def trainable_variables(self):
        return [self.kernel.variance, self.kernel.lengthscales, self.likelihood.variance]

    # -- objective ---------------------------------------------------------------------------------------------
    def _launch_elbo(self):
        var = hyper_value(self.kernel.variance)
        s2 = hyper_value(self.likelihood.variance)
        Kuu, dKuu = self.inducing_features.make_Kuu_device(self.kernel, want_grad=True)
        kuu = ops.kuu_chain_1d(Kuu, dKuu, self.basis, chunks=self._chunks)     # once: it does not depend on y
        for acc, out in zip(self._accs, self._outs):
            ops.elbo_grad_1d(Kuu, dKuu, acc, self.basis, var, s2, chunks=self._chunks, out=out, kuu=kuu, join_late=True)
        return self._out

    @staticmethod
    def _bound(outs, v, s2, n):
        """(elbo, grad[3], info) of the D output columns from their rows outs[D, 16] (Bound1D) at variance v and sigma2 s2;
        n() returns the number of data points (called for D > 1 only).  T = (-N v + trace) / (2 s2) counts once:
        dT/dv = (-N + trace / v) / (2 s2) (trace is linear in v), dT/dl = (dtrace/dl) / (2 s2), dT/ds2 = -T / s2."""
        def shared():
            N, tr = n(), outs[0, Bound1D.TRACE]
            T = 0.5 * (-N * v + tr) / s2
            return np.array([T, 0.5 * (-N + tr / v) / s2, 0.5 * outs[0, Bound1D.DTRACE_DL] / s2, -T / s2])
        return _combine_columns(outs[:, Bound1D.ELBO_GRAD], outs[:, Bound1D.INFO], shared)

    def elbo_and_grad(self):
        """ELBO (reference gpr.py:49-89) and {id(param): dELBO/dparam} for variance, lengthscales, sigma^2."""
        self._launch_elbo()
        outs = torch.stack(self._outs).cpu().numpy()
        v, s2 = hyper_value(self.kernel.variance), hyper_value(self.likelihood.variance)
        elbo, g, info = self._bound(outs, v, s2, lambda: float(self._scal[1].item()))
        if info != 0:
            raise np.linalg.LinAlgError("banded Cholesky failed: non-positive pivot %d" % int(info))
        row = outs[0]
        self.last_terms = dict(log_det_Kuu=row[Bound1D.LOG_DET_KUU], log_det_P=row[Bound1D.LOG_DET_P],
                               quad=outs[:, Bound1D.QUAD].sum(), trace=row[Bound1D.TRACE])
        return float(elbo), _grad_dict(zip(self.trainable_variables, g))

    def training_loss_and_gradients_batch(self, U):
        """training_loss_and_gradients at B settings at once, without changing the model's parameters.

        U[B, 3]: unconstrained values in the order of `trainable_variables` (1 <= B <= 64).  Returns (loss[B], grad[B, 3],
        info[B]); row b equals training_loss_and_gradients() with the parameters set to U[b], bit for bit.  A setting whose
        banded Cholesky fails gets loss = +inf, NaN gradients and its first failing pivot in info (nothing is raised).  All
        settings share the accumulators and run as one batch of chains on the GPU (asvgp_elbo_grad_1d_batched); the results
        come back in one device-to-host copy."""
        params = self.trainable_variables
        U = np.asarray(U, dtype=np.float64)
        if U.ndim != 2 or U.shape[1] != len(params):
            raise ValueError("U must be [B, %d] (unconstrained values of trainable_variables), got shape %s"
                             % (len(params), U.shape))
        if not 1 <= U.shape[0] <= _lib.MAX_BATCH:
            raise ValueError("U has %d rows; a batch holds 1..%d settings" % (U.shape[0], _lib.MAX_BATCH))
        if not np.isfinite(U).all():
            raise ValueError("U must be finite")
        vals = _values_at(params, U)
        var, ell, s2 = vals[:, 0], vals[:, 1], vals[:, 2]
        Kuu, dKuu = self.inducing_features.make_Kuu_device_batched(self.kernel, ell, var, want_grad=True)
        if self._acc_batch is None:
            self._acc_batch = self._acc.view(1, -1) if len(self._accs) == 1 else torch.stack(self._accs)
        if len(self._accs) > 1 and self._n_host is None:
            self._n_host = float(self._scal[1].item())
        outs = ops.elbo_grad_1d_batched(Kuu, dKuu, self._acc_batch, self.basis, var, s2, chunks=self._chunks).cpu().numpy()
        bounds = [self._bound(outs[b], var[b], s2[b], lambda: self._n_host) for b in range(len(U))]
        return _losses(bounds, params, U)

    def elbo(self):
        """Variational bound on the log marginal likelihood (reference gpr.py:49-89)."""
        return np.float64(self.elbo_and_grad()[0])

    # -- prediction ----------------------------------------------------------------------------------------------
    def posterior_weights(self):
        """(alpha, S) on the device: alpha = P^-1 Kuf_y / sigma2, S = band(P^-1) - band(Kuu^-1)."""
        s2 = hyper_value(self.likelihood.variance)
        Kuu, _ = self.inducing_features.make_Kuu_device(self.kernel, want_grad=False)
        alpha, S, info = ops.posterior_1d(Kuu, self._acc, self.basis, s2, chunks=self._chunks)
        if len(self._accs) > 1:          # one solve per output column; S does not depend on y
            cols = [alpha]
            for acc in self._accs[1:]:
                a_d, _, info_d = ops.posterior_1d(Kuu, acc, self.basis, s2, chunks=self._chunks)
                cols.append(a_d)
                info = torch.maximum(info, info_d)
            alpha = torch.stack(cols, 0)
        return alpha, S, info

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False, batch=False):
        """Posterior mean (n*, D) and variance (n*, 1) at Xnew (reference gpr.py:91-136).  numpy in -> numpy out,
        CUDA tensor in -> CUDA tensors out.  `batch` is accepted for compatibility; no chunking is needed (and the
        reference's silent drop of the last n* mod 10000 points, SURVEY Q6, is not reproduced)."""
        assert not full_output_cov
        if full_cov:
            raise NotImplementedError
        alpha, S, info = self.posterior_weights()
        xs = ops.to_device(Xnew).reshape(-1)
        v = hyper_value(self.kernel.variance)
        if alpha.dim() == 1:
            mean, var = ops.predict_1d(xs, self.basis, alpha, S, v)
            mean = mean.view(-1, 1)
        else:
            cols = [ops.predict_1d(xs, self.basis, a_d, S, v) for a_d in alpha]
            mean, var = torch.stack([c[0] for c in cols], 1), cols[0][1]
        if info.any().item():
            raise np.linalg.LinAlgError("banded Cholesky failed in predict_f")
        return _like_input(Xnew, mean, var.view(-1, 1))


class GPR_1d_many:
    """S independent 1-D regressions (GPR_1d each) that share one B-spline basis and one Matern kind, fitted together.

    data = (X[N, 1], y[N] or y[N, 1]) holds all series concatenated, sorted by series: series s is rows offsets[s] ..
    offsets[s+1] - 1 (offsets: host array or tensor of S + 1 integers, 0 first, non-decreasing, N last; empty series are
    allowed).  X and y are CUDA tensors or host arrays (copied to the device once), float32 or float64.  One O(N) pass fills one
    packed accumulator per series (asvgp_accum_1d_segmented); every later step evaluates up to 64 series per batch of launches,
    each slot reading its own series' accumulator, with the bits of GPR_1d on that series alone.

    Per-series parameters are the unconstrained array U[S, 3] in the order (variance, lengthscale, sigma2), initialised from the
    template `kernel` and Gaussian() (or from U0); `variance`, `lengthscales` and `noise_variance` read them back constrained.
    An empty series has ELBO 0, gradient 0 and predicts the prior."""

    def __init__(self, data, offsets, kernel, basis, check_inputs=True, chunks=0, U0=None):
        if _dist.is_distributed("auto"):
            raise NotImplementedError("GPR_1d_many runs on one GPU; torch.distributed is initialised with world size > 1")
        self._kind = kernel_kind(kernel)
        X, y = data
        if X.ndim == 2:
            assert X.shape[1] == 1
        _output_columns(y, "GPR_1d_many", 1, NotImplementedError)   # one column per series
        n = int(X.shape[0])
        if int(y.shape[0]) != n:
            raise ValueError("X and y must have the same number of rows")
        self._offsets = ops.validate_offsets(offsets, n)
        self.num_series = S = self._offsets.size - 1
        self._counts = np.diff(self._offsets)
        if check_inputs and n:
            _check_domain(X.reshape(-1, 1), [basis])
        self.kernel = kernel
        self.basis = basis
        self.inducing_features = SplineFeatures1D(kernel, basis)
        self._chunks = chunks
        # transforms of the three per-series parameters (value_at / dvalue_dunconstrained_at of these templates)
        self._params = [Parameter(hyper_value(kernel.variance), name="variance"),
                        Parameter(hyper_value(kernel.lengthscales), name="lengthscales"), Gaussian().variance]
        if U0 is None:
            self.U = np.tile([p.unconstrained for p in self._params], (S, 1))
        else:
            self.U = np.array(U0, dtype=np.float64)
            if self.U.shape != (S, 3) or not np.isfinite(self.U).all():
                raise ValueError("U0 must be finite [%d, 3], got shape %s" % (S, self.U.shape))
        self._acc = ops.accum_1d_segmented(X.reshape(-1), y.reshape(-1), self._offsets, basis)

    @property
    def variance(self):
        return _values_at(self._params, self.U)[:, 0]

    @property
    def lengthscales(self):
        return _values_at(self._params, self.U)[:, 1]

    @property
    def noise_variance(self):
        return _values_at(self._params, self.U)[:, 2]

    def _evaluate(self, U, ids):
        """(loss[n], grad[n, 3], info[n]) of series ids[i] at unconstrained U[i]: -ELBO and its gradient in U, as
        GPR_1d.training_loss_and_gradients on that series alone.  A failed factorisation gives loss +inf, NaN gradients and its
        pivot in info; an empty series gives 0, 0."""
        U = np.asarray(U, dtype=np.float64).reshape(-1, 3)
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        n = ids.size
        loss, grad, info = np.zeros(n), np.zeros((n, 3)), np.zeros(n, dtype=np.int64)
        live = np.flatnonzero(self._counts[ids] > 0)
        outs = []
        for c in range(0, live.size, _lib.MAX_BATCH):
            sel = live[c: c + _lib.MAX_BATCH]
            vals = _values_at(self._params, U[sel])
            Kuu, dKuu = self.inducing_features.make_Kuu_device_batched(self.kernel, vals[:, 1], vals[:, 0], want_grad=True)
            outs.append(ops.elbo_grad_1d_batched(Kuu, dKuu, self._acc, self.basis, vals[:, 0], vals[:, 2], chunks=self._chunks,
                                                 rows=ids[sel])[:, 0])
        if not outs:
            return loss, grad, info
        out = torch.cat(outs).cpu().numpy()           # one device-to-host copy per call
        bounds = [(o[Bound1D.ELBO], o[Bound1D.GRAD], o[Bound1D.INFO]) for o in out]
        loss[live], grad[live], info[live] = _losses(bounds, self._params, U[live])
        return loss, grad, info

    def training_loss_and_gradients(self):
        """(loss[S], grad[S, 3], info[S]) at the current U: -ELBO of every series and its gradient in U."""
        return self._evaluate(self.U, np.arange(self.num_series))

    def elbo(self):
        """ELBO of every series [S] (-inf where the factorisation fails)."""
        return -self.training_loss_and_gradients()[0]

    def optimize(self, method="L-BFGS-B", wave=256, **scipy_kwargs):
        """One L-BFGS-B (scipy) per series from the current U, in waves of at most `wave` series whose runs advance in lockstep
        (lockstep_minimize): each round evaluates the running series 64 at a time.  Every run takes the iterates of a serial
        run on its series.  A failing series ends with fun = +inf and keeps its starting U; the others go on.  Sets U and
        returns the S results."""
        from .optimizers import lockstep_minimize

        S = self.num_series
        results = [None] * S
        for w0 in range(0, S, int(wave)):
            ids = np.arange(w0, min(S, w0 + int(wave)))
            res = lockstep_minimize(lambda Uw, idx, ids=ids: self._evaluate(Uw, ids[idx]), self.U[ids], method=method,
                                    pass_ids=True, **scipy_kwargs)
            for s, r in zip(ids, res):
                results[s] = r
                if np.isfinite(r.fun):
                    self.U[s] = r.x
        return results

    def posterior_weights(self):
        """(alpha [S, m], S_band [S, k+1, m], info [S, 2]) on the device at the current U (zeros for empty series)."""
        k, m, S = self.basis.order, self.basis.m, self.num_series
        dev = self._acc.device
        alpha = torch.zeros((S, m), dtype=torch.float64, device=dev)
        S_band = torch.zeros((S, k + 1, m), dtype=torch.float64, device=dev)
        info = torch.zeros((S, 2), dtype=torch.float64, device=dev)
        live = np.flatnonzero(self._counts > 0)
        for c in range(0, live.size, _lib.MAX_BATCH):
            sel = live[c: c + _lib.MAX_BATCH]
            vals = _values_at(self._params, self.U[sel])
            Kuu, _ = self.inducing_features.make_Kuu_device_batched(self.kernel, vals[:, 1], vals[:, 0], want_grad=False)
            a, sb, inf = ops.posterior_1d_batched(Kuu, self._acc, self.basis, vals[:, 2], sel, chunks=self._chunks)
            idx = torch.from_numpy(sel).to(dev)
            alpha[idx], S_band[idx], info[idx] = a, sb, inf
        return alpha, S_band, info

    def predict_f(self, Xnew, offsets_new):
        """Posterior mean (n*, 1) and variance (n*, 1) of every series at its test points: rows offsets_new[s] ..
        offsets_new[s+1] - 1 of Xnew belong to series s.  numpy in -> numpy out, CUDA tensor in -> CUDA tensors out."""
        alpha, S_band, info = self.posterior_weights()
        variances = torch.from_numpy(self.variance).to(alpha.device)
        mean, var = ops.predict_1d_segmented(ops.to_device(Xnew).reshape(-1), offsets_new, self.basis, alpha, S_band, variances)
        if info.any().item():
            raise np.linalg.LinAlgError("banded Cholesky failed in predict_f")
        return _like_input(Xnew, mean.view(-1, 1), var.view(-1, 1))


class _PerDimension(_ModelBase):
    """What GPR_kron and GPR_additive share: a kernel, a basis and a banded Kuu factor per input dimension."""

    @property
    def trainable_variables(self):
        out = []
        for k in self.kernels:
            out += [k.variance, k.lengthscales]
        return _unique(out + [self.likelihood.variance])

    def _factors(self, want_grad, defer=False):
        """Per-dimension Kuu factors, their lengthscale derivatives, and the bands of their inverses.  The banded
        inversions run on side streams so that they overlap the factorisation of P; with `defer` the caller joins them
        itself (`self._join()`) right before it reads the bands."""
        Ks, dKs = [], []
        for feat, kern in zip(self.inducing_features, self.kernels):
            K, dK = feat.make_Kuu_device(kern, want_grad=True)
            Ks.append(K); dKs.append(dK)
        Ss, dSs, scals, self._join = ops.band_inverses_beside(Ks, dKs, self.bases)
        if not defer:
            self._join()
        return Ks, dKs, Ss, dSs, scals


def _kron_column_bound(N, s2, v, m1, m2, sc1, sc2, logdetP, Q, yy, T, want_grad):
    """ELBO of the Kronecker model for one output column and, with want_grad, its derivatives: [elbo] or [elbo, v1, l1, v2,
    l2, sigma2]; sc_i = {log|K_i|, dlog|K_i|, ...}, T = the 11 slots of asvgp_kron_terms.  Returns (that row, log|Kuu|)."""
    M = m1 * m2
    logdetK = m2 * sc1[0] + m1 * sc2[0]                       # log|K1 (x) K2|
    tr = T[8]
    v12 = v[0] * v[1]
    elbo = (-0.5 * N * np.log(2 * np.pi * s2) - 0.5 * logdetP + 0.5 * logdetK - 0.5 * yy / s2
            + 0.5 * Q / s2**2 - 0.5 * N * v12 / s2 + 0.5 * tr / s2)
    if not want_grad:
        return np.array([elbo]), logdetK
    trPG, trPdK1, trPdK2, trPK = T[0:4]
    xGx, xdK1x, xdK2x, xKx = T[4:8]
    d_l1 = -0.5 * trPdK1 + 0.5 * m2 * sc1[1] - 0.5 * xdK1x / s2**2 + 0.5 * T[9] / s2
    d_l2 = -0.5 * trPdK2 + 0.5 * m1 * sc2[1] - 0.5 * xdK2x / s2**2 + 0.5 * T[10] / s2
    # Kuu is proportional to 1 / (v1 v2): dKuu/dv_i = -Kuu / v_i
    common = 0.5 * trPK - 0.5 * M + 0.5 * xKx / s2**2 + 0.5 * tr / s2
    d_v1 = common / v[0] - 0.5 * N * v[1] / s2
    d_v2 = common / v[1] - 0.5 * N * v[0] / s2
    d_s2 = (-0.5 * N / s2 + 0.5 * trPG / s2**2 + 0.5 * yy / s2**2 + 0.5 * xGx / s2**4 - Q / s2**3
            + 0.5 * N * v12 / s2**2 - 0.5 * tr / s2**2)
    return np.array([elbo, d_v1, d_l1, d_v2, d_l2, d_s2]), logdetK


def _kron_shared(N, s2, v, T):
    """The terms -N v1 v2 / (2 s2) + trace / (2 s2) of one column's bound, which count once for all output columns, and
    their derivatives: [T, v1, l1, v2, l2, sigma2].  trace = T[8] is proportional to v1 v2 (S_i = K_i^-1 is proportional
    to v_i)."""
    T0 = 0.5 * (-N * v[0] * v[1] + T[8]) / s2
    return np.array([T0, 0.5 * (-N * v[1] + T[8] / v[0]) / s2, 0.5 * T[9] / s2, 0.5 * (-N * v[0] + T[8] / v[1]) / s2,
                     0.5 * T[10] / s2, -T0 / s2])


class GPR_kron(_PerDimension):
    """Collapsed-bound sparse GP regression on 2-D inputs with Kronecker-structured B-spline inducing features
    (reference gpr.py:239-359).  Same constructor, attributes and methods; what differs is only *how*:

      * the reference materialises the Khatri-Rao Kuf ((k+1)^2 N non-zeros), KufKfu as a DENSE M x M matrix and
        factorises P densely (gpr.py:268-272, 293) — infeasible at M = 200 x 200.  Here the O(N) pass accumulates
        per-cell polynomial moments (asvgp_accum_2d) that expand into the (k+1)(2k+1)-row stencil of KufKfu, P is
        factorised as a band of scalar bandwidth k (m2 + 1) = `self.bandwidth` (gpr.py:262), and everything else
        the bound, its gradients and the predictor need from P^-1 / Kuu^-1 are entries on the stencil pattern and
        the bands of K1^-1, K2^-1 (SURVEY §8(a) a14, a15);
      * `elbo_and_grad()` returns the five hyper-parameter derivatives with the bound (the reference gets them from
        TF reverse mode through the dense factorisations);
      * with torch.distributed initialised the data passed in are this rank's shard: the packed accumulator
        [G stencil | Kuf_y | sum y^2 | N] is all-reduced once, the factorisation is replicated.
    """

    n_outputs = 1           # output columns (y[N, D]); class defaults for objects assembled without the constructor
    _extra = None

    def __init__(self, data, kernels, bases, distributed="auto", check_inputs=True, method=None, raster_shape=None):
        """raster_shape=(n1, n2): the caller's statement that X is np.meshgrid(x1, x2, indexing="ij") flattened (x1 slow),
        the eNATL60-shaped input — skips the on-device input classification (a wrong statement is slow, never wrong).
        X[n, 2] and y may each be float32 or float64 (CUDA tensors or host arrays) and are read as they are; the model
        equals the one built from the float64-converted data up to summation order.
        y[n, D] (D <= ops.MAX_RHS, method "nd"): D output columns on the same points share one factorisation of P per step;
        the bound is the reference's multi-output bound (as GPR_1d), predict_f returns means (n*, D) and variances (n*, 1)."""
        X, y = data
        self.X, self.y = X, y
        self.n = X.shape[0]
        self._method = method          # None: ops.KRON_METHOD ("nd" nested-dissection fronts; "band": tile DAG over the band)
        self.d = X.shape[1]

        # Check dimensionality of inputs / valid kernels (reference gpr.py:247-252)
        assert len(kernels) == len(bases) == self.d
        y, n_out = _output_columns(y, "GPR_kron", ops.MAX_RHS)
        self.n_outputs = n_out
        if n_out > 1 and (method or ops.KRON_METHOD) != "nd":
            raise NotImplementedError("several output columns need method='nd' (the scalar-band method takes one column)")
        self._kinds = [kernel_kind(k) for k in kernels]
        if self.d != 2:
            raise NotImplementedError("GPR_kron is implemented for d = 2 (as reference utils.py:57)")
        if check_inputs and self.n:
            _check_domain(X, bases)

        self.kernel = kernels[-1]               # the reference hands the last loop kernel to GPModel (SURVEY Q8)
        self.likelihood = Gaussian()
        self.mean_function = None
        self.num_latent_gps = 1
        self.bases = list(bases)
        self.kernels = list(kernels)

        # Bandwidth (reference gpr.py:260-262; equals order * (m2 + 1) for d = 2)
        self.m = self.bases[0].m
        self.order = self.bases[0].order
        self.bandwidth = self.order * (self.bases[1].m + 1)

        self.inducing_features = [SplineFeatures1D(self.kernels[i], self.bases[i]) for i in range(self.d)]

        # Precompute static quantities (reference gpr.py:268-274): one fused pass over this rank's points
        dev = ops.device()
        if raster_shape is not None:
            assert int(raster_shape[0]) * int(raster_shape[1]) == self.n, "raster_shape does not match the number of points"
        row_len = None if raster_shape is None else int(raster_shape[1])
        if n_out == 1:
            self._acc = torch.zeros(ops.accum_size_2d(self.bases), dtype=torch.float64, device=dev)
            _, _, scal = ops.split_accum_2d(self._acc, self.bases)
            cellmom = ops.moment_table_2d(self.bases)
            if isinstance(X, torch.Tensor) and X.is_cuda:
                if raster_shape is not None:
                    ops.accum_2d(X, y.reshape(-1), self.bases, cellmom, scal, raster_row_len=row_len)
                else:
                    ops.accum_2d(X, y.reshape(-1), self.bases, cellmom, scal, binned="auto")
            else:
                ops.accum_2d_host(X, y, self.bases, cellmom, scal, raster_row_len=row_len)
            ops.expand_moments_2d(cellmom, self.bases, self._acc)
            del cellmom
            self._distributed = _dist.is_distributed(distributed)
            if self._distributed:
                _dist.allreduce_packed(self._acc)
            self._extra = None
        else:
            self._accumulate_columns(X, y, dev, row_len)
            self._distributed = _dist.is_distributed(distributed)
            if self._distributed:               # ONE collective over the packed accumulator and the other columns' [b_d | sum y_d^2 | N]
                _dist.allreduce_packed(self._packed)
        self._Gs, self._b, self._scal = ops.split_accum_2d(self._acc, self.bases)

    def _accumulate_columns(self, X, y, dev, row_len):
        """O(N) pass for D > 1 output columns: column 0 gives G, b_1 and its scalars exactly as a single-column model; every
        further column is accumulated into a scratch moment table of its own, of which only b_d and (sum y_d^2, N) are kept.
        All of it lives in one packed buffer [accumulator | (b_d, sum y_d^2, N) for d = 2 ... D] (one all-reduce)."""
        n_out, M = self.n_outputs, self.bases[0].m * self.bases[1].m
        na = ops.accum_size_2d(self.bases)
        self._packed = torch.zeros(na + (n_out - 1) * (M + 2), dtype=torch.float64, device=dev)
        self._acc = self._packed[:na]
        self._extra = self._packed[na:].view(n_out - 1, M + 2)
        accs = [self._acc] + [torch.zeros(na, dtype=torch.float64, device=dev) for _ in range(n_out - 1)]
        scals = [ops.split_accum_2d(a, self.bases)[2] for a in accs]
        cellmoms = [ops.moment_table_2d(self.bases) for _ in range(n_out)]
        if isinstance(X, torch.Tensor) and X.is_cuda:
            binned = False if row_len else ops.choose_binned_2d(X, self.bases)     # the order of X is probed once
            for d in range(n_out):
                yd = y[:, d].contiguous()
                ops.accum_2d(X, yd, self.bases, cellmoms[d], scals[d], binned=binned, raster_row_len=row_len)
        else:                   # host data: each chunk of X is staged and sent once for all columns
            ops.accum_2d_host(X, y, self.bases, cellmoms, scals, raster_row_len=row_len)
        for d in range(n_out):
            ops.expand_moments_2d(cellmoms[d], self.bases, accs[d])
            if d:
                _, b_d, sc_d = ops.split_accum_2d(accs[d], self.bases)
                self._extra[d - 1, :M].copy_(b_d)
                self._extra[d - 1, M:].copy_(sc_d)

    def _rhs(self):
        """Kuf_y of every output column as one device tensor [D, M]."""
        M = self._b.numel()
        if self._extra is None:
            return self._b.view(1, M)
        return torch.cat([self._b.view(1, M), self._extra[:, :M]], 0)

    def _device_stats(self):
        yy = self._scal[0:1] if self._extra is None else torch.cat([self._scal[0:1], self._extra[:, -2]])
        return self._Gs, self._rhs(), yy, self._scal[1]

    @property
    def KufKfu_sparse(self):
        """Full symmetric KufKfu as a SciPy CSR matrix (reference gpr.py:271)."""
        from . import utils

        return utils.stencil_to_sparse(self._host_stats()[0], self.bases[0].m, self.bases[1].m, self.order)

    @property
    def KufKfu_band(self):
        from . import utils

        return utils.sparse_to_band(self.KufKfu_sparse, self.bandwidth)

    # -- objective ---------------------------------------------------------------------------------------------
    def _evaluate(self, want_grad):
        s2 = hyper_value(self.likelihood.variance)
        v = [hyper_value(k.variance) for k in self.kernels]
        m1, m2 = self.bases[0].m, self.bases[1].m
        D = self.n_outputs
        ws = ops.kron_workspace(m1, m2, self.order, getattr(self, "_method", None), n_rhs=D)
        Ks, dKs, Ss, dSs, scals = self._factors(want_grad, defer=True)
        ops.kron_factor(Ks[0], Ks[1], self._acc, self.bases, s2, ws, b=self._rhs() if D > 1 else None)
        # (x_d, in ws.x_cols, is only read with want_grad: the value needs no selected inverse)
        SigP = ops.kron_selinv(self.bases, ws)[0] if want_grad else ws.sigma_stencil.zero_()
        self._join()
        # one factorisation, the xT Op x terms per column (slots 0..3 and 8..10 are the same in every column)
        for x_d, terms_d in zip(ws.x_cols, ws.terms_cols):
            ops.kron_terms(SigP, self._acc, x_d, Ks[0], dKs[0], Ks[1], dKs[1], Ss[0], dSs[0], Ss[1], dSs[1], self.bases, terms_d)
        yy_rest = [] if self._extra is None else [self._extra[:, -2]]          # sum(y_d^2) of columns 2 ... D
        packed = torch.cat([scals[0], scals[1], ws.scal, ws.terms_flat, self._scal] + yy_rest).cpu().numpy()   # one D2H read
        sc1, sc2, p = packed[0:4], packed[4:8], 8 + ws.scal.numel()
        logdetP, infoP, Qs = ws.unpack_scal(packed[8:p])
        Ts = packed[p: p + 11 * D].reshape(D, 11); p += 11 * D
        N = packed[p + 1]
        yys = [packed[p], *packed[p + 2:]]
        cols = [_kron_column_bound(N, s2, v, m1, m2, sc1, sc2, logdetP, Qs[d], yys[d], Ts[d], want_grad) for d in range(D)]
        elbo, g, info = _combine_columns([c[0] for c in cols], [infoP, sc1[2], sc2[2]], lambda: _kron_shared(N, s2, v, Ts[0]))
        if info != 0:
            raise np.linalg.LinAlgError("Cholesky failed: non-positive pivot %d" % int(info))
        self.last_terms = dict(log_det_Kuu=cols[0][1], log_det_P=logdetP, quad=float(Qs.sum()), trace=Ts[0][8])
        if not want_grad:
            return float(elbo), None
        grads = _grad_dict([(self.kernels[0].variance, g[0]), (self.kernels[0].lengthscales, g[1]),
                            (self.kernels[1].variance, g[2]), (self.kernels[1].lengthscales, g[3]),
                            (self.likelihood.variance, g[4])])
        return float(elbo), grads

    def elbo_and_grad(self):
        """ELBO (reference gpr.py:282-308) and {id(param): dELBO/dparam} for (v1, l1, v2, l2, sigma^2)."""
        return self._evaluate(True)

    def elbo(self):
        """Variational bound on the log marginal likelihood (reference gpr.py:282-308)."""
        return np.float64(self._evaluate(False)[0])

    def training_loss_and_gradients_batch(self, U, max_slots=None):
        """training_loss_and_gradients at B settings at once, without changing the model's parameters.

        U[B, len(trainable_variables)]: unconstrained values in the order of `trainable_variables` (1 <= B <= 64; 3 columns when
        one kernel object serves both dimensions).  Returns (loss[B], grad[B, len(trainable_variables)], info[B]); row b equals
        training_loss_and_gradients() with the parameters set to U[b] up to the summation order of the factorisation's fp64
        REDs.  info is the first non-zero of the pivots of P and of the two per-dimension factors; such a setting gets loss =
        +inf and NaN gradients (nothing is raised).  All settings share the accumulator: each group of settings is one
        factorisation of P per setting through one plan (asvgp_kron_factor_batched and friends), and its results come back in
        one device-to-host copy.  Groups hold at most `max_slots` settings (default: as many as fit in the free device
        memory; a slot takes ~1.1 GB at 200 x 200, order 3); the results do not depend on the grouping."""
        params = self.trainable_variables
        U = np.asarray(U, dtype=np.float64)
        if U.ndim != 2 or U.shape[1] != len(params):
            raise ValueError("U must be [B, %d] (unconstrained values of trainable_variables), got shape %s"
                             % (len(params), U.shape))
        if not 1 <= U.shape[0] <= _lib.MAX_BATCH:
            raise ValueError("U has %d rows; a batch holds 1..%d settings" % (U.shape[0], _lib.MAX_BATCH))
        if not np.isfinite(U).all():
            raise ValueError("U must be finite")
        if (getattr(self, "_method", None) or ops.KRON_METHOD) != "nd":
            raise NotImplementedError("batched evaluation runs the nested-dissection factorisation (method='nd')")
        vals = _values_at(params, U)
        # columns of vals holding (v1, l1, v2, l2, sigma2); one shared kernel object maps both dimensions to the same columns
        roles = [self.kernels[0].variance, self.kernels[0].lengthscales, self.kernels[1].variance, self.kernels[1].lengthscales,
                 self.likelihood.variance]
        col = [next(j for j, p in enumerate(params) if p is r) for r in roles]
        m1, m2, D = self.bases[0].m, self.bases[1].m, self.n_outputs
        slot_bytes = ops.kron_batch_slot_bytes(m1, m2, self.order, D)
        groups = ops.kron_batch_groups(len(U), slot_bytes, ops.kron_batch_free_bytes(m1, m2, self.order, D), max_slots)
        bounds = []
        for first, n in groups:
            bounds += self._evaluate_batch(vals[first:first + n], col, params)
        return _losses(bounds, params, U)

    def _evaluate_batch(self, vals, col, params):
        """(elbo, grad[len(params)], info) of each row of vals (constrained values of params) through one batch of slots."""
        B = len(vals)
        v1, l1, v2, l2, s2 = (vals[:, c] for c in col)
        m1, m2, D = self.bases[0].m, self.bases[1].m, self.n_outputs
        Ks, dKs = [], []
        for feat, kern, ell, var in zip(self.inducing_features, self.kernels, (l1, l2), (v1, v2)):
            K, dK = feat.make_Kuu_device_batched(kern, ell, var, want_grad=True)
            Ks.append(K); dKs.append(dK)
        Ss, dSs, scals, join = ops.band_inverses_beside(Ks, dKs, self.bases)
        ws = ops.kron_batch_workspace(m1, m2, self.order, D, B)
        ops.kron_factor_batched(Ks[0], Ks[1], self._acc, self.bases, s2, ws, b=self._rhs())
        SigP, x = ops.kron_selinv_batched(self.bases, ws, B)
        join()
        ops.kron_terms_batched(SigP, self._acc, x, Ks[0], dKs[0], Ks[1], dKs[1], Ss[0], dSs[0], Ss[1], dSs[1], self.bases,
                               ws.terms[:B])
        yy_rest = [] if self._extra is None else [self._extra[:, -2]]          # sum(y_d^2) of columns 2 ... D
        packed = torch.cat([scals[0].view(-1), scals[1].view(-1), ws.scal[:B].reshape(-1), ws.terms[:B].reshape(-1), self._scal]
                           + yy_rest).cpu().numpy()                             # one D2H read
        p = 0
        sc1 = packed[p: p + 4 * B].reshape(B, 4); p += 4 * B
        sc2 = packed[p: p + 4 * B].reshape(B, 4); p += 4 * B
        scal = packed[p: p + (2 + D) * B].reshape(B, 2 + D); p += (2 + D) * B        # {log|P|, info, Q_1 ... Q_D} per slot
        Ts = packed[p: p + 11 * D * B].reshape(B, D, 11); p += 11 * D * B
        N = packed[p + 1]
        yys = [packed[p], *packed[p + 2:]]
        roles = [self.kernels[0].variance, self.kernels[0].lengthscales, self.kernels[1].variance, self.kernels[1].lengthscales,
                 self.likelihood.variance]
        out = []
        for b in range(B):
            infos = [scal[b, 1], sc1[b, 2], sc2[b, 2]]
            if any(i != 0 for i in infos):
                out.append((np.nan, np.full(len(params), np.nan), next(i for i in infos if i != 0)))
                continue
            v = [v1[b], v2[b]]
            cols = [_kron_column_bound(N, s2[b], v, m1, m2, sc1[b], sc2[b], scal[b, 0], scal[b, 2 + d], yys[d], Ts[b, d], True)
                    for d in range(D)]
            elbo, g, info = _combine_columns([c[0] for c in cols], infos, lambda: _kron_shared(N, s2[b], v, Ts[b, 0]))
            gd = _grad_dict(zip(roles, g))
            out.append((elbo, np.array([gd[id(p)] for p in params]), info))
        return out

    # -- prediction ----------------------------------------------------------------------------------------------
    def posterior_weights(self):
        """(alpha, SigP stencil, S1, S2) on the device: alpha = P^-1 Kuf_y / sigma2 ([D, M] for D > 1 output columns),
        SigP = stencil entries of P^-1, S_i = band(K_i^-1)."""
        s2 = hyper_value(self.likelihood.variance)
        D = self.n_outputs
        ws = ops.kron_workspace(self.bases[0].m, self.bases[1].m, self.order, getattr(self, "_method", None), n_rhs=D)
        Ks, _, Ss, _, scals = self._factors(False)
        ops.kron_factor(Ks[0], Ks[1], self._acc, self.bases, s2, ws, b=self._rhs() if D > 1 else None)
        SigP, x = ops.kron_selinv(self.bases, ws)
        info = torch.stack([ws.info, scals[0][2], scals[1][2]])
        return x / s2, SigP, Ss[0], Ss[1], info

    def _hyper_state(self):
        return tuple(hyper_value(p) for p in self.trainable_variables)

    def posterior_table(self):
        """Per-cell polynomial form of the posterior (device table of asvgp_predict_2d_prepare), cached until a
        hyper-parameter changes: the reference's scripts predict in chunks of 10 000 points (eNATL60.py:96-102), and
        every chunk after the first reuses the factorisation, the selected inverse and this table."""
        state = self._hyper_state()
        cached = getattr(self, "_table", None)
        if cached is None or cached[0] != state:
            alpha, SigP, S1, S2, info = self.posterior_weights()
            if self.n_outputs == 1:
                table = ops.predict_2d_prepare(self.bases, alpha, SigP, S1, S2)
            else:                   # one table per output column (the variance part is the same in all of them)
                table = [ops.predict_2d_prepare(self.bases, a_d, SigP, S1, S2) for a_d in alpha]
            if info.any().item():
                raise np.linalg.LinAlgError("Cholesky failed in predict_f")
            self._table = cached = (state, table)
        return cached[1]

    def predict_f(self, Xnew, full_cov=False, full_output_cov=False, raster_shape=None):
        """Posterior mean (n*, D) and variance (n*, 1) at Xnew[n*, 2] (reference gpr.py:310-334).  raster_shape: as in the
        constructor, for gridded test points."""
        assert not full_output_cov
        if full_cov:
            raise NotImplementedError
        table = self.posterior_table()
        prior = hyper_value(self.kernels[0].variance) * hyper_value(self.kernels[1].variance)
        row_len = None if raster_shape is None else int(raster_shape[1])
        if self.n_outputs == 1:
            mean, var = ops.predict_2d_apply(Xnew, self.bases, table, prior, raster_row_len=row_len)
        else:
            Xs = ops.to_device(Xnew)
            cols = [ops.predict_2d_apply(Xs, self.bases, t, prior, raster_row_len=row_len) for t in table]
            mean, var = torch.stack([c[0] for c in cols], 1), cols[0][1]
        return _like_input(Xnew, mean.reshape(mean.shape[0], -1), var.view(-1, 1))

    def predict_f_sparse(self, Xnew, full_cov=False, full_output_cov=False):
        """Same numbers as predict_f (reference gpr.py:336-359 is its CHOLMOD twin)."""
        return self.predict_f(Xnew, full_cov=full_cov, full_output_cov=full_output_cov)


def _additive_column_bound(N, s2, v, vsum, ms, sc, logdetP, logdetK, trace, trn, Q, yy, T, dn, want_grad):
    """ELBO of the additive model for one output column and, with want_grad, its derivatives: [elbo] or [elbo, v_1, l_1, ...,
    v_D, l_D, sigma2]; T[i] = asvgp_additive_terms of P^-1 and this column's x, dn = asvgp_dense_terms."""
    elbo = (-0.5 * N * np.log(2 * np.pi * s2) - 0.5 * logdetP + 0.5 * logdetK - 0.5 * yy / s2
            + 0.5 * Q / s2**2 - 0.5 * N * vsum / s2 + 0.5 * trace / s2)
    if not want_grad:
        return np.array([elbo])
    g = [elbo]
    for i, m in enumerate(ms):
        trPK, trPdK, xKx, xdKx = T[i]
        d_l = -0.5 * trPdK + 0.5 * sc[i, 1] - 0.5 * xdKx / s2**2 + 0.5 * trn[i, 1] / s2
        # K_d is proportional to 1 / v_d: dK_d/dv_d = -K_d / v_d, trace(K_d^-1 G_dd) is proportional to v_d
        d_v = (0.5 * trPK - 0.5 * m + 0.5 * xKx / s2**2 + 0.5 * trn[i, 0] / s2) / v[i] - 0.5 * N / s2
        g += [d_v, d_l]
    trPG, xGx = dn
    d_s2 = (-0.5 * N / s2 + 0.5 * trPG / s2**2 + 0.5 * yy / s2**2 + 0.5 * xGx / s2**4 - Q / s2**3
            + 0.5 * N * vsum / s2**2 - 0.5 * trace / s2**2)
    return np.array(g + [d_s2])


def _additive_shared(N, s2, v, vsum, trace, trn):
    """The terms -N sum(v) / (2 s2) + trace / (2 s2) of one column's bound, which count once for all output columns, and
    their derivatives: [T, v_1, l_1, ..., v_D, l_D, sigma2].  trace(K_d^-1 G_dd) = trn[d, 0] is proportional to v_d."""
    T = 0.5 * (-N * vsum + trace) / s2
    dT = []
    for i in range(len(v)):
        dT += [0.5 * (-N + trn[i, 0] / v[i]) / s2, 0.5 * trn[i, 1] / s2]
    return np.array([T] + dT + [-T / s2])


class GPR_additive(_PerDimension):
    """Collapsed-bound sparse GP regression with an ADDITIVE kernel, f(x) = sum_d f_d(x_d), each f_d on B-spline inducing
    features (reference gpr.py:139-236).  Same constructor, attributes and methods; what differs is only *how*:

      * the reference stacks the per-dimension Kuf and forms KufKfu by a sparse product (gpr.py:172-176).  Here the banded
        diagonal blocks come from the fused 1-D accumulate (asvgp_accum_1d, one pass per dimension) and the dense
        off-diagonal blocks from asvgp_accum_cross (one pass per pair); Kuf is never formed;
      * P = Kuu + KufKfu / sigma2 is dense (sum m_d)^2 — the reference factorises it with tf.linalg.cholesky (gpr.py:192-195).
        Here it is one dense front of the tile-DAG kernels of the Kronecker model (asvgp_dense_factor / asvgp_dense_selinv,
        fp64 tensor cores), which also returns P^-1 Kuf_y and P^-1;
      * trace(Kuu^-1 KufKfu) (gpr.py:209: a dense solve there) only touches the banded diagonal blocks: per dimension
        band(K_d^-1) from asvgp_band_inverse_1d, as in GPR_kron;
      * `elbo_and_grad()` returns the 2 D + 1 derivatives with the bound (TF reverse mode in the reference).
    """

    n_outputs = 1
    _B = None

    def __init__(self, data, kernels, bases, distributed="auto", check_inputs=True):
        X, y = data
        self.X, self.y = X, y
        self.n = X.shape[0]
        self.d = X.shape[1]

        # Check dimensionality of inputs / valid kernels (reference gpr.py:146-152)
        assert len(kernels) == len(bases) == self.d
        y, n_out = _output_columns(y, "GPR_additive", ops.MAX_RHS)
        self.n_outputs = n_out
        self._kinds = [kernel_kind(k) for k in kernels]
        if self.d > 8:
            raise NotImplementedError("GPR_additive is implemented for at most 8 input dimensions")
        if check_inputs and self.n:
            _check_domain(X, bases)

        self.kernel = kernels[-1]               # as the reference: the last loop kernel goes to GPModel (SURVEY Q8)
        self.likelihood = Gaussian()
        self.mean_function = None
        self.num_latent_gps = 1
        self.bases = list(bases)
        self.kernels = list(kernels)
        self.inducing_features = [SplineFeatures1D(self.kernels[i], self.bases[i]) for i in range(self.d)]

        # Bandwidth (reference gpr.py:163-166)
        bandwidths = [basis.order for basis in self.bases]
        assert all(x == bandwidths[0] for x in bandwidths)
        self.bandwidth = self.order = self.bases[0].order

        # Precompute static quantities (reference gpr.py:169-176): D banded passes + D (D - 1) / 2 cross passes
        Xd = ops.to_device(X)
        yall = ops.to_device(y)
        yd = yall[:, 0].contiguous() if n_out > 1 else yall.reshape(-1)
        self._offsets = np.concatenate([[0], np.cumsum([b.m for b in self.bases])]).astype(int)
        self.M = int(self._offsets[-1])
        self._accs = [ops.accum_1d(Xd[:, i].contiguous(), yd, self.bases[i], binned="auto") for i in range(self.d)]
        # further output columns: Kuf_y and sum(y^2) per (dimension, column); G comes from column 0 only
        self._col_accs = [[ops.accum_1d(Xd[:, i].contiguous(), yall[:, c].contiguous(), self.bases[i], binned="auto")
                           for i in range(self.d)] for c in range(1, n_out)]
        self._cross = {}
        for i in range(self.d):
            for j in range(i + 1, self.d):
                self._cross[(i, j)] = ops.accum_cross(Xd, i, j, self.bases[i], self.bases[j])
        self._distributed = _dist.is_distributed(distributed)
        if self._distributed:
            for acc in self._accs + [a for col in self._col_accs for a in col]:
                _dist.allreduce_packed(acc)
            for c in self._cross.values():
                _dist.allreduce_packed(c)
        # dense KufKfu and the stacked Kuf_y
        self._G = torch.zeros((self.M, self.M), dtype=torch.float64, device=Xd.device)
        self._b = torch.empty(self.M, dtype=torch.float64, device=Xd.device)
        for i, (acc, basis) in enumerate(zip(self._accs, self.bases)):
            Gi, bi, scal = ops.split_accum_1d(acc, basis)
            o = int(self._offsets[i])
            ops.additive_put_band(Gi, basis, o, self._G)
            self._b[o: o + basis.m].copy_(bi)
        for (i, j), c in self._cross.items():
            ops.additive_put_cross(c, self._offsets[i], self._offsets[j], self._G)
        self._scal = ops.split_accum_1d(self._accs[0], self.bases[0])[2]          # {sum y^2, N}: the same in every dimension
        self._B, self._yy = None, None
        if n_out > 1:               # right-hand sides [D, M] and sum(y_d^2) per column
            self._B = torch.empty((n_out, self.M), dtype=torch.float64, device=Xd.device)
            self._B[0].copy_(self._b)
            self._yy = torch.empty(n_out, dtype=torch.float64, device=Xd.device)
            self._yy[0:1].copy_(self._scal[0:1])
            for c, accs in enumerate(self._col_accs, start=1):
                for i, (acc, basis) in enumerate(zip(accs, self.bases)):
                    _, bi, scal = ops.split_accum_1d(acc, basis)
                    o = int(self._offsets[i])
                    self._B[c, o: o + basis.m].copy_(bi)
                self._yy[c: c + 1].copy_(ops.split_accum_1d(accs[0], self.bases[0])[2][0:1])
        del self._col_accs
        self._P = torch.empty_like(self._G)

    def _device_stats(self):
        if self._B is None:
            return self._G, self._b.view(1, -1), self._scal[0:1], self._scal[1]
        return self._G, self._B, self._yy, self._scal[1]

    @property
    def KufKfu(self):
        return self._host_stats()[0]

    @property
    def KufKfu_sparse(self):
        import scipy.sparse as sp

        return sp.csr_matrix(self.KufKfu)

    # -- objective ----------------------------------------------------------------------------------------------------------------
    def _factor(self, want_inverse):
        s2 = hyper_value(self.likelihood.variance)
        Ks, dKs, Ss, dSs, scals = self._factors(True, defer=True)   # the short banded chains overlap the dense factorisation
        # P = KufKfu / sigma2 + Kuu  (reference gpr.py:192)
        ops.additive_scale(self._G, s2, self._P)
        for K, basis, o in zip(Ks, self.bases, self._offsets):
            ops.additive_put_band(K, basis, o, self._P, add=True)
        ws = ops.dense_workspace(self.M, self.n_outputs)
        ops.dense_factor(self._P, self._device_stats()[1], ws)
        x, Pinv = ops.dense_selinv(ws) if want_inverse else (None, None)
        self._join()
        return Ks, dKs, Ss, dSs, scals, ws, x, Pinv

    def _evaluate(self, want_grad):
        s2 = hyper_value(self.likelihood.variance)
        v = [hyper_value(k.variance) for k in self.kernels]
        Ks, dKs, Ss, dSs, scals, ws, x, Pinv = self._factor(want_grad)
        D, R = self.d, self.n_outputs
        dev = self._G.device
        xs = ws.x_cols if want_grad else [None] * R
        # trace(Kuu^-1 KufKfu) and its lengthscale derivatives: per dimension, on the bands
        tr = torch.zeros((D, 4), dtype=torch.float64, device=dev)         # sum S_d .* G_dd, sum dS_d .* G_dd, -, -
        terms = torch.zeros((R, D, 4), dtype=torch.float64, device=dev)  # per output column: the x-dependent terms
        dense = torch.zeros((R, 2), dtype=torch.float64, device=dev)
        zero_x = torch.zeros(self.M, dtype=torch.float64, device=dev)
        for i, (basis, o) in enumerate(zip(self.bases, self._offsets)):
            # (the same contraction kernel with S := KufKfu's diagonal block and K := band(K_d^-1))
            ops.additive_terms(self._G, zero_x, o, basis, Ss[i], dSs[i], tr[i])
            if want_grad:
                for c in range(R):
                    ops.additive_terms(Pinv, xs[c], o, basis, Ks[i], dKs[i], terms[c, i])
        if want_grad:
            for c in range(R):
                ops.dense_terms(Pinv, self._G, xs[c], dense[c])
        packed = torch.cat([torch.stack(scals).reshape(-1), ws.scal, tr.reshape(-1), terms.reshape(-1), dense.reshape(-1),
                            self._scal, self._device_stats()[2]]).cpu().numpy()
        sc = packed[: 4 * D].reshape(D, 4); p = 4 * D
        logdetP, infoP, Qs = ws.unpack_scal(packed[p: p + ws.scal.numel()]); p += ws.scal.numel()
        trn = packed[p: p + 4 * D].reshape(D, 4); p += 4 * D
        T = packed[p: p + 4 * D * R].reshape(R, D, 4); p += 4 * D * R
        dn = packed[p: p + 2 * R].reshape(R, 2); p += 2 * R
        N = packed[p + 1]; p += 2
        yys = packed[p: p + R]
        logdetK = float(sc[:, 0].sum())
        trace = float(trn[:, 0].sum())
        vsum = float(np.sum(v))
        ms = [basis.m for basis in self.bases]
        cols = [_additive_column_bound(N, s2, v, vsum, ms, sc, logdetP, logdetK, trace, trn, Qs[c], yys[c], T[c], dn[c],
                                       want_grad) for c in range(R)]
        elbo, g, info = _combine_columns(cols, [infoP] + list(sc[:, 2]),
                                         lambda: _additive_shared(N, s2, v, vsum, trace, trn))
        if info != 0:
            raise np.linalg.LinAlgError("Cholesky failed: non-positive pivot %d" % int(info))
        self.last_terms = dict(log_det_Kuu=logdetK, log_det_P=logdetP, quad=float(Qs.sum()), trace=trace)
        if not want_grad:
            return float(elbo), None
        pairs = []
        for i, kern in enumerate(self.kernels):
            pairs += [(kern.variance, g[2 * i]), (kern.lengthscales, g[2 * i + 1])]
        pairs.append((self.likelihood.variance, g[2 * D]))
        return float(elbo), _grad_dict(pairs)

    def elbo_and_grad(self):
        """ELBO (reference gpr.py:181-210) and {id(param): dELBO/dparam} for (v_1, l_1, ..., v_D, l_D, sigma^2)."""
        return self._evaluate(True)

    def elbo(self):
        return np.float64(self._evaluate(False)[0])

    # -- prediction -----------------------------------------------------------------------------------------------------------------
    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        """Posterior mean (n*, R) and variance (n*, 1) at Xnew[n*, D] for R output columns (reference gpr.py:212-236)."""
        assert not full_output_cov
        if full_cov:
            raise NotImplementedError
        s2 = hyper_value(self.likelihood.variance)
        Ks, dKs, Ss, dSs, scals, ws, x, Pinv = self._factor(True)
        info = torch.stack([ws.info] + [s[2] for s in scals])
        Xs = ops.to_device(Xnew)
        assert Xs.dim() == 2 and Xs.shape[1] == self.d
        prepared = ops.predict_additive_prepare(self.bases, self._offsets, Ss)
        alphas = x / s2
        prior = float(sum(hyper_value(k.variance) for k in self.kernels))
        cols = [ops.predict_additive(Xs, self.bases, prepared, alpha, Pinv, prior)          # one pass per output column
                for alpha in alphas.view(self.n_outputs, self.M)]
        if info.any().item():
            raise np.linalg.LinAlgError("Cholesky failed in predict_f")
        return _like_input(Xnew, torch.stack([c[0] for c in cols], 1), cols[0][1].view(-1, 1))
