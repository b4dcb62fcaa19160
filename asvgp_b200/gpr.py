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
from .kernels import Gaussian, Parameter, hyper_value, kernel_kind


class _ModelBase:
    """The slice of gpflow.models.GPModel + InternalDataTrainingLossMixin the reference's scripts use."""

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
            lo, hi = (torch.aminmax(X) if isinstance(X, torch.Tensor) else (X.min(), X.max()))
            assert float(lo) > basis.a
            assert float(hi) < basis.b

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
        self._host = None
        self._outs = [torch.empty(16, dtype=torch.float64, device=self._acc.device) for _ in self._accs]
        self._out = self._outs[0]

    # -- the reference's cached attributes (host copies, fetched lazily) --------------------------------------
    def _host_stats(self):
        if self._host is None:
            parts = [ops.split_accum_1d(acc, self.basis) for acc in self._accs]
            b = torch.stack([p[1] for p in parts], 1).cpu().numpy()
            scal = self._scal.cpu().numpy().copy()
            scal[0] = float(sum(p[2][0] for p in parts).item())
            self._host = (self._G.cpu().numpy(), b, scal)
        return self._host

    @property
    def KufKfu(self):
        return self._host_stats()[0]

    @property
    def Kuf_y(self):
        return self._host_stats()[1]

    @property
    def tr_yTy(self):
        return float(self._host_stats()[2][0])

    @property
    def num_data(self):
        """Global number of datapoints (all shards)."""
        return int(self._host_stats()[2][1])

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
    def _combine_columns(outs, v, s2, n):
        """Bound for D output columns from the D single-column evaluations outs[D, 16] at variance v, sigma2 s2 and n data
        points (v, s2, n are only read for D > 1).  The reference scales the log-dets by D and sums the data-fit terms over
        columns, but counts -sum(K_diag)/2s2 + trace/2s2 ONCE (gpr.py:81-87); summing the columns counts it D times, so
        D - 1 copies of T = (-N v + trace)/(2 s2) are taken out again: dT/dv = (-N + trace/v)/(2 s2) (trace is linear in
        v), dT/dl = (dtrace/dl)/(2 s2), dT/ds2 = -T/s2."""
        out = outs[0].copy()
        extra = len(outs) - 1
        if extra:
            tr, dtr_dl = out[7], out[15]
            T = 0.5 * (-n * v + tr) / s2
            out[0:4] = outs[:, 0:4].sum(0) - extra * np.array([T, 0.5 * (-n + tr / v) / s2, 0.5 * dtr_dl / s2, -T / s2])
            out[6] = outs[:, 6].sum()
            bad = outs[:, 8][outs[:, 8] != 0]
            out[8] = bad[0] if bad.size else 0.0
        return out

    def _combine_outputs(self):
        outs = torch.stack(self._outs).cpu().numpy()
        if len(outs) == 1:
            return self._combine_columns(outs, None, None, None)
        v, s2 = hyper_value(self.kernel.variance), hyper_value(self.likelihood.variance)
        return self._combine_columns(outs, v, s2, float(self._scal[1].item()))

    def _grads(self, out):
        return _grad_dict([(self.kernel.variance, out[1]), (self.kernel.lengthscales, out[2]),
                           (self.likelihood.variance, out[3])])

    def elbo_and_grad(self):
        """ELBO (reference gpr.py:49-89) and {id(param): dELBO/dparam} for variance, lengthscales, sigma^2."""
        self._launch_elbo()
        out = self._combine_outputs()
        if out[8] != 0:
            raise np.linalg.LinAlgError("banded Cholesky failed: non-positive pivot %d" % int(out[8]))
        grads = self._grads(out)
        self.last_terms = dict(log_det_Kuu=out[4], log_det_P=out[5], quad=out[6], trace=out[7])
        return float(out[0]), grads

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
        vals = np.array([[p.value_at(float(u)) for p, u in zip(params, row)] for row in U])
        var, ell, s2 = vals[:, 0], vals[:, 1], vals[:, 2]
        Kuu, dKuu = self.inducing_features.make_Kuu_device_batched(self.kernel, ell, var, want_grad=True)
        if self._acc_batch is None:
            self._acc_batch = self._acc.view(1, -1) if len(self._accs) == 1 else torch.stack(self._accs)
        D = len(self._accs)
        if D > 1 and self._n_host is None:
            self._n_host = float(self._scal[1].item())
        outs = ops.elbo_grad_1d_batched(Kuu, dKuu, self._acc_batch, self.basis, var, s2, chunks=self._chunks).cpu().numpy()
        B = U.shape[0]
        loss, grad, info = np.empty(B), np.empty((B, len(params))), np.zeros(B, dtype=np.int64)
        for b in range(B):
            out = self._combine_columns(outs[b], var[b], s2[b], self._n_host)
            if out[8] != 0:
                loss[b], grad[b], info[b] = np.inf, np.nan, int(out[8])
                continue
            grads = self._grads(out)
            loss[b] = -float(out[0])
            grad[b] = [-(grads[id(p)] * p.dvalue_dunconstrained_at(float(u))) for p, u in zip(params, U[b])]
        return loss, grad, info

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
        var = var.view(-1, 1)
        if isinstance(Xnew, torch.Tensor) and Xnew.is_cuda:
            return mean, var
        return mean.cpu().numpy(), var.cpu().numpy()


def _kron_column_bound(N, s2, v, m1, m2, sc1, sc2, logdetP, Q, yy, T, want_grad):
    """ELBO of the Kronecker model for one output column and, with want_grad, its derivatives [v1, l1, v2, l2, sigma2];
    sc_i = {log|K_i|, dlog|K_i|, ...}, T = the 11 slots of asvgp_kron_terms.  Returns (elbo, grads or None, log|Kuu|)."""
    M = m1 * m2
    logdetK = m2 * sc1[0] + m1 * sc2[0]                       # log|K1 (x) K2|
    tr = T[8]
    v12 = v[0] * v[1]
    elbo = (-0.5 * N * np.log(2 * np.pi * s2) - 0.5 * logdetP + 0.5 * logdetK - 0.5 * yy / s2
            + 0.5 * Q / s2**2 - 0.5 * N * v12 / s2 + 0.5 * tr / s2)
    if not want_grad:
        return elbo, None, logdetK
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
    return elbo, np.array([d_v1, d_l1, d_v2, d_l2, d_s2]), logdetK


class GPR_kron(_ModelBase):
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
        if y.ndim == 1:
            y = y.reshape(-1, 1)
        n_out = self.n_outputs = int(y.shape[1])
        if not 1 <= n_out <= ops.MAX_RHS:
            raise ValueError("GPR_kron takes 1 ... %d output columns, got %d" % (ops.MAX_RHS, n_out))
        if n_out > 1 and (method or ops.KRON_METHOD) != "nd":
            raise NotImplementedError("several output columns need method='nd' (the scalar-band method takes one column)")
        self._kinds = [kernel_kind(k) for k in kernels]
        if self.d != 2:
            raise NotImplementedError("GPR_kron is implemented for d = 2 (as reference utils.py:57)")
        if check_inputs and self.n:
            for i, basis in enumerate(bases):
                col = X[:, i]
                lo, hi = (torch.aminmax(col) if isinstance(col, torch.Tensor) else (col.min(), col.max()))
                assert float(lo) > basis.a and float(hi) < basis.b, "inputs must lie strictly inside the basis domain"

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
        self._host = None

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

    # -- the reference's cached attributes (host copies, fetched lazily) --------------------------------------
    def _host_stats(self):
        if self._host is None:
            b, scal = self._b.cpu().numpy().reshape(-1, 1), self._scal.cpu().numpy()
            if self._extra is not None:         # (M, D) and the sum of y^2 over all columns (reference gpr.py:274, 78-79)
                extra = self._extra.cpu().numpy()
                M = b.shape[0]
                b = np.concatenate([b, extra[:, :M].T], 1)
                scal = scal.copy()
                scal[0] = scal[0] + extra[:, M].sum()
            self._host = (self._Gs.cpu().numpy(), b, scal)
        return self._host

    def _rhs(self):
        """Kuf_y of every output column as one device tensor [D, M] (D > 1 only)."""
        M = self._b.numel()
        return torch.cat([self._b.view(1, M), self._extra[:, :M]], 0)

    @property
    def Kuf_y(self):
        return self._host_stats()[1]

    @property
    def tr_yTy(self):
        return float(self._host_stats()[2][0])

    @property
    def num_data(self):
        return int(self._host_stats()[2][1])

    @property
    def KufKfu_sparse(self):
        """Full symmetric KufKfu as a SciPy CSR matrix (reference gpr.py:271)."""
        from . import utils

        return utils.stencil_to_sparse(self._host_stats()[0], self.bases[0].m, self.bases[1].m, self.order)

    @property
    def KufKfu_band(self):
        from . import utils

        return utils.sparse_to_band(self.KufKfu_sparse, self.bandwidth)

    @property
    def trainable_variables(self):
        out = []
        for k in self.kernels:
            out += [k.variance, k.lengthscales]
        return _unique(out + [self.likelihood.variance])

    # -- objective ---------------------------------------------------------------------------------------------
    def _factors(self, want_grad, defer=False):
        """Per-dimension Kuu factors, their lengthscale derivatives, and the bands of their inverses.  The two banded
        inversions (one short chain each, ~0.1 ms) run on side streams so that they overlap the factorisation of P;
        with `defer` the caller joins them itself (`_join`) right before it reads the bands."""
        main = torch.cuda.current_stream()
        Ks, dKs, Ss, dSs, scals = [], [], [], [], []
        for feat, kern in zip(self.inducing_features, self.kernels):
            K, dK = feat.make_Kuu_device(kern, want_grad=True)
            Ks.append(K); dKs.append(dK)
        self._side = ops.side_streams(len(self.bases))
        for i, (side, basis) in enumerate(zip(self._side, self.bases)):
            side.wait_stream(main)
            with torch.cuda.stream(side):
                S, dS, sc = ops.band_inverse_1d(Ks[i], dKs[i], basis, slot=1 + i)
            for t in (S, dS, sc):
                t.record_stream(main)
            Ss.append(S); dSs.append(dS); scals.append(sc)
        if not defer:
            self._join()
        return Ks, dKs, Ss, dSs, scals

    def _join(self):
        main = torch.cuda.current_stream()
        for side in self._side:
            main.wait_stream(side)

    def _evaluate(self, want_grad):
        s2 = hyper_value(self.likelihood.variance)
        v = [hyper_value(k.variance) for k in self.kernels]
        m1, m2 = self.bases[0].m, self.bases[1].m
        D = self.n_outputs
        ws = ops.kron_workspace(m1, m2, self.order, getattr(self, "_method", None), n_rhs=D)
        Ks, dKs, Ss, dSs, scals = self._factors(want_grad, defer=True)
        ops.kron_factor(Ks[0], Ks[1], self._acc, self.bases, s2, ws, b=self._rhs() if D > 1 else None)
        if want_grad:
            SigP, x = ops.kron_selinv(self.bases, ws)
        else:
            ws.sigma_stencil.zero_()
            SigP, x = ws.sigma_stencil, ws.rhs[: ws.M * D].view(D, ws.M).squeeze(0)   # x unused for the value
        self._join()
        if D == 1:
            ops.kron_terms(SigP, self._acc, x, Ks[0], dKs[0], Ks[1], dKs[1], Ss[0], dSs[0], Ss[1], dSs[1], self.bases,
                           ws.terms)
            packed = torch.cat([scals[0], scals[1], ws.scal, ws.terms, self._scal]).cpu().numpy()   # one D2H read
            sc1, sc2, scP, T, (yy, N) = packed[0:4], packed[4:8], packed[8:11], packed[11:22], packed[22:24]
            info = scP[2] or sc1[2] or sc2[2]
            if info != 0:
                raise np.linalg.LinAlgError("Cholesky failed: non-positive pivot %d" % int(info))
            elbo, g, logdetK = _kron_column_bound(N, s2, v, m1, m2, sc1, sc2, scP[0], scP[1], yy, T, want_grad)
            self.last_terms = dict(log_det_Kuu=logdetK, log_det_P=scP[0], quad=scP[1], trace=T[8])
        else:
            # one factorisation, the xT Op x terms per column (slots 0..3 and 8..10 are the same in every column)
            for d in range(D):
                ops.kron_terms(SigP, self._acc, x[d], Ks[0], dKs[0], Ks[1], dKs[1], Ss[0], dSs[0], Ss[1], dSs[1], self.bases,
                               ws.terms[d])
            packed = torch.cat([scals[0], scals[1], ws.scal, ws.terms.reshape(-1), self._scal,
                                self._extra[:, -2]]).cpu().numpy()
            sc1, sc2, p = packed[0:4], packed[4:8], 8
            logdetP, info, Qs = packed[p], packed[p + 1], packed[p + 2: p + 2 + D]; p += 2 + D
            Ts = packed[p: p + 11 * D].reshape(D, 11); p += 11 * D
            N = packed[p + 1]
            yys = np.concatenate([[packed[p]], packed[p + 2: p + 1 + D]])
            info = info or sc1[2] or sc2[2]
            if info != 0:
                raise np.linalg.LinAlgError("Cholesky failed: non-positive pivot %d" % int(info))
            cols = [_kron_column_bound(N, s2, v, m1, m2, sc1, sc2, logdetP, Qs[d], yys[d], Ts[d], want_grad) for d in range(D)]
            logdetK, tr = cols[0][2], Ts[0][8]
            # -N v1 v2 / 2 s2 + trace / 2 s2 count once (reference gpr.py:81-87), not once per column: take D - 1 copies of
            # T = (-N v1 v2 + tr) / (2 s2) out again.  tr is proportional to v1 v2 (S_i = K_i^-1 is proportional to v_i).
            T0 = 0.5 * (-N * v[0] * v[1] + tr) / s2
            elbo = sum(c[0] for c in cols) - (D - 1) * T0
            g = None
            if want_grad:
                dT = np.array([0.5 * (-N * v[1] + tr / v[0]) / s2, 0.5 * Ts[0][9] / s2,
                               0.5 * (-N * v[0] + tr / v[1]) / s2, 0.5 * Ts[0][10] / s2, -T0 / s2])
                g = np.sum([c[1] for c in cols], 0) - (D - 1) * dT
            self.last_terms = dict(log_det_Kuu=logdetK, log_det_P=logdetP, quad=float(np.sum(Qs)), trace=tr)
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

    def maximum_log_likelihood_objective(self):
        return self.elbo()

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
        info = torch.stack([ws.scal[2 if D == 1 else 1], scals[0][2], scals[1][2]])
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
        mean, var = mean.reshape(mean.shape[0], -1), var.view(-1, 1)
        if isinstance(Xnew, torch.Tensor) and Xnew.is_cuda:
            return mean, var
        return mean.cpu().numpy(), var.cpu().numpy()

    def predict_f_sparse(self, Xnew, full_cov=False, full_output_cov=False):
        """Same numbers as predict_f (reference gpr.py:336-359 is its CHOLMOD twin)."""
        return self.predict_f(Xnew, full_cov=full_cov, full_output_cov=full_output_cov)


def _additive_column_bound(N, s2, v, vsum, ms, sc, logdetP, logdetK, trace, trn, Q, yy, T, dn, want_grad):
    """ELBO of the additive model for one output column and, with want_grad, its derivatives [v_1, l_1, ..., v_D, l_D,
    sigma2]; T[i] = asvgp_additive_terms of P^-1 and this column's x, dn = asvgp_dense_terms.  Returns (elbo, grads or None)."""
    elbo = (-0.5 * N * np.log(2 * np.pi * s2) - 0.5 * logdetP + 0.5 * logdetK - 0.5 * yy / s2
            + 0.5 * Q / s2**2 - 0.5 * N * vsum / s2 + 0.5 * trace / s2)
    if not want_grad:
        return elbo, None
    g = []
    for i, m in enumerate(ms):
        trPK, trPdK, xKx, xdKx = T[i]
        d_l = -0.5 * trPdK + 0.5 * sc[i, 1] - 0.5 * xdKx / s2**2 + 0.5 * trn[i, 1] / s2
        # K_d is proportional to 1 / v_d: dK_d/dv_d = -K_d / v_d, trace(K_d^-1 G_dd) is proportional to v_d
        d_v = (0.5 * trPK - 0.5 * m + 0.5 * xKx / s2**2 + 0.5 * trn[i, 0] / s2) / v[i] - 0.5 * N / s2
        g += [d_v, d_l]
    trPG, xGx = dn
    d_s2 = (-0.5 * N / s2 + 0.5 * trPG / s2**2 + 0.5 * yy / s2**2 + 0.5 * xGx / s2**4 - Q / s2**3
            + 0.5 * N * vsum / s2**2 - 0.5 * trace / s2**2)
    return elbo, np.array(g + [d_s2])


class GPR_additive(_ModelBase):
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
        if y.ndim == 1:
            y = y.reshape(-1, 1)
        n_out = self.n_outputs = int(y.shape[1])
        if not 1 <= n_out <= ops.MAX_RHS:
            raise ValueError("GPR_additive takes 1 ... %d output columns, got %d" % (ops.MAX_RHS, n_out))
        self._kinds = [kernel_kind(k) for k in kernels]
        if self.d > 8:
            raise NotImplementedError("GPR_additive is implemented for at most 8 input dimensions")
        if check_inputs and self.n:
            for i, basis in enumerate(bases):
                col = X[:, i]
                lo, hi = (torch.aminmax(col) if isinstance(col, torch.Tensor) else (col.min(), col.max()))
                assert float(lo) > basis.a and float(hi) < basis.b, "inputs must lie strictly inside the basis domain"

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
            ops._lib.call("asvgp_additive_put_band", ops._p(Gi), basis.m, basis.order, o, self.M, 1.0, 0, ops._p(self._G), ops._stream())
            self._b[o: o + basis.m].copy_(bi)
        for (i, j), c in self._cross.items():
            ops._lib.call("asvgp_additive_put_cross", ops._p(c), self.bases[i].m, self.bases[j].m, int(self._offsets[i]),
                          int(self._offsets[j]), self.M, ops._p(self._G), ops._stream())
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
        self._host = None

    # -- the reference's cached attributes ------------------------------------------------------------------------------------
    def _host_stats(self):
        if self._host is None:
            if self._B is None:
                self._host = (self._G.cpu().numpy(), self._b.cpu().numpy().reshape(-1, 1), self._scal.cpu().numpy())
            else:                   # Kuf_y (M, D); tr_yTy sums over the columns (reference gpr.py:78-79)
                scal = self._scal.cpu().numpy().copy()
                scal[0] = float(self._yy.sum().item())
                self._host = (self._G.cpu().numpy(), self._B.cpu().numpy().T.copy(), scal)
        return self._host

    @property
    def KufKfu(self):
        return self._host_stats()[0]

    @property
    def KufKfu_sparse(self):
        import scipy.sparse as sp

        return sp.csr_matrix(self.KufKfu)

    @property
    def Kuf_y(self):
        return self._host_stats()[1]

    @property
    def tr_yTy(self):
        return float(self._host_stats()[2][0])

    @property
    def num_data(self):
        return int(self._host_stats()[2][1])

    @property
    def trainable_variables(self):
        out = []
        for k in self.kernels:
            out += [k.variance, k.lengthscales]
        return _unique(out + [self.likelihood.variance])

    # -- objective ----------------------------------------------------------------------------------------------------------------
    def _factor(self, want_inverse):
        s2 = hyper_value(self.likelihood.variance)
        main = torch.cuda.current_stream()
        Ks, dKs, Ss, dSs, scals = [], [], [], [], []
        for feat, kern in zip(self.inducing_features, self.kernels):
            K, dK = feat.make_Kuu_device(kern, want_grad=True)
            Ks.append(K); dKs.append(dK)
        side = ops.side_streams(self.d)
        for i, basis in enumerate(self.bases):                 # short banded chains: overlap them with the dense factorisation
            side[i].wait_stream(main)
            with torch.cuda.stream(side[i]):
                S, dS, sc = ops.band_inverse_1d(Ks[i], dKs[i], basis, slot=1 + i)
            for t in (S, dS, sc):
                t.record_stream(main)
            Ss.append(S); dSs.append(dS); scals.append(sc)
        # P = KufKfu / sigma2 + Kuu  (reference gpr.py:192)
        ops._lib.call("asvgp_additive_scale", ops._p(self._G), self.M, float(s2), ops._p(self._P), ops._stream())
        for i, basis in enumerate(self.bases):
            ops._lib.call("asvgp_additive_put_band", ops._p(Ks[i]), basis.m, basis.order, int(self._offsets[i]), self.M, 1.0, 1,
                          ops._p(self._P), ops._stream())
        ws = ops.dense_workspace(self.M, self.n_outputs)
        ops.dense_factor(self._P, self._b if self._B is None else self._B, ws)
        x, Pinv = ops.dense_selinv(ws) if want_inverse else (None, None)
        for s in side:
            main.wait_stream(s)
        return Ks, dKs, Ss, dSs, scals, ws, x, Pinv

    def _evaluate(self, want_grad):
        s2 = hyper_value(self.likelihood.variance)
        v = [hyper_value(k.variance) for k in self.kernels]
        Ks, dKs, Ss, dSs, scals, ws, x, Pinv = self._factor(want_grad)
        D, R = self.d, self.n_outputs
        dev = self._G.device
        xs = [x] if R == 1 else (list(x) if x is not None else [None] * R)
        # trace(Kuu^-1 KufKfu) and its lengthscale derivatives: per dimension, on the bands
        tr = torch.zeros((D, 4), dtype=torch.float64, device=dev)         # sum S_d .* G_dd, sum dS_d .* G_dd, -, -
        terms = torch.zeros((R, D, 4), dtype=torch.float64, device=dev)  # per output column: the x-dependent terms
        dense = torch.zeros((R, 2), dtype=torch.float64, device=dev)
        zero_x = torch.zeros(self.M, dtype=torch.float64, device=dev)
        for i, basis in enumerate(self.bases):
            o = int(self._offsets[i])
            # (the same contraction kernel with S := KufKfu's diagonal block and K := band(K_d^-1))
            ops._lib.call("asvgp_additive_terms", ops._p(self._G), ops._p(zero_x), self.M, o, basis.m, basis.order, ops._p(Ss[i]),
                          ops._p(dSs[i]), ops._p(tr[i]), ops._stream())
            if want_grad:
                for c in range(R):
                    ops._lib.call("asvgp_additive_terms", ops._p(Pinv), ops._p(xs[c]), self.M, o, basis.m, basis.order,
                                  ops._p(Ks[i]), ops._p(dKs[i]), ops._p(terms[c, i]), ops._stream())
        if want_grad:
            for c in range(R):
                ops._lib.call("asvgp_dense_terms", ops._p(Pinv), ops._p(self._G), ops._p(xs[c]), self.M, ops._p(dense[c]),
                              ops._stream())
        yy_cols = self._scal[0:1] if R == 1 else self._yy
        packed = torch.cat([torch.stack(scals).reshape(-1), ws.scal, tr.reshape(-1), terms.reshape(-1), dense.reshape(-1),
                            self._scal, yy_cols]).cpu().numpy()
        sc = packed[: 4 * D].reshape(D, 4); p = 4 * D
        scP = packed[p: p + ws.scal.numel()]; p += ws.scal.numel()
        trn = packed[p: p + 4 * D].reshape(D, 4); p += 4 * D
        T = packed[p: p + 4 * D * R].reshape(R, D, 4); p += 4 * D * R
        dn = packed[p: p + 2 * R].reshape(R, 2); p += 2 * R
        N = packed[p + 1]; p += 2
        yys = packed[p: p + R]
        # scal layouts of asvgp_dense_factor (one rhs) and asvgp_dense_factor_multi
        logdetP, infoP, Qs = (scP[0], scP[2], scP[1:2]) if R == 1 else (scP[0], scP[1], scP[2:])
        info = infoP or next((s[2] for s in sc if s[2] != 0), 0.0)
        if info != 0:
            raise np.linalg.LinAlgError("Cholesky failed: non-positive pivot %d" % int(info))
        logdetK = float(sc[:, 0].sum())
        trace = float(trn[:, 0].sum())
        vsum = float(np.sum(v))
        ms = [basis.m for basis in self.bases]
        cols = [_additive_column_bound(N, s2, v, vsum, ms, sc, logdetP, logdetK, trace, trn, Qs[c], yys[c], T[c], dn[c],
                                       want_grad) for c in range(R)]
        self.last_terms = dict(log_det_Kuu=logdetK, log_det_P=logdetP, quad=float(np.sum(Qs)) if R > 1 else Qs[0], trace=trace)
        if R == 1:
            elbo, g = cols[0]
        else:
            # -N sum(v) / 2 s2 + trace / 2 s2 count once (reference gpr.py:81-87), not once per column: take R - 1 copies of
            # T = (-N sum(v) + trace) / (2 s2) out again.  trace(K_d^-1 G_dd) is proportional to v_d.
            T0 = 0.5 * (-N * vsum + trace) / s2
            elbo = sum(c[0] for c in cols) - (R - 1) * T0
            if want_grad:
                dT = []
                for i in range(D):
                    dT += [0.5 * (-N + trn[i, 0] / v[i]) / s2, 0.5 * trn[i, 1] / s2]
                g = np.sum([c[1] for c in cols], 0) - (R - 1) * np.array(dT + [-T0 / s2])
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

    def maximum_log_likelihood_objective(self):
        return self.elbo()

    # -- prediction -----------------------------------------------------------------------------------------------------------------
    def predict_f(self, Xnew, full_cov=False, full_output_cov=False):
        """Posterior mean (n*, R) and variance (n*, 1) at Xnew[n*, D] for R output columns (reference gpr.py:212-236)."""
        assert not full_output_cov
        if full_cov:
            raise NotImplementedError
        s2 = hyper_value(self.likelihood.variance)
        Ks, dKs, Ss, dSs, scals, ws, x, Pinv = self._factor(True)
        info = torch.stack([ws.scal[2 if self.n_outputs == 1 else 1]] + [s[2] for s in scals])
        Xs = ops.to_device(Xnew)
        assert Xs.dim() == 2 and Xs.shape[1] == self.d
        n = Xs.shape[0]
        dev = Xs.device
        meshes = torch.cat([ops.device_mesh(b) for b in self.bases])
        meta, koff = [], 0
        for i, b in enumerate(self.bases):
            nk = ops.device_mesh(b).numel()
            meta += [koff, nk, int(self._offsets[i]), b.m]
            koff += nk
        meta = torch.tensor(meta, dtype=torch.int32, device=dev)
        S_all = torch.cat([S.reshape(-1) for S in Ss])
        alphas = x / s2
        prior = float(sum(hyper_value(k.variance) for k in self.kernels))
        cols = []
        for alpha in ([alphas] if self.n_outputs == 1 else list(alphas)):       # one pass per output column
            mean = torch.empty(n, dtype=torch.float64, device=dev)
            var = torch.empty(n, dtype=torch.float64, device=dev)
            ops._lib.call("asvgp_predict_additive", ops._p(Xs), n, self.d, ops._p(meshes), ops._p(meta), self.M, self.order,
                          ops._p(alpha), ops._p(Pinv), ops._p(S_all), prior, ops._p(mean), ops._p(var), ops._stream())
            cols.append((mean, var))
        if info.any().item():
            raise np.linalg.LinAlgError("Cholesky failed in predict_f")
        mean, var = torch.stack([c[0] for c in cols], 1), cols[0][1].view(-1, 1)
        if isinstance(Xnew, torch.Tensor) and Xnew.is_cuda:
            return mean, var
        return mean.cpu().numpy(), var.cpu().numpy()
