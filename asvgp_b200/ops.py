"""Thin Python faces of the C-ABI entry points.  torch is used for device memory and streams only; every
operator below runs a hand-written sm_100a kernel through ctypes (no torch math on the hot path, no CPU
fallback).  Inputs may be numpy arrays, torch tensors or any object exporting `__dlpack__`."""
import ctypes

import numpy as np
import torch

from . import _lib

F64 = torch.float64
F32 = torch.float32
# element-type codes of the typed entry points (ASVGP_F64 / ASVGP_F32 in include/asvgp_b200.h)
ELEM_TYPES = {F64: 0, F32: 1}


_HAVE_CUDA = None
_DEVICES = {}


def device():
    global _HAVE_CUDA
    if _HAVE_CUDA is None:                      # asked once: torch.cuda.is_available() costs microseconds on every call
        _HAVE_CUDA = bool(torch.cuda.is_available())
    if not _HAVE_CUDA:
        raise _lib.AsvgpNativeError("asvgp_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    i = torch.cuda.current_device()
    d = _DEVICES.get(i)
    if d is None:
        d = _DEVICES[i] = torch.device("cuda", i)
    return d


def _as_tensor(a):
    """numpy / torch / DLPack object -> torch tensor (no copy where the source allows, dtype and device unchanged)."""
    if isinstance(a, torch.Tensor):
        return a
    if isinstance(a, np.ndarray):
        return torch.from_numpy(np.ascontiguousarray(a))
    if hasattr(a, "__dlpack__"):
        return torch.from_dlpack(a)
    return torch.as_tensor(np.asarray(a))


def to_device(a, dtype=F64):
    """numpy / torch / DLPack object -> contiguous CUDA tensor of `dtype` on the current device."""
    if isinstance(a, torch.Tensor) and a.is_cuda and a.dtype == dtype and a.is_contiguous() and \
            a.device.index == torch.cuda.current_device():
        return a                                # the hot path's inputs are already where they belong
    return _as_tensor(a).to(device=device(), dtype=dtype).contiguous()


def point_dtype(dtype):
    """The dtype training points are read in: float32 and float64 as they are, anything else converted to float64."""
    return dtype if dtype in ELEM_TYPES else F64


def points_to_device(a):
    """Training points (x, X or y) -> (contiguous CUDA tensor, element-type code).  float32 / float64 data keep their
    dtype, so the accumulate kernels read it without a widened copy (they convert each value in registers, exactly)."""
    t = _as_tensor(a)
    t = to_device(t, dtype=point_dtype(t.dtype))
    return t, ELEM_TYPES[t.dtype]


def points_to_host(a):
    """Host-resident training points -> CPU tensor of their point dtype (no copy for float32 / float64 data)."""
    t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a))
    return t.to(dtype=point_dtype(t.dtype))


def _p(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def _stream():
    # the raw cudaStream_t of torch's current stream (torch.cuda.current_stream() builds a Python Stream object every call)
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))


def device_mesh(basis):
    """The basis' knot mesh as a CUDA tensor (cached on the basis object per device)."""
    dev = device()
    cache = basis.__dict__.setdefault("_dev_mesh", {})
    if dev not in cache:
        cache[dev] = torch.from_numpy(np.ascontiguousarray(basis.mesh, dtype=np.float64)).to(dev)
    return cache[dev]


def basis_eval_1d(X, basis, dx=0):
    """(idx[n] int64, vals[(k+1), n]) as numpy arrays — rows idx+r of Kuf (reference basis.py:51-80)."""
    x = to_device(X).reshape(-1)
    n, k = x.numel(), basis.order
    mesh = device_mesh(basis)
    idx = torch.empty(n, dtype=torch.int64, device=x.device)
    vals = torch.empty((k + 1, n), dtype=F64, device=x.device)
    coef = to_device(basis.piece_coefficients(dx)) if dx > 0 else None
    _lib.call("asvgp_basis_eval_1d", _p(x), n, _p(mesh), mesh.numel(), k, int(dx), _p(coef), _p(idx), _p(vals),
              _stream())
    return idx.cpu().numpy(), vals.cpu().numpy()


def accum_size_1d(basis):
    return (basis.order + 2) * basis.m + 2


BINNED_MIN_POINTS = 1 << 18      # below this the partition passes cost more than the REDs they save
BINNED_JUMP_FRACTION = 0.05


def order_probe_1d(x, basis):
    """Fraction of sampled neighbour pairs of x that lie more than one knot interval apart (one small D2H read)."""
    x, xt = points_to_device(x)
    x = x.reshape(-1)
    mesh = device_mesh(basis)
    out = torch.empty(1, dtype=F64, device=x.device)
    _lib.call("asvgp_order_probe_1d_typed", _p(x), xt, x.numel(), _p(mesh), mesh.numel(), _p(out), _stream())
    return float(out.item())


def accum_1d(x, y, basis, acc=None, binned=False):
    """Adds sum_n w_n w_n^T (lower band), sum_n w_n y_n, sum y^2 and the count of the points (x, y) into the
    packed accumulator [G_band | b | sum(y^2) | count] (allocated zeroed if None).  Reference gpr.py:39-44.
    binned: False = streaming kernel (any order is exact; fast when consecutive points share knot intervals),
    True = bucket-partition first (inputs in no particular order), "auto" = sample the order on the device and choose
    (one host synchronisation).  x and y may each be float32 or float64 and are read as they are (other dtypes are
    converted to float64); the sums are float64 and equal those of the float64-converted points up to summation order."""
    x, xt = points_to_device(x)
    y, yt = points_to_device(y)
    x, y = x.reshape(-1), y.reshape(-1)
    if x.numel() != y.numel():
        raise ValueError("x and y must have the same number of points")
    mesh = device_mesh(basis)
    if acc is None:
        acc = torch.zeros(accum_size_1d(basis), dtype=F64, device=x.device)
    if binned == "auto":
        binned = x.numel() >= BINNED_MIN_POINTS and order_probe_1d(x, basis) > BINNED_JUMP_FRACTION
    if binned:
        nbytes = _lib.load().asvgp_accum_1d_binned_work_bytes(x.numel())
        work = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        _lib.call("asvgp_accum_1d_binned_typed", _p(x), xt, _p(y), yt, x.numel(), _p(mesh), mesh.numel(), basis.order,
                  _p(acc), _p(work), nbytes, _stream())
        return acc
    _lib.call("asvgp_accum_1d_typed", _p(x), xt, _p(y), yt, x.numel(), _p(mesh), mesh.numel(), basis.order, _p(acc),
              _stream())
    return acc


def split_accum_1d(acc, basis):
    """Views (G_band (k+1, M), b (M,), scal (2,)) into the packed accumulator."""
    k, m = basis.order, basis.m
    return acc[: (k + 1) * m].view(k + 1, m), acc[(k + 1) * m: (k + 2) * m], acc[(k + 2) * m:]


def predict_1d(xnew, basis, alpha, S_band, variance, mean=None, var=None):
    """Posterior mean/variance at xnew from alpha = P^-1 b / sigma2 and S = band(P^-1) - band(Kuu^-1)
    (reference gpr.py:91-136)."""
    x = to_device(xnew).reshape(-1)
    n = x.numel()
    mesh = device_mesh(basis)
    alpha = to_device(alpha).reshape(-1)
    S_band = to_device(S_band)
    if mean is None:
        mean = torch.empty(n, dtype=F64, device=x.device)
    if var is None:
        var = torch.empty(n, dtype=F64, device=x.device)
    _lib.call("asvgp_predict_1d", _p(x), n, _p(mesh), mesh.numel(), basis.order, _p(alpha), _p(S_band),
              float(variance), _p(mean), _p(var), _stream())
    return mean, var


# ---- banded (latency-bound) operators ----------------------------------------------------------------------------------
def workspace_1d(m, order, chunks=0, slot=0):
    """Scratch tensor for elbo_grad_1d / posterior_1d (cached per (device, m, order, chunks, slot); callers that run on
    several streams at once use one slot per stream)."""
    dev = device()
    key = (dev, m, order, chunks, slot)
    ws = _WORKSPACES.get(key)
    if ws is None:
        nbytes = _lib.load().asvgp_workspace_bytes_1d(m, order, chunks)
        if nbytes < 0:
            raise _lib.AsvgpNativeError("asvgp_workspace_bytes_1d rejected m=%d order=%d" % (m, order))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _WORKSPACES[key] = ws
    return ws


_WORKSPACES = {}


def device_tables(basis, names):
    """The named static bands of the basis stacked as one CUDA tensor [len(names), k+1, m] (cached)."""
    dev = device()
    cache = basis.__dict__.setdefault("_dev_tables", {})
    key = (dev, tuple(names))
    if key not in cache:
        stack = np.stack([np.asarray(getattr(basis, n), dtype=np.float64) for n in names])
        cache[key] = torch.from_numpy(np.ascontiguousarray(stack)).to(dev)
    return cache[key]


def kuu_assemble(basis, names, coef, dcoef=None, want_grad=True):
    """Kuu = sum coef[n] * basis.<n> (and its lengthscale derivative) as CUDA bands (reference
    inducing_features.py:12-44)."""
    tables = device_tables(basis, names)
    k, m = basis.order, basis.m
    Kuu = torch.empty((k + 1, m), dtype=F64, device=tables.device)
    dKuu = torch.empty_like(Kuu) if want_grad else None
    c = (ctypes.c_double * len(names))(*[float(v) for v in coef])
    dc = (ctypes.c_double * len(names))(*[float(v) for v in (dcoef if dcoef is not None else [0.0] * len(names))])
    _lib.call("asvgp_kuu_assemble", _p(tables), len(names), ctypes.cast(c, ctypes.c_void_p),
              ctypes.cast(dc, ctypes.c_void_p), m, k, _p(Kuu), _p(dKuu), _stream())
    return Kuu, dKuu


def kuu_assemble_batched(basis, names, coefs, dcoefs=None, want_grad=True):
    """kuu_assemble for B coefficient sets, the rows of coefs / dcoefs [B, len(names)]: (Kuu, dKuu) as [B, k+1, m] CUDA
    bands; slot b equals kuu_assemble(basis, names, coefs[b], dcoefs[b]) bit for bit."""
    tables = device_tables(basis, names)
    k, m, n = basis.order, basis.m, len(names)
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    dcoefs = np.zeros_like(coefs) if dcoefs is None else np.ascontiguousarray(dcoefs, dtype=np.float64)
    if coefs.ndim != 2 or coefs.shape[1] != n or dcoefs.shape != coefs.shape:
        raise ValueError("coefs / dcoefs must be [B, %d], got %s / %s" % (n, coefs.shape, dcoefs.shape))
    B = coefs.shape[0]
    Kuu = torch.empty((B, k + 1, m), dtype=F64, device=tables.device)
    dKuu = torch.empty_like(Kuu) if want_grad else None
    _lib.call("asvgp_kuu_assemble_batched", _p(tables), n, B, ctypes.c_void_p(coefs.ctypes.data),
              ctypes.c_void_p(dcoefs.ctypes.data), m, k, _p(Kuu), _p(dKuu), _stream())
    return Kuu, dKuu


def workspace_1d_batched(m, order, chunks, B, D):
    """Scratch tensor for elbo_grad_1d_batched (cached per (device, m, order, chunks, B, D))."""
    dev = device()
    key = (dev, m, order, chunks, "batched", B, D)
    ws = _WORKSPACES.get(key)
    if ws is None:
        nbytes = _lib.load().asvgp_workspace_bytes_1d_batched(m, order, chunks, B, D)
        if nbytes < 0:
            raise _lib.AsvgpNativeError("asvgp_workspace_bytes_1d_batched rejected m=%d order=%d B=%d D=%d" % (m, order, B, D))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _WORKSPACES[key] = ws
    return ws


def elbo_grad_1d_batched(Kuu, dKuu, accs, basis, variances, sigma2s, chunks=0, out=None):
    """B settings of the bound in one stream of launches: Kuu, dKuu [B, k+1, m] (kuu_assemble_batched), accs [D, L] (D
    packed accumulators, or one [L]), variances / sigma2s [B] on the host.  Returns out [B, D, 16] on the device; out[b, d]
    equals elbo_grad_1d of slot b and column d bit for bit in slots 0..8 and 15 (see include/asvgp_b200.h)."""
    k, m = basis.order, basis.m
    accs = accs.reshape(1, -1) if accs.dim() == 1 else accs
    variances = np.ascontiguousarray(variances, dtype=np.float64).reshape(-1)
    sigma2s = np.ascontiguousarray(sigma2s, dtype=np.float64).reshape(-1)
    B, D = variances.size, accs.shape[0]
    if sigma2s.size != B or tuple(Kuu.shape) != (B, k + 1, m) or tuple(dKuu.shape) != (B, k + 1, m):
        raise ValueError("elbo_grad_1d_batched: %d variances, %d sigma2s, Kuu %s, dKuu %s" % (B, sigma2s.size, tuple(Kuu.shape),
                                                                                            tuple(dKuu.shape)))
    if accs.shape[1] != accum_size_1d(basis) or not accs.is_contiguous():
        raise ValueError("elbo_grad_1d_batched: accs must be contiguous [D, %d]" % accum_size_1d(basis))
    if not 1 <= B <= _lib.MAX_BATCH or not 1 <= D <= _lib.MAX_BATCH_COLUMNS:
        raise ValueError("elbo_grad_1d_batched: B=%d not in 1..%d or D=%d not in 1..%d"
                         % (B, _lib.MAX_BATCH, D, _lib.MAX_BATCH_COLUMNS))
    ws = workspace_1d_batched(m, k, int(chunks), B, D)
    if out is None:
        out = torch.empty((B, D, 16), dtype=F64, device=accs.device)
    _lib.call("asvgp_elbo_grad_1d_batched", _p(Kuu), _p(dKuu), _p(accs), m, k, B, D, ctypes.c_void_p(variances.ctypes.data),
              ctypes.c_void_p(sigma2s.ctypes.data), int(chunks), _p(out), _p(ws), ws.numel(), _stream())
    return out


class KuuChain:
    """Handle of a Kuu chain in flight on the side stream (kuu_chain_1d): its state buffer, the event that marks it
    complete, and the operands it reads (kept alive until the bound has consumed the state)."""
    __slots__ = ("state", "event", "operands")

    def __init__(self, state, event, operands):
        self.state, self.event, self.operands = state, event, operands


# The Kuu chain that runs BESIDE a streaming kernel (gate=True) takes a cluster of 4 CTAs (512 chunks) instead of 8: it is hidden
# anyway, and the accumulate — which leaves exactly 4 SMs' worth of CTA slots free — runs at the rate of the SMs it keeps.
KUU_CHUNKS_BESIDE_STREAMING = 0
_KUU_STATES = {}
_KUU_STREAM = {}
_KUU_LAST = {}


def kuu_chain_1d(Kuu, dKuu, basis, chunks=0, gate=False, timing=False):
    """Launches the part of the bound that depends on the hyper-parameters only — log|Kuu|, band(Kuu^-1) and their
    lengthscale tangents (reference gpr.py:56-70) — on a side stream, ordered after the current stream's work so far
    (the Kuu assembly).  Launch it BEFORE accum_1d and the O(N) pass hides it; elbo_grad_1d(..., kuu=handle) joins.
    gate=True: the current stream waits until the chain kernel is next in line on the side stream (its pre-pass is done), so
    that a machine-filling kernel launched next does not take every SM before the chain's few CTAs are dispatched."""
    k, m = basis.order, basis.m
    if gate and chunks == 0:
        chunks = KUU_CHUNKS_BESIDE_STREAMING
    dev = device()
    side = _KUU_STREAM.get(dev)
    if side is None:
        # high priority: its few CTAs must get their SMs although a full-machine streaming kernel is being dispatched
        side = _KUU_STREAM[dev] = torch.cuda.Stream(device=dev, priority=-1)
    key = (dev, m, k)
    state = _KUU_STATES.get(key)
    if state is None:
        state = _KUU_STATES[key] = torch.empty(_lib.load().asvgp_kuu_state_doubles(m, k), dtype=F64, device=dev)
    ws = workspace_1d(m, k, chunks, slot="kuu")
    main = torch.cuda.current_stream()
    side.wait_stream(main)
    gate_ev = torch.cuda.Event() if gate else None
    if gate:
        gate_ev.record(side)          # creates the underlying cudaEvent_t; the library re-records it before the chain kernel
    _lib.call("asvgp_kuu_chain_1d", _p(Kuu), _p(dKuu), m, k, int(chunks), _p(state), _p(ws), ws.numel(),
              ctypes.c_void_p(gate_ev.cuda_event if gate else 0), ctypes.c_void_p(side.cuda_stream))
    done = torch.cuda.Event(enable_timing=timing)
    done.record(side)
    if gate:
        main.wait_event(gate_ev)
    # the operands stay referenced until the next chain is launched (by then this one has been joined or superseded: the
    # side stream is in order), so the allocator cannot hand their memory out while the side stream still reads it
    handle = _KUU_LAST[dev] = KuuChain(state, done, (Kuu, dKuu))
    return handle


def elbo_grad_1d(Kuu, dKuu, acc, basis, variance, sigma2, chunks=0, out=None, kuu=None, join_late=None):
    """Launches the ELBO+gradient kernels; returns the 16-slot device result (see include/asvgp_b200.h).  The Kuu chain
    runs on a side stream next to the two P chains (`kuu`: a handle from kuu_chain_1d launched earlier, e.g. before the
    accumulate; shared by the output columns of a multi-output model)."""
    k, m = basis.order, basis.m
    if join_late is None:
        join_late = kuu is None      # forked right here: the P chains run beside it; a handle from earlier is joined up front
    if kuu is None:
        kuu = kuu_chain_1d(Kuu, dKuu, basis, chunks)
    ws = workspace_1d(m, k, chunks)
    if out is None:
        out = torch.empty(16, dtype=F64, device=acc.device)
    _lib.call("asvgp_elbo_grad_1d_prepared", _p(kuu.state), _p(Kuu), _p(dKuu), _p(acc), m, k, float(variance),
              float(sigma2), int(chunks), _p(out), _p(ws), ws.numel(), ctypes.c_void_p(kuu.event.cuda_event), int(join_late),
              _stream())
    return out


def elbo_grad_1d_single_stream(Kuu, dKuu, acc, basis, variance, sigma2, chunks=0, out=None):
    """The same bound as ONE C call on the current stream (asvgp_elbo_grad_1d: Kuu chain, then P chains)."""
    k, m = basis.order, basis.m
    ws = workspace_1d(m, k, chunks)
    if out is None:
        out = torch.empty(16, dtype=F64, device=acc.device)
    _lib.call("asvgp_elbo_grad_1d", _p(Kuu), _p(dKuu), _p(acc), m, k, float(variance), float(sigma2), int(chunks),
              _p(out), _p(ws), ws.numel(), _stream())
    return out


def posterior_1d(Kuu, acc, basis, sigma2, chunks=0):
    """alpha = P^-1 b / sigma2 and S = band(P^-1) - band(Kuu^-1) on the device (reference gpr.py:96-108)."""
    k, m = basis.order, basis.m
    ws = workspace_1d(m, k, chunks)
    alpha = torch.empty(m, dtype=F64, device=acc.device)
    S = torch.empty((k + 1, m), dtype=F64, device=acc.device)
    info = torch.zeros(2, dtype=F64, device=acc.device)
    _lib.call("asvgp_posterior_1d", _p(Kuu), _p(acc), m, k, float(sigma2), int(chunks), _p(alpha), _p(S), _p(info),
              _p(ws), ws.numel(), _stream())
    return alpha, S, info


# ---- host-resident data: stream it through pinned staging buffers ------------------------------------------------------
_STAGING = {}


def _staging(dev, key, nbytes):
    """Double-buffered pinned and device staging areas of `nbytes` bytes each, cached per (device, key)."""
    key = (dev,) + key
    st = _STAGING.get(key)
    if st is None:
        st = dict(
            host=[torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(2)],
            dev=[torch.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(2)],
            copy_stream=torch.cuda.Stream(device=dev),
            filled=[torch.cuda.Event() for _ in range(2)],
            drained=[torch.cuda.Event() for _ in range(2)],
            staged=[torch.cuda.Event() for _ in range(2)],
        )
        _STAGING[key] = st
    return st


def _split_staging(buf, parts):
    """Typed views of consecutive regions of a uint8 staging buffer: parts = [(dtype, count), ...], every region starting
    at a 32-byte boundary (the kernels' vector loads)."""
    out, off = [], 0
    for dtype, count in parts:
        nb = count * dtype.itemsize
        out.append(buf[off: off + nb].view(dtype))
        off += -(-nb // 32) * 32
    return out


def _staging_bytes(parts):
    return sum(-(-count * dtype.itemsize // 32) * 32 for dtype, count in parts)


def accum_1d_host(x, y, basis, acc=None, chunk=1 << 23):
    """accum_1d for HOST arrays (numpy or CPU tensors): the points are streamed to the GPU in `chunk`-point pieces,
    host->pinned staging (unless already pinned), async H2D on a copy stream, double-buffered against the accumulate
    kernel — the device never holds more than two chunks.  float32 / float64 arrays are staged and sent in their own dtype
    (float32 halves the PCIe bytes); other dtypes are converted to float64."""
    dev = device()
    xt = points_to_host(x).reshape(-1)
    yt = points_to_host(y).reshape(-1)
    n = xt.numel()
    if yt.numel() != n:
        raise ValueError("x and y must have the same number of points")
    mesh = device_mesh(basis)
    if acc is None:
        acc = torch.zeros(accum_size_1d(basis), dtype=F64, device=dev)
    if n == 0:
        return acc
    chunk = min(chunk, n + (n & 1))
    parts = [(xt.dtype, chunk), (yt.dtype, chunk)]
    st = _staging(dev, ("1d", chunk, xt.dtype, yt.dtype), _staging_bytes(parts))
    xc, yc = ELEM_TYPES[xt.dtype], ELEM_TYPES[yt.dtype]
    pinned = xt.is_pinned() and yt.is_pinned()
    main = torch.cuda.current_stream()
    cs = st["copy_stream"]
    n_chunks = -(-n // chunk)
    for c in range(n_chunks):
        lo, hi = c * chunk, min((c + 1) * chunk, n)
        s = c & 1
        dx, dy = _split_staging(st["dev"][s], parts)
        # the kernel that last read this buffer (two chunks ago, or the previous CALL: the staging buffers are cached and
        # shared between calls) has finished; waiting on a never-recorded event is a no-op
        cs.wait_event(st["drained"][s])
        with torch.cuda.stream(cs):
            if pinned:
                dx[: hi - lo].copy_(xt[lo:hi], non_blocking=True)
                dy[: hi - lo].copy_(yt[lo:hi], non_blocking=True)
            else:
                hx, hy = _split_staging(st["host"][s], parts)
                st["staged"][s].synchronize()          # previous H2D out of this pinned buffer (also a previous call's) is done
                hx[: hi - lo].copy_(xt[lo:hi])
                hy[: hi - lo].copy_(yt[lo:hi])
                dx[: hi - lo].copy_(hx[: hi - lo], non_blocking=True)
                dy[: hi - lo].copy_(hy[: hi - lo], non_blocking=True)
                st["staged"][s].record(cs)
            st["filled"][s].record(cs)
        main.wait_event(st["filled"][s])
        _lib.call("asvgp_accum_1d_typed", _p(dx), xc, _p(dy), yc, hi - lo, _p(mesh), mesh.numel(), basis.order, _p(acc),
                  ctypes.c_void_p(main.cuda_stream))
        st["drained"][s].record(main)
    return acc


# =====================================================================================================================
# 2-D (Kronecker) operators
# =====================================================================================================================
def _check_bases_2d(bases):
    if len(bases) != 2:
        raise NotImplementedError("the Kronecker kernels are written for d = 2 (as reference utils.py:57)")
    if bases[0].order != bases[1].order:
        raise ValueError("all bases of a Kronecker model must have the same order (reference gpr.py:260-262)")
    return bases[0].order, bases[0].m, bases[1].m


def stencil_rows(order):
    """Rows of the stencil layout: offsets d1 in [0, k], d2 in [-k, k]."""
    return (order + 1) * (2 * order + 1)


def accum_size_2d(bases):
    """Doubles of the packed 2-D accumulator [G stencil (n_e x M) | b (M) | sum y^2 | count]."""
    k, m1, m2 = _check_bases_2d(bases)
    return (stencil_rows(k) + 1) * m1 * m2 + 2


def split_accum_2d(acc, bases):
    k, m1, m2 = _check_bases_2d(bases)
    M, ne = m1 * m2, stencil_rows(k)
    return acc[: ne * M].view(ne, M), acc[ne * M: (ne + 1) * M], acc[(ne + 1) * M:]


def moment_table_2d(bases):
    """Zeroed per-cell moment table for accum_2d."""
    k, _, _ = _check_bases_2d(bases)
    n = _lib.load().asvgp_accum_2d_moment_doubles(bases[0].mesh.shape[0], bases[1].mesh.shape[0], k)
    return torch.zeros(n, dtype=F64, device=device())


def order_probe_2d(X, bases):
    """Fraction of sampled neighbour pairs of X[n,2] that lie more than one cell apart (one small D2H read)."""
    X, xt = points_to_device(X)
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    out = torch.empty(1, dtype=F64, device=X.device)
    _lib.call("asvgp_order_probe_2d_typed", _p(X), xt, X.shape[0], _p(mesh1), mesh1.numel(), _p(mesh2), mesh2.numel(), _p(out),
              _stream())
    return float(out.item())


def choose_binned_2d(X, bases):
    """accum_2d's binned="auto" choice for the device points X[n, 2] (one order probe, one host synchronisation): callers
    that accumulate several target columns over the same X probe once and pass the answer to every call."""
    return X.shape[0] >= BINNED_MIN_POINTS and order_probe_2d(X, bases) > BINNED_JUMP_FRACTION


def accum_2d(X, y, bases, cellmom, scal, binned=False, raster_row_len=None):
    """Adds the per-cell moments of the points (X[n,2], y[n]) into `cellmom` and (sum y^2, n) into `scal`
    (reference gpr.py:268-274 without materialising the Khatri-Rao Kuf).  binned: as accum_1d.
    raster_row_len: the caller's statement that X is a flattened raster (meshgrid, x1 slow) with rows of that many points
    — skips the on-device classification (asvgp_accum_2d_raster); a wrong statement is slow, never wrong.
    X and y may each be float32 or float64 and are read as they are (other dtypes are converted to float64)."""
    k, _, _ = _check_bases_2d(bases)
    X, xt = points_to_device(X)
    y, yt = points_to_device(y)
    y = y.reshape(-1)
    if X.dim() != 2 or X.shape[1] != 2 or X.shape[0] != y.numel():
        raise ValueError("X must be [n, 2] and y [n]")
    if X.data_ptr() % 16:            # the kernel reads one point / two targets per load (a clone keeps the dtype)
        X = X.clone()
    if y.data_ptr() % 16:
        y = y.clone()
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    if raster_row_len:
        _lib.call("asvgp_accum_2d_raster_typed", _p(X), xt, _p(y), yt, X.shape[0], int(raster_row_len), _p(mesh1),
                  mesh1.numel(), _p(mesh2), mesh2.numel(), k, _p(cellmom), _p(scal), _stream())
        return cellmom, scal
    if binned == "auto":
        binned = choose_binned_2d(X, bases)
    if binned:
        nbytes = _lib.load().asvgp_accum_2d_binned_work_bytes(X.shape[0])
        work = torch.empty(nbytes, dtype=torch.uint8, device=X.device)
        _lib.call("asvgp_accum_2d_binned_typed", _p(X), xt, _p(y), yt, X.shape[0], _p(mesh1), mesh1.numel(), _p(mesh2),
                  mesh2.numel(), k, _p(cellmom), _p(scal), _p(work), nbytes, _stream())
        return cellmom, scal
    _lib.call("asvgp_accum_2d_typed", _p(X), xt, _p(y), yt, X.shape[0], _p(mesh1), mesh1.numel(), _p(mesh2), mesh2.numel(), k,
              _p(cellmom), _p(scal), _stream())
    return cellmom, scal


def _expansion_tables(order, dev):
    key = (dev, order)
    t = _EXPANSION.get(key)
    if t is None:
        from . import _spline_tables as tab

        t = (torch.from_numpy(np.ascontiguousarray(tab.product_bernstein_float(order))).to(dev),
             torch.from_numpy(np.ascontiguousarray(tab.piece_bernstein_float(order))).to(dev))
        _EXPANSION[key] = t
    return t


_EXPANSION = {}


def expand_moments_2d(cellmom, bases, acc):
    """Adds the Gram stencil and the projection implied by the moment table into the packed accumulator."""
    k, _, _ = _check_bases_2d(bases)
    Gs, b, _ = split_accum_2d(acc, bases)
    Cprod, Dy = _expansion_tables(k, acc.device)
    _lib.call("asvgp_expand_moments_2d", _p(cellmom), _p(Cprod), _p(Dy), bases[0].mesh.shape[0],
              bases[1].mesh.shape[0], k, _p(Gs), _p(b), _stream())
    return acc


def accum_2d_host(X, y, bases, cellmom, scal, chunk=1 << 22, raster_row_len=None):
    """accum_2d for HOST arrays: streamed through pinned staging buffers, double-buffered against the kernel.
    raster_row_len: as accum_2d (the chunks are then whole rows).  float32 / float64 arrays are staged and sent in their own
    dtype; other dtypes are converted to float64.
    Several target columns: y [n, D] with D moment tables and scalar pairs (cellmom, scal: sequences of D) — every chunk of X
    crosses PCIe once and the accumulate runs once per column on it."""
    dev = device()
    Xt = points_to_host(X)
    yt = points_to_host(y)
    multi = isinstance(cellmom, (list, tuple))
    ycols = [yt[:, d] for d in range(yt.shape[1])] if multi else [yt.reshape(-1)]
    cellmoms, scals = (list(cellmom), list(scal)) if multi else ([cellmom], [scal])
    n = Xt.shape[0]
    if Xt.dim() != 2 or Xt.shape[1] != 2 or any(c.numel() != n for c in ycols):
        raise ValueError("X must be [n, 2] and y [n] (or [n, D] with D moment tables)")
    if not (len(ycols) == len(cellmoms) == len(scals)):
        raise ValueError("one moment table and one scalar pair per target column")
    Xt = Xt.contiguous()
    if n == 0:
        return cellmom, scal
    k, _, _ = _check_bases_2d(bases)
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    if raster_row_len:
        if n % int(raster_row_len):
            raise ValueError("n is not a whole number of rows of raster_row_len points")
        chunk = max(1, chunk // int(raster_row_len)) * int(raster_row_len)
        if chunk & 1:
            chunk *= 2
    chunk = min(chunk, n + (n & 1))
    n_cols = len(ycols)
    parts = [(Xt.dtype, 2 * chunk)] + [(yt.dtype, chunk)] * n_cols
    key = ("2d", chunk, Xt.dtype, yt.dtype) if not multi else ("2d", chunk, Xt.dtype, yt.dtype, n_cols)
    st = _staging(dev, key, _staging_bytes(parts))
    xc, yc = ELEM_TYPES[Xt.dtype], ELEM_TYPES[yt.dtype]
    pinned = Xt.is_pinned() and all(c.is_pinned() and c.is_contiguous() for c in ycols)
    main, cs = torch.cuda.current_stream(), st["copy_stream"]
    for c in range(-(-n // chunk)):
        lo, hi = c * chunk, min((c + 1) * chunk, n)
        cnt, s = hi - lo, c & 1
        dXf, *dyfs = _split_staging(st["dev"][s], parts)
        dX, dys = dXf[: 2 * cnt].view(cnt, 2), [dyf[:cnt] for dyf in dyfs]
        cs.wait_event(st["drained"][s])                # also covers the previous call (cached, shared staging buffers)
        with torch.cuda.stream(cs):
            if pinned:
                dX.copy_(Xt[lo:hi], non_blocking=True)
                for dy, yc_host in zip(dys, ycols):
                    dy.copy_(yc_host[lo:hi], non_blocking=True)
            else:
                hXf, *hyfs = _split_staging(st["host"][s], parts)
                st["staged"][s].synchronize()
                hXf[: 2 * cnt].view(cnt, 2).copy_(Xt[lo:hi])
                for hyf, yc_host in zip(hyfs, ycols):
                    hyf[:cnt].copy_(yc_host[lo:hi])
                dXf[: 2 * cnt].copy_(hXf[: 2 * cnt], non_blocking=True)
                for dy, hyf in zip(dys, hyfs):
                    dy.copy_(hyf[:cnt], non_blocking=True)
                st["staged"][s].record(cs)
            st["filled"][s].record(cs)
        main.wait_event(st["filled"][s])
        for dy, cm, sc in zip(dys, cellmoms, scals):
            if raster_row_len:
                _lib.call("asvgp_accum_2d_raster_typed", _p(dX), xc, _p(dy), yc, cnt, int(raster_row_len), _p(mesh1),
                          mesh1.numel(), _p(mesh2), mesh2.numel(), k, _p(cm), _p(sc), ctypes.c_void_p(main.cuda_stream))
            else:
                _lib.call("asvgp_accum_2d_typed", _p(dX), xc, _p(dy), yc, cnt, _p(mesh1), mesh1.numel(), _p(mesh2), mesh2.numel(),
                          k, _p(cm), _p(sc), ctypes.c_void_p(main.cuda_stream))
        st["drained"][s].record(main)
    return cellmom, scal


_SIDE_STREAMS = {}


def side_streams(n):
    """n cached side streams of the current device (for small independent launches that should overlap a long kernel)."""
    dev = device()
    pool = _SIDE_STREAMS.setdefault(dev, [])
    while len(pool) < n:
        pool.append(torch.cuda.Stream(device=dev))
    return pool[:n]


def band_inverse_1d(A, dA, basis, chunks=0, slot=0):
    """(band(A^-1), band(-A^-1 dA A^-1), scal[4] = {log|A|, dlog|A|, info, -}) of one banded SPD factor."""
    k, m = basis.order, basis.m
    ws = workspace_1d(m, k, chunks, slot)
    sig = torch.empty((k + 1, m), dtype=F64, device=A.device)
    dsig = torch.empty_like(sig)
    scal = torch.empty(4, dtype=F64, device=A.device)
    _lib.call("asvgp_band_inverse_1d", _p(A), _p(dA if dA is not None else A), m, k, int(chunks), _p(sig), _p(dsig),
              _p(scal), _p(ws), ws.numel(), _stream())
    return sig, dsig, scal


KRON_METHODS = ("nd", "band")
KRON_METHOD = "nd"        # default factorisation of the 2-D model: nested-dissection fronts; "band" = tile DAG over the scalar band


MAX_RHS = 32       # ASVGP_MAX_RHS of include/asvgp_b200.h: right-hand sides (output columns) per factorisation


def _check_n_rhs(n_rhs):
    n_rhs = int(n_rhs)
    if not 1 <= n_rhs <= MAX_RHS:
        raise ValueError("n_rhs must lie in [1, %d], got %d" % (MAX_RHS, n_rhs))
    return n_rhs


class KronWorkspace:
    """Device buffers of the factorisation of P = K1 (x) K2 + G / sigma2 (cached per (device, m1, m2, k, method, n_rhs)).
    n_rhs > 1: one factorisation for n_rhs right-hand sides (asvgp_kron_*_multi; rhs is [n_rhs * M], scal
    {log|P|, info, Q_1 ... Q_n_rhs}, terms [n_rhs, 11]); n_rhs = 1 is the single-rhs layout of asvgp_kron_factor."""

    def __init__(self, m1, m2, order, method="nd", n_rhs=1):
        lib = _lib.load()
        dev = device()
        if method not in KRON_METHODS:
            raise ValueError("method must be one of %r" % (KRON_METHODS,))
        n_rhs = _check_n_rhs(n_rhs)
        if n_rhs > 1 and method != "nd":
            raise NotImplementedError("several right-hand sides need method='nd' (the scalar-band method takes one)")
        self.m1, self.m2, self.order, self.method, self.n_rhs = m1, m2, order, method, n_rhs
        self.M = m1 * m2
        self.prefix = "asvgp_kron_" if method == "nd" else "asvgp_kronband_"
        if n_rhs == 1:
            nb, nw, ns, nr = (getattr(lib, self.prefix + q)(m1, m2, order) for q in ("band_doubles", "work_doubles", "sig_doubles", "rhs_doubles"))
            if min(nb, nw, ns, nr) < 0:
                raise _lib.AsvgpNativeError("kron workspace query rejected m=%d,%d order=%d" % (m1, m2, order))
        else:
            sizes = (ctypes.c_int64 * 4)()
            _lib.call("asvgp_kron_doubles_multi", m1, m2, order, n_rhs, ctypes.cast(sizes, ctypes.c_void_p))
            nb, ns, nw, nr = sizes
        self.band = torch.empty(nb, dtype=F64, device=dev)
        self.sig_band = None                     # allocated on first selected inverse
        self.n_sig = ns
        self.work = torch.empty(nw, dtype=F64, device=dev)
        self.rhs = torch.zeros(nr, dtype=F64, device=dev)
        self.scal = torch.zeros(3 if n_rhs == 1 else 2 + n_rhs, dtype=F64, device=dev)
        self.sigma_stencil = torch.zeros((stencil_rows(order), self.M), dtype=F64, device=dev)
        self.terms = torch.zeros(11 if n_rhs == 1 else (n_rhs, 11), dtype=F64, device=dev)


_KRON_WS = {}


def kron_workspace(m1, m2, order, method=None, n_rhs=1):
    method = method or KRON_METHOD
    key = (device(), m1, m2, order, method, int(n_rhs))
    ws = _KRON_WS.get(key)
    if ws is None:
        ws = _KRON_WS[key] = KronWorkspace(m1, m2, order, method, n_rhs)
    return ws


def kron_plan_info(m1, m2, order, with_fronts=False, n_rhs=None):
    """Shape of the nested-dissection elimination tree (host-side query, no GPU needed): dict of counts and, with
    `with_fronts`, the list of fronts as (level, separator ids, boundary ids); id m1*m2 is the right-hand-side row
    (n_rhs given: ids m1*m2 ... m1*m2 + n_rhs - 1 are the rows of the n_rhs right-hand sides)."""
    lib = _lib.load()
    out = (ctypes.c_double * 8)()
    if n_rhs is None:
        query = lambda o, buf, cap: lib.asvgp_kron_plan_info(m1, m2, order, o, buf, cap)   # noqa: E731
    else:
        query = lambda o, buf, cap: lib.asvgp_kron_plan_info_multi(m1, m2, order, int(n_rhs), o, buf, cap)   # noqa: E731
    need = query(ctypes.cast(out, ctypes.c_void_p), None, 0)
    if need < 0:
        raise _lib.AsvgpNativeError("kron_plan_info rejected m=%d,%d order=%d n_rhs=%s" % (m1, m2, order, n_rhs))
    info = dict(zip(("fronts", "levels", "tiles", "separator_block_columns", "chain_columns", "chain_block_columns",
                     "largest_front", "flops"), [float(v) for v in out]))
    if with_fronts:
        buf = np.zeros(need, dtype=np.int32)
        query(None, buf.ctypes.data_as(ctypes.c_void_p), need)
        fronts, w = [], 0
        while w < need:
            level, ns, nb = (int(v) for v in buf[w:w + 3])
            fronts.append((level, buf[w + 3:w + 3 + ns].copy(), buf[w + 3 + ns:w + 3 + ns + nb].copy()))
            w += 3 + ns + nb
        info["front_list"] = fronts
    return info


def kron_factor(K1, K2, acc, bases, sigma2, ws, b=None):
    """Factorisation of P and forward substitution of Kuf_y; ws.scal = {log|P|, ||L^-1 b||^2, info}.
    b: right-hand sides [D, M] (D = ws.n_rhs; default: the projection in acc, D = 1).  With D > 1 one factorisation
    serves all columns and ws.scal = {log|P|, info, ||L^-1 b_1||^2, ..., ||L^-1 b_D||^2}."""
    k, m1, m2 = _check_bases_2d(bases)
    Gs, b_acc, _ = split_accum_2d(acc, bases)
    if b is None:
        b = b_acc
    if b.numel() != ws.n_rhs * ws.M:
        raise ValueError("b must hold n_rhs = %d columns of %d entries" % (ws.n_rhs, ws.M))
    if ws.method == "band":
        ws.rhs.zero_()
    ws.rhs[: ws.n_rhs * ws.M].view_as(b).copy_(b)
    if ws.n_rhs == 1:
        _lib.call(ws.prefix + "factor", _p(K1), _p(K2), _p(Gs), m1, m2, k, float(sigma2), _p(ws.band), _p(ws.rhs),
                  _p(ws.scal), _stream())
    else:
        _lib.call("asvgp_kron_factor_multi", _p(K1), _p(K2), _p(Gs), m1, m2, k, ws.n_rhs, float(sigma2), _p(ws.band),
                  _p(ws.rhs), _p(ws.scal), _stream())
    return ws


def kron_selinv(bases, ws):
    """Selected inverse of P on the stencil pattern (ws.sigma_stencil) and x = P^-1 Kuf_y (ws.rhs[:M]; [D, M] for a
    workspace of D > 1 right-hand sides)."""
    k, m1, m2 = _check_bases_2d(bases)
    if ws.sig_band is None:
        ws.sig_band = torch.empty(ws.n_sig, dtype=F64, device=ws.band.device)
    if ws.n_rhs == 1:
        _lib.call(ws.prefix + "selinv", _p(ws.band), m1, m2, k, _p(ws.sig_band), _p(ws.rhs), _p(ws.sigma_stencil),
                  _p(ws.work), _stream())
        return ws.sigma_stencil, ws.rhs[: ws.M]
    _lib.call("asvgp_kron_selinv_multi", _p(ws.band), m1, m2, k, ws.n_rhs, _p(ws.sig_band), _p(ws.rhs), _p(ws.sigma_stencil),
              _p(ws.work), _stream())
    return ws.sigma_stencil, ws.rhs.view(ws.n_rhs, ws.M)


def kron_terms(SigP, acc, x, K1, dK1, K2, dK2, S1, dS1, S2, dS2, bases, out):
    k, m1, m2 = _check_bases_2d(bases)
    Gs, _, _ = split_accum_2d(acc, bases)
    _lib.call("asvgp_kron_terms", _p(SigP), _p(Gs), _p(x), _p(K1), _p(dK1), _p(K2), _p(dK2), _p(S1), _p(dS1), _p(S2),
              _p(dS2), m1, m2, k, _p(out), _stream())
    return out


def predict_2d_prepare(bases, alpha, SigP, S1, S2, work=None):
    """Per-cell polynomial form of the posterior (asvgp_predict_2d_prepare): done once per set of hyper-parameters, then any
    number of predict_2d_apply calls stream test points through it."""
    k, _, _ = _check_bases_2d(bases)
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    if work is None:
        nw = _lib.load().asvgp_predict_2d_work_doubles(mesh1.numel(), mesh2.numel(), k)
        work = torch.empty(nw, dtype=F64, device=alpha.device)
    _lib.call("asvgp_predict_2d_prepare", mesh1.numel(), mesh2.numel(), k, _p(alpha), _p(SigP), _p(S1), _p(S2), _p(work), _stream())
    return work


def predict_2d_apply(Xnew, bases, work, prior_var, raster_row_len=None, mean=None, var=None):
    """Posterior mean / variance at Xnew[n, 2] from the prepared table (reference gpr.py:310-359)."""
    k, _, _ = _check_bases_2d(bases)
    X = to_device(Xnew)
    if X.dim() != 2 or X.shape[1] != 2:
        raise ValueError("Xnew must be [n, 2]")
    if X.data_ptr() % 16:
        X = X.clone()
    n = X.shape[0]
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    mean = torch.empty(n, dtype=F64, device=X.device) if mean is None else mean
    var = torch.empty(n, dtype=F64, device=X.device) if var is None else var
    _lib.call("asvgp_predict_2d_apply", _p(X), n, int(raster_row_len or 0), _p(mesh1), mesh1.numel(), _p(mesh2), mesh2.numel(), k,
              float(prior_var), _p(mean), _p(var), _p(work), _stream())
    return mean, var


def predict_2d(Xnew, bases, alpha, SigP, S1, S2, prior_var):
    """Posterior mean / variance of the Kronecker model at Xnew[n, 2] (reference gpr.py:310-359)."""
    k, _, _ = _check_bases_2d(bases)
    X = to_device(Xnew)
    if X.dim() != 2 or X.shape[1] != 2:
        raise ValueError("Xnew must be [n, 2]")
    n = X.shape[0]
    mesh1, mesh2 = device_mesh(bases[0]), device_mesh(bases[1])
    mean = torch.empty(n, dtype=F64, device=X.device)
    var = torch.empty(n, dtype=F64, device=X.device)
    key = (X.device, mesh1.numel(), mesh2.numel(), k)
    work = _PREDICT_WORK.get(key)
    if work is None:
        nw = _lib.load().asvgp_predict_2d_work_doubles(mesh1.numel(), mesh2.numel(), k)
        work = _PREDICT_WORK[key] = torch.empty(nw, dtype=F64, device=X.device)
    _lib.call("asvgp_predict_2d", _p(X), n, _p(mesh1), mesh1.numel(), _p(mesh2), mesh2.numel(), k, _p(alpha),
              _p(SigP), _p(S1), _p(S2), float(prior_var), _p(mean), _p(var), _p(work), _stream())
    return mean, var


_PREDICT_WORK = {}


# =====================================================================================================================
# dense SPD matrices (one front of the nested-dissection kernels) and the additive model's operators
# =====================================================================================================================
class DenseWorkspace:
    """Device buffers of asvgp_dense_factor / asvgp_dense_selinv for n x n matrices (cached per (device, n, n_rhs)).
    n_rhs > 1: asvgp_dense_*_multi, x is [n_rhs, n] and scal {log|A|, info, rhs_1^T A^-1 rhs_1, ...}."""

    def __init__(self, n, n_rhs=1):
        lib = _lib.load()
        dev = device()
        n_rhs = _check_n_rhs(n_rhs)
        if n_rhs == 1:
            nb, ns, nw = lib.asvgp_dense_band_doubles(n), lib.asvgp_dense_sig_doubles(n), lib.asvgp_dense_work_doubles(n)
            if min(nb, ns, nw) < 0:
                raise _lib.AsvgpNativeError("dense workspace query rejected n=%d" % n)
        else:
            sizes = (ctypes.c_int64 * 4)()
            _lib.call("asvgp_dense_doubles_multi", n, n_rhs, ctypes.cast(sizes, ctypes.c_void_p))
            nb, ns, nw, _ = sizes
        self.n, self.n_rhs = n, n_rhs
        self.band = torch.empty(nb, dtype=F64, device=dev)
        self.sig_band = torch.empty(ns, dtype=F64, device=dev)
        self.work = torch.empty(nw, dtype=F64, device=dev)
        self.scal = torch.zeros(3 if n_rhs == 1 else 2 + n_rhs, dtype=F64, device=dev)
        self.x = torch.empty(n if n_rhs == 1 else (n_rhs, n), dtype=F64, device=dev)
        self.inv = torch.empty((n, n), dtype=F64, device=dev)


_DENSE_WS = {}


def dense_workspace(n, n_rhs=1):
    key = (device(), n, int(n_rhs))
    ws = _DENSE_WS.get(key)
    if ws is None:
        ws = _DENSE_WS[key] = DenseWorkspace(n, n_rhs)
    return ws


def dense_factor(A, rhs, ws):
    """Cholesky of the dense SPD matrix A (lower triangle read); ws.scal = {log|A|, rhs^T A^-1 rhs, info}.  rhs may be
    [D, n] for a workspace of D = ws.n_rhs > 1 right-hand sides: ws.scal = {log|A|, info, rhs_1^T A^-1 rhs_1, ...}."""
    if rhs.numel() != ws.n_rhs * ws.n:
        raise ValueError("rhs must hold n_rhs = %d columns of %d entries" % (ws.n_rhs, ws.n))
    rhs = rhs.contiguous()
    if ws.n_rhs == 1:
        _lib.call("asvgp_dense_factor", _p(A), ws.n, _p(rhs), _p(ws.band), _p(ws.scal), _stream())
    else:
        _lib.call("asvgp_dense_factor_multi", _p(A), ws.n, ws.n_rhs, _p(rhs), _p(ws.band), _p(ws.scal), _stream())
    return ws


def dense_selinv(ws):
    """(A^-1 rhs, A^-1) from the factor held in ws (consumed); A^-1 rhs is [D, n] for D = ws.n_rhs > 1."""
    if ws.n_rhs == 1:
        _lib.call("asvgp_dense_selinv", _p(ws.band), ws.n, _p(ws.sig_band), _p(ws.x), _p(ws.inv), _p(ws.work), _stream())
    else:
        _lib.call("asvgp_dense_selinv_multi", _p(ws.band), ws.n, ws.n_rhs, _p(ws.sig_band), _p(ws.x), _p(ws.inv), _p(ws.work),
                  _stream())
    return ws.x, ws.inv


def accum_cross(X, da, db, basis_a, basis_b, out=None):
    """out[m_a, m_b] += Kuf_a Kuf_b^T for columns da, db of the device tensor X[n, D] (reference gpr.py:174-175)."""
    X = to_device(X)
    if out is None:
        out = torch.zeros((basis_a.m, basis_b.m), dtype=F64, device=X.device)
    ma, mb = device_mesh(basis_a), device_mesh(basis_b)
    if basis_a.order != basis_b.order:
        raise ValueError("all bases of an additive model must have the same order (reference gpr.py:163-165)")
    D = X.shape[1]
    _lib.call("asvgp_accum_cross", ctypes.c_void_p(X.data_ptr() + 8 * da), ctypes.c_void_p(X.data_ptr() + 8 * db), D, X.shape[0],
              _p(ma), ma.numel(), _p(mb), mb.numel(), basis_a.order, _p(out), _stream())
    return out
