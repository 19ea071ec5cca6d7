"""Many small, independent RLVI problems in one launch: the drop-ins of rlvi_b200.rlvi for sweeps.

    update_weights(losses, tol=1e-3, maxiter=100)       rlvi.py:8-20   [B, n] -> [B, n];  list of 1-D -> list
    mean(samples, maxiter=100, tol=1e-3)                rlvi.py:46-65  [B, n, d] or list of [n_b, d] -> theta [B, d]
    linear_regression(X, y, maxiter=100, tol=1e-3)      rlvi.py:68-89  [B, n, d], [B, n] or lists -> theta [B, d]
    logistic_regression(X, y, maxiter=100, tol=1e-2, mstep="sklearn")
                                                        rlvi.py:92-108 [B, n, d], [B, n] or lists -> theta [B, d + 1]

The reference's experiment driver (standard-learning/main.py) fits thousands of tiny problems -- Monte-Carlo runs over a
grid of corruption rates at N = 40..100 -- and so do bootstrap replicates and per-group fits.  One call per problem through
rlvi_b200.rlvi costs about ten launches and two host synchronisations per EM iteration; here every problem runs its whole
EM loop inside one warp of one kernel (rlvi_batched_em_f64), so a sweep is one launch.  Each problem gets the result the
single-problem drop-in computes, to rounding: the same fixed point, the same M-step (the normal equations; for logistic
regression the drop-in's Newton solve of utils.sklearn_log_reg or the MM iteration of utils.mm_log_reg, both in the
warp, rlvi_batched_logistic_f64), the same stop test.

A batch is a stacked array ([B, n, ...], every problem the same size) or a list of per-problem arrays (ragged).  NumPy in
gives NumPy out (the problems are packed on the host and copied to the GPU once); CUDA float64 tensors in gives tensors out.
A problem may have at most `rlvi_b200.ops.batched_max_rows(d)` rows (at least 1024 at every d <= 64); larger ones raise
ValueError and belong to the single-problem functions.  Linear-regression problems whose normal equations fail the
drop-in's pivot test (rank-deficient or ill-conditioned designs, n_b < d) are re-solved one by one with
rlvi_b200.rlvi.linear_regression, whose eigen-decomposition route gives the minimum-norm answer.  Logistic problems take
at most `rlvi_b200.ops.batched_logistic_max_rows(d)` rows (at least 1024 at every d <= 63, 2000 at d <= 8); those whose
Newton solve does not converge in 60 steps, or whose MM majoriser fails the pivot test, are re-solved one by one with
rlvi_b200.rlvi.logistic_regression.  An exception a re-solve raises names the problem.  There is no CPU fallback.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from . import rlvi as _rlvi
from ._host import default_device

__all__ = ["update_weights", "mean", "linear_regression", "logistic_regression"]

HOST_SOLVE = 2       # status of rlvi_batched_em_f64 / _logistic_f64: the problem needs the single-problem drop-in
_LOGREG_MSTEP = {"sklearn": ops.BATCHED_LOGREG_NEWTON, "mm": ops.BATCHED_LOGREG_MM}


def _gather(a, pdim, name):
    """The caller's problems, stacked [B, *problem] or a list of `pdim`-dimensional arrays, as their rows back to back.
    Returns (flat rows: float64 NumPy array or tensor, lengths, stacked, is_torch)."""
    if isinstance(a, (list, tuple)):
        if len(a) == 0:
            raise ValueError(f"{name}: no problems given")
        is_t = isinstance(a[0], torch.Tensor)
        if is_t:
            parts = [p.to(device=a[0].device, dtype=torch.float64) for p in a]
        else:
            parts = [np.asarray(p, dtype=np.float64) for p in a]
        if any(p.ndim != pdim for p in parts):
            raise ValueError(f"{name}: every problem must have {pdim} dimension(s)")
        lengths = np.array([p.shape[0] for p in parts], dtype=np.int64)
        flat = torch.cat(parts) if is_t else np.concatenate(parts)
        return flat, lengths, False, is_t
    is_t = isinstance(a, torch.Tensor)
    a = a.to(torch.float64) if is_t else np.asarray(a, dtype=np.float64)
    if a.ndim != pdim + 1:
        raise ValueError(f"{name}: expected a stacked [B, n{', d' if pdim == 2 else ''}] array or a list of problems")
    B, n = a.shape[0], a.shape[1]
    return a.reshape(B * n, *a.shape[2:]), np.full(B, n, dtype=np.int64), True, is_t


def _offsets(lengths):
    return np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)


def _check_cap(lengths, d, fn, cap=None, d_max=64):
    cap = ops.batched_max_rows(d) if cap is None else cap
    if cap == 0:
        raise ValueError(f"batched.{fn} supports 1 <= d <= {d_max} (got d = {d}); use rlvi_b200.rlvi.{fn} per problem")
    if lengths.size and int(lengths.max()) > cap:
        raise ValueError(f"batched.{fn}: a problem has {int(lengths.max())} rows, the batched kernels admit at most {cap} "
                         f"rows per problem at d = {d}; fit larger problems with rlvi_b200.rlvi.{fn}")


def _to_device(*flats):
    """Host arrays -> one H2D copy of their concatenation, returned as device views of the original shapes;
    tensors are moved (if on the CPU) and made contiguous."""
    if isinstance(flats[0], torch.Tensor):
        dev = flats[0].device if flats[0].is_cuda else default_device()
        return [f.to(dev).contiguous() for f in flats]
    buf = torch.from_numpy(np.concatenate([f.ravel() for f in flats])).to(default_device())
    out, at = [], 0
    for f in flats:
        out.append(buf[at:at + f.size].view(f.shape))
        at += f.size
    return out


def update_weights(losses, tol=1e-3, maxiter=100):
    """rlvi.py:8-20 on every problem: [B, n] -> pi [B, n]; a list of 1-D loss vectors -> a list of pi vectors."""
    flat, lengths, stacked, is_t = _gather(losses, 1, "losses")
    _check_cap(lengths, 1, "update_weights")
    (l,) = _to_device(flat)
    off = _offsets(lengths)
    pi, _ = ops.batched_fixed_point(l, off, tol=tol, maxiter=maxiter)
    if stacked:
        pi = pi.view(lengths.size, int(lengths[0]))
        return pi if is_t else pi.cpu().numpy()
    if is_t:
        return list(torch.split(pi, lengths.tolist()))
    return np.split(pi.cpu().numpy(), off[1:-1])


def mean(samples, maxiter=100, tol=1e-3):
    """rlvi.py:46-65 on every problem: [B, n, d] or a list of [n_b, d] -> theta [B, d]."""
    flat, lengths, _, is_t = _gather(samples, 2, "samples")
    d = flat.shape[1]
    _check_cap(lengths, d, "mean")
    (X,) = _to_device(flat)
    theta, _, _ = ops.batched_em(ops.BATCHED_MEAN, X, None, _offsets(lengths), tol=tol, maxiter=maxiter)
    return theta if is_t else theta.cpu().numpy()


def _fit_xy(fn, X, y, fit, cap, d_max, **dropin_kw):
    """The body of linear_regression and logistic_regression: packs X and y, checks them against `cap(d)`, runs
    `fit(X, y, offsets)` (one batched call) and re-fits the HOST_SOLVE problems with rlvi.<fn>(..., **dropin_kw); an
    exception the drop-in raises names the problem."""
    fx, lengths, _, is_t = _gather(X, 2, "X")
    fy, ly, _, _ = _gather(y, 1, "y")
    if not np.array_equal(lengths, ly):
        raise ValueError("X and y must describe the same problems with the same numbers of rows")
    d = fx.shape[1]
    _check_cap(lengths, d, fn, cap(d), d_max)
    Xd, yd = _to_device(fx, fy.to(fx.device) if is_t else fy)
    off = _offsets(lengths)
    theta, _, status = fit(Xd, yd, off)
    for b in np.flatnonzero(status.cpu().numpy() == HOST_SOLVE):
        s, e = int(off[b]), int(off[b + 1])
        # fresh copies: the drop-in's kernels choose their load path by alignment, and a copy gives the bits of the
        # problem fitted on its own
        try:
            theta[b] = getattr(_rlvi, fn)(Xd[s:e].clone(), yd[s:e].clone(), **dropin_kw)
        except Exception as exc:
            exc.args = (f"batched.{fn}, problem {b}: {exc.args[0] if exc.args else exc}",) + exc.args[1:]
            raise
    return theta if is_t else theta.cpu().numpy()


def linear_regression(X, y, maxiter=100, tol=1e-3):
    """rlvi.py:68-89 on every problem: X [B, n, d] or a list of [n_b, d], y [B, n] or a list of [n_b] -> theta [B, d]."""
    return _fit_xy("linear_regression", X, y,
                   lambda Xd, yd, off: ops.batched_em(ops.BATCHED_LINREG, Xd, yd, off, tol=tol, maxiter=maxiter),
                   ops.batched_max_rows, 64, maxiter=maxiter, tol=tol)


def logistic_regression(X, y, maxiter=100, tol=1e-2, mstep="sklearn"):
    """rlvi.py:92-108 on every problem: X [B, n, d] or a list of [n_b, d], y [B, n] or a list of [n_b] -> theta [B, d + 1]
    (intercept first).  `mstep` as in rlvi.logistic_regression: "sklearn" (the reference's default) or "mm"."""
    if mstep not in _LOGREG_MSTEP:
        raise ValueError(f'mstep must be "sklearn" or "mm" (got {mstep!r})')
    return _fit_xy("logistic_regression", X, y,
                   lambda Xd, yd, off: ops.batched_logistic(Xd, yd, off, mstep=_LOGREG_MSTEP[mstep], tol=tol,
                                                            maxiter=maxiter),
                   ops.batched_logistic_max_rows, 63, maxiter=maxiter, tol=tol, mstep=mstep)
