"""Device-tensor front end of the C ABI (include/rlvi_b200.h): one Python function per entry point.

Every function takes CUDA `torch.Tensor`s (torch is the allocator / stream provider only), passes raw
device pointers and the CURRENT torch stream to librlvi_b200.so, and returns tensors on the same device.
Nothing here computes: there is no CPU fallback, and a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (BATCHED_LINREG, BATCHED_LOGREG_MM, BATCHED_LOGREG_NEWTON, BATCHED_MEAN, FP_DEEP, FP_ONLINE, FP_STANDARD, LOSS_GAUSSIAN, LOSS_LOGISTIC_CE,
                   LOSS_PCA, LOSS_SOFTPLUS, LOSS_SQDIST, LOSS_SQRES, TF32X1, TF32X3)

__all__ = ["FP_STANDARD", "FP_ONLINE", "FP_DEEP", "LOSS_LOGISTIC_CE", "LOSS_SOFTPLUS", "LOSS_SQRES",
           "LOSS_SQDIST", "LOSS_PCA", "LOSS_GAUSSIAN", "fixed_point", "fixed_point_deep", "shift_sum", "shift_sum_e", "loss",
           "weighted_moments", "split_moments", "logistic_grad", "wce_fwd_bwd", "fn_threshold", "read_result",
           "em_step_logistic_host", "launch_count", "TF32X3", "TF32X1", "sigmoid", "online_ce", "irls_weights", "rrm_sum",
           "BATCHED_MEAN", "BATCHED_LINREG", "batched_max_rows", "batched_fixed_point", "batched_results", "batched_em",
           "BATCHED_LOGREG_NEWTON", "BATCHED_LOGREG_MM", "batched_logistic_max_rows", "batched_logistic"]

_RESULT_DTYPE = np.dtype([("eps", "<f8"), ("rho", "<f8"), ("sum_pi", "<f8"), ("err", "<f8"), ("iters", "<i4"),
                          ("converged", "<i4")])
assert _RESULT_DTYPE.itemsize == C.sizeof(_lib.FpResult) == 40


def _dev(t: torch.Tensor) -> int:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("rlvi_b200.ops works on CUDA tensors only (there is no CPU path)")
    return t.device.index if t.device.index is not None else torch.cuda.current_device()


def _chk(t, dtype, name):
    if t is None:
        return None
    if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
        raise TypeError(f"{name} must be a contiguous CUDA tensor of dtype {dtype} (got {t.dtype}, "
                        f"cuda={t.is_cuda}, contiguous={t.is_contiguous()})")
    return t


def _len(t, n, name):
    """The C side sees raw pointers only: every length is checked here."""
    if t is not None and t.numel() != n:
        raise ValueError(f"{name} must have {n} elements (got {t.numel()})")
    return t


def _same_device(ref, *tensors):
    for t in tensors:
        if t is not None and t.device != ref.device:
            raise ValueError(f"all tensors of one call must live on {ref.device} (got {t.device})")


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ctx(dev):
    """The library context of torch's CURRENT stream on `dev`: contexts own scratch, so each stream has
    its own and calls issued from different streams never share it."""
    return _lib.context(dev, torch.cuda.current_stream(dev).cuda_stream)


def launch_count(device=0) -> int:
    """Kernels launched by the library on `device` since its contexts were created."""
    return _lib.launches(int(device))


def read_result(result: torch.Tensor) -> dict:
    """Copy a device rlvi_fp_result (5 doubles = 40 bytes) to the host (synchronises the stream)."""
    raw = result.cpu().numpy().view(np.uint8)[:40].view(_RESULT_DTYPE)[0]
    out = {k: raw[k].item() for k in _RESULT_DTYPE.names}
    if out["iters"] < 0:
        raise _lib.RlviError("fixed-point kernel aborted: a grid/peer barrier timed out")
    return out


def fixed_point(losses=None, *, e_work=None, scale=None, variant=FP_STANDARD, tol=1e-3, maxiter=100, out=None,
                result=None, dist=None, pi0=None):
    """rlvi_fixed_point_f64.  Returns (pi, result_tensor); `result_tensor` stays on the device (see
    `read_result`).  With `losses=None`, `e_work` must already hold e_i = exp(-l_i)."""
    ref = losses if losses is not None else e_work
    dev = _dev(ref)
    f64 = torch.float64
    losses = _chk(losses, f64, "losses")
    n = ref.numel()
    if e_work is None:
        e_work = torch.empty(n, dtype=f64, device=ref.device)
    _chk(e_work, f64, "e_work")
    if out is None:
        out = torch.empty(n, dtype=f64, device=ref.device)
    _chk(out, f64, "out")
    _chk(scale, f64, "scale")
    if n == 0:
        raise ValueError("empty loss vector")
    _len(e_work, n, "e_work")
    _len(out, n, "out")
    _len(scale, 1, "scale")
    if result is None:
        result = torch.empty(5, dtype=f64, device=ref.device)
    _chk(result, f64, "result")
    _len(result, 5, "result")
    _same_device(ref, e_work, out, scale, result)
    ctx = _ctx(dev)
    dptr = C.byref(dist) if dist is not None else None
    if pi0 is None:
        rc = ctx.lib.rlvi_fixed_point_f64(ctx.handle, int(variant), _p(losses), _p(scale), _p(e_work), n, float(tol),
                                          int(maxiter), _p(out), _p(result), dptr, _stream(dev))
    else:      # opt-in: start from a carried-over mean posterior (rlvi_fixed_point_init_f64)
        rc = ctx.lib.rlvi_fixed_point_init_f64(ctx.handle, int(variant), _p(losses), _p(scale), _p(e_work), n,
                                               float(tol), int(maxiter), float(pi0), _p(out), _p(result), dptr,
                                               _stream(dev))
    _lib.check(rc, "rlvi_fixed_point_f64")
    return out, result


def fixed_point_deep(residuals, weights, *, e_work=None, tol=1e-3, maxiter=40, result=None, dist=None):
    """rlvi_fixed_point_deep_f32: in place on `residuals` and `weights` (train_rlvi.py:14-38)."""
    dev = _dev(residuals)
    f32 = torch.float32
    _chk(residuals, f32, "residuals")
    _chk(weights, f32, "weights")
    n = residuals.numel()
    if weights.numel() != n:
        raise ValueError("residuals and weights must have the same length")
    if e_work is None:
        e_work = torch.empty(n, dtype=f32, device=residuals.device)
    _len(_chk(e_work, f32, "e_work"), n, "e_work")
    if result is None:
        result = torch.empty(5, dtype=torch.float64, device=residuals.device)
    _len(_chk(result, torch.float64, "result"), 5, "result")
    _same_device(residuals, weights, e_work, result)
    ctx = _ctx(dev)
    dptr = C.byref(dist) if dist is not None else None
    rc = ctx.lib.rlvi_fixed_point_deep_f32(ctx.handle, _p(residuals), _p(weights), _p(e_work), n, float(tol),
                                           int(maxiter), _p(result), dptr, _stream(dev))
    _lib.check(rc, "rlvi_fixed_point_deep_f32")
    return result


def shift_sum(losses, shift, c, *, pi_out=None, out=None):
    """rlvi_shift_sum_f64: out[0] = sum_i t_i/(c+t_i), t_i = exp(-l_i + shift) (rlvi.py:34-39)."""
    dev = _dev(losses)
    _chk(losses, torch.float64, "losses")
    _len(_chk(pi_out, torch.float64, "pi_out"), losses.numel(), "pi_out")
    if out is None:
        out = torch.empty(1, dtype=torch.float64, device=losses.device)
    _len(_chk(out, torch.float64, "out"), 1, "out")
    _same_device(losses, pi_out, out)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_shift_sum_f64(ctx.handle, _p(losses), losses.numel(), float(shift), float(c), _p(pi_out),
                                    _p(out), _stream(dev))
    _lib.check(rc, "rlvi_shift_sum_f64")
    return out


def shift_sum_e(e, scale_t, c, *, pi_out=None, out=None):
    """rlvi_shift_sum_e_f64: out[0] = sum_i t_i/(c+t_i), t_i = e_i * scale_t (e = exp(-l), scale_t = exp(shift))."""
    dev = _dev(e)
    _chk(e, torch.float64, "e")
    _len(_chk(pi_out, torch.float64, "pi_out"), e.numel(), "pi_out")
    if out is None:
        out = torch.empty(1, dtype=torch.float64, device=e.device)
    _len(_chk(out, torch.float64, "out"), 1, "out")
    _same_device(e, pi_out, out)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_shift_sum_e_f64(ctx.handle, _p(e), e.numel(), float(scale_t), float(c), _p(pi_out), _p(out),
                                      _stream(dev))
    _lib.check(rc, "rlvi_shift_sum_e_f64")
    return out


def _chk_x(X):
    """X is float64 (the reference's precision) or float32 (FP32-stored mode: the rlvi_*_f32 entry points).
    Returns True for float32."""
    is32 = isinstance(X, torch.Tensor) and X.dtype == torch.float32
    _chk(X, torch.float32 if is32 else torch.float64, "X")
    return is32


def loss(kind, X, params, *, y=None, intercept=False, weights=None, want_losses=True, want_e=False,
         losses_out=None, e_out=None, wsum_out=None):
    """rlvi_loss_f64 (float64 X) / rlvi_loss_f32 (float32 X).  Returns (losses | None, e | None, wsum | None)."""
    dev = _dev(X)
    f64 = torch.float64
    x32 = _chk_x(X)
    if x32 and kind == LOSS_GAUSSIAN:
        raise ValueError("the Gaussian loss has no FP32-stored variant")
    if X.dim() != 2:
        raise ValueError("X must be [n, d]")
    n, d = X.shape
    _chk(params, f64, "params")
    n_params = 1 + d + d * d if kind == LOSS_GAUSSIAN else d + (1 if intercept else 0)
    if kind in (LOSS_SQDIST, LOSS_PCA, LOSS_GAUSSIAN) and intercept:
        raise ValueError("this loss kind has no intercept")
    _len(params, n_params, "params")
    _len(_chk(y, f64, "y"), n, "y")
    _len(_chk(weights, f64, "weights"), n, "weights")
    _len(_chk(losses_out, f64, "losses_out"), n, "losses_out")
    _len(_chk(e_out, f64, "e_out"), n, "e_out")
    _len(_chk(wsum_out, f64, "wsum_out"), 2, "wsum_out")
    _same_device(X, params, y, weights, losses_out, e_out, wsum_out)
    if want_losses and losses_out is None:
        losses_out = torch.empty(n, dtype=f64, device=X.device)
    if want_e and e_out is None:
        e_out = torch.empty(n, dtype=f64, device=X.device)
    if weights is not None and wsum_out is None:
        wsum_out = torch.empty(2, dtype=f64, device=X.device)
    ctx = _ctx(dev)
    fn = ctx.lib.rlvi_loss_f32 if x32 else ctx.lib.rlvi_loss_f64
    rc = fn(ctx.handle, int(kind), 1 if intercept else 0, _p(X), _p(y), n, d, _p(params),
            _p(weights), _p(losses_out), _p(e_out), _p(wsum_out), _stream(dev))
    _lib.check(rc, "rlvi_loss_f32" if x32 else "rlvi_loss_f64")
    return losses_out, e_out, wsum_out


def weighted_moments(X, weights, *, y=None, power=1, want_gram=True, out=None, center=None, precision=TF32X3):
    """rlvi_weighted_moments_f64 (or, with `center`, rlvi_weighted_moments_centered_f64: x_i -> x_i - center);
    float32 X -> rlvi_weighted_moments_f32 (tcgen05 TF32 tensor-core Gram, `precision` = TF32X3 | TF32X1).
    Returns the flat device buffer [S0, Swy, S1(d), Sy(d), G(d*d)] (FP64); `split_moments` gives views."""
    dev = _dev(X)
    f64 = torch.float64
    x32 = _chk_x(X)
    if x32 and center is not None:
        raise ValueError("the centred statistics have no FP32-stored variant")
    if X.dim() != 2:
        raise ValueError("X must be [n, d]")
    n, d = X.shape
    _len(_chk(weights, f64, "weights"), n, "weights")
    _len(_chk(y, f64, "y"), n, "y")
    ctx = _ctx(dev)
    if out is None:
        out = torch.zeros(ctx.lib.rlvi_moments_out_doubles(d), dtype=f64, device=X.device)
    _len(_chk(out, f64, "out"), ctx.lib.rlvi_moments_out_doubles(d), "out")
    _same_device(X, weights, y, out, center)
    if x32:
        rc = ctx.lib.rlvi_weighted_moments_f32(ctx.handle, _p(X), _p(y), _p(weights), n, d, int(power),
                                               1 if want_gram else 0, int(precision), _p(out), _stream(dev))
        _lib.check(rc, "rlvi_weighted_moments_f32")
        return out
    if center is None:
        rc = ctx.lib.rlvi_weighted_moments_f64(ctx.handle, _p(X), _p(y), _p(weights), n, d, int(power),
                                               1 if want_gram else 0, _p(out), _stream(dev))
    else:
        _chk(center, f64, "center")
        if center.numel() != d:
            raise ValueError("center must have d elements")
        rc = ctx.lib.rlvi_weighted_moments_centered_f64(ctx.handle, _p(X), _p(y), _p(weights), _p(center), n, d,
                                                        int(power), 1 if want_gram else 0, _p(out), _stream(dev))
    _lib.check(rc, "rlvi_weighted_moments_f64")
    return out


def split_moments(out, d):
    """Views into the flat moments buffer: dict(S0, Swy, S1, Sy, G)."""
    return {"S0": out[0], "Swy": out[1], "S1": out[2:2 + d], "Sy": out[2 + d:2 + 2 * d],
            "G": out[2 + 2 * d:2 + 2 * d + d * d].view(d, d)}


def logistic_grad(X, y, weights, params, *, out=None):
    """rlvi_logistic_grad_f64: [sum c, X^T c], c = w (sigmoid(b + x.theta) - y) (utils.py:40-41)."""
    dev = _dev(X)
    f64 = torch.float64
    _chk(X, f64, "X")
    if X.dim() != 2:
        raise ValueError("X must be [n, d]")
    n, d = X.shape
    _len(_chk(y, f64, "y"), n, "y")
    _len(_chk(weights, f64, "weights"), n, "weights")
    _len(_chk(params, f64, "params"), d + 1, "params")
    if out is None:
        out = torch.empty(d + 1, dtype=f64, device=X.device)
    _len(_chk(out, f64, "out"), d + 1, "out")
    _same_device(X, y, weights, params, out)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_logistic_grad_f64(ctx.handle, _p(X), _p(y), _p(weights), n, d, _p(params), _p(out),
                                        _stream(dev))
    _lib.check(rc, "rlvi_logistic_grad_f64")
    return out


def sigmoid(x, *, out=None):
    """rlvi_sigmoid_f64: utils.py:7-16 on an N-vector (any shape, flattened)."""
    dev = _dev(x)
    _chk(x, torch.float64, "x")
    if out is None:
        out = torch.empty_like(x)
    _len(_chk(out, torch.float64, "out"), x.numel(), "out")
    _same_device(x, out)
    if x.numel() == 0:
        return out
    ctx = _ctx(dev)
    _lib.check(ctx.lib.rlvi_sigmoid_f64(ctx.handle, _p(x), x.numel(), _p(out), _stream(dev)), "rlvi_sigmoid_f64")
    return out


def online_ce(log_proba, targets, *, out=None):
    """rlvi_online_ce_f64: -t l - (1 - t) l (online-learning/main.py:84-85)."""
    dev = _dev(log_proba)
    _chk(log_proba, torch.float64, "log_proba")
    n = log_proba.numel()
    _len(_chk(targets, torch.float64, "targets"), n, "targets")
    if out is None:
        out = torch.empty_like(log_proba)
    _len(_chk(out, torch.float64, "out"), n, "out")
    _same_device(log_proba, targets, out)
    if n == 0:
        return out
    ctx = _ctx(dev)
    _lib.check(ctx.lib.rlvi_online_ce_f64(ctx.handle, _p(log_proba), _p(targets), n, _p(out), _stream(dev)),
               "rlvi_online_ce_f64")
    return out


def irls_weights(e, weights, *, out=None):
    """rlvi_irls_weights_f64: out_i = weights_i e_i (1 - e_i)."""
    dev = _dev(e)
    _chk(e, torch.float64, "e")
    n = e.numel()
    _len(_chk(weights, torch.float64, "weights"), n, "weights")
    if out is None:
        out = torch.empty_like(e)
    _len(_chk(out, torch.float64, "out"), n, "out")
    _same_device(e, weights, out)
    ctx = _ctx(dev)
    _lib.check(ctx.lib.rlvi_irls_weights_f64(ctx.handle, _p(e), _p(weights), n, _p(out), _stream(dev)),
               "rlvi_irls_weights_f64")
    return out


def rrm_sum(losses, inv_alpha, cutoff=1e-16, *, norm=0.0, w_out=None, out=None):
    """rlvi_rrm_sum_f64: out[0] = sum_i max(exp(-l_i inv_alpha), cutoff); w_out_i = exp(-l_i inv_alpha) norm."""
    dev = _dev(losses)
    _chk(losses, torch.float64, "losses")
    _len(_chk(w_out, torch.float64, "w_out"), losses.numel(), "w_out")
    if out is None:
        out = torch.empty(1, dtype=torch.float64, device=losses.device)
    _len(_chk(out, torch.float64, "out"), 1, "out")
    _same_device(losses, w_out, out)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_rrm_sum_f64(ctx.handle, _p(losses), losses.numel(), float(inv_alpha), float(cutoff), float(norm),
                                  _p(w_out), _p(out), _stream(dev))
    _lib.check(rc, "rlvi_rrm_sum_f64")
    return out


def batched_max_rows(d) -> int:
    """rlvi_batched_max_rows: rows one problem of a batched call may have at `d` features (0 outside 1..64)."""
    return int(_lib.load().rlvi_batched_max_rows(int(d)))


def _batched_offsets(offsets, rows, cap, ref):
    """Checks the caller's problem boundaries on the host (the kernels index X, y and pi with them) and uploads them once:
    offsets[0] == 0, strictly increasing, offsets[-1] == rows, every length <= cap.  Returns (device int64 tensor, nprob)."""
    if isinstance(offsets, torch.Tensor):
        if offsets.is_cuda:
            raise TypeError("offsets must be a host array (they are checked on the host before any launch)")
        offsets = offsets.numpy()
    off = np.asarray(offsets)
    if off.ndim != 1 or off.size < 2 or not np.issubdtype(off.dtype, np.integer):
        raise TypeError("offsets must be a 1-D integer array of nprob + 1 row boundaries")
    off = np.ascontiguousarray(off, dtype=np.int64)
    lengths = np.diff(off)
    if off[0] != 0 or off[-1] != rows:
        raise ValueError(f"offsets must start at 0 and end at the number of rows ({rows}); got {off[0]} .. {off[-1]}")
    if np.any(lengths <= 0):
        raise ValueError("offsets must be strictly increasing (every problem needs at least one row)")
    if int(lengths.max()) > cap:
        raise ValueError(f"a problem has {int(lengths.max())} rows; batched calls admit at most {cap} at this d")
    return torch.from_numpy(off).to(ref.device), off.size - 1


def batched_fixed_point(losses, offsets, *, tol=1e-3, maxiter=100, out=None, results=None):
    """rlvi_batched_fixed_point_f64: update_weights (rlvi.py:8-20) on every segment [offsets[b], offsets[b+1]) of `losses`.
    `offsets` is a host integer array.  Returns (pi, results): `results` is a device float64 [nprob, 5] buffer holding one
    rlvi_fp_result per problem (`batched_results` decodes it)."""
    dev = _dev(losses)
    f64 = torch.float64
    _chk(losses, f64, "losses")
    if losses.dim() != 1:
        raise ValueError("losses must be 1-D (the problems packed back to back)")
    n = losses.numel()
    ctx = _ctx(dev)
    offs, nprob = _batched_offsets(offsets, n, ctx.lib.rlvi_batched_max_rows(1), losses)
    if out is None:
        out = torch.empty(n, dtype=f64, device=losses.device)
    _len(_chk(out, f64, "out"), n, "out")
    if results is None:
        results = torch.empty(nprob, 5, dtype=f64, device=losses.device)
    _len(_chk(results, f64, "results"), 5 * nprob, "results")
    _same_device(losses, out, results)
    rc = ctx.lib.rlvi_batched_fixed_point_f64(ctx.handle, _p(losses), _p(offs), nprob, n, float(tol), int(maxiter),
                                              _p(out), _p(results), _stream(dev))
    _lib.check(rc, "rlvi_batched_fixed_point_f64")
    return out, results


def batched_results(results):
    """The [nprob, 5] device buffer of batched_fixed_point as a NumPy structured array (fields of rlvi_fp_result)."""
    return results.cpu().numpy().reshape(-1).view(_RESULT_DTYPE).copy()


def _batched_xy(entry, max_rows, X, y, offsets, code, D_extra, d_max, d_what, tol, maxiter):
    """The body of batched_em and batched_logistic: checks X [rows, d] (1 <= d <= d_max) and y [rows] (when given),
    uploads the offsets against the cap `max_rows` at d, allocates (theta [nprob, d + D_extra], iters, status) and calls
    the C entry point `entry` with model / mstep `code`."""
    dev = _dev(X)
    f64 = torch.float64
    _chk(X, f64, "X")
    if X.dim() != 2:
        raise ValueError("X must be [rows, d]")
    rows, d = X.shape
    if not 1 <= d <= d_max:
        raise ValueError(f"{d_what} 1 <= d <= {d_max} (got d = {d})")
    if y is not None:
        _len(_chk(y, f64, "y"), rows, "y")
    _same_device(X, y)
    if int(maxiter) < 0:
        raise ValueError("maxiter must be >= 0")
    ctx = _ctx(dev)
    offs, nprob = _batched_offsets(offsets, rows, getattr(ctx.lib, max_rows)(d), X)
    theta = torch.empty(nprob, d + D_extra, dtype=f64, device=X.device)
    iters = torch.empty(nprob, dtype=torch.int32, device=X.device)
    status = torch.empty(nprob, dtype=torch.int32, device=X.device)
    rc = getattr(ctx.lib, entry)(ctx.handle, int(code), _p(X), _p(y), _p(offs), nprob, rows, d, float(tol), int(maxiter),
                                 _p(theta), _p(iters), _p(status), _stream(dev))
    _lib.check(rc, entry)
    return theta, iters, status


def batched_em(model, X, y, offsets, *, tol=1e-3, maxiter=100):
    """rlvi_batched_em_f64: the EM loop of rlvi.mean (model BATCHED_MEAN, y None) or rlvi.linear_regression
    (BATCHED_LINREG) on every segment of the rows of X [rows, d] (and y [rows]).  `offsets` is a host integer array.
    Returns device tensors (theta [nprob, d] float64, iters [nprob] int32, status [nprob] int32); status 0 = stop test met,
    1 = maxiter reached, 2 = the normal equations failed the pivot test: theta is NaN, solve that problem with
    rlvi.linear_regression."""
    if model not in (BATCHED_MEAN, BATCHED_LINREG):
        raise ValueError("model must be BATCHED_MEAN or BATCHED_LINREG")
    if model == BATCHED_MEAN and y is not None:
        raise ValueError("the mean model takes no y")
    if model == BATCHED_LINREG and y is None:
        raise ValueError("linear regression needs y")
    return _batched_xy("rlvi_batched_em_f64", "rlvi_batched_max_rows", X, y, offsets, model, 0, 64,
                       "batched calls support", tol, maxiter)


def batched_logistic_max_rows(d) -> int:
    """rlvi_batched_logistic_max_rows: rows one problem of batched_logistic may have at `d` features (0 outside 1..63)."""
    return int(_lib.load().rlvi_batched_logistic_max_rows(int(d)))


def batched_logistic(X, y, offsets, *, mstep, tol=1e-2, maxiter=100):
    """rlvi_batched_logistic_f64: the EM loop of rlvi.logistic_regression on every segment of the rows of X [rows, d] and
    y [rows], with the Newton M-step of utils.sklearn_log_reg (mstep BATCHED_LOGREG_NEWTON) or utils.mm_log_reg
    (BATCHED_LOGREG_MM).  `offsets` is a host integer array.  Returns device tensors (theta [nprob, d + 1] float64,
    intercept first; iters [nprob] int32; status [nprob] int32): status 0 = stop test met, 1 = maxiter reached, 2 = theta
    is NaN, solve that problem with rlvi.logistic_regression."""
    if mstep not in (BATCHED_LOGREG_NEWTON, BATCHED_LOGREG_MM):
        raise ValueError("mstep must be BATCHED_LOGREG_NEWTON or BATCHED_LOGREG_MM")
    if y is None:
        raise ValueError("logistic regression needs y")
    return _batched_xy("rlvi_batched_logistic_f64", "rlvi_batched_logistic_max_rows", X, y, offsets, mstep, 1, 63,
                       "batched logistic regression supports", tol, maxiter)


def sever_pass(X, u, op, scalar, *, a=None, b=None, active=None, out0=None, out1=None, out2=None):
    """rlvi_sever_pass_f64 (sever.py:22-31 / :95-104).  op 0: c = scalar (X u - b) -> (c, active c^2, 1/c);
    op 1: scores (a (X u) - scalar)^2, -1 for inactive rows.  Returns (out0, out1, out2)."""
    dev = _dev(X)
    f64 = torch.float64
    _chk(X, f64, "X")
    if X.dim() != 2:
        raise ValueError("X must be [n, d]")
    n, d = X.shape
    _len(_chk(u, f64, "u"), d, "u")
    _len(_chk(a, f64, "a"), n, "a")
    _len(_chk(b, f64, "b"), n, "b")
    _len(_chk(active, f64, "active"), n, "active")
    if op not in (0, 1):
        raise ValueError("op must be 0 or 1")
    if op == 1 and a is None:
        raise ValueError("op 1 needs the coefficients a")
    if out0 is None:
        out0 = torch.empty(n, dtype=f64, device=X.device)
    if op == 0:
        if out1 is None:
            out1 = torch.empty(n, dtype=f64, device=X.device)
        if out2 is None:
            out2 = torch.empty(n, dtype=f64, device=X.device)
    for t, name in ((out0, "out0"), (out1, "out1"), (out2, "out2")):
        _len(_chk(t, f64, name), n, name)
    _same_device(X, u, a, b, active, out0, out1, out2)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_sever_pass_f64(ctx.handle, _p(X), n, d, _p(u), int(op), float(scalar), _p(a), _p(b), _p(active),
                                     _p(out0), _p(out1), _p(out2), _stream(dev))
    _lib.check(rc, "rlvi_sever_pass_f64")
    return out0, out1, out2


def wce_fwd_bwd(logits, labels, weights, residuals, *, indexes=None, want_grad=True, want_per_sample=False,
                want_correct=False):
    """rlvi_wce_fwd_bwd_f32.  Returns dict(loss [1], dlogits | None, per_sample | None, correct | None)."""
    dev = _dev(logits)
    f32 = torch.float32
    _chk(logits, f32, "logits")
    if logits.dim() != 2:
        raise ValueError("logits must be [batch, classes]")
    b, c = logits.shape
    _len(_chk(labels, torch.int64, "labels"), b, "labels")
    _len(_chk(indexes, torch.int64, "indexes"), b, "indexes")
    _chk(weights, f32, "weights")
    _chk(residuals, f32, "residuals")
    _same_device(logits, labels, indexes, weights, residuals)
    n_train = weights.numel()
    if residuals.numel() != n_train:
        raise ValueError("residuals and weights must have the same length")
    if indexes is None and n_train < b:
        raise ValueError("identity indexes need n_train >= batch")
    out_loss = torch.empty(1, dtype=f32, device=logits.device)
    dlogits = torch.empty_like(logits) if want_grad else None
    per = torch.empty(b, dtype=f32, device=logits.device) if want_per_sample else None
    correct = torch.empty(2, dtype=torch.int32, device=logits.device) if want_correct else None
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_wce_fwd_bwd_f32(ctx.handle, _p(logits), _p(labels), _p(indexes), _p(weights), _p(residuals), b,
                                      c, n_train, _p(per), _p(dlogits), _p(out_loss), _p(correct), _stream(dev))
    _lib.check(rc, "rlvi_wce_fwd_bwd_f32")
    return {"loss": out_loss, "dlogits": dlogits, "per_sample": per, "correct": correct}


def fn_threshold(weights, alpha=0.05, prev_threshold=0.0, truncate=False, *, out=None):
    """rlvi_fn_threshold_f32: false_negative_criterion (+ optional truncation), train_rlvi.py:41-49,102-103."""
    dev = _dev(weights)
    _chk(weights, torch.float32, "weights")
    if out is None:
        out = torch.empty(1, dtype=torch.float32, device=weights.device)
    _len(_chk(out, torch.float32, "out"), 1, "out")
    _same_device(weights, out)
    ctx = _ctx(dev)
    rc = ctx.lib.rlvi_fn_threshold_f32(ctx.handle, _p(weights), weights.numel(), float(alpha),
                                       float(prev_threshold), 1 if truncate else 0, _p(out), _stream(dev))
    _lib.check(rc, "rlvi_fn_threshold_f32")
    return out


def em_step_logistic_host(X, y, params, *, tol=1e-3, maxiter=100, want_pi=True, device=0, pi_out=None,
                          moments_out=None, group=None, n_global=None):
    """rlvi_em_step_logistic_host on HOST arrays (NumPy or CPU torch tensors, FP64, C-contiguous; pinned
    memory makes the copies asynchronous).  Returns dict(pi, moments, result)."""
    def host_ptr(a, name):
        if isinstance(a, torch.Tensor):
            if a.is_cuda or a.dtype != torch.float64 or not a.is_contiguous():
                raise TypeError(f"{name}: need a contiguous CPU float64 tensor")
            return C.c_void_p(a.data_ptr()), tuple(a.shape)
        a = np.ascontiguousarray(a, dtype=np.float64)
        return C.c_void_p(a.ctypes.data), a.shape, a

    hx = host_ptr(X, "X")
    hy = host_ptr(y, "y")
    hp = host_ptr(params, "params")
    n, d = hx[1]
    if hy[1] != (n,) or hp[1] != (d + 1,):
        raise ValueError("shape mismatch: X [n,d], y [n], params [d+1]")
    nm = _lib.load().rlvi_moments_out_doubles(d)

    def chk_out(a, count, name):
        """The C side copies `count` doubles into a raw host pointer: length, dtype and layout are checked here."""
        if a is None:
            return
        if isinstance(a, torch.Tensor):
            ok = (not a.is_cuda) and a.dtype == torch.float64 and a.is_contiguous() and a.numel() == count
        else:
            ok = isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"] and a.size == count
        if not ok:
            raise ValueError(f"{name} must be a C-contiguous CPU float64 buffer of exactly {count} elements")

    chk_out(pi_out, n, "pi_out")
    chk_out(moments_out, nm, "moments_out")
    ctx = _lib.context(int(device))
    if want_pi and pi_out is None:
        pi_out = np.empty(n, dtype=np.float64)
    if moments_out is None:
        moments_out = np.empty(nm, dtype=np.float64)
    res = _lib.FpResult()

    def out_ptr(a):
        if a is None:
            return None
        return C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else C.c_void_p(a.ctypes.data)

    if group is None or group.world == 1:
        rc = ctx.lib.rlvi_em_step_logistic_host(ctx.handle, hx[0], hy[0], n, d, hp[0], float(tol), int(maxiter),
                                                out_ptr(pi_out) if want_pi else None, out_ptr(moments_out),
                                                C.byref(res))
    else:      # this rank's shard of a sample-sharded data set (rlvi_b200.dist.ShardGroup)
        fpd = group.fp_dist(int(n_global))
        std = group.stats_dist()
        rc = ctx.lib.rlvi_em_step_logistic_host_sharded(ctx.handle, hx[0], hy[0], n, d, hp[0], float(tol),
                                                        int(maxiter), out_ptr(pi_out) if want_pi else None,
                                                        out_ptr(moments_out), C.byref(res), C.byref(fpd),
                                                        C.byref(std))
    _lib.check(rc, "rlvi_em_step_logistic_host")
    if res.iters < 0:
        raise _lib.RlviError("fixed-point kernel aborted: a grid barrier timed out")
    return {"pi": pi_out if want_pi else None, "moments": moments_out,
            "result": {"eps": res.eps, "rho": res.rho, "sum_pi": res.sum_pi, "err": res.err, "iters": res.iters,
                       "converged": res.converged}}
