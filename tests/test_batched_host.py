"""Host logic of the batched entry points without a GPU.

1. rlvi_b200.ops.batched_fixed_point / batched_em against a recording stub of the library: well-formed calls reach the C
   entry points with the right scalars, and every bad offset vector, dtype, d or length is refused on the host before a
   pointer is handed over (the kernels index the packed arrays with the offsets).
2. rlvi_b200.batched's packing and unpacking (stacked arrays, ragged lists, NumPy vs tensor returns) and its substitution
   of the host-solve problems, with the two ops.batched_* functions replaced by a torch-CPU double that runs the NumPy
   oracle per segment; checked against the reference's goldens.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import rlvi_np
from rlvi_b200 import batched, ops, rlvi

CAP = {1: 1530, 2: 1522, 10: 1386, 64: 1024}


class _Recorder:
    def __init__(self):
        self.calls = []

    def rlvi_batched_max_rows(self, d):
        return CAP.get(d, 1024) if 1 <= d <= 64 else 0

    def __getattr__(self, name):
        if not name.startswith("rlvi_"):
            raise AttributeError(name)

        def fn(*args):
            self.calls.append((name, args))
            return 0
        return fn


class _Ctx:
    def __init__(self):
        self.lib = _Recorder()
        self.handle = C.c_void_p(1)


@pytest.fixture
def rec(monkeypatch):
    ctx = _Ctx()

    def chk(t, dtype, name):            # ops._chk minus the is_cuda requirement
        if t is None:
            return None
        if t.dtype != dtype or not t.is_contiguous():
            raise TypeError(f"{name} must be a contiguous tensor of dtype {dtype}")
        return t

    monkeypatch.setattr(ops, "_dev", lambda t: 0)
    monkeypatch.setattr(ops, "_stream", lambda dev: None)
    monkeypatch.setattr(ops, "_ctx", lambda dev: ctx)
    monkeypatch.setattr(ops, "_chk", chk)
    return ctx.lib


def f64(*shape):
    return torch.zeros(shape, dtype=torch.float64)


def test_well_formed_calls_reach_the_abi(rec):
    pi, res = ops.batched_fixed_point(f64(100), [0, 40, 100], tol=1e-4, maxiter=7)
    assert pi.shape == (100,) and res.shape == (2, 5)
    theta, iters, status = ops.batched_em(ops.BATCHED_LINREG, f64(100, 10), f64(100), np.array([0, 40, 100]), maxiter=3)
    assert theta.shape == (2, 10) and iters.dtype == torch.int32 and status.shape == (2,)
    ops.batched_em(ops.BATCHED_MEAN, f64(64, 64), None, torch.tensor([0, 64]))
    (n1, a1), (n2, a2), (n3, a3) = rec.calls
    assert n1 == "rlvi_batched_fixed_point_f64" and a1[3:7] == (2, 100, 1e-4, 7)
    assert n2 == "rlvi_batched_em_f64" and a2[1] == ops.BATCHED_LINREG and a2[5:10] == (2, 100, 10, 1e-3, 3)
    assert n3 == "rlvi_batched_em_f64" and a3[1] == ops.BATCHED_MEAN and a3[3] is None and a3[5:8] == (1, 64, 64)


@pytest.mark.parametrize("offsets, err", [
    ([0, 40, 40, 100], ValueError),         # empty problem
    ([0, 60, 40, 100], ValueError),         # decreasing
    ([5, 40, 100], ValueError),             # does not start at 0
    ([0, 40, 99], ValueError),              # does not end at the rows
    ([0, 40, 101], ValueError),             # past the rows
    ([0], TypeError),                       # no problem
    ([[0, 100]], TypeError),                # not 1-D
    ([0.0, 100.0], TypeError),              # not integers
])
def test_bad_offsets_are_refused(rec, offsets, err):
    with pytest.raises(err):
        ops.batched_fixed_point(f64(100), offsets)
    with pytest.raises(err):
        ops.batched_em(ops.BATCHED_LINREG, f64(100, 3), f64(100), offsets)
    assert rec.calls == []


def test_bad_shapes_dtypes_and_sizes_are_refused(rec):
    off = [0, 50, 100]
    with pytest.raises(TypeError):
        ops.batched_fixed_point(torch.zeros(100, dtype=torch.float32), off)
    with pytest.raises(TypeError):
        ops.batched_em(ops.BATCHED_LINREG, torch.zeros(100, 4, dtype=torch.float32), f64(100), off)
    with pytest.raises(TypeError):
        ops.batched_em(ops.BATCHED_LINREG, f64(4, 100).t(), f64(100), off)            # not contiguous
    for d in (0, 65):
        with pytest.raises(ValueError, match="1 <= d <= 64"):
            ops.batched_em(ops.BATCHED_MEAN, f64(100, d), None, off)
    with pytest.raises(ValueError):
        ops.batched_em(ops.BATCHED_LINREG, f64(100, 4), f64(99), off)                 # y length != rows
    with pytest.raises(ValueError):
        ops.batched_em(ops.BATCHED_LINREG, f64(100, 4), None, off)                    # LINREG without y
    with pytest.raises(ValueError):
        ops.batched_em(ops.BATCHED_MEAN, f64(100, 4), f64(100), off)                  # MEAN with y
    with pytest.raises(ValueError):
        ops.batched_em(7, f64(100, 4), f64(100), off)                                 # unknown model
    with pytest.raises(ValueError, match="at most 1024"):
        ops.batched_em(ops.BATCHED_MEAN, f64(1100, 64), None, [0, 1025, 1100])        # over the cap
    with pytest.raises(ValueError, match="at most 1530"):
        ops.batched_fixed_point(f64(1600), [0, 1531, 1600])
    with pytest.raises(ValueError):
        ops.batched_fixed_point(f64(100, 1), off)                                     # losses not 1-D
    assert rec.calls == []


# ---- rlvi_b200.batched on a torch-CPU double of the two ops entry points ------------------------------------------------
def _segments(off):
    return [(int(off[b]), int(off[b + 1])) for b in range(len(off) - 1)]


def _fake_fixed_point(losses, offsets, *, tol=1e-3, maxiter=100, out=None, results=None):
    off = np.asarray(offsets)
    l = losses.numpy()
    pi = np.empty_like(l)
    res = np.zeros((len(off) - 1, 5))
    for b, (s, e) in enumerate(_segments(off)):
        pi[s:e] = rlvi_np.update_weights(l[s:e], tol=tol, maxiter=maxiter)
    return torch.from_numpy(pi), torch.from_numpy(res)


def _fake_em(model, X, y, offsets, *, tol=1e-3, maxiter=100):
    off = np.asarray(offsets)
    Xn = X.numpy()
    theta, iters, status = [], [], []
    for s, e in _segments(off):
        if model == ops.BATCHED_MEAN:
            theta.append(rlvi_np.mean(Xn[s:e], maxiter=maxiter, tol=tol))
            iters.append(0)
            status.append(0)
        elif np.linalg.matrix_rank(Xn[s:e]) < Xn.shape[1]:
            theta.append(np.full(Xn.shape[1], np.nan))
            iters.append(0)
            status.append(batched.HOST_SOLVE)
        else:
            trace = []
            theta.append(rlvi_np.linear_regression(Xn[s:e], y.numpy()[s:e], maxiter=maxiter, tol=tol, trace=trace))
            iters.append(len(trace))
            status.append(0)
    return (torch.from_numpy(np.array(theta)), torch.tensor(iters, dtype=torch.int32),
            torch.tensor(status, dtype=torch.int32))


@pytest.fixture
def double(monkeypatch):
    host_solved = []

    def fake_linreg(X, y, maxiter=100, tol=1e-3):
        host_solved.append(X.shape)
        return torch.from_numpy(rlvi_np.linear_regression(X.numpy(), y.numpy(), maxiter=maxiter, tol=tol))

    monkeypatch.setattr(batched, "default_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(ops, "batched_fixed_point", _fake_fixed_point)
    monkeypatch.setattr(ops, "batched_em", _fake_em)
    monkeypatch.setattr(ops, "batched_max_rows", lambda d: CAP.get(d, 1024) if 1 <= d <= 64 else 0)
    monkeypatch.setattr(rlvi, "linear_regression", fake_linreg)
    return host_solved


def relmax(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def test_stacked_and_ragged_linear_regression(double):
    g = load_golden("config1_linreg_fixed_eps")
    theta = batched.linear_regression(g["X"][:5], g["y"][:5])
    assert isinstance(theta, np.ndarray) and theta.shape == (5, 10)
    assert relmax(theta, g["theta_rlvi"][:5]) < 1e-9
    gl = load_golden("linreg_n40_d10")
    X = [g["X"][0][:31], gl["X"], g["X"][1]]
    y = [g["y"][0][:31], gl["y"], g["y"][1]]
    theta = batched.linear_regression(X, y)
    assert theta.shape == (3, 10) and relmax(theta[1], gl["theta"]) < 1e-9
    assert relmax(theta[2], g["theta_rlvi"][1]) < 1e-9
    t = batched.linear_regression([torch.from_numpy(a) for a in X], [torch.from_numpy(a) for a in y])
    assert isinstance(t, torch.Tensor) and torch.equal(t, torch.from_numpy(theta))
    with pytest.raises(ValueError, match="same problems"):
        batched.linear_regression(X, y[:2])


def test_host_solve_problems_are_substituted(double):
    g = load_golden("linreg_n40_d10")
    Xdup = g["X"].copy()
    Xdup[:, 2] = Xdup[:, 6]
    theta = batched.linear_regression([g["X"], Xdup, g["X"][:6]], [g["y"], g["y"], g["y"][:6]])
    assert double == [(40, 10), (6, 10)]
    assert relmax(theta[0], g["theta"]) < 1e-9
    assert relmax(theta[1], rlvi_np.linear_regression(Xdup, g["y"])) == 0.0
    assert relmax(theta[2], rlvi_np.linear_regression(g["X"][:6], g["y"][:6])) == 0.0


@pytest.mark.parametrize("tag", ["mean_n100_d2", "mean_n768_d64"])
def test_mean_stacked_and_ragged(double, tag):
    g = load_golden(tag)
    X = g["X"]
    theta = batched.mean([X[:50], X, X[7:]])
    assert theta.shape == (3, X.shape[1]) and relmax(theta[1], g["theta"]) < 1e-9
    t = batched.mean(torch.from_numpy(np.stack([X, X])))
    assert isinstance(t, torch.Tensor) and t.shape == (2, X.shape[1]) and relmax(t[0].numpy(), g["theta"]) < 1e-9


def test_update_weights_shapes(double):
    g40, g1000 = load_golden("update_weights_n40"), load_golden("update_weights_n1000")
    pis = batched.update_weights([g40["losses"], g1000["losses"]])
    assert isinstance(pis, list) and pis[0].shape == (40,) and pis[1].shape == (1000,)
    assert relmax(pis[0], g40["pi"]) < 1e-9 and relmax(pis[1], g1000["pi"]) < 1e-9
    st = batched.update_weights(np.stack([g40["losses"], g40["losses"]]))
    assert isinstance(st, np.ndarray) and st.shape == (2, 40) and relmax(st[1], g40["pi"]) < 1e-9
    tl = batched.update_weights([torch.from_numpy(g40["losses"]), torch.from_numpy(g1000["losses"])])
    assert isinstance(tl, list) and isinstance(tl[1], torch.Tensor) and relmax(tl[1].numpy(), g1000["pi"]) < 1e-9
    ts = batched.update_weights(torch.from_numpy(np.stack([g40["losses"]] * 3)))
    assert isinstance(ts, torch.Tensor) and ts.shape == (3, 40)


def test_oversize_and_unsupported_problems_raise(double):
    with pytest.raises(ValueError, match=r"at most 1386 .*rlvi_b200\.rlvi\.linear_regression"):
        batched.linear_regression([np.zeros((1387, 10))], [np.zeros(1387)])
    with pytest.raises(ValueError, match=r"at most 1024 .*rlvi_b200\.rlvi\.mean"):
        batched.mean(np.zeros((2, 1025, 64)))
    with pytest.raises(ValueError, match=r"at most 1530 .*rlvi_b200\.rlvi\.update_weights"):
        batched.update_weights([np.zeros(1531)])
    with pytest.raises(ValueError, match="1 <= d <= 64"):
        batched.mean(np.zeros((2, 100, 65)))
    with pytest.raises(ValueError, match="no problems"):
        batched.mean([])
