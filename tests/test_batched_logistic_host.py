"""Host logic of the batched logistic regression without a GPU.

1. rlvi_b200.ops.batched_logistic against a recording stub of the library: well-formed calls reach
   rlvi_batched_logistic_f64 with the right scalars, and every bad offset vector, dtype, d, y, mstep or length is refused
   on the host before a pointer is handed over.
2. rlvi_b200.batched.logistic_regression's packing and unpacking (stacked arrays, ragged lists, NumPy vs tensor returns)
   and its substitution of the host-solve problems, with ops.batched_logistic replaced by a torch-CPU double that runs
   the NumPy oracle's MM fit per segment.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import rlvi_np
from rlvi_b200 import batched, ops, rlvi, synth

CAP = {1: 2071, 8: 2008, 10: 1981, 63: 1024}


def cap(d):
    return CAP.get(d, 1024) if 1 <= d <= 63 else 0


class _Recorder:
    def __init__(self):
        self.calls = []

    def rlvi_batched_logistic_max_rows(self, d):
        return cap(d)

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
    theta, iters, status = ops.batched_logistic(f64(100, 10), f64(100), np.array([0, 40, 100]),
                                                mstep=ops.BATCHED_LOGREG_MM, tol=1e-3, maxiter=3)
    assert theta.shape == (2, 11) and iters.dtype == torch.int32 and status.shape == (2,)
    ops.batched_logistic(f64(1024, 63), f64(1024), torch.tensor([0, 1024]), mstep=ops.BATCHED_LOGREG_NEWTON)
    ops.batched_logistic(f64(5, 1), f64(5), [0, 5], mstep=ops.BATCHED_LOGREG_NEWTON, maxiter=0)
    (n1, a1), (n2, a2), (n3, a3) = rec.calls
    assert n1 == n2 == n3 == "rlvi_batched_logistic_f64"
    assert a1[1] == ops.BATCHED_LOGREG_MM == 1 and a1[5:10] == (2, 100, 10, 1e-3, 3)
    assert a2[1] == ops.BATCHED_LOGREG_NEWTON == 0 and a2[5:10] == (1, 1024, 63, 1e-2, 100)
    assert a3[5:10] == (1, 5, 1, 1e-2, 0)
    assert all(a is not None for a in a1[2:5] + a1[10:13])


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
    for mstep in (ops.BATCHED_LOGREG_NEWTON, ops.BATCHED_LOGREG_MM):
        with pytest.raises(err):
            ops.batched_logistic(f64(100, 3), f64(100), offsets, mstep=mstep)
    assert rec.calls == []


def test_bad_shapes_dtypes_and_sizes_are_refused(rec):
    off = [0, 50, 100]
    N = ops.BATCHED_LOGREG_NEWTON
    with pytest.raises(TypeError):
        ops.batched_logistic(torch.zeros(100, 4, dtype=torch.float32), f64(100), off, mstep=N)
    with pytest.raises(TypeError):
        ops.batched_logistic(f64(100, 4), torch.zeros(100, dtype=torch.float32), off, mstep=N)
    with pytest.raises(TypeError):
        ops.batched_logistic(f64(4, 100).t(), f64(100), off, mstep=N)                # not contiguous
    for d in (0, 64):
        with pytest.raises(ValueError, match="1 <= d <= 63"):
            ops.batched_logistic(f64(100, d), f64(100), off, mstep=N)
    with pytest.raises(ValueError):
        ops.batched_logistic(f64(100, 4), f64(99), off, mstep=N)                      # y length != rows
    with pytest.raises(ValueError):
        ops.batched_logistic(f64(100, 4), None, off, mstep=N)                         # no y
    with pytest.raises(ValueError):
        ops.batched_logistic(f64(100), f64(100), off, mstep=N)                        # X not 2-D
    for bad in (2, -1, "mm"):
        with pytest.raises(ValueError, match="mstep"):
            ops.batched_logistic(f64(100, 4), f64(100), off, mstep=bad)
    with pytest.raises(ValueError, match="maxiter"):
        ops.batched_logistic(f64(100, 4), f64(100), off, mstep=N, maxiter=-1)
    with pytest.raises(ValueError, match="at most 1024"):
        ops.batched_logistic(f64(1100, 63), f64(1100), [0, 1025, 1100], mstep=N)     # over the cap
    with pytest.raises(ValueError, match="at most 2008"):
        ops.batched_logistic(f64(2100, 8), f64(2100), [0, 2009, 2100], mstep=N)
    assert rec.calls == []


# ---- rlvi_b200.batched.logistic_regression on a torch-CPU double of ops.batched_logistic --------------------------------
def _fake_logistic(X, y, offsets, *, mstep, tol=1e-2, maxiter=100):
    off = np.asarray(offsets)
    Xn, yn = X.numpy(), y.numpy()
    theta, iters, status = [], [], []
    for b in range(len(off) - 1):
        s, e = int(off[b]), int(off[b + 1])
        Xa = np.hstack([np.ones((e - s, 1)), Xn[s:e]])
        if np.linalg.matrix_rank(Xa) < Xa.shape[1]:
            theta.append(np.full(Xa.shape[1], np.nan))
            status.append(batched.HOST_SOLVE)
        else:
            theta.append(rlvi_np.logistic_regression_mm(Xn[s:e], yn[s:e], maxiter=maxiter, tol=tol))
            status.append(0)
        iters.append(0)
    return (torch.from_numpy(np.array(theta)), torch.tensor(iters, dtype=torch.int32),
            torch.tensor(status, dtype=torch.int32))


@pytest.fixture
def double(monkeypatch):
    host_solved = []

    def fake_logreg(X, y, maxiter=100, tol=1e-2, mstep="sklearn"):
        assert isinstance(X, torch.Tensor) and X.is_contiguous()
        host_solved.append((tuple(X.shape), mstep))
        if X.shape[0] < 3:
            raise RuntimeError("sklearn_log_reg: Newton iteration did not converge in 60 steps")
        return torch.full((X.shape[1] + 1,), X.shape[0] + maxiter + 1000 * tol, dtype=torch.float64)

    monkeypatch.setattr(batched, "default_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(ops, "batched_logistic", _fake_logistic)
    monkeypatch.setattr(ops, "batched_logistic_max_rows", cap)
    monkeypatch.setattr(rlvi, "logistic_regression", fake_logreg)
    return host_solved


def problem(n, d, seed, eps=0.2):
    X, y, _ = synth.logistic_data(n, d, corruption=eps, seed=seed)
    return X, y


def test_stacked_and_ragged(double):
    g = load_golden("logreg_mm_n1500_d8")
    pads = [problem(n, 8, seed=10 + k) for k, n in enumerate((60, 333, 1200))]
    X = [pads[0][0], g["X"], pads[1][0], pads[2][0]]
    y = [pads[0][1], g["y"], pads[1][1], pads[2][1]]
    theta = batched.logistic_regression(X, y, mstep="mm")
    assert isinstance(theta, np.ndarray) and theta.shape == (4, 9)
    for b in range(4):
        assert np.array_equal(theta[b], rlvi_np.logistic_regression_mm(X[b], y[b]))
    t = batched.logistic_regression([torch.from_numpy(a) for a in X], [torch.from_numpy(a) for a in y], mstep="mm")
    assert isinstance(t, torch.Tensor) and torch.equal(t, torch.from_numpy(theta))
    Xs = np.stack([g["X"][:200], g["X"][200:400]])
    ys = np.stack([g["y"][:200], g["y"][200:400]])
    st = batched.logistic_regression(Xs, ys, mstep="mm", maxiter=5, tol=1e-3)
    rg = batched.logistic_regression(list(Xs), list(ys), mstep="mm", maxiter=5, tol=1e-3)
    assert st.shape == (2, 9) and np.array_equal(st, rg)
    assert np.array_equal(st[1], rlvi_np.logistic_regression_mm(Xs[1], ys[1], maxiter=5, tol=1e-3))
    assert double == []
    with pytest.raises(ValueError, match="same problems"):
        batched.logistic_regression(X, y[:3])
    with pytest.raises(ValueError, match="mstep"):
        batched.logistic_regression(X, y, mstep="newton")


def test_host_solve_problems_are_substituted(double):
    X0, y0 = problem(80, 5, seed=1)
    Xdup, ydup = problem(90, 5, seed=2)
    Xdup[:, 1] = Xdup[:, 3]
    X2, y2 = problem(70, 5, seed=3)
    theta = batched.logistic_regression([X0, Xdup, X2], [y0, ydup, y2], maxiter=7, mstep="sklearn")
    assert double == [((90, 5), "sklearn")]
    assert np.array_equal(theta[1], np.full(6, 90 + 7 + 10.0))
    assert np.array_equal(theta[[0, 2]], batched.logistic_regression([X0, X2], [y0, y2], maxiter=7))


def test_a_drop_in_exception_names_the_problem(double):
    X0, y0 = problem(80, 3, seed=4)
    with pytest.raises(RuntimeError, match=r"problem 1: sklearn_log_reg: Newton iteration did not converge"):
        batched.logistic_regression([X0, X0[:2], X0], [y0, y0[:2], y0])


def test_oversize_and_unsupported_problems_raise(double):
    with pytest.raises(ValueError, match=r"at most 1981 .*rlvi_b200\.rlvi\.logistic_regression"):
        batched.logistic_regression([np.zeros((1982, 10))], [np.zeros(1982)])
    with pytest.raises(ValueError, match=r"1 <= d <= 63 .*rlvi_b200\.rlvi\.logistic_regression"):
        batched.logistic_regression(np.zeros((2, 100, 64)), np.zeros((2, 100)))
    with pytest.raises(ValueError, match="no problems"):
        batched.logistic_regression([], [])
    assert double == []
