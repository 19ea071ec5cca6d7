"""Series passes of the STANDARD fixed point against streaming every pass (RLVI_FP_SERIES=0) on the same e."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from rlvi_b200 import fp_series, ops  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

pytestmark = pytest.mark.gpu


def _e(name, n):
    """e = exp(-l) of a stored loss vector, tiled to n samples (collapse data: update_weights_n16384; losses below
    zero, eps ~ 0.3: update_weights_neg)."""
    losses = np.load(os.path.join(GOLDEN, "update_weights_%s.npz" % name))["losses"]
    return torch.from_numpy(np.exp(-np.resize(losses, n))).cuda()


def _run(e, series, **kw):
    old = os.environ.get("RLVI_FP_SERIES")
    os.environ["RLVI_FP_SERIES"] = "1" if series else "0"
    try:
        pi, res = ops.fixed_point(None, e_work=e, **kw)
        return pi.cpu().numpy(), ops.read_result(res)
    finally:
        if old is None:
            del os.environ["RLVI_FP_SERIES"]
        else:
            os.environ["RLVI_FP_SERIES"] = old


def _rel(a, b):
    return abs(a - b) / abs(b)


def _check_close(e, **kw):
    pi_s, r_s = _run(e, True, **kw)
    pi_t, r_t = _run(e, False, **kw)
    assert r_s["iters"] == r_t["iters"], (r_s, r_t)
    assert r_s["converged"] == r_t["converged"]
    assert _rel(r_s["eps"], r_t["eps"]) <= 1e-14
    assert _rel(r_s["sum_pi"], r_t["sum_pi"]) <= 1e-14
    nz = pi_t != 0.0                                  # e underflows to 0 for the largest losses: pi = 0 both ways
    assert np.array_equal(pi_s[~nz], pi_t[~nz])
    assert float(np.max(np.abs(pi_s[nz] - pi_t[nz]) / pi_t[nz])) <= 1e-13
    pi_2, r_2 = _run(e, True, **kw)                  # same bits on repeat
    assert r_2 == r_s and np.array_equal(pi_2, pi_s)
    return r_s


# 2^20: resident head in shared memory; 2^23 + 17: bulk-copy ring, odd n; 300001: ragged, grid kernel
@pytest.mark.parametrize("n", [1 << 20, (1 << 23) + 17, 300001])
def test_series_matches_streaming(n):
    e = _e("n16384", n)
    r = _check_close(e)
    if n <= 1 << 20:                                         # the model's schedule on the same e reaches the series
        passes, ref = fp_series.replay(e.cpu().numpy())
        assert any(p["mode"] == "series" for p in passes)
        assert r["iters"] == ref["iters"]


@pytest.mark.parametrize("maxiter", [12, 32])
def test_series_maxiter(maxiter):
    e = _e("n16384", (1 << 23) + 17)
    r = _check_close(e, tol=-1.0, maxiter=maxiter)
    assert r["iters"] == maxiter and r["converged"] == 0


def test_series_either_side_of_switch():
    n = 1 << 20
    e = _e("n16384", n)
    passes, _ = fp_series.replay(e.cpu().numpy())
    first = next(p["k"] for p in passes if p["mode"] == "series")
    for maxiter in (first - 1, first, first + 1):
        r = _check_close(e, maxiter=maxiter)
        assert r["iters"] == maxiter


@pytest.mark.parametrize("n", [1 << 20, (1 << 23) + 17])
def test_no_switch_is_bit_identical(n):
    e = _e("neg", n)
    pi_s, r_s = _run(e, True)
    pi_t, r_t = _run(e, False)
    assert 0.3 < r_t["eps"] < 0.5
    assert r_s == r_t
    assert np.array_equal(pi_s, pi_t)
