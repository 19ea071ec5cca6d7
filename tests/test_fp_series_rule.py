"""The switch rule and the series evaluation of the fixed point's series passes (rlvi_b200/fp_series.py, the NumPy
restatement of fixed_point.cu), against the direct sums of every pass."""
import math
import os
import re

import numpy as np
import pytest

from rlvi_b200 import fp_series

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden_e(name):
    return np.exp(-np.load(os.path.join(GOLDEN, "update_weights_%s.npz" % name))["losses"])


def _collapse_e(n=1 << 15, seed=7):
    """e = sigmoid(margin) of a noisy logistic model, as bench.py's loss pass makes it: all of e in (0, 1)."""
    rng = np.random.default_rng(seed)
    m = rng.normal(1.0, 2.5, n)
    return 1.0 / (1.0 + np.exp(-m))


def _trajectory(e, maxiter=40, pi0=0.95):
    """(rho_new, rho_old) of every pass k >= 2 of the streamed recurrence (tol = -1: no stop test)."""
    n = float(e.size)
    eps = 1.0 - pi0
    rho, out = eps / (1.0 - eps), []
    s = math.fsum(e / (rho + e))
    for _ in range(maxiter - 1):
        eps = 1.0 - s / n
        rho_next = eps / (1.0 - eps)
        if not (math.isfinite(rho_next) and rho_next > 0):
            break
        out.append((rho_next, rho))
        rho = rho_next
        s = math.fsum(e / (rho + e))
    return out


def _rel(a, b):
    return abs(a - b) / abs(b)


@pytest.mark.parametrize("data", ["n40", "n1000", "n4096", "n16384", "collapse"])
def test_admitted_passes_match_direct_sums(data):
    e = _golden_e(data) if data != "collapse" else _collapse_e()
    two_e = fp_series.scale(float(e.max()))
    P = fp_series.power_sums(e, two_e)
    admitted = rejected_bad = 0
    for rho_new, rho_old in _trajectory(e):
        q = two_e / min(rho_new, rho_old)
        s1, s2 = fp_series.series_sums(P, two_e, rho_new, rho_old)
        d1, d2 = fp_series.direct_sums(e, rho_new, rho_old)
        worst = max(_rel(s1, d1), _rel(s2, d2))
        if fp_series.admits(q):
            admitted += 1
            assert worst <= 1e-15, (q, worst)
        elif worst > 1e-15:
            rejected_bad += 1
    assert admitted >= 5               # collapse data: the series takes over
    assert rejected_bad >= 1           # and the passes before it would have been wrong


def test_rule_bounds_are_bounds():
    """Where the rule would admit a pass, the true truncation error of each series is below its a-priori bound:
    checked with the worst case for the bound, every z = 1 (P_j = n), against exact closed forms."""
    for q in np.geomspace(1e-4, 0.3, 60):
        b1, b2 = fp_series.bounds(q)
        rho_new = 1.0 / q
        rho_old = rho_new + 1.0                      # drho != 0; q = 2^E / min(rho', rho) with 2^E = 1
        P = np.full(fp_series.J, 1.0)
        s1, s2 = fp_series.series_sums(P, 1.0, rho_new, rho_old)
        exact1 = 1.0 / (rho_new + 1.0)
        exact2 = (rho_old - rho_new) ** 2 / ((rho_new + 1.0) ** 2 * (rho_old + 1.0) ** 2)
        assert _rel(s1, exact1) <= b1 + 2e-15       # plus rounding
        assert _rel(s2, exact2) <= b2 + 2e-15


def test_non_collapse_never_builds():
    """eps ~ 0.4 (losses below zero): the power sums are never built, so the kernel streams every pass as before."""
    e = np.exp(-np.resize(np.load(os.path.join(GOLDEN, "update_weights_neg.npz"))["losses"], 1 << 14))
    passes, r = fp_series.replay(e)
    assert 0.3 < r["eps"] < 0.5
    assert all(p["mode"] in ("stream", "sum_only", "sum_only+full") for p in passes)


@pytest.mark.parametrize("data", ["n1000", "n16384"])
def test_schedule_same_result_as_streaming(data):
    e = _golden_e(data)
    passes, r = fp_series.replay(e)
    _, r0 = fp_series.replay(e, series=False)
    assert any(p["mode"] == "build" for p in passes)
    assert sum(p["mode"] == "build" for p in passes) == 1
    assert r["iters"] == r0["iters"] and r["converged"] == r0["converged"]
    assert fp_series.streamed_passes(passes) < r["iters"] // 2


def test_model_constants_match_kernel():
    src = open(os.path.join(ROOT, "rlvi_b200", "csrc", "fixed_point.cu")).read()
    assert int(re.search(r"constexpr int kFpSeriesJ = (\d+);", src).group(1)) == fp_series.J
    assert "0x1p-40" in src and fp_series.NEAR_TOL == 2.0 ** -40
