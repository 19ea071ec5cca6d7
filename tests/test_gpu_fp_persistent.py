"""The persistent fixed-point kernels (fp_kernel_f64, fp_kernel_deep_f32: every n above the single-CTA kernel's 28 672
doubles / 57 344 floats) against restated reference loops, where they are most likely to go wrong:

* rcp_fast's range edges.  From pass 2 on the aligned (VEC) path takes pi' from rcp.approx.ftz.f64, which flushes a
  result below 2^-1022 to zero: an argument in [2^1022, 2^1024) gives a finite 0, not a NaN / inf that the trip's
  non-finite test would catch.  Losses near -354.5 put the STANDARD full trip's (rho' + e)(rho + e) there, losses near
  -709 the sum-only trip's rho' + e; 720 (e subnormal) and 800 (e = 0) go through the existing IEEE fallback.
* the ONLINE variant, the warm start (rlvi_fixed_point_init_f64) and the FP32 deep variant at persistent-kernel sizes,
  through every route: streaming modes (RLVI_FP_CACHE_SLOTS), series passes off, 8-byte aligned views (scalar path),
  a precomputed e and a scale tensor.

Tolerances as in test_gpu_parity.py.  The iteration count is asserted only where no pass's err lies within 1e-9 of tol
(the seeds below keep every decision well away from it).
"""
import functools

import numpy as np
import pytest
import torch

from oracle import deep_ref, rlvi_np

pytestmark = pytest.mark.gpu

F64_TOL = 1e-9
F32_TOL = 1e-5
STANDARD, ONLINE = 0, 1
FLUSH = 2.0 ** 1022          # rcp.approx.ftz.f64 returns 0 for every finite argument from here on
LN2 = float(np.log(2.0))


@pytest.fixture(scope="module")
def dev():
    from rlvi_b200 import _lib
    _lib.load()
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def relmax(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def pi_tol(ref_pi):
    return max(F64_TOL, 4 * 2.0 ** -53 / max(float(np.mean(ref_pi)), 1e-300))


# ---- reference ---------------------------------------------------------------------------------------------------
def ref_loop(losses, variant, tol, maxiter=100, pi0=None):
    """standard-learning/rlvi.py:8-20 (STANDARD) or online-learning/main.py:45-58 (ONLINE), in the reference's operation
    order, started from the constant pi0 (default 0.95 / 0.5), recording (eps, rho, err, sum pi') of every pass.
    Returns dict(pi = the last pi' (ONLINE: normalised by max(pi') n), raw = the last pi', passes, iters)."""
    e = np.exp(-losses)
    pi = np.full_like(e, (0.95 if variant == STANDARD else 0.5) if pi0 is None else pi0)
    passes = []
    for k in range(1, maxiter + 1):
        avg = np.mean(pi)
        eps = 1 - avg
        if variant == STANDARD:
            rho = eps / (1 - eps)
            new = e / (rho + e)
        else:
            rho = avg / (1 - avg)
            new = rho * e / (1 + rho * e)
        err = np.linalg.norm(new - pi)
        passes.append((eps, rho, err, new.sum()))
        if err < tol:
            break
        pi = new
    out = new if variant == STANDARD else new / (np.max(new) * len(new))
    return {"pi": out, "raw": new, "passes": passes, "iters": k}


def decided_with_margin(ref, tol):
    """No pass's stop test err < tol is within 1e-9 relative of tol: the kernel's sums, rounded differently, decide alike."""
    return all(abs(p[2] - tol) > 1e-9 * abs(tol) for p in ref["passes"])


def flush_hits(ref, e_x, variant):
    """Passes k >= 2 whose fast-reciprocal argument at e = e_x lands in [2^1022, inf): (full trip, sum-only trip)."""
    full = summ = 0
    with np.errstate(over="ignore"):
        for (_, r_old, _, _), (_, r_new, _, _) in zip(ref["passes"], ref["passes"][1:]):
            a = (r_new + e_x) * (r_old + e_x) if variant == STANDARD else (1 + r_new * e_x) * (1 + r_old * e_x)
            full += FLUSH <= a < np.inf
            summ += variant == STANDARD and FLUSH <= r_new + e_x < np.inf
    return full, summ


def check(pi, res, ref, tol, variant):
    from rlvi_b200 import ops
    r = ops.read_result(res)
    eps, _, err, s = ref["passes"][-1]
    tpi = pi_tol(ref["pi"]) if variant == STANDARD else F64_TOL
    assert relmax(pi.cpu().numpy(), ref["pi"]) < tpi
    if decided_with_margin(ref, tol):
        assert r["iters"] == ref["iters"]
    assert abs(r["eps"] - eps) <= F64_TOL * abs(eps) + 4 * 2.0 ** -53      # eps = 1 - mean(pi) is quantised to ulp(1)
    # rho = eps / (1 - eps) inherits that quantum (SURVEY.md H1), and err with it
    assert abs(r["err"] - err) <= max(1e-6, pi_tol(ref["raw"])) * err + 1e-15
    assert abs(r["sum_pi"] - s) <= (pi_tol(ref["raw"]) if variant == STANDARD else F64_TOL) * s


# ---- data ----------------------------------------------------------------------------------------------------------
def base_losses(n):
    """The collapse regime (mostly large losses, eps -> 1), as in test_fixed_point_stop_decision_across_regimes."""
    return 0.5 * np.random.default_rng(n).chisquare(4, size=n) + 2.0


def place(losses, value, where):
    out = losses.copy()
    n = out.size
    if where == "first":
        out[0] = value
    elif where == "last":
        out[n - 1] = value
    elif where == "middle":
        out[n // 2] = value
    else:                                                   # a 1 % sprinkle
        out[np.random.default_rng(n + 1).choice(n, size=n // 100, replace=False)] = value
    return out


def online_edge(n, where, tol):
    """A loss whose e puts ONLINE's (1 + rho' e)(1 + rho e) at ~2^1023 in the last pass: pi' ~ 1 for such a sample
    whatever its exact loss, so rho' and rho are read off a run with a large negative loss at the same places."""
    ref = ref_loop(place(base_losses(n), -300.0, where), ONLINE, tol)
    r_old, r_new = ref["passes"][-2][1], ref["passes"][-1][1]
    return -(511.5 * LN2 - 0.5 * np.log(r_old * r_new))


@functools.lru_cache(maxsize=2)
def case(variant, n, value, where, tol, scale):
    """(losses as passed to the kernel, reference).  value None: the base data alone; "edge": online_edge.  With a
    scale s the kernel gets l / s and forms s (l / s) as the reference does."""
    if value is None:
        losses = base_losses(n)
    else:
        losses = place(base_losses(n), online_edge(n, where, tol) if value == "edge" else value, where)
    if scale is not None:
        losses = losses / scale
    return losses, ref_loop(losses * scale if scale is not None else losses, variant, tol)


ROUTES = ["default", "slots-1", "slots0", "slots8", "series0", "unaligned", "ework", "scale"]
SCALE = 0.37


def run_route(dev, monkeypatch, variant, n, value, where, tol, route, pi0=None):
    from rlvi_b200 import ops
    scale = SCALE if route == "scale" else None
    losses, ref = case(variant, n, value, where, tol, scale)
    if route.startswith("slots"):
        monkeypatch.setenv("RLVI_FP_CACHE_SLOTS", route[5:])
    if route == "series0":
        monkeypatch.setenv("RLVI_FP_SERIES", "0")
    kw = {"variant": variant, "tol": tol}
    if route == "unaligned":
        buf = cu(np.concatenate([[0.0], losses]), dev)
        pi, res = ops.fixed_point(buf[1:], **kw)            # 8-byte aligned only: the scalar IEEE path
    elif route == "ework":
        pi, res = ops.fixed_point(None, e_work=cu(np.exp(-losses), dev), **kw)
    elif route == "scale":
        pi, res = ops.fixed_point(cu(losses, dev), scale=torch.tensor([SCALE], dtype=torch.float64, device=dev), **kw)
    else:
        pi, res = ops.fixed_point(cu(losses, dev), **kw)
    check(pi, res, ref, tol, variant)
    return ref


# ---- 1. STANDARD at rcp_fast's range edges ---------------------------------------------------------------------------
WINDOW_VALUES = [-354.5, -354.21, -354.88, -709.0, -708.5, -709.7]
EDGE_VALUES = WINDOW_VALUES + [720.0, 800.0]
PLACES = ["first", "last", "middle", "sprinkle"]
BIG = (1 << 22) + 3                                         # above 2^22: the bulk-copy ring by default


def _standard_cases():
    out = []
    for n in (28673, 300001, BIG):
        for value in EDGE_VALUES:
            for where in (PLACES if n < BIG else ["sprinkle"]):
                for tol in ((1e-3, 1e-6) if n < BIG else (1e-6,)):
                    for route in ROUTES:
                        out.append(pytest.param(n, value, where, tol, route, id=f"n{n}-l{value:g}-{where}-tol{tol:g}-{route}"))
    return out


@pytest.mark.parametrize("n,value,where,tol,route", _standard_cases())
def test_standard_range_edges(dev, monkeypatch, n, value, where, tol, route):
    ref = run_route(dev, monkeypatch, STANDARD, n, value, where, tol, route)
    if value in WINDOW_VALUES:                  # the case really reaches the flush window of the fast reciprocal
        assert sum(flush_hits(ref, np.exp(-value), STANDARD)) > 0


# ---- 2. ONLINE on the persistent kernel -------------------------------------------------------------------------------
def _online_cases():
    out = []
    for n in (28673, 70001, 606209, BIG):
        routes = ROUTES if n < BIG else ["slots-1"]
        for value in (None, "edge"):
            for where in ((PLACES if n < BIG else ["first", "sprinkle"]) if value else ["-"]):
                for tol in ((1e-3, 1e-6) if n < BIG else (1e-6,)):
                    for route in routes:
                        out.append(pytest.param(n, value, where, tol, route, id=f"n{n}-{value or 'plain'}-{where}-tol{tol:g}-{route}"))
    return out


@pytest.mark.parametrize("n,value,where,tol,route", _online_cases())
def test_online_persistent(dev, monkeypatch, n, value, where, tol, route):
    ref = run_route(dev, monkeypatch, ONLINE, n, value, where, tol, route)
    if value is None and route == "default":    # the reference function itself, not only the restated loop
        assert relmax(ref["pi"], rlvi_np.update_weights_online(base_losses(n), tol=tol)) == 0.0
    if value == "edge" and route != "scale":
        losses, _ = case(ONLINE, n, value, where, tol, None)
        assert flush_hits(ref, np.exp(-losses.min()), ONLINE)[0] > 0


# ---- 3. warm start ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [STANDARD, ONLINE], ids=["standard", "online"])
@pytest.mark.parametrize("n", [70001, 300001])
@pytest.mark.parametrize("pi0", [0.3, 0.7, 0.999])
@pytest.mark.parametrize("slots", [None, "-1"], ids=["default", "ring"])
def test_warm_start(dev, monkeypatch, variant, n, pi0, slots):
    """rlvi_fixed_point_init_f64: the loop started from the constant pi0 instead of 0.95 / 0.5
    (test_online_carry_over_extension's reference, generalised to both variants and the persistent kernel)."""
    from rlvi_b200 import ops
    if slots is not None:
        monkeypatch.setenv("RLVI_FP_CACHE_SLOTS", slots)
    rng = np.random.default_rng(n + int(1000 * pi0))
    losses = np.where(rng.random(n) < 0.3, 6.0 + rng.normal(size=n), -1.0 + 0.3 * rng.normal(size=n))   # bimodal
    tol = 1e-6
    ref = ref_loop(losses, variant, tol, pi0=pi0)
    pi, res = ops.fixed_point(cu(losses, dev), variant=variant, tol=tol, pi0=pi0)
    check(pi, res, ref, tol, variant)


# ---- 4. FP32 deep variant on one GPU ------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [57345, 60000, 300001, (1 << 22) + 1])
@pytest.mark.parametrize("offset", [0, 1], ids=["vec", "scalar"])
def test_deep_persistent(dev, n, offset):
    """fp_kernel_deep_f32 against deep_ref.update_sample_weights (train_rlvi.py:14-38); offset 1 makes residuals,
    weights and e_work 4-byte aligned views, which takes the scalar path."""
    from rlvi_b200 import ops
    rng = np.random.default_rng(n)
    r = (0.5 * rng.chisquare(2, size=n) + rng.normal(size=n)).astype(np.float32)
    w = (0.5 + 0.5 * rng.random(n)).astype(np.float32)                # incoming weights of an earlier epoch
    r_ref, w_ref = torch.from_numpy(r.copy()), torch.from_numpy(w.copy())
    k = deep_ref.update_sample_weights(r_ref, w_ref)

    def view(a):
        buf = torch.zeros(n + offset, dtype=torch.float32, device=dev)
        if a is not None:
            buf[offset:] = torch.from_numpy(a).to(dev)
        return buf[offset:]

    rd, wd, ed = view(r), view(w), view(None)
    res = ops.fixed_point_deep(rd, wd, e_work=ed)
    out = ops.read_result(res)
    assert out["iters"] == k
    assert relmax(rd.cpu().numpy(), r_ref.numpy()) < F32_TOL
    assert np.max(np.abs(wd.cpu().numpy() - w_ref.numpy())) < F32_TOL
