"""NumPy restatement of the series passes of the STANDARD fixed point (fixed_point.cu, DESIGN.md section 4).

Once rho dominates max e, the two sums a pass needs follow from the power sums P_j = sum z^j of z = e / 2^E, where 2^E
is the smallest power of two >= max e.  The kernel builds them once, in a sum-only streamed pass predicted to lie
within two passes of the switch, and evaluates every pass that `admits` from them.  This module mirrors the rule, the
series evaluation and the pass schedule, for tests and for tools/fp_series_time.py."""
from __future__ import annotations

import math

import numpy as np

J = 17                     # power sums (kFpSeriesJ)
TRUNC = 2.0 ** -60         # a-priori relative truncation bound the rule requires of both series
NEAR_TOL = 2.0 ** -40      # a series err this close to tol (relative) is re-taken from the streamed sums


def bounds(q, j=J):
    """Relative truncation bounds of (sum pi', sum t^2) after j power sums, at q = 2^E / min(rho', rho); inf when the
    tail estimate does not apply."""
    r = q * (j + 3) / j
    if not (q > 0.0 and r < 1.0):
        return math.inf, math.inf
    qm = q ** (j - 1)
    b1 = qm * q * (1.0 + q) / (1.0 - q)
    b2 = (1.0 + q) ** 4 * (j + 2) * (j + 1) * j / 6.0 * qm / (1.0 - r)
    return b1, b2


def admits(q, j=J):
    b1, b2 = bounds(q, j)
    return b1 <= TRUNC and b2 <= TRUNC


def scale(emax):
    """2^E: the smallest power of two >= emax (None outside the range the kernel accepts)."""
    if not (2.0 ** -1000 < emax < 2.0 ** 1000):
        return None
    m, ex = math.frexp(emax)
    return emax if m == 0.5 else math.ldexp(1.0, ex)


def power_sums(e, two_e, j=J):
    z = np.asarray(e, dtype=np.float64) / two_e
    out, p = np.empty(j), z.copy()
    for i in range(j):
        out[i] = math.fsum(p)
        p *= z
    return out


def series_sums(P, two_e, rho_new, rho_old):
    """(sum pi', sum (pi' - pi)^2) from the power sums, in the kernel's operation order."""
    j = len(P)
    a, b = two_e / rho_new, two_e / rho_old
    h = P[j - 1]
    for i in range(j - 2, -1, -1):
        h = -a * h + P[i]
    s1 = a * h
    ab = a * b
    d1, d2, d3, d4 = 2.0 * (a + b), a * a + (b * b + 4.0 * ab), 2.0 * ab * (a + b), ab * ab
    g0, g1, g2, g3, acc = 1.0, 0.0, 0.0, 0.0, P[1]
    for m in range(1, j - 1):      # g_m = (-1)^m c_m from the recurrence of 1 / ((1 + a x)^2 (1 + b x)^2)
        g = -(d1 * g0 + (d2 * g1 + (d3 * g2 + d4 * g3)))
        g0, g1, g2, g3 = g, g0, g1, g2
        acc = g * P[m + 1] + acc
    w = a * b / two_e
    drho = rho_old - rho_new
    return s1, (drho * drho) * ((w * w) * acc)


def direct_sums(e, rho_new, rho_old):
    """The streamed pass's two sums, accurately rounded (math.fsum)."""
    e = np.asarray(e, dtype=np.float64)
    t = e / ((rho_new + e) * (rho_old + e))
    return math.fsum(e / (rho_new + e)), (rho_old - rho_new) ** 2 * math.fsum(t * t)


def replay(e, tol=1e-3, maxiter=100, pi0=0.95, series=True, j=J):
    """The STANDARD recurrence with the kernel's schedule: per pass, whether it streamed or came from the series and
    whether it built the power sums.  Sums are the direct ones (the series agrees to rounding where admitted).
    Returns (passes, result) with passes a list of dicts k, q, mode ('stream', 'sum_only', 'build', 'series')."""
    e = np.asarray(e, dtype=np.float64)
    n = float(e.size)
    eps = 1.0 - pi0
    rho_new, rho_old = eps / (1.0 - eps), 0.0
    S, sqrt_n = n * pi0, math.sqrt(n)
    bound_prev = bound_prev2 = 0.0
    two_e, P, state = None, None, 0
    passes, k, converged, err = [], 1, 0, 0.0
    while True:
        if k == 1:
            pn = e / (rho_new + e)
            s1, s2, mode = math.fsum(pn), math.fsum((pn - pi0) ** 2), "stream"
            two_e = scale(float(e.max()))
            state = 0 if two_e is not None else -1
            q = math.inf
        else:
            q = two_e / min(rho_new, rho_old) if two_e else math.inf
            mode = None
            if state == 1 and admits(q, j):
                s1, s2 = series_sums(P, two_e, rho_new, rho_old)
                if not abs(math.sqrt(s2) - tol) <= NEAR_TOL * abs(tol):
                    mode = "series"
            if mode is None:
                sum_only = k < maxiter and bound_prev2 > 0.0 and bound_prev * min(1.0, bound_prev / bound_prev2) > 2 * tol
                r = rho_new / rho_old
                build = series and sum_only and state == 0 and admits(two_e / min(rho_new, rho_old) / (r * r), j)
                s1, s2 = direct_sums(e, rho_new, rho_old)
                mode = "build" if build else ("sum_only" if sum_only else "stream")
                if build:
                    P = power_sums(e, two_e, j)
                    state = 1 if np.all(np.isfinite(P)) and e.min() >= 0 else -1
                bound = abs(s1 - S) / sqrt_n
                if sum_only and not bound > tol * (1.0 + 1e-6):
                    mode += "+full"
                    sum_only = False
                if sum_only:
                    s2 = None
        bound = abs(s1 - S) / sqrt_n
        bound_prev2, bound_prev = bound_prev, bound
        S = s1
        passes.append({"k": k, "q": q, "mode": mode})
        if s2 is None:
            err = bound
        else:
            err = math.sqrt(s2)
            if err < tol:
                converged = 1
                break
        if k >= maxiter:
            break
        rho_old = rho_new
        avg = S / n
        eps = 1.0 - avg
        rho_new = eps / (1.0 - eps)
        k += 1
    return passes, {"eps": eps, "rho": rho_new, "sum_pi": S, "err": err, "iters": k, "converged": converged}


def streamed_passes(passes):
    """Passes that read e (the series passes do not); the final pi pass is not counted."""
    return sum(1 for p in passes if p["mode"] != "series")
