"""Entry-wise accuracy bounds, biased test inputs and a NumPy emulation for the TF32 weighted Gram
(rlvi_weighted_moments_f32) -- a helper of the test modules, not a test file.

Why entry-wise.  TF32 rounding errors are zero-mean on random data, so measured against max |G| they shrink like
1/sqrt(n) and a kernel that skips a correction product can pass `max|G - G_ref| / max|G_ref| < 1e-5`.  The check here
holds every entry to its own scale, |G - G_ref| <= tau B with B = |X|^T diag(w) |X|, and `biased_inputs` builds samples
whose TF32 remainders all have one sign, so the error of a missing product is a bias that does not average out.

References are FP64 on the same float32 samples: NumPy up to ~1e10 multiply-adds, torch float64 on the samples' device
beyond that.  Their own error, ~n 2^-53 B, is far below either tolerance.
"""
from __future__ import annotations

import math

import numpy as np
import torch

TAU_TF32X3 = 1e-5        # RLVI_TF32X3 (include/rlvi_b200.h)
TAU_F64 = 1e-12          # shapes converted to FP64 (d % 4 != 0, d > 512, unaligned X)
NUMPY_MAX_MACS = 1e10


def reference(X, w, y, power):
    """FP64 moments and their entry-wise scales on the float32 samples X (NumPy or torch on any device; w, y: float64).
    Returns numpy arrays: G, BG = |X|^T diag(w^p) |X|, S1 = X^T w, B1 = |X|^T w, Sy = X^T (w^p y),
    By = |X|^T |w^p y|, S0, Swy."""
    X, w, y = (torch.as_tensor(t) if t is not None else None for t in (X, w, y))
    n, d = X.shape
    if X.device.type != "cpu" and n * d * d > NUMPY_MAX_MACS:
        X64 = X.double()
        w64, y64 = w.to(X.device), None if y is None else y.to(X.device)
        dot = torch.matmul
        absx = X64 if bool((X >= 0).all()) else X64.abs()     # skip the copy for all-positive samples
        fin = lambda t: t.cpu().numpy()                    # noqa: E731
    else:
        X64 = X.cpu().numpy().astype(np.float64)
        w64, y64 = w.cpu().numpy(), None if y is None else y.cpu().numpy()
        dot = np.matmul
        absx = np.abs(X64)
        fin = np.asarray
    we = w64 * w64 if power == 2 else w64
    r = {"G": fin(dot(X64.T, X64 * we[:, None])), "S1": fin(dot(X64.T, w64)), "S0": float(we.sum())}
    r["G"] = 0.5 * (r["G"] + r["G"].T)                     # BLAS need not return an exactly symmetric product
    r["BG"] = r["G"] if absx is X64 else fin(dot(absx.T, absx * we[:, None]))
    r["B1"] = r["S1"] if absx is X64 else fin(dot(absx.T, w64))
    if y64 is None:
        r["Sy"] = r["By"] = np.zeros(d)
        r["Swy"] = 0.0
    else:
        wy = we * y64
        r["Sy"] = fin(dot(X64.T, wy))
        r["By"] = fin(dot(absx.T, wy.abs() if torch.is_tensor(wy) else np.abs(wy)))
        r["Swy"] = float(wy.sum())
    return r


def max_ratio(a, b, bound):
    """max |a - b| / bound over the entries (inf where bound == 0 and a != b)."""
    err = np.abs(np.asarray(a, dtype=np.float64) - b)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(err == 0, 0.0, err / bound)
    return float(np.max(q)) if q.size else 0.0


def check_moments(m, r, tau, with_y, want_gram=True):
    """Assert the kernel's moments `m` (split_moments, any device) against `reference` entry by entry; S0 and Swy at
    1e-9 relative.  Returns max |G - G_ref| / B (0 when the Gram was not asked for)."""
    m = {k: (v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in m.items()}
    assert np.all(np.isfinite(m["S1"])) and (not want_gram or np.all(np.isfinite(m["G"])))
    q1 = max_ratio(m["S1"], r["S1"], tau * r["B1"])
    assert q1 <= 1.0, f"S1: max err / (tau B) = {q1:.3g}"
    assert abs(float(m["S0"]) - r["S0"]) <= 1e-9 * r["S0"]
    if with_y:
        qy = max_ratio(m["Sy"], r["Sy"], tau * r["By"])
        assert qy <= 1.0, f"Sy: max err / (tau B) = {qy:.3g}"
        assert abs(float(m["Swy"]) - r["Swy"]) <= 1e-9 * abs(r["Swy"]) + 1e-12
    if not want_gram:
        return 0.0
    qg = max_ratio(m["G"], r["G"], r["BG"])
    assert qg <= tau, f"G: max |G - G_ref| / B = {qg:.3g} > {tau:g}"
    assert np.array_equal(m["G"], m["G"].T)
    return qg


def biased_inputs(n, d, *, seed, device="cpu", col_exp=(-3, 3), max_k=6, zero_frac=0.05):
    """Float32 samples whose TF32 remainders are all positive and large, with exactly representable row scales.

    Every x_ij > 0 is a TF32 value (random 10 mantissa bits; exponent col_exp[j], or uniform in the (lo, hi) range per
    column) plus r in [2048, 3686] in its 13 low bits: the remainder below the TF32 rounding is 0.25 .. 0.45 of a TF32
    ulp, always of one sign, so hi = tf32(x) rounds down on every element.  The weights are powers of four 4^-k,
    k <= max_k, with max exactly 1 (row 0) and a fraction `zero_frac` of zeros: the kernels normalise them by an even
    power of two, so s_i = pi_i or sqrt(pi_i) is exact and z = s x has the remainders of x for both powers.
    Returns X (float32) and w (float64) on `device`."""
    g = torch.Generator(device=device).manual_seed(seed)
    i32 = dict(dtype=torch.int32, device=device, generator=g)
    if isinstance(col_exp, tuple):
        e = torch.randint(col_exp[0], col_exp[1] + 1, (d,), **i32)
    else:
        e = torch.as_tensor(col_exp, dtype=torch.int32, device=device)
    bits = torch.randint(0, 1024, (n, d), **i32) << 13
    bits |= torch.randint(2048, 3687, (n, d), **i32)
    bits |= (e + 127) << 23
    X = bits.view(torch.float32)
    k = torch.randint(0, max_k + 1, (n,), device=device, generator=g).double()
    w = torch.pow(4.0, -k)
    w[torch.rand(n, device=device, generator=g) < zero_frac] = 0.0
    w[0] = 1.0
    return X, w


# ---- NumPy emulation of the tensor-core products (exact products and sums: accumulation error not included) ----------
def tf32_rn(z):
    """Round-to-nearest onto the TF32 grid on the bit pattern (tf32.cuh to_tf32)."""
    b = np.asarray(z, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def bf16_rn(z):
    """Round-to-nearest-even onto BF16 (cvt.rn.bf16x2.f32), returned as float32."""
    b = np.asarray(z, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)).view(np.float32)


def row_scale(w, power):
    """s_i of z_i = s_i x_i as the kernels form it: pi normalised by the even power of two 2^e >= max pi, then
    pi 2^-e (power 2) or sqrt(pi 2^-e) (power 1), rounded to float32."""
    m = float(np.max(w))
    e = 0
    if m > 0 and math.isfinite(m):
        e = math.frexp(m)[1]
        e += e & 1
    pis = w * 2.0 ** -e
    return (pis if power == 2 else np.sqrt(pis)).astype(np.float32)


def emulated_gram(Z, mode):
    """Z^T Z with the operand splits of one kernel mode, products and sums in FP64:
    'x1' hi.hi (RLVI_TF32X1); 'drop' hi.hi + lo.hi (one correction missing); 'x3' hi.hi + lo.hi + hi.lo with lo on the
    TF32 grid; 'bf16' hi.hi + bf16(lo).bf16(z) + bf16(z).bf16(lo) (the CTA-pair kernel's default corrections)."""
    Z = np.asarray(Z, dtype=np.float32)
    hi = tf32_rn(Z)
    lo = Z - hi                                            # exact in FP32
    h = hi.astype(np.float64)
    G = h.T @ h
    if mode == "x1":
        return G
    if mode == "bf16":
        l16, z16 = bf16_rn(lo).astype(np.float64), bf16_rn(Z).astype(np.float64)
        c = l16.T @ z16
        return G + c + c.T
    c = tf32_rn(lo).astype(np.float64).T @ h
    if mode == "drop":
        return G + c
    assert mode == "x3", mode
    return G + c + c.T
