"""The biased inputs of tests/tf32_bounds.py make a missing TF32 correction product visible entry by entry: checked on
the CPU with the NumPy emulation of the kernels' operand splits (exact products and sums, so this is the error of the
products alone).  tests/test_gpu_fp32_mode.py relies on it: a kernel that runs single-pass TF32 or drops one correction
misses its entry-wise check on these inputs by an order of magnitude."""
import numpy as np
import pytest

import tf32_bounds as tb


@pytest.mark.parametrize("n,power", [(4000, 1), (4000, 2), (50000, 2)])
def test_biased_inputs_expose_missing_corrections(n, power):
    X, w = tb.biased_inputs(n, 64, seed=n + power)
    X, w = X.numpy(), w.numpy()
    assert X.dtype == np.float32 and np.all(X > 0) and w.max() == 1.0 and np.any(w == 0)
    s = tb.row_scale(w, power)
    assert np.array_equal(s.astype(np.float64), w / 4 if power == 2 else np.sqrt(w / 4))     # exact row scales
    Z = s[:, None] * X
    assert np.array_equal(Z.astype(np.float64), s.astype(np.float64)[:, None] * X)        # z = s x exact in FP32
    Z64 = Z.astype(np.float64)
    G = Z64.T @ Z64
    B = G                                                # all-positive samples: B = |Z|^T |Z| = G
    err = {m: np.abs(tb.emulated_gram(Z, m) - G) / B for m in ("x1", "drop", "x3", "bf16")}
    assert err["x1"].min() >= 1e-4, err["x1"].min()
    assert err["drop"].min() >= 5e-5, err["drop"].min()
    assert err["x3"].max() <= 1e-6, err["x3"].max()
    assert err["bf16"].max() <= 1e-6, err["bf16"].max()


def test_reference_bounds_and_check():
    """`reference` gives B = |X|^T diag(w) |X| (not |G|) on signed samples, and `check_moments` rejects an error of
    just over tau B in one entry."""
    rng = np.random.default_rng(0)
    import torch
    X = torch.from_numpy(rng.normal(size=(300, 8)).astype(np.float32))
    w = torch.from_numpy(rng.random(300))
    y = torch.from_numpy(rng.normal(size=300))
    r = tb.reference(X, w, y, 2)
    X64, we = X.numpy().astype(np.float64), w.numpy() ** 2
    assert np.allclose(r["BG"], np.abs(X64).T @ (np.abs(X64) * we[:, None]), rtol=1e-14)
    assert np.all(r["BG"] >= np.abs(r["G"])) and np.all(r["By"] >= np.abs(r["Sy"]))
    m = {"G": r["G"].copy(), "S1": r["S1"], "Sy": r["Sy"], "S0": r["S0"], "Swy": r["Swy"]}
    assert tb.check_moments(m, r, 1e-5, True) == 0.0
    m["G"][2, 5] += 1.01e-5 * r["BG"][2, 5]
    m["G"][5, 2] = m["G"][2, 5]
    with pytest.raises(AssertionError):
        tb.check_moments(m, r, 1e-5, True)
