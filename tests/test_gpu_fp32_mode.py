"""FP32-stored-X mode (SURVEY.md section 8d, BASELINE.json config 3): rlvi_weighted_moments_f32 (tcgen05 TF32 Gram)
and rlvi_loss_f32 against the NumPy oracle evaluated in FP64 on the SAME float32 samples.  Tolerance: north_star's
1e-5 for FP32 quantities (3xTF32 is ~1e-6; single-pass TF32 is bounded at its own, looser, level)."""
import os

import numpy as np
import pytest
import torch

from oracle import rlvi_np

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
TOL32 = 1e-5


def rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def gpu_moments(X32, w, y=None, power=1, precision=0, want_gram=True):
    from rlvi_b200 import ops
    dev = torch.device("cuda", 0)
    out = ops.weighted_moments(torch.from_numpy(X32).to(dev), torch.from_numpy(w).to(dev),
                               y=None if y is None else torch.from_numpy(y).to(dev), power=power, precision=precision,
                               want_gram=want_gram)
    return {k: v.cpu().numpy() for k, v in ops.split_moments(out, X32.shape[1]).items()}


def oracle_moments(X32, w, y, power):
    we = w * w if power == 2 else w
    r = rlvi_np.weighted_moments(X32.astype(np.float64), we, y)
    r["S1"] = X32.astype(np.float64).T @ w          # first power even when power == 2 (header contract)
    return r


@pytest.mark.parametrize("n,d,power,with_y", [(768, 64, 2, False), (4096, 128, 2, False), (5000, 256, 1, True),
                                              (20000, 512, 2, False), (777, 100, 1, True), (33, 512, 2, False),
                                              (1, 64, 1, False), (17, 4, 1, True), (100000, 384, 1, False),
                                              (3000, 132, 2, True),
                                              # CTA-pair kernel edges: partial third / fourth feature block, 2-D boxes
                                              # (d % 32 != 0), fewer tiles than pairs, y with both powers
                                              (2049, 260, 1, True), (999, 500, 2, True), (70000, 448, 1, True),
                                              (40, 256, 2, True)])
def test_moments_f32_tf32x3_matches_oracle(n, d, power, with_y):
    rng = np.random.default_rng(n + d)
    X = rng.normal(size=(n, d)).astype(np.float32)
    X[:, 0] += 3.0
    w = rng.random(n) ** 4
    y = rng.normal(size=n) if with_y else None
    m = gpu_moments(X, w, y, power)
    r = oracle_moments(X, w, y, power)
    assert rel(m["G"], r["G"]) < TOL32
    assert rel(m["S1"], r["S1"]) < TOL32
    assert abs(m["S0"] - r["S0"]) < 1e-9 * r["S0"]
    assert np.array_equal(m["G"], m["G"].T)                      # exact symmetry
    if with_y:
        assert rel(m["Sy"], r["Sy"]) < TOL32
        assert abs(m["Swy"] - r["Swy"]) < 1e-9 * abs(r["Swy"]) + 1e-12


@pytest.mark.parametrize("scale", [1e-7, 1e-20, 1e-150, 1e40])
def test_moments_f32_collapse_regime_weights(scale):
    """SURVEY.md H1: the posteriors of a converged fixed point are ~1e-7 and smaller; pi^2 x^2 would leave the FP32 range.
    The kernel normalises the weights by a power of two and scales the statistics back: same accuracy at any scale."""
    rng = np.random.default_rng(21)
    n, d = 30000, 256
    X = rng.normal(size=(n, d)).astype(np.float32)
    w = scale * rng.random(n) ** 3
    y = rng.normal(size=n)
    for power in (1, 2):
        m = gpu_moments(X, w, y, power)
        r = oracle_moments(X, w, y, power)
        assert rel(m["G"], r["G"]) < TOL32 and rel(m["S1"], r["S1"]) < TOL32 and rel(m["Sy"], r["Sy"]) < TOL32
        assert abs(m["S0"] - r["S0"]) < 1e-9 * r["S0"]


def test_moments_f32_fallback_shapes():
    """d % 4 != 0, d > 512 and an unaligned X take the FP64 route: FP64-level agreement."""
    rng = np.random.default_rng(5)
    for n, d in ((500, 10), (2000, 130), (300, 600)):
        X = rng.normal(size=(n, d)).astype(np.float32)
        w = rng.random(n)
        m = gpu_moments(X, w, None, 1)
        r = oracle_moments(X, w, None, 1)
        assert rel(m["G"], r["G"]) < 1e-12 and rel(m["S1"], r["S1"]) < 1e-12
    from rlvi_b200 import ops
    dev = torch.device("cuda", 0)
    X = rng.normal(size=(1001, 64)).astype(np.float32)
    base = torch.from_numpy(np.concatenate([np.zeros(1, np.float32), X.reshape(-1)])).to(dev)
    Xu = base[1:].view(1001, 64)                                 # 4-byte aligned only
    w = rng.random(1001)
    out = ops.weighted_moments(Xu, torch.from_numpy(w).to(dev))
    G = ops.split_moments(out, 64)["G"].cpu().numpy()
    assert rel(G, oracle_moments(X, w, None, 1)["G"]) < 1e-12


def test_moments_f32_single_pass_tf32_is_bounded():
    for d in (256, 128):                          # CTA pairs / the single-CTA kernel
        rng = np.random.default_rng(9)
        X = rng.normal(size=(50000, d)).astype(np.float32)
        w = rng.random(50000)
        m1 = gpu_moments(X, w, None, 2, precision=1)
        r = oracle_moments(X, w, None, 2)
        assert rel(m1["G"], r["G"]) < 2e-4, d     # 2^-11 operand rounding, zero-mean: ~1e-3 / sqrt(rows)


@pytest.mark.parametrize("n,d,power,with_y", [(30000, 512, 2, False), (9000, 256, 1, True), (5000, 388, 2, True)])
def test_moments_f32_correction_modes_agree(n, d, power, with_y, monkeypatch):
    """The ~1e-6 mode of the CTA-pair kernel runs its two correction products (lo.hi + hi.lo) as BF16 by default and as
    TF32 with RLVI_TF32_PURE3=1: both meet the oracle at the FP32 tolerance, and they agree with each other far below it
    (the BF16 rounding of the corrections is a 2^-19 relative, zero-mean perturbation of each product)."""
    rng = np.random.default_rng(n)
    X = rng.normal(size=(n, d)).astype(np.float32)
    X[:, :3] += 2.0
    w = rng.random(n) ** 3
    y = rng.normal(size=n) if with_y else None
    r = oracle_moments(X, w, y, power)
    monkeypatch.delenv("RLVI_TF32_PURE3", raising=False)
    mixed = gpu_moments(X, w, y, power)
    monkeypatch.setenv("RLVI_TF32_PURE3", "1")
    pure = gpu_moments(X, w, y, power)
    for m in (mixed, pure):
        assert rel(m["G"], r["G"]) < TOL32
        assert rel(m["S1"], r["S1"]) < TOL32
        if with_y:
            assert rel(m["Sy"], r["Sy"]) < TOL32
    assert rel(mixed["G"], pure["G"]) < 3e-6
    # column sums do not go through the tensor core; the two modes split the row tiles over the pair types differently,
    # so their FP32 partial sums group differently
    assert rel(mixed["S1"], pure["S1"]) < 1e-6


def test_moments_f32_deterministic_and_linear():
    for d in (512, 128):                                         # CTA pairs / the single-CTA kernel
        rng = np.random.default_rng(11)
        X = rng.normal(size=(70001, d)).astype(np.float32)
        w = rng.random(70001)
        a = gpu_moments(X, w, None, 1)
        b = gpu_moments(X, w, None, 1)
        assert np.array_equal(a["G"], b["G"]) and np.array_equal(a["S1"], b["S1"]), d
        c = gpu_moments(X, 4.0 * w, None, 1)                     # exact power-of-two scaling of every product
        assert rel(c["G"], 4.0 * a["G"]) < 1e-6, d


def test_moments_f32_large_n_d512_against_oracle():
    """N = 2^20, d = 512 (a sixteenth of config 3): the oracle finishes in seconds."""
    n, d = 1 << 20, 512
    rng = np.random.default_rng(3)
    X = rng.standard_normal(size=(n, d), dtype=np.float32)
    w = rng.random(n) ** 2
    m = gpu_moments(X, w, None, 2)
    X64 = X.astype(np.float64)
    Gr = (X64 * (w * w)[:, None]).T @ X64
    assert rel(m["G"], Gr) < TOL32
    assert rel(m["S1"], X64.T @ w) < TOL32


@pytest.mark.parametrize("kind_name", ["LOGISTIC_CE", "SOFTPLUS", "SQRES", "SQDIST", "PCA"])
@pytest.mark.parametrize("n,d", [(1000, 64), (333, 512), (50, 7), (4097, 200)])
def test_loss_f32_matches_oracle(kind_name, n, d):
    from rlvi_b200 import ops
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(d)
    X = rng.normal(size=(n, d)).astype(np.float32)
    X64 = X.astype(np.float64)
    th = rng.normal(size=d) / np.sqrt(d)
    y = (rng.random(n) < 0.5).astype(np.float64)
    w = rng.random(n)
    kind = getattr(ops, "LOSS_" + kind_name)
    icpt = kind_name in ("LOGISTIC_CE", "SOFTPLUS")
    params = np.concatenate([[0.3], th]) if icpt else th
    if kind_name == "LOGISTIC_CE":
        ref = rlvi_np.cross_entropy(np.hstack([np.ones((n, 1)), X64]), params, y)
    elif kind_name == "SOFTPLUS":
        ref = rlvi_np.softplus_loss(X64, params)
    elif kind_name == "SQRES":
        ref = (y - X64 @ th) ** 2
    elif kind_name == "SQDIST":
        ref = np.linalg.norm(th - X64, axis=1) ** 2
    else:
        th = th / np.linalg.norm(th)
        params = th
        ref = rlvi_np.pca_losses(X64, th)
    l, e, ws = ops.loss(kind, torch.from_numpy(X).to(dev), torch.from_numpy(params).to(dev),
                        y=torch.from_numpy(y).to(dev), intercept=icpt, weights=torch.from_numpy(w).to(dev), want_e=True)
    assert rel(l.cpu().numpy(), ref) < 1e-12
    assert rel(e.cpu().numpy(), np.exp(-ref)) < 1e-11
    ws = ws.cpu().numpy()
    assert abs(ws[0] - w @ ref) < 1e-11 * abs(w @ ref) and abs(ws[1] - w.sum()) < 1e-12 * w.sum()


def test_utils_pca_f32_against_golden_problem():
    """utils.pca on the float32 cast of the golden problem pca_n768_d64: theta and losses against the oracle run in
    FP64 on the same float32 samples (1e-5), and against the FP64 golden itself (storage rounding only)."""
    from rlvi_b200 import utils
    g = np.load(os.path.join(GOLD, "pca_n768_d64.npz"))
    X32 = g["X"].astype(np.float32)
    th, losses = utils.pca(X32, g["w"].copy())
    th_ref, l_ref = rlvi_np.pca_mstep(X32.astype(np.float64), g["w"])
    assert rel(th, th_ref) < TOL32
    assert rel(losses, l_ref) < TOL32
    assert rel(th, g["theta_mstep"]) < 1e-4      # float32 storage of X vs the FP64 golden


def test_rlvi_pca_f32_end_to_end():
    from rlvi_b200 import rlvi
    g = np.load(os.path.join(GOLD, "pca_n768_d64.npz"))
    X32 = g["X"].astype(np.float32)
    th = rlvi.pca(X32, theta_init=g["theta_init"])
    th_ref = rlvi_np.pca(X32.astype(np.float64), theta_init=g["theta_init"])
    assert rel(th, th_ref) < 1e-4                # maxiter-bounded loop: eigenvector sensitivity x 1e-6 statistics
