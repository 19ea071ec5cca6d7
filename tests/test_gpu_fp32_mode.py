"""FP32-stored-X mode (SURVEY.md section 8d, BASELINE.json config 3): rlvi_weighted_moments_f32 (tcgen05 TF32 Gram)
and rlvi_loss_f32 against the NumPy oracle evaluated in FP64 on the SAME float32 samples.  Tolerance: north_star's
1e-5 for FP32 quantities, entry by entry: |G - G_ref| <= 1e-5 |X|^T diag(w) |X| (tests/tf32_bounds.py); single-pass TF32 is
bounded at its own, looser, level.  The tests on `biased_inputs` make a missing correction product fail that check on
every entry, which zero-mean rounding on random samples hides."""
import os

import numpy as np
import pytest
import torch

import tf32_bounds as tb
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
    tb.check_moments(m, tb.reference(X, w, y, power), TOL32, with_y)      # includes exact symmetry


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
        tb.check_moments(gpu_moments(X, w, y, power), tb.reference(X, w, y, power), TOL32, True)


def test_moments_f32_fallback_shapes():
    """d % 4 != 0, d > 512 and an unaligned X take the FP64 route: FP64-level agreement."""
    rng = np.random.default_rng(5)
    for n, d in ((500, 10), (2000, 130), (300, 600)):
        X = rng.normal(size=(n, d)).astype(np.float32)
        w = rng.random(n)
        tb.check_moments(gpu_moments(X, w, None, 1), tb.reference(X, w, None, 1), tb.TAU_F64, False)
    from rlvi_b200 import ops
    dev = torch.device("cuda", 0)
    X = rng.normal(size=(1001, 64)).astype(np.float32)
    base = torch.from_numpy(np.concatenate([np.zeros(1, np.float32), X.reshape(-1)])).to(dev)
    Xu = base[1:].view(1001, 64)                                 # 4-byte aligned only
    w = rng.random(1001)
    out = ops.weighted_moments(Xu, torch.from_numpy(w).to(dev))
    tb.check_moments(ops.split_moments(out, 64), tb.reference(X, w, None, 1), tb.TAU_F64, False)


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
    r = tb.reference(X, w, y, power)
    monkeypatch.delenv("RLVI_TF32_PURE3", raising=False)
    mixed = gpu_moments(X, w, y, power)
    monkeypatch.setenv("RLVI_TF32_PURE3", "1")
    pure = gpu_moments(X, w, y, power)
    for m in (mixed, pure):
        tb.check_moments(m, r, TOL32, with_y)
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
    tb.check_moments(m, tb.reference(torch.from_numpy(X).cuda(), torch.from_numpy(w), None, 2), TOL32, False)


# ---- biased inputs (tests/tf32_bounds.py): every TF32 remainder of the same sign, so a missing product is a bias ----
SINGLE_CTA_D = (4, 36, 64, 100, 128)             # d % 32 != 0: four 2-D boxes; d % 32 == 0: one 3-D box
PAIR_D = (132, 256, 260, 384, 388, 448, 512)     # one pair type (d <= 256), three types; 257..384 run as 512
DEV = "cuda"


def dev_moments(X, w, y=None, power=1, precision=0, want_gram=True, out=None):
    from rlvi_b200 import ops
    o = ops.weighted_moments(X, w, y=y, power=power, precision=precision, want_gram=want_gram, out=out)
    return ops.split_moments(o, X.shape[1])


def report(what, q):
    print(f"[tf32] {what}: max |G - G_ref| / B = {q:.3g}")


@pytest.mark.parametrize("power,with_y", [(1, False), (1, True), (2, False), (2, True)])
@pytest.mark.parametrize("d", SINGLE_CTA_D + PAIR_D)
def test_moments_f32_biased_inputs_every_route(d, power, with_y, monkeypatch):
    """Both kernels, both powers, with and without y, BF16 and TF32 corrections (RLVI_TF32_PURE3=1, pair kernel only):
    entry-wise within 1e-5 B.  RLVI_TF32X1 on the same inputs -- the kernel without its corrections -- must miss by
    more than 1e-4 B on every diagonal entry, which shows the check sees a missing correction."""
    n = 3000 + 7 * d
    X, w = tb.biased_inputs(n, d, seed=d * 4 + power * 2 + with_y, device=DEV)
    y = torch.randn(n, dtype=torch.float64, device=DEV) if with_y else None
    r = tb.reference(X, w, y, power)
    modes = ("0", "1") if d > 128 else ("0",)
    for pure in modes:
        monkeypatch.setenv("RLVI_TF32_PURE3", pure)
        q = tb.check_moments(dev_moments(X, w, y, power), r, TOL32, with_y)
        report(f"d={d} p={power} y={with_y} {'pure TF32' if pure == '1' else 'default'} corrections", q)
    monkeypatch.delenv("RLVI_TF32_PURE3")
    G1 = dev_moments(X, w, y, power, precision=1)["G"].cpu().numpy()
    q1 = np.abs(G1 - r["G"]) / r["BG"]
    report(f"d={d} p={power} y={with_y} TF32X1", float(q1.max()))
    assert np.diag(q1).min() > 1e-4


@pytest.mark.parametrize("d", (64, 256, 512))
@pytest.mark.parametrize("n", (1, 15, 16, 17, 127, 128, 129))
def test_moments_f32_row_count_edges(n, d):
    """Partial and single tiles, fewer tiles than CTAs and fewer than the pairs of one pair type."""
    X, w = tb.biased_inputs(n, d, seed=n * 1000 + d, device=DEV)
    y = torch.randn(n, dtype=torch.float64, device=DEV)
    power = 1 + n % 2
    tb.check_moments(dev_moments(X, w, y, power), tb.reference(X, w, y, power), TOL32, True)


@pytest.mark.parametrize("d,power", [(128, 2), (256, 1), (512, 1)])
def test_moments_f32_register_flush_depth(d, power):
    """Every slot runs at least one full 32 Ki-row FP32 register accumulation (chunks_per_flush = 256 chunks of 128
    rows) on all-positive data: the worst case for one-signed FP32 rounding.  The single-CTA kernel has one slot per SM;
    the CTA-pair kernel has at most SMs / 2 pairs of one type, so these n reach a full flush in every slot whatever the
    plan picks."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    slots = sms if d <= 128 else sms // 2
    n = slots * 32768 + 16 * slots + 5
    X, w = tb.biased_inputs(n, d, seed=d, device=DEV)
    y = torch.randn(n, dtype=torch.float64, device=DEV)
    q = tb.check_moments(dev_moments(X, w, y, power), tb.reference(X, w, y, power), TOL32, True)
    report(f"flush depth n={n} d={d} p={power} ({torch.cuda.get_device_name(0)})", q)


@pytest.mark.parametrize("power", (1, 2))
@pytest.mark.parametrize("d", (64, 256, 512))
def test_moments_f32_weight_range(d, power):
    """Weights from 1 down to 1e-300 in one call, with exact zeros and subnormal doubles: the kernels normalise by a
    power of two and the rows whose scaled weight leaves the FP32 range contribute below the bound."""
    n = 6000
    X, _ = tb.biased_inputs(n, d, seed=7 + d, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(d + power)
    w = torch.pow(10.0, -300.0 * torch.rand(n, dtype=torch.float64, device=DEV, generator=g))
    w[::97] = 0.0
    w[1:4] = torch.tensor([5e-324, 1e-310, 2.2e-308], dtype=torch.float64)
    w[4] = 1.0
    y = torch.randn(n, dtype=torch.float64, device=DEV, generator=g)
    tb.check_moments(dev_moments(X, w, y, power), tb.reference(X, w, y, power), TOL32, True)


@pytest.mark.parametrize("power", (1, 2))
@pytest.mark.parametrize("d", (64, 256, 512))
def test_moments_f32_column_magnitudes(d, power):
    """Columns scaled from 2^-20 to 2^20 in one X: every entry meets its own bound."""
    X, w = tb.biased_inputs(5000, d, seed=11 + d, device=DEV, col_exp=np.linspace(-20, 20, d).round().astype(int))
    y = torch.randn(5000, dtype=torch.float64, device=DEV)
    tb.check_moments(dev_moments(X, w, y, power), tb.reference(X, w, y, power), TOL32, True)


# The supported range of the scaled samples z = s x (include/rlvi_b200.h, RLVI_TF32X3): 2^Z_LO <= |z| < 2^Z_HI.  Measured
# on a B200: still within the bound at 2^-66, 2.6e-5 B at 2^-68; non-finite at 2^61 (32 rows per CTA).
Z_LO, Z_HI = -60, 56


@pytest.mark.parametrize("end", ("low", "high"))
@pytest.mark.parametrize("power", (1, 2))
@pytest.mark.parametrize("d", (64, 256))
def test_moments_f32_supported_range_ends(d, power, end):
    """All samples at one end of the supported range of |s x|: unit weights give s = 1/2 (power 1) or 1/4 (power 2)
    after the kernels' normalisation, so x = 2^(E + 1) or 2^(E + 2) puts z in [2^E, 2^(E + 1))."""
    e = (Z_LO if end == "low" else Z_HI - 1) + power
    X, w = tb.biased_inputs(4096, d, seed=d + power, device=DEV, col_exp=[e] * d, max_k=0, zero_frac=0.0)
    q = tb.check_moments(dev_moments(X, w, None, power), tb.reference(X, w, None, power), TOL32, False)
    report(f"range end {end}: |z| in [2^{e - power}, 2^{e - power + 1}) d={d} p={power}", q)


@pytest.mark.parametrize("n,d", [(5000, 64), (5000, 256), (5000, 512), (1_700_000, 10)])
def test_moments_f32_want_gram_0_leaves_G_untouched(n, d):
    """want_gram = 0 on the three routes (single CTA, CTA pairs, FP64 conversion over three chunks): the G region of
    `out` comes back bit-identical, the vectors within their bounds."""
    X, w = tb.biased_inputs(n, d, seed=n + d, device=DEV)
    y = torch.randn(n, dtype=torch.float64, device=DEV)
    out = torch.randn(2 + 2 * d + d * d, dtype=torch.float64, device=DEV) * 1e300      # sentinel
    g0 = out[2 + 2 * d:].clone()
    m = dev_moments(X, w, y, 2, want_gram=False, out=out)
    assert torch.equal(out[2 + 2 * d:].view(torch.int64), g0.view(torch.int64))
    tau = tb.TAU_F64 if d % 4 else TOL32
    tb.check_moments(m, tb.reference(X, w, y, 2), tau, True, want_gram=False)


@pytest.mark.parametrize("power", (1, 2))
@pytest.mark.parametrize("n,d,aligned", [(2_100_000, 10, True), (40000, 516, True), (20561, 1020, True),
                                         (300_001, 64, False)])
def test_moments_f32_fp64_route_chunks(n, d, aligned, power):
    """The FP64 conversion route (d % 4 != 0, d > 512, unaligned X) over three chunks of 64 MiB / (8 d) rows: the
    chunk loop, its y / weights offsets and the accumulation of the chunk results, entry-wise at FP64 level."""
    g = torch.Generator(device=DEV).manual_seed(n + power)
    X = torch.randn((n, d), dtype=torch.float32, device=DEV, generator=g) + 0.5
    if not aligned:
        base = torch.zeros(n * d + 1, dtype=torch.float32, device=DEV)
        base[1:].copy_(X.view(-1))
        X = base[1:].view(n, d)                                       # 4-byte aligned only
    assert n > 2 * (64 << 20) // (8 * d)
    w = torch.rand(n, dtype=torch.float64, device=DEV, generator=g) ** 2
    y = torch.randn(n, dtype=torch.float64, device=DEV, generator=g)
    tb.check_moments(dev_moments(X, w, y, power), tb.reference(X, w, y, power), tb.TAU_F64, True)


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
