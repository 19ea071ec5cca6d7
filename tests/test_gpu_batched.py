"""rlvi_b200.batched and the rlvi_batched_* kernels on the GPU: many independent update_weights / mean / linear_regression
problems in one launch, each against the reference's goldens, the NumPy oracle and the single-problem drop-in.

Tolerances as in test_gpu_parity.py: 1e-9 relative for theta, SURVEY.md H1's max(1e-9, 4 * 2^-53 / mean pi) for pi."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import rlvi_np

pytestmark = pytest.mark.gpu

F64_TOL = 1e-9


@pytest.fixture(scope="module")
def dev():
    from rlvi_b200 import _lib
    _lib.load()
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def relmax(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def pi_tol(ref_pi):
    return max(F64_TOL, 4 * 2.0 ** -53 / max(float(np.mean(ref_pi)), 1e-300))


def linreg_problem(n, d, seed, eps=0.2):
    from rlvi_b200 import synth
    return synth.linear_regression_data(n, d, eps=eps, seed=seed)


def mean_problem(n, d, seed, eps=0.2):
    from rlvi_b200 import synth
    return synth.mean_data(n, d, eps=eps, seed=seed)


def test_config1_in_one_call(dev):
    """BASELINE.json configs[0]: the 100 problems of standard-learning/main.py:308-357 as ONE batch; per-run theta against
    the reference's own estimates and BASELINE.md section 2a's fingerprint, as test_config1_monte_carlo_replay checks
    for the per-problem loop."""
    from rlvi_b200 import batched
    g = load_golden("config1_linreg_fixed_eps")
    theta = batched.linear_regression(g["X"], g["y"])
    assert isinstance(theta, np.ndarray) and theta.shape == (100, 10)
    err = []
    for th, ref in zip(theta, g["theta_rlvi"]):
        assert relmax(th, ref) < F64_TOL
        err.append(np.linalg.norm(1.0 - th) / np.sqrt(10.0))
    assert abs(np.mean(err) - 0.02654) < 5e-5 and abs(np.median(err) - 0.02625) < 5e-5
    # CUDA tensors in -> CUDA tensors out, the same bits
    t = batched.linear_regression(torch.from_numpy(g["X"]).to(dev), torch.from_numpy(g["y"]).to(dev))
    assert t.is_cuda and np.array_equal(t.cpu().numpy(), theta)


@pytest.mark.parametrize("name", ["linreg_n40_d10", "mean_n100_d2", "linreg_n768_d64", "mean_n768_d64"])
def test_goldens_as_batch_members(dev, name):
    from rlvi_b200 import batched, ops
    g = load_golden(name)
    d = g["X"].shape[1]
    cap = ops.batched_max_rows(d)
    rng = np.random.default_rng(sum(map(ord, name)))
    sizes = [int(s) for s in rng.integers(max(2, 2 * d), cap + 1, size=6)]
    if name.startswith("linreg"):
        pads = [linreg_problem(n, d, seed=100 + k) for k, n in enumerate(sizes)]
        Xs = [p[0] for p in pads[:3]] + [g["X"]] + [p[0] for p in pads[3:]]
        ys = [p[1] for p in pads[:3]] + [g["y"]] + [p[1] for p in pads[3:]]
        theta = batched.linear_regression(Xs, ys)
    else:
        pads = [mean_problem(n, d, seed=100 + k) for k, n in enumerate(sizes)]
        theta = batched.mean(pads[:3] + [g["X"]] + pads[3:])
    assert theta.shape == (7, d)
    assert relmax(theta[3], g["theta"]) < F64_TOL


def test_update_weights_goldens_as_segments(dev):
    from rlvi_b200 import batched, synth
    g40, g1000, gneg = (load_golden(n) for n in ("update_weights_n40", "update_weights_n1000", "update_weights_neg"))
    pads = [synth.losses_mixture(n, seed=n) for n in (7, 513, 1200)]
    segs = [pads[0], g40["losses"], pads[1], g1000["losses"], gneg["losses"], pads[2]]
    pis = batched.update_weights(segs)
    assert isinstance(pis, list) and [p.shape for p in pis] == [s.shape for s in segs]
    assert relmax(pis[1], g40["pi"]) < pi_tol(g40["pi"])
    assert relmax(pis[3], g1000["pi"]) < pi_tol(g1000["pi"])
    ref_neg = rlvi_np.update_weights(gneg["losses"])          # the golden itself was made with tol 1e-5, maxiter 7
    assert relmax(pis[4], ref_neg) < pi_tol(ref_neg)
    for p, s in zip(pis, segs):
        ref = rlvi_np.update_weights(s)
        assert relmax(p, ref) < pi_tol(ref)
    pis = batched.update_weights(segs, float(gneg["tol"]), int(gneg["maxiter"]))
    assert relmax(pis[4], gneg["pi"]) < pi_tol(gneg["pi"])
    # stacked in -> stacked out
    stacked = np.stack([g40["losses"], g40["losses"][::-1].copy()])
    out = batched.update_weights(stacked)
    assert out.shape == (2, 40) and relmax(out[0], g40["pi"]) < pi_tol(g40["pi"])


def _sweep(seed, count):
    """`count` ragged problems: d in 1..64, n in [max(2, 2d), cap], eps in [0, 0.4]; grouped by d."""
    from rlvi_b200 import ops
    rng = np.random.default_rng(seed)
    groups = {}
    for k in range(count):
        d = int(rng.integers(1, 65))
        n = int(rng.integers(max(2, 2 * d), ops.batched_max_rows(d) + 1))
        groups.setdefault(d, []).append((n, float(rng.uniform(0.0, 0.4)), 1000 * seed + k))
    return groups


def test_linear_regression_sweep_against_the_oracle(dev):
    from rlvi_b200 import batched, ops
    checked = beyond = 0
    for d, probs in sorted(_sweep(7, 400).items()):
        data = [linreg_problem(n, d, seed=s, eps=e) for n, e, s in probs]
        theta = batched.linear_regression([p[0] for p in data], [p[1] for p in data])
        X = torch.from_numpy(np.concatenate([p[0] for p in data])).to(dev)
        y = torch.from_numpy(np.concatenate([p[1] for p in data])).to(dev)
        off = np.concatenate([[0], np.cumsum([n for n, _, _ in probs])])
        _, iters, status = ops.batched_em(ops.BATCHED_LINREG, X, y, off)
        iters, status = iters.cpu().numpy(), status.cpu().numpy()
        for b, (Xb, yb) in enumerate(data):
            trace = []
            ref = rlvi_np.linear_regression(Xb, yb, trace=trace)
            cond = max([np.linalg.cond(Xb)] + [np.linalg.cond(np.sqrt(w)[:, None] * Xb) for _, w in trace])
            if cond > 1e3:
                # the weights collapsed onto too few rows: the normal equations (the drop-in's M-step, which the kernel
                # follows) keep 1e-9 only up to cond ~ 1e3 (DESIGN.md section 6); the drop-in differs from gelsd here too
                beyond += 1
                continue
            assert relmax(theta[b], ref) < F64_TOL, (d, b)
            if status[b] in (0, 1):
                assert iters[b] == len(trace), (d, b, iters[b], len(trace))
            checked += 1
    assert checked + beyond == 400 and beyond <= 4


def test_mean_sweep_against_the_oracle(dev):
    from rlvi_b200 import batched
    checked = 0
    for d, probs in sorted(_sweep(8, 400).items()):
        data = [mean_problem(n, d, seed=s, eps=e) for n, e, s in probs]
        theta = batched.mean(data)
        for b, Xb in enumerate(data):
            assert relmax(theta[b], rlvi_np.mean(Xb)) < F64_TOL, (d, b)
            checked += 1
    assert checked == 400


def test_update_weights_sweep_against_the_oracle(dev):
    from rlvi_b200 import batched, ops, synth
    rng = np.random.default_rng(9)
    cap = ops.batched_max_rows(1)
    segs = [synth.losses_mixture(int(rng.integers(2, cap + 1)), seed=k) * rng.uniform(0.2, 5.0) for k in range(400)]
    pis = batched.update_weights(segs)
    off = np.concatenate([[0], np.cumsum([len(s) for s in segs])])
    _, res = ops.batched_fixed_point(torch.from_numpy(np.concatenate(segs)).to(dev), off)
    res = ops.batched_results(res)
    for b, s in enumerate(segs):
        ref, eps, k, _ = rlvi_np.fixed_point_trace(s)
        assert relmax(pis[b], ref) < pi_tol(ref), b
        assert res["iters"][b] == k and abs(res["eps"][b] - eps) < F64_TOL, b


def test_host_solve_route(dev):
    """Rank-deficient designs are flagged (status 2) and re-solved by the drop-in; the other problems do not notice."""
    from rlvi_b200 import batched, ops, rlvi
    d = 10
    good = [linreg_problem(40 + 7 * k, d, seed=200 + k) for k in range(6)]
    Xdup, ydup = linreg_problem(60, d, seed=301)
    Xdup[:, 3] = Xdup[:, 7]
    Xfew, yfew = linreg_problem(6, d, seed=302)
    Xzero, yzero = linreg_problem(50, d, seed=303)
    Xzero[:, 5] = 0.0
    bad = [(Xdup, ydup), (Xfew, yfew), (Xzero, yzero)]
    probs = good[:2] + bad[:1] + good[2:4] + bad[1:] + good[4:]
    where_bad = [2, 5, 6]
    X = [p[0] for p in probs]
    y = [p[1] for p in probs]
    off = np.concatenate([[0], np.cumsum([len(v) for v in y])])
    _, _, status = ops.batched_em(ops.BATCHED_LINREG, torch.from_numpy(np.concatenate(X)).to(dev),
                                  torch.from_numpy(np.concatenate(y)).to(dev), off)
    status = status.cpu().numpy()
    assert [int(status[b]) for b in where_bad] == [2, 2, 2]
    theta = batched.linear_regression(X, y)
    for b, (Xb, yb) in zip(where_bad, bad):
        assert np.array_equal(theta[b], rlvi.linear_regression(Xb, yb)), b
    alone = batched.linear_regression([p[0] for p in good], [p[1] for p in good])
    keep = [b for b in range(len(probs)) if b not in where_bad]
    assert np.array_equal(theta[keep], alone)


def test_isolation_and_determinism(dev):
    from rlvi_b200 import batched, ops
    d = 10
    probe = linreg_problem(57, d, seed=400)
    rng = np.random.default_rng(401)
    others = [linreg_problem(int(rng.integers(20, 300)), d, seed=402 + k) for k in range(1999)]
    ref = batched.linear_regression([probe[0]], [probe[1]])[0]
    assert np.array_equal(batched.linear_regression([probe[0]], [probe[1]])[0], ref)        # same batch twice
    for batch_size in (1, 37, 2000):
        for place in ("first", "last", "repeated"):
            rest = others[:batch_size - 1] if place != "repeated" else others[:max(0, batch_size - 3)]
            if place == "first":
                probs, idx = [probe] + rest, [0]
            elif place == "last":
                probs, idx = rest + [probe], [len(rest)]
            else:
                probs = [probe] + rest[:len(rest) // 2] + [probe] + rest[len(rest) // 2:] + ([probe] if batch_size > 1 else [])
                idx = [i for i, p in enumerate(probs) if p is probe]
            th = batched.linear_regression([p[0] for p in probs], [p[1] for p in probs])
            for i in idx:
                assert np.array_equal(th[i], ref), (batch_size, place, i)
    # a NaN in one problem changes no other problem's bits (in the kernel: the NaN problem fails the pivot test and is
    # handed back with status 2; the drop-in then raises on it, as it does for that problem alone)
    probs = others[:36] + [probe]
    off = np.concatenate([[0], np.cumsum([len(p[1]) for p in probs])])
    y = torch.from_numpy(np.concatenate([p[1] for p in probs])).to(dev)
    X = np.concatenate([p[0] for p in probs])
    base = [t.cpu().numpy() for t in ops.batched_em(ops.BATCHED_LINREG, torch.from_numpy(X).to(dev), y, off)]
    X[off[10] + 3, 4] = np.nan
    got = [t.cpu().numpy() for t in ops.batched_em(ops.BATCHED_LINREG, torch.from_numpy(X).to(dev), y, off)]
    assert got[2][10] == 2 and np.isnan(got[0][10]).all()
    keep = [b for b in range(len(probs)) if b != 10]
    for g, b in zip(got, base):
        assert np.array_equal(g[keep], b[keep])
    # the mean model and the fixed point are just as position-independent
    m = [mean_problem(int(rng.integers(3, 400)), 5, seed=500 + k) for k in range(37)]
    assert np.array_equal(batched.mean(m)[20], batched.mean([m[20]])[0])
    segs = [rng.random(int(rng.integers(1, 500))) * 10 for _ in range(37)]
    assert np.array_equal(batched.update_weights(segs)[20], batched.update_weights([segs[20]])[0])


def test_limits_against_the_single_problem_dropins(dev):
    from rlvi_b200 import batched, ops, rlvi

    def same(a, b):
        a, b = np.asarray(a), np.asarray(b)
        assert np.array_equal(np.isnan(a), np.isnan(b))
        ok = ~np.isnan(b)
        if ok.any():
            assert relmax(a[ok], b[ok]) < F64_TOL

    cap10 = ops.batched_max_rows(10)
    assert ops.batched_max_rows(10) >= 200 and ops.batched_max_rows(64) >= 1024
    # n_b = 1: the mean's sigma2 is 0 and the drop-in returns NaN; the batched call must too
    one = mean_problem(1, 3, seed=600)
    th = batched.mean([one, mean_problem(50, 3, seed=601)])
    same(th[0], rlvi.mean(one))
    assert np.isnan(th[0]).all()
    # n_b = cap, d = 1, d = 64
    for n, d in ((cap10, 10), (ops.batched_max_rows(1), 1), (300, 1), (ops.batched_max_rows(64), 64), (130, 64)):
        X, y = linreg_problem(n, d, seed=602 + d)
        same(batched.linear_regression([X], [y])[0], rlvi.linear_regression(X, y))
        M = mean_problem(n, d, seed=603 + d)
        same(batched.mean([M])[0], rlvi.mean(M))
    lw = [np.array([0.3]), np.random.default_rng(604).random(ops.batched_max_rows(1)) * 4]
    for got, l in zip(batched.update_weights(lw), lw):
        same(got, rlvi.update_weights(l))
    # maxiter = 1, 2 stop on maxiter (status 1)
    g = load_golden("config1_linreg_fixed_eps")
    X, y = g["X"][:4], g["y"][:4]
    for maxiter in (1, 2):
        th = batched.linear_regression(X, y, maxiter=maxiter)
        _, iters, status = ops.batched_em(ops.BATCHED_LINREG, torch.from_numpy(X.reshape(-1, 10)).to(dev),
                                          torch.from_numpy(y.reshape(-1)).to(dev), np.arange(5) * 40, maxiter=maxiter)
        assert (status.cpu().numpy() == 1).all() and (iters.cpu().numpy() == maxiter).all()
        for b in range(4):
            same(th[b], rlvi.linear_regression(X[b], y[b], maxiter=maxiter))
        M = mean_problem(100, 2, seed=605)
        same(batched.mean([M], maxiter=maxiter)[0], rlvi.mean(M, maxiter=maxiter))
    # a segment over the cap is refused on the host, before any launch
    before = ops.launch_count(0)
    Xbig, ybig = linreg_problem(cap10 + 1, 10, seed=606)
    with pytest.raises(ValueError, match=f"at most {cap10}.*rlvi.linear_regression"):
        batched.linear_regression([Xbig], [ybig])
    with pytest.raises(ValueError, match="at most"):
        ops.batched_em(ops.BATCHED_LINREG, torch.from_numpy(Xbig).to(dev), torch.from_numpy(ybig).to(dev),
                       [0, cap10 + 1])
    assert ops.launch_count(0) == before


def test_no_out_of_bounds_writes(dev):
    """Guard bands around every output of the two entry points (called through the C ABI with views into larger buffers)
    survive, also for rejected segments."""
    from rlvi_b200 import _lib
    G, SENT = 64, -7.25e300
    d, lengths = 7, [1, 33, 40, 700]
    rows = sum(lengths)
    rng = np.random.default_rng(700)
    X = torch.from_numpy(rng.normal(size=(rows, d))).to(dev)
    y = torch.from_numpy(rng.normal(size=rows)).to(dev)
    stream = torch.cuda.current_stream(dev)
    ctx = _lib.context(0, stream.cuda_stream)

    def guarded(count, dtype=torch.float64, sent=SENT):
        buf = torch.full((count + 2 * G,), sent, dtype=dtype, device=dev)
        return buf, buf[G:G + count]

    def intact(buf, count, sent=SENT):
        return bool((buf[:G] == sent).all()) and bool((buf[G + count:] == sent).all())

    good = [0] + list(np.cumsum(lengths))
    bad = [0, 1, 1, 30, rows + 5]           # an empty and an overlong segment among good ones
    for offs in (good, bad):
        nprob = len(offs) - 1
        off = torch.tensor(offs, dtype=torch.int64, device=dev)
        bt, th = guarded(nprob * d)
        bi, it = guarded(nprob, torch.int32, -77)
        bs, st = guarded(nprob, torch.int32, -77)
        for model in (0, 1):
            rc = ctx.lib.rlvi_batched_em_f64(ctx.handle, model, C.c_void_p(X.data_ptr()),
                                             C.c_void_p(y.data_ptr()) if model else None, C.c_void_p(off.data_ptr()),
                                             nprob, rows, d, 1e-3, 100, C.c_void_p(th.data_ptr()),
                                             C.c_void_p(it.data_ptr()), C.c_void_p(st.data_ptr()),
                                             C.c_void_p(stream.cuda_stream))
            assert rc == 0
            torch.cuda.synchronize()
            assert intact(bt, nprob * d) and intact(bi, nprob, -77) and intact(bs, nprob, -77)
        bp, pi = guarded(rows)
        br, res = guarded(nprob * 5)
        rc = ctx.lib.rlvi_batched_fixed_point_f64(ctx.handle, C.c_void_p(y.data_ptr()), C.c_void_p(off.data_ptr()), nprob,
                                                  rows, 1e-3, 100, C.c_void_p(pi.data_ptr()), C.c_void_p(res.data_ptr()),
                                                  C.c_void_p(stream.cuda_stream))
        assert rc == 0
        torch.cuda.synchronize()
        assert intact(bp, rows) and intact(br, nprob * 5)
        if offs is bad:
            s = st.cpu().numpy()
            assert list(s[[1, 3]]) == [-1, -1] and np.isnan(th.view(nprob, d)[[1, 3]].cpu().numpy()).all()
            r = res.view(nprob, 5).cpu().numpy().view(np.uint8).reshape(nprob, 40)[:, 32:].view(np.int32)
            assert list(r[[1, 3], 0]) == [-1, -1]
