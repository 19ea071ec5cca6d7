"""rlvi_b200.batched.logistic_regression and rlvi_batched_logistic_f64 on the GPU: many independent logistic-regression
fits in one launch, with either M-step, against the reference's goldens, the NumPy oracle (MM) and the single-problem
drop-in rlvi.logistic_regression (both M-steps).

Bars: the MM fit to 1e-8 relative of the oracle (test_gpu_parity.py's bar for the drop-in's MM route), the Newton fit to
1e-9 relative of the drop-in."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import rlvi_np

pytestmark = pytest.mark.gpu

MM_TOL = 1e-8
NEWTON_TOL = 1e-9


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


def problem(n, d, seed, eps=0.2):
    from rlvi_b200 import synth
    X, y, _ = synth.logistic_data(n, d, corruption=eps, seed=seed)
    return X, y


def run_ops(probs, mstep, dev, **kw):
    """ops.batched_logistic on a list of (X, y): (theta, iters, status) as NumPy arrays."""
    from rlvi_b200 import ops
    off = np.concatenate([[0], np.cumsum([len(p[1]) for p in probs])])
    X = torch.from_numpy(np.concatenate([p[0] for p in probs])).to(dev)
    y = torch.from_numpy(np.concatenate([p[1] for p in probs])).to(dev)
    return [t.cpu().numpy() for t in ops.batched_logistic(X, y, off, mstep=mstep, **kw)]


def padded(g, rng, d, count=6):
    from rlvi_b200 import ops
    cap = ops.batched_logistic_max_rows(d)
    sizes = [int(s) for s in rng.integers(8 * (d + 1), cap + 1, size=count)]
    pads = [problem(n, d, seed=100 + k) for k, n in enumerate(sizes)]
    probs = pads[:3] + [(g["X"], g["y"])] + pads[3:]
    return [p[0] for p in probs], [p[1] for p in probs]


def test_goldens_as_batch_members(dev):
    from rlvi_b200 import batched, rlvi
    rng = np.random.default_rng(1)
    g = load_golden("logreg_mm_n1500_d8")
    X, y = padded(g, rng, 8)
    theta = batched.logistic_regression(X, y, mstep="mm")
    assert theta.shape == (7, 9)
    assert relmax(theta[3], g["theta"]) < MM_TOL
    g = load_golden("logreg_sklearn_n2000_d8")
    X, y = padded(g, rng, 8)
    theta = batched.logistic_regression(X, y)
    assert relmax(theta[3], rlvi.logistic_regression(g["X"], g["y"])) < NEWTON_TOL
    assert relmax(theta[3], g["theta"]) < 2e-2                             # test_round2_dropins.py's bar on liblinear
    cos = theta[3][1:] @ g["theta"][1:] / np.linalg.norm(theta[3][1:]) / np.linalg.norm(g["theta"][1:])
    assert cos > 1 - 1e-4


def _sweep(seed, count):
    """`count` ragged problems: d in 1..63, n in [8(d + 1), cap], corruption in [0.05, 0.4]; grouped by d."""
    from rlvi_b200 import ops
    rng = np.random.default_rng(seed)
    groups = {}
    for k in range(count):
        d = int(rng.integers(1, 64))
        n = int(rng.integers(8 * (d + 1), ops.batched_logistic_max_rows(d) + 1))
        groups.setdefault(d, []).append(problem(n, d, seed=1000 * seed + k, eps=float(rng.uniform(0.05, 0.4))))
    return groups


def test_mm_sweep_against_the_oracle(dev):
    from rlvi_b200 import batched, ops
    checked = 0
    for d, probs in sorted(_sweep(11, 300).items()):
        theta = batched.logistic_regression([p[0] for p in probs], [p[1] for p in probs], mstep="mm")
        _, _, status = run_ops(probs, ops.BATCHED_LOGREG_MM, dev)
        for b, (Xb, yb) in enumerate(probs):
            assert status[b] in (0, 1), (d, b, status[b])
            r = relmax(theta[b], rlvi_np.logistic_regression_mm(Xb, yb))
            assert r < MM_TOL, (d, b, len(yb), r)
            checked += 1
    assert checked == 300


def test_newton_sweep_against_the_dropin(dev):
    from rlvi_b200 import batched, ops, rlvi
    groups = _sweep(12, 200)
    g = load_golden("sklearn_sep_n800_d6")                                  # nearly separable
    groups.setdefault(6, []).append((g["X"], g["y"]))
    checked, beyond = 0, []
    for d, probs in sorted(groups.items()):
        theta = batched.logistic_regression([p[0] for p in probs], [p[1] for p in probs])
        _, iters, status = run_ops(probs, ops.BATCHED_LOGREG_NEWTON, dev)
        for b, (Xb, yb) in enumerate(probs):
            assert status[b] in (0, 1), (d, b, status[b])
            r = relmax(theta[b], rlvi.logistic_regression(Xb, yb))
            if r >= NEWTON_TOL:
                beyond.append((d, b, len(yb), int(iters[b]), r))
            checked += 1
    assert checked == 201
    assert beyond == []


def test_isolation_and_determinism(dev):
    """The kernel's outputs for one problem (theta, iters, status) do not depend on its place in the batch or the batch
    size.  Checked on ops.batched_logistic: a random batch may hold problems the drop-in itself cannot fit (see
    test_host_solve_route), which batched.logistic_regression would hand over and raise on."""
    from rlvi_b200 import ops
    d = 10
    probe = problem(157, d, seed=400)
    rng = np.random.default_rng(401)
    others = [problem(int(rng.integers(90, 400)), d, seed=402 + k) for k in range(1999)]
    for mstep in (ops.BATCHED_LOGREG_NEWTON, ops.BATCHED_LOGREG_MM):
        ref = [a[0] for a in run_ops([probe], mstep, dev)]
        assert all(np.array_equal(a[0], r) for a, r in zip(run_ops([probe], mstep, dev), ref))    # same batch twice
        for batch_size in (1, 37, 2000):
            for place in ("first", "last", "repeated"):
                rest = others[:batch_size - 1] if place != "repeated" else others[:max(0, batch_size - 3)]
                if place == "first":
                    probs, idx = [probe] + rest, [0]
                elif place == "last":
                    probs, idx = rest + [probe], [len(rest)]
                else:
                    probs = ([probe] + rest[:len(rest) // 2] + [probe] + rest[len(rest) // 2:]
                             + ([probe] if batch_size > 1 else []))
                    idx = [i for i, p in enumerate(probs) if p is probe]
                got = run_ops(probs, mstep, dev)
                for i in idx:
                    assert all(np.array_equal(a[i], r) for a, r in zip(got, ref)), (mstep, batch_size, place, i)
    # a NaN in one problem: status 2 there, no other problem's bits change
    probs = others[:36] + [probe]
    for mstep in (ops.BATCHED_LOGREG_NEWTON, ops.BATCHED_LOGREG_MM):
        base = run_ops(probs, mstep, dev)
        Xn = probs[10][0].copy()
        Xn[3, 4] = np.nan
        got = run_ops(probs[:10] + [(Xn, probs[10][1])] + probs[11:], mstep, dev)
        assert got[2][10] == 2 and np.isnan(got[0][10]).all()
        keep = [b for b in range(len(probs)) if b != 10]
        for a, b in zip(got, base):
            assert np.array_equal(a[keep], b[keep])


def _same_as_dropin_alone(probs, b, mstep, ref_batch_without_b):
    """batched.logistic_regression on `probs` returns at b exactly what the drop-in returns on problem b alone (NaN-aware)
    or raises what the drop-in raises, naming the problem; the other problems keep the bits of a batch without b."""
    from rlvi_b200 import batched, rlvi
    X, y = [p[0] for p in probs], [p[1] for p in probs]
    try:
        ref = rlvi.logistic_regression(probs[b][0], probs[b][1], mstep=mstep)
    except Exception as exc:                                               # noqa: BLE001 -- whatever the drop-in raises
        with pytest.raises(type(exc), match=f"problem {b}: "):
            batched.logistic_regression(X, y, mstep=mstep)
        return "raised"
    theta = batched.logistic_regression(X, y, mstep=mstep)
    assert np.array_equal(theta[b], ref, equal_nan=True)
    assert np.array_equal(np.delete(theta, b, axis=0), ref_batch_without_b)
    return "returned"


def test_host_solve_route(dev):
    """Status 2 hands a problem to rlvi.logistic_regression: MM's Q fails the pivot test on a duplicated column; the Newton
    solve stalls on a small problem whose posterior weights collapse (the drop-in's own Newton solve stalls there too)."""
    from rlvi_b200 import batched, ops
    d = 6
    good = [problem(120 + 13 * k, d, seed=500 + k) for k in range(6)]
    Xdup, ydup = problem(150, d, seed=510)
    Xdup[:, 1] = Xdup[:, 4]
    probs = good[:3] + [(Xdup, ydup)] + good[3:]
    _, _, status = run_ops(probs, ops.BATCHED_LOGREG_MM, dev)
    assert status[3] == 2 and (np.delete(status, 3) != 2).all()
    alone = batched.logistic_regression([p[0] for p in good], [p[1] for p in good], mstep="mm")
    _same_as_dropin_alone(probs, 3, "mm", alone)
    # n = 98, d = 10: the kernel's Newton solve does not converge in 60 steps at some EM iteration
    good = [problem(150 + 11 * k, 10, seed=520 + k) for k in range(4)]
    probs = good[:1] + [problem(98, 10, seed=1077)] + good[1:]
    _, _, status = run_ops(probs, ops.BATCHED_LOGREG_NEWTON, dev)
    assert (np.delete(status, 1) != 2).all()
    if status[1] == 2:
        alone = batched.logistic_regression([p[0] for p in good], [p[1] for p in good])
        _same_as_dropin_alone(probs, 1, "sklearn", alone)


def test_limits_against_the_single_problem_dropin(dev):
    from rlvi_b200 import batched, ops, rlvi
    assert ops.batched_logistic_max_rows(8) >= 2000 and ops.batched_logistic_max_rows(63) >= 1024
    assert ops.batched_logistic_max_rows(64) == 0 and ops.batched_logistic_max_rows(0) == 0
    for d in (1, 8, 63):
        for n in (8 * (d + 1), ops.batched_logistic_max_rows(d)):
            X, y = problem(n, d, seed=600 + d + n)
            for mstep, bar in (("sklearn", NEWTON_TOL), ("mm", MM_TOL)):
                r = relmax(batched.logistic_regression([X], [y], mstep=mstep)[0],
                           rlvi.logistic_regression(X, y, mstep=mstep))
                assert r < bar, (d, n, mstep, r)
    # maxiter = 0, 1, 2 stop on maxiter (status 1) on problems that take more than two EM iterations; 0 returns the
    # first fit
    for mstep, code, bar in (("sklearn", ops.BATCHED_LOGREG_NEWTON, NEWTON_TOL), ("mm", ops.BATCHED_LOGREG_MM, MM_TOL)):
        cand = [problem(300, 5, seed=610 + k, eps=0.4) for k in range(40)]
        _, iters, status = run_ops(cand, code, dev)
        probs = [p for p, i, s in zip(cand, iters, status) if s in (0, 1) and i > 2][:4]
        assert len(probs) == 4
        for maxiter in (0, 1, 2):
            th = batched.logistic_regression([p[0] for p in probs], [p[1] for p in probs], maxiter=maxiter, mstep=mstep)
            _, iters, status = run_ops(probs, code, dev, maxiter=maxiter)
            assert (status == 1).all() and (iters == maxiter).all()
            for b, (Xb, yb) in enumerate(probs):
                assert relmax(th[b], rlvi.logistic_regression(Xb, yb, maxiter=maxiter, mstep=mstep)) < bar
    # over the cap, d = 64: refused on the host, before any launch
    before = ops.launch_count(0)
    cap = ops.batched_logistic_max_rows(10)
    Xbig, ybig = problem(cap + 1, 10, seed=620)
    with pytest.raises(ValueError, match=f"at most {cap}.*rlvi.logistic_regression"):
        batched.logistic_regression([Xbig], [ybig])
    with pytest.raises(ValueError, match="at most"):
        ops.batched_logistic(torch.from_numpy(Xbig).to(dev), torch.from_numpy(ybig).to(dev), [0, cap + 1],
                             mstep=ops.BATCHED_LOGREG_MM)
    X64, y64 = problem(200, 64, seed=621)
    with pytest.raises(ValueError, match="rlvi.logistic_regression"):
        batched.logistic_regression([X64], [y64], mstep="mm")
    assert ops.launch_count(0) == before


def test_no_out_of_bounds_writes(dev):
    """Guard bands around every output of rlvi_batched_logistic_f64 (called through the C ABI with views into larger
    buffers) survive, also for rejected segments, which get status -1 and NaN theta."""
    from rlvi_b200 import _lib
    G, SENT = 64, -7.25e300
    d, lengths = 7, [40, 33, 90, 700]
    D = d + 1
    rows = sum(lengths)
    Xn, yn = problem(rows, d, seed=700)
    X = torch.from_numpy(Xn).to(dev)
    y = torch.from_numpy(yn).to(dev)
    stream = torch.cuda.current_stream(dev)
    ctx = _lib.context(0, stream.cuda_stream)

    def guarded(count, dtype=torch.float64, sent=SENT):
        buf = torch.full((count + 2 * G,), sent, dtype=dtype, device=dev)
        return buf, buf[G:G + count]

    def intact(buf, count, sent=SENT):
        return bool((buf[:G] == sent).all()) and bool((buf[G + count:] == sent).all())

    good = [0] + list(np.cumsum(lengths))
    bad = [0, 40, 40, 100, rows + 5]          # an empty and an overlong segment among good ones
    for offs in (good, bad):
        nprob = len(offs) - 1
        off = torch.tensor(offs, dtype=torch.int64, device=dev)
        for mstep in (0, 1):
            bt, th = guarded(nprob * D)
            bi, it = guarded(nprob, torch.int32, -77)
            bs, st = guarded(nprob, torch.int32, -77)
            rc = ctx.lib.rlvi_batched_logistic_f64(ctx.handle, mstep, C.c_void_p(X.data_ptr()), C.c_void_p(y.data_ptr()),
                                                   C.c_void_p(off.data_ptr()), nprob, rows, d, 1e-2, 100,
                                                   C.c_void_p(th.data_ptr()), C.c_void_p(it.data_ptr()),
                                                   C.c_void_p(st.data_ptr()), C.c_void_p(stream.cuda_stream))
            assert rc == 0
            torch.cuda.synchronize()
            assert intact(bt, nprob * D) and intact(bi, nprob, -77) and intact(bs, nprob, -77)
            s = st.cpu().numpy()
            if offs is bad:
                assert list(s[[1, 3]]) == [-1, -1] and np.isnan(th.view(nprob, D)[[1, 3]].cpu().numpy()).all()
                assert (s[[0, 2]] >= 0).all()
            else:
                assert (s >= 0).all()
    rc = ctx.lib.rlvi_batched_logistic_f64(ctx.handle, 0, C.c_void_p(X.data_ptr()), C.c_void_p(y.data_ptr()),
                                           C.c_void_p(off.data_ptr()), 1, rows, 64, 1e-2, 100, C.c_void_p(th.data_ptr()),
                                           C.c_void_p(it.data_ptr()), C.c_void_p(st.data_ptr()),
                                           C.c_void_p(stream.cuda_stream))
    assert rc != 0 and b"outside 1..63" in ctx.lib.rlvi_last_error()


def test_calling_conventions(dev):
    from rlvi_b200 import batched
    probs = [problem(250, 4, seed=800 + k) for k in range(5)]
    X, y = [p[0] for p in probs], [p[1] for p in probs]
    for mstep in ("sklearn", "mm"):
        ragged = batched.logistic_regression(X, y, mstep=mstep)
        assert isinstance(ragged, np.ndarray) and ragged.shape == (5, 5)
        stacked = batched.logistic_regression(np.stack(X), np.stack(y), mstep=mstep)
        assert isinstance(stacked, np.ndarray) and np.array_equal(stacked, ragged)
        t = batched.logistic_regression(torch.from_numpy(np.stack(X)).to(dev), torch.from_numpy(np.stack(y)).to(dev),
                                        mstep=mstep)
        assert isinstance(t, torch.Tensor) and t.is_cuda and np.array_equal(t.cpu().numpy(), ragged)
        tl = batched.logistic_regression([torch.from_numpy(a).to(dev) for a in X],
                                         [torch.from_numpy(a).to(dev) for a in y], mstep=mstep)
        assert isinstance(tl, torch.Tensor) and np.array_equal(tl.cpu().numpy(), ragged)
