"""Time the batched RLVI fits (rlvi_b200.batched) against the per-problem drop-in loop and the NumPy oracle on the
reference experiment driver's Monte-Carlo sweeps (standard-learning/main.py: test_linear_regression, N = 40, d = 10;
test_mean, N = 100, d = 2; 20 corruption rates linspace(0, 0.4, 20) x 100 runs = 2000 problems each), plus one larger point
(1184 linear-regression problems of N = 1024, d = 64: 8 problems per SM).  The logistic sweeps follow the driver's
test_logistic_regression_fixed_eps (standard-learning/main.py:422-472, N = 200; BASELINE.md section 2a): 20 corruption
rates linspace(0.05, 0.4, 20) x 100 runs of synth.logistic_data, at d = 10 (the driver's d is not recorded here), plus
1184 problems of N = 1024, d = 63, each with both M-steps (mstep "sklearn" = Newton, "mm").  Prints one JSON line.

For every sweep:
  batched_device_s   one batched call on device-resident CUDA tensors, host clock around call + synchronise, median of --reps
                     after one warm-up call
  batched_numpy_s    the same call with NumPy in and out (packing, one H2D copy, D2H of theta), median of --reps
  dropin_loop_s      rlvi_b200.rlvi.{linear_regression, mean} called once per problem with NumPy in and out (what a
                     config-1 driver does today), one pass after a warm-up problem
  oracle_s           oracle.rlvi_np (the NumPy restatement of the reference) per problem, one process on the host
  max_rel_theta_*    max over problems of max|theta - ref| / max|ref| against the oracle and against the drop-in;
                     problems_over_1e-9_vs_oracle counts the problems past 1e-9, and dropin_problems_over_1e-9_vs_oracle
                     the same count for the single-problem drop-in (weights collapsed onto too few rows, DESIGN.md section 6)
  host_solve         problems the kernel handed back to rlvi.linear_regression (status 2)
The large point runs the loop and the oracle on its first --large-subset problems only (problems_timed says how many).
The logistic sweeps (logreg_*) report the same keys, with the loop and the oracle on the first --logistic-subset
(--logistic-large-subset at d = 63) problems, the oracle for mstep "mm" only (it has no liblinear), and in addition
  batched_kernel_s   ops.batched_logistic alone on device tensors (one launch; status-2 problems are left NaN)
  host_solve         problems the kernel handed back to rlvi.logistic_regression (status 2)
  dropin_raised      timed problems on which the drop-in itself raises (Newton not converged); they are left out of the
                     parity figures, and batched_device_s / batched_numpy_s are null when the batch holds one (the
                     batched call raises what the drop-in raises; batched_error has the message)

    python tools/batched_time.py [--reps 20] [--large-subset 128] [--logistic-subset 200] [--logistic-large-subset 32]
                                 [--out r05_batched_logistic.json]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from rlvi_b200 import batched, ops, rlvi, synth  # noqa: E402

# The NumPy oracle is the host baseline and the parity reference of this measurement, as in bench.py's CPU leg; it is
# loaded by name because nothing outside tests/ and the two checkers imports it statically.
rlvi_np = importlib.import_module("oracle.rlvi_np")

EPS_GRID = np.linspace(0.0, 0.4, 20)
LOGISTIC_EPS_GRID = np.linspace(0.05, 0.4, 20)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else ("?", "?", "?")
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi_name": name, "power_limit": power, "max_sm_clock": clock}


def relmax(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def sweep_linreg(n, d, runs, seed0):
    data = [synth.linear_regression_data(n, d, eps=float(e), seed=seed0 + 1000 * i + r)
            for i, e in enumerate(EPS_GRID) for r in range(runs)]
    return np.stack([p[0] for p in data]), np.stack([p[1] for p in data])


def sweep_mean(n, d, runs, seed0):
    return np.stack([synth.mean_data(n, d, eps=float(e), seed=seed0 + 1000 * i + r)
                     for i, e in enumerate(EPS_GRID) for r in range(runs)])


def sweep_logistic(n, d, runs, seed0):
    data = [synth.logistic_data(n, d, corruption=float(e), seed=seed0 + 1000 * i + r)
            for i, e in enumerate(LOGISTIC_EPS_GRID) for r in range(runs)]
    return np.stack([p[0] for p in data]), np.stack([p[1] for p in data])


def median_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def measure(model, X, y, reps, subset=None):
    dev = torch.device("cuda", 0)
    B, n, d = X.shape
    Xd = torch.from_numpy(X).to(dev)
    yd = torch.from_numpy(y).to(dev) if y is not None else None
    if model == "linreg":
        dev_call = lambda: batched.linear_regression(Xd, yd)          # noqa: E731
        np_call = lambda: batched.linear_regression(X, y)             # noqa: E731
        single = lambda b: rlvi.linear_regression(X[b], y[b])         # noqa: E731
        oracle = lambda b: rlvi_np.linear_regression(X[b], y[b])      # noqa: E731
    else:
        dev_call = lambda: batched.mean(Xd)                           # noqa: E731
        np_call = lambda: batched.mean(X)                             # noqa: E731
        single = lambda b: rlvi.mean(X[b])                            # noqa: E731
        oracle = lambda b: rlvi_np.mean(X[b])                         # noqa: E731
    out = {"problems": B, "n": n, "d": d}
    out["batched_device_s"] = median_time(dev_call, reps)
    out["batched_numpy_s"] = median_time(np_call, reps)
    out["reps"] = reps
    theta = np_call()
    idx = range(B if subset is None else min(subset, B))
    single(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    th_single = [single(b) for b in idx]
    torch.cuda.synchronize()
    out["dropin_loop_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    th_oracle = [oracle(b) for b in idx]
    out["oracle_s"] = time.perf_counter() - t0
    out["problems_timed"] = len(th_single)
    k = len(th_single)
    vs_oracle = [relmax(theta[b], th_oracle[b]) for b in idx]
    vs_dropin = [relmax(theta[b], th_single[b]) for b in idx]
    out["max_rel_theta_vs_oracle"] = max(vs_oracle)
    out["max_rel_theta_vs_dropin"] = max(vs_dropin)
    out["problems_over_1e-9_vs_oracle"] = sum(r > 1e-9 for r in vs_oracle)
    out["dropin_problems_over_1e-9_vs_oracle"] = sum(relmax(th_single[i], th_oracle[i]) > 1e-9 for i in range(k))
    if model == "linreg":
        _, _, status = ops.batched_em(ops.BATCHED_LINREG, Xd.view(B * n, d), yd.view(-1), np.arange(B + 1) * n)
        out["host_solve"] = int((status.cpu() == batched.HOST_SOLVE).sum())
    # per-problem figures for like-for-like comparison when the loop ran on a subset
    out["batched_device_us_per_problem"] = 1e6 * out["batched_device_s"] / B
    out["dropin_loop_us_per_problem"] = 1e6 * out["dropin_loop_s"] / k
    out["oracle_us_per_problem"] = 1e6 * out["oracle_s"] / k
    out["speedup_vs_dropin_loop"] = out["dropin_loop_us_per_problem"] / out["batched_device_us_per_problem"]
    out["speedup_vs_oracle"] = out["oracle_us_per_problem"] / out["batched_device_us_per_problem"]
    out["numpy_speedup_vs_oracle"] = out["oracle_us_per_problem"] / (1e6 * out["batched_numpy_s"] / B)
    return out


def measure_logistic(mstep, X, y, reps, subset):
    dev = torch.device("cuda", 0)
    B, n, d = X.shape
    Xd, yd = torch.from_numpy(X).to(dev), torch.from_numpy(y).to(dev)
    code = {"sklearn": ops.BATCHED_LOGREG_NEWTON, "mm": ops.BATCHED_LOGREG_MM}[mstep]
    off = np.arange(B + 1) * n
    out = {"problems": B, "n": n, "d": d, "mstep": mstep, "reps": reps}
    out["batched_kernel_s"] = median_time(lambda: ops.batched_logistic(Xd.view(B * n, d), yd.view(-1), off, mstep=code),
                                          reps)
    _, _, status = ops.batched_logistic(Xd.view(B * n, d), yd.view(-1), off, mstep=code)
    out["host_solve"] = int((status.cpu() == batched.HOST_SOLVE).sum())
    try:
        out["batched_device_s"] = median_time(lambda: batched.logistic_regression(Xd, yd, mstep=mstep), reps)
        out["batched_numpy_s"] = median_time(lambda: batched.logistic_regression(X, y, mstep=mstep), reps)
        theta = batched.logistic_regression(X, y, mstep=mstep)
    except RuntimeError as exc:
        out["batched_device_s"] = out["batched_numpy_s"] = None
        out["batched_error"] = str(exc)
        theta = ops.batched_logistic(Xd.view(B * n, d), yd.view(-1), off, mstep=code)[0].cpu().numpy()
    k = min(subset, B)
    rlvi.logistic_regression(X[0], y[0], mstep=mstep)
    torch.cuda.synchronize()
    th_single, raised = [], []
    t0 = time.perf_counter()
    for b in range(k):
        try:
            th_single.append(rlvi.logistic_regression(X[b], y[b], mstep=mstep))
        except RuntimeError:
            th_single.append(None)
            raised.append(b)
    torch.cuda.synchronize()
    out["dropin_loop_s"] = time.perf_counter() - t0
    out["problems_timed"] = k
    out["dropin_raised"] = len(raised)
    ok = [b for b in range(k) if th_single[b] is not None and not np.isnan(theta[b]).any()]
    vs_dropin = [relmax(theta[b], th_single[b]) for b in ok]
    out["max_rel_theta_vs_dropin"] = max(vs_dropin)
    out["problems_over_1e-9_vs_dropin"] = sum(r > 1e-9 for r in vs_dropin)
    out["batched_kernel_us_per_problem"] = 1e6 * out["batched_kernel_s"] / B
    out["dropin_loop_us_per_problem"] = 1e6 * out["dropin_loop_s"] / k
    out["kernel_speedup_vs_dropin_loop"] = out["dropin_loop_us_per_problem"] / out["batched_kernel_us_per_problem"]
    if out["batched_device_s"] is not None:
        out["batched_device_us_per_problem"] = 1e6 * out["batched_device_s"] / B
        out["speedup_vs_dropin_loop"] = out["dropin_loop_us_per_problem"] / out["batched_device_us_per_problem"]
    if mstep == "mm":
        t0 = time.perf_counter()
        th_oracle = [rlvi_np.logistic_regression_mm(X[b], y[b]) for b in range(k)]
        out["oracle_s"] = time.perf_counter() - t0
        out["oracle_us_per_problem"] = 1e6 * out["oracle_s"] / k
        vs_oracle = [relmax(theta[b], th_oracle[b]) for b in ok]
        out["max_rel_theta_vs_oracle"] = max(vs_oracle)
        out["problems_over_1e-8_vs_oracle"] = sum(r > 1e-8 for r in vs_oracle)
        out["dropin_problems_over_1e-8_vs_oracle"] = sum(relmax(th_single[b], th_oracle[b]) > 1e-8 for b in ok)
        out["kernel_speedup_vs_oracle"] = out["oracle_us_per_problem"] / out["batched_kernel_us_per_problem"]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--large-subset", type=int, default=128)
    ap.add_argument("--logistic-subset", type=int, default=200)
    ap.add_argument("--logistic-large-subset", type=int, default=32)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batched_time.py measures on a GPU; none is visible")
    res = {"tool": "batched_time", **gpu_info(), "cpu_count": os.cpu_count(), "torch": torch.__version__}
    X, y = sweep_linreg(40, 10, 100, seed0=0)
    res["linreg_sweep_n40_d10"] = measure("linreg", X, y, a.reps)
    M = sweep_mean(100, 2, 100, seed0=0)
    res["mean_sweep_n100_d2"] = measure("mean", M, None, a.reps)
    X, y = sweep_linreg(1024, 64, 1184 // 20 + 1, seed0=7)
    res["linreg_1184_n1024_d64"] = measure("linreg", X[:1184], y[:1184], max(3, a.reps // 4), subset=a.large_subset)
    X, y = sweep_logistic(200, 10, 100, seed0=0)
    for mstep in ("sklearn", "mm"):
        res[f"logreg_{mstep}_sweep_n200_d10"] = measure_logistic(mstep, X, y, a.reps, a.logistic_subset)
    X, y = sweep_logistic(1024, 63, 1184 // 20 + 1, seed0=7)
    for mstep in ("sklearn", "mm"):
        res[f"logreg_{mstep}_1184_n1024_d63"] = measure_logistic(mstep, X[:1184], y[:1184], max(3, a.reps // 4),
                                                                 a.logistic_large_subset)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
