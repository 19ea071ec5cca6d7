"""Time the batched RLVI fits (rlvi_b200.batched) against the per-problem drop-in loop and the NumPy oracle on the
reference experiment driver's Monte-Carlo sweeps (standard-learning/main.py: test_linear_regression, N = 40, d = 10;
test_mean, N = 100, d = 2; 20 corruption rates linspace(0, 0.4, 20) x 100 runs = 2000 problems each), plus one larger point
(1184 linear-regression problems of N = 1024, d = 64: 8 problems per SM).  Prints one JSON line.

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

    python tools/batched_time.py [--reps 20] [--large-subset 128] [--out r04_batched.json]
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--large-subset", type=int, default=128)
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
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
