"""Times ops.fixed_point on bench.py's data with the series passes on and off (RLVI_FP_SERIES), alternating in one
process, at 2^26 samples (one GPU) and 2^23 (the shard of eight).  Prints ms per call, iterations, and the streamed
passes of the kernel's schedule (rlvi_b200/fp_series.py replayed on a 2^20-sample prefix of the same e).

    python tools/fp_series_time.py [--reps 20] [--rounds 3]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from rlvi_b200 import fp_series, ops, synth  # noqa: E402


def bench_e(log2n, dev):
    n = 1 << log2n
    X, y, theta = synth.logistic_rows_torch(0, n, 64, dev, seed=1234)
    params = torch.cat([torch.zeros(1, dtype=torch.float64, device=dev), theta]).contiguous()
    _, e, _ = ops.loss(ops.LOSS_LOGISTIC_CE, X, params, y=y, intercept=True, want_losses=False, want_e=True)
    del X, y
    return e


def time_calls(e, series, reps):
    os.environ["RLVI_FP_SERIES"] = "1" if series else "0"
    pi = torch.empty_like(e)
    res = torch.empty(5, dtype=torch.float64, device=e.device)
    ops.fixed_point(None, e_work=e, out=pi, result=res)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        ops.fixed_point(None, e_work=e, out=pi, result=res)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps, ops.read_result(res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(dev)
    print(json.dumps({"gpu": props.name}))
    for log2n in (26, 23):
        e = bench_e(log2n, dev)
        passes, _ = fp_series.replay(e[: 1 << 20].cpu().numpy())
        for rnd in range(args.rounds):
            for series in (True, False):
                ms, r = time_calls(e, series, args.reps)
                streamed = fp_series.streamed_passes(passes) if series else r["iters"]
                print(json.dumps({"log2n": log2n, "series": series, "round": rnd, "ms_per_call": round(ms, 4),
                                  "iters": r["iters"], "eps": r["eps"], "streamed_passes_model": streamed}))
        del e
        torch.cuda.empty_cache()
    os.environ.pop("RLVI_FP_SERIES", None)


if __name__ == "__main__":
    main()
