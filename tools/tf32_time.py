"""Times rlvi_weighted_moments_f32 at config-3 width: python tools/tf32_time.py [log2n] [d] [reps]."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from rlvi_b200 import ops

log2n = int(sys.argv[1]) if len(sys.argv) > 1 else 22
d = int(sys.argv[2]) if len(sys.argv) > 2 else 512
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 5
dev = torch.device("cuda", 0)
n = 1 << log2n
X = torch.randn((n, d), device=dev, dtype=torch.float32)
w = torch.rand(n, device=dev, dtype=torch.float64)
for prec, name in ((ops.TF32X3, "x3"), (ops.TF32X1, "x1")):
    out = None
    for _ in range(2):
        out = ops.weighted_moments(X, w, power=2, precision=prec, out=out)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        ops.weighted_moments(X, w, power=2, precision=prec, out=out)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    print(f"{name} n=2^{log2n} d={d} {ms:.3f} ms  {n * d * 4 / ms / 1e6:.0f} GB/s", flush=True)
