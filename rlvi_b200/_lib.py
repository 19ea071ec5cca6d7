"""ctypes binding of librlvi_b200.so (the C ABI declared in include/rlvi_b200.h).

There is NO CPU fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
Build the library with `python -c "import __graft_entry__ as g; g.build()"` (or `make -C rlvi_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librlvi_b200.so")

# every symbol include/rlvi_b200.h declares (tests/test_boundary.py checks the header against this)
SYMBOLS = (
    "rlvi_version", "rlvi_last_error", "rlvi_ctx_create", "rlvi_ctx_destroy", "rlvi_ctx_sm_count",
    "rlvi_ctx_launch_count", "rlvi_fp_dist_inbox_doubles", "rlvi_fixed_point_f64", "rlvi_fixed_point_init_f64",
    "rlvi_fixed_point_deep_f32", "rlvi_shift_sum_f64", "rlvi_shift_sum_e_f64", "rlvi_loss_f64", "rlvi_moments_out_doubles",
    "rlvi_weighted_moments_f64", "rlvi_weighted_moments_centered_f64", "rlvi_logistic_grad_f64", "rlvi_wce_fwd_bwd_f32", "rlvi_fn_threshold_f32",
    "rlvi_em_step_logistic_host", "rlvi_dist_window_create", "rlvi_dist_window_open", "rlvi_dist_window_close",
    "rlvi_stats_allreduce_f64", "rlvi_em_step_logistic_host_sharded", "rlvi_weighted_moments_f32", "rlvi_loss_f32", "rlvi_sigmoid_f64", "rlvi_online_ce_f64", "rlvi_irls_weights_f64", "rlvi_rrm_sum_f64", "rlvi_sever_pass_f64",
    "rlvi_batched_max_rows", "rlvi_batched_fixed_point_f64", "rlvi_batched_em_f64", "rlvi_batched_logistic_max_rows",
    "rlvi_batched_logistic_f64",
)

FP_STANDARD, FP_ONLINE, FP_DEEP = 0, 1, 2
LOSS_LOGISTIC_CE, LOSS_SOFTPLUS, LOSS_SQRES, LOSS_SQDIST, LOSS_PCA, LOSS_GAUSSIAN = range(6)
TF32X3, TF32X1 = 0, 1
BATCHED_MEAN, BATCHED_LINREG = 0, 1
BATCHED_LOGREG_NEWTON, BATCHED_LOGREG_MM = 0, 1


class FpResult(C.Structure):
    """struct rlvi_fp_result (include/rlvi_b200.h)."""
    _fields_ = [("eps", C.c_double), ("rho", C.c_double), ("sum_pi", C.c_double), ("err", C.c_double),
                ("iters", C.c_int32), ("converged", C.c_int32)]


class FpDist(C.Structure):
    """struct rlvi_fp_dist (include/rlvi_b200.h)."""
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("n_global", C.c_int64), ("inbox", C.c_void_p),
                ("peer_inbox", C.c_void_p), ("call_index", C.c_uint64)]


_lib = None
_lock = threading.RLock()       # re-entrant: context() -> Context() -> load()


def load():
    """dlopen the library once; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: the CUDA extension is not built and rlvi_b200 has no CPU fallback. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` in the repo root.")
        lib = C.CDLL(LIB_PATH)
        vp, i64, i32, f64, f32 = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_float
        lib.rlvi_version.restype = i32
        lib.rlvi_last_error.restype = C.c_char_p
        lib.rlvi_ctx_create.argtypes = [i32, C.POINTER(vp)]
        lib.rlvi_ctx_destroy.argtypes = [vp]
        lib.rlvi_ctx_sm_count.argtypes = [vp]
        lib.rlvi_ctx_launch_count.argtypes = [vp]
        lib.rlvi_ctx_launch_count.restype = i64
        lib.rlvi_fp_dist_inbox_doubles.argtypes = [i32]
        lib.rlvi_fixed_point_f64.argtypes = [vp, i32, vp, vp, vp, i64, f64, i32, vp, vp, C.POINTER(FpDist), vp]
        lib.rlvi_fixed_point_init_f64.argtypes = [vp, i32, vp, vp, vp, i64, f64, i32, f64, vp, vp, C.POINTER(FpDist), vp]
        lib.rlvi_fixed_point_deep_f32.argtypes = [vp, vp, vp, vp, i64, f32, i32, vp, C.POINTER(FpDist), vp]
        lib.rlvi_shift_sum_f64.argtypes = [vp, vp, i64, f64, f64, vp, vp, vp]
        lib.rlvi_shift_sum_e_f64.argtypes = [vp, vp, i64, f64, f64, vp, vp, vp]
        lib.rlvi_loss_f64.argtypes = [vp, i32, i32, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp]
        lib.rlvi_moments_out_doubles.argtypes = [i32]
        lib.rlvi_weighted_moments_f64.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, vp, vp]
        lib.rlvi_weighted_moments_centered_f64.argtypes = [vp, vp, vp, vp, vp, i64, i32, i32, i32, vp, vp]
        lib.rlvi_weighted_moments_f32.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp, vp]
        lib.rlvi_loss_f32.argtypes = [vp, i32, i32, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp]
        lib.rlvi_sigmoid_f64.argtypes = [vp, vp, i64, vp, vp]
        lib.rlvi_online_ce_f64.argtypes = [vp, vp, vp, i64, vp, vp]
        lib.rlvi_irls_weights_f64.argtypes = [vp, vp, vp, i64, vp, vp]
        lib.rlvi_rrm_sum_f64.argtypes = [vp, vp, i64, f64, f64, f64, vp, vp, vp]
        lib.rlvi_sever_pass_f64.argtypes = [vp, vp, i64, i32, vp, i32, f64, vp, vp, vp, vp, vp, vp, vp]
        lib.rlvi_logistic_grad_f64.argtypes = [vp, vp, vp, vp, i64, i32, vp, vp, vp]
        lib.rlvi_wce_fwd_bwd_f32.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, i64, vp, vp, vp, vp, vp]
        lib.rlvi_fn_threshold_f32.argtypes = [vp, vp, i64, f32, f32, i32, vp, vp]
        lib.rlvi_em_step_logistic_host.argtypes = [vp, vp, vp, i64, i32, vp, f64, i32, vp, vp, C.POINTER(FpResult)]
        lib.rlvi_em_step_logistic_host_sharded.argtypes = [vp, vp, vp, i64, i32, vp, f64, i32, vp, vp, C.POINTER(FpResult),
                                                           C.POINTER(FpDist), C.POINTER(FpDist)]
        lib.rlvi_batched_max_rows.argtypes = [i32]
        lib.rlvi_batched_fixed_point_f64.argtypes = [vp, vp, vp, i32, i64, f64, i32, vp, vp, vp]
        lib.rlvi_batched_em_f64.argtypes = [vp, i32, vp, vp, vp, i32, i64, i32, f64, i32, vp, vp, vp, vp]
        lib.rlvi_batched_logistic_max_rows.argtypes = [i32]
        lib.rlvi_batched_logistic_f64.argtypes = [vp, i32, vp, vp, vp, i32, i64, i32, f64, i32, vp, vp, vp, vp]
        lib.rlvi_dist_window_create.argtypes = [vp, i32, C.POINTER(vp), C.c_char_p]
        lib.rlvi_dist_window_open.argtypes = [vp, i32, i32, vp, C.c_char_p, C.POINTER(vp)]
        lib.rlvi_dist_window_close.argtypes = [vp, i32, i32, vp, vp]
        lib.rlvi_stats_allreduce_f64.argtypes = [vp, vp, i32, C.POINTER(FpDist), vp]
        for name in SYMBOLS:
            fn = getattr(lib, name)            # AttributeError here == the .so does not export the header
            if name not in ("rlvi_last_error", "rlvi_ctx_launch_count"):
                fn.restype = i32
        _lib = lib
    return _lib


class RlviError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        msg = load().rlvi_last_error().decode("utf-8", "replace")
        raise RlviError(f"{what} failed (code {rc}): {msg}")


class Context:
    """One rlvi_ctx per (device, stream); owns the library's device scratch.  Calls on one context must be
    stream-ordered (include/rlvi_b200.h, Conventions), so `context()` hands out one per CUDA stream."""

    def __init__(self, device: int):
        self.lib = load()
        self.device = int(device)
        h = C.c_void_p()
        check(self.lib.rlvi_ctx_create(self.device, C.byref(h)), "rlvi_ctx_create")
        self.handle = h
        self.sm_count = self.lib.rlvi_ctx_sm_count(h)

    @property
    def launches(self) -> int:
        return int(self.lib.rlvi_ctx_launch_count(self.handle))

    def close(self):
        if getattr(self, "handle", None):
            self.lib.rlvi_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_contexts: dict = {}


def context(device: int, stream: int = 0) -> Context:
    """The context of (device, stream handle); stream 0 = the legacy default stream (torch's default)."""
    key = (int(device), int(stream or 0))
    ctx = _contexts.get(key)
    if ctx is None:
        load()
        with _lock:
            ctx = _contexts.get(key)
            if ctx is None:
                ctx = _contexts[key] = Context(device)
    return ctx


def launches(device: int) -> int:
    """Kernels launched by the library on `device`, over all its contexts."""
    return sum(c.launches for (d, _), c in list(_contexts.items()) if d == int(device))
