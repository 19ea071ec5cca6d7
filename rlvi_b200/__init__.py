"""rlvi_b200 -- the data-parallel hot path of RLVI (akarakulev/rlvi) on B200 (sm_100a).

Drop-in modules (reference file they mirror):
    rlvi_b200.rlvi    standard-learning/rlvi.py
    rlvi_b200.utils   standard-learning/utils.py
    rlvi_b200.deep    deep-learning/methods/train_rlvi.py
    rlvi_b200.online  online-learning/main.py (update_weights_rlvi, cross_entropy)
    rlvi_b200.ops     one function per C-ABI entry point (include/rlvi_b200.h), on CUDA tensors
    rlvi_b200.dist    sample-dimension sharding over the GPUs of one box
    rlvi_b200.batched many small independent update_weights / mean / linear_regression problems in one launch

The compute lives in rlvi_b200/librlvi_b200.so (hand-written CUDA, built by `__graft_entry__.build()`);
there is no CPU fallback -- importing the drop-ins works anywhere, calling them needs the library and a GPU.
"""
__version__ = "0.1.0"
