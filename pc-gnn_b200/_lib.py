"""ctypes binding of libpcgnn_b200.so (the C ABI declared in include/pcgnn_b200.h).

There is no CPU fallback: if the library has not been built, or a kernel call fails, this raises.
Build it with ``python -c "import __graft_entry__ as g; g.build()"`` (or ``make -C pc-gnn_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PCG_LIB_VARIANT=trace selects the per-item phase tracer build (profiles/trace_choose.py; `make trace`)
SO_PATH = os.path.join(_HERE, "libpcgnn_b200_trace.so" if os.environ.get("PCG_LIB_VARIANT") == "trace"
                       else "libpcgnn_b200.so")

SLOT = 64            # PCG_SLOT
MAX_REL = 8          # PCG_MAX_REL
STATUS_WORDS = 12    # PCG_STATUS_WORDS
ST_SLOTS, ST_OVERFLOW = 0, 3
NORM_MEAN, NORM_RSQRT = 0, 1
KB_MAX_POOL = 8192   # PCG_KB_WORDS * 32: pools up to this size use the per-item kept-pool bitmap
# PCG_METRICS_WORDS doubles written by pcg_binary_metrics, in the order of the PCG_MT_* word indices
METRICS_KEYS = ("auc", "f1", "f1_macro", "recall", "precision", "recall_macro", "precision_macro", "accuracy", "gmean",
                "best_f1_macro", "best_threshold", "n_pos", "n_neg", "tp", "fp", "tn", "fn",
                "ap", "recall_at_k", "best_gmean", "best_gmean_threshold")
METRICS_WORDS = len(METRICS_KEYS)
POINT_WORDS = 5      # PCG_POINT_WORDS: doubles per pcg_binary_points request
POINTS_MAX = 1024    # PCG_POINTS_MAX
POINT_TOP_K, POINT_TPR_AT_FPR, POINT_PAUC = 0, 1, 2

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_z = C.c_size_t
_d = C.c_double
_u64 = C.c_uint64

# name -> (restype, argtypes); mirrors include/pcgnn_b200.h one to one
SIGNATURES = {
    "pcg_last_error": (C.c_char_p, []),
    "pcg_version": (_i, []),
    "pcg_device_sms": (_i, []),
    "pcg_set_pdl": (_i, [_i]),
    "pcg_score_table": (_i, [_p, _l, _i, _l, _p, _p, _p, _p, _i, _p, _p, _p, _p, _z, _p]),
    "pcg_pool_scores": (_i, [_p, _i, _l, _p, _p, _p, _i, _p, _p]),
    "pcg_stage": (_i, [_p, _p, _z, _p]),
    "pcg_host_device_ptr": (_p, [_p]),
    "pcg_pool_scores_stage": (_i, [_p, _i, _l, _p, _p, _p, _i, _p, _p, _p, _z, _p, C.c_uint32, _l, _p]),
    "pcg_stage_indexed": (_i, [_p, _p, _z, _p, C.c_uint32, _l, _l, _i, _p]),
    "pcg_sort_pool_workspace_bytes": (_z, [_i]),
    "pcg_sort_pool": (_i, [_p, _p, _i, _p, _p, _p, _p, _z, _p]),
    "pcg_choose_workspace_bytes": (_z, [_i, _i, _l, _l]),
    "pcg_choose_sticky_offset": (_z, [_l]),
    "pcg_choose_workspace_init": (_i, [_p, _z, _l, _p]),
    "pcg_pool_positions": (_i, [_p, _i, _l, _p, _p]),
    "pcg_entry_pool_positions": (_i, [_p, _l, _p, _p, _p]),
    "pcg_choose": (_i, [_p, _p, _l, _l, _i, _p, _p, _p, _p, _p, _i, C.POINTER(_d), _p, _d, _p, _p, _p, _p, _i, _i, _l,
                        _p, _p, _l, _p, _p, _p, _p, _p, _p, _p, _z, _p, _i, _p]),
    "pcg_select_all": (_i, [_p, _p, _l, _i, _p, _i, _i, _l, _p, _p, _p, _p, _p, _p, _p, _p]),
    "pcg_aggregate": (_i, [_p, _l, _p, _p, _p, _p, _p, _p, _p, _i, _i, _l, _p, _i, _p, _p, _p, _p]),
    "pcg_aggregate_bwd": (_i, [_p, _l, _p, _p, _p, _p, _p, _p, _i, _l, _p, _i, _p, _p]),
    "pcg_dense_fwd": (_i, [_p, _l, _i, _p, _i, _i, _i, _p, _p, C.POINTER(_p), _p, _p, _p, _p]),
    "pcg_dense_bwd_scratch_floats": (_z, [_i, _i, _i, _i]),
    "pcg_dense_bwd": (_i, [_l, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, C.POINTER(_p), _p, _p, _p]),
    "pcg_tile_supported": (_i, [_i, _i, _i, _i]),
    "pcg_tile_fwd": (_i, [_p, _l, _i, _p, _i, _i, _i, _p, _l, _p, C.POINTER(_p), _p, _p, _p, _i, _p, _p, _p, _p]),
    "pcg_tile_scratch_floats": (_z, [_i, _i, _i, _i]),
    "pcg_tile_train": (_i, [_p, _l, _i, _p, _i, _i, _i, _p, _l, _p, C.POINTER(_p), _p, _p, _p, _p, _p, C.c_float,
                            _p, _p, _p, _p, C.POINTER(_p), _p, _p, _p, _p, _p, _i, _p]),
    "pcg_head_scratch_floats": (_z, [_i, _i, _i]),
    "pcg_center_fwd": (_i, [_p, _l, _i, _p, _i, _p, _p, _p, _p]),
    "pcg_center_bwd": (_i, [_p, _l, _i, _p, _i, _p, _p, _p, _p, _p, _p]),
    "pcg_head_loss_fwd": (_i, [_p, _i, _i, _p, _p, _p, C.c_float, _p, _p, _p, _p, _p, _p, _p]),
    "pcg_head_loss_bwd": (_i, [_p, _i, _i, _p, _p, _p, _p, C.c_float, _p, _p, _p, _p, _p, _p, _p]),
    "pcg_encoder_scratch_floats": (_z, [_i, _i, _i]),
    "pcg_encoder_fwd": (_i, [_p, _l, _p, _l, _p, _i, _p, _i, _i, _p, _p]),
    "pcg_encoder_bwd": (_i, [_p, _l, _p, _l, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p]),
    "pcg_comm_region_bytes": (_z, [_l]),
    "pcg_comm_alloc": (_i, [C.POINTER(_p), _z]),
    "pcg_comm_free": (_i, [_p]),
    "pcg_comm_export": (_i, [_p, C.c_char_p]),
    "pcg_comm_import": (_i, [C.c_char_p, C.POINTER(_p)]),
    "pcg_comm_unmap": (_i, [_p]),
    "pcg_allreduce_adam": (_i, [_p, _p, _p, _p, _l, C.POINTER(_p), _i, _i, _p, _p, C.c_float, C.c_float, C.c_float,
                                C.c_float, C.c_float, _i, _p]),
    "pcg_score_region_bytes": (_z, [_l]),
    "pcg_score_bcast": (_i, [_p, _l, _i, _l, _p, _p, _l, _l, C.POINTER(_p), _i, _i, _p, _p]),
    "pcg_pick_step": (_i, [_p, _l, _p, _l, _p, _p, _p]),
    "pcg_pick_step_philox": (_i, [_p, _l, _u64, _u64, _l, _p, _p, _p]),
    "pcg_eval_head": (_i, [_p, _i, _i, _p, _i, _l, _p, C.c_uint32, _p, _p]),
    "pcg_binary_metrics_workspace_bytes": (_z, [_l]),
    "pcg_binary_metrics": (_i, [_p, _p, _l, _p, _p, _z, _p]),
    "pcg_binary_curve": (_i, [_p, _z, _l, _p, _p, _p, _p, _p]),
    "pcg_binary_points_workspace_bytes": (_z, [_l, _i]),
    "pcg_binary_points": (_i, [_p, _z, _l, _p, _p, _i, _p, _p, _z, _p]),
}

_lib = None


class PcgError(RuntimeError):
    pass


def lib():
    """The loaded library (dlopen on first use). Raises if it was never built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise PcgError(
                f"{SO_PATH} is missing: the CUDA extension has not been built "
                "(run `python -c \"import __graft_entry__ as g; g.build()\"`). There is no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().pcg_last_error().decode("utf-8", "replace")
        raise PcgError(f"{what or 'pcgnn_b200'} failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def host_device_ptr(pinned_tensor) -> int:
    """Device address of a pinned (page-locked) host tensor; raises when the memory is not device-mapped."""
    dev = lib().pcg_host_device_ptr(pinned_tensor.data_ptr())
    if not dev:
        raise PcgError(lib().pcg_last_error().decode("utf-8", "replace"))
    return int(dev)


class capture:
    """``with capture(graph):`` = ``with torch.cuda.graph(graph):`` with Python's garbage collector out of the way.
    Destroying a CUDA graph while a stream is capturing invalidates the capture, and the collector may decide at any
    moment, also in the middle of a recording, to free cyclic garbage that owns graphs (an InterAgg and its graph cache
    reference each other). So: collect first, then keep the collector off until the recording has ended."""

    def __init__(self, graph, **kw):
        import torch

        self._ctx = torch.cuda.graph(graph, **kw)
        self._was = False

    def __enter__(self):
        import gc

        gc.collect()
        self._was = gc.isenabled()
        gc.disable()
        try:
            return self._ctx.__enter__()
        except BaseException:
            if self._was:
                gc.enable()
            raise

    def __exit__(self, *exc):
        import gc

        try:
            return self._ctx.__exit__(*exc)
        finally:
            if self._was:
                gc.enable()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream
