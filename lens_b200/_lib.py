"""ctypes binding of the C ABI declared in include/lens_b200.h.

The CUDA library is the product: if it is missing or cannot be loaded this module
raises -- there is no CPU or PyTorch fallback for any compute call.
"""
import ctypes as C
import os

from . import build as _build

_lib = None


class LensError(RuntimeError):
    pass


def _declare(L):
    vp, i32, i64, u32, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_float
    pi32, pi64 = C.POINTER(C.c_int), C.POINTER(C.c_int64)
    f64 = C.c_double
    sig = {
        "lens_version": (i32, [pi32, pi32]),
        "lens_last_error": (C.c_char_p, []),
        "lens_device_sm_count": (i32, [pi32]),
        "lens_launch_count": (i32, [pi64]),
        "lens_snn_set_timing": (i32, [vp, i32]),
        "lens_snn_get_timing": (i32, [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), pi64, pi64]),
        "lens_bin_events": (i32, [vp, vp, vp, i64, u32, u32, i32, i32, i32, i32, i32, i32,
                                  vp, vp, vp, vp, i64, vp]),
        "lens_pool_frames": (i32, [vp, i64, i32, i32, vp, vp]),
        "lens_check_sorted_u32": (i32, [vp, i64, vp, vp]),
        "lens_bin_event_streams": (i32, [vp, vp, vp, i64, vp, vp, i32, i32, u32, i32, i32, i32, i32, i32, i32,
                                         vp, vp, vp, vp, vp]),
        "lens_check_sorted_segments_u32": (i32, [vp, i64, vp, i32, vp, vp]),
        "lens_snn_create": (i32, [i32, i32, i32, i32, f32, f32, vp, vp, vp, i32,
                                  C.POINTER(vp), pi64, vp]),
        "lens_snn_destroy": (i32, [vp]),
        "lens_snn_reset": (i32, [vp, vp]),
        "lens_snn_reset_streams": (i32, [vp, vp, vp]),
        "lens_snn_get_state": (i32, [vp, vp, vp, vp, vp]),
        "lens_snn_get_overflow": (i32, [vp, vp, vp]),
        "lens_snn_forward": (i32, [vp, vp, i32, i32, vp, vp, vp, i32, vp]),
        "lens_snn_forward_range": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, i32, vp]),
        "lens_snn_forward_float": (i32, [vp, vp, i32, i32, vp, vp]),
        "lens_snn_forward_streams": (i32, [vp, vp, vp, i32, i32, vp, i32, vp]),
        "lens_seqmatch_topk": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp]),
        "lens_seqmatch_topk_stream": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, i64, vp, vp, vp]),
        "lens_seqmatch_topk_stream_ids": (i32, [vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp]),
        "lens_sad_matrix": (i32, [vp, vp, i32, i32, i32, vp, vp]),
        "lens_reciprocal": (i32, [vp, i64, vp, vp]),
        "lens_online_accumulate": (i32, [vp, vp, i32, i32, vp, vp]),
        "lens_online_match": (i32, [vp, i32, i32, i32, vp, vp, vp]),
        "lens_event_windows": (i32, [vp, vp, vp, i64, vp, i32, i32, i32, f64, f64, i64, vp, vp, vp, vp, vp, vp]),
        "lens_bin_events_lut": (i32, [vp, vp, vp, i32, i32, vp, vp, i64, i32, i32, i64, vp, vp, vp]),
        "lens_pr_counts": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, i32]),
        "lens_pr_counts_multi": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, i32]),
        "lens_recall": (i32, [vp, i32, i32, i32, i32, vp, i64, vp, i32, pi32, i32, vp, vp, vp]),
        "lens_recall_bounds": (i32, [vp, vp, i32, i32, pi32, i32, vp, vp, vp, vp]),
        "lens_seq_recall_bounds": (i32, [vp, i32, i32, i32, i32, vp, i64, vp, i32, pi32, i32, vp, vp, vp, vp]),
        "lens_seq_recall_bounds_stream": (i32, [vp, i32, i32, i32, i32, vp, vp, i64, vp, i32, pi32, i32, vp, vp, vp,
                                                vp]),
        "lens_seq_recall_bounds_stream_ids": (i32, [vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, i32, pi32, i32, vp,
                                                    vp, vp, vp]),
        "lens_topn_merge": (i32, [vp, vp, i32, i64, i32, vp, vp, vp]),
        "lens_seqpr_records_bytes": (i32, [i32, i32, i32, i32, i32, pi64]),
        "lens_seqpr_scan": (i32, [vp, i32, i32, i32, i32, i32, vp, i64, vp, i32, vp, vp, vp, vp]),
        "lens_seqpr_counts": (i32, [vp, i32, i32, i32, i32, i32, vp, i64, vp, i32, vp, vp, i32, vp, vp, vp]),
        "lens_seqpr_stream_bytes": (i32, [i32, i32, i32, i32, pi64]),
        "lens_seqpr_stream_accumulate": (i32, [vp, i32, i32, i32, i32, vp, vp, i64, vp, i32, vp, vp, vp, vp]),
        "lens_seqpr_stream_accumulate_ids": (i32, [vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp,
                                                   vp]),
        "lens_seqpr_stream_histogram": (i32, [vp, i32, i32, i32, i32, vp, vp, vp, vp]),
        "lens_seqpr_hist_counts": (i32, [vp, i32, i32, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    return sig


EXPORTS = None


def lib():
    """Load lens_b200/liblens_b200.so (building it with nvcc if the sources are newer)."""
    global _lib, EXPORTS
    if _lib is None:
        path = os.environ.get("LENS_B200_LIB")      # e.g. an instrumented build from tools/ (profiling only)
        if not path:
            path = _build.SO_PATH
            if _build.needs_build():
                path = _build.build()
        if not os.path.exists(path):
            raise LensError(f"{path} is missing: run `python -m lens_b200.build`")
        L = C.CDLL(path)
        EXPORTS = _declare(L)
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().lens_last_error().decode(errors="replace")
        raise LensError(f"{what} failed (rc={rc}): {msg}")


def stream_ptr():
    """cudaStream_t of torch's current stream, as a void* for the C ABI."""
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require_cuda(*tensors):
    import torch
    if not torch.cuda.is_available():
        raise LensError("lens_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback")
    for t in tensors:
        if t is not None and (not t.is_cuda or not t.is_contiguous()):
            raise LensError("lens_b200 expects contiguous CUDA tensors")


def launch_count():
    """Kernels launched by liblens_b200.so since it was loaded."""
    n = C.c_int64(0)
    check(lib().lens_launch_count(C.byref(n)), "lens_launch_count")
    return int(n.value)
