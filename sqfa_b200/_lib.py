"""ctypes binding of libsqfa_b200.so (the C ABI in include/sqfa_b200.h).

There is no CPU fallback: if the shared library is missing, or a kernel is asked to run without a
CUDA device, the call raises. PyTorch is used only for device memory and streams; every compute
call goes through the `extern "C"` entry points with raw device pointers.
"""

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsqfa_b200.so")

_lib = None

c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_u32 = ctypes.c_uint32
c_f32 = ctypes.c_float
c_ptr = ctypes.c_void_p
c_size = ctypes.c_size_t
c_int = ctypes.c_int

# element codes of the *_h entry points (SQFA_ELEM_* in include/sqfa_b200.h)
ELEM_CODES = {torch.bfloat16: 1, torch.float16: 2}

# name -> (restype, argtypes); mirrors include/sqfa_b200.h one to one
SIGNATURES = {
    "sqfa_version": (c_int, []),
    "sqfa_build_id": (ctypes.c_char_p, []),
    "sqfa_last_error": (ctypes.c_char_p, []),
    "sqfa_device_sm_count": (c_int, []),
    "sqfa_label_max": (c_int, [c_ptr, c_i64, c_ptr, c_ptr]),
    "sqfa_bucket_workspace_bytes": (c_size, [c_i64, c_i32]),
    "sqfa_bucket_labels": (c_int, [c_ptr, c_i64, c_i32, c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_ptr]),
    "sqfa_class_sums_workspace_bytes": (c_size, [c_i64, c_i32, c_i32]),
    "sqfa_class_sums": (
        c_int,
        [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_means": (c_int, [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_class_gram_workspace_bytes": (c_size, [c_i64, c_i32, c_i32]),
    "sqfa_class_gram": (
        c_int,
        [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_int, c_ptr, c_i32, c_i32, c_i32,
         c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_gram_group_signals": (c_i64, [c_i64, c_i32, c_i32, c_i32, c_i32]),
    "sqfa_stream_wait_geq": (c_int, [c_ptr, c_ptr, c_i32]),
    "sqfa_gram_packed_floats": (c_size, [c_i32, c_i32]),
    "sqfa_gram_executed_tile_area": (c_i64, [c_i32]),
    "sqfa_class_gram_sum_splits": (c_i32, [c_i64, c_i32, c_i32]),
    "sqfa_class_pilot_shift": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_class_gram_sums": (
        c_int,
        [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_means_from_partials": (c_int, [c_ptr, c_i32, c_ptr, c_ptr, c_i32, c_i32, c_ptr, c_ptr, c_ptr]),
    "sqfa_class_gram_sum_splits_h": (c_i32, [c_i64, c_i32, c_i32, c_i32]),
    "sqfa_class_pilot_shift_h": (c_int, [c_ptr, c_i64, c_i32, c_ptr, c_ptr, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_class_gram_sums_h": (
        c_int,
        [c_ptr, c_i64, c_i32, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_counts_pack": (c_int, [c_ptr, c_i32, c_ptr, c_ptr]),
    "sqfa_counts_unpack": (c_int, [c_ptr, c_i32, c_ptr, c_ptr]),
    "sqfa_stats_epilogue_workspace_bytes": (c_size, [c_i32]),
    "sqfa_stats_epilogue": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_int, c_int, c_ptr, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_stats_epilogue_reduce": (
        c_int,
        [c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_int, c_int, c_ptr, c_ptr, c_ptr,
         c_size, c_ptr],
    ),
    "sqfa_peer_push": (c_int, [c_ptr, c_ptr, c_size, c_ptr]),
    "sqfa_class_statistics_workspace_bytes": (c_size, [c_i64, c_i32, c_i32]),
    "sqfa_class_statistics": (
        c_int,
        [c_ptr, c_i64, c_ptr, c_i64, c_i32, c_i32, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
         c_size, c_ptr],
    ),
    "sqfa_class_sums_h": (
        c_int,
        [c_ptr, c_i64, c_i32, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_gram_workspace_bytes_h": (c_size, [c_i64, c_i32, c_i32, c_i32]),
    "sqfa_class_gram_h": (
        c_int,
        [c_ptr, c_i64, c_i32, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_int, c_ptr, c_i32, c_i32,
         c_i32, c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_gram_group_signals_h": (c_i64, [c_i64, c_i32, c_i32, c_i32, c_i32, c_i32]),
    "sqfa_class_statistics_workspace_bytes_h": (c_size, [c_i64, c_i32, c_i32, c_i32]),
    "sqfa_class_statistics_h": (
        c_int,
        [c_ptr, c_i64, c_i32, c_ptr, c_i64, c_i32, c_i32, c_int, c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
         c_ptr, c_size, c_ptr],
    ),
    "sqfa_transform_h": (c_int, [c_ptr, c_i64, c_i32, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_class_sums_f64": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_ptr]),
    "sqfa_class_means_f64": (c_int, [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_class_gram_f64": (c_int, [c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_int, c_ptr]),
    "sqfa_stats_epilogue_f64": (
        c_int, [c_ptr, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_int, c_int, c_ptr, c_ptr, c_ptr]),
    "sqfa_lbfgs_max_n": (c_i64, []),
    "sqfa_lbfgs_max_history": (c_i32, []),
    "sqfa_lbfgs_direction": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_f32, c_int, c_ptr, c_f32, c_f32, c_ptr,
         c_ptr],
    ),
    "sqfa_lbfgs_max_n_f64": (c_i64, []),
    "sqfa_lbfgs_direction_f64": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i32, c_ptr, c_int, c_ptr, c_ptr, c_ptr],
    ),
    "sqfa_project_workspace_bytes": (c_size, [c_i32, c_i32, c_i32]),
    "sqfa_project_fwd": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_ptr, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_project_bwd": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_transform": (c_int, [c_ptr, c_i64, c_ptr, c_i64, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_embed_fwd": (c_int, [c_ptr, c_ptr, c_f32, c_i32, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_embed_bwd": (c_int, [c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_ptr, c_ptr]),
    "sqfa_class_factor_floats": (c_size, [c_i32, c_i32]),
    "sqfa_class_factor": (c_int, [c_ptr, c_i32, c_i32, c_i32, c_ptr, c_ptr, c_ptr]),
    "sqfa_pair_distances_workspace_bytes": (c_size, [c_i32, c_i32, c_i32, c_i32, c_i32, c_i64, c_i64]),
    "sqfa_pair_distances": (
        c_int,
        [c_ptr, c_ptr, c_i32, c_i32, c_i32, c_i32, c_i32, c_i64, c_i64, c_f32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
         c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_class_factor_bwd": (c_int, [c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_ptr]),
    "sqfa_gauss_pair_workspace_bytes": (c_size, [c_i32, c_i32, c_i32, c_i32]),
    "sqfa_gauss_pair_distances": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_i32, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_size,
         c_ptr, c_ptr],
    ),
    "sqfa_fused_loss_workspace_bytes": (c_size, [c_i32, c_i32, c_i32, c_i32, c_i64, c_i64]),
    "sqfa_fused_loss": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_f32, c_i32, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_size, c_ptr],
    ),
    "sqfa_fused_loss_exchange_span": (c_int, [c_i32, c_i32, c_i32, c_i32, c_i64, c_i64, c_i32, c_ptr, c_ptr]),
    "sqfa_fused_loss_sharded": (
        c_int,
        [c_i32, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_f32, c_i32, c_i32, c_i32, c_i64, c_i64, c_ptr, c_ptr,
         c_size, c_ptr],
    ),
    "sqfa_closure_eval": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_f32, c_i32, c_i32, c_i32, c_i64, c_i64, c_ptr, c_ptr, c_ptr,
         c_ptr, c_size, c_ptr],
    ),
    "sqfa_fused_loss_workspace_bytes_f64": (c_size, [c_i32, c_i32, c_i32, c_i32, c_i64, c_i64]),
    "sqfa_closure_eval_f64": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_i32, c_i32, c_i32, c_i64, c_i64, c_ptr, c_ptr, c_ptr,
         c_ptr, c_size, c_ptr],
    ),
    "sqfa_fused_loss_exchange_span_f64": (c_int, [c_i32, c_i32, c_i32, c_i32, c_i64, c_i64, c_i32, c_ptr, c_ptr]),
    "sqfa_fused_loss_sharded_f64": (
        c_int,
        [c_i32, c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_i32, c_i32, c_i32, c_i64, c_i64, c_ptr, c_ptr,
         c_size, c_ptr],
    ),
    "sqfa_gauss_closure_workspace_bytes_f64": (c_size, [c_i32, c_i32, c_i32, c_i32, c_i64, c_i64]),
    "sqfa_gauss_closure_eval_f64": (
        c_int,
        [c_ptr, c_ptr, c_ptr, c_i32, c_i32, c_i32, c_ptr, c_i32, c_i32, c_i32, c_i64, c_i64, c_ptr, c_ptr, c_ptr,
         c_ptr, c_size, c_ptr],
    ),
}


class SqfaNativeError(RuntimeError):
    """Raised when a native call reports failure."""


def load():
    """Load libsqfa_b200.so and declare every prototype. Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SqfaNativeError(
            f"{LIB_PATH} not found. Build it with `python -m sqfa_b200.build` (needs nvcc). "
            "sqfa_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    missing = []
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:  # header / library drift; tests/test_abi.py fails on this
            missing.append(name)
            continue
        fn.restype = restype
        fn.argtypes = argtypes
    lib.sqfa_missing_symbols = tuple(missing)
    if "sqfa_build_id" not in missing and os.environ.get("SQFA_ALLOW_STALE_LIB") != "1":
        # a library built from other sources than the ones next to it would be tested / run silently
        from . import build as _build

        want = _build.source_build_id()
        have = lib.sqfa_build_id().decode()
        if want is not None and have != want:
            raise SqfaNativeError(
                f"{LIB_PATH} was built from different sources (build id {have}, sources {want}); "
                "rebuild it with `python -m sqfa_b200.build`"
            )
    _lib = lib
    return lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def check(code, what):
    if code != 0:
        msg = load().sqfa_last_error()
        raise SqfaNativeError(f"{what} failed with code {code}: {msg.decode() if msg else ''}")


def require_cuda(*tensors):
    """The kernels only run on a CUDA device; fail loudly instead of falling back."""
    if not torch.cuda.is_available():
        raise SqfaNativeError(
            "sqfa_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback."
        )
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise SqfaNativeError("internal error: expected CUDA tensors at the native boundary")


def compute_device(*tensors):
    """Device the kernels run on: the device of the first CUDA input, else the current device."""
    for t in tensors:
        if isinstance(t, torch.Tensor) and t.is_cuda:
            return t.device
    if not torch.cuda.is_available():
        raise SqfaNativeError(
            "sqfa_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback."
        )
    return torch.device("cuda", torch.cuda.current_device())
