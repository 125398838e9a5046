"""ctypes binding of libcsmpn_b200.so (the C ABI declared in include/csmpn_b200.h).

There is no CPU fallback: if the shared library is missing this module raises at first use, and every
compute entry point refuses non-CUDA tensors.  PyTorch is only used for device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint8, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcsmpn_b200.so")

_lib = None


class CsmpnError(RuntimeError):
    pass


def _declare(lib):
    P = c_void_p
    i64, i32 = c_int64, c_int
    f = c_float
    sigs = {
        "csmpn_version": (c_int, []),
        "csmpn_status_string": (c_char_p, [i32]),
        "csmpn_last_cuda_error": (c_char_p, []),
        "csmpn_sm_count": (c_int, []),
        "csmpn_launch_count": (i64, []),
        "csmpn_algebra_tables": (c_int, [i32, P, P, P, P, P]),
        "csmpn_gp_fwd": (c_int, [i32, P, P, P, P, i64, i32, i32, P]),
        "csmpn_gp_bwd": (c_int, [i32, P, P, P, P, P, P, i64, i32, i32, P]),
        "csmpn_grade_forms_fwd": (c_int, [i32, P, P, P, i64, i32, P]),
        "csmpn_grade_forms_bwd": (c_int, [i32, P, P, P, P, i64, i32, P]),
        "csmpn_mvlinear_fwd": (c_int, [i32, P, P, P, P, i64, i32, i32, i32, P]),
        "csmpn_mvlinear_bwd_input": (c_int, [i32, P, P, P, i64, i32, i32, i32, P]),
        "csmpn_mvlinear_bwd_weight_workspace": (i64, [i32, i64, i32, i32]),
        "csmpn_mvlinear_bwd_weight": (c_int, [i32, P, P, P, P, i64, i32, i32, i32, P, i64, P]),
        "csmpn_mvsilu_fwd": (c_int, [i32, P, P, P, P, P, i64, i32, P]),
        "csmpn_mvsilu_bwd": (c_int, [i32, P, P, P, P, P, P, P, P, i64, i32, P, i64, P]),
        "csmpn_mvnorm_fwd": (c_int, [i32, P, P, P, P, i64, i32, P]),
        "csmpn_mvnorm_bwd": (c_int, [i32, P, P, P, P, P, P, i64, i32, P, i64, P]),
        "csmpn_mvlayernorm_fwd": (c_int, [i32, P, P, P, P, i64, i32, P]),
        "csmpn_mvlayernorm_bwd": (c_int, [i32, P, P, P, P, P, P, i64, i32, P, i64, P]),
        "csmpn_wgp_fwd": (c_int, [i32, P, P, P, P, P, f, P, i64, i32, P]),
        "csmpn_wgp_bwd": (c_int, [i32, P, P, P, P, P, f, P, P, P, i64, i32, P, i64, P]),
        "csmpn_param_grad_workspace": (i64, [i64]),
        "csmpn_csr_workspace": (i64, [i64, i64]),
        "csmpn_csr_build": (c_int, [P, i64, i64, P, P, P, i64, P]),
        "csmpn_gather_diff": (c_int, [P, P, P, P, i64, i64, P]),
        "csmpn_segment_reduce": (c_int, [P, P, P, P, i64, i64, i32, P]),
        "csmpn_scatter_diff": (c_int, [P, P, P, P, P, P, i64, i64, i32, P]),
        "csmpn_segment_expand": (c_int, [P, P, P, P, i64, i64, i32, P]),
        # fused CEMLP block / sorted-order EGCL helpers (descriptor structs are passed by reference)
        "csmpn_block_fwd": (c_int, [i32, P, P]),
        "csmpn_block_tc_supported": (c_int, [i32, i32, i32]),
        "csmpn_block_tc_plan": (c_int, [i32, i32, i32]),
        "csmpn_block_tc_passes": (c_int, [i32, i32, i32]),
        "csmpn_block_fwd_workspace": (i64, [i32, P]),
        "csmpn_block_simt_resident": (c_int, [i32, i32, i32]),
        "csmpn_bpt_floats": (i64, [i32, i64, i32]),
        "csmpn_block_bwd_workspace": (i64, [i32, P]),
        "csmpn_block_bwd": (c_int, [i32, P, P, P, i64, P]),
        "csmpn_csr_sorted_indices": (c_int, [P, P, P, P, P, i64, P]),
        "csmpn_csr_rank": (c_int, [P, P, i64, P]),
        "csmpn_csr_build_pair": (c_int, [P, P, i64, i64, P, P, P, P, P, P, P, P, i64, P]),
        "csmpn_segment_reduce_sorted": (c_int, [P, P, P, i64, i64, i32, P]),
        "csmpn_segment_expand_sorted": (c_int, [P, P, P, P, i64, i64, i32, P]),
        "csmpn_scatter_diff_sorted": (c_int, [P, i64, P, P, P, P, P, i64, i64, i32, P]),
        "csmpn_scatter_rows": (c_int, [P, i64, i64, P, P, i64, i64, P]),
        "csmpn_add3_rows": (c_int, [P, i64, P, i64, P, i64, P, i64, i64, P]),
        "csmpn_scatter_pair_sorted": (c_int, [P, i64, i64, i64, P, P, P, P, P, i64, i64, P]),
        # simplicial lifting
        "csmpn_lift_count": (c_int, [P, P, P, P, P, P]),
        "csmpn_lift_fill": (c_int, [P, P, P, i64, P, P, P, P, P]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return sigs


EXPORTED = None


def lib():
    """Load (once) and return the shared library; raise loudly if it is not built."""
    global _lib, EXPORTED
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CsmpnError(
                f"csmpn_b200: native library not found at {LIB_PATH}. Build it with "
                f"`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback."
            )
        l = ctypes.CDLL(LIB_PATH)
        EXPORTED = _declare(l)
        _lib = l
    return _lib


def check(status: int, what: str = ""):
    if status != 0:
        l = lib()
        msg = l.csmpn_status_string(status).decode()
        if status == -4:
            msg += ": " + l.csmpn_last_cuda_error().decode()
        raise CsmpnError(f"csmpn_b200 {what} failed: {msg} (status {status})")


def ptr(t: torch.Tensor | None):
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors, what="op"):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise CsmpnError(
                f"csmpn_b200.{what}: expected CUDA tensors (got device {t.device}); this package has no CPU path"
            )


def f32c(t: torch.Tensor) -> torch.Tensor:
    """fp32 + contiguous view/copy (the C ABI only takes dense fp32)."""
    if t.dtype != torch.float32:
        raise CsmpnError(f"csmpn_b200 kernels are fp32-only (got {t.dtype})")
    return t if t.is_contiguous() else t.contiguous()


def metric_host(metric) -> ctypes.Array:
    vals = [float(m) for m in metric]
    return (c_float * len(vals))(*vals)


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
