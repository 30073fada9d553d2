"""ctypes binding of libhnr.so (the C ABI declared in include/hnr.h).

The product path has NO fallback: if the shared library is missing or was not built for the
device in use, importing/calling raises.  PyTorch is only used for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libhnr.so")

_lib = None

vp, i64, i32, f32c = C.c_void_p, C.c_int64, C.c_int32, C.c_float


class GridT(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("cell", C.c_float * 3), ("dims", C.c_int32 * 3), ("radius2", C.c_float),
                ("n_cells", C.c_int64), ("P", C.c_int32), ("layers", C.c_int32), ("qhalf_lo", C.c_int32 * 3),
                ("qhalf_hi", C.c_int32 * 3)]


_SIGS = {
    "hnr_abi_version": (C.c_int, []),
    "hnr_last_error": (C.c_char_p, []),
    "hnr_device_arch": (C.c_int, []),
    "hnr_scan_scratch_elems": (i64, [i64]),
    "hnr_exclusive_scan_i32": (C.c_int, [vp, vp, i64, vp, vp]),
    "hnr_grid_build": (C.c_int, [vp, i64, C.POINTER(GridT), i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "hnr_query": (C.c_int, [vp, vp, vp, vp, i64, i64, i64, i64, i64, C.POINTER(GridT)] + [vp] * 19 + [vp]),
    "hnr_nbr_weights": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, vp, vp, vp, vp]),
    "hnr_nbr_features": (C.c_int, [vp] * 10 + [vp, i64, i64, i64, vp, vp, vp]),
    "hnr_nbr_features_bwd": (C.c_int, [vp] * 7 + [vp, i64, i64, vp, vp, vp, vp]),
    "hnr_alpha_ksum_fwd": (C.c_int, [vp] * 7 + [vp, i64, i64, i64, vp, vp, vp, vp]),
    "hnr_alpha_ksum_bwd": (C.c_int, [vp] * 8 + [i64, i64, i64, vp, vp, vp, vp, vp]),
    "hnr_conf_bwd": (C.c_int, [vp] * 5 + [i64, i64, i64, vp, vp]),
    "hnr_project_views": (C.c_int, [vp] * 5 + [i64, i64, vp, vp, vp]),
    "hnr_image_gather_fwd": (C.c_int, [C.POINTER(vp), C.POINTER(i64), vp, vp, i64, i64, i64, vp, vp, i64, vp, vp]),
    "hnr_image_gather_bwd": (C.c_int, [C.POINTER(vp), C.POINTER(i64), vp, vp, vp, i64, i64, i64, vp]),
    "hnr_blend_fwd": (C.c_int, [vp, vp, vp, vp, i64, i64, i64, vp, i64, vp]),
    "hnr_blend_bwd": (C.c_int, [vp, vp, vp, vp, vp, i64, i64, vp, vp, vp]),
    "hnr_linear_head_bwd": (C.c_int, [vp, vp, C.c_int, vp, vp, i64, i64, i64, vp, i64, vp, vp, vp]),
    "hnr_peer_sum_f32": (C.c_int, [C.POINTER(vp), C.c_int, i64, vp, vp]),
    "hnr_multimem_sum_f32": (C.c_int, [vp, i64, vp, vp]),
    "hnr_blend_bwd_ld": (C.c_int, [vp, i64, vp, vp, vp, vp, i64, i64, vp, i64, vp, vp]),
    "hnr_image_gather_bwd_ld": (C.c_int, [C.POINTER(vp), C.POINTER(i64), vp, vp, vp, i64, i64, i64, i64, vp]),
    "hnr_linear_fwd": (C.c_int, [C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, vp, vp, i64, vp, i64, i64, i64,
                                 i64, C.c_int, vp]),
    "hnr_linear_bwd_data": (C.c_int, [vp, i64, vp, i64, vp, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), i64, i64, i64, C.c_int, vp]),
    "hnr_linear_bwd_data_narrow": (C.c_int, [vp, i64, vp, i64, C.c_int, vp, i64, i64, i64, vp, i64, i64, i64, vp]),
    "hnr_linear_bwd_weight": (C.c_int, [vp, i64, vp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, vp, i64,
                                        i64, i64, C.c_int, vp]),
    "hnr_composite_fwd": (C.c_int, [vp, vp, vp, C.c_int, vp, vp, f32c, C.c_int, i64, i64, vp, vp, vp, vp, vp, vp, vp]),
    "hnr_composite_bwd": (C.c_int, [vp] * 11 + [i64, i64, vp, vp]),
    "hnr_blur_select_fwd": (C.c_int, [vp, vp, vp, i64, i64, i64, i64, vp, vp, vp]),
    "hnr_blur_select_bwd": (C.c_int, [vp, vp, vp, i64, i64, i64, i64, vp, vp]),
    "hnr_blur_gray_fwd": (C.c_int, [vp, vp, i64, i64, vp, vp]),
    "hnr_blur_gray_bwd": (C.c_int, [vp, i64, i64, vp, vp]),
    "hnr_blur_learn_fwd": (C.c_int, [vp, vp, i64, i64, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp]),
    "hnr_blur_learn_bwd": (C.c_int, [vp, vp, i64, vp, i64, i64, i64, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "hnr_linear_tc_packed_bytes": (i64, [i64, i64]),
    "hnr_linear_tc_fwd": (C.c_int, [C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, i64, i64, vp, vp, i64, vp, i64, i64,
                                    i64, i64, C.c_int, vp, vp, C.c_int, vp, vp]),
    "hnr_linear_tc_bwd_data": (C.c_int, [vp, i64, vp, i64, C.c_int, vp, i64, i64, vp, i64, i64, i64, i64, vp]),
    "hnr_linear_tc_bwd_weight": (C.c_int, [vp, i64, vp, i64, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp, vp, i64,
                                           i64, i64, C.c_int, vp]),
    "hnr_adam_step": (C.c_int, [vp, vp, vp, vp, i64, f32c, f32c, f32c, f32c, f32c, i64, vp]),
    "hnr_adam_multi": (C.c_int, [i64, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), f32c, f32c, f32c, f32c, f32c,
                                 i64, vp, vp]),
    "hnr_frame_rays": (C.c_int, [vp, i64, i64, i64, i64, i64, vp, vp, C.c_int, vp, vp, vp, vp, vp]),
    "hnr_frame_views": (C.c_int, [vp, vp, i64, i64, vp, vp]),
    "hnr_nbr_mlp_f16_packed_bytes": (i64, []),
    "hnr_chain_f16_chunk_bytes": (i64, [i64]),
    "hnr_chain_f16_set_trace": (None, [vp]),
    "hnr_chain_f16_forward": (C.c_int, [C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), f32c, C.c_int, C.POINTER(i64),
                                        C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_int), vp, C.POINTER(i64), vp, C.POINTER(f32c),
                                        C.POINTER(f32c), C.POINTER(vp), C.POINTER(i64), vp, i64, vp, vp, C.c_int, vp, i64, vp, vp]),
    "hnr_nbr_mlp_f16_forward": (C.c_int, [vp] * 17 + [C.POINTER(C.c_float), f32c, f32c, f32c, i64, i64, vp, vp, vp, vp, vp, vp]),
    "hnr_nbr_mlp_f16_forward_pp": (C.c_int, [vp] * 17 + [C.POINTER(C.c_float), f32c, f32c, f32c, i64, i64, vp, vp, vp, vp]),
    "hnr_nbr_mlp_f16_forward_train": (C.c_int, [vp] * 17 + [C.POINTER(C.c_float), f32c, f32c, f32c, i64, i64] + [vp] * 11),
    "hnr_alpha_ksum_bwd_img": (C.c_int, [vp] * 8 + [i64, i64, vp, vp, vp, vp, vp, vp]),
    "hnr_nbr_bwd_f16_packed_bytes": (i64, []),
    "hnr_nbr_bwd_f16": (C.c_int, [vp] * 8 + [i64, i64, vp, i64, vp]),
    "hnr_dz_extras_bwd": (C.c_int, [vp, vp, i64, i64, i64, vp, vp]),
    "hnr_wgrad_img_jobs": (C.c_int, [C.c_int, C.POINTER(vp), C.POINTER(i64), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), C.POINTER(i64),
                                     C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), vp]),
    "hnr_chain_f16_forward_train": (C.c_int, [C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), f32c, C.c_int, C.POINTER(i64),
                                              C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_int), vp, C.POINTER(i64), vp, C.POINTER(f32c),
                                              C.POINTER(f32c), C.POINTER(vp), C.POINTER(i64), vp, i64, vp, vp, C.c_int, vp, i64, vp, vp,
                                              C.POINTER(vp), vp]),
    "hnr_chain_f16_forward_add0": (C.c_int, [C.POINTER(vp), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), f32c, C.c_int, C.POINTER(i64),
                                             C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_int), vp, C.POINTER(i64), vp, C.POINTER(f32c),
                                             C.POINTER(f32c), C.POINTER(vp), C.POINTER(i64), vp, i64, vp, vp, C.c_int, vp, i64, vp, vp,
                                             C.POINTER(vp), vp, i64, i64, f32c, vp]),
    "hnr_img_sum_views": (C.c_int, [vp, i64, i64, i64, vp, i64, vp]),
    "hnr_chain_bwd_f16": (C.c_int, [C.c_int, C.POINTER(i64), C.POINTER(i64), i64, C.c_int, vp, i64, vp, i64, C.POINTER(vp), C.POINTER(vp), vp,
                                    C.POINTER(i64), vp, i64, i64, vp]),
    "hnr_train_loss": (C.c_int, [vp, vp, vp, i64, vp, i64, f32c, f32c, vp, vp, vp, vp, vp]),
    "hnr_pyramid_fwd": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64, i64, i64, vp]),
    "hnr_pyramid_bwd": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64, i64, i64, vp]),
    "hnr_pack_job_bytes": (i64, []),
    "hnr_bias_job_bytes": (i64, []),
    "hnr_pack_weights": (C.c_int, [vp, i64, i64, vp, i64, vp, vp]),
    "hnr_nbr_features_bwd_ld": (C.c_int, [vp, i64] + [vp] * 7 + [i64, i64, vp, vp, vp, vp]),
}

EXPORTED = sorted(_SIGS)


def lib():
    """Return the loaded library, loading it on first use.  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)       # AttributeError if the symbol is missing -> loud
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().hnr_last_error().decode()
        raise RuntimeError(f"libhnr {what} failed ({code}): {msg}")


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream():
    """raw handle of torch's current stream on the current device.  torch.cuda.current_stream() builds a Stream object through several
    Python layers (~20 us; ~60 launches per training step): the raw-stream accessor is ~50x cheaper"""
    if _RAW_STREAM is not None:
        return C.c_void_p(_RAW_STREAM(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("hybridneuralrendering_b200: tensors must live on a CUDA device (no CPU fallback)")


def ptr_array(ts: Sequence[Optional[torch.Tensor]]):
    arr = (vp * len(ts))()
    for i, t in enumerate(ts):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


def i64_array(vals: Sequence[int]):
    return (i64 * len(vals))(*[int(v) for v in vals])
