"""ctypes binding of libnuhtc_b200.so (the C ABI declared in include/nuhtc_b200.h).

There is no fallback: if the shared library is missing or a call fails, the op raises.
Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C nuhtc_b200/csrc``.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnuhtc_b200.so")

# constants of include/nuhtc_b200.h
LAYOUT_NCHW, LAYOUT_NHWC, LAYOUT_CG32 = 0, 1, 2
ROI_ROUTE, ROI_SUM = 0, 1
IMPL_AUTO, IMPL_DIRECT = 0, 1
NMS_AGNOSTIC, NMS_OFFSET, NMS_PERCLASS, NMS_PERCLASS_RAW = 0, 1, 2, 3
PASTE_PROB, PASTE_BIN, PASTE_BITS = 0, 1, 2
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
MAX_LEVELS = 8

_c = ctypes
_vp, _i, _i64, _f, _d, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_double, _c.c_size_t

# name -> (restype, argtypes); the not-gpu test-suite checks every name is exported
SIGNATURES = {
    "nuhtc_abi_version": (_i, []),
    "nuhtc_last_error": (_c.c_char_p, []),
    "nuhtc_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "nuhtc_roi_align_fwd": (_i, [_c.POINTER(_vp), _c.POINTER(_i), _c.POINTER(_i), _c.POINTER(_f), _i, _i, _i, _i, _vp, _i,
                                 _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp]),
    "nuhtc_to_cg32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "nuhtc_roi_align_workspace_bytes": (_sz, [_c.POINTER(_i), _c.POINTER(_i), _i, _i, _i, _i, _i]),
    "nuhtc_roi_align_cg32": (_i, [_c.POINTER(_vp), _c.POINTER(_i), _c.POINTER(_i), _c.POINTER(_f), _i, _i, _i, _vp, _i, _i, _i, _i,
                                  _i, _i, _f, _c.POINTER(_i), _vp, _vp, _vp, _sz, _vp]),
    "nuhtc_to_cg32_dt": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "nuhtc_roi_align_cg32_dt": (_i, [_c.POINTER(_vp), _c.POINTER(_i), _c.POINTER(_i), _c.POINTER(_f), _i, _i, _i, _vp, _i, _i, _i,
                                     _i, _i, _i, _f, _c.POINTER(_i), _vp, _i, _vp, _vp, _sz, _vp]),
    "nuhtc_attention_pool_workspace_bytes": (_sz, [_i, _i]),
    "nuhtc_attention_pool": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "nuhtc_nms_workspace_bytes": (_sz, [_i64, _i, _i64, _i]),
    "nuhtc_nms": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i64, _f, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nuhtc_paste_masks": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp, _vp]),
    "nuhtc_paste_masks_dense_bits": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _vp]),
    "nuhtc_pack_masks": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "nuhtc_mask_nms_workspace_bytes": (_sz, [_i, _i, _i]),
    "nuhtc_mask_nms": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _d, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nuhtc_merge_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "nuhtc_merge": (_i, [_vp, _vp, _vp, _i64, _i64, _d, _i, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nuhtc_merge_graph": (_i, [_vp, _vp, _vp, _i64, _i64, _d, _i64, _vp, _vp, _vp, _c.POINTER(_i64), _vp, _vp, _sz, _vp]),
    "nuhtc_merge_rounds": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _i, _vp]),
    "nuhtc_mask_contours": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "nuhtc_contour_rings": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _vp, _vp]),
    "nuhtc_delta2bbox": (_i, [_vp, _i, _vp, _i64, _c.POINTER(_f * 4), _c.POINTER(_f * 4), _i, _i, _d, _f, _vp, _vp]),
    "nuhtc_multiclass_candidates": (_i, [_vp, _i, _vp, _i, _vp, _i, _i64, _i, _f, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nuhtc_detection_slots": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nuhtc_tile_filter": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "nuhtc_rpn_topk_supported": (_i, [_vp, _vp, _i, _i, _i]),
    "nuhtc_rpn_topk_decode": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _d, _f, _vp, _vp, _vp, _vp, _vp]),
    "nuhtc_mask_components_workspace_bytes": (_c.c_size_t, [_i, _i, _i]),
    "nuhtc_mask_components": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _c.c_size_t, _vp]),
    "nuhtc_ring_yextent": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "nuhtc_keep_flags": (_i, [_vp, _vp, _vp, _i, _i, _i64, _vp, _vp]),
    "nuhtc_preprocess_tiles": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _c.POINTER(_f * 3), _c.POINTER(_f * 3), _vp, _vp]),
}

_lib = None


class NuhtcError(RuntimeError):
    pass


def lib():
    """The loaded library.  Raises loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NuhtcError(
                f"{LIB_PATH} is missing: the CUDA library has not been built "
                "(run `make -C nuhtc_b200/csrc` or `__graft_entry__.build()`). There is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().nuhtc_last_error()
        raise NuhtcError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


# element types the RoIAlign path takes natively (include/nuhtc_b200.h NUHTC_DTYPE_*)
DTYPE_CODES = {torch.float32: DTYPE_F32, torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16}


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise NuhtcError(f"{name} must be a CUDA tensor: nuhtc_b200 ops run on the GPU only (no CPU fallback)")


# ---- launch accounting: how many of OUR kernels each C-ABI call enqueues (bench.py reports the sum as
# "gpu_launches"; library kernels such as cub's radix sort are not counted)
LAUNCHES = {"n": 0}
KERNELS_PER_CALL = {"nchw_to_nhwc": 1, "to_cg32": 1, "roi_align_strip": 5, "attention_pool": 4, "roi_align": 1, "nms": 9, "paste": 2, "paste_dual": 1, "pack": 3, "mask_nms": 8, "merge": 16, "contours": 2, "rings": 1, "glue": 1, "rpn_topk": 1, "components": 8, "preprocess": 1}


def count(op: str, n: int = 1) -> None:
    LAUNCHES["n"] += KERNELS_PER_CALL[op] * n
