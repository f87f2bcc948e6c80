"""ctypes binding of libfrr.so (include/frr.h).  There is no CPU fallback: if the library is
missing or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os
import re
import threading

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
LIB_PATH = os.path.join(PKG, "libfrr.so")
HEADER = os.path.join(REPO, "include", "frr.h")

_lock = threading.Lock()
_lib = None

_p = C.c_void_p
_i = C.c_int
_f = C.c_float
_d = C.c_double

# name -> (restype, argtypes); mirrors include/frr.h one to one
SIGNATURES = {
    "frr_abi_version": (_i, []),
    "frr_last_error": (C.c_char_p, []),
    "frr_launch_count": (C.c_uint64, []),
    "frr_anchor_base_host": (_i, [_p, _i]),
    "frr_tv_anchor_base_host": (_i, [_f, _p, _i, _p]),
    "frr_anchors_pyramid": (_i, [_p, _i, _p, _p, _i, _i, _i, _p]),
    "frr_anchors": (_i, [_p, _i, _i, _i, _p, _i, _p]),
    "frr_rpn_decode": (_i, [_p, _p, _i, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p, _i, _i, _p]),
    "frr_topk_desc_opt": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _i, _p]),
    "frr_nms_sorted": (_i, [_p, _p, _i, _i, _d, _i, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p]),
    "frr_rpn_proposals_workspace_bytes": (C.c_size_t, [_i, _i, _i, _i]),
    "frr_rpn_proposals": (_i, [_p, _p, _i, _p, _p, _i, _i, _i, _p, _i, _f, _i, _i, _i, _i, _d, _p, _p, _p, C.c_size_t, _i,
                               _p]),
    "frr_nms_variant": (_i, [_i, _i, _d, _i, _i, _i, _i, _p]),
    "frr_rpn_proposals_workspace_layout": (_i, [_i, _i, _i, _i, _p]),
    "frr_nms_sorted_indirect": (_i, [_p, _i, _p, _p, _i, _i, _d, _i, _p, _p, _p, _i, _i, _p]),
    "frr_rois5": (_i, [_p, _p, _i, _i, _i, _i, _p, _i, _p, _p]),
    "frr_roi_pool_fwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _p, _i, _p, _p, _p]),
    "frr_roi_pool_bwd": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _p, _p]),
    "frr_roi_align_fwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _p, _p]),
    "frr_roi_align_bwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _p, _p]),
    "frr_roi_pool_bwd_deterministic": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _p, _i, _p, _p]),
    "frr_roi_align_bwd_deterministic": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _p, _p]),
    "frr_roi_variant": (_i, [_i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "frr_fpn_level_rois": (_i, [_p, _i, _i, _i, _i, _f, _i, _p, _p, _p]),
    "frr_region_loss": (_i, [_p, _p, _p, _p, _i, _i, _p, _p, _p, _p, _i, _i, _i, _f, _f, _p, _p, _p, _p, _p, _p]),
    "frr_sample_targets": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _i, _p, _p, _i, _p]),
    "frr_rpn_targets_assign": (_i, [_p, _p, _i, _i, _p, _p, _i, _i, _i, _p, _i, _i, _f, _f, _f, _i, _i, _p, _p, _p, _p, _p, _p,
                                    _p]),
    "frr_rpn_targets_finalize": (_i, [_p, _i, _i, _p, _p, _i, _i, _i, _p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "frr_frcnn_targets_assign": (_i, [_p, _p, _i, _i, _p, _p, _i, _f, _f, _p, _p, _p, _p, _p, _p, _p]),
    "frr_frcnn_targets_finalize": (_i, [_p, _p, _i, _i, _p, _p, _i, _p, _p, _p, _p, _p, _i, _p, _i, _p, _p, _p, _p, _p]),
    "frr_decode_classwise": (_i, [_p, _p, _p, _i, _i, _p, _p, _p, _p]),
    "frr_pack_detections": (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _i, _p, _p, _p]),
    "frr_pack_detections_ranked_workspace_bytes": (C.c_size_t, [_i, _i, _i]),
    "frr_pack_detections_ranked": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _p, _p, _p, C.c_size_t, _p]),
    "frr_class_nms_workspace_bytes": (C.c_size_t, [_i, _i, _i]),
    "frr_class_nms": (_i, [_p, _p, _p, _i, _i, _i, _f, _d, _i, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    # mixed-size batch: per-image sizes image_hw [B,2] on the device
    "frr_rpn_decode_sized": (_i, [_p, _p, _i, _p, _i, _p, _i, _i, _i, _f, _p, _p, _p, _i, _i, _p]),
}


class FrrError(RuntimeError):
    pass


def declared_symbols() -> list[str]:
    """Entry points declared in include/frr.h."""
    with open(HEADER) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(frr_[a-z0-9_]+)\s*\(", text)))


def load():
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise FrrError(
                f"{LIB_PATH} is missing: build it with `python -m faster_rcnn_pytorch_b200.build` "
                "(there is no CPU fallback for the region stage)")
        # libfrr.so links the CUDA runtime dynamically (no second, static copy inside the library): torch has already
        # loaded its libcudart.so.12 into the process, and the loader resolves the NEEDED entry to that copy
        import torch  # noqa: F401
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.frr_abi_version() != 3:
            raise FrrError("libfrr.so ABI version mismatch")
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().frr_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise FrrError(f"{what} failed ({rc}): {msg}")


def launch_count() -> int:
    return int(load().frr_launch_count())
