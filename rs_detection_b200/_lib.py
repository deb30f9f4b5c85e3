"""ctypes binding of librsdet.so (include/rsdet.h) + the small amount of torch plumbing the host
side needs (device buffers, current stream, a cached workspace).

There is no CPU fallback: if the shared library is missing, or an op is called without a CUDA
device, this module raises.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librsdet.so")

NMS_ROTATED, NMS_ROTATED_GE, NMS_POLY, NMS_MERGE, NMS_HBB, NMS_HBB_P1, NMS_HBB_P1_F64 = 0, 1, 2, 3, 4, 5, 6
MAX_LEVELS = 8

_vp = C.c_void_p


class RoiAlignCfg(C.Structure):
    _fields_ = [("num_levels", C.c_int), ("batch", C.c_int), ("channels", C.c_int),
                ("height", C.c_int * MAX_LEVELS), ("width", C.c_int * MAX_LEVELS),
                ("spatial_scale", C.c_float * MAX_LEVELS),
                ("pooled_h", C.c_int), ("pooled_w", C.c_int), ("sampling_ratio", C.c_int), ("version", C.c_int),
                ("extend_w", C.c_float), ("extend_h", C.c_float), ("finest_scale", C.c_float),
                ("channels_last", C.c_int)]


class RpnCfg(C.Structure):
    _fields_ = [("num_levels", C.c_int), ("height", C.c_int * MAX_LEVELS), ("width", C.c_int * MAX_LEVELS),
                ("num_anchors", C.c_int), ("use_sigmoid", C.c_int), ("nms_pre", C.c_int), ("nms_post", C.c_int),
                ("nms_thresh", C.c_double), ("min_bbox_size", C.c_float), ("means", C.c_float * 6), ("stds", C.c_float * 6),
                ("wh_ratio_clip", C.c_float)]


# name -> (restype, argtypes); every symbol include/rsdet.h declares
SIGNATURES = {
    "rsdet_version": (C.c_int, []),
    "rsdet_error_string": (C.c_char_p, [C.c_int]),
    "rsdet_launch_count": (C.c_ulonglong, []),
    "rsdet_obb2poly": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "rsdet_obb2hbb": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "rsdet_poly2hbb": (C.c_int, [_vp, C.c_int, C.c_int, _vp, _vp]),
    "rsdet_poly2origpoly": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    "rsdet_iou_poly_pairs": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp]),
    "rsdet_box_iou_rotated_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "rsdet_box_iou_rotated": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_size_t, _vp]),
    "rsdet_assign_workspace_bytes": (C.c_size_t, [C.c_int]),
    "rsdet_assign_wrt_overlaps": (C.c_int, [_vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int,
                                            C.c_int, _vp, C.c_int32, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "rsdet_nms_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "rsdet_nms": (C.c_int, [C.c_int, _vp, _vp, _vp, C.c_int, C.c_double, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp,
                            C.c_size_t, _vp]),
    "rsdet_multiclass_nms_rotated_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "rsdet_multiclass_nms_rotated": (C.c_int, [_vp, C.c_int, _vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, _vp,
                                               _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "rsdet_roi_align_rotated_workspace_bytes": (C.c_size_t, [C.POINTER(RoiAlignCfg), C.c_int, C.c_int]),
    "rsdet_roi_align_rotated_forward": (C.c_int, [C.POINTER(RoiAlignCfg), C.POINTER(_vp), _vp, C.c_int, _vp, _vp, _vp,
                                                  C.c_size_t, _vp]),
    "rsdet_roi_align_rotated_backward": (C.c_int, [C.POINTER(RoiAlignCfg), _vp, _vp, C.c_int, C.POINTER(_vp), _vp,
                                                   C.c_size_t, _vp]),
    "rsdet_oriented_head_results_workspace_bytes": (C.c_size_t, [C.c_int]),
    "rsdet_oriented_head_results": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                              C.c_float, C.POINTER(C.c_float), C.c_float, C.c_int, _vp, _vp, _vp, _vp, C.c_size_t,
                                              _vp]),
    "rsdet_voc_match": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int, C.c_int, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rsdet_rpn_num_candidates": (C.c_int, [C.POINTER(RpnCfg)]),
    "rsdet_rpn_proposals_workspace_bytes": (C.c_size_t, [C.POINTER(RpnCfg)]),
    "rsdet_rpn_proposals": (C.c_int, [C.POINTER(RpnCfg), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _vp, _vp, _vp,
                                      _vp, _vp, C.c_size_t, _vp]),
    "rsdet_roi_align_profile_events": (C.c_int, [_vp, _vp]),
    "rsdet_nchw_to_nhwc": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    "rsdet_nhwc_to_nchw": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
}

_lib = None


def load():
    """Load librsdet.so; raise (never fall back) if it is missing or incomplete."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m rs_detection_b200.build` "
                               "(there is no CPU / PyTorch fallback for the rotated-box ops)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str):
    if rc == 0:
        return
    msg = load().rsdet_error_string(rc).decode()
    if rc == -1:
        raise ValueError(f"{what}: {msg}")
    raise RuntimeError(f"{what}: {msg} (code {rc})")


def launch_count() -> int:
    return int(load().rsdet_launch_count())


# ------------------------------------------------------------------------------- torch plumbing
def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("rs_detection_b200 ops need a CUDA device (sm_100a); there is no CPU fallback")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


_workspaces: dict = {}
# A CUDA graph keeps the raw address of every scratch buffer it was captured with, so a buffer handed out while a graph
# was being captured must never go back to the caching allocator: every replay would write into whatever tensor the
# allocator placed there next.  `_graph_held` names the keys whose current buffer a capture used; when such a buffer is
# replaced (growth) or released it moves to `_retired`, which lives as long as the process.  Sizes grow by more than
# 1.25x per replacement, so growth alone retires at most 4x the live buffer of a key; each release_workspaces() after a
# capture retires one more buffer per key that capture used.
_graph_held: set = set()
_retired: list = []


def workspace(nbytes: int, tag: str = "default") -> torch.Tensor:
    """Cached per-(device, stream, tag) scratch buffer, grown geometrically; contents are undefined.
    Keyed by the current stream so that tiles processed on different streams never share scratch.
    A buffer handed out during a CUDA-graph capture stays alive for the rest of the process."""
    dev = torch.cuda.current_device()
    key = (dev, torch.cuda.current_stream().cuda_stream, tag)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        if key in _graph_held:
            _retired.append(buf)
            _graph_held.discard(key)
        size = max(int(nbytes * 1.25) + 4096, 1 << 20)
        buf = torch.empty(size, dtype=torch.uint8, device=f"cuda:{dev}")
        _workspaces[key] = buf
    if torch.cuda.is_current_stream_capturing():
        _graph_held.add(key)
    return buf


def release_workspaces():
    """Drop the cached scratch buffers, except those a captured CUDA graph still uses (they are retired, not freed)."""
    _retired.extend(_workspaces[k] for k in _graph_held if k in _workspaces)
    _graph_held.clear()
    _workspaces.clear()


def to_device(x, dtype):
    """torch CUDA tensor (contiguous, dtype) from a torch tensor or numpy array; second value tells
    whether the caller passed HOST data (then results are returned as numpy)."""
    require_cuda()
    if isinstance(x, torch.Tensor):
        host = not x.is_cuda
        t = x.to(device="cuda", dtype=dtype, non_blocking=True).contiguous()
        return t, host
    a = np.ascontiguousarray(x)
    t = torch.from_numpy(a).to(device="cuda", non_blocking=True).to(dtype).contiguous()
    return t, True


def from_device(t, host: bool, like=None):
    if not host:
        return t
    if isinstance(like, torch.Tensor):
        return t.cpu()
    return t.cpu().numpy()
