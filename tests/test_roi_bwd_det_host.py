"""CPU: the deterministic RoIAlignRotated backward (include/rsdet.h) without a GPU.

The workspace query is host-only and returns 0 outside the contract (adaptive sampling grid, bad dtypes, the entry and
pixel limits); the entry point reports argument errors before it launches anything, so these calls carry null or
dummy device pointers and no CUDA call is made; `core.roi_align_rotated_backward(..., deterministic=True)` rejects what
the atomic call rejects."""
import ctypes

import pytest
import torch

F32, F16, BF16 = 0, 1, 2
EINVAL, ELIMIT = -1, -3
PYRAMID = [(1, 256, 256, 256), (1, 256, 128, 128), (1, 256, 64, 64), (1, 256, 32, 32)]


def _cfg(shapes=PYRAMID, channels_last=False, out=7, sr=2):
    from rs_detection_b200 import core
    return core.make_roi_cfg(shapes, [1 / 4, 1 / 8, 1 / 16, 1 / 32][:len(shapes)], out, sr, 1, (1.4, 1.2),
                             channels_last=channels_last)


def _lib():
    from rs_detection_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_workspace_query(channels_last):
    L = _lib()
    cfg = _cfg(channels_last=channels_last)
    c = ctypes.byref(cfg)
    q = L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes
    pixels = sum(s[2] * s[3] for s in PYRAMID)
    for K in (0, 1, 512, 4096):
        entries = K * 49 * 4 * 4
        for dt in (F32, F16, BF16):
            b = q(c, K, dt)
            # keys and entry indices twice, weights, the bin-major grad_out
            assert b >= 5 * 4 * entries + 4 * K * 49 * 256
            if not channels_last:       # fp32 channels-last accumulators
                assert b >= 4 * pixels * 256
        assert q(c, K, F16) == q(c, K, F32) == q(c, K, BF16)
    assert q(c, 4096, F32) > q(c, 512, F32) > q(c, 1, F32)
    other = q(ctypes.byref(_cfg(channels_last=not channels_last)), 512, F32)
    assert (other > q(c, 512, F32)) == channels_last      # the NCHW call needs the accumulators


def test_workspace_query_returns_zero_outside_the_contract():
    L = _lib()
    q = L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes
    cfg = _cfg()
    c = ctypes.byref(cfg)
    assert q(c, 100, 3) == 0 and q(c, 100, -1) == 0                         # dtypes
    assert q(c, -1, F32) == 0
    for sr in (0, -1):                                                      # adaptive grid
        assert q(ctypes.byref(_cfg(sr=sr)), 100, F32) == 0
    # entry limit: K * 7 * 7 * 2^2 * 4 <= 2^28
    k_max = (1 << 28) // (49 * 16)
    assert q(c, k_max, F32) > 0 and q(c, k_max + 1, F32) == 0
    big = _cfg(out=64, sr=16)                                               # one RoI = 2^22 entries
    assert q(ctypes.byref(big), 64, F32) > 0 and q(ctypes.byref(big), 65, F32) == 0
    assert q(ctypes.byref(_cfg(out=(1 << 14, 1 << 14), sr=1)), 1, F32) == 0  # one RoI above the limit
    # pixel limit: the keys are 32-bit
    huge = _cfg([(1 << 16, 4, 256, 256)], sr=1)
    assert q(ctypes.byref(huge), 1, F32) == 0
    assert q(ctypes.byref(_cfg([(16, 4, 256, 256)], sr=1)), 1, F32) > 0
    bad = _cfg()
    bad.num_levels = 0
    assert q(ctypes.byref(bad), 100, F32) == 0


def test_entry_point_rejects_before_any_launch():
    """Real sizes and dummy device pointers: only the argument checks may stop these calls, and they must (no CUDA call
    is made on this machine)."""
    L = _lib()
    f = L.rsdet_roi_align_rotated_backward_deterministic
    cfg = _cfg()
    c = ctypes.byref(cfg)
    maps = (ctypes.c_void_p * 8)(*([8] * 4 + [0] * 4))
    big_ws = 1 << 40
    for gdt, fdt in [(F32, 3), (F16, BF16), (BF16, F32), (9, F16), (F32, -1)]:
        assert f(c, gdt, 8, 8, 100, fdt, maps, 8, big_ws, None) == EINVAL, (gdt, fdt)
    for sr in (0, -2):
        assert f(ctypes.byref(_cfg(sr=sr)), F32, 8, 8, 100, F32, maps, 8, big_ws, None) == EINVAL
    assert f(c, F32, 8, 8, -1, F32, maps, 8, big_ws, None) == EINVAL
    assert f(None, F32, 8, 8, 100, F32, maps, 8, big_ws, None) == EINVAL
    assert f(c, F32, 8, 8, 100, F32, None, 8, big_ws, None) == EINVAL
    holes = (ctypes.c_void_p * 8)(*([8, 8, 0, 8] + [0] * 4))
    assert f(c, F32, 8, 8, 100, F32, holes, 8, big_ws, None) == EINVAL
    assert f(c, F32, None, 8, 100, F32, maps, 8, big_ws, None) == EINVAL    # null grad_out
    assert f(c, F32, 8, None, 100, F32, maps, 8, big_ws, None) == EINVAL    # null rois
    k_max = (1 << 28) // (49 * 16)
    assert f(c, F32, 8, 8, k_max + 1, F32, maps, 8, big_ws, None) == ELIMIT
    assert f(ctypes.byref(_cfg([(1 << 16, 4, 256, 256)], sr=1)), F32, 8, 8, 1, F32, maps, 8, big_ws, None) == ELIMIT
    # a workspace smaller than the query
    need = L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(c, 100, F32)
    assert f(c, F32, 8, 8, 100, F32, maps, 8, need - 1, None) == -2


@pytest.mark.parametrize("deterministic", [False, True])
def test_core_rejects_the_same_inputs(deterministic):
    from rs_detection_b200 import core
    cfg = _cfg(PYRAMID[:2])
    rois = torch.zeros((3, 6))
    with pytest.raises(ValueError, match="float32, float16 or bfloat16"):
        core.roi_align_rotated_backward(cfg, torch.zeros((3, 256, 7, 7)), rois, PYRAMID[:2], feat_dtype=torch.float64,
                                        deterministic=deterministic)
    with pytest.raises(RuntimeError, match="CUDA"):          # no CPU fallback on either path
        core.roi_align_rotated_backward(cfg, torch.zeros((3, 256, 7, 7)), rois, PYRAMID[:2], deterministic=deterministic)
