"""CPU: the layout bits of `rsdet_roi_align_cfg.channels_last` (RSDET_ROI_NHWC_MAPS, RSDET_ROI_NHWC_ROIS) without a GPU.

Workspace sizes per flag value, bits outside the two that must be rejected before anything is launched, and the
`memory_format` argument of the jdet mirror's RoIAlignRotated layers."""
import ctypes

import pytest
import torch

F32, F16, BF16 = 0, 1, 2
MAPS, ROIS = 1, 2
PYRAMID = [(1, 256, 256, 256), (1, 256, 128, 128), (1, 256, 64, 64), (1, 256, 32, 32)]


def _cfg(flags=0, out=7, sr=2):
    from rs_detection_b200 import core
    cfg = core.make_roi_cfg(PYRAMID, [1 / 4, 1 / 8, 1 / 16, 1 / 32], out, sr, 1, (1.4, 1.2))
    cfg.channels_last = flags
    return cfg


def _align256(n):
    return (n + 255) // 256 * 256


def test_header_and_binding_agree_on_the_bits():
    from rs_detection_b200 import _lib
    assert (_lib.ROI_NHWC_MAPS, _lib.ROI_NHWC_ROIS) == (MAPS, ROIS)
    import os
    src = open(os.path.join(os.path.dirname(_lib.__file__), "..", "include", "rsdet.h")).read()
    assert "#define RSDET_ROI_NHWC_MAPS 1" in src and "#define RSDET_ROI_NHWC_ROIS 2" in src


@pytest.mark.parametrize("shape", [(7, 2), (5, 2), (7, 0)], ids=["fwd77", "fwd5x5", "generic"])
def test_atomic_workspace_ignores_the_roi_layout(shape):
    """The forward and the atomic backward read out / grad_out in place in either layout: only the maps bit counts."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    for K in (0, 1, 4000):
        for bwd in (0, 1):
            for dt in (F32, F16, BF16):
                q = {f: L.rsdet_roi_align_rotated_workspace_bytes_typed(ctypes.byref(_cfg(f, *shape)), K, bwd, dt)
                     for f in (0, 1, 2, 3)}
                assert q[0] > 0 and q[1] > 0
                assert q[2] == q[0] and q[3] == q[1], (K, bwd, dt, q)
            assert L.rsdet_roi_align_rotated_workspace_bytes(ctypes.byref(_cfg(2, *shape)), K, bwd) == \
                L.rsdet_roi_align_rotated_workspace_bytes(ctypes.byref(_cfg(0, *shape)), K, bwd)


@pytest.mark.parametrize("out,sr,channels", [(7, 2, 256), (5, 3, 260)])
def test_deterministic_workspace_drops_the_bin_major_copy_for_fp32(out, sr, channels):
    """An NHWC fp32 grad_out is the bin-major array the deterministic gather reads: no copy, no workspace for it.  The
    query does not know a half call's grad_out dtype, so half maps keep the fp32 copy reserved."""
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    shapes = [(1, channels) + s[2:] for s in PYRAMID]
    for K in (1, 600, 4000):
        copy = _align256(4 * K * out * out * channels)
        for maps in (0, MAPS):
            q = {}
            for f in (maps, maps | ROIS):
                cfg = core.make_roi_cfg(shapes, [1 / 4, 1 / 8, 1 / 16, 1 / 32], out, sr, 1, (1.4, 1.2))
                cfg.channels_last = f
                q[f] = {dt: L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(ctypes.byref(cfg), K, dt)
                        for dt in (F32, F16, BF16)}
            assert all(v > 0 for d in q.values() for v in d.values())
            assert q[maps][F32] - q[maps | ROIS][F32] == copy, (K, maps)
            assert q[maps | ROIS][F16] == q[maps][F16] and q[maps | ROIS][BF16] == q[maps][BF16]


@pytest.mark.parametrize("flags", [4, 5, 7, 8, 1 << 30, -1, -2])
def test_other_bits_are_rejected_before_any_launch(flags):
    """Values that set a bit other than the two layout bits: every workspace query returns 0 and every entry point
    RSDET_EINVAL.  The calls carry real sizes and non-null fake device pointers, so only the flag check may stop them
    (no CUDA call is made on this machine)."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    c = ctypes.byref(_cfg(flags))
    for dt in (F32, F16, BF16):
        for bwd in (0, 1):
            assert L.rsdet_roi_align_rotated_workspace_bytes_typed(c, 100, bwd, dt) == 0
        assert L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(c, 100, dt) == 0
    assert L.rsdet_roi_align_rotated_workspace_bytes(c, 100, 0) == 0
    feats = (ctypes.c_void_p * 8)(*([256] * 4 + [0] * 4))
    assert L.rsdet_roi_align_rotated_forward(c, feats, 256, 100, 256, None, 256, 1 << 30, None) == -1
    assert L.rsdet_roi_align_rotated_forward_typed(c, F16, feats, 256, 100, F16, 256, None, 256, 1 << 30, None) == -1
    assert L.rsdet_roi_align_rotated_backward(c, 256, 256, 100, feats, 256, 1 << 30, None) == -1
    assert L.rsdet_roi_align_rotated_backward_typed(c, F32, 256, 256, 100, F32, feats, 256, 1 << 30, None) == -1
    assert L.rsdet_roi_align_rotated_backward_deterministic(c, F32, 256, 256, 100, F32, feats, 256, 1 << 30, None) == -1


BAD_FORMATS = [torch.preserve_format, "channels_last", None, 1]


@pytest.mark.parametrize("bad", BAD_FORMATS, ids=[str(b) for b in BAD_FORMATS])
def test_bad_memory_format_raises_value_error(bad):
    from rs_detection_b200 import core
    from rs_detection_b200.jdet.ops import roi_align_rotated, roi_align_rotated_v1
    for cls in (roi_align_rotated_v1.ROIAlignRotated_v1, roi_align_rotated.ROIAlignRotated):
        with pytest.raises(ValueError, match="memory_format"):
            cls(7, 1 / 16, 2, memory_format=bad)
    feat, rois = torch.zeros((1, 256, 16, 16)), torch.zeros((3, 6))
    for fn in (roi_align_rotated_v1.roi_align, roi_align_rotated.roi_align):
        with pytest.raises(ValueError, match="memory_format"):
            fn(feat, rois, 7, 1 / 16, 2, memory_format=bad)
    with pytest.raises(ValueError, match="memory_format"):
        core.roi_align_rotated_forward(_cfg(), [torch.zeros(s) for s in PYRAMID], rois, memory_format=bad)


def test_memory_format_reaches_the_layers_and_repr():
    from rs_detection_b200.jdet.models.roi_extractors.oriented_single_level import OrientedSingleRoIExtractor
    from rs_detection_b200.jdet.models.roi_extractors.rbox_single_level import RboxSingleRoIExtractor
    from rs_detection_b200.jdet.ops.roi_align_rotated import ROIAlignRotated
    from rs_detection_b200.jdet.ops.roi_align_rotated_v1 import ROIAlignRotated_v1
    assert repr(ROIAlignRotated_v1(7, 0.25, 2)) == "ROIAlignRotated_v1(output_size=(7, 7), spatial_scale=0.25, sampling_ratio=2)"
    assert repr(ROIAlignRotated(7, 0.25)) == "ROIAlignRotated(output_size=(7, 7), spatial_scale=0.25, sampling_ratio=0)"
    assert ROIAlignRotated_v1(7, 0.25, 2).memory_format is torch.contiguous_format
    cl = ROIAlignRotated_v1(7, 0.25, 2, memory_format=torch.channels_last)
    assert repr(cl) == ("ROIAlignRotated_v1(output_size=(7, 7), spatial_scale=0.25, sampling_ratio=2, "
                        "memory_format=torch.channels_last)")
    ext = OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=2,
                                          memory_format=torch.channels_last), 256, [4, 8, 16, 32])
    assert all(l.memory_format is torch.channels_last for l in ext.roi_layers)
    rb = RboxSingleRoIExtractor(dict(type='ROIAlignRotated', output_size=7, sampling_ratio=2,
                                     memory_format=torch.channels_last), 256, [4, 8, 16, 32])
    assert all(l.memory_format is torch.channels_last for l in rb.roi_layers)
    with pytest.raises(ValueError, match="memory_format"):
        OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=2,
                                        memory_format=torch.preserve_format), 256, [4, 8, 16, 32])
