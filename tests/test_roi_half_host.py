"""CPU: the half-precision RoIAlignRotated entry points (include/rsdet.h, RSDET_DTYPE_*) without a GPU.

Workspace sizes, argument errors that must be reported before anything is launched, the mixed-dtype rule of
`core.roi_align_rotated_forward`, and the float16 `jt.code` bodies of the Jittor adapter compiled for sm_100a against the
stub executor.h and the real header (the way tests/test_jittor_adapter.py checks the fp32 bodies)."""
import ctypes
import os
import subprocess

import pytest
import torch

from test_jittor_adapter import NVCC, ROOT, V, _wrap, fake_jt  # noqa: F401  (fake_jt is a fixture)

F32, F16, BF16 = 0, 1, 2
PYRAMID = [(1, 256, 256, 256), (1, 256, 128, 128), (1, 256, 64, 64), (1, 256, 32, 32)]


def _cfg(shapes=PYRAMID, channels_last=False, out=7, sr=2):
    from rs_detection_b200 import core
    return core.make_roi_cfg(shapes, [1 / 4, 1 / 8, 1 / 16, 1 / 32][:len(shapes)], out, sr, 1, (1.4, 1.2),
                             channels_last=channels_last)


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("shape", [(7, 2), (5, 2), (7, 0)], ids=["fwd77", "fwd5x5", "generic"])
def test_typed_workspace_query(channels_last, shape):
    from rs_detection_b200 import _lib
    L = _lib.load()
    cfg = _cfg(channels_last=channels_last, out=shape[0], sr=shape[1])
    c = ctypes.byref(cfg)
    pixels = sum(s[2] * s[3] for s in PYRAMID) * 256
    for K in (0, 1, 4000):
        for bwd in (0, 1):
            assert L.rsdet_roi_align_rotated_workspace_bytes_typed(c, K, bwd, F32) == \
                L.rsdet_roi_align_rotated_workspace_bytes(c, K, bwd)
        fast_nchw = not channels_last and shape[1] > 0
        f32, f16, bf16 = (L.rsdet_roi_align_rotated_workspace_bytes_typed(c, K, 0, d) for d in (F32, F16, BF16))
        assert f16 == bf16
        if fast_nchw:       # the NHWC copy of the pyramid halves
            assert f16 < f32 and f32 - f16 >= pixels * 2
        else:
            assert f16 == f32
        # half gradient maps: fp32 accumulators on every path
        b32, b16 = (L.rsdet_roi_align_rotated_workspace_bytes_typed(c, K, 1, d) for d in (F32, F16))
        assert b16 >= pixels * 4 and (b16 == b32 if fast_nchw else b16 - b32 >= pixels * 4)


def test_bad_dtypes_are_rejected_before_any_launch():
    """These calls carry real sizes and null device pointers: only the dtype check may stop them, and it must come first
    (no CUDA call is made on this machine)."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    cfg = _cfg()
    c = ctypes.byref(cfg)
    feats = (ctypes.c_void_p * 8)(*([8] * 4 + [0] * 4))
    assert L.rsdet_roi_align_rotated_workspace_bytes_typed(c, 100, 0, 3) == 0
    assert L.rsdet_roi_align_rotated_workspace_bytes_typed(c, 100, 1, -1) == 0
    fwd = L.rsdet_roi_align_rotated_forward_typed
    for fdt, odt in [(3, F32), (-1, F32), (F16, BF16), (BF16, F16), (F32, F16), (F16, 7)]:
        assert fwd(c, fdt, feats, 8, 100, odt, 8, None, 8, 1 << 30, None) == -1, (fdt, odt)
    bwd = L.rsdet_roi_align_rotated_backward_typed
    for gdt, fdt in [(F32, 3), (F16, BF16), (BF16, F32), (9, F16)]:
        assert bwd(c, gdt, 8, 8, 100, fdt, feats, 8, 1 << 30, None) == -1, (gdt, fdt)


def test_core_rejects_mixed_half_levels():
    from rs_detection_b200 import core
    cfg = _cfg(PYRAMID[:2])
    rois = torch.zeros((3, 6))
    mixed = [torch.zeros(PYRAMID[0], dtype=torch.bfloat16), torch.zeros(PYRAMID[1], dtype=torch.float32)]
    with pytest.raises(ValueError, match="mix"):
        core.roi_align_rotated_forward(cfg, mixed, rois)
    two_halves = [torch.zeros(PYRAMID[0], dtype=torch.bfloat16), torch.zeros(PYRAMID[1], dtype=torch.float16)]
    with pytest.raises(ValueError, match="mix"):
        core.roi_align_rotated_forward(cfg, two_halves, rois)
    with pytest.raises(ValueError, match="float32, float16 or bfloat16"):
        core.roi_align_rotated_backward(cfg, torch.zeros((3, 256, 7, 7)), rois, PYRAMID[:2], feat_dtype=torch.float64)


def test_core_checks_out_dtype():
    from rs_detection_b200 import core
    cfg = _cfg(PYRAMID[:1])
    feats = [torch.zeros(PYRAMID[0], dtype=torch.float16)]
    with pytest.raises(ValueError, match="out_dtype"):
        core.roi_align_rotated_forward(cfg, feats, torch.zeros((3, 6)), out_dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="out has dtype"):
        core.roi_align_rotated_forward(cfg, feats, torch.zeros((3, 6)), out=torch.zeros((3, 256, 7, 7)),
                                       out_dtype=torch.float16)


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_float16_jt_code_bodies_compile_against_rsdet_h(fake_jt, tmp_path):
    from rs_detection_b200 import jittor_adapter as A
    h = lambda *s: V(s, "float16")
    for version in (0, 1):
        A.make_roi_align(version).apply(h(2, 256, 64, 64), V((30, 6)), (7, 7), 1 / 16., 2)
    A.make_roi_align(1).apply(h(2, 256, 64, 64), V((30, 6), "float16"), (7, 7), 1 / 16., 2)      # rois cast to fp32
    fused = A.make_fused_extractor(1)
    fused.apply(h(1, 256, 256, 256), h(1, 256, 128, 128), h(1, 256, 64, 64), h(1, 256, 32, 32), V((4000, 6)),
                [4, 8, 16, 32], 7, 2, (1.4, 1.2), 56)
    with pytest.raises(ValueError, match="mix"):
        fused.apply(h(1, 256, 64, 64), V((1, 256, 32, 32)), V((30, 6)), [16, 32], 7, 2, (1.4, 1.2), 56)
    recs = [r for r in fake_jt if "_typed" in r["src"]]
    assert len(recs) == 8 and all(r["outs"][0][1] == "float16" for r in recs)
    assert all("(const float*)in" in r["src"] for r in recs)
    # the float16 gradient of a float16 output goes in as RSDET_DTYPE_F16
    assert all("backward_typed(&cfg, RSDET_DTYPE_F16" in r["src"] for r in recs if "backward" in r["src"])
    src = tmp_path / "adapter_half_ops.cu"
    body = recs[0]["header"] + "\nnamespace jittor { Executor exe; }\n"
    for i, r in enumerate(recs):
        # Jittor declares a float16 Var's pointer with its own 2-byte type: a distinct type here
        w = _wrap(i, dict(r, header=""))
        for k, v in enumerate(r["ins"]):
            if v.dtype == "float16":
                w = w.replace(f"  float* in{k}_p = nullptr;", f"  jt_half* in{k}_p = nullptr;")
        for k, (_, dt) in enumerate(r["outs"]):
            if dt == "float16":
                w = w.replace(f"  float* out{k}_p = nullptr;", f"  jt_half* out{k}_p = nullptr;")
        assert "jt_half* in0_p" in w
        body += w
    src.write_text(body.replace("namespace jittor { Executor exe; }",
                                "namespace jittor { Executor exe; }\nstruct jt_half { unsigned short x; };", 1))
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-c", str(src), "-o", str(tmp_path / "h.o"),
           "-I", os.path.join(ROOT, "tests", "jittor_stub"), "-Wno-deprecated-gpu-targets"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-4000:]
