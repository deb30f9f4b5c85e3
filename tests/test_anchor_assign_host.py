"""CPU: the horizontal IoU (BboxOverlaps2D) and the fused anchor assignment (rsdet_bbox_overlaps, rsdet_assign_hbb)
without a GPU.

The test oracle's bbox_overlaps (tests/hbb_oracle.py) is checked against a scalar float32 evaluation of the formula in include/rsdet.h; the
workspace query is host-only and returns 0 outside the contract; the entry points report argument errors before they
launch anything, so these calls carry null or dummy device pointers and no CUDA call is made; the mirror rejects what
the calculator does not implement; the Jittor adapter's new bodies compile against rsdet.h."""
import os
import subprocess

import numpy as np
import pytest
import torch

from hbb_oracle import bbox_overlaps
from test_jittor_adapter import NVCC, ROOT, V, _wrap, fake_jt  # noqa: F401  (fake_jt is a fixture)

EINVAL, EWORKSPACE, ELIMIT = -1, -2, -3
MAX_GTS, MAX_ANCHORS = 1 << 24, 1 << 30
f = np.float32


def _lib():
    from rs_detection_b200 import _lib
    return _lib.load()


def _iou_scalar(a, b):
    """The formula of include/rsdet.h, one numpy float32 scalar operation at a time."""
    area_a = (f(a[2]) - f(a[0])) * (f(a[3]) - f(a[1]))
    area_b = (f(b[2]) - f(b[0])) * (f(b[3]) - f(b[1]))
    w = max(min(f(a[2]), f(b[2])) - max(f(a[0]), f(b[0])), f(0))
    h = max(min(f(a[3]), f(b[3])) - max(f(a[1]), f(b[1])), f(0))
    overlap = f(w * h)
    union = max(f(f(area_a + area_b) - overlap), f(1e-6))
    return f(overlap / union)


def _edge_boxes():
    base = np.array([10, 20, 50, 60], np.float32)
    return np.array([
        base,                         # identical
        [50, 20, 90, 60],             # touching on x
        [10, 60, 50, 100],            # touching on y
        [20, 30, 40, 50],             # nested inside
        [0, 0, 100, 100],             # contains
        [200, 200, 300, 300],         # disjoint
        [30, 40, 30, 80],             # zero width, crosses base
        [30, 40, 30, 40],             # a point inside base
        [60, 70, 50, 65],             # inverted (negative area)
        [10.1, 20.3, 49.7, 60.2],     # near-identical
        [49.999, 20, 90, 60],         # sliver overlap
        [-5.5, -7.25, 12.75, 21.5],   # negative coordinates
    ], np.float32)


def test_oracle_bbox_overlaps_is_the_formula():
    rng = np.random.default_rng(3)
    xy = rng.uniform(0, 200, (60, 2))
    wh = 2.0 ** rng.uniform(-3, 7, (60, 2))
    rnd = np.concatenate([xy, xy + wh], 1).astype(np.float32)
    boxes = np.concatenate([_edge_boxes(), rnd])
    got = bbox_overlaps(boxes, boxes[::-1])
    assert got.dtype == np.float32 and got.shape == (len(boxes), len(boxes))
    want = np.array([[_iou_scalar(a, b) for b in boxes[::-1]] for a in boxes], np.float32)
    assert np.array_equal(got, want)                        # -0.0 == +0.0: the sign of a zero is not in the contract
    nz = want != 0
    assert np.array_equal(got[nz].view(np.int32), want[nz].view(np.int32))
    e = bbox_overlaps(_edge_boxes()[:1], _edge_boxes())[0]
    assert e[0] == 1 and e[1] == 0 and e[2] == 0 and e[5] == 0 and e[6] == 0 and e[7] == 0 and e[8] == 0
    assert e[3] == f(400) / f(1600) and 0 < e[10] < 1e-4
    assert (got >= 0).all() and (got <= 1).all()


def test_workspace_query_is_host_only():
    q = _lib().rsdet_assign_hbb_workspace_bytes
    assert q(1, 1) > 0
    assert q(2048, 261888) >= 2048 * 8 + 4
    assert q(4096, 261888) > q(2048, 261888)
    assert q(2048, 261888) == q(2048, 1)                    # per-GT keys only: nothing grows with the anchors
    for G, n in [(0, 10), (-1, 10), (10, 0), (10, -5), (MAX_GTS + 1, 10), (10, MAX_ANCHORS + 1)]:
        assert q(G, n) == 0, (G, n)
    assert q(MAX_GTS, MAX_ANCHORS) > 0


def test_bbox_overlaps_rejects_before_any_launch():
    L = _lib()
    fn = L.rsdet_bbox_overlaps
    assert fn(8, -1, 8, 5, 8, None) == EINVAL
    assert fn(8, 5, 8, -1, 8, None) == EINVAL
    assert fn(None, 5, 8, 5, 8, None) == EINVAL
    assert fn(8, 5, None, 5, 8, None) == EINVAL
    assert fn(8, 5, 8, 5, None, None) == EINVAL
    assert fn(8, 1 << 30, 8, 1 << 11, 8, None) == ELIMIT        # 2^41 pairs
    assert fn(None, 0, None, 7, None, None) == 0                # empty: nothing to do, nothing launched


def test_assign_hbb_rejects_before_any_launch():
    L = _lib()
    fn = L.rsdet_assign_hbb
    big = 1 << 40

    def call(G=4, n=100, gt=8, anc=8, inds=8, mlq=1, ws=8, wsb=big):
        return fn(gt, G, anc, n, None, 0.7, 0.0, 0.3, 0.3, mlq, 1, None, -1, inds, 8, None, ws, wsb, None)

    assert call(G=0) == EINVAL and call(G=-3) == EINVAL
    assert call(n=0) == EINVAL and call(n=-1) == EINVAL
    assert call(gt=None) == EINVAL and call(anc=None) == EINVAL and call(inds=None) == EINVAL
    assert call(G=MAX_GTS + 1) == ELIMIT
    assert call(n=MAX_ANCHORS + 1) == ELIMIT
    need = L.rsdet_assign_hbb_workspace_bytes(4, 100)
    assert call(wsb=need - 1) == EWORKSPACE
    assert call(ws=None, wsb=0) == EWORKSPACE                  # the low-quality pass needs its keys


def test_core_and_mirror_reject_on_the_host():
    from rs_detection_b200 import core
    from rs_detection_b200.jdet.models.boxes.assigner import MaxIoUAssigner
    from rs_detection_b200.jdet.models.boxes.iou_calculator import BboxOverlaps2D
    calc = BboxOverlaps2D()
    a, b = torch.zeros((3, 4)), torch.zeros((5, 5))
    with pytest.raises(AssertionError):
        calc(a, b, mode='iof')
    with pytest.raises(AssertionError):
        calc(a, b, is_aligned=True)
    with pytest.raises(AssertionError):
        calc(torch.zeros((3, 6)), b)
    assert repr(calc) == "BboxOverlaps2D()"
    m = MaxIoUAssigner(0.7, 0.3, 0.3, iou_calculator=dict(type='BboxOverlaps2D'))
    assert isinstance(m.iou_calculator, BboxOverlaps2D)
    with pytest.raises(ValueError):
        m.assign(torch.zeros((0, 4)), torch.zeros((3, 4)))
    with pytest.raises(RuntimeError, match="CUDA"):              # no CPU fallback
        core.assign_hbb(torch.zeros((3, 4)), torch.zeros((5, 4)), 0.7, 0.3)
    with pytest.raises(RuntimeError, match="CUDA"):
        core.bbox_overlaps(torch.zeros((3, 4)), torch.zeros((5, 4)))


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_adapter_bodies_compile_against_rsdet_h(fake_jt, tmp_path):  # noqa: F811
    from rs_detection_b200 import jittor_adapter as A
    A.bbox_overlaps(V((7, 4)), V((9, 4)))
    A.assign_hbb(V((6, 4)), V((1000, 4)), 0.7, 0.3, 0.3, True, True, V((6,), "int32"), -1, V((1000,), "uint8"))
    A.assign_hbb(V((6, 4)), V((1000, 4)), 0.5, (0.1, 0.5), 0.5, False, False)
    assert A.bbox_overlaps(V((0, 4)), V((9, 4))).shape == (0, 9) and len(fake_jt) == 3
    with pytest.raises(ValueError):
        A.assign_hbb(V((0, 4)), V((10, 4)), 0.7, 0.3)
    src = tmp_path / "adapter_hbb.cu"
    body = fake_jt[0]["header"] + "\nnamespace jittor { Executor exe; }\n"
    for i, r in enumerate(fake_jt):
        body += _wrap(i, dict(r, header=""))
    src.write_text(body)
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-c", str(src), "-o", str(tmp_path / "a.o"),
           "-I", os.path.join(ROOT, "tests", "jittor_stub"), "-Wno-deprecated-gpu-targets"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-4000:]
