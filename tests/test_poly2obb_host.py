"""CPU: the restatement of cv2.minAreaRect (tests/min_area_rect_oracle.c) against the installed OpenCV, and the poly2obb
entry points' host-side contract.

The restatement is the checker of rsdet_poly2obb, so it is pinned first: bit for bit against cv2.minAreaRect (centre,
size and angle) and against jdet.ops.bbox_transforms.poly2obb (the mirror's OpenCV loop plus the le90 step) on
about 1.3 million seeded quads: jittered rotated rectangles in scene coordinates, near-squares, axis-aligned boxes, every
start vertex in both winding orders, integer-grid quads with collinear or coincident corners (two- and one-point
hulls), and the golden merge fixture."""
import os
import subprocess

import numpy as np
import pytest
import torch

import min_area_rect_oracle as M
from test_jittor_adapter import NVCC, ROOT, V, _wrap, fake_jt  # noqa: F401  (fake_jt is a fixture)

EINVAL = -1
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "merge_golden.npz")


def _rows():
    fam = M.families(seed=11, m=400_000)
    fam["golden"] = np.load(GOLDEN)["p2o_polys"]
    return fam


@pytest.fixture(scope="module")
def rows():
    return _rows()


def test_families_cover_the_cases(rows):
    assert sum(r.shape[0] for r in rows.values()) >= 1_000_000
    grid = M.min_area_rect(rows["grid"])
    assert ((grid[:, 2] == 0) & (grid[:, 3] == 0)).any()          # one-point hulls
    assert ((grid[:, 2] == 0) != (grid[:, 3] == 0)).any()         # two-point hulls
    assert (M.min_area_rect(rows["axis_aligned"])[:, 4] == -90).all()


@pytest.mark.parametrize("family", ["rotated", "near_square", "axis_aligned", "orders", "grid", "grid_orders", "golden"])
def test_restatement_is_cv2_min_area_rect(rows, family):
    got, want = M.min_area_rect(rows[family]), M.cv2_min_area_rect(rows[family])
    bad = np.nonzero((got.view(np.int32) != want.view(np.int32)).any(1))[0]
    assert bad.size == 0, (family, bad.size, rows[family][bad[:3]], got[bad[:3]], want[bad[:3]])


@pytest.mark.parametrize("family", ["rotated", "near_square", "axis_aligned", "orders", "grid", "grid_orders", "golden"])
def test_restatement_is_the_mirror_poly2obb(rows, family):
    from rs_detection_b200.jdet.ops.bbox_transforms import poly2obb
    got, want = M.poly2obb(rows[family]), poly2obb(rows[family])
    assert want.dtype == np.float64 and got.shape == want.shape
    bad = np.nonzero((got.view(np.int64) != want.view(np.int64)).any(1))[0]
    assert bad.size == 0, (family, bad.size, rows[family][bad[:3]], got[bad[:3]], want[bad[:3]])


def test_restatement_reproduces_the_golden_obb():
    g = np.load(GOLDEN)
    assert np.array_equal(M.poly2obb(g["p2o_polys"]).view(np.int64), g["p2o_obb"].view(np.int64))


def test_poly2obb_rejects_before_any_launch():
    from rs_detection_b200 import _lib
    L = _lib.load()
    before = L.rsdet_launch_count()
    assert L.rsdet_poly2obb(8, -1, 8, None) == EINVAL
    assert L.rsdet_poly2obb(None, 5, 8, None) == EINVAL
    assert L.rsdet_poly2obb(8, 5, None, None) == EINVAL
    assert L.rsdet_poly2obb(None, 0, None, None) == 0             # empty: nothing to do, nothing launched
    assert L.rsdet_launch_count() == before


def test_core_poly2obb_rejects_on_the_host():
    from rs_detection_b200 import core
    with pytest.raises(RuntimeError, match="CUDA"):              # no CPU fallback
        core.poly2obb(torch.zeros((3, 8), dtype=torch.float64))


@pytest.mark.skipif(not os.path.exists(NVCC), reason="nvcc not available")
def test_adapter_poly2obb_compiles_against_rsdet_h(fake_jt, tmp_path):  # noqa: F811
    from rs_detection_b200 import jittor_adapter as A
    assert A.poly2obb(V((7, 8), "float64")).shape == (7, 5)
    assert A.poly2obb(V((2, 3, 8), "float64")).shape == (2, 3, 5)
    assert A.poly2obb(V((0, 8), "float64")).shape == (0, 5) and len(fake_jt) == 2
    with pytest.raises(AssertionError):
        A.poly2obb(V((4, 10), "float64"))
    src = tmp_path / "adapter_poly2obb.cu"
    body = fake_jt[0]["header"] + "\nnamespace jittor { Executor exe; }\n"
    for i, r in enumerate(fake_jt):
        body += _wrap(i, dict(r, header=""))
    src.write_text(body)
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-c", str(src), "-o", str(tmp_path / "a.o"),
           "-I", os.path.join(ROOT, "tests", "jittor_stub"), "-Wno-deprecated-gpu-targets"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-4000:]
