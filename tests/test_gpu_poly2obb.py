"""GPU: rsdet_poly2obb (core.poly2obb) against the host poly2obb (cv2.minAreaRect + le90) and its C restatement, bit for
bit, and the two merge pipelines that use it against the host-poly2obb route they replaced."""
import os

import numpy as np
import pytest
import torch

import min_area_rect_oracle as M
import workloads as W

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "merge_golden.npz")
FAMILIES = ["rotated", "near_square", "axis_aligned", "orders", "grid", "grid_orders", "golden"]


@pytest.fixture(scope="module")
def rows():
    fam = M.families(seed=23, m=400_000)
    fam["golden"] = np.load(GOLDEN)["p2o_polys"]
    return fam


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _device(polys):
    from rs_detection_b200 import core
    out = core.poly2obb(torch.from_numpy(np.ascontiguousarray(polys, np.float64)).cuda())
    assert out.dtype == torch.float64 and out.is_cuda
    return out.cpu().numpy()


def _mismatch(got, want):
    return np.nonzero((_bits(got) != _bits(want)).any(1))[0]


@pytest.mark.parametrize("family", FAMILIES)
def test_device_equals_host_and_restatement(cuda, rows, family):
    from rs_detection_b200.jdet.ops.bbox_transforms import poly2obb
    q = rows[family]
    got = _device(q)
    for want in (poly2obb(q), M.poly2obb(q)):
        bad = _mismatch(got, want)
        assert bad.size == 0, (family, bad.size, q[bad[:3]], got[bad[:3]], want[bad[:3]])


def test_large_n(cuda):
    """4.2 million rows in one call: every family, concatenated and shuffled."""
    from rs_detection_b200.jdet.ops.bbox_transforms import poly2obb
    fam = M.families(seed=29, m=1_320_000)
    q = np.concatenate(list(fam.values()))
    q = q[np.random.default_rng(0).permutation(q.shape[0])]
    assert q.shape[0] >= 4_000_000
    got = _device(q)
    bad = _mismatch(got, M.poly2obb(q))
    assert bad.size == 0, (bad.size, q[bad[:3]])
    sub = np.random.default_rng(1).choice(q.shape[0], 200_000, replace=False)
    assert _mismatch(got[sub], poly2obb(q[sub])).size == 0


def test_n_zero_and_one(cuda):
    from rs_detection_b200 import _lib, core
    before = _lib.launch_count()
    empty = core.poly2obb(torch.zeros((0, 8), dtype=torch.float64, device="cuda"))
    assert empty.shape == (0, 5) and empty.dtype == torch.float64 and _lib.launch_count() == before
    one = np.array([[911., 109., 873., 208., 699., 141., 737., 41.]])
    assert _mismatch(_device(one), M.poly2obb(one)).size == 0
    # float32 input is widened losslessly; the kernel then rounds it back to the same float32 corners
    q32 = torch.from_numpy(np.ascontiguousarray(M.families(seed=2, m=800)["rotated"], np.float32)).cuda()
    assert _mismatch(core.poly2obb(q32).cpu().numpy(), M.poly2obb(q32.cpu().numpy().astype(np.float64))).size == 0


def test_argument_errors_launch_nothing(cuda):
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    buf = torch.zeros((4, 8), dtype=torch.float64, device="cuda")
    before = _lib.launch_count()
    assert L.rsdet_poly2obb(buf.data_ptr(), -1, buf.data_ptr(), None) == -1
    assert L.rsdet_poly2obb(None, 4, buf.data_ptr(), None) == -1
    assert L.rsdet_poly2obb(buf.data_ptr(), 4, None, None) == -1
    assert _lib.launch_count() == before
    with pytest.raises(ValueError):
        core.poly2obb(torch.zeros((4, 10), dtype=torch.float64, device="cuda"))


def test_non_default_stream_and_graph_capture(cuda, rows):
    from rs_detection_b200 import core
    q = rows["orders"][:100_000]
    want = M.poly2obb(q)
    x = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        y = core.poly2obb(x)
    torch.cuda.current_stream().wait_stream(s)
    assert _mismatch(y.cpu().numpy(), want).size == 0

    static_in = torch.zeros_like(x)
    g = torch.cuda.CUDAGraph()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        core.poly2obb(static_in)  # warm-up outside the capture
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            static_out = core.poly2obb(static_in)
    for fam in ("orders", "grid_orders"):
        static_in.copy_(torch.from_numpy(np.ascontiguousarray(rows[fam][:100_000])).cuda())
        g.replay()
        torch.cuda.synchronize()
        assert _mismatch(static_out.cpu().numpy(), M.poly2obb(rows[fam][:100_000])).size == 0


# ------------------------------------------------------------------------------------------ the pipelines that use it
@pytest.fixture()
def host_route(monkeypatch):
    """Swap core.poly2obb for the host OpenCV loop: the route these pipelines took before the device call."""
    from rs_detection_b200 import core
    from rs_detection_b200.jdet.ops.bbox_transforms import poly2obb

    def host(polys):
        return torch.from_numpy(poly2obb(polys.cpu().numpy())).to(polys.device)

    def use():
        monkeypatch.setattr(core, "poly2obb", host)
    return use


@pytest.mark.parametrize("seed", [0, 1])
def test_csv_ensemble_matches_the_host_route(cuda, host_route, seed):
    from rs_detection_b200.jdet import merge as PM
    subs = W.csv_submissions(num_images=12, objects_per_image=400, seed=seed)
    thr_d = {c: 0.3 + 0.05 * i for i, c in enumerate(PM.FAIR1M_1_5_CLASSES)}
    got = [PM.merge_csv_with_class(subs, 0.625), PM.merge_csv_with_class(subs, thr_d), PM.merge_csv_without_class(subs, 0.9)]
    host_route()
    want = [PM.merge_csv_with_class(subs, 0.625), PM.merge_csv_with_class(subs, thr_d), PM.merge_csv_without_class(subs, 0.9)]
    n = subs[0].shape[0] + subs[1].shape[0]
    for a, b in zip(got, want):
        assert a.shape == b.shape and np.array_equal(_bits(a), _bits(b)) and 0 < a.shape[0] < n


def test_py_cpu_nms_obb_and_mergebyobb_match_the_host_route(cuda, host_route, tmp_path):
    from oracle import formats as F
    from rs_detection_b200.jdet.data.devkits import result_merge as RM
    sc = W.merge_scene(num_objects=400, scene=2500, seed=9)
    dets = np.concatenate([sc["polys"], sc["scores"][:, None]], 1)
    got = [RM.py_cpu_nms_obb(dets, t) for t in (0.1, 0.3)]
    F.write_before_nms(W.tile_results(150, 4, 2200, 2, seed=12), tmp_path / "before", W.FAIR1M_CLASSES)
    RM.mergebyobb(str(tmp_path / "before"), str(tmp_path / "got"))
    host_route()
    want = [RM.py_cpu_nms_obb(dets, t) for t in (0.1, 0.3)]
    RM.mergebyobb(str(tmp_path / "before"), str(tmp_path / "want"))
    for a, b in zip(got, want):
        assert np.array_equal(a, b) and 0 < len(a) < len(dets)
    files = sorted(os.listdir(tmp_path / "want"))
    assert files == sorted(os.listdir(tmp_path / "got")) and files
    for f in files:
        assert (tmp_path / "got" / f).read_text() == (tmp_path / "want" / f).read_text(), f
