"""GPU parity: nms_rotated / ml_nms_rotated / multiclass_nms_rotated / poly_nms through the jdet mirror
-> C ABI vs the oracle.  Contract: keep indices bit-exact (pairs inside the 1e-6 band are counted)."""
import os

import numpy as np
import pytest
import torch

import workloads as W
from helpers import band_pairs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_drift_golden.npz")


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_known_answer(cuda):
    from rs_detection_b200.jdet.ops.nms_rotated import ml_nms_rotated, nms_rotated
    dets = _t(np.array([[0, 0, 1, 1, 0], [0, 0, 0.5, 0.5, 0.3], [0, 0, 0.9, 0.9, 0]], np.float32))
    scores = _t(np.array([0.1, 0.2, 0.3], np.float32))
    labels = _t(np.array([1, 1, 1]))
    assert nms_rotated(dets, scores, 0.3).tolist() == [2]           # nms_rotated.py:598-603
    assert ml_nms_rotated(dets, scores, labels, 0.3).tolist() == [2]
    assert nms_rotated(torch.zeros((0, 5), device="cuda"), torch.zeros((0,), device="cuda"), 0.3).numel() == 0


@pytest.mark.parametrize("n,canvas", [(1, 1024), (63, 256), (64, 256), (65, 256), (1000, 1024), (5000, 1024),
                                      (9000, 2048)])  # 9000 boxes = 141 blocks: the multi-CTA cooperative scan
@pytest.mark.parametrize("thr", [0.1, 0.5])
def test_nms_rotated_vs_oracle(cuda, oracle, n, canvas, thr):
    from rs_detection_b200.jdet.ops.nms_rotated import nms_rotated
    d = W.rotated_boxes(n, 100 + n, canvas=canvas, smin=8, smax=128)
    s = W.distinct_scores(n, 100 + n)
    got = nms_rotated(_t(d), _t(s), thr).cpu().numpy()
    want = oracle.nms_rotated(d, s, thr, ge=False)
    if n <= 1000:
        print("band pairs:", band_pairs(oracle.box_iou_rotated(d, d, 0, 1), thr))
    assert np.array_equal(got, want)
    assert np.all(np.diff(got) > 0)  # ascending original index (jt.where(keep)[0])


def test_nms_cpu_cuda_rule_and_explicit_order(cuda, oracle):
    from rs_detection_b200.jdet.ops.nms_rotated import nms_rotated_cpu, nms_rotated_cuda
    n = 800
    d = W.rotated_boxes(n, 7, canvas=512, smin=16, smax=128)
    d[100:200] = d[0:100]  # exact duplicates: IoU == 1 -> `>=` and `>` agree; thr 1.0 separates them
    s = W.distinct_scores(n, 7)
    order = np.argsort(-s.astype(np.float64), kind="stable").astype(np.int32)
    for thr in (0.3, 1.0):
        for fn, ge in ((nms_rotated_cpu, True), (nms_rotated_cuda, False)):
            got = fn(_t(d), _t(order.astype(np.int64)), thr, box_length=5).cpu().numpy()
            assert np.array_equal(got, oracle.nms_rotated_keep(d, order, thr, 5, ge, 1)), (thr, ge)


@pytest.mark.parametrize("n,ncls", [(3000, 15), (4000, 1), (500, 500), (20000, 2)])
def test_ml_nms_rotated_vs_oracle(cuda, oracle, n, ncls):
    from rs_detection_b200.jdet.ops.nms_rotated import ml_nms_rotated
    d = W.rotated_boxes(n, 31, canvas=700, smin=16, smax=128)
    s = W.distinct_scores(n, 31)
    lab = np.random.default_rng(1).integers(0, ncls, n)
    got = ml_nms_rotated(_t(d), _t(s), _t(lab), 0.1).cpu().numpy()
    assert np.array_equal(got, oracle.ml_nms_rotated(d, s, lab, 0.1))


@pytest.mark.parametrize("max_num", [-1, 2000, 50])
@pytest.mark.parametrize("per_class_boxes", [False, True])
def test_multiclass_nms_rotated_vs_oracle(cuda, oracle, max_num, per_class_boxes):
    from rs_detection_b200.jdet.ops.nms_rotated import multiclass_nms_rotated
    n, C = 1500, 15
    sc = W.class_scores(n, C, 3)
    if per_class_boxes:
        bb = np.concatenate([W.rotated_boxes(n, 40 + c, smin=16, smax=160) for c in range(C + 1)], 1)
    else:
        bb = W.rotated_boxes(n, 40, smin=16, smax=160)
    fac = np.random.default_rng(9).uniform(0.5, 1.0, n).astype(np.float32)
    for sf in (None, fac):
        wd, wl = oracle.multiclass_nms_rotated(bb, sc, 0.05, dict(type='nms_rotated', iou_thr=0.1), max_num, sf)
        gd, gl = multiclass_nms_rotated(_t(bb), _t(sc), 0.05, dict(type='nms_rotated', iou_thr=0.1), max_num,
                                        None if sf is None else _t(sf))
        assert gd.shape == wd.shape and gd.shape[1] == 6
        assert np.array_equal(gd.cpu().numpy(), wd)
        assert np.array_equal(gl.cpu().numpy(), wl)
    # nothing above the score threshold -> (0,6), (0,)
    gd, gl = multiclass_nms_rotated(_t(bb), _t(sc), 2.0, dict(iou_thr=0.1), max_num)
    assert tuple(gd.shape) == (0, 6) and gl.numel() == 0


def test_poly_nms_vs_oracle(cuda, oracle):
    from rs_detection_b200.jdet.ops.nms_poly import multiclass_poly_nms, poly_nms
    n = 1200
    pp = oracle.obb2poly(W.rotated_boxes(n, 51, canvas=600, smin=16, smax=128))
    s = W.distinct_scores(n, 51)
    b9 = np.concatenate([pp, s[:, None]], 1)
    for thr in (0.1, 0.5):
        got = poly_nms(_t(b9), thr).cpu().numpy()
        want = oracle.poly_nms(b9, thr)
        assert np.array_equal(got, want)
    lab = np.random.default_rng(2).integers(0, 15, n)
    gd, gl = multiclass_poly_nms(_t(pp), _t(s), _t(lab), 0.1)
    wd, wl = oracle.multiclass_poly_nms(pp, s, lab, 0.1)
    assert np.array_equal(gd.cpu().numpy(), wd) and np.array_equal(gl.cpu().numpy(), wl)


def test_large_nms_properties(cuda):
    """50k boxes: too slow for the CPU oracle; size-independent properties of greedy NMS instead:
    (a) idempotence, (b) survivors are pairwise below threshold, (c) every suppressed box has a
    higher-scored survivor above threshold."""
    from rs_detection_b200 import core
    from rs_detection_b200._lib import NMS_ROTATED
    n, thr = 50000, 0.3
    d = _t(W.rotated_boxes(n, 77, canvas=4096, smin=8, smax=128))
    s = _t(W.distinct_scores(n, 77))
    res = core.nms(NMS_ROTATED, d, s, thr)
    keep = res.sorted_idx
    k = keep.numel()
    assert 0 < k < n
    again = core.nms(NMS_ROTATED, d[keep], s[keep], thr).sorted_idx
    assert again.numel() == k                                                      # (a)
    sub = keep[torch.randperm(k, device="cuda")[:3000]]
    iou = core.box_iou_rotated(d[sub], d[keep], 0)
    iou[torch.arange(sub.numel(), device="cuda"), torch.searchsorted(keep, sub)] = 0
    assert float(iou.max()) <= thr                                                 # (b)
    mask = res.keep_mask
    supp = torch.nonzero(~mask)[:, 0]
    supp = supp[torch.randperm(supp.numel(), device="cuda")[:3000]]
    iou = core.box_iou_rotated(d[supp], d[keep], 0)
    higher = s[keep][None, :] > s[supp][:, None]
    assert bool(((iou > thr) & higher).any(1).all())                               # (c)


@pytest.mark.parametrize("K,C,score_thr", [(4000, 10, 0.001), (2000, 15, 0.05)])
def test_multiclass_nms_rotated_baseline_sizes(cuda, oracle, K, C, score_thr):
    """BASELINE config 2 (K=4000, 10 classes, score_thr 0.001: ~40k candidates, 63-block staged scan, pair queue near
    capacity) and config 1 (K=2000, 15 classes, 0.05) -- the exact tiles bench.py times -- against the oracle, and
    per class against the reference's own NMS source compiled for the host (oracle/_ref, where it is built from the
    reference tree).  Everywhere, the per-class keep counts are also compared with the ORACLE's counts stored in
    tests/golden/oracle_drift_golden.npz: a drift guard, not reference output."""
    import bench as B
    from rs_detection_b200.jdet.ops.nms_rotated import multiclass_nms_rotated
    boxes = W.rotated_boxes(K, 500)                                   # = bench.tile_inputs(0) boxes for K = 4000
    scores = W.class_scores(K, C, 0, logit_scale=1.0)
    if K == B.K_ROIS and C == B.NUM_CLASSES:
        _, _, b0, s0 = B.tile_inputs(0)
        assert np.array_equal(b0, boxes) and np.array_equal(s0, scores)
    wd, wl = oracle.multiclass_nms_rotated(boxes, scores, score_thr, dict(iou_thr=0.1), 2000)
    gd, gl = multiclass_nms_rotated(_t(boxes), _t(scores), score_thr, dict(type='nms_rotated', iou_thr=0.1), 2000)
    assert np.array_equal(gd.cpu().numpy(), wd) and np.array_equal(gl.cpu().numpy(), wl)
    # per-class keep counts (the label gate of ml_nms_rotated = one NMS per class): the oracle's stored counts, checked
    # against the reference's CUDA-rule NMS source where oracle/_ref is built
    gd_all, gl_all = multiclass_nms_rotated(_t(boxes), _t(scores), score_thr, dict(type='nms_rotated', iou_thr=0.1), -1)
    gl_all = gl_all.cpu().numpy()
    kept = np.load(GOLD)[f"mcnms_class_kept_K{K}_C{C}"]
    from oracle import ref as R
    if R.ensure_built():
        for c in range(C):
            m = scores[:, c + 1] > np.float32(score_thr)
            sc = scores[m, c + 1]
            order = np.argsort(-sc.astype(np.float64), kind="stable").astype(np.int32)
            assert int(R.nms_keep(boxes[m], order, 0.1, 5, ge=False).sum()) == kept[c]
    total = int(kept.sum())
    assert total - 1 == gd_all.shape[0]      # max_num=-1 drops the last detection (nms_rotated.py:590-591)
    print(f"K={K} C={C}: {int((scores[:, 1:] > score_thr).sum())} candidates -> {total} kept")


def test_poly_nms_exact_zero_skip_adversarial(cuda, oracle):
    """csrc/poly_iou.cuh drops pairs whose 16 fan terms are provably exactly zero (angular sectors, seen from the
    origin, disjoint by a safety margin).  The oracle evaluates every pair literally; threshold 0 turns ANY non-zero
    cancellation noise into a suppression, so the keep lists agree only if the skipped pairs really are exact zeros.
    Layouts: a fan of boxes around the origin with gaps down to the margin, boxes with radial edges, boxes that contain
    or touch the origin, the reference's class-offset layout far from the origin, integer coordinates (exact ties in
    the cross products)."""
    from rs_detection_b200.jdet.ops.nms_poly import poly_nms
    rng = np.random.default_rng(123)
    sets = []
    # (a) fan around the origin: radius 40..3000, angular pitch barely above / below the box's own angular width
    for R, npts, jitter in ((60.0, 90, 0.002), (400.0, 300, 0.0005), (3000.0, 400, 0.0002)):
        ang = np.linspace(0, 2 * np.pi, npts, endpoint=False) + rng.normal(0, jitter, npts)
        w = 2 * np.pi * R / npts * rng.uniform(0.6, 1.3, npts)
        h = rng.uniform(4, 30, npts)
        th = ang + np.pi / 2 + rng.normal(0, 0.2, npts)          # tangential boxes, some rotated
        th[::7] = ang[::7]                                        # radial boxes: edge lines through the origin region
        obb = np.stack([R * np.cos(ang), R * np.sin(ang), w, h, th], 1).astype(np.float32)
        sets.append(oracle.obb2poly(obb))
    # (b) boxes containing / touching the origin and tiny boxes next to it
    obb = W.rotated_boxes(150, 9, canvas=80, smin=2, smax=60)
    obb[:, :2] -= 40
    sets.append(oracle.obb2poly(obb))
    # (c) class-offset layout of multiclass_poly_nms (nms_poly.py:235-237), far from the origin
    obb = W.rotated_boxes(500, 10, canvas=500, smin=8, smax=90)
    p = oracle.obb2poly(obb)
    lab = rng.integers(0, 6, 500)
    sets.append((p + (lab * (float(p.max() - p.min()) + 1))[:, None]).astype(np.float32))
    # (d) integer coordinates
    sets.append(np.round(oracle.obb2poly(W.rotated_boxes(300, 11, canvas=300, smin=8, smax=60))).astype(np.float32) + 1000)
    for k, pp in enumerate(sets):
        pp = np.ascontiguousarray(pp, np.float32)
        sc = W.distinct_scores(pp.shape[0], 60 + k)
        b9 = np.concatenate([pp, sc[:, None]], 1)
        for thr in (0.0, 0.02, 0.3):
            got = poly_nms(_t(b9), thr).cpu().numpy()
            want = oracle.poly_nms(b9, thr)
            assert np.array_equal(got, want), (k, thr, len(got), len(want))


@pytest.mark.parametrize("n,canvas,thr", [(40000, 1024, 0.1), (40000, 4096, 0.5), (100000, 2048, 0.3)])
def test_sparse_rotated_path_equals_dense_engine(cuda, n, canvas, thr):
    """n >= 32768 unlabelled rotated boxes take the sparse path (sweep-and-prune candidates, CSR of suppressing pairs,
    fixed-point greedy); the same call WITH (all-equal) labels stays on the dense tiles + scan.  Both apply the same
    exact filter cascade and clipper, so the keep sets must be identical."""
    from rs_detection_b200 import core
    from rs_detection_b200._lib import NMS_ROTATED, NMS_ROTATED_GE
    d = _t(W.rotated_boxes(n, n + 3, canvas=canvas, smin=8, smax=128))
    s = _t(W.distinct_scores(n, n + 3))
    for kind in (NMS_ROTATED, NMS_ROTATED_GE):
        sparse = core.nms(kind, d, s, thr)
        dense = core.nms(kind, d, s, thr, labels=torch.zeros(n, dtype=torch.int32, device="cuda"))
        assert torch.equal(sparse.keep_mask, dense.keep_mask)
        assert torch.equal(sparse.sorted_idx, dense.sorted_idx) and 0 < sparse.count < n
