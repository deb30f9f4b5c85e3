"""Pin the C restatement (oracle/rsdet_oracle.c) to the reference's own source compiled for the host
(oracle/_ref, built by oracle/build_ref.py from the strings inside the reference's python/jdet/ops/*.py).
Bit-for-bit: any difference is a failure.

oracle/_ref can only be built from the reference tree, which is not part of the repository.  Where it is built, the
tests compare the oracle with it (`live_ref`).  Everywhere, they also compare the oracle with
tests/golden/oracle_drift_golden.npz: the ORACLE's own output on these inputs, stored as a drift guard (like the
`merge_*` entries of rotated_path_golden.npz), NOT reference output.  Reference output on smaller inputs is stored in
tests/golden/rotated_path_golden.npz and checked by tests/test_golden.py; it does not cover the degenerate IoU boxes,
the reference's CUDA hull-sort flavour itself, RoIAlign v0 forward with sampling_ratio 0, the backward with
sampling_ratio 0, or reversed / far-from-origin poly IoU, which only a run with oracle/_ref pins to the reference."""
import os

import numpy as np
import pytest

import workloads as W

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_drift_golden.npz")


def same_as_stored(a, gold, key):
    """a equals the stored array, or, where only a sample of it is stored, equals it at the stored flat indices"""
    a = np.asarray(a).ravel()
    idx = gold.get(key + "_idx")
    return np.array_equal(a if idx is None else a[idx], gold[key])


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLD))


@pytest.fixture(scope="module")
def live_ref():
    """oracle/_ref where it is built (or buildable from the reference tree), else None"""
    from oracle import ref as R
    return R if R.ensure_built() else None


def _pairs(seed=0, n=1500, g=192):
    P = W.rotated_boxes(n, seed)
    G = W.jittered_copies(P, g, seed + 1)
    return G, P


DEGENERATE = np.array([[5, 5, 4, 2, 0.3], [5, 5, 4, 2, 0.3], [5, 5, 0, 2, 0], [5, 5, 1e-8, 1e-8, 0], [9, 5, 4, 2, 0.3],
                       [5, 5, 2, 4, 0.3 + np.pi / 2], [7, 5, 4, 2, 0.3], [5, 5, 4, 2, -0.3]], np.float32)


def nms_inputs(n=2500, seed=3):
    d = W.rotated_boxes(n, seed, smin=16, smax=128)
    s = W.distinct_scores(n, seed)
    return d, np.argsort(-s.astype(np.float64), kind="stable").astype(np.int32)


def ml_nms_inputs(n=2500):
    d, order = nms_inputs(n, 4)
    lab = np.random.default_rng(0).integers(0, 15, n)
    return np.concatenate([d, lab[:, None].astype(np.float32)], 1), order


def roi_inputs():
    """(feat, rois, grad_rng): the gradient of the backward check is drawn from grad_rng after the forward"""
    rng = np.random.default_rng(0)
    feat = rng.standard_normal((2, 8, 64, 64)).astype(np.float32)
    rois = W.proposals(60, 0, batch=2)
    rois[:4, 3:5] = [[0.5, 0.5], [3000, 20], [20, 3000], [1, 900]]  # clamped / huge / out-of-map RoIs
    rois[4, 1:3] = [-40, 1100]
    return feat, rois, rng


def poly_inputs():
    """(polys, the same quads with reversed vertex order and far from the origin, their partners)"""
    from oracle import oracle as O
    pp = O.obb2poly(W.rotated_boxes(300, 5, smin=16, smax=128))
    return pp, pp[:, [0, 1, 6, 7, 4, 5, 2, 3]] + np.float32(7000), pp + np.float32(7000)


def poly_nms_inputs(n=600):
    from oracle import oracle as O
    pp = O.obb2poly(W.rotated_boxes(n, 6, smin=16, smax=128))
    s = W.distinct_scores(n, 6)
    return np.concatenate([pp, s[:, None]], 1), np.argsort(-s.astype(np.float64), kind="stable")


@pytest.mark.parametrize("version", [0, 1])
@pytest.mark.parametrize("cudasort", [False, True])
def test_iou_bit_exact(oracle, gold, live_ref, version, cudasort):
    G, P = _pairs()
    a = oracle.box_iou_rotated(G, P, version, int(cudasort))
    assert (a > 0.5).sum() > 50 and (a == 0).mean() > 0.5  # the sample spans both regimes
    assert same_as_stored(a, gold, f"iou_v{version}_cudasort{int(cudasort)}")
    if live_ref:
        assert np.array_equal(a, live_ref.box_iou(G, P, version, cudasort))


def test_iou_known_answer(oracle, live_ref):
    # the reference's own self-test boxes, box_iou_rotated.py:513-514 -> [[1,0.2],[0.2,1]]
    b = np.array([[0, 0, 1, 1, 0], [0.5, 0.5, 1, 2, 0]], np.float32)
    fns = [lambda: oracle.box_iou_rotated(b, b)] + ([lambda: live_ref.box_iou(b, b)] if live_ref else [])
    for f in fns:
        np.testing.assert_allclose(f(), [[1, 0.2], [0.2, 1]], rtol=0, atol=1e-7)


def test_iou_degenerate_inputs(oracle, gold, live_ref):
    b = DEGENERATE
    for v in (0, 1):
        for cs in (0, 1):
            a = oracle.box_iou_rotated(b, b, v, cs)
            assert np.array_equal(a, gold[f"iou_degenerate_v{v}_cudasort{cs}"])
            if live_ref:
                assert np.array_equal(a, live_ref.box_iou(b, b, v, bool(cs)))


@pytest.mark.parametrize("thr", [0.1, 0.5])
@pytest.mark.parametrize("ge", [False, True])
def test_nms_keep_exact(oracle, gold, live_ref, thr, ge):
    d, order = nms_inputs()
    k = oracle.nms_rotated_keep(d, order, thr, 5, ge)
    assert 0 < k.sum() < d.shape[0]
    assert np.array_equal(k, gold[f"nms_keep_{thr}_ge{int(ge)}"])
    if live_ref:
        assert np.array_equal(k, live_ref.nms_keep(d, order, thr, 5, ge))


def test_ml_nms_keep_exact(oracle, gold, live_ref):
    d6, order = ml_nms_inputs()
    k = oracle.nms_rotated_keep(d6, order, 0.1, 6, False)
    assert np.array_equal(k, gold["ml_nms_keep_0.1"])
    if live_ref:
        assert np.array_equal(k, live_ref.nms_keep(d6, order, 0.1, 6, False))


def test_nms_known_answer(oracle, live_ref):
    # nms_rotated.py:598-603 -> keep [2]
    dets = np.array([[0, 0, 1, 1, 0], [0, 0, 0.5, 0.5, 0.3], [0, 0, 0.9, 0.9, 0]], np.float32)
    scores = np.array([0.1, 0.2, 0.3], np.float32)
    assert oracle.nms_rotated(dets, scores, 0.3).tolist() == [2]
    assert oracle.ml_nms_rotated(dets, scores, np.array([1, 1, 1]), 0.3).tolist() == [2]
    if live_ref:
        order = np.argsort(-scores).astype(np.int32)
        assert np.nonzero(live_ref.nms_keep(dets, order, 0.3, 5, False))[0].tolist() == [2]


@pytest.mark.parametrize("version", [0, 1])
@pytest.mark.parametrize("sampling_ratio", [2, 0])
def test_roi_align_bit_exact(oracle, gold, live_ref, version, sampling_ratio):
    feat, rois, rng = roi_inputs()
    a = oracle.roi_align_rotated_fwd(feat, rois, (7, 7), 1 / 16, sampling_ratio, version)
    assert same_as_stored(a, gold, f"roi_fwd_v{version}_sr{sampling_ratio}")
    g = rng.standard_normal(a.shape).astype(np.float32)
    ab = oracle.roi_align_rotated_bwd(g, rois, feat.shape, 1 / 16, sampling_ratio, version)
    assert same_as_stored(ab, gold, f"roi_bwd_v{version}_sr{sampling_ratio}")
    if live_ref:
        assert np.array_equal(a, live_ref.roi_fwd(feat, rois, (7, 7), 1 / 16, sampling_ratio, version))
        assert np.array_equal(ab, live_ref.roi_bwd(g, rois, feat.shape, 1 / 16, sampling_ratio, version))


def test_poly_iou_bit_exact(oracle, gold, live_ref):
    pp, q, far = poly_inputs()
    a = oracle.poly_iou_matrix(pp, pp)
    assert (a > 0.3).sum() > 300
    assert same_as_stored(a, gold, "poly_iou")
    # clockwise / counter-clockwise vertex order and far-from-origin quads (multiclass offsets)
    b = oracle.poly_iou_matrix(q, far)
    assert same_as_stored(b, gold, "poly_iou_far_reversed")
    if live_ref:
        assert np.array_equal(a, live_ref.poly_iou_matrix(pp, pp))
        assert np.array_equal(b, live_ref.poly_iou_matrix(q, far))


def test_poly_nms_exact(oracle, gold, live_ref):
    b9, order = poly_nms_inputs()
    keep = oracle.poly_nms(b9, 0.1)
    assert np.array_equal(keep, gold["poly_nms_keep_0.1"])
    if live_ref:
        assert np.array_equal(keep, order[live_ref.poly_nms_sorted_keep(b9[order], 0.1)])


def test_fma_contraction_stays_inside_band(oracle, ref):
    """nvcc contracts a*b+c by default, g++ does not: the reference's CUDA and CPU paths differ by < 1e-6
    (SURVEY appendix A), which is where the 1e-6 exclusion band of the parity contract comes from."""
    G, P = _pairs(7)
    a = ref.box_iou(G, P, 1, False, fma=False)
    b = ref.box_iou(G, P, 1, False, fma=True)
    assert np.abs(a - b).max() < 1e-6
