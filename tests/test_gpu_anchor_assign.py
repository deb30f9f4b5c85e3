"""The horizontal IoU matrix (rsdet_bbox_overlaps) and the fused RPN anchor assignment (rsdet_assign_hbb) on the GPU.

The fused call must equal, bit for bit, the materialised route rsdet_assign_wrt_overlaps(rsdet_bbox_overlaps(...)) on the
1024^2 tile's 261 888 anchors, and the oracle (oracle.max_iou_assign over tests/hbb_oracle.bbox_overlaps) on smaller
scenes, including the cases where skipping the GTs that miss a CTA's anchor strip could change a decision: all-zero
columns with pos_iou_thr <= 0, and a GT that overlaps nothing with min_pos_iou = 0."""
import numpy as np
import pytest
import torch

import workloads as W
from hbb_oracle import bbox_overlaps

pytestmark = pytest.mark.gpu

TILE_LEVELS = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
# make_golden_refpy.py:125-128: the R-CNN, RPN and RPN-one-match assigner configs
THRESHOLDS = {"rcnn": (0.5, 0.5, 0.5, False, True), "rpn": (0.7, 0.3, 0.3, True, True), "rpn_one": (0.7, 0.3, 0.3, True, False)}


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def tile_anchors(levels=TILE_LEVELS):
    from rs_detection_b200.jdet.models.boxes.anchor_generator import AnchorGenerator
    gen = AnchorGenerator(strides=[4, 8, 16, 32, 64][:len(levels)], ratios=[0.5, 1.0, 2.0], scales=[8])
    return torch.cat(gen.grid_anchors(levels, device="cuda")).contiguous()


def gt_hbb(G, seed, canvas=W.TILE, smax=256):
    from oracle import oracle as O
    src = W.rotated_boxes(max(G, 16), seed, canvas=canvas, smin=8, smax=smax)
    return O.obb2hbb(W.jittered_copies(src, G, seed + 1))


def fused(gt, anc, cfg, labels=None, valid=None, fill=-1):
    from rs_detection_b200 import core
    pos, neg, mpos, mlq, allm = cfg
    return core.assign_hbb(gt, anc, pos, neg, mpos, mlq, allm, labels, fill, valid=valid)


def materialised(gt, anc, cfg, labels=None, fill=-1, ov=None):
    from rs_detection_b200 import core
    pos, neg, mpos, mlq, allm = cfg
    ov = core.bbox_overlaps(gt, anc) if ov is None else ov
    return core.assign_wrt_overlaps(ov, pos, neg, mpos, mlq, allm, labels, fill)


def oracle_assign(oracle, gt, anc, cfg, labels=None, fill=-1):
    pos, neg, mpos, mlq, allm = cfg
    return oracle.max_iou_assign(bbox_overlaps(gt, anc), pos, neg, mpos, mlq, allm, gt_labels=labels,
                                 assigned_labels_filled=fill)


def same(a, b, what):
    """Bit-identical outputs (gt_inds, max_overlaps, labels or None)."""
    assert torch.equal(a[0], b[0]), f"{what}: gt_inds ({int((a[0] != b[0]).sum())} differ)"
    assert torch.equal(a[1].view(torch.int32), b[1].view(torch.int32)), f"{what}: max_overlaps bits"
    assert (a[2] is None) == (b[2] is None) and (a[2] is None or torch.equal(a[2], b[2])), f"{what}: labels"


def like_oracle(got, want, what):
    """Equal to the oracle: exact indices and labels, equal max_overlaps (bit-equal where nonzero)."""
    assert np.array_equal(got[0].cpu().numpy(), want[0]), f"{what}: gt_inds"
    assert np.array_equal(got[1].cpu().numpy(), want[1]), f"{what}: max_overlaps"
    if want[2] is not None:
        assert np.array_equal(got[2].cpu().numpy(), want[2]), f"{what}: labels"


# ---------------------------------------------------------------------------------------------- the IoU matrix
def test_bbox_overlaps_matches_oracle(cuda):
    from rs_detection_b200 import core
    rng = np.random.default_rng(5)
    xy = rng.uniform(0, 500, (1000, 2))
    wh = 2.0 ** rng.uniform(-2, 8, (1000, 2))
    b1 = np.concatenate([xy, xy + wh], 1).astype(np.float32)
    b1[:10] = b1[10:20]                                          # identical rows
    b1[20:25, 2] = b1[20:25, 0]                                  # zero width
    b1[25:30, 2:] = b1[25:30, :2] - 1                            # inverted
    b2 = np.concatenate([b1[::7], np.concatenate([b1[::5, 2:4], b1[::5, 2:4] + 9], 1)]).astype(np.float32)  # touching
    for x, y in [(b1, b2), (b2, b1), (b1[:1], b2), (b1, b2[:1]), (b1[:777], b2[:129])]:
        got = core.bbox_overlaps(_t(x), _t(y)).cpu().numpy()
        want = bbox_overlaps(x, y)
        assert np.array_equal(got, want)
        nz = want != 0
        assert nz.sum() > 0 and np.array_equal(got[nz].view(np.int32), want[nz].view(np.int32))
        assert not np.signbit(got[~nz]).any()                    # the library writes +0.0
    assert core.bbox_overlaps(_t(b1[:0]), _t(b2)).shape == (0, len(b2))


# ---------------------------------------------------------------------------------------------- fused == materialised
@pytest.mark.parametrize("G", [1, 8, 64, 512, 2048])
def test_fused_equals_materialised_on_the_tile(cuda, G):
    anc = tile_anchors()
    assert anc.shape[0] == 261888
    gt = _t(gt_hbb(G, 40 + G))
    labels = _t(np.random.default_rng(G).integers(1, 16, G).astype(np.int32))
    from rs_detection_b200 import core
    ov = core.bbox_overlaps(gt, anc)
    positives = 0
    for tag, cfg in THRESHOLDS.items():
        for lab in (None, labels):
            want = materialised(gt, anc, cfg, lab, ov=ov)
            got = fused(gt, anc, cfg, lab)
            same(got, want, f"G={G} {tag} labels={lab is not None}")
            positives += int((got[0] > 0).sum())
    assert positives > 0
    del ov
    torch.cuda.empty_cache()


def test_fused_equals_oracle_on_a_small_scene(cuda, oracle):
    levels = [(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]          # a 256^2 tile: 16 368 anchors
    anc = tile_anchors(levels)
    an = anc.cpu().numpy()
    gt = gt_hbb(40, 7, canvas=256, smax=96)
    labels = np.random.default_rng(8).integers(1, 16, 40).astype(np.int32)
    for tag, cfg in THRESHOLDS.items():
        want = oracle_assign(oracle, gt, an, cfg, labels, 0)
        like_oracle(fused(_t(gt), anc, cfg, _t(labels), fill=0), want, tag)
    # more GTs than one shared-memory chunk (1024)
    big = gt_hbb(1500, 9, canvas=256, smax=96)
    for tag, cfg in THRESHOLDS.items():
        like_oracle(fused(_t(big), anc, cfg), oracle_assign(oracle, big, an, cfg), f"G=1500 {tag}")


# ---------------------------------------------------------------------------------------------- edge cases
def _check_all(oracle, gt, an, cfgs, what, labels=None):
    for cfg in cfgs:
        got = fused(_t(gt), _t(an), cfg, None if labels is None else _t(labels))
        like_oracle(got, oracle_assign(oracle, gt, an, cfg, labels), f"{what} {cfg}")
        same(got, materialised(_t(gt), _t(an), cfg, None if labels is None else _t(labels)), f"{what} {cfg}")


def test_duplicates_and_ties(cuda, oracle):
    """Equal GTs (the first maximal GT wins the column; the last low-quality match wins) and equal anchors (the first
    maximal anchor is a GT's argmax)."""
    an = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]).cpu().numpy()
    an = np.concatenate([an[:3000], an[:3000][::-1], an[3000:]]).astype(np.float32)
    gt = gt_hbb(30, 11, canvas=256, smax=96)
    gt = np.concatenate([gt, gt[:10], gt[5:15]]).astype(np.float32)
    gt[3] = an[100]                                          # a GT equal to an anchor: IoU 1
    cfgs = list(THRESHOLDS.values()) + [(0.5, 0.4, 0.0, True, True), (0.5, 0.4, 0.0, True, False)]
    _check_all(oracle, gt, an, cfgs, "duplicates", labels=np.arange(1, len(gt) + 1, dtype=np.int32))


@pytest.mark.parametrize("pos", [0.0, -0.1])
def test_all_zero_columns_with_nonpositive_pos_thr(cuda, oracle, pos):
    """Anchors far from every GT: max 0, argmax GT 0, positive under pos_iou_thr <= 0 (GT 0 misses their strips)."""
    an = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]).cpu().numpy()
    far = an[:2000] + np.float32(5000)
    an = np.concatenate([an, far]).astype(np.float32)
    gt = gt_hbb(20, 13, canvas=256, smax=96)
    cfgs = [(pos, 0.3, 0.3, False, True), (pos, (-1.0, 0.3), 0.3, True, True), (pos, 0.3, 0.3, True, False)]
    _check_all(oracle, gt, an, cfgs, f"pos={pos}")
    got = fused(_t(gt), _t(an), cfgs[0])
    assert (got[0][-2000:] == 1).all() and (got[1][-2000:] == 0).all() and not torch.signbit(got[1][-2000:]).any()


@pytest.mark.parametrize("assign_all", [True, False])
def test_gt_overlapping_nothing_with_min_pos_iou_zero(cuda, oracle, assign_all):
    """gt_max = 0 >= min_pos_iou = 0: under gt_max_assign_all the GT low-quality-matches every IoU-0 anchor, otherwise
    the first anchor; the GT misses almost every strip and must not be skipped."""
    an = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]).cpu().numpy()
    gt = gt_hbb(20, 15, canvas=256, smax=96)
    gt = np.concatenate([gt[:7], [[9000, 9000, 9050, 9040]], gt[7:], [[-800, 40, -700, 90]]]).astype(np.float32)
    cfgs = [(0.7, 0.3, 0.0, True, assign_all), (0.7, (0.0, 0.3), 0.0, True, assign_all), (0.5, 0.5, 0.0, True, assign_all)]
    _check_all(oracle, gt, an, cfgs, f"nothing all={assign_all}")
    got = fused(_t(gt), _t(an), cfgs[0])[0].cpu().numpy()
    assert (got == len(gt)).any()                            # the last zero-max GT took anchors


def test_neg_iou_thr_tuple(cuda, oracle):
    an = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]).cpu().numpy()
    gt = gt_hbb(30, 17, canvas=256, smax=96)
    cfgs = [(0.7, (0.1, 0.3), 0.3, True, True), (0.7, (0.0, 0.0), 0.3, False, True), (0.5, (0.2, 0.6), 0.5, True, False)]
    _check_all(oracle, gt, an, cfgs, "neg tuple")


@pytest.mark.parametrize("n", [1, 31, 255, 257, 1037, 5003])
def test_anchor_counts_off_the_block_size(cuda, oracle, n):
    an = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)]).cpu().numpy()
    an = an[np.random.default_rng(n).permutation(len(an))[:n]]   # scattered: wide strips
    gt = gt_hbb(25, 19, canvas=256, smax=96)
    _check_all(oracle, gt, an, list(THRESHOLDS.values()), f"n={n}")


# ---------------------------------------------------------------------------------------------- masks
def _compacted(gt, anc, cfg, mask, labels, fill):
    n = anc.shape[0]
    idx = mask.nonzero().reshape(-1)
    sub = fused(gt, anc[idx].contiguous(), cfg, labels, fill=fill)
    ref = materialised(gt, anc[idx].contiguous(), cfg, labels, fill=fill)
    same(sub, ref, "compacted fused vs materialised")
    inds = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    mx = torch.zeros((n,), dtype=torch.float32, device="cuda")
    inds[idx], mx[idx] = sub[0], sub[1]
    lab = None
    if labels is not None:
        lab = torch.full((n,), fill, dtype=torch.int32, device="cuda")
        lab[idx] = sub[2]
    return inds, mx, lab


def test_masks_equal_compaction(cuda):
    anc = tile_anchors()
    gt = _t(gt_hbb(64, 21))
    labels = _t(np.random.default_rng(22).integers(1, 16, 64).astype(np.int32))
    border = 0
    inside = ((anc[:, 0] >= -border) & (anc[:, 1] >= -border) & (anc[:, 2] < W.TILE + border) &
              (anc[:, 3] < W.TILE + border))                     # anchor_inside_flags
    rnd = torch.from_numpy(np.random.default_rng(23).random(anc.shape[0]) < 0.6).cuda()
    first_off = inside.clone()
    first_off[:5000] = False                                     # the first valid anchor is not anchor 0
    assert 0 < int(inside.sum()) < anc.shape[0]
    for name, mask in [("border", inside), ("random", rnd), ("late start", first_off)]:
        for tag, cfg in list(THRESHOLDS.items()) + [("zero_min_pos", (0.7, 0.3, 0.0, True, False))]:
            for lab in (None, labels):
                got = fused(gt, anc, cfg, lab, valid=mask, fill=7)
                want = _compacted(gt, anc, cfg, mask, lab, 7)
                same(got, want, f"{name} {tag} labels={lab is not None}")
                assert not torch.signbit(got[1]).any()
    none = torch.zeros(anc.shape[0], dtype=torch.bool, device="cuda")
    inds, mx, lab = fused(gt, anc, THRESHOLDS["rpn"], labels, valid=none, fill=7)
    assert (inds == -1).all() and (mx == 0).all() and (lab == 7).all()


# ---------------------------------------------------------------------------------------------- reproducibility
def test_repeat_graph_and_streams(cuda):
    anc = tile_anchors()
    gts = [_t(gt_hbb(512, 31)), _t(gt_hbb(512, 33))]
    cfg = THRESHOLDS["rpn"]
    labels = _t(np.random.default_rng(34).integers(1, 16, 512).astype(np.int32))
    direct = [fused(g, anc, cfg, labels) for g in gts]
    same(fused(gts[0], anc, cfg, labels), direct[0], "second run")

    # CUDA graph: capture once, replay on new GTs (the keys must be re-initialised by the replay itself)
    static_gt = gts[0].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fused(static_gt, anc, cfg, labels)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fused(static_gt, anc, cfg, labels)
    for k in (0, 1, 0):
        static_gt.copy_(gts[k])
        graph.replay()
        torch.cuda.synchronize()
        same(out, direct[k], f"graph replay {k}")

    # two streams at once, each with its own workspace (core's scratch is per stream)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    res = {}
    for _ in range(3):
        with torch.cuda.stream(s1):
            res[1] = fused(gts[0], anc, cfg, labels)
        with torch.cuda.stream(s2):
            res[2] = fused(gts[1], anc, cfg, labels)
        torch.cuda.synchronize()
        same(res[1], direct[0], "stream 1")
        same(res[2], direct[1], "stream 2")


# ---------------------------------------------------------------------------------------------- the mirror
def test_max_iou_assigner_bbox_overlaps2d(cuda, oracle):
    from rs_detection_b200.jdet.models.boxes.assigner import MaxIoUAssigner
    anc = tile_anchors([(64, 64), (32, 32), (16, 16), (8, 8), (4, 4)])
    an = anc.cpu().numpy()
    gt = gt_hbb(24, 41, canvas=256, smax=96)
    labels = np.random.default_rng(42).integers(1, 16, 24).astype(np.int32)
    scored = np.concatenate([gt, np.ones((24, 1), np.float32)], 1)      # a score column is dropped
    for kw in (dict(pos_iou_thr=0.7, neg_iou_thr=0.3, min_pos_iou=0.3, match_low_quality=True),
               dict(pos_iou_thr=0.7, neg_iou_thr=0.3, min_pos_iou=0.3, match_low_quality=True, gt_max_assign_all=False),
               dict(pos_iou_thr=0.5, neg_iou_thr=(0.1, 0.5), min_pos_iou=0.5, match_low_quality=False)):
        a = MaxIoUAssigner(**kw, iou_calculator=dict(type='BboxOverlaps2D'))
        cfg = (kw["pos_iou_thr"], kw["neg_iou_thr"], kw["min_pos_iou"], kw["match_low_quality"],
               kw.get("gt_max_assign_all", True))
        want = oracle_assign(oracle, gt, an, cfg, labels, 0)
        for g in (_t(gt), _t(scored)):
            r = a.assign(anc, g, gt_labels=_t(labels))
            assert r.num_gts == 24
            like_oracle((r.gt_inds, r.max_overlaps, r.labels), want, str(kw))
        r = a.assign(torch.from_numpy(an), torch.from_numpy(gt), gt_labels=torch.from_numpy(labels))   # host tensors
        assert not r.gt_inds.is_cuda
        like_oracle((r.gt_inds, r.max_overlaps, r.labels), want, f"host {kw}")
