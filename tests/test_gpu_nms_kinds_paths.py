"""The polygon, merge and horizontal NMS kinds of `csrc/nms.cu` on every dispatch path, against the oracle, exactly.

`rsdet_nms` runs POLY (`poly_nms`), MERGE (`py_cpu_nms_poly_fast`), HBB (merge.py `nms`), HBB_P1_F64 (`py_cpu_nms`)
and HBB_P1 (`jt.nms`) through the same `nms_run` as the rotated kinds.  The rows, and the condition in `nms.cu` that
selects each one:

  row                             taken when
  staged                          a label group of fewer than kCoopMinBlocks = 128 blocks of 64 boxes (nms.cu:567):
                                  `reduce_ov_staged_kernel<2,true>` (nms.cu:2058)
  cooperative                     a group of >= 8129 boxes: cooperative `reduce_kernel`, launched when the call has
                                  ceil(n / 64) >= 128 (nms.cu:2061); it skips the small groups (`skip_small = 1`)
  mixed                           a labelled call with staged groups and a cooperative group: both kernels share it
  many segments                   more than kFastSegs = 2048 label groups: the chunked-scan branch of
                                  `segment_table_kernel` (nms.cu:296)
  sparse                          MERGE with n >= kSparseMinBoxes = 8192 (nms.cu:1420, 1989): sweep, candidate graph and
                                  fixed-point resolve; 16 more launches (nms.cu:2045)
  sparse many segments            the sparse path over more than 2048 groups
  sparse crowd fallback           a crowded group makes the sweep's visit estimate exceed kSparseMaxVisits per box
                                  (nms.cu:1585): the gate opens and the dense kernels take the whole call
  sparse per-label zero fallback  a per-label threshold at which an IoU of 0 suppresses: `sp_keys_kernel` opens the
                                  gate (nms.cu:1531)
  per-label thresholds            `thr_per_label`; labels outside [0, num_thr) use the scalar thr (nms.cu:342)
  all pairs                       a group whose threshold suppresses an IoU of 0 (`zero_suppressed`: thr < 0, or thr <= 0
                                  for HBB): `mask_tiles_kernel<KIND, true>` sends every pair to the exact predicate
                                  (nms.cu:484), and a scalar such threshold skips the sparse path (nms.cu:1988-1989)

Every case asserts the launches its path adds (16 for the sparse path, 1 for the cooperative scan) over the same call on
two boxes.  Keep lists are compared with `oracle.poly_nms`, `py_cpu_nms_poly_fast(stable_ties=True)` (once per group),
`hbb_nms(stable_ties=True)`, `py_cpu_nms` and `jt_nms`.  Ties: the float64 kinds put the higher index first, POLY and
HBB_P1 (and the rotated kinds) the lower index first; -0.0 and +0.0 tie.
"""
import numpy as np
import pytest
import torch

import workloads as W
from rs_detection_b200._lib import (NMS_HBB, NMS_HBB_P1, NMS_HBB_P1_F64, NMS_MERGE, NMS_POLY, NMS_ROTATED,
                                    NMS_ROTATED_GE)

gpu = pytest.mark.gpu             # the case-table test runs without a device

DISPATCH = (
    "staged", "cooperative", "mixed", "many segments", "sparse", "sparse many segments", "sparse crowd fallback",
    "sparse per-label zero fallback", "per-label thresholds", "all pairs",
)
NAMES = {NMS_POLY: "poly", NMS_MERGE: "merge", NMS_HBB: "hbb", NMS_HBB_P1_F64: "hbb_p1_f64", NMS_HBB_P1: "hbb_p1",
         NMS_ROTATED: "rotated", NMS_ROTATED_GE: "rotated_ge"}
KINDS = (NMS_POLY, NMS_MERGE, NMS_HBB, NMS_HBB_P1_F64, NMS_HBB_P1)
F64 = (NMS_MERGE, NMS_HBB, NMS_HBB_P1_F64)
USUAL = {NMS_POLY: 0.1, NMS_MERGE: 0.1, NMS_HBB: 0.5, NMS_HBB_P1_F64: 0.3, NMS_HBB_P1: 0.7, NMS_ROTATED: 0.1,
         NMS_ROTATED_GE: 0.1}
ZERO_THR = {k: (0.0 if k in (NMS_HBB, NMS_ROTATED_GE) else -0.1) for k in NAMES}   # a threshold at which IoU 0 suppresses
THRESHOLDS = (-0.1, 0.0, 1e-12, "usual", 1.0, 1.5)
COOP_MIN = 8129                    # ceil(n / 64) >= kCoopMinBlocks
SPARSE_MIN = 8192                  # kSparseMinBoxes (MERGE)
SPARSE_LAUNCHES = 16


# ------------------------------------------------------------------------------------------ path model
def zero_suppressed(kind, thr):
    """Traits<KIND>::zero_suppressed: does the kind's rule suppress a pair of IoU 0 at this threshold?"""
    if kind in (NMS_ROTATED, NMS_POLY):
        return bool(np.float32(0) > np.float32(thr))
    if kind == NMS_ROTATED_GE:
        return bool(np.float32(0) >= np.float32(thr))
    if kind == NMS_HBB:
        return not (0.0 < thr)
    if kind == NMS_HBB_P1:
        return 0.0 > thr
    return not (0.0 <= thr)                                      # MERGE, HBB_P1_F64


def group_thr(label, thr, tpl):
    """segment_table_kernel (nms.cu:339-343): thr_per_label[label] for 0 <= label < num_thr, the scalar thr otherwise."""
    return float(tpl[label]) if tpl is not None and 0 <= label < len(tpl) else thr


def crowd_opens_gate(n, crowd):
    """A group of `crowd` boxes that all contain one point: every later box of the same (group, y band) run is visited
    by the sweep, and the y1 of such boxes span at most two bands, so the visits are at least crowd^2 / 4."""
    return crowd * crowd / 4 > 640 * n + 4096


def kinds_path(kind, sizes, label_values, thr, tpl=None, crowd=0):
    """(rows of DISPATCH, launches over the two-box call).  label_values None: an unlabelled call of one group."""
    n = int(sum(sizes))
    labelled = label_values is not None
    thrs = [group_thr(int(l), thr, tpl if labelled else None) for l in (label_values if labelled else [0])]
    zero = [zero_suppressed(kind, t) for t in thrs]
    per_label = labelled and tpl is not None
    sparse = kind == NMS_MERGE and n >= SPARSE_MIN and not (not per_label and zero_suppressed(kind, thr))
    coop_launch = -(-n // 64) >= 128
    rows = set()
    resolved = sparse
    if sparse and crowd_opens_gate(n, crowd):
        rows.add("sparse crowd fallback")
        resolved = False
    if sparse and any(zero):
        rows.add("sparse per-label zero fallback")
        resolved = False
    if resolved:
        rows.add("sparse")
        if len(sizes) > 2048:
            rows.add("sparse many segments")
    else:
        big = [s for s in sizes if s >= COOP_MIN]
        if len(big) < len(sizes):
            rows.add("staged")
        if big:
            rows.add("cooperative")
            if labelled and len(big) < len(sizes):
                rows.add("mixed")
        if any(zero):
            rows.add("all pairs")
    if labelled and len(sizes) > 2048:
        rows.add("many segments")
    if per_label:
        rows.add("per-label thresholds")
    return rows, SPARSE_LAUNCHES * sparse + coop_launch


# ------------------------------------------------------------------------------------------ inputs
def clustered_obb(n, seed, crowd=False):
    """(n,5) float32 boxes in clusters of ~24 on a grid of 80 px: every cluster suppresses down to a few boxes, so the
    oracles' greedy loops stay short.  crowd: every box contains the point (500, 500)."""
    rng = np.random.default_rng(seed)
    if crowd:
        c = 500 + rng.uniform(-3, 3, (n, 2))
        wh = rng.uniform(20, 60, (n, 2))
    else:
        k = max(1, n // 24)
        g = int(np.ceil(np.sqrt(k)))
        centres = np.stack([np.arange(k) % g, np.arange(k) // g], 1) * 80.0 + 40
        spread = rng.uniform(1, 10, k)
        cid = rng.integers(0, k, n)
        c = centres[cid] + rng.normal(0, 1, (n, 2)) * spread[cid, None]
        wh = rng.uniform(14, 40, (k, 2))[cid] * rng.uniform(0.8, 1.25, (n, 2))
    th = rng.uniform(-np.pi / 2, np.pi / 2, n)
    return np.concatenate([c, wh, th[:, None]], 1).astype(np.float32)


def kind_dets(kind, obb):
    if kind in (NMS_ROTATED, NMS_ROTATED_GE):
        return obb
    if kind in (NMS_POLY, NMS_MERGE):
        p = W.obb_to_poly64(obb)
        return p.astype(np.float32) if kind == NMS_POLY else p
    o = obb.astype(np.float64)
    h = np.round(np.stack([o[:, 0] - o[:, 2] / 2, o[:, 1] - o[:, 3] / 2, o[:, 0] + o[:, 2] / 2, o[:, 1] + o[:, 3] / 2], 1) * 4) / 4
    return h.astype(np.float32) if kind == NMS_HBB_P1 else h


def make_scores(n, seed, mode, kind):
    rng = np.random.default_rng(seed + 7)
    if mode == "quantised":            # text-format scores (four decimals) plus signed zeros: many ties
        s = np.round(rng.uniform(0, 1, n), 4)
        z = rng.uniform(size=n)
        s[z < 0.05] = 0.0
        s[(z >= 0.05) & (z < 0.1)] = -0.0
    else:
        s = W.distinct_scores(n, seed)
    return s.astype(np.float64 if kind in F64 else np.float32)


def make_case(kind, sizes, label_values, seed, scores="distinct", crowd=0):
    """Boxes of group g come from their own clustered scene (crowd: the first group is a crowd of that size); rows of
    all groups are shuffled together."""
    parts = [clustered_obb(s, seed + 101 * g, crowd=(g == 0 and crowd > 0)) for g, s in enumerate(sizes)]
    obb = np.concatenate(parts)
    n = obb.shape[0]
    perm = np.random.default_rng(seed + 3).permutation(n)
    dets = np.ascontiguousarray(kind_dets(kind, obb)[perm])
    s = make_scores(n, seed, scores, kind)
    labels = None
    if label_values is not None:
        labels = np.repeat(np.asarray(label_values, np.int32), sizes)[perm]
    return dets, s, labels


# ------------------------------------------------------------------------------------------ reference
def global_order(kind, scores):
    """Descending score, ties by the kind's rule: higher index first for the float64 kinds, lower index first else."""
    if kind in F64:
        return np.argsort(scores, kind="stable")[::-1]
    return np.argsort(-scores.astype(np.float64), kind="stable")


def oracle_group(O, kind, dets, scores, thr):
    """Kept local indices of ONE group, from the oracle of the kind."""
    if kind == NMS_POLY:
        return np.asarray(O.poly_nms(np.concatenate([dets, scores[:, None]], 1), thr), np.int64)
    if kind == NMS_MERGE:
        return np.asarray(O.py_cpu_nms_poly_fast(np.concatenate([dets, scores[:, None]], 1), thr, stable_ties=True), np.int64)
    if kind == NMS_HBB:
        return np.asarray(O.hbb_nms(np.concatenate([dets, scores[:, None]], 1), thr, stable_ties=True), np.int64)
    if kind == NMS_HBB_P1_F64:
        return np.asarray(O.py_cpu_nms(np.concatenate([dets, scores[:, None]], 1), thr), np.int64)
    if kind == NMS_HBB_P1:
        return np.asarray(O.jt_nms(np.concatenate([dets, scores[:, None]], 1).astype(np.float32), thr), np.int64)
    order = O._argsort_desc(scores)
    keep = O.nms_rotated_keep(dets, order, thr, 5, kind == NMS_ROTATED_GE)
    return order[keep[order]].astype(np.int64)


def reference(O, kind, dets, scores, thr, labels=None, tpl=None):
    """Kept original indices in the call's descending-score order."""
    n = scores.shape[0]
    kept = np.zeros(n, bool)
    if labels is None:
        kept[oracle_group(O, kind, dets, scores, thr)] = True
    else:
        for l in np.unique(labels):
            sel = np.flatnonzero(labels == l)
            kept[sel[oracle_group(O, kind, dets[sel], scores[sel], group_thr(int(l), thr, tpl))]] = True
    order = global_order(kind, scores)
    return order[kept[order]].astype(np.int64)


# ------------------------------------------------------------------------------------------ engine calls
def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run(kind, dets, scores, thr, labels=None, tpl=None):
    """core.nms -> (kept indices in score order, launches of the call)."""
    from rs_detection_b200 import _lib, core
    d, s, l, t = _t(dets), _t(scores), _t(labels), _t(None if tpl is None else np.asarray(tpl, np.float64))
    l0 = _lib.launch_count()
    res = core.nms(kind, d, s, thr, labels=l, thr_per_label=t, want_mask=False, want_sorted=False, want_score=True)
    launches = _lib.launch_count() - l0
    return res.score_idx.cpu().numpy(), launches


def check_case(O, kind, dets, scores, thr, labels=None, tpl=None, crowd=0, sizes=None, label_values=None, want_rows=()):
    n = scores.shape[0]
    rows, extra = kinds_path(kind, sizes or [n], label_values, thr, tpl, crowd)
    for r in want_rows:
        assert r in rows, (r, rows)
    _, base = run(kind, dets[:2], scores[:2], thr, None if labels is None else labels[:2], tpl)
    got, launches = run(kind, dets, scores, thr, labels, tpl)
    assert launches == base + extra, (launches, base, extra, sorted(rows))
    want = reference(O, kind, dets, scores, thr, labels, tpl)
    print(f"{NAMES[kind]} n={n} thr={thr}: {want.size} kept, rows {sorted(rows)}")
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.array_equal(got, want)
    return got


# ------------------------------------------------------------------------------------------ case table
def _neg_labels(g):
    """g distinct label values, half of them negative, not contiguous"""
    return (np.arange(g) - g // 2) * 3 - 1


def _cases():
    cases = []   # id, kind, sizes, label values (None: unlabelled), thr ("usual" or a number), tpl, scores, crowd, row
    for k in KINDS:
        nm = NAMES[k]
        for n in (1, 63, 64, 65, 3000):
            cases.append((f"{nm}_staged_{n}", k, [n], None, "usual", None, "distinct", 0, "staged"))
        for n in (8128, 8129):
            cases.append((f"{nm}_unlabelled_{n}", k, [n], None, "usual", None, "distinct", 0,
                          "cooperative" if n >= COOP_MIN else "staged"))
        if k == NMS_MERGE:        # n >= 8192 is sparse: a crowd sends the mixed call back to the dense kernels
            cases.append((f"{nm}_mixed_crowd", k, [8200] + [40] * 30, list(range(31)), "usual", None, "distinct", 8200,
                          "mixed"))
            cases.append((f"{nm}_sparse_9000", k, [9000], None, "usual", None, "distinct", 0, "sparse"))
            cases.append((f"{nm}_sparse_2100_groups", k, [4] * 2100, list(_neg_labels(2100)), "usual", None, "distinct",
                          0, "sparse many segments"))
            cases.append((f"{nm}_sparse_per_label", k, [1200] * 8, list(range(-2, 6)), "usual",
                          [0.1, 0.05, 0.3, 0.2], "distinct", 0, "sparse"))
            cases.append((f"{nm}_sparse_per_label_zero", k, [1200] * 8, list(range(-2, 6)), "usual",
                          [0.1, 0.05, 0.3, ZERO_THR[k]], "distinct", 0, "sparse per-label zero fallback"))
            cases.append((f"{nm}_sparse_quantised", k, [9000], None, "usual", None, "quantised", 0, "sparse"))
        else:
            cases.append((f"{nm}_mixed", k, [8200] + [40] * 30, list(range(31)), "usual", None, "distinct", 0, "mixed"))
        for g in (2048, 2049):
            cases.append((f"{nm}_groups_{g}", k, [3] * g, list(_neg_labels(g)), "usual", None, "distinct", 0,
                          "many segments" if g > 2048 else "staged"))
        cases.append((f"{nm}_per_label", k, [200] * 8, list(range(-2, 6)), "usual", [USUAL[k], 0.05, 0.3, ZERO_THR[k]],
                      "distinct", 0, "per-label thresholds"))
        cases.append((f"{nm}_ties_staged", k, [3000], None, "usual", None, "quantised", 0, "staged"))
        cases.append((f"{nm}_ties_coop", k, [8150], None, "usual", None, "quantised", 0, "cooperative"))
        cases.append((f"{nm}_ties_labelled", k, [3000, 500, 20], [7, -3, 0], "usual", None, "quantised", 0, "staged"))
        for thr in THRESHOLDS:
            cases.append((f"{nm}_thr_{thr}", k, [300, 200, 100], [0, 1, 2], thr, None, "distinct", 0, "staged"))
        for thr in (-0.1, 0.0):
            cases.append((f"{nm}_coop_thr_{thr}", k, [8150], None, thr, None, "distinct", 0,
                          "all pairs" if zero_suppressed(k, thr) else "cooperative"))
    for k in (NMS_ROTATED, NMS_ROTATED_GE):
        for thr in THRESHOLDS:
            cases.append((f"{NAMES[k]}_thr_{thr}", k, [300, 200, 100], [0, 1, 2], thr, None, "distinct", 0, "staged"))
    return cases


CASES = _cases()


def _resolve(k, thr):
    return USUAL[k] if thr == "usual" else thr


# ------------------------------------------------------------------------------------------ tests
def test_case_table_covers_every_row():
    covered = set()
    for cid, k, sizes, lv, thr, tpl, _, crowd, row in CASES:
        rows, _ = kinds_path(k, sizes, lv, _resolve(k, thr), tpl, crowd)
        assert row in rows, (cid, row, rows)
        covered |= rows
    assert covered == set(DISPATCH), sorted(set(DISPATCH) - covered)
    # the model's edges
    assert kinds_path(NMS_HBB, [8128], None, 0.5)[1] == 0 and kinds_path(NMS_HBB, [8129], None, 0.5)[1] == 1
    assert kinds_path(NMS_MERGE, [8191], None, 0.1)[1] == 1 and kinds_path(NMS_MERGE, [8192], None, 0.1)[1] == 17
    assert kinds_path(NMS_MERGE, [8192], None, -0.1) == ({"cooperative", "all pairs"}, 1)
    assert zero_suppressed(NMS_HBB, 0.0) and not zero_suppressed(NMS_HBB_P1_F64, 0.0)
    assert zero_suppressed(NMS_ROTATED_GE, 0.0) and not zero_suppressed(NMS_ROTATED, 0.0)
    assert not zero_suppressed(NMS_ROTATED_GE, 1e-12) and not zero_suppressed(NMS_HBB, 1e-12)


@gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_path(cuda, oracle, case):
    cid, k, sizes, lv, thr, tpl, scores, crowd, row = case
    dets, s, labels = make_case(k, sizes, lv, seed=len(cid) * 1009 + sum(sizes) % 997, scores=scores, crowd=crowd)
    check_case(oracle, k, dets, s, _resolve(k, thr), labels, tpl, crowd, sizes, lv, want_rows=(row,))


@gpu
@pytest.mark.parametrize("kind", KINDS, ids=[NAMES[k] for k in KINDS])
def test_staged_equals_cooperative(cuda, kind):
    """8128 boxes (the staged scan) and 8129 (the cooperative one, the last box far from every other): the first 8128
    rows keep the same boxes, in the same order."""
    dets, s, _ = make_case(kind, [8129], None, seed=77)
    far = kind_dets(kind, np.array([[1e5, 1e5, 20, 20, 0.3]], np.float32))
    dets[-1] = far[0]
    a, la = run(kind, dets[:-1], s[:-1], USUAL[kind])
    b, lb = run(kind, dets, s, USUAL[kind])
    assert lb == la + 1
    assert np.array_equal(b[b != 8128], a)


@gpu
def test_merge_dense_equals_sparse(cuda):
    """8191 boxes run the dense engine, 8192 the sparse path: the same keep list, bit for bit, when the extra box
    overlaps nothing."""
    dets, s, _ = make_case(NMS_MERGE, [8192], None, seed=78)
    dets[-1] = kind_dets(NMS_MERGE, np.array([[1e5, 1e5, 20, 20, 0.3]], np.float32))[0]
    a, la = run(NMS_MERGE, dets[:-1], s[:-1], 0.1)
    b, lb = run(NMS_MERGE, dets, s, 0.1)
    assert lb == la + SPARSE_LAUNCHES
    assert np.array_equal(b[b != 8191], a)


# ------------------------------------------------------------------------------------------ degenerate boxes
HBB_DEGENERATE = np.array([
    [0, 0, 10, 10], [10, 0, 20, 10],                 # touching: x2 == x1' exactly
    [30, 0, 40, 10], [40.5, 0, 50, 10],              # a gap below one pixel: the "+1" boxes overlap
    [60, 0, 70, 10], [71, 0, 80, 10],                # a gap of one pixel: the "+1" boxes touch
    [100, 0, 100, 10], [100, 0, 100, 10],            # zero width
    [120, 5, 120, 5], [120, 5, 120, 5],              # zero width and height
    [150, 0, 140, 10], [150, 0, 140, 10],            # negative width
    [200, 0, 199, 10], [300, 0, 299, 10],            # "+1" areas 0 and 0: 0/0 for the "+1" kinds
    [400, 0, 401, 1], [500, 0, 497, 1],              # "+1" areas 4 and -4
    [600, 0, 620, 20], [600, 0, 620, 20], [600, 0, 620, 20],   # identical
    [700, 0, 720, 20], [690, -5, 730, 30],           # nested
], np.float64)


def _degenerate(kind):
    if kind in (NMS_POLY, NMS_MERGE):
        obb = np.array([[10, 10, 20, 20, 0], [30, 10, 20, 20, 0],           # squares sharing an edge
                        [60, 10, 0, 20, 0.3], [60, 10, 0, 20, 0.3],         # zero width
                        [90, 10, 0, 0, 0], [90, 10, 0, 0, 0],               # points
                        [120, 10, 20, 8, 0.4], [120, 10, 20, 8, 0.4], [120, 10, 20, 8, 0.4],   # identical
                        [150, 10, 30, 30, 0], [150, 10, 10, 10, 0.7],       # nested
                        [180, 10, -10, 20, 0.2], [180, 10, 10, 20, 0.2]], np.float32)   # negative width
        return kind_dets(kind, obb)
    return HBB_DEGENERATE.astype(np.float32 if kind == NMS_HBB_P1 else np.float64)


@gpu
@pytest.mark.parametrize("thr", [0.3, 1e-12, 0.0, 1.0])
@pytest.mark.parametrize("kind", KINDS, ids=[NAMES[k] for k in KINDS])
def test_degenerate_boxes(cuda, oracle, kind, thr):
    """Touching, sub-pixel gaps, zero and negative widths, zero "+1" area sums, identical and nested boxes, with tied
    scores; unlabelled, and labelled in three groups of neighbouring rows."""
    d = _degenerate(kind)
    s = (np.arange(d.shape[0]) % 3 / 4).astype(np.float64 if kind in F64 else np.float32)
    check_case(oracle, kind, d, s, thr)
    lab = ((np.arange(d.shape[0]) // 4) % 3).astype(np.int32)
    check_case(oracle, kind, d, s, thr, lab, sizes=list(np.bincount(lab)), label_values=[0, 1, 2])


# ------------------------------------------------------------------------------------------ C ABI outputs
@gpu
@pytest.mark.parametrize("kind", [NMS_POLY, NMS_HBB_P1_F64], ids=["poly", "hbb_p1_f64"])
def test_null_output_combinations(cuda, oracle, kind):
    """All 16 NULL / non-NULL combinations of keep_mask, keep_sorted_idx, keep_score_idx and num_keep, on a workspace
    filled with 0xFF before every call: each output that is asked for matches the oracle."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    sizes, lv = [1500, 900, 40, 1], [3, -1, 0, 9]
    dets, s, labels = make_case(kind, sizes, lv, seed=90, scores="quantised")
    n = s.shape[0]
    thr = USUAL[kind]
    want = reference(oracle, kind, dets, s, thr, labels)
    mask_want = np.zeros(n, np.uint8)
    mask_want[want] = 1
    d, sc, lab = _t(dets), _t(s), _t(labels)
    wsb = L.rsdet_nms_workspace_bytes(kind, n)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    for combo in range(16):
        ws.fill_(0xFF)
        km = torch.full((n,), 0x7F, dtype=torch.uint8, device="cuda") if combo & 1 else None
        ks = torch.full((n,), -5, dtype=torch.int64, device="cuda") if combo & 2 else None
        kc = torch.full((n,), -5, dtype=torch.int64, device="cuda") if combo & 4 else None
        nk = torch.full((1,), -5, dtype=torch.int32, device="cuda") if combo & 8 else None
        p = lambda t: 0 if t is None else t.data_ptr()
        rc = L.rsdet_nms(kind, d.data_ptr(), sc.data_ptr(), lab.data_ptr(), n, thr, None, 0, p(km), p(ks), p(kc), p(nk),
                         ws.data_ptr(), wsb, _lib.stream_ptr())
        assert rc == 0, (combo, rc)
        k = want.size
        if km is not None:
            assert np.array_equal(km.cpu().numpy(), mask_want), combo
        if ks is not None:
            assert np.array_equal(ks.cpu().numpy()[:k], np.sort(want)), combo
        if kc is not None:
            assert np.array_equal(kc.cpu().numpy()[:k], want), combo
        if nk is not None:
            assert int(nk.item()) == k, combo


# ------------------------------------------------------------------------------------------ thresholds
@gpu
@pytest.mark.parametrize("thr", [0.0, 1e-12, 0.1, 1.0, 1.5])
@pytest.mark.parametrize("engine", ["fast", "generic"])
def test_multiclass_thresholds(cuda, oracle, engine, thr):
    from rs_detection_b200 import core
    n, C = 300, 3
    mb = clustered_obb(n, 91)
    ms = W.class_scores(n, C, 92)
    box = mb if engine == "fast" else np.tile(mb, (1, C + 1))
    wd, wl = oracle.multiclass_nms_rotated(mb, ms, 0.05, dict(iou_thr=thr), 10 ** 6)
    d, lab, cnt = core.multiclass_nms_rotated(_t(box), _t(ms), 0.05, thr, 10 ** 6)
    k = int(cnt.item())
    assert np.array_equal(d[:k].cpu().numpy().view(np.int32), wd.view(np.int32)) and np.array_equal(lab[:k].cpu().numpy(), wl)


@gpu
@pytest.mark.parametrize("engine", ["fast", "generic"])
def test_multiclass_negative_iou_thr_refused(cuda, engine):
    """iou_thr < 0 would suppress disjoint pairs, which the decision matrix never evaluates: RSDET_EINVAL."""
    from rs_detection_b200 import core
    n, C = 50, 2
    mb = clustered_obb(n, 93)
    box = mb if engine == "fast" else np.tile(mb, (1, C + 1))
    with pytest.raises(ValueError):
        core.multiclass_nms_rotated(_t(box), _t(W.class_scores(n, C, 94)), 0.05, -0.1, 100)


@gpu
@pytest.mark.parametrize("kind", [NMS_ROTATED, NMS_ROTATED_GE], ids=["rotated", "rotated_ge"])
def test_rotated_zero_threshold_skips_sparse(cuda, oracle, kind):
    """An unlabelled rotated call of 32768 boxes takes the sparse path, except at a threshold where IoU 0 suppresses:
    then the dense kernels evaluate every pair and each box suppresses every later one."""
    thr = ZERO_THR[kind]
    dets = W.rotated_boxes(32768, 95, canvas=2048, smin=8, smax=128)
    s = W.distinct_scores(32768, 95)
    _, base = run(kind, dets[:2], s[:2], thr)
    got, launches = run(kind, dets, s, thr)
    assert launches == base + 1                      # cooperative scan, no sparse path
    assert np.array_equal(got, reference(oracle, kind, dets, s, thr)) and got.size == 1
