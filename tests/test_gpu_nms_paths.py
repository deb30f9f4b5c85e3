"""Every dispatch path of the rotated NMS engine (`csrc/nms.cu`) against the oracle, bit for bit.

`rsdet_multiclass_nms_rotated` and `rsdet_nms` pick their kernels from n (boxes), C (classes), the box layout
(`bbox_dim` 5: one box per row shared by every class; 5(C+1): one box per class), the per-class candidate counts and
the labels.  The paths, as `nms.cu` selects them (DESIGN.md §4.4):

  row                                  taken when
  fast pipe<1>                         bbox_dim 5, n <= 4096, C <= 4096: `reduce_ov_pipe_kernel<1,512>`
  fast pipe<2>                         4097 <= n <= 8128 (three row buffers fit 227 KB)
  fast staged<2>                       8129 <= n <= 8192: `reduce_ov_staged_kernel<2,false>`
  fast classes > scan CTAs             C > 148: a scan CTA takes several classes
  fast class-sort sizes                `mc_class_sort_kernel` networks of P < 64, 64, 128..1024, 2048 and > 2048 keys
  matrix split                         `mask_cap > used + flag_words + 4096` (C >= 2 in practice): filter -> pair queue ->
                                       clip -> flagged tiles
  matrix unsplit                       otherwise (C = 1 in most cases): `ov_tiles_kernel` over every tile
  generic shared reduce_ov             bbox_dim 5, n > 8192 (so C <= 127): `reduce_ov_kernel`
  generic shared segment_table         bbox_dim 5, C > 4096 (so n <= 256): no class counts, `segment_table_kernel`
  generic per-class staged             bbox_dim 5(C+1): `reduce_ov_staged_kernel<2,true>`
  generic per-class cooperative        a class with >= 8129 candidates: cooperative `reduce_kernel`
  many segments                        more than 2048 label groups of a rotated kind: the chunked-scan branch of
                                       `segment_table_kernel`
  ge dense cooperative                 `NMS_ROTATED_GE` (`nms_rotated_cpu`) with n >= 8129 on the dense engine
  sparse unlabelled                    unlabelled rotated kinds with n >= 32768 (checked at 32767 / 32768 against the
                                       dense engine)

Every case asserts the path it is meant to reach: the fast path counts 8 launches (10 with a split matrix) and the
generic engine more; `expected_path` mirrors the conditions of `nms.cu` for the rest.  Multiclass calls with more
candidates than the oracle's all-pairs `ml_nms_rotated` can take go through `per_class_reference`, which runs the
oracle's NMS on each class alone.  Replicating a class-agnostic box into every class column forces the generic
per-class engine on the same problem, so the engines are also compared with each other, bit for bit.

-0.0 and +0.0 scores compare equal and tie: the lower index comes first in the fp32 kinds (the higher index in the
float64 merge kinds), as in the oracle's stable sorts.
"""
import functools
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import workloads as W
from rs_detection_b200._lib import NMS_HBB, NMS_ROTATED, NMS_ROTATED_GE

pytestmark = pytest.mark.gpu

DISPATCH = (
    "fast pipe<1>", "fast pipe<2>", "fast staged<2>", "fast classes > scan CTAs", "fast class-sort sizes",
    "matrix split", "matrix unsplit", "generic shared reduce_ov", "generic shared segment_table",
    "generic per-class staged", "generic per-class cooperative", "many segments", "ge dense cooperative",
    "sparse unlabelled",
)
IOU_THR = 0.1
FAST_LAUNCHES = 8                  # mc_fast_run's count_launch(8); launch_ov_matrix adds 2 when it splits


# ------------------------------------------------------------------------------------------ path model
def _matrix_split(n, C):
    """launch_ov_matrix (nms.cu:1805-1815) with mask_cap = mc_mask_words(n, C) (nms.cu:2500-2503)."""
    tov = -(-n // 64)
    pitch = (tov + 1) & ~1
    tiles = tov * (tov + 1) // 2
    mask_cap = max(C, 1) * n * (tov + 1)
    used, flag_words = n * pitch, (tiles + 7) // 8 + 1
    return tiles < (1 << 22) and mask_cap > used + flag_words + 4096


def _sort_size(cnt):
    p = 2                                    # mc_class_sort_kernel (nms.cu:2313-2314)
    while p < cnt:
        p <<= 1
    return p


def expected_path(n, C, bbox_dim, counts):
    """Rows of DISPATCH that `rsdet_multiclass_nms_rotated` takes for these per-class candidate counts.  Mirrors
    mc_fast_ok (nms.cu:2432), mc_fast_run (2478-2492), the use_counts rule (2542), nms_run's shared scan (1937,
    1958-1964) and generic scan (2038-2055), and segment_table_kernel (280)."""
    counts = np.asarray(counts)
    rows = set()
    tov = -(-n // 64)
    ts = tov | 1
    segs = int((counts > 0).sum())
    if bbox_dim == 5 and 1 <= n <= 8192 and C <= 4096:
        piped = 8 * (ts + 3 * 64 * ts) + 4 * n
        if piped + 2048 <= 227 * 1024:
            rows.add("fast pipe<1>" if tov <= 64 else "fast pipe<2>")
        else:
            rows.add("fast staged<2>")
        if C > 148:
            rows.add("fast classes > scan CTAs")
        sizes = {_sort_size(int(c)) for c in counts}
        if (min(sizes) < 64 and 64 in sizes and any(64 < p < 2048 for p in sizes) and 2048 in sizes
                and max(sizes) > 2048):
            rows.add("fast class-sort sizes")
        rows.add("matrix split" if _matrix_split(n, C) else "matrix unsplit")
    elif bbox_dim == 5:
        rows.add("matrix split" if _matrix_split(n, C) else "matrix unsplit")
        staged = 8 * (5 * ts + 2 * 64 * ts) + 4 * n
        if not (tov <= 128 and staged <= 200 * 1024):
            rows.add("generic shared reduce_ov")
        if C > 1024:                                        # kMcHist: no class counts
            rows.add("generic shared segment_table")
            if segs > 2048:
                rows.add("many segments")
    else:
        rows.add("generic per-class staged")
        if counts.max() >= 8129:
            rows.add("generic per-class cooperative")
        if segs > 2048:
            rows.add("many segments")
    return rows


def engine_path(kind, n, num_labels):
    """Rows of DISPATCH that `rsdet_nms` takes: nms_run (nms.cu:1970-1971 sparse, 2043 cooperative scan) and
    segment_table_kernel (280).  num_labels None: an unlabelled call."""
    if num_labels is None and n >= 32768:
        return {"sparse unlabelled"}
    rows = set()
    if num_labels is not None and num_labels > 2048:
        rows.add("many segments")
    if kind == NMS_ROTATED_GE and num_labels is None and -(-n // 64) >= 128:
        rows.add("ge dense cooperative")
    return rows


# ------------------------------------------------------------------------------------------ reference
def per_class_keep(oracle, mb, ms, score_thr, iou_thr, sf=None):
    """`oracle.multiclass_nms_rotated` up to its final sort, one class at a time: (boxes, scores, labels) of the kept
    candidates in expansion order.  A stable sort restricted to one class is that class's stable sort, and the label
    gate makes the NMS independent per class.  The oracle's ctypes calls release the GIL."""
    mb, ms = np.ascontiguousarray(mb, np.float32), np.ascontiguousarray(ms, np.float32)
    n, nc = ms.shape[0], ms.shape[1] - 1
    boxes = mb.reshape(n, -1, 5)[:, 1:] if mb.shape[1] > 5 else np.broadcast_to(mb[:, None], (n, nc, 5))
    scores = ms[:, 1:]
    valid = scores > np.float32(score_thr)
    if sf is not None:
        scores = scores * np.ascontiguousarray(sf, np.float32)[:, None]
    cb, cs, cl = np.ascontiguousarray(boxes[valid]), scores[valid], np.nonzero(valid)[1]
    by_class = np.argsort(cl, kind="stable")
    groups = np.split(by_class, np.flatnonzero(np.diff(cl[by_class])) + 1) if cl.size else []

    def one(sel):
        return sel, oracle.nms_rotated_keep(cb[sel], oracle._argsort_desc(cs[sel]), iou_thr, 5, False)

    keep = np.zeros(cl.shape, bool)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        for sel, k in ex.map(one, groups):
            keep[sel[k]] = True
    return cb[keep], cs[keep], cl[keep]


def apply_max_num(oracle, kept, max_num):
    """The final stable score sort and the `keep.size(0) > max_num` slice of oracle.multiclass_nms_rotated."""
    b, s, l = kept
    if b.shape[0] == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.int32)
    inds = oracle._argsort_desc(s)
    if b.shape[0] > max_num:
        inds = inds[:max_num]
    return np.concatenate([b[inds], s[inds][:, None]], 1), l[inds].astype(np.int32)


def per_class_reference(oracle, mb, ms, score_thr, iou_thr, max_num=-1, sf=None):
    return apply_max_num(oracle, per_class_keep(oracle, mb, ms, score_thr, iou_thr, sf), max_num)


# ------------------------------------------------------------------------------------------ engine calls
def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _mc(mb, ms, score_thr, max_num=-1, sf=None):
    """core.multiclass_nms_rotated -> (dets, labels, launches of the call)."""
    from rs_detection_b200 import _lib, core
    mb_t, ms_t, sf_t = _t(mb), _t(ms), None if sf is None else _t(sf)
    l0 = _lib.launch_count()
    d, lab, cnt = core.multiclass_nms_rotated(mb_t, ms_t, score_thr, IOU_THR, max_num, sf_t)
    launches = _lib.launch_count() - l0
    k = int(cnt.item())
    return d[:k].cpu().numpy(), lab[:k].cpu().numpy(), launches


def _replicate(mb, C):
    """The class-agnostic box in every class column (background included): bbox_dim = 5(C+1)."""
    return np.ascontiguousarray(np.tile(mb, (1, C + 1)))


def _counts(ms, score_thr):
    return (ms[:, 1:] > np.float32(score_thr)).sum(0)


def _same(got, want, what):
    gd, gl = got
    wd, wl = want
    assert gd.shape == wd.shape, f"{what}: {gd.shape} vs {wd.shape}"
    assert np.array_equal(gd.view(np.int32), wd.view(np.int32)), what
    assert np.array_equal(gl, wl), what


# ------------------------------------------------------------------------------------------ inputs
def _uniform_inputs(n, C, seed, frac, factors, canvas=1024):
    """Boxes of 16..160 px; class scores uniform below 0.999, a fraction `frac` above the threshold.  The last box is a
    copy of box 0, which tops every class: whatever the scan reads of the decision matrix's last columns matters."""
    rng = np.random.default_rng(seed)
    mb = W.rotated_boxes(n, seed, canvas=canvas, smin=16, smax=160)
    ms = rng.uniform(0, 0.999, (n, C + 1)).astype(np.float32)
    thr = float(np.float32(1 - frac))
    if n > 1:
        mb[n - 1] = mb[0]
        ms[0, 1:], ms[n - 1, 1:] = 0.9995, 0.9993
    sf = None
    if factors:
        sf = rng.uniform(0.5, 1.0, n).astype(np.float32)
        sf[0] = sf[n - 1] = 1.0
    return mb, ms, sf, thr


FAST_CASES = [   # id, n, C, fraction of candidates above the threshold, score factors, the row the case is for
    ("pipe1_4096", 4096, 3, 0.3, False, "fast pipe<1>"),
    ("pipe2_4097", 4097, 3, 0.3, False, "fast pipe<2>"),
    ("pipe2_4160", 4160, 2, 0.4, True, "fast pipe<2>"),
    ("pipe2_6000", 6000, 4, 0.25, False, "fast pipe<2>"),
    ("pipe2_8128", 8128, 2, 0.4, True, "fast pipe<2>"),
    ("staged_8129", 8129, 2, 0.4, False, "fast staged<2>"),
    ("unsplit_1500", 1500, 1, 0.8, False, "matrix unsplit"),
    ("unsplit_8000", 8000, 1, 0.6, True, "matrix unsplit"),
    ("split_8192_tiny_queue", 8192, 1, 0.9, False, "matrix split"),
    ("classes_149", 1000, 149, 0.05, False, "fast classes > scan CTAs"),
    ("classes_600", 1500, 600, 0.02, True, "fast classes > scan CTAs"),
    ("classes_4096", 256, 4096, 0.02, False, "fast classes > scan CTAs"),
]

SORT_COUNTS = [0, 1, 2, 32, 33, 64, 65, 1024, 1025, 2047, 2048, 2049, 4096, 4097, 8191, 8192]


def _sort_size_inputs(quantised):
    """n = 8192, one class per entry of SORT_COUNTS with exactly that many candidates above 0.45."""
    n, C = 8192, len(SORT_COUNTS)
    rng = np.random.default_rng(20 + quantised)
    mb = W.rotated_boxes(n, 21, canvas=1024, smin=16, smax=160)
    ms = rng.uniform(0, 0.4, (n, C + 1)).astype(np.float32)
    for c, k in enumerate(SORT_COUNTS):
        live = rng.permutation(n)[:k]
        u = rng.uniform(0, 1, k)
        ms[live, c + 1] = 0.5 + (np.floor(u * 8) / 16 if quantised else u * 0.49)   # quantised: 8 levels, many ties
    return mb, ms, None, 0.45


LABELLED_CASES = [   # kind, n, number of distinct labels (None: unlabelled), as the tests below call them
    (NMS_ROTATED, 6000, 2048), (NMS_ROTATED, 6000, 2049), (NMS_ROTATED, 3000, 11), (NMS_ROTATED_GE, 9000, None),
    (NMS_ROTATED, 32767, None), (NMS_ROTATED, 32768, None), (NMS_ROTATED_GE, 32767, None), (NMS_ROTATED_GE, 32768, None),
]

GENERIC_CASES = [   # id, n, C, box layout, the row the case is for
    ("perclass_coop_9000", 9000, 2, "per-class", "generic per-class cooperative"),
    ("perclass_3000_classes", 300, 3000, "per-class", "many segments"),
    ("shared_9000_C1", 9000, 1, "shared", "generic shared reduce_ov"),
    ("shared_9000_C2", 9000, 2, "shared", "generic shared reduce_ov"),
    ("shared_5000_classes", 200, 5000, "shared", "generic shared segment_table"),
]


def _generic_inputs(n, C, layout):
    rng = np.random.default_rng(n + C)
    if layout == "per-class":
        canvas = 1024 if n > 1000 else 256
        mb = W.rotated_boxes(n * (C + 1), n + C, canvas=canvas, smin=16, smax=160).reshape(n, 5 * (C + 1))
    else:
        mb = W.rotated_boxes(n, n + C, canvas=1024, smin=16, smax=160)
    ms = rng.uniform(0, 0.999, (n, C + 1)).astype(np.float32)
    if n > 8192:
        ms[:, 1] = rng.uniform(0.6, 0.999, n)        # class 0: every box is a candidate
        thr = 0.5 if C > 1 else 0.3                  # class 1: about half
    else:
        thr = float(np.float32(0.99))                # 1 % of n x C: more than 2048 non-empty classes
    return mb, ms, None, thr


# ------------------------------------------------------------------------------------------ tests
def test_reference_helper_matches_oracle(oracle):
    """per_class_reference == oracle.multiclass_nms_rotated on inputs small enough for the all-pairs oracle."""
    n, C = 400, 6
    rng = np.random.default_rng(3)
    ms = W.class_scores(n, C, 3)
    sf = rng.uniform(0.5, 1.0, n).astype(np.float32)
    for mb in (W.rotated_boxes(n, 4, canvas=300, smin=16, smax=120),
               W.rotated_boxes(n * (C + 1), 5, canvas=300, smin=16, smax=120).reshape(n, -1)):
        for max_num in (-1, -5, 0, 7, 10 ** 6):
            for f in (None, sf):
                want = oracle.multiclass_nms_rotated(mb, ms, 0.05, dict(iou_thr=IOU_THR), max_num, f)
                got = per_class_reference(oracle, mb, ms, 0.05, IOU_THR, max_num, f)
                _same(got, want, f"max_num={max_num} bbox_dim={mb.shape[1]} factors={f is not None}")
    # nothing above the threshold
    _same(per_class_reference(oracle, mb, ms, 2.0, IOU_THR), (np.zeros((0, 6), np.float32), np.zeros((0,), np.int32)),
          "empty")


def test_case_tables_cover_every_dispatch_row():
    covered = set()
    for _, n, C, frac, factors, row in FAST_CASES:
        mb, ms, _, thr = _uniform_inputs(n, C, n + C, frac, factors)
        rows = expected_path(n, C, 5, _counts(ms, thr))
        assert row in rows, (n, C, row, rows)
        covered |= rows
    for quantised in (False, True):
        mb, ms, _, thr = _sort_size_inputs(quantised)
        rows = expected_path(8192, len(SORT_COUNTS), 5, _counts(ms, thr))
        assert "fast class-sort sizes" in rows
        covered |= rows
    for _, n, C, layout, row in GENERIC_CASES:
        mb, ms, _, thr = _generic_inputs(n, C, layout)
        rows = expected_path(n, C, mb.shape[1], _counts(ms, thr))
        assert row in rows, (n, C, layout, row, rows)
        covered |= rows
        covered |= expected_path(n, C, 5 * (C + 1), _counts(ms, thr))      # the replicated comparison
    for kind, n, labels in LABELLED_CASES:
        covered |= engine_path(kind, n, labels)
    assert engine_path(NMS_ROTATED, 32767, None) == set() and engine_path(NMS_ROTATED_GE, 9000, None)
    assert covered == set(DISPATCH), sorted(set(DISPATCH) - covered)


@pytest.mark.parametrize("case", FAST_CASES, ids=[c[0] for c in FAST_CASES])
def test_fast_path(cuda, oracle, case):
    _, n, C, frac, factors, row = case
    mb, ms, sf, thr = _uniform_inputs(n, C, n + C, frac, factors)
    rows = expected_path(n, C, 5, _counts(ms, thr))
    assert row in rows
    gd, gl, launches = _mc(mb, ms, thr, 10 ** 6, sf)
    assert launches == FAST_LAUNCHES + 2 * ("matrix split" in rows), launches
    want = per_class_reference(oracle, mb, ms, thr, IOU_THR, 10 ** 6, sf)
    print(f"n={n} C={C}: {int(_counts(ms, thr).sum())} candidates, {want[0].shape[0]} kept, {launches} launches")
    _same((gd, gl), want, "fast path vs per-class reference")
    # the same problem through the generic per-class engine
    rd, rl, rlaunches = _mc(_replicate(mb, C), ms, thr, 10 ** 6, sf)
    assert rlaunches > FAST_LAUNCHES + 2, rlaunches
    _same((rd, rl), (gd, gl), "generic per-class engine vs fast path")


@pytest.mark.parametrize("quantised", [False, True], ids=["distinct", "quantised"])
def test_class_sort_sizes(cuda, oracle, quantised):
    """One class per bitonic network size of mc_class_sort_kernel; quantised scores tie inside every class."""
    mb, ms, _, thr = _sort_size_inputs(quantised)
    counts = _counts(ms, thr)
    assert counts.tolist() == SORT_COUNTS
    assert "fast class-sort sizes" in expected_path(8192, len(SORT_COUNTS), 5, counts)
    gd, gl, launches = _mc(mb, ms, thr, 10 ** 6)
    assert launches == FAST_LAUNCHES + 2 * _matrix_split(8192, len(SORT_COUNTS))
    _same((gd, gl), per_class_reference(oracle, mb, ms, thr, IOU_THR, 10 ** 6), "fast path vs per-class reference")
    rd, rl, _ = _mc(_replicate(mb, len(SORT_COUNTS)), ms, thr, 10 ** 6)
    _same((rd, rl), (gd, gl), "generic per-class engine vs fast path")


MAX_NUMS = {"-1": lambda nk: -1, "-2": lambda nk: -2, "-nk": lambda nk: -nk, "-nk-1": lambda nk: -nk - 1, "0": lambda nk: 0,
            "1": lambda nk: 1, "nk-1": lambda nk: nk - 1, "nk": lambda nk: nk, "nk+1": lambda nk: nk + 1,
            "1e6": lambda nk: 10 ** 6}


@functools.lru_cache(maxsize=1)
def _max_num_problem():
    from oracle import oracle as O
    n, C = 1500, 15
    mb = W.rotated_boxes(n, 40, smin=16, smax=160)
    ms = W.class_scores(n, C, 3)
    sf = np.random.default_rng(9).uniform(0.5, 1.0, n).astype(np.float32)
    return mb, ms, sf, per_class_keep(O, mb, ms, 0.05, IOU_THR, sf)


@pytest.mark.parametrize("max_num", list(MAX_NUMS))
@pytest.mark.parametrize("engine", ["fast", "generic"])
def test_max_num(cuda, oracle, engine, max_num):
    """python `inds[:max_num]` after `keep.size(0) > max_num`, in mc_fast_output_kernel and in mc_output_kernel."""
    mb, ms, sf, kept = _max_num_problem()
    nk = kept[0].shape[0]
    assert nk > 2
    m = MAX_NUMS[max_num](nk)
    C = ms.shape[1] - 1
    gd, gl, launches = _mc(mb if engine == "fast" else _replicate(mb, C), ms, 0.05, m, sf)
    assert (launches <= FAST_LAUNCHES + 2) == (engine == "fast"), launches
    _same((gd, gl), apply_max_num(oracle, kept, m), f"max_num={m} nk={nk}")


@pytest.mark.parametrize("case", GENERIC_CASES, ids=[c[0] for c in GENERIC_CASES])
def test_generic_engine(cuda, oracle, case):
    _, n, C, layout, row = case
    mb, ms, sf, thr = _generic_inputs(n, C, layout)
    counts = _counts(ms, thr)
    rows = expected_path(n, C, mb.shape[1], counts)
    assert row in rows
    if C == 2:
        assert counts.min() > 0
    gd, gl, launches = _mc(mb, ms, thr, 10 ** 6, sf)
    assert launches > FAST_LAUNCHES + 2, launches
    want = per_class_reference(oracle, mb, ms, thr, IOU_THR, 10 ** 6, sf)
    print(f"n={n} C={C} {layout}: {int(counts.sum())} candidates in {int((counts > 0).sum())} classes, "
          f"{want[0].shape[0]} kept, {launches} launches")
    _same((gd, gl), want, "generic engine vs per-class reference")
    if layout == "shared":                 # the same problem through the per-class engine
        rd, rl, _ = _mc(_replicate(mb, C), ms, thr, 10 ** 6, sf)
        _same((rd, rl), (gd, gl), "generic per-class engine vs generic shared engine")


# ------------------------------------------------------------------------------------------ labelled engine

@pytest.mark.parametrize("num_labels", [2048, 2049])
def test_ml_nms_many_labels(cuda, oracle, num_labels):
    """2048 label groups fit the segment table's in-CTA sort; 2049 take its chunked-scan branch."""
    from rs_detection_b200.jdet.ops.nms_rotated import ml_nms_rotated
    n = 6000
    assert ("many segments" in engine_path(NMS_ROTATED, n, num_labels)) == (num_labels > 2048)
    d = W.rotated_boxes(n, 61, canvas=400, smin=16, smax=128)
    s = W.distinct_scores(n, 61)
    lab = np.random.default_rng(62).permutation(np.arange(n) % num_labels)
    assert np.unique(lab).size == num_labels
    got = ml_nms_rotated(_t(d), _t(s), _t(lab), IOU_THR).cpu().numpy()
    want = oracle.ml_nms_rotated(d, s, lab, IOU_THR)
    print(f"{num_labels} labels: {want.size} of {n} kept")
    assert want.size < n
    assert np.array_equal(got, want)


def test_ml_nms_negative_labels(cuda, oracle):
    """Arbitrary int32 labels take the sign-flipped 32-bit label key; |label| <= 2^24 so that the oracle's float32
    label column holds them exactly."""
    from rs_detection_b200.jdet.ops.nms_rotated import ml_nms_rotated
    n = 3000
    vals = np.array([-2 ** 24, -2 ** 24 + 1, -70000, -256, -1, 0, 1, 255, 65536, 2 ** 24 - 1, 2 ** 24], np.int64)
    lab = vals[np.random.default_rng(63).integers(0, vals.size, n)]
    d = W.rotated_boxes(n, 64, canvas=700, smin=16, smax=128)
    s = W.distinct_scores(n, 64)
    got = ml_nms_rotated(_t(d), _t(s), _t(lab), IOU_THR).cpu().numpy()
    assert np.array_equal(got, oracle.ml_nms_rotated(d, s, lab, IOU_THR))


@pytest.mark.parametrize("thr", [0.3, 1.0])
def test_nms_rotated_cpu_cooperative(cuda, oracle, thr):
    """The `>=` rule on a 141-block group: the dense engine's cooperative scan.  Exact duplicates have IoU 1, which
    `>=` suppresses at thr 1.0 and `>` would not."""
    from rs_detection_b200.jdet.ops.nms_rotated import nms_rotated_cpu
    n = 9000
    assert "ge dense cooperative" in engine_path(NMS_ROTATED_GE, n, None)
    d = W.rotated_boxes(n, 65, canvas=1024, smin=16, smax=160)
    d[4000:4100] = d[0:100]
    s = W.distinct_scores(n, 65)
    order = np.argsort(-s.astype(np.float64), kind="stable").astype(np.int32)
    got = nms_rotated_cpu(_t(d), _t(order.astype(np.int64)), thr, box_length=5).cpu().numpy()
    want = oracle.nms_rotated_keep(d, order, thr, 5, True, 1)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("n", [32767, 32768])
def test_sparse_boundary_equals_dense_engine(cuda, n):
    """At n = 32768 unlabelled rotated calls take the sparse path (16 more launches), at 32767 the dense engine;
    the same call with all-equal labels stays dense (5 more launches for the label sort)."""
    from rs_detection_b200 import _lib, core
    d = _t(W.rotated_boxes(n, 66, canvas=2048, smin=8, smax=128))
    s = _t(W.distinct_scores(n, 66))
    zeros = torch.zeros(n, dtype=torch.int32, device="cuda")
    for kind in (NMS_ROTATED, NMS_ROTATED_GE):
        sparse = "sparse unlabelled" in engine_path(kind, n, None)
        assert sparse == (n >= 32768)
        l0 = _lib.launch_count()
        unl = core.nms(kind, d, s, 0.3)
        l1 = _lib.launch_count()
        lab = core.nms(kind, d, s, 0.3, labels=zeros)
        l2 = _lib.launch_count()
        assert (l1 - l0 > l2 - l1) == sparse, (l1 - l0, l2 - l1)
        assert torch.equal(unl.keep_mask, lab.keep_mask)
        assert torch.equal(unl.sorted_idx, lab.sorted_idx) and 0 < unl.count < n


# ------------------------------------------------------------------------------------------ C ABI buffers
GUARD = 16
LABEL_FILL = -7


@pytest.mark.parametrize("layout", ["shared", "per-class"])
def test_guarded_outputs_and_dirty_workspace(cuda, oracle, layout):
    """Rows below the count match the reference; rows at and above it and the guards on both sides keep their
    prefill.  The result does not depend on what the workspace holds: zeros, ones, or what a larger call left."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    n, C, max_num = 2000, 5, 300

    def inputs(n, C, seed):
        mb = W.rotated_boxes(n * (C + 1) if layout == "per-class" else n, seed, canvas=800, smin=16, smax=160)
        return mb.reshape(n, -1), W.class_scores(n, C, seed)

    mb, ms = inputs(n, C, 70)
    big_mb, big_ms = inputs(4000, 10, 71)
    assert (mb.shape[1] == 5) == (layout == "shared")
    wd, wl = per_class_reference(oracle, mb, ms, 0.05, IOU_THR, max_num)
    wsb = max(L.rsdet_multiclass_nms_rotated_workspace_bytes(n, C), L.rsdet_multiclass_nms_rotated_workspace_bytes(4000, 10))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

    def call(mb, ms, max_num):
        n, C = ms.shape[0], ms.shape[1] - 1
        cap = n * C
        dets = torch.full(((cap + 2 * GUARD) * 6,), float("nan"), device="cuda")
        labs = torch.full((cap + 2 * GUARD,), LABEL_FILL, dtype=torch.int32, device="cuda")
        cnt = torch.full((1,), LABEL_FILL, dtype=torch.int32, device="cuda")
        mb_t, ms_t = _t(mb), _t(ms)
        rc = L.rsdet_multiclass_nms_rotated(mb_t.data_ptr(), mb.shape[1], ms_t.data_ptr(), n, C, 0.05, IOU_THR, max_num, None,
                                            dets.data_ptr() + GUARD * 24, labs.data_ptr() + GUARD * 4, cnt.data_ptr(),
                                            ws.data_ptr(), wsb, _lib.stream_ptr())
        assert rc == 0, rc
        return dets.cpu().numpy().reshape(-1, 6), labs.cpu().numpy(), int(cnt.item())

    results = []
    for prep in ("zeros", "ones", "larger call"):
        if prep == "zeros":
            ws.fill_(0)
        elif prep == "ones":
            ws.fill_(0xFF)
        else:
            ws.fill_(0)
            call(big_mb, big_ms, -1)
        dets, labs, k = call(mb, ms, max_num)
        assert k == wd.shape[0], (prep, k, wd.shape[0])
        rows = dets[GUARD:GUARD + k]
        assert np.array_equal(rows.view(np.int32), wd.view(np.int32)) and np.array_equal(labs[GUARD:GUARD + k], wl), prep
        assert np.isnan(np.delete(dets, np.s_[GUARD:GUARD + k], 0)).all(), prep
        assert (np.delete(labs, np.s_[GUARD:GUARD + k]) == LABEL_FILL).all(), prep
        results.append(dets.view(np.int32))
    assert all(np.array_equal(r, results[0]) for r in results[1:])


# ------------------------------------------------------------------------------------------ score keys
TINY = np.float32(np.finfo(np.float32).smallest_subnormal)
SCORE_CLUSTERS = [   # scores of identical boxes: each cluster keeps exactly the first of them in score order
    (-0.0, 0.0), (0.0, -0.0), (-0.0, -0.0), (0.0, 0.0, -0.0), (-0.0, 0.0, 0.0), (np.inf, np.inf), (np.inf, 1e38),
    (1e38, np.inf), (TINY, 0.0), (-0.0, TINY), (0.0, TINY, -0.0), (-TINY, -0.0), (-0.0, -TINY), (-TINY, 0.0, -TINY),
]


def _clusters(seed):
    """Identical boxes per cluster, clusters apart from each other; cluster order shuffled."""
    rng = np.random.default_rng(seed)
    boxes, scores, cid = [], [], []
    for k in rng.permutation(len(SCORE_CLUSTERS)):
        for v in SCORE_CLUSTERS[k]:
            boxes.append([100.0 * k + 50, 60.0, 40.0, 20.0, 0.3])
            scores.append(v)
            cid.append(k)
    return np.array(boxes, np.float32), np.array(scores, np.float32), np.array(cid)


def test_signed_zero_scores_tie_nms_rotated(cuda, oracle):
    from rs_detection_b200.jdet.ops.nms_rotated import ml_nms_rotated, nms_rotated
    d, s, cid = _clusters(80)
    want = oracle.nms_rotated(d, s, 0.5)
    assert want.size == len(SCORE_CLUSTERS)
    assert np.array_equal(nms_rotated(_t(d), _t(s), 0.5).cpu().numpy(), want)
    lab = (cid * 7919) % 13 - 6
    assert np.array_equal(ml_nms_rotated(_t(d), _t(s), _t(lab), 0.5).cpu().numpy(), oracle.ml_nms_rotated(d, s, lab, 0.5))


def test_signed_zero_scores_tie_hbb(cuda, oracle):
    """The float64 kinds key through desc_key(double); their ties put the higher index first."""
    from rs_detection_b200 import core
    d, s, _ = _clusters(81)
    hbb = np.stack([d[:, 0] - 20, d[:, 1] - 10, d[:, 0] + 20, d[:, 1] + 10], 1).astype(np.float64)
    res = core.nms(NMS_HBB, _t(hbb), _t(s.astype(np.float64)), 0.5, want_score=True)
    want = oracle.hbb_nms(np.concatenate([hbb, s.astype(np.float64)[:, None]], 1), 0.5, stable_ties=True)
    assert want.size == len(SCORE_CLUSTERS)
    assert np.array_equal(res.score_idx.cpu().numpy(), want)


@pytest.mark.parametrize("engine", ["fast", "generic"])
def test_signed_zero_scores_tie_multiclass(cuda, oracle, engine):
    """-0.0 and +0.0 scores from score factors of -0.0, +0.0 and 1 on raw scores of 0 and 0.25 (score_thr < 0 lets
    a zero raw score through), plus +inf and the smallest subnormal; C = 3 classes on clustered boxes."""
    d, s, _ = _clusters(82)
    n, C = d.shape[0], 3
    rng = np.random.default_rng(83)
    ms = rng.choice(np.array([0.0, 0.25, TINY, np.inf], np.float32), (n, C + 1)).astype(np.float32)
    sf = rng.choice(np.array([-0.0, 0.0, 1.0], np.float32), n).astype(np.float32)
    sf[np.isinf(ms).any(1)] = 1.0                                    # inf * 0 would be NaN
    ms[:, 1] = np.where(sf == 1.0, s, ms[:, 1])                      # the cluster scores where the factor keeps them
    mb = d if engine == "fast" else _replicate(d, C)
    want = oracle.multiclass_nms_rotated(d, ms, -1.0, dict(iou_thr=0.5), 10 ** 6, sf)
    prod = ms[:, 1:] * sf[:, None]
    assert (np.signbit(prod) & (prod == 0)).any() and (~np.signbit(prod) & (prod == 0)).any()
    from rs_detection_b200 import core
    d_t, lab, cnt = core.multiclass_nms_rotated(_t(mb), _t(ms), -1.0, 0.5, 10 ** 6, _t(sf))
    k = int(cnt.item())
    _same((d_t[:k].cpu().numpy(), lab[:k].cpu().numpy()), want, engine)
