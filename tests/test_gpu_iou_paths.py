"""The loops of `box_iou_tiles_kernel` (csrc/box_iou.cu) that small matrices never reach, and MaxIoU assignment on
given overlap matrices, against the oracle.

  loop                 reached when
  grid-stride tiles    more 64x64 tiles than the grid's 6 * 148 = 888 CTAs (box_iou.cu:206-208): a CTA takes a second,
                       third ... tile, crowded and empty ones in turn
  stage-2 chunks       a tile with more than kQ2 = 1024 bounding-circle survivors (box_iou.cu:105): a 64x64 tile of
                       mutually overlapping boxes has 4096, four chunks
  zero_tiny            the v1 wrapper's guard, boxes with a side below 1e-3 (box_iou.cu:28), for both versions

IoU values meet the parity contract (1e-6 absolute); assignment is bit-exact.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
TILES_PER_GRID = 6 * 148


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _iou(b1, b2, version, zero_tiny):
    """rsdet_box_iou_rotated through the C ABI."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    t1, t2 = _t(b1), _t(b2)
    out = torch.full((b1.shape[0], b2.shape[0]), float("nan"), device="cuda")
    wsb = L.rsdet_box_iou_rotated_workspace_bytes(b1.shape[0], b2.shape[0])
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device="cuda")
    rc = L.rsdet_box_iou_rotated(t1.data_ptr(), b1.shape[0], t2.data_ptr(), b2.shape[0], version, int(zero_tiny),
                                 out.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr())
    assert rc == 0, rc
    return out.cpu().numpy()


def _want(oracle, b1, b2, version, zero_tiny):
    w = oracle.box_iou_rotated(b1, b2, version, 1)
    if zero_tiny:
        w[b1[:, 2:4].min(1) < np.float32(0.001), :] = 0.0
        w[:, b2[:, 2:4].min(1) < np.float32(0.001)] = 0.0
    return w


def _close(got, want, what):
    err = float(np.abs(got.astype(np.float64) - want).max()) if got.size else 0.0
    print(f"{what}: max |d| = {err:.3g}")
    assert not np.isnan(got).any(), what
    assert err <= 1e-6, what


def _crowd(n, seed, centre=(500.0, 500.0)):
    """n boxes that all contain `centre`: every pair overlaps."""
    rng = np.random.default_rng(seed)
    c = np.asarray(centre) + rng.uniform(-3, 3, (n, 2))
    wh = rng.uniform(20, 60, (n, 2))
    return np.concatenate([c, wh, rng.uniform(-np.pi / 2, np.pi / 2, (n, 1))], 1).astype(np.float32)


def _striped(n, seed):
    """Blocks of 64 rows: even blocks are crowds around one of three spots, odd blocks are boxes scattered far apart,
    so tiles alternate between 4096 overlapping pairs and none."""
    rng = np.random.default_rng(seed)
    out = []
    for b in range(-(-n // 64)):
        if b % 2 == 0:
            out.append(_crowd(64, seed + b, centre=(500.0 + 400 * (b // 2 % 3), 500.0)))
        else:
            xy = rng.uniform(5000, 1e6, (64, 2))
            out.append(np.concatenate([xy, rng.uniform(5, 30, (64, 2)), rng.uniform(-1.5, 1.5, (64, 1))], 1).astype(np.float32))
    return np.concatenate(out)[:n]


@pytest.mark.parametrize("version", [0, 1])
def test_grid_stride_tiles(cuda, oracle, version):
    n = 3000
    tiles = (-(-n // 64)) ** 2
    assert tiles >= 2200 > 2 * TILES_PER_GRID
    b1, b2 = _striped(n, 10), _striped(n, 11)
    got = _iou(b1, b2, version, False)
    want = _want(oracle, b1, b2, version, False)
    crowded = (want > 0).sum()
    assert 0.03 * want.size < crowded < 0.5 * want.size
    _close(got, want, f"v{version} {n}x{n}, {tiles} tiles")


SIDES = [1, 63, 64, 65, 129]


@pytest.mark.parametrize("version", [0, 1])
def test_stage2_chunks(cuda, oracle, version):
    """Crowds: a full 64x64 tile holds 4096 survivors (four chunks of 1024); partial tiles at every edge size."""
    for n1 in SIDES:
        for n2 in SIDES:
            b1, b2 = _crowd(n1, n1), _crowd(n2, 1000 + n2)
            want = _want(oracle, b1, b2, version, False)
            assert (want > 0).all()
            _close(_iou(b1, b2, version, False), want, f"v{version} crowd {n1}x{n2}")


@pytest.mark.parametrize("version", [0, 1])
@pytest.mark.parametrize("zero_tiny", [False, True])
def test_zero_tiny(cuda, oracle, version, zero_tiny):
    """Sides at 1e-3 (kept) and the float just below (zeroed when zero_tiny), zero and negative sides, among crowds."""
    b = _crowd(200, 12)
    below = np.nextafter(np.float32(0.001), np.float32(0))
    rng = np.random.default_rng(13)
    for i, (w, h) in enumerate([(0.001, 5), (5, 0.001), (below, 5), (5, below), (0.001, 0.001), (below, below),
                                (0, 10), (-3, 10), (10, -3), (1e-8, 1e-8)]):
        for r in rng.choice(200, 3, replace=False):
            b[r, 2], b[r, 3] = w, h
    b2 = np.concatenate([b[::3], _crowd(70, 14)])
    tiny1 = b[:, 2:4].min(1) < np.float32(0.001)
    assert tiny1.any() and (b[:, 2:4].min(1) == np.float32(0.001)).any()
    got = _iou(b, b2, version, zero_tiny)
    want = _want(oracle, b, b2, version, zero_tiny)
    _close(got, want, f"v{version} zero_tiny={zero_tiny}")
    if zero_tiny:
        assert (got[tiny1] == 0).all()


# ------------------------------------------------------------------------------------------ assignment
def _overlaps(G, n, seed):
    """Quantised overlaps: equal maxima in columns and rows, all-zero rows and columns."""
    rng = np.random.default_rng(seed)
    ov = rng.choice(np.array([0, 0, 0, 0.1, 0.3, 0.5, 0.7, 0.9], np.float32), (G, n))
    if G > 2:
        ov[1] = 0                               # an all-zero gt row
        ov[2] = ov[0]                           # equal rows: every column maximum ties between gt 0 and 2
    ov[:, 5] = 0                                # an all-zero proposal column
    ov[:, 7] = ov[:, 6]                         # equal columns: row maxima tie between proposals 6 and 7
    return ov


@pytest.mark.parametrize("low_quality", [(False, True), (True, True), (True, False)], ids=["plain", "lq_all", "lq_one"])
@pytest.mark.parametrize("G", [1, 33, 3000])
def test_assign_bit_exact(cuda, oracle, G, low_quality):
    from rs_detection_b200 import core
    n = 1037                                    # not a multiple of 128
    ov = _overlaps(G, n, G)
    gl = np.random.default_rng(G + 1).integers(0, 15, G).astype(np.int32)
    mlq, assign_all = low_quality
    for min_pos in (0.0, 0.3):
        for neg in (0.4, (0.1, 0.5)):
            w_inds, w_max, w_lab = oracle.max_iou_assign(ov, 0.5, neg, min_pos, mlq, assign_all, gt_labels=gl,
                                                         assigned_labels_filled=-1)
            inds, mx, lab = core.assign_wrt_overlaps(_t(ov), 0.5, neg, min_pos, mlq, assign_all, gt_labels=_t(gl))
            what = f"G={G} mlq={mlq} all={assign_all} min_pos={min_pos} neg={neg}"
            assert np.array_equal(inds.cpu().numpy(), w_inds), what
            assert np.array_equal(mx.cpu().numpy().view(np.int32), w_max.view(np.int32)), what
            assert np.array_equal(lab.cpu().numpy(), w_lab), what


def test_assign_null_outputs(cuda, oracle):
    """NULL gt_labels (the labels output is the fill value) and NULL max_overlaps through the C ABI."""
    from rs_detection_b200 import _lib
    L = _lib.load()
    G, n = 33, 1037
    ov = _overlaps(G, n, 5)
    w_inds, _, _ = oracle.max_iou_assign(ov, 0.5, 0.4, 0.0, True, True)
    ov_t = _t(ov)
    ws = torch.empty(L.rsdet_assign_workspace_bytes(G), dtype=torch.uint8, device="cuda")
    inds = torch.full((n,), -9, dtype=torch.int32, device="cuda")
    lab = torch.full((n,), -9, dtype=torch.int32, device="cuda")
    rc = L.rsdet_assign_wrt_overlaps(ov_t.data_ptr(), G, n, 0.5, 0.0, 0.4, 0.0, 1, 1, None, -3, inds.data_ptr(), None,
                                     lab.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
    assert rc == 0
    assert np.array_equal(inds.cpu().numpy(), w_inds)
    assert (lab.cpu().numpy() == -3).all()
