"""Every dispatch path of `rsdet_roi_align_rotated_forward` / `_backward` against the oracle.

The two entry points choose a prologue and a gather kernel from the layout (NCHW or channels-last), the RoI count K,
the alignment of the caller's buffers, the geometry and whether the fast path applies (include/rsdet.h, DESIGN.md
§4.1).  Forward, 7x7 bins, sampling ratio 2, C % 256 == 0:

  * 16-byte aligned output, NCHW, 256 <= K <= 16384: the order block and the geometry blocks ride with the pyramid
    transpose (`transpose_prep_kernel`); above K = 4160 the order block recomputes buckets in its scatter pass;
  * aligned output, NCHW, K < 256 or K > 16384, and every aligned channels-last call: `roi_prep_kernel`;
  * output not 16-byte aligned: the prologue of the other geometries (`roi_order_kernel` or the ride-along order
    block, then `roi_geometry_kernel`) and `roi_align_fwd_kernel<2>`; otherwise the persistent
    `roi_align_fwd77p_kernel`.

Other geometries run `roi_align_fwd_kernel<2>` (C % 256 == 0) or `<1>`, and configurations outside the fast path run
`roi_align_generic_kernel`.  The order (K >= 256) changes only which CTA takes a RoI, and the persistent kernel is
bit-identical to `roi_align_fwd_kernel<2>`, so every forward path is checked bit for bit against one reference: NCHW,
aligned, K split into calls of at most 4000 RoIs.  A seeded subset of rows is checked against the oracle at 1e-5 of
the tensor scale, every output buffer is prefilled with NaN (every row must be written, nothing outside it), and the
levels written through `levels_out` must equal the oracle's.  Backward: both layouts, K below and above the order threshold, 256 and 260
channels (`roi_align_bwd_kernel<2>` / `<1>` with a ragged second chunk), against the oracle at 1e-4, with the
caller's gradient buffers prefilled with NaN so that their zero fill is checked too.

The tests marked "misaligned" pass caller buffers that are offset by one float from a 16-byte boundary: a
`grad_out`, and channels-last feature maps and gradient maps.  They exist to check the library's fallback for such
pointers (scalar staging of `grad_out`, the generic kernel for channels-last maps).  Do not run them against a build
of the library that lacks that fallback: there the fast kernels issue 16-byte vector accesses on misaligned
addresses.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import workloads as W
from helpers import close_report

pytestmark = pytest.mark.gpu

NAN = float("nan")
STRIDES = [4, 8, 16, 32]
EXTEND = (1.4, 1.2)          # (h, w) extension of the Oriented R-CNN extractor
TILE = 256
ALIGNED, SHIFTED = 4, 1      # float offset of a view into its buffer: 16 bytes, or 4 bytes off a 16-byte boundary
REF_CALL = 4000              # RoIs per call of the reference
ORACLE_ROWS = 200            # seeded rows per case checked against the oracle


# ------------------------------------------------------------------------------------------ helpers
def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check(got, want, tol, what):
    assert not np.isnan(got).any(), f"{what}: NaN in the result"      # close_report does not count NaN
    scale = float(np.abs(want).max()) or 1.0
    nbad, maxerr, _ = close_report(got, want, tol, tol * scale)
    print(f"{what}: max abs err {maxerr:.3g} (scale {scale:.3g}), violations {nbad}/{want.size}")
    assert nbad == 0, what


class Placed:
    """A tensor of `shape` at `offset` floats into a buffer with guard floats on both sides."""

    def __init__(self, shape, offset, fill=NAN, src=None):
        self.n = int(np.prod(shape))
        self.offset = offset
        self.buf = torch.full((self.n + 8,), fill, dtype=torch.float32, device="cuda")
        self.t = self.buf[offset:offset + self.n].view(shape)
        if src is not None:
            self.t.copy_(src)

    def guards_intact(self):
        g = torch.cat([self.buf[:self.offset], self.buf[self.offset + self.n:]])
        return bool(torch.isnan(g).all())


def _cfg(shapes, scales, out=7, sr=2, version=1, extend=EXTEND, channels_last=False):
    from rs_detection_b200 import core
    return core.make_roi_cfg(shapes, scales, out, sr, version, extend, 56.0, channels_last=channels_last)


def _forward(cfg, feats, rois, out, lv=None):
    """The C ABI forward into caller buffers (core allocates its own)."""
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    K = rois.shape[0]
    ws = torch.empty(max(L.rsdet_roi_align_rotated_workspace_bytes(C.byref(cfg), K, 0), 1), dtype=torch.uint8, device="cuda")
    rc = L.rsdet_roi_align_rotated_forward(C.byref(cfg), core._ptr_array(feats), rois.data_ptr() if K else None, K,
                                           out.data_ptr(), None if lv is None else lv.data_ptr(), ws.data_ptr(),
                                           ws.numel(), _lib.stream_ptr())
    assert rc == 0, rc


def _backward(cfg, grad_out, rois, grads):
    """The C ABI backward into caller buffers; grad_out is a tensor or None (K = 0)."""
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    K = rois.shape[0]
    ws = torch.empty(L.rsdet_roi_align_rotated_workspace_bytes(C.byref(cfg), K, 1), dtype=torch.uint8, device="cuda")
    rc = L.rsdet_roi_align_rotated_backward(C.byref(cfg), None if grad_out is None else grad_out.data_ptr(),
                                            rois.data_ptr() if K else None, K, core._ptr_array(grads), ws.data_ptr(),
                                            ws.numel(), _lib.stream_ptr())
    assert rc == 0, rc


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _reference(cfg, feats, rois):
    """NCHW, aligned output, calls of at most REF_CALL RoIs."""
    K = rois.shape[0]
    ref = Placed((K, cfg.channels, cfg.pooled_h, cfg.pooled_w), ALIGNED)
    for i in range(0, K, REF_CALL):
        _forward(cfg, feats, rois[i:i + REF_CALL], ref.t[i:i + REF_CALL])
    assert not torch.isnan(ref.t).any()
    return ref.t


def _levels(rois, num_levels=4, extend=EXTEND):
    from oracle import oracle as O
    if num_levels == 1:
        return np.zeros(rois.shape[0], np.int64)
    return O.map_roi_levels(O.roi_rescale(rois, extend), num_levels)


def _subset(K, seed):
    return np.sort(np.random.default_rng(seed).choice(K, min(K, ORACLE_ROWS), replace=False))


class Scene:
    """A pyramid (numpy, NCHW and NHWC on the device) and its RoIs."""

    def __init__(self, feats, rois, scales, out=7, sr=2, version=1, extend=EXTEND):
        self.np = feats
        self.shapes = [f.shape for f in feats]
        self.nchw = [_t(f) for f in feats]
        self.nhwc = [_nhwc(x) for x in self.nchw]
        self.rois_np = rois
        self.rois = _t(rois)
        self.scales = scales
        self.out, self.sr, self.version, self.extend = out, sr, version, extend

    def cfg(self, channels_last):
        return _cfg(self.shapes, self.scales, self.out, self.sr, self.version, self.extend, channels_last)

    def feats(self, channels_last):
        return self.nhwc if channels_last else self.nchw

    def oracle_fwd(self, oracle, rows):
        r = self.rois_np[rows]
        osz = (self.out, self.out) if isinstance(self.out, int) else tuple(self.out)
        if len(self.np) == 1:
            assert self.extend == (1.0, 1.0)
            return oracle.roi_align_rotated_fwd(self.np[0], r, osz, self.scales[0], self.sr, self.version)
        want, _ = oracle.oriented_extractor_fwd(self.np, r, STRIDES, osz, self.sr, self.extend, 56, self.version)
        return want

    def oracle_bwd(self, oracle, g):
        if len(self.np) == 1:
            assert self.extend == (1.0, 1.0)
            return [oracle.roi_align_rotated_bwd(g, self.rois_np, self.shapes[0], self.scales[0], self.sr, self.version)]
        return oracle.oriented_extractor_bwd(g, self.shapes, self.rois_np, STRIDES, self.sr, self.extend, 56, self.version)


def _fpn_scene(batch, K, seed, channels=256, tile=TILE, rois=None, **kw):
    feats = W.fpn_pyramid(batch, seed, tile=tile, channels=channels)
    if rois is None:
        rois = W.proposals(K, seed, batch=batch, canvas=tile)
    return Scene(feats, rois, [1 / s for s in STRIDES], **kw)


def _check_forward_call(scene, oracle, channels_last, offset, ref, what, rows=None, want=None, bitwise=True):
    """One forward call into a NaN-prefilled output at `offset` with levels: against `ref` and the oracle."""
    K = scene.rois.shape[0]
    cfg = scene.cfg(channels_last)
    out = Placed((K, cfg.channels, cfg.pooled_h, cfg.pooled_w), offset)
    lv = torch.full((K,), -1, dtype=torch.int32, device="cuda")
    _forward(cfg, scene.feats(channels_last), scene.rois, out.t, lv)
    assert out.guards_intact(), f"{what}: write outside the output"
    assert not torch.isnan(out.t.view(K, -1)).any(dim=1).any(), f"{what}: an output row kept its NaN prefill"
    assert np.array_equal(lv.cpu().numpy(), _levels(scene.rois_np, len(scene.np), scene.extend)), f"{what}: levels"
    if bitwise:
        assert torch.equal(out.t, ref), f"{what}: not bit-identical to the reference calls"
    else:
        _check(out.t.cpu().numpy(), ref.cpu().numpy(), 1e-5, f"{what} vs reference calls")
    if rows is None:
        rows = _subset(K, K)
    if want is None:
        want = scene.oracle_fwd(oracle, rows)
    _check(out.t[torch.from_numpy(rows).cuda()].cpu().numpy(), want, 1e-5, f"{what} vs oracle")
    return out.t


def _check_forward_all(scene, oracle, what):
    """Reference calls, then every (layout, output alignment) against them."""
    ref = _reference(scene.cfg(False), scene.nchw, scene.rois)
    rows = _subset(scene.rois.shape[0], 1)
    want = scene.oracle_fwd(oracle, rows)
    for cl in (False, True):
        for off in (ALIGNED, SHIFTED):
            _check_forward_call(scene, oracle, cl, off, ref, f"{what} channels_last={cl} offset={off}", rows, want)


# ------------------------------------------------------------------------------------------ forward path matrix
KS = [1, 255, 256, 4096, 4097, 4160, 4161, 16384, 16385]
MATRIX = [(cl, off, K) for cl in (False, True) for off in (ALIGNED, SHIFTED) for K in KS] + \
         [(False, off, 10000) for off in (ALIGNED, SHIFTED)]


@pytest.fixture(scope="module")
def matrix_scene(cuda):
    scene = _fpn_scene(1, max(KS), 3)
    return scene, _reference(scene.cfg(False), scene.nchw, scene.rois)


@pytest.mark.parametrize("channels_last,offset,K", MATRIX,
                         ids=[f"{'nhwc' if cl else 'nchw'}-{'aligned' if off == ALIGNED else 'shifted'}-K{K}"
                              for cl, off, K in MATRIX])
def test_forward_path_matrix(oracle, matrix_scene, channels_last, offset, K):
    """K straddles the order threshold (256), the ride-along bucket cache (4160), the ride-along limit (16384)."""
    full, ref = matrix_scene
    scene = Scene(full.np, full.rois_np[:K], full.scales)
    scene.nchw, scene.nhwc = full.nchw, full.nhwc
    _check_forward_call(scene, oracle, channels_last, offset, ref[:K], f"K={K} channels_last={channels_last} offset={offset}")


@pytest.mark.parametrize("batch", [2, 8, 9, 12])
def test_forward_batches(oracle, cuda, batch):
    """Batch above 8 wraps the image slot of the locality order's buckets."""
    _check_forward_all(_fpn_scene(batch, 1500, 20 + batch), oracle, f"batch {batch}")


def test_forward_single_level_batch(oracle, cuda):
    feat = np.random.default_rng(30).standard_normal((3, 256, 48, 40)).astype(np.float32)
    rois = W.proposals(700, 30, batch=3, canvas=640)
    _check_forward_all(Scene([feat], rois, [1 / 16], extend=(1.0, 1.0)), oracle, "one level, batch 3")


def test_forward_identical_rois(oracle, cuda):
    """Every RoI in one bucket of the locality order; 4500 > 4160 also recomputes buckets in the scatter pass."""
    rois = np.repeat(np.array([[0, 130.5, 77.25, 90, 40, 0.6]], np.float32), 4500, axis=0)
    _check_forward_all(_fpn_scene(1, 0, 31, rois=rois), oracle, "identical RoIs")


def test_forward_unsorted_batch_indices(oracle, cuda):
    rois = W.proposals(1200, 32, batch=4, canvas=TILE)
    rois[:, 0] = np.sort(rois[:, 0])[::-1]           # descending image index
    rois[::7, 0] = np.arange(len(rois[::7])) % 4       # interleaved
    _check_forward_all(_fpn_scene(4, 0, 32, rois=rois), oracle, "unsorted batch indices")


# ------------------------------------------------------------------------------------------ fast-path neighbours
@pytest.mark.parametrize("channels,out,sr", [(512, 5, 2), (512, 7, 3), (36, 7, 2)],
                         ids=["fwd2-C512-5x5", "fwd2-C512-sr3", "fwd1-C36"])
def test_forward_fast_neighbours(oracle, cuda, channels, out, sr):
    """roi_align_fwd_kernel<2> (C % 256 == 0, not 7x7 / sr 2) and <1>, with the locality order (K >= 256)."""
    _check_forward_all(_fpn_scene(2, 400, 40 + channels + sr, channels=channels, out=out, sr=sr), oracle,
                       f"C={channels} out={out} sr={sr}")


# ------------------------------------------------------------------------------------------ generic kernel, channels-last
@pytest.mark.parametrize("channels,out,sr", [(6, 7, 0), (8, 8, 5)], ids=["C6-sr0", "C8-8x8-sr5"])
def test_generic_channels_last(oracle, cuda, channels, out, sr):
    """roi_align_generic_kernel: C % 4 != 0 with an adaptive grid, and 8x8 bins x 25 samples (> 1024 samples)."""
    scene = _fpn_scene(2, 300, 50 + channels, channels=channels, out=out, sr=sr)
    ref = _reference(scene.cfg(False), scene.nchw, scene.rois)
    rows = _subset(300, 2)
    want = scene.oracle_fwd(oracle, rows)
    for cl in (False, True):
        for off in (ALIGNED, SHIFTED):
            _check_forward_call(scene, oracle, cl, off, ref, f"generic channels_last={cl} offset={off}", rows, want)
    g = torch.randn(ref.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(channels))
    wb = scene.oracle_bwd(oracle, g.cpu().numpy())
    got = {}
    for cl in (False, True):
        grads = [Placed(s if not cl else (s[0], s[2], s[3], s[1]), ALIGNED) for s in scene.shapes]
        _backward(scene.cfg(cl), g, scene.rois, [p.t for p in grads])
        got[cl] = [(p.t.permute(0, 3, 1, 2) if cl else p.t).cpu().numpy() for p in grads]
        for l in range(len(wb)):
            assert grads[l].guards_intact()
            _check(got[cl][l], wb[l], 1e-4, f"generic bwd channels_last={cl} level {l}")
    for l in range(len(wb)):
        _check(got[True][l], got[False][l], 1e-4, f"generic bwd channels-last vs NCHW level {l}")


# ------------------------------------------------------------------------------------------ backward matrix
BWD = [(cl, K, ch, kind) for cl in (False, True) for K in (100, 600) for ch in (256, 260) for kind in ("v0", "v1", "fpn")]


def _bwd_scene(K, channels, kind, seed):
    if kind == "fpn":
        return _fpn_scene(2, K, seed, channels=channels)
    rng = np.random.default_rng(seed)
    feat = rng.standard_normal((2, channels, 40, 36)).astype(np.float32)
    rois = W.proposals(K, seed, batch=2, canvas=600)
    rois[:3, 3:5] = [[0.5, 0.5], [2000, 20], [20, 1500]]
    rois[3, 1:3] = [-40, 700]
    return Scene([feat], rois, [1 / 16], version=0 if kind == "v0" else 1, extend=(1.0, 1.0))


def _check_backward(scene, oracle, channels_last, g, what, grad_offset=ALIGNED, want=None):
    cfg = scene.cfg(channels_last)
    shapes = [(s[0], s[2], s[3], s[1]) if channels_last else s for s in scene.shapes]
    grads = [Placed(s, grad_offset) for s in shapes]
    _backward(cfg, g, scene.rois, [p.t for p in grads])
    got = []
    for l, p in enumerate(grads):
        assert p.guards_intact(), f"{what}: write outside level {l}'s gradient"
        got.append((p.t.permute(0, 3, 1, 2) if channels_last else p.t).cpu().numpy())
    if want is not None:
        for l in range(len(got)):
            _check(got[l], want[l], 1e-4, f"{what} level {l}")
    return got


@pytest.mark.parametrize("channels_last,K,channels,kind", BWD,
                         ids=[f"{'nhwc' if cl else 'nchw'}-K{K}-C{ch}-{kind}" for cl, K, ch, kind in BWD])
def test_backward_matrix(oracle, cuda, channels_last, K, channels, kind):
    scene = _bwd_scene(K, channels, kind, 60 + K + channels)
    osz = (len(scene.rois_np), channels, 7, 7)
    g = torch.randn(osz, device="cuda", generator=torch.Generator(device="cuda").manual_seed(K + channels))
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    _check_backward(scene, oracle, channels_last, g, f"bwd {kind} K={K} C={channels} channels_last={channels_last}", want=want)


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_backward_no_rois_zero_fills(cuda, oracle, channels_last):
    scene = _fpn_scene(2, 0, 70, rois=np.zeros((0, 6), np.float32))
    got = _check_backward(scene, oracle, channels_last, None, f"bwd K=0 channels_last={channels_last}")
    for l, a in enumerate(got):
        assert not np.isnan(a).any() and not a.any(), f"level {l} not zero-filled"


# ------------------------------------------------------------------------------------------ misaligned caller buffers
@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("channels", [256, 260])
def test_misaligned_grad_out(oracle, cuda, channels_last, channels):
    """grad_out 4 bytes off a 16-byte boundary: the fast backward stages it with scalar loads."""
    scene = _fpn_scene(2, 600, 80 + channels, channels=channels)
    g = torch.randn((600, channels, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(81))
    want = _check_backward(scene, oracle, channels_last, g, "aligned grad_out")
    gs = Placed(g.shape, SHIFTED, src=g)
    _check_backward(scene, oracle, channels_last, gs.t, f"shifted grad_out channels_last={channels_last}", want=want)


def test_misaligned_channels_last_features(oracle, cuda):
    """Channels-last maps 4 bytes off a 16-byte boundary: the forward runs the generic kernel, whose per-sample sums
    differ from the fast kernels' merged taps in the last bits, so it is held to the forward tolerance."""
    scene = _fpn_scene(2, 1500, 90)
    ref = _reference(scene.cfg(False), scene.nchw, scene.rois)
    shifted = [Placed(x.shape, SHIFTED, src=x) for x in scene.nhwc]
    scene.nhwc = [p.t for p in shifted]
    rows = _subset(1500, 3)
    want = scene.oracle_fwd(oracle, rows)
    for off in (ALIGNED, SHIFTED):
        _check_forward_call(scene, oracle, True, off, ref, f"shifted NHWC maps, output offset={off}", rows, want,
                            bitwise=False)


@pytest.mark.parametrize("channels", [256, 260])
def test_misaligned_channels_last_grads(oracle, cuda, channels):
    """Channels-last gradient maps 4 bytes off a 16-byte boundary: the backward runs the generic kernel."""
    scene = _fpn_scene(2, 600, 100 + channels, channels=channels)
    g = torch.randn((600, channels, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(101))
    want = _check_backward(scene, oracle, True, g, "aligned NHWC gradients")
    _check_backward(scene, oracle, True, g, f"shifted NHWC gradients C={channels}", grad_offset=SHIFTED, want=want)
