"""fp16 / bf16 feature pyramids through RoIAlignRotated: the typed entry points of include/rsdet.h and the mirror.

Contract under test: a half value converts exactly to fp32 and the arithmetic after that is the fp32 arithmetic
unchanged.  So every half-input forward must be BIT-IDENTICAL to the fp32 entry point called on the maps converted to
fp32 (`maps.float()`), in the same layout and with an output of the same alignment class (both calls then run the same
kernel family), and a half-output forward must equal that result rounded once (`.to(half)`).  The backward accumulates
in fp32 and rounds once; its atomic order is unspecified, so it is held to 1e-4 of the scale plus one half-precision
ulp per element of the rounded fp32 backward.  Outputs and gradient maps are NaN-prefilled with guard elements on both
sides; the "shifted" buffers sit one element off a 16-byte boundary.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_roi_paths import EXTEND, STRIDES, Scene, _fpn_scene, _levels, _subset, _bwd_scene, _check

pytestmark = pytest.mark.gpu

HALF = [torch.bfloat16, torch.float16]
HALF_IDS = ["bf16", "f16"]
CODE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
MANT = {torch.float16: 10, torch.bfloat16: 7}            # explicit mantissa bits
MIN_ULP = {torch.float16: 2.0 ** -24, torch.bfloat16: 2.0 ** -133}
NAN = float("nan")


class Placed:
    """A tensor of `shape` and `dtype`, 16 bytes (aligned) or one element (shifted) into a NaN-filled buffer with guard
    elements on both sides."""

    def __init__(self, shape, shifted, dtype, fill=NAN, src=None):
        self.n = int(np.prod(shape))
        esize = torch.empty((), dtype=dtype).element_size()
        self.offset = 1 if shifted else 16 // esize
        self.buf = torch.full((self.n + 2 * (16 // esize),), fill, dtype=dtype, device="cuda")
        self.t = self.buf[self.offset:self.offset + self.n].view(shape)
        if src is not None:
            self.t.copy_(src)

    def guards_intact(self):
        g = torch.cat([self.buf[:self.offset], self.buf[self.offset + self.n:]])
        return bool(torch.isnan(g.float()).all())


def _lib():
    from rs_detection_b200 import _lib
    return _lib


def _forward(cfg, feats, rois, out, lv=None):
    """The typed forward: element types from the tensors."""
    from rs_detection_b200 import core
    lib, L = _lib(), _lib().load()
    K, fdt = rois.shape[0], CODE[feats[0].dtype]
    ws = torch.empty(max(L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 0, fdt), 1), dtype=torch.uint8,
                     device="cuda")
    rc = L.rsdet_roi_align_rotated_forward_typed(C.byref(cfg), fdt, core._ptr_array(feats), rois.data_ptr() if K else None, K,
                                                 CODE[out.dtype], out.data_ptr(), None if lv is None else lv.data_ptr(),
                                                 ws.data_ptr(), ws.numel(), lib.stream_ptr())
    assert rc == 0, rc


def _backward(cfg, grad_out, rois, grads):
    from rs_detection_b200 import core
    lib, L = _lib(), _lib().load()
    K, fdt = rois.shape[0], CODE[grads[0].dtype]
    ws = torch.empty(L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 1, fdt), dtype=torch.uint8, device="cuda")
    gdt = CODE[grad_out.dtype] if grad_out is not None else fdt
    rc = L.rsdet_roi_align_rotated_backward_typed(C.byref(cfg), gdt, None if grad_out is None else grad_out.data_ptr(),
                                                  rois.data_ptr() if K else None, K, fdt, core._ptr_array(grads),
                                                  ws.data_ptr(), ws.numel(), lib.stream_ptr())
    assert rc == 0, rc


def _clone(scene):
    s = object.__new__(Scene)
    s.__dict__.update(scene.__dict__)
    return s


def _as(scene, dtype):
    """The scene with its pyramid rounded to `dtype` (device tensors; the numpy copy becomes the fp32 upcast)."""
    s = _clone(scene)
    s.nchw = [x.to(dtype) for x in scene.nchw]
    s.nhwc = [x.to(dtype) for x in scene.nhwc]
    s.np = [x.float().cpu().numpy() for x in s.nchw]
    return s


def _up(scene):
    s = _clone(scene)
    s.nchw = [x.float() for x in scene.nchw]
    s.nhwc = [x.float() for x in scene.nhwc]
    return s


def _run_fwd(scene, channels_last, shifted, dtype):
    K = scene.rois.shape[0]
    cfg = scene.cfg(channels_last)
    out = Placed((K, cfg.channels, cfg.pooled_h, cfg.pooled_w), shifted, dtype)
    lv = torch.full((K,), -1, dtype=torch.int32, device="cuda")
    _forward(cfg, scene.feats(channels_last), scene.rois, out.t, lv)
    assert out.guards_intact(), "write outside the output"
    assert not torch.isnan(out.t.float()).any(), "NaN left in the output"
    return out.t, lv


def _check_pair(half_scene, up_scene, channels_last, shifted, out_dtype, what, ref=None):
    """half call vs the fp32 call on the upcast maps (same layout, same output alignment class)"""
    if ref is None:
        ref = _run_fwd(up_scene, channels_last, shifted, torch.float32)
    got, lv = _run_fwd(half_scene, channels_last, shifted, out_dtype)
    want = ref[0] if out_dtype == torch.float32 else ref[0].to(out_dtype)
    assert torch.equal(lv, ref[1]), f"{what}: levels differ from the fp32 call"
    assert torch.equal(got.view(torch.int16) if out_dtype != torch.float32 else got.view(torch.int32),
                       want.view(torch.int16) if out_dtype != torch.float32 else want.view(torch.int32)), \
        f"{what}: not bit-identical to the fp32 call on the upcast maps"
    return ref


# ------------------------------------------------------------------------------------------ 1. forward matrix
KS = [1, 255, 256, 4160, 4161, 16385]
FWD = [(dt, cl, sh, K) for dt in HALF for cl in (False, True) for sh in (False, True) for K in KS]


@pytest.fixture(scope="module")
def half_scenes(cuda):
    base = _fpn_scene(1, max(KS), 3)
    scenes = {}
    for dt in HALF:
        h = _as(base, dt)
        scenes[dt] = (h, _up(h))
    return scenes


def _sub(scene, K):
    s = _clone(scene)
    s.rois_np, s.rois = scene.rois_np[:K], scene.rois[:K]
    return s


@pytest.mark.parametrize("dtype,channels_last,shifted,K", FWD,
                         ids=[f"{HALF_IDS[HALF.index(dt)]}-{'nhwc' if cl else 'nchw'}-{'shifted' if sh else 'aligned'}-K{K}"
                              for dt, cl, sh, K in FWD])
def test_forward_matrix(half_scenes, dtype, channels_last, shifted, K):
    h, up = half_scenes[dtype]
    ref = None
    for odt in (torch.float32, dtype):
        ref = _check_pair(_sub(h, K), _sub(up, K), channels_last, shifted, odt,
                          f"{dtype} K={K} channels_last={channels_last} shifted={shifted} out={odt}", ref)


@pytest.fixture(scope="module")
def batch8_scene(cuda):
    return _fpn_scene(8, 32000, 11)


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_forward_batch8_32000(batch8_scene, dtype, channels_last):
    """The benchmark's batched call: 8 tiles, 32 000 RoIs (the roi_prep_kernel prologue)."""
    h = _clone(batch8_scene)
    h.nchw = [x.to(dtype) for x in batch8_scene.nchw]
    h.nhwc = [x.to(dtype) for x in batch8_scene.nhwc]
    ref = None
    for odt in (torch.float32, dtype):
        ref = _check_pair(h, _up(h), channels_last, False, odt, f"batch 8 {dtype} channels_last={channels_last} out={odt}", ref)


# ------------------------------------------------------------------------------------------ 2. other paths
OTHER = [("fwd2-5x5", dict(channels=256, out=5, sr=2)), ("fwd1-C260", dict(channels=260, out=7, sr=2)),
         ("generic-sr0", dict(channels=256, out=7, sr=0)), ("generic-C6", dict(channels=6, out=7, sr=2))]


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("name,kw", OTHER, ids=[o[0] for o in OTHER])
def test_forward_other_paths(cuda, dtype, name, kw):
    """roi_align_fwd_kernel<2> / <1> and the generic kernel, both layouts and output alignments."""
    h = _as(_fpn_scene(2, 400, 40 + kw["channels"] + kw["sr"], **kw), dtype)
    up = _up(h)
    for cl in (False, True):
        for sh in (False, True):
            ref = None
            for odt in (torch.float32, dtype):
                ref = _check_pair(h, up, cl, sh, odt, f"{name} {dtype} channels_last={cl} shifted={sh} out={odt}", ref)


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_forward_v0_single_level(cuda, dtype):
    h = _as(_bwd_scene(700, 256, "v0", 5), dtype)
    up = _up(h)
    for cl in (False, True):
        ref = None
        for odt in (torch.float32, dtype):
            ref = _check_pair(h, up, cl, False, odt, f"v0 {dtype} channels_last={cl} out={odt}", ref)


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_forward_shifted_channels_last_maps(cuda, dtype):
    """Half NHWC maps one element off an 8-byte boundary run the generic kernel, like fp32 maps off a 16-byte one."""
    h = _as(_fpn_scene(2, 1500, 90), dtype)
    up = _up(h)
    hs = [Placed(x.shape, True, dtype, src=x) for x in h.nhwc]
    us = [Placed(x.shape, True, torch.float32, src=x) for x in up.nhwc]
    h.nhwc, up.nhwc = [p.t for p in hs], [p.t for p in us]
    for sh in (False, True):
        ref = None
        for odt in (torch.float32, dtype):
            ref = _check_pair(h, up, True, sh, odt, f"shifted NHWC {dtype} out shifted={sh} out={odt}", ref)


# ------------------------------------------------------------------------------------------ 3. oracle anchor
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_oracle_anchor(oracle, cuda, dtype):
    h = _as(_fpn_scene(2, 3000, 12), dtype)
    rows = _subset(3000, 4)
    want = h.oracle_fwd(oracle, rows)      # h.np holds the upcast maps
    for cl in (False, True):
        got, lv = _run_fwd(h, cl, False, torch.float32)
        _check(got[torch.from_numpy(rows).cuda()].cpu().numpy(), want, 1e-5, f"{dtype} channels_last={cl} vs oracle")
        assert np.array_equal(lv.cpu().numpy(), _levels(h.rois_np, 4, EXTEND))


def test_fp16_output_subnormals(cuda):
    """Features of about 1e-6: fp16 outputs fall in the subnormal range and must round exactly like torch."""
    base = _fpn_scene(1, 2000, 13)
    base.nchw = [x * 1e-6 for x in base.nchw]
    base.nhwc = [x * 1e-6 for x in base.nhwc]
    h = _as(base, torch.float16)
    assert (h.nchw[0].abs() < 6.1e-5).float().mean() > 0.99
    up = _up(h)
    for cl in (False, True):
        ref = _check_pair(h, up, cl, False, torch.float16, f"subnormal fp16 channels_last={cl}")
        assert ((ref[0].abs() < 6.1e-5) & (ref[0] != 0)).any()


# ------------------------------------------------------------------------------------------ 4. backward matrix
def _ulp(a, dtype):
    a = np.abs(a.astype(np.float64))
    with np.errstate(divide="ignore"):
        e = np.floor(np.log2(np.where(a > 0, a, 1.0)))
    return np.maximum(np.where(a > 0, 2.0 ** (e - MANT[dtype]), 0.0), MIN_ULP[dtype])


def _check_half_grads(got, want, dtype, what):
    """got, want: half tensors in the same layout; want = (fp32 backward).to(half)"""
    g, w = got.float().cpu().numpy(), want.float().cpu().numpy()
    assert not np.isnan(g).any(), f"{what}: NaN left in the gradient"
    scale = float(np.abs(w).max()) or 1.0
    tol = 1e-4 * scale + np.maximum(_ulp(g, dtype), _ulp(w, dtype))
    bad = np.abs(g - w) > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} elements off, max err {float(np.abs(g - w).max()):.3g} (scale {scale:.3g})"


def _grads(scene, channels_last, g, dtype, shifted=False):
    cfg = scene.cfg(channels_last)
    shapes = [(s[0], s[2], s[3], s[1]) if channels_last else s for s in scene.shapes]
    ps = [Placed(s, shifted, dtype) for s in shapes]
    _backward(cfg, g, scene.rois, [p.t for p in ps])
    for l, p in enumerate(ps):
        assert p.guards_intact(), f"write outside level {l}'s gradient"
    return [p.t for p in ps]


BWD = [(dt, cl, K, ch, kind, gh) for dt in HALF for cl in (False, True) for K in (100, 600) for ch in (256, 260)
       for kind in ("v0", "v1", "fpn") for gh in (False, True)]


@pytest.mark.parametrize("dtype,channels_last,K,channels,kind,half_grad", BWD,
                         ids=[f"{HALF_IDS[HALF.index(dt)]}-{'nhwc' if cl else 'nchw'}-K{K}-C{ch}-{kind}-g{'half' if gh else 'f32'}"
                              for dt, cl, K, ch, kind, gh in BWD])
def test_backward_matrix(cuda, dtype, channels_last, K, channels, kind, half_grad):
    scene = _bwd_scene(K, channels, kind, 60 + K + channels)
    g = torch.randn((K, channels, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(K + channels))
    if half_grad:
        g = g.to(dtype)
    want = [x.to(dtype) for x in _grads(scene, channels_last, g.float(), torch.float32)]
    got = _grads(scene, channels_last, g, dtype)
    for l in range(len(got)):
        _check_half_grads(got[l], want[l], dtype, f"bwd {dtype} {kind} K={K} C={channels} channels_last={channels_last} "
                                                  f"half grad_out={half_grad} level {l}")


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_backward_no_rois_zero_fills(cuda, dtype, channels_last):
    scene = _fpn_scene(2, 0, 70, rois=np.zeros((0, 6), np.float32))
    for p in _grads(scene, channels_last, None, dtype):
        assert not torch.isnan(p.float()).any() and not p.float().any(), "not zero-filled"


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("channels", [256, 260])
def test_backward_shifted_buffers(cuda, dtype, channels_last, channels):
    """A half grad_out one element off an 8-byte boundary (scalar staging) and shifted half gradient maps."""
    scene = _fpn_scene(2, 600, 80 + channels, channels=channels)
    g = torch.randn((600, channels, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(81)).to(dtype)
    want = [x.to(dtype) for x in _grads(scene, channels_last, g.float(), torch.float32)]
    gs = Placed(g.shape, True, dtype, src=g)
    for l, x in enumerate(_grads(scene, channels_last, gs.t, dtype)):
        _check_half_grads(x, want[l], dtype, f"shifted grad_out channels_last={channels_last} level {l}")
    for l, x in enumerate(_grads(scene, channels_last, g, dtype, shifted=True)):
        _check_half_grads(x, want[l], dtype, f"shifted gradient maps channels_last={channels_last} level {l}")


# ------------------------------------------------------------------------------------------ 5. autograd through the mirror
def test_mirror_autograd_bf16(cuda):
    from rs_detection_b200.jdet.models.roi_extractors.oriented_single_level import OrientedSingleRoIExtractor
    from rs_detection_b200.jdet.ops.roi_align_rotated_v1 import ROIAlignRotated_v1
    scene = _fpn_scene(2, 900, 14)
    g = torch.randn((900, 256, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(14))
    ext = OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=2), 256, STRIDES,
                                     extend_factor=EXTEND)
    single = ROIAlignRotated_v1(7, 1 / 8, 2)
    cases = [("extractor", lambda xs: ext(xs, scene.rois), scene.nchw),
             ("ROIAlignRotated_v1", lambda xs: single(xs[0], scene.rois), scene.nchw[1:2])]
    for name, fn, maps in cases:
        leaf = [m.to(torch.bfloat16).requires_grad_(True) for m in maps]
        # the parent commit's path: the op casts bf16 to fp32 and autograd casts the fp32 gradient back
        cast = [x.detach().clone().requires_grad_(True) for x in leaf]
        y_cast = fn([x.float() for x in cast])
        y = fn(leaf)
        assert y.dtype == torch.float32 and torch.equal(y, y_cast), f"{name}: output differs from the cast path"
        y.backward(g)
        y_cast.backward(g)
        for l, (a, b) in enumerate(zip(leaf, cast)):
            assert a.grad.dtype == torch.bfloat16
            _check_half_grads(a.grad, b.grad, torch.bfloat16, f"{name} level {l} .grad")


# ------------------------------------------------------------------------------------------ 6. no hidden fp32 copy
def test_no_hidden_fp32_copy(batch8_scene):
    from rs_detection_b200 import _lib as lib, core
    scene = batch8_scene
    maps = [x.to(torch.bfloat16) for x in scene.nchw]
    maps32 = [x.float() for x in maps]
    cfg = scene.cfg(False)
    n0 = lib.launch_count()
    core.roi_align_rotated_forward(cfg, maps32, scene.rois)
    launches32 = lib.launch_count() - n0
    del maps32
    lib.release_workspaces()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    n0 = lib.launch_count()
    out = core.roi_align_rotated_forward(cfg, maps, scene.rois)
    torch.cuda.synchronize()
    assert lib.launch_count() - n0 == launches32
    ws = lib.load().rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), 32000, 0, CODE[torch.bfloat16])
    growth = torch.cuda.max_memory_allocated() - before
    # the scratch cache rounds its buffer up to 1.25x + 4 KB (rs_detection_b200/_lib.py)
    allowed = out.numel() * 4 + int(ws * 1.25) + 4096 + (1 << 20)
    assert growth <= allowed, f"peak grew by {growth} bytes, output + workspace allow {allowed}"
    assert ws < sum(m.numel() for m in maps) * 4     # no fp32 copy of the pyramid in the workspace either


# ------------------------------------------------------------------------------------------ 7. CUDA graph
@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_cuda_graph_replay(batch8_scene, dtype):
    from rs_detection_b200 import core
    scene = batch8_scene
    maps = [x.to(dtype) for x in scene.nchw]
    cfg = scene.cfg(False)
    g = torch.randn((32000, 256, 7, 7), device="cuda", generator=torch.Generator(device="cuda").manual_seed(16)).to(dtype)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out = torch.empty((32000, 256, 7, 7), dtype=dtype, device="cuda")
        core.roi_align_rotated_forward(cfg, maps, scene.rois, out=out, out_dtype=dtype)
        eager_f = out.clone()
        eager_b = [x.clone() for x in core.roi_align_rotated_backward(cfg, g, scene.rois, scene.shapes, feat_dtype=dtype)]
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            core.roi_align_rotated_forward(cfg, maps, scene.rois, out=out, out_dtype=dtype)
            grads = core.roi_align_rotated_backward(cfg, g, scene.rois, scene.shapes, feat_dtype=dtype)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        out.fill_(NAN)
        for x in grads:
            x.fill_(NAN)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out.view(torch.int16), eager_f.view(torch.int16)), "forward replay differs from the eager call"
        for l, (a, b) in enumerate(zip(grads, eager_b)):
            # atomics: the order of the fp32 sums is unspecified, so the rounded maps may differ by an ulp
            _check_half_grads(a, b, dtype, f"backward replay level {l}")
