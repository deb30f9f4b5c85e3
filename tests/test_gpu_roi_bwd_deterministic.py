"""The deterministic RoIAlignRotated backward (`rsdet_roi_align_rotated_backward_deterministic`, include/rsdet.h).

Contract under test: every gradient element is the reference's sequential fp32 sum, terms (top * w) / count in the order
RoI, bin row, bin column, sample row, sample column, tap.  Hence
  1. at theta = 0 (where the device's cosf / sinf equal the host's) the gradient maps equal the oracle's BIT FOR BIT, and
     half maps equal the oracle's fp32 maps rounded once;
  2. at general angles they are within the backward tolerance of the oracle and of the atomic path;
  3. the bits do not depend on the run, the stream, graph replay, the layout, the buffers' alignment or the batch split;
  4. under torch.use_deterministic_algorithms(True) the autograd functions take this path.
Gradient buffers are NaN-prefilled with guard elements on both sides (every element written, nothing outside).
"""
import ctypes as C

import numpy as np
import pytest
import torch

import workloads as W
from test_gpu_roi_half import Placed
from test_gpu_roi_paths import EXTEND, STRIDES, Scene, _check, _fpn_scene, _levels

pytestmark = pytest.mark.gpu

CODE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
HALF = [torch.bfloat16, torch.float16]
HALF_IDS = ["bf16", "f16"]


# ------------------------------------------------------------------------------------------ helpers
def _call(cfg, grad_out, rois, grads):
    """The C ABI into caller buffers; element types from the tensors (grad_out None: K = 0)."""
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    K, fdt = rois.shape[0], CODE[grads[0].dtype]
    wsb = L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(C.byref(cfg), K, fdt)
    assert wsb > 0
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    gdt = CODE[grad_out.dtype] if grad_out is not None else fdt
    rc = L.rsdet_roi_align_rotated_backward_deterministic(C.byref(cfg), gdt, None if grad_out is None else grad_out.data_ptr(),
                                                          rois.data_ptr() if K else None, K, fdt, core._ptr_array(grads),
                                                          ws.data_ptr(), ws.numel(), _lib.stream_ptr())
    assert rc == 0, rc


def _det(scene, channels_last, g, dtype=torch.float32, shifted=False):
    """-> gradient maps in NCHW order (permuted views when channels-last)"""
    cfg = scene.cfg(channels_last)
    shapes = [(s[0], s[2], s[3], s[1]) if channels_last else s for s in scene.shapes]
    ps = [Placed(s, shifted, dtype) for s in shapes]
    _call(cfg, g, scene.rois, [p.t for p in ps])
    for l, p in enumerate(ps):
        assert p.guards_intact(), f"write outside level {l}'s gradient"
        assert not torch.isnan(p.t.float()).any(), f"level {l}: element left unwritten"
    return [p.t.permute(0, 3, 1, 2) if channels_last else p.t for p in ps]


def _atomic(scene, channels_last, g):
    from rs_detection_b200 import core
    gs = core.roi_align_rotated_backward(scene.cfg(channels_last), g, scene.rois, scene.shapes)
    return [x.permute(0, 3, 1, 2) if channels_last else x for x in gs]


def _bits(x):
    x = x.contiguous()
    return x.view(torch.int32) if x.dtype == torch.float32 else x.view(torch.int16)


def _same_bits(a, b, what):
    for l, (x, y) in enumerate(zip(a, b)):
        assert x.dtype == y.dtype and torch.equal(_bits(x), _bits(y)), f"{what}: level {l} differs"


def _np_bits_equal(got, want, what):
    got = np.ascontiguousarray(got, dtype=np.float32)
    want = np.ascontiguousarray(want, dtype=np.float32)
    bad = got.view(np.int32) != want.view(np.int32)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements differ from the oracle, max abs diff "
                           f"{float(np.abs(got - want).max()):.3g}")


def _edge_rois(h, w, stride, batch, seed, K):
    """Proposals plus RoIs that straddle every border and corner, clamp to 1 px, or exceed the map (image coordinates)."""
    ih, iw = h * stride, w * stride
    edge = []
    for cx, cy in [(0, ih / 2), (iw, ih / 2), (iw / 2, 0), (iw / 2, ih), (0, 0), (iw, ih), (0, ih), (iw, 0),
                   (-stride, ih / 3), (iw + stride, ih / 3), (iw / 3, -1.5 * stride), (iw / 3, ih + stride)]:
        edge.append([cx, cy, 6 * stride, 3 * stride, 0.0])
    edge += [[iw / 2, ih / 2, 0.5, 0.5, 0.0], [iw / 4, ih / 4, 0.1, 40.0, 0.0], [iw / 2, ih / 2, 4 * iw, 3 * ih, 0.0],
             [iw / 3, ih / 2, 2 * iw, 5.0, 0.0], [-4 * iw, ih / 2, 30.0, 30.0, 0.0]]
    edge = np.array(edge, np.float32)
    rng = np.random.default_rng(seed)
    edge = np.concatenate([rng.integers(0, batch, len(edge)).astype(np.float32)[:, None], edge], 1)
    props = W.proposals(K - len(edge), seed, batch=batch, canvas=max(ih, iw))
    rois = np.concatenate([edge, props]).astype(np.float32)
    return rois[rng.permutation(len(rois))]


def _single_scene(K, channels, version, out, sr, seed, theta0=True):
    rng = np.random.default_rng(seed)
    feat = rng.standard_normal((2, channels, 40, 36)).astype(np.float32)
    rois = _edge_rois(40, 36, 16, 2, seed, K)
    if theta0:
        rois[:, 5] = 0
    return Scene([feat], rois, [1 / 16], out=out, sr=sr, version=version, extend=(1.0, 1.0))


def _grad(shape, seed, dtype=torch.float32):
    return torch.randn(shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed)).to(dtype)


def _osz(scene):
    return (scene.out, scene.out) if isinstance(scene.out, int) else tuple(scene.out)


# ------------------------------------------------------------------------------------------ 1. bit-identical at theta = 0
SINGLE = [(v, sr, out, ch, K) for v in (0, 1) for sr in (1, 2, 3) for out in (7, (5, 3)) for ch in (256, 16, 6)
          for K in ((300,) if (sr + ch) % 2 else (200,))]


@pytest.mark.parametrize("version,sr,out,channels,K", SINGLE,
                         ids=[f"v{v}-sr{sr}-{'7x7' if o == 7 else '5x3'}-C{ch}-K{K}" for v, sr, o, ch, K in SINGLE])
def test_bitwise_vs_oracle_theta0(oracle, cuda, version, sr, out, channels, K):
    scene = _single_scene(K, channels, version, out, sr, 7 * sr + channels + version)
    g = _grad((K, channels) + _osz(scene), K + channels)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    for cl in (False, True):
        got = _det(scene, cl, g)
        _np_bits_equal(got[0].cpu().numpy(), want[0], f"v{version} sr={sr} out={out} C={channels} K={K} channels_last={cl}")


@pytest.mark.parametrize("K", [255, 256, 1500])
def test_bitwise_extractor_vs_oracle_theta0(oracle, cuda, K):
    """4 levels with extension and level mapping, restricted to RoIs whose device level equals the oracle's."""
    from rs_detection_b200 import core
    full = _fpn_scene(2, K, 90 + K)
    rois = full.rois_np.copy()
    rois[:, 5] = 0
    _, lv = core.roi_align_rotated_forward(full.cfg(False), full.nchw, torch.from_numpy(rois).cuda(), want_levels=True)
    keep = lv.cpu().numpy() == _levels(rois, 4, EXTEND)
    assert keep.mean() > 0.5
    scene = Scene(full.np, rois[keep], full.scales)
    g = _grad((int(keep.sum()), 256, 7, 7), K)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    for cl in (False, True):
        got = _det(scene, cl, g)
        for l in range(4):
            _np_bits_equal(got[l].cpu().numpy(), want[l], f"extractor K={K} channels_last={cl} level {l}")


@pytest.mark.parametrize("dtype", HALF, ids=HALF_IDS)
def test_half_maps_are_the_oracle_rounded_once(oracle, cuda, dtype):
    scene = _single_scene(300, 256, 1, 7, 2, 21)
    g = _grad((300, 256, 7, 7), 22)
    want = torch.from_numpy(scene.oracle_bwd(oracle, g.cpu().numpy())[0]).cuda().to(dtype)
    for cl in (False, True):
        got = _det(scene, cl, g, dtype)
        _same_bits([got[0]], [want], f"{dtype} maps channels_last={cl} vs oracle.to({dtype})")
        # a half grad_out converts exactly: the same as the fp32 call on the upcast grad_out
        gh = g.to(dtype)
        _same_bits(_det(scene, cl, gh, dtype), _det(scene, cl, gh.float(), dtype), f"{dtype} grad_out channels_last={cl}")


# ------------------------------------------------------------------------------------------ 2. general angles
GENERAL = [(kind, ch) for kind in ("v0", "v1", "fpn") for ch in (256, 260)]


@pytest.mark.parametrize("kind,channels", GENERAL, ids=[f"{k}-C{c}" for k, c in GENERAL])
def test_general_angles_vs_oracle_and_atomic(oracle, cuda, kind, channels):
    from test_gpu_roi_paths import _bwd_scene
    scene = _bwd_scene(600, channels, kind, 160 + channels)
    g = _grad((600, channels, 7, 7), 161 + channels)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    for cl in (False, True):
        got = _det(scene, cl, g)
        atomic = _atomic(scene, cl, g)
        for l in range(len(want)):
            _check(got[l].cpu().numpy(), want[l], 1e-4, f"{kind} C={channels} channels_last={cl} level {l} vs oracle")
            _check(got[l].cpu().numpy(), atomic[l].cpu().numpy(), 1e-4, f"{kind} C={channels} channels_last={cl} level {l} vs atomic")


def test_full_size_adjoint(cuda):
    """BASELINE config-1 sizes (K = 2000, C = 256, 1024^2 tile): <fwd(x), g> == <x, bwd(g)>."""
    from rs_detection_b200 import core
    shapes = W.fpn_shapes()
    gen = torch.Generator(device="cuda").manual_seed(3)
    xs = [torch.randn(s, device="cuda", generator=gen) for s in shapes]
    rois = torch.from_numpy(W.proposals(2000, 3)).cuda()
    cfg = core.make_roi_cfg(shapes, [1 / s for s in W.STRIDES], 7, 2, 1, (1.4, 1.2), 56.0)
    fx = core.roi_align_rotated_forward(cfg, xs, rois)
    g = torch.randn(fx.shape, device="cuda", generator=gen)
    gx = core.roi_align_rotated_backward(cfg, g, rois, shapes, deterministic=True)
    lhs = float((fx.double() * g.double()).sum())
    rhs = float(sum((a.double() * b.double()).sum() for a, b in zip(xs, gx)))
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), abs(rhs), 1.0)


# ------------------------------------------------------------------------------------------ 3. reproducible bits
@pytest.fixture(scope="module")
def repro(cuda):
    scene = _fpn_scene(2, 3000, 170)
    return scene, _grad((3000, 256, 7, 7), 171)


def test_two_calls(repro):
    scene, g = repro
    for cl in (False, True):
        _same_bits(_det(scene, cl, g), _det(scene, cl, g), f"two calls channels_last={cl}")


def test_layouts_agree(repro):
    scene, g = repro
    _same_bits(_det(scene, False, g), [x.contiguous() for x in _det(scene, True, g)], "NCHW vs channels-last")


def test_alignment_does_not_matter(repro):
    scene, g = repro
    ref = _det(scene, False, g)
    gs = Placed(g.shape, True, torch.float32, src=g)
    for cl in (False, True):
        _same_bits(ref, [x.contiguous() for x in _det(scene, cl, gs.t)], f"misaligned grad_out channels_last={cl}")
        _same_bits(ref, [x.contiguous() for x in _det(scene, cl, g, shifted=True)], f"misaligned maps channels_last={cl}")


def test_two_streams_at_once(repro):
    from rs_detection_b200 import core
    scene, g = repro
    cfg = scene.cfg(False)
    ref = _det(scene, False, g)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = []
    torch.cuda.synchronize()
    for s in streams:
        with torch.cuda.stream(s):
            outs.append(core.roi_align_rotated_backward(cfg, g, scene.rois, scene.shapes, deterministic=True))
    torch.cuda.synchronize()
    for i, o in enumerate(outs):
        _same_bits(ref, o, f"stream {i}")


def test_cuda_graph_replays(repro):
    from rs_detection_b200 import core
    scene, g0 = repro
    cfg = scene.cfg(False)
    g = g0.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        core.roi_align_rotated_backward(cfg, g, scene.rois, scene.shapes, deterministic=True)    # warm-up, workspace
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            grads = core.roi_align_rotated_backward(cfg, g, scene.rois, scene.shapes, deterministic=True)
    torch.cuda.current_stream().wait_stream(s)
    for i in range(10):
        gi = _grad(g.shape, 1000 + i)
        g.copy_(gi)
        for x in grads:
            x.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        _same_bits(grads, _det(scene, False, gi), f"replay {i}")


def test_batch_split(cuda):
    """One 8-image call vs eight single-image calls, each with that image's RoIs in the same relative order."""
    scene = _fpn_scene(8, 4000, 180)
    g = _grad((4000, 256, 7, 7), 181)
    batched = _det(scene, False, g)
    for i in range(8):
        rows = np.flatnonzero(scene.rois_np[:, 0] == i)
        rois = scene.rois_np[rows].copy()
        rois[:, 0] = 0
        one = Scene([f[i:i + 1] for f in scene.np], rois, scene.scales)
        got = _det(one, False, g[torch.from_numpy(rows).cuda()].contiguous())
        _same_bits([x[i:i + 1] for x in batched], got, f"image {i}")


# ------------------------------------------------------------------------------------------ 4. torch integration
@pytest.fixture
def deterministic_mode(request):
    before = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    request.addfinalizer(lambda: torch.use_deterministic_algorithms(before[0], warn_only=before[1]))
    return torch.use_deterministic_algorithms


def _modules(sr):
    from rs_detection_b200.jdet.models.roi_extractors.oriented_single_level import OrientedSingleRoIExtractor
    from rs_detection_b200.jdet.ops.roi_align_rotated import ROIAlignRotated
    from rs_detection_b200.jdet.ops.roi_align_rotated_v1 import ROIAlignRotated_v1
    ext = OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=sr), 256, STRIDES,
                                     extend_factor=EXTEND)
    return [("ROIAlignRotated_v1", ROIAlignRotated_v1(7, 1 / 8, sr), 1, False),
            ("ROIAlignRotated", ROIAlignRotated(7, 1 / 8, sr), 0, False),
            ("OrientedSingleRoIExtractor", ext, 1, True)]


def _autograd(scene, mod, multi, g):
    maps = scene.nchw if multi else scene.nchw[1:2]
    leaf = [m.detach().clone().requires_grad_(True) for m in maps]
    y = mod(leaf, scene.rois) if multi else mod(leaf[0], scene.rois)
    return leaf, y


def _direct(scene, version, multi, sr, g, deterministic):
    from rs_detection_b200 import core
    if multi:
        cfg = core.make_roi_cfg(scene.shapes, scene.scales, 7, sr, 1, EXTEND, 56.0)
        shapes = scene.shapes
    else:
        shapes = [scene.shapes[1]]
        cfg = core.make_roi_cfg(shapes, [1 / 8], 7, sr, version, (1.0, 1.0), 56.0)
    return core.roi_align_rotated_backward(cfg, g, scene.rois, shapes, deterministic=deterministic)


@pytest.fixture(scope="module")
def torch_scene(cuda):
    return _fpn_scene(2, 900, 190), _grad((900, 256, 7, 7), 191)


def test_autograd_under_deterministic_mode(torch_scene, deterministic_mode):
    scene, g = torch_scene
    deterministic_mode(True)
    for name, mod, version, multi in _modules(2):
        leaf, y = _autograd(scene, mod, multi, g)
        y.backward(g)
        _same_bits([x.grad for x in leaf], _direct(scene, version, multi, 2, g, True), name)


def test_adaptive_grid_raises_or_warns(torch_scene, deterministic_mode):
    scene, g = torch_scene
    deterministic_mode(True)
    for name, mod, version, multi in _modules(0):
        leaf, y = _autograd(scene, mod, multi, g)
        with pytest.raises(RuntimeError, match="deterministic"):
            y.backward(g)
    deterministic_mode(True, warn_only=True)
    for name, mod, version, multi in _modules(0):
        leaf, y = _autograd(scene, mod, multi, g)
        with pytest.warns(UserWarning, match="deterministic"):
            y.backward(g)
        want = _direct(scene, version, multi, 0, g, False)
        for l, (a, b) in enumerate(zip(leaf, want)):
            _check(a.grad.cpu().numpy(), b.cpu().numpy(), 1e-4, f"{name} warn_only level {l}")


def test_flag_off_keeps_the_atomic_path(torch_scene):
    from rs_detection_b200 import _lib
    scene, g = torch_scene
    assert not torch.are_deterministic_algorithms_enabled()
    for name, mod, version, multi in _modules(2):
        leaf, y = _autograd(scene, mod, multi, g)
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        y.backward(g)
        autograd_launches = _lib.launch_count() - n0
        n0 = _lib.launch_count()
        want = _direct(scene, version, multi, 2, g, False)
        assert autograd_launches == _lib.launch_count() - n0, f"{name}: not the atomic entry point"
        for l, (a, b) in enumerate(zip(leaf, want)):
            _check(a.grad.cpu().numpy(), b.cpu().numpy(), 1e-4, f"{name} flag off level {l}")


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_no_rois_gives_zero_maps(cuda, channels_last):
    from rs_detection_b200 import core
    scene = _fpn_scene(2, 0, 200, rois=np.zeros((0, 6), np.float32))
    for det in (False, True):
        for dt in (torch.float32, torch.bfloat16):
            gs = core.roi_align_rotated_backward(scene.cfg(channels_last), torch.zeros((0, 256, 7, 7), device="cuda"),
                                                 scene.rois, scene.shapes, feat_dtype=dt, deterministic=det)
            for x in gs:
                assert not torch.isnan(x.float()).any() and not x.float().any(), f"deterministic={det} {dt}: not zero"
    # the C ABI into NaN-prefilled buffers
    for x in _det(scene, channels_last, None):
        assert not x.any()
