"""RoIAlignRotated with channels-last RoI tensors (RSDET_ROI_NHWC_ROIS) and channels_last torch tensors.

Contract under test (include/rsdet.h): the RoI-tensor layout changes where values are stored, never what they are.
  * forward: a (K, ph, pw, C) output is, bit for bit, the (K, C, ph, pw) output of the same call permuted -- for every
    dispatch path (persistent kernel behind either prologue, roi_align_fwd_kernel<2> / <1>, the misaligned output,
    the generic kernel), both map layouts, fp32 / fp16 / bf16 maps and fp32 or half output;
  * deterministic backward: a (K, ph, pw, C) grad_out gives the same bits as the (K, C, ph, pw) one, and at theta = 0
    the oracle's bits;
  * atomic backward: agrees with the NCHW-style grad_out and with the oracle to 1e-4.
Output buffers are NaN-prefilled with guard elements on both sides; "shifted" buffers sit one element off a 16-byte
boundary.  The mirror part checks the torch layer: channels_last pyramids are read in place (no transpose launch),
their gradients come back channels_last, and `memory_format=torch.channels_last` gives a channels_last output.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import workloads as W
from test_gpu_roi_bwd_deterministic import _bits, _grad, _np_bits_equal, _same_bits, _single_scene
from test_gpu_roi_half import CODE, Placed
from test_gpu_roi_paths import STRIDES, _bwd_scene, _check, _fpn_scene, _levels

pytestmark = pytest.mark.gpu

MAPS, ROIS = 1, 2


def _cfg(scene, maps_nhwc, rois_nhwc):
    cfg = scene.cfg(maps_nhwc)
    cfg.channels_last = (MAPS if maps_nhwc else 0) | (ROIS if rois_nhwc else 0)
    return cfg


def _ws(nbytes):
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")


def _forward(cfg, feats, rois, out, lv):
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    K, fdt = rois.shape[0], CODE[feats[0].dtype]
    ws = _ws(L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 0, fdt))
    rc = L.rsdet_roi_align_rotated_forward_typed(C.byref(cfg), fdt, core._ptr_array(feats), rois.data_ptr(), K, CODE[out.dtype],
                                                 out.data_ptr(), lv.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr())
    assert rc == 0, rc


def _backward(cfg, g, rois, grads, deterministic):
    from rs_detection_b200 import _lib, core
    L = _lib.load()
    K, fdt = rois.shape[0], CODE[grads[0].dtype]
    if deterministic:
        ws = _ws(L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(C.byref(cfg), K, fdt))
        fn = L.rsdet_roi_align_rotated_backward_deterministic
    else:
        ws = _ws(L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 1, fdt))
        fn = L.rsdet_roi_align_rotated_backward_typed
    rc = fn(C.byref(cfg), CODE[g.dtype], g.data_ptr(), rois.data_ptr(), K, fdt, core._ptr_array(grads), ws.data_ptr(),
            ws.numel(), _lib.stream_ptr())
    assert rc == 0, rc


# ------------------------------------------------------------------------------------------ forward through the C ABI
def _fwd_pair(scene, maps_nhwc, shifted, fdt, odt, what):
    """The same call with an NCHW-style and an NHWC output of the same alignment class: bit-identical after permuting."""
    K = scene.rois.shape[0]
    feats = [x.to(fdt) for x in scene.feats(maps_nhwc)]
    res = {}
    for rois_nhwc in (False, True):
        cfg = _cfg(scene, maps_nhwc, rois_nhwc)
        shape = (K, cfg.pooled_h, cfg.pooled_w, cfg.channels) if rois_nhwc else (K, cfg.channels, cfg.pooled_h, cfg.pooled_w)
        out = Placed(shape, shifted, odt)
        lv = torch.full((K,), -1, dtype=torch.int32, device="cuda")
        _forward(cfg, feats, scene.rois, out.t, lv)
        assert out.guards_intact(), f"{what} rois_nhwc={rois_nhwc}: write outside the output"
        assert not torch.isnan(out.t.float()).any(), f"{what} rois_nhwc={rois_nhwc}: element left unwritten"
        assert np.array_equal(lv.cpu().numpy(), _levels(scene.rois_np, len(scene.np), scene.extend)), f"{what}: levels"
        res[rois_nhwc] = out.t.permute(0, 3, 1, 2) if rois_nhwc else out.t
    assert torch.equal(_bits(res[True]), _bits(res[False])), f"{what}: NHWC output is not the NCHW output permuted"
    return res[False]


DTYPES = [(torch.float32, torch.float32), (torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16),
          (torch.float16, torch.float32), (torch.float16, torch.float16)]
DT_IDS = ["f32", "bf16-f32out", "bf16", "f16-f32out", "f16"]
KS = [255, 256, 16384, 16385]


@pytest.fixture(scope="module")
def big_scene(cuda):
    return _fpn_scene(1, max(KS), 3)


@pytest.mark.parametrize("dts", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("shifted", [False, True], ids=["aligned", "shifted"])
@pytest.mark.parametrize("maps_nhwc", [False, True], ids=["nchw", "nhwc"])
def test_forward_77_paths(big_scene, maps_nhwc, shifted, K, dts):
    """7x7 / sr 2 / C 256, behind the ride-along prologue for NCHW maps and 256 <= K <= 16384 and roi_prep_kernel
    otherwise: aligned -> persistent kernel, shifted -> roi_align_fwd_kernel<2> with scalar stores."""
    from test_gpu_roi_paths import Scene
    scene = Scene(big_scene.np, big_scene.rois_np[:K], big_scene.scales)
    scene.nchw, scene.nhwc = big_scene.nchw, big_scene.nhwc
    _fwd_pair(scene, maps_nhwc, shifted, dts[0], dts[1], f"7x7 K={K} maps_nhwc={maps_nhwc} shifted={shifted} {dts}")


@pytest.mark.parametrize("dts", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("channels,out,sr", [(512, 5, 2), (36, 7, 2), (6, 7, 0), (8, 8, 5)],
                         ids=["fwd2-C512-5x5", "fwd1-C36", "generic-C6-sr0", "generic-C8-8x8-sr5"])
def test_forward_other_paths(oracle, cuda, channels, out, sr, dts):
    scene = _fpn_scene(2, 300, 40 + channels + sr, channels=channels, out=out, sr=sr)
    for maps_nhwc in (False, True):
        for shifted in (False, True):
            got = _fwd_pair(scene, maps_nhwc, shifted, dts[0], dts[1], f"C={channels} out={out} sr={sr} {dts}")
    if dts == (torch.float32, torch.float32):
        rows = np.arange(0, 300, 7)
        _check(got[torch.from_numpy(rows).cuda()].cpu().numpy(), scene.oracle_fwd(oracle, rows), 1e-5, "vs oracle")


def test_forward_misaligned_nhwc_maps(cuda):
    """Channels-last maps off their four-element alignment run the generic kernel for both output layouts."""
    scene = _fpn_scene(2, 600, 90)
    shifted = [Placed(x.shape, True, torch.float32, src=x) for x in scene.nhwc]
    scene.nhwc = [p.t for p in shifted]
    for out_shifted in (False, True):
        _fwd_pair(scene, True, out_shifted, torch.float32, torch.float32, f"shifted NHWC maps, out shifted={out_shifted}")


# ------------------------------------------------------------------------------------------ atomic backward
BWD = [(maps, K, ch, kind) for maps in (False, True) for K in (100, 600) for ch in (256, 260) for kind in ("v0", "fpn")]


def _atomic_maps(scene, maps_nhwc, g, rois_nhwc, dtype=torch.float32):
    cfg = _cfg(scene, maps_nhwc, rois_nhwc)
    shapes = [(s[0], s[2], s[3], s[1]) if maps_nhwc else s for s in scene.shapes]
    ps = [Placed(s, False, dtype) for s in shapes]
    _backward(cfg, g, scene.rois, [p.t for p in ps], False)
    for l, p in enumerate(ps):
        assert p.guards_intact(), f"write outside level {l}"
    return [(p.t.permute(0, 3, 1, 2) if maps_nhwc else p.t).float().cpu().numpy() for p in ps]


def _nhwc_copy(g, shifted):
    """g (K, C, ph, pw) as a (K, ph, pw, C) buffer, aligned or one element off."""
    return Placed(tuple(g.permute(0, 2, 3, 1).shape), shifted, g.dtype, src=g.permute(0, 2, 3, 1)).t


@pytest.mark.parametrize("maps_nhwc,K,channels,kind", BWD,
                         ids=[f"{'nhwc' if m else 'nchw'}-K{K}-C{ch}-{kind}" for m, K, ch, kind in BWD])
def test_atomic_backward(oracle, cuda, maps_nhwc, K, channels, kind):
    scene = _bwd_scene(K, channels, kind, 60 + K + channels)
    g = _grad((K, channels, 7, 7), K + channels)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    ref = _atomic_maps(scene, maps_nhwc, g, False)
    for shifted in (False, True):
        got = _atomic_maps(scene, maps_nhwc, _nhwc_copy(g, shifted), True)
        for l in range(len(want)):
            _check(got[l], want[l], 1e-4, f"NHWC grad_out shifted={shifted} level {l} vs oracle")
            _check(got[l], ref[l], 1e-4, f"NHWC grad_out shifted={shifted} level {l} vs NCHW grad_out")


@pytest.mark.parametrize("channels,out,sr", [(6, 7, 0), (8, 8, 5)], ids=["C6-sr0", "C8-8x8-sr5"])
def test_atomic_backward_generic(oracle, cuda, channels, out, sr):
    scene = _fpn_scene(2, 300, 50 + channels, channels=channels, out=out, sr=sr)
    g = _grad((300, channels, out, out), channels)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    for maps_nhwc in (False, True):
        for shifted in (False, True):
            got = _atomic_maps(scene, maps_nhwc, _nhwc_copy(g, shifted), True)
            for l in range(len(want)):
                _check(got[l], want[l], 1e-4, f"generic maps_nhwc={maps_nhwc} shifted={shifted} level {l}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_atomic_backward_half(cuda, dtype):
    scene = _fpn_scene(2, 600, 77)
    g = _grad((600, 256, 7, 7), 77, dtype)
    for maps_nhwc in (False, True):
        ref = _atomic_maps(scene, maps_nhwc, g, False, dtype)
        got = _atomic_maps(scene, maps_nhwc, _nhwc_copy(g, True), True, dtype)
        for l in range(len(ref)):
            scale = float(np.abs(ref[l]).max())
            assert np.abs(got[l] - ref[l]).max() <= 1e-4 * scale + scale * 2.0 ** -7, f"{dtype} level {l}"


# ------------------------------------------------------------------------------------------ deterministic backward
def _det_maps(scene, maps_nhwc, g, rois_nhwc, dtype):
    cfg = _cfg(scene, maps_nhwc, rois_nhwc)
    shapes = [(s[0], s[2], s[3], s[1]) if maps_nhwc else s for s in scene.shapes]
    ps = [Placed(s, False, dtype) for s in shapes]
    _backward(cfg, g, scene.rois, [p.t for p in ps], True)
    for l, p in enumerate(ps):
        assert p.guards_intact() and not torch.isnan(p.t.float()).any(), f"level {l}"
    return [p.t.permute(0, 3, 1, 2) if maps_nhwc else p.t for p in ps]


@pytest.mark.parametrize("maps_dtype,g_dtype", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16),
                                                (torch.float16, torch.float16), (torch.bfloat16, torch.float32)],
                         ids=["f32", "bf16", "f16", "bf16-maps-f32-grad"])
@pytest.mark.parametrize("K,channels", [(600, 256), (300, 260)])
def test_deterministic_layouts_agree(cuda, maps_dtype, g_dtype, K, channels):
    scene = _fpn_scene(2, K, 110 + channels, channels=channels)
    g = _grad((K, channels, 7, 7), K, g_dtype)
    for maps_nhwc in (False, True):
        ref = _det_maps(scene, maps_nhwc, g, False, maps_dtype)
        for shifted in (False, True):
            got = _det_maps(scene, maps_nhwc, _nhwc_copy(g, shifted), True, maps_dtype)
            _same_bits(got, ref, f"maps_nhwc={maps_nhwc} NHWC grad_out shifted={shifted}")


@pytest.mark.parametrize("version", [0, 1])
def test_deterministic_theta0_vs_oracle(oracle, cuda, version):
    scene = _single_scene(300, 256, version, 7, 2, 130 + version)
    g = _grad((300, 256, 7, 7), 131)
    want = scene.oracle_bwd(oracle, g.cpu().numpy())
    for maps_nhwc in (False, True):
        got = _det_maps(scene, maps_nhwc, _nhwc_copy(g, False), True, torch.float32)
        _np_bits_equal(got[0].cpu().numpy(), want[0], f"v{version} maps_nhwc={maps_nhwc}")


# ------------------------------------------------------------------------------------------ the torch mirror
def _launches():
    from rs_detection_b200 import _lib
    return _lib.launch_count()


def _modules(kind, memory_format=torch.contiguous_format):
    from rs_detection_b200.jdet.models.roi_extractors.oriented_single_level import OrientedSingleRoIExtractor
    from rs_detection_b200.jdet.ops.roi_align_rotated import ROIAlignRotated
    from rs_detection_b200.jdet.ops.roi_align_rotated_v1 import ROIAlignRotated_v1
    if kind == "extractor":
        return OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=2,
                                               memory_format=memory_format), 256, STRIDES, extend_factor=(1.4, 1.2))
    cls = ROIAlignRotated_v1 if kind == "v1" else ROIAlignRotated
    return cls(7, 1 / 16, 2, memory_format=memory_format)


def _run(kind, mod, feats, rois, g, deterministic=False):
    xs = [f.detach().requires_grad_(True) for f in feats]      # same storage: a misaligned level stays misaligned
    torch.cuda.synchronize()
    n0 = _launches()
    y = mod(xs, rois) if kind == "extractor" else mod(xs[0], rois)
    torch.cuda.synchronize()
    n = _launches() - n0
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(deterministic)
    try:
        y.backward(g)
    finally:
        torch.use_deterministic_algorithms(prev)
    return y.detach(), [x.grad for x in xs], n


def _mirror_scene(kind, dtype=torch.float32):
    if kind == "extractor":
        feats = [torch.from_numpy(f).cuda().to(dtype) for f in W.fpn_pyramid(2, 140, tile=256, channels=256)]
        rois = torch.from_numpy(W.proposals(200, 140, batch=2, canvas=256)).cuda()
    else:
        rng = np.random.default_rng(141)
        feats = [torch.from_numpy(rng.standard_normal((2, 256, 40, 36)).astype(np.float32)).cuda().to(dtype)]
        rois = torch.from_numpy(W.proposals(200, 141, batch=2, canvas=600)).cuda()
    return feats, rois


KINDS = ["extractor", "v1", "v0"]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("kind", KINDS)
def test_mirror_channels_last_maps(cuda, kind, dtype):
    """200 RoIs (below the locality-order threshold): NCHW maps take prologue + transpose + gather, channels-last maps
    prologue + gather."""
    feats, rois = _mirror_scene(kind, dtype)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    g = _grad((200, 256, 7, 7), 142)
    mod = _modules(kind)
    y0, g0, n0 = _run(kind, mod, feats, rois, g)
    y1, g1, n1 = _run(kind, mod, cl, rois, g)
    assert torch.equal(_bits(y1), _bits(y0)), "channels_last maps change the output"
    assert n1 == n0 - 1, f"launches: {n1} with channels_last maps, {n0} with contiguous maps (one transpose fewer expected)"
    for a, b in zip(g1, g0):
        assert a.is_contiguous(memory_format=torch.channels_last) and not a.is_contiguous(), "gradient is not channels_last"
        assert a.dtype == dtype
        scale = float(b.float().abs().max())
        tol = 1e-4 * scale + (0 if dtype == torch.float32 else scale * 2.0 ** -7)
        assert float((a.float() - b.float()).abs().max()) <= tol
    _, d0, _ = _run(kind, mod, feats, rois, g, deterministic=True)
    _, d1, _ = _run(kind, mod, cl, rois, g, deterministic=True)
    for a, b in zip(d1, d0):
        assert a.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(_bits(a), _bits(b)), "deterministic gradient differs between layouts"


@pytest.mark.parametrize("kind", KINDS)
def test_mirror_channels_last_output(cuda, kind):
    feats, rois = _mirror_scene(kind)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    g = _grad((200, 256, 7, 7), 143)
    y0, g0, _ = _run(kind, _modules(kind), feats, rois, g, deterministic=True)
    for maps in (feats, cl):
        for grad in (g, g.contiguous(memory_format=torch.channels_last)):
            y, gs, _ = _run(kind, _modules(kind, torch.channels_last), maps, rois, grad, deterministic=True)
            assert y.is_contiguous(memory_format=torch.channels_last) and not y.is_contiguous()
            assert torch.equal(_bits(y), _bits(y0))
            for a, b in zip(gs, g0):
                assert torch.equal(_bits(a), _bits(b)), "deterministic gradient depends on the RoI layout"


def test_mirror_fallbacks(cuda):
    """Mixed layouts across levels, and a channels_last level off the fast kernels' alignment, take the contiguous
    route: same output bits, same launches."""
    feats, rois = _mirror_scene("extractor")
    g = _grad((200, 256, 7, 7), 144)
    mod = _modules("extractor")
    y0, g0, n0 = _run("extractor", mod, feats, rois, g, deterministic=True)
    mixed = [f.contiguous(memory_format=torch.channels_last) if i % 2 else f for i, f in enumerate(feats)]
    shifted = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    n, c, h, w = feats[2].shape
    buf = torch.empty(n * c * h * w + 1, device="cuda")
    shifted[2] = buf[1:].view(n, h, w, c).permute(0, 3, 1, 2)
    shifted[2].copy_(feats[2])
    assert shifted[2].is_contiguous(memory_format=torch.channels_last) and shifted[2].data_ptr() % 16
    for what, fs in (("mixed", mixed), ("misaligned", shifted)):
        y, gs, n1 = _run("extractor", mod, fs, rois, g, deterministic=True)
        assert torch.equal(_bits(y), _bits(y0)), what
        assert n1 == n0, f"{what}: {n1} launches vs {n0}"
        for a, b in zip(gs, g0):
            assert torch.equal(_bits(a), _bits(b)), what


def test_mirror_cuda_graph(cuda):
    feats, rois = _mirror_scene("extractor")
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    mod = _modules("extractor", torch.channels_last)
    eager = mod(cl, rois).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        mod(cl, rois)                       # warm-up on the capture stream (workspace sizing)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y = mod(cl, rois)
    y.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert y.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(_bits(y), _bits(eager))
