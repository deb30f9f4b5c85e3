"""The timed step of bench.py, as it runs, against the oracle.

bench.py measures one 8-tile step (`run_ours` -> `device_step`): eight obb2poly + multiclass_nms_rotated chains on
high-priority side streams (each multiclass call forks its class sort onto a library-internal side lane) and ONE
extractor call over all 8 tiles -- 32 000 RoIs, batch 8, which takes the lean `roi_prep_kernel` prologue
(K > kPrepMaxRois) instead of the transpose ride-along every per-tile call takes -- captured once into a CUDA graph
and replayed.  These tests rebuild that step, check every output of an eager step against the oracle and against
per-tile extractor calls, check that graph replays (also after the inputs are overwritten in place) reproduce the
eager step bit for bit for several stream / batch layouts, tie the test's step to bench's own through
`bench.py --dump-outputs`, and check that scratch buffers a captured graph uses outlive workspace growth and
`release_workspaces()`.

All 8 tiles of the step are checked against the oracle: its multiclass NMS takes about 5 s per tile of 4000 x 10
candidates on one CPU core, and the 8 tiles run in parallel threads, once per module.
"""
import concurrent.futures as cf
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
import workloads as W
from helpers import close_report

pytestmark = pytest.mark.gpu

T = bench.TILES_PER_GPU
K = bench.K_ROIS
ROWS_PER_TILE = 64                       # seeded RoI rows per tile checked against the oracle
LAYOUTS = [(1, 8), (2, 1), (8, 8), (8, 2)]   # (streams, tiles per extractor call)
POLY_TOL = 1e-4 * W.TILE                 # obb2poly tolerance of tests/test_gpu_fuzz.py
NAN = float("nan")


def _rows(t):
    return np.sort(np.random.default_rng(t).choice(K, ROWS_PER_TILE, replace=False))


def _oracle_tile(O, inp, t):
    feats, rois, boxes, scores = inp
    dets, labels = O.multiclass_nms_rotated(boxes, scores, bench.SCORE_THR, dict(iou_thr=bench.IOU_THR), bench.MAX_NUM)
    feat_rows, _ = O.oriented_extractor_fwd(feats, rois[_rows(t)], list(W.STRIDES), extend_factor=bench.EXTEND)
    return dict(dets=dets, labels=labels, polys=O.obb2poly(boxes), rows=_rows(t), feat_rows=feat_rows)


@pytest.fixture(scope="module")
def tiles_np():
    return [bench.tile_inputs(t) for t in range(T)]


@pytest.fixture(scope="module")
def want(oracle, tiles_np):
    """oracle results of the 8 bench tiles (NMS, polygons, 64 RoI rows each), computed once"""
    with cf.ThreadPoolExecutor(T) as ex:        # the oracle's C calls release the GIL
        return list(ex.map(lambda t: _oracle_tile(oracle, tiles_np[t], t), range(T)))


class Inputs:
    """The bench tiles on the device, laid out as bench.py run_ours does: the 8 pyramids as one batch per level,
    a tile's own pyramid a view into it."""

    def __init__(self, tiles_np):
        self.feats8 = [torch.from_numpy(np.concatenate([t[0][l] for t in tiles_np], 0)).cuda() for l in range(len(W.STRIDES))]
        self.rois = [torch.from_numpy(t[1]).cuda() for t in tiles_np]
        self.boxes = [torch.from_numpy(t[2]).cuda() for t in tiles_np]
        self.scores = [torch.from_numpy(t[3]).cuda() for t in tiles_np]

    def feats(self, i):
        return [f8[i:i + 1] for f8 in self.feats8]


@pytest.fixture(scope="module")
def base(cuda, tiles_np):
    return Inputs(tiles_np)


def _cfg(batch):
    from rs_detection_b200 import core
    return core.make_roi_cfg([(batch,) + tuple(sh[1:]) for sh in W.fpn_shapes()], [1.0 / s for s in W.STRIDES], 7, 2, 1,
                             bench.EXTEND, 56.0)


@pytest.fixture(scope="module")
def ref8(base):
    """RoI features of every tile from its own per-tile extractor call (4000 RoIs, batch 1: the `ride` prologue), in
    the row order of the batched output"""
    from rs_detection_b200 import core
    cfg = _cfg(1)
    out = torch.empty((T * K, W.CHANNELS, 7, 7), dtype=torch.float32, device="cuda")
    for i in range(T):
        core.roi_align_rotated_forward(cfg, base.feats(i), base.rois[i], out=out[i * K:(i + 1) * K])
    torch.cuda.synchronize()
    return out


@pytest.fixture(scope="module")
def streams(cuda):
    """created once per module (the NMS side lanes are per caller stream, at most 256 per process)"""
    n = max(8, bench.NSTREAMS)
    return ([torch.cuda.Stream(priority=bench.NMS_PRIO) for _ in range(n)],
            [torch.cuda.Stream() for _ in range(n)])


class Step:
    """bench.py run_ours `device_step` on a private copy of the inputs, for `nstreams` NMS streams (and as many
    extractor streams) and `roi_batch` tiles per extractor call."""

    def __init__(self, base, streams, nstreams, roi_batch):
        assert roi_batch in (1, 2, 4, 8)
        self.base, self.nstreams, self.roi_batch = base, nstreams, roi_batch
        self.side = streams[0][:nstreams]
        self.side2 = streams[1][:nstreams]
        self.feats8 = [f.clone() for f in base.feats8]
        self.tiles = [([f8[i:i + 1] for f8 in self.feats8], base.rois[i].clone(), base.boxes[i].clone(), base.scores[i].clone())
                      for i in range(T)]
        self.rois8 = torch.cat([torch.cat([torch.full((K, 1), float(i), device="cuda"), t[1][:, 1:]], 1)
                                for i, t in enumerate(self.tiles)], 0).contiguous()
        self.cfg8, self.cfgb = _cfg(T), _cfg(roi_batch)
        self.roisb = [torch.cat([torch.cat([torch.full((K, 1), float(j), device="cuda"), self.tiles[g * roi_batch + j][1][:, 1:]], 1)
                                 for j in range(roi_batch)], 0).contiguous() for g in range(T // roi_batch)]
        self.out8 = torch.empty((T * K, W.CHANNELS, 7, 7), dtype=torch.float32, device="cuda")

    def load(self, perm):
        """overwrite the inputs IN PLACE: slot i gets bench tile perm[i] (captured graphs keep their addresses)"""
        for i, t in enumerate(perm):
            for f8, b8 in zip(self.feats8, self.base.feats8):
                f8[i].copy_(b8[t])
            _, rois, boxes, scores = self.tiles[i]
            rois.copy_(self.base.rois[t])
            boxes.copy_(self.base.boxes[t])
            scores.copy_(self.base.scores[t])
            self.rois8[i * K:(i + 1) * K, 1:].copy_(self.base.rois[t][:, 1:])
            g, j = divmod(i, self.roi_batch)
            self.roisb[g][j * K:(j + 1) * K, 1:].copy_(self.base.rois[t][:, 1:])

    def __call__(self):
        # Issues exactly what bench.py `device_step` (run_ours, bench.py:403-427) issues: fork every stream from the
        # current one, per tile obb2poly + multiclass_nms_rotated on side[i % nstreams], the extractor call(s) on
        # side2[g % nstreams], join.  Keep the two in step.
        from rs_detection_b200 import core
        main = torch.cuda.current_stream()
        for st in self.side + self.side2:
            st.wait_stream(main)
        results = []
        for i, (feats, rois, boxes, scores) in enumerate(self.tiles):
            with torch.cuda.stream(self.side[i % self.nstreams]):
                polys = core.obb2poly(boxes)
                results.append((polys,) + core.multiclass_nms_rotated(boxes, scores, bench.SCORE_THR, bench.IOU_THR, bench.MAX_NUM))
        for g in range(T // self.roi_batch):
            with torch.cuda.stream(self.side2[g % self.nstreams]):
                if self.roi_batch == T:
                    core.roi_align_rotated_forward(self.cfg8, self.feats8, self.rois8, out=self.out8)
                else:
                    lo, hi = g * self.roi_batch, (g + 1) * self.roi_batch
                    core.roi_align_rotated_forward(self.cfgb, [f8[lo:hi] for f8 in self.feats8], self.roisb[g],
                                                   out=self.out8[lo * K:hi * K])
        for st in self.side + self.side2:
            main.wait_stream(st)
        return results


def _snapshot(step, results):
    """copies of what a step left behind (detections cut to the kept count)"""
    torch.cuda.synchronize()
    counts = [int(r[3].item()) for r in results]
    return dict(out8=step.out8.clone(), counts=counts, polys=[r[0].clone() for r in results],
                dets=[r[1][:k].clone() for r, k in zip(results, counts)],
                labels=[r[2][:k].clone() for r, k in zip(results, counts)])


def _assert_identical(got, ref, what):
    assert got["counts"] == ref["counts"], f"{what}: kept counts {got['counts']} != {ref['counts']}"
    for i in range(T):
        assert torch.equal(got["polys"][i], ref["polys"][i]), f"{what}: tile slot {i} polygons differ"
        assert torch.equal(got["dets"][i], ref["dets"][i]), f"{what}: tile slot {i} detections differ"
        assert torch.equal(got["labels"][i], ref["labels"][i]), f"{what}: tile slot {i} labels differ"
    _assert_rows_equal(got["out8"], ref["out8"], what)


def _assert_rows_equal(got, ref, what):
    if torch.equal(got, ref):
        return
    diff = (got != ref).flatten(1).any(1)
    err = (got - ref).abs().nan_to_num(float("inf")).max().item()
    raise AssertionError(f"{what}: {int(diff.sum())} of {got.shape[0]} RoI feature rows differ (max abs err {err:.3g}); "
                         f"first differing rows {torch.nonzero(diff).flatten()[:8].tolist()}")


def _check_vs_reference(snap, want, ref8, perm=tuple(range(T))):
    """every output of a step against the oracle (slot i holds bench tile perm[i]) and the RoI features against the
    per-tile extractor calls"""
    out8 = snap["out8"]
    nan_rows = torch.isnan(out8).flatten(1).any(1)
    assert not bool(nan_rows.any()), \
        f"{int(nan_rows.sum())} RoI feature rows keep the NaN prefill, e.g. rows {torch.nonzero(nan_rows).flatten()[:8].tolist()}"
    for i, t in enumerate(perm):
        w = want[t]
        k = snap["counts"][i]
        assert k == w["dets"].shape[0], f"slot {i} (tile {t}): {k} detections kept, oracle keeps {w['dets'].shape[0]}"
        assert np.array_equal(snap["dets"][i].cpu().numpy(), w["dets"]), f"slot {i} (tile {t}): detections differ from the oracle"
        assert np.array_equal(snap["labels"][i].cpu().numpy(), w["labels"]), f"slot {i} (tile {t}): labels differ from the oracle"
        perr = float(np.abs(snap["polys"][i].cpu().numpy().astype(np.float64) - w["polys"]).max())
        assert perr <= POLY_TOL, f"slot {i} (tile {t}): obb2poly max abs err {perr:.3g}"
        got = out8[i * K + torch.from_numpy(w["rows"]).cuda()].cpu().numpy()
        scale = float(np.abs(w["feat_rows"]).max())
        nbad, err, _ = close_report(got, w["feat_rows"], 1e-5, 1e-5 * scale)
        assert nbad == 0, f"slot {i} (tile {t}): {nbad} RoI feature values off the oracle (max abs err {err:.3g}, scale {scale:.3g})"
        # The batched call (lean prologue, batch-aware locality order) and the per-tile call (prologue riding with the
        # transpose) run the same geometry and gather arithmetic per RoI: only WHICH CTA takes a RoI differs.
        _assert_rows_equal(out8[i * K:(i + 1) * K], ref8[t * K:(t + 1) * K], f"slot {i} (tile {t}) vs its per-tile extractor call")


def _eager(step):
    step.out8.fill_(NAN)
    return _snapshot(step, step())


def _capture(step, warmup=2):
    """warm up, then capture the step once, as bench.py does"""
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        results = step()
    return graph, results


def _replay(graph, step, results):
    step.out8.fill_(NAN)       # a row the replay skips cannot inherit an earlier step's value
    graph.replay()
    return _snapshot(step, results)


@pytest.mark.parametrize("nstreams,roi_batch", LAYOUTS, ids=[f"s{s}-b{b}" for s, b in LAYOUTS])
def test_eager_step_vs_oracle(base, streams, want, ref8, nstreams, roi_batch):
    step = Step(base, streams, nstreams, roi_batch)
    _check_vs_reference(_eager(step), want, ref8)


@pytest.mark.parametrize("nstreams,roi_batch", LAYOUTS, ids=[f"s{s}-b{b}" for s, b in LAYOUTS])
def test_graph_replay(base, streams, want, ref8, nstreams, roi_batch):
    step = Step(base, streams, nstreams, roi_batch)
    eager = _eager(step)
    graph, results = _capture(step)
    for r in range(3):
        _assert_identical(_replay(graph, step, results), eager, f"replay {r} vs the eager step")
    # new inputs in the captured tensors: nothing may have been decided on the host at capture time, and the device
    # state a step leaves behind (work counter of the persistent gather, NMS counters) must be reset by the replay
    perm = [(i + 1) % T for i in range(T)]
    step.load(perm)
    replayed = _replay(graph, step, results)
    _check_vs_reference(replayed, want, ref8, perm)
    _assert_identical(replayed, _eager(step), "replay on new inputs vs an eager step on them")
    del graph


def test_bench_dump_matches(base, streams, tiles_np, want, oracle, tmp_path):
    """bench.py's own timed step (what its `value` measures) dumps what it computed: it must agree with the oracle
    and, bit for bit, with a replay of this module's copy of the step."""
    env = dict(os.environ)
    cmd = [sys.executable, os.path.join(bench.ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--no-cpu-baseline", "--no-verify", "--dump-outputs", str(tmp_path)]
    p = subprocess.run(cmd, cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0, p.stderr[-4000:]
    json.loads(p.stdout.strip().splitlines()[-1])
    d = {n: np.load(tmp_path / f"{n}.npy") for n in
         ("roi_feature_rows", "roi_features", "polygons", "detections", "labels", "detections_per_tile")}

    # against the oracle
    counts = [w["dets"].shape[0] for w in want]
    assert d["detections_per_tile"].tolist() == counts
    assert np.array_equal(d["detections"], np.concatenate([w["dets"] for w in want]))
    assert np.array_equal(d["labels"], np.concatenate([w["labels"] for w in want]).astype(np.float32))
    assert d["polygons"].shape == (T, K, 8)
    assert float(np.abs(d["polygons"].astype(np.float64) - np.stack([w["polys"] for w in want])).max()) <= POLY_TOL
    rows = d["roi_feature_rows"].astype(np.int64)
    wf = np.empty_like(d["roi_features"])
    for t in range(T):
        m = rows // K == t
        wf[m], _ = oracle.oriented_extractor_fwd(tiles_np[t][0], tiles_np[t][1][rows[m] % K], list(W.STRIDES),
                                                 extend_factor=bench.EXTEND)
    scale = float(np.abs(wf).max())
    nbad, err, _ = close_report(d["roi_features"], wf, 1e-5, 1e-5 * scale)
    assert nbad == 0, f"{nbad} dumped RoI feature values off the oracle (max abs err {err:.3g}, scale {scale:.3g})"

    # against a replay of this module's step in bench's layout
    step = Step(base, streams, bench.NSTREAMS, bench.ROI_BATCH)
    graph, results = _capture(step)
    snap = _replay(graph, step, results)
    assert np.array_equal(snap["out8"][torch.from_numpy(rows).cuda()].cpu().numpy(), d["roi_features"])
    assert np.array_equal(np.stack([p_.cpu().numpy() for p_ in snap["polys"]]), d["polygons"])
    assert snap["counts"] == counts
    assert np.array_equal(np.concatenate([x.cpu().numpy() for x in snap["dets"]]), d["detections"])
    assert np.array_equal(np.concatenate([x.cpu().numpy() for x in snap["labels"]]).astype(np.float32), d["labels"])
    del graph


@pytest.fixture(scope="module")
def lifetime_streams(cuda):
    return {"grow": torch.cuda.Stream(), "release": torch.cuda.Stream()}


@pytest.mark.parametrize("how", ["grow", "release"])
def test_graph_scratch_outlives_workspace_cache(base, tiles_np, want, lifetime_streams, how):
    """A captured graph keeps the raw addresses of its scratch.  Growing the stream's cached NMS workspace after the
    capture, or releasing the cache, must not hand that scratch to another tensor: replays would write into it."""
    from rs_detection_b200 import _lib, core
    S = lifetime_streams[how]
    key = (torch.cuda.current_device(), S.cuda_stream, "nms")
    nms = lambda b, s: core.multiclass_nms_rotated(b, s, bench.SCORE_THR, bench.IOU_THR, bench.MAX_NUM)
    with torch.cuda.stream(S):
        nms(base.boxes[0], base.scores[0])          # eager: S's scratch comes from S's ordinary pool
    S.synchronize()
    old = _lib._workspaces[key]
    old_ptr, old_bytes = old.data_ptr(), old.numel()
    del old
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=S):
        dets, labels, cnt = nms(base.boxes[0], base.scores[0])
    assert _lib._workspaces[key].data_ptr() == old_ptr

    if how == "grow":                               # n = 8000, 10 classes: a larger "nms" workspace on S
        big_b = torch.from_numpy(np.concatenate([tiles_np[0][2], tiles_np[1][2]])).cuda()
        big_s = torch.from_numpy(np.concatenate([tiles_np[0][3], tiles_np[1][3]])).cuda()
        with torch.cuda.stream(S):
            nms(big_b, big_s)
        assert _lib._workspaces[key].data_ptr() != old_ptr
    else:
        _lib.release_workspaces()
    with torch.cuda.stream(S):                      # the caching allocator pools blocks per stream
        victims = [torch.full((old_bytes,), 0xA5, dtype=torch.uint8, device="cuda") for _ in range(4)]
    landed = [v.data_ptr() for v in victims if old_ptr <= v.data_ptr() < old_ptr + old_bytes]
    with torch.cuda.stream(S):
        graph.replay()
    torch.cuda.synchronize()
    changed = [i for i, v in enumerate(victims) if not bool((v == 0xA5).all())]
    assert not changed, f"graph replay wrote into tensors allocated after the workspace cache was changed ({how}): victims {changed}"
    assert not landed, f"the graph's scratch at {old_ptr:#x} was freed and reallocated to {landed}"
    k = int(cnt.item())
    assert k == want[0]["dets"].shape[0]
    assert np.array_equal(dets[:k].cpu().numpy(), want[0]["dets"])
    assert np.array_equal(labels[:k].cpu().numpy(), want[0]["labels"])
    del graph
