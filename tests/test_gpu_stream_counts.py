"""Per-stream change counts (cbinfer_b200.trackStreamChanges, the cb_*_streams entry points): each
counting kernel against torch's bucketing of its own outputs at its shape edges, the models against an
untracked twin, the consequences the contract promises (skipped, re-fed, reset streams; an unchanged
output), CUDA graphs, FramePipeline and the launch list of a tracked step."""
import copy
import json
import os
import subprocess
import sys
from collections import Counter

import pytest
import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _rows(B, n=1):
    """a fresh counts row (garbage) and its accumulator (zero, B + 1 words as the models allocate it)"""
    return (torch.full((n * B,), -7, dtype=torch.int32, device="cuda"),
            torch.zeros(B + 1, dtype=torch.int32, device="cuda"))


def _popcount_per_stream(bits, B):
    w = bits.view(B, -1).to(torch.int64) & 0xffffffff
    return sum(((w >> i) & 1).sum(1) for i in range(32)).to(torch.int32)


def _bucket(idx, B, HW):
    idx = idx.to(torch.int64)
    return torch.bincount(idx // HW, minlength=B)[:B].to(torch.int32)


# ---- dilation + compaction: list, list + tiles, tiles only ----------------------------------------

SHAPES = [(B, W) for B in (1, 3, 8, 64) for W in (31, 32, 33, 640)]


def _raw_bits(B, H, W, fill, g):
    from cbinfer_b200 import _lib
    Wd = (W + 31) // 32
    if fill == "empty":
        m = torch.zeros(B, H, W, dtype=torch.bool)
    elif fill == "full":
        m = torch.ones(B, H, W, dtype=torch.bool)
    else:
        m = torch.rand(B, H, W, generator=g) < 0.002
        m[B // 2] = False                               # one stream without any change
    bits = torch.zeros(B * H * Wd, dtype=torch.int32, device="cuda")
    if B * H * W:
        _lib.check(_lib.C.cb_map_to_bits(_lib.stream_ptr(), m.to(torch.int8).cuda().data_ptr(), bits.data_ptr(),
                                         B, H, W))
    return bits


@pytest.mark.parametrize("k", [1, 3, 7])
@pytest.mark.parametrize("B,W", SHAPES)
def test_dilate_compact_counts_by_stream(B, W, k):
    """All three modes of dilate_compact_kernel, clear_raw on and off, empty / sparse / full maps: the row
    is the per-stream popcount of the launch's own dilated bitmap (bit-exact), every other output equals
    the untracked launch, and a second launch and two graph replays are right too (accumulator left 0).
    H = 120 at B = 64, W = 640 gives the ticketed grid (> 264 tiles); the others are fully resident, and
    whenever H * Wd is not a multiple of 512 streams straddle blocks."""
    from cbinfer_b200 import conv2d_cg as cg
    H = 120 if (B, W) == (64, 640) else 5
    Wd = (W + 31) // 32
    g = torch.Generator().manual_seed(B * 1000 + W * 10 + k)
    shape = (B, H, W)
    for fill in ("empty", "sparse", "full"):
        raw0 = _raw_bits(B, H, W, fill, g)
        for mode in ("list", "tiles", "tiles_only"):
            for clear in (False, True):
                s = cg.alloc_scratch(shape, "cuda")
                tw = cg.alloc_tile_ws(shape, "cuda")

                def run(streams):
                    raw = raw0.clone()
                    if mode == "tiles_only":
                        cg.dilate_tiles(raw, shape, (k, k), s["count"], s["ws"], s["dil_bits"], tw, clear_raw=clear,
                                        streams=streams)
                        lst = None
                    else:
                        cg.dilate_compact(raw, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"],
                                          clear_raw=clear, tile_ws=tw if mode == "tiles" else None, streams=streams)
                        lst = s["idx"][:int(s["count"].item())].clone()
                    return dict(raw=raw, bits=s["dil_bits"].clone(), count=s["count"].clone(), idx=lst,
                                ntiles=tw[1].clone() if mode != "list" else None)

                ref = run(None)
                exp = _popcount_per_stream(ref["bits"][:B * H * Wd], B)
                assert int(exp.sum()) == int(ref["count"])
                sc, acc = _rows(B)
                for rep in range(2):
                    got = run((sc, acc))
                    for key in ref:
                        if ref[key] is not None:
                            assert torch.equal(got[key], ref[key]), (fill, mode, clear, key, rep)
                    assert torch.equal(sc, exp), (fill, mode, clear, rep)
                    assert int(acc.abs().sum()) == 0
                if fill == "sparse" and clear:
                    raw = raw0.clone()
                    sc.fill_(-1)
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        if mode == "tiles_only":
                            cg.dilate_tiles(raw, shape, (k, k), s["count"], s["ws"], s["dil_bits"], tw, streams=(sc, acc))
                        else:
                            cg.dilate_compact(raw, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"],
                                              tile_ws=tw if mode == "tiles" else None, streams=(sc, acc))
                    for _ in range(2):
                        raw.copy_(raw0)
                        sc.fill_(-1)
                        graph.replay()
                        torch.cuda.synchronize()
                        assert torch.equal(sc, exp) and int(acc.abs().sum()) == 0, (mode, "graph")


# ---- small-map one-launch detection + compaction ---------------------------------------------------

@pytest.mark.parametrize("k", [1, 3, 7])
@pytest.mark.parametrize("B,W", [(1, 31), (3, 33), (8, 32), (8, 46), (64, 31)])
def test_sparse_compact_counts_by_stream(B, W, k):
    """cb_change_detect_sparse_compact_streams: the row is the popcount of the launch's dilated bitmap per
    stream; bitmaps, list, count and state equal the untracked launch; twice, and clear_raw on / off."""
    from cbinfer_b200 import _lib
    from cbinfer_b200 import conv2d_cg as cg
    H = 3 if B == 64 else 9
    C = 8
    g = torch.Generator().manual_seed(B * 100 + W + k)
    state0, sbuf = cg.pixel_major((B, C, H, W), torch.float32, "cuda", 0)
    state0.copy_(torch.rand(B, C, H, W, generator=g))
    x = state0.clone().contiguous(memory_format=torch.channels_last)
    for density in (0.0, 0.05, 1.0):
        chg = torch.rand(B, H, W, generator=g) < density
        x.copy_(state0 + chg.unsqueeze(1).cuda() * 1.0)
        cand = torch.nonzero(torch.rand(B * H * W, generator=g) < 0.5).flatten().int().cuda()
        cands = cg.ChangeIndexes.from_tensor(cand, (B, H, W))
        for clear in (False, True):
            s = cg.alloc_scratch((B, H, W), "cuda")
            sync = torch.zeros(1, dtype=torch.int32, device="cuda")

            def run(streams):
                st, _ = cg.pixel_major((B, C, H, W), torch.float32, "cuda", 0)
                st.copy_(state0)
                s["raw_bits"].zero_()
                cg.detect_sparse_compact(x, st, s["raw_bits"], 0.5, _lib.UPDATE_ALL, cands, (k, k), s["idx"],
                                         s["count"], sync, bits_are_clear=True, dil_bits=s["dil_bits"],
                                         clear_raw=clear, streams=streams)
                return [s["raw_bits"].clone(), s["dil_bits"].clone(), s["count"].clone(),
                        s["idx"][:int(s["count"].item())].clone(), st.clone()]

            ref = run(None)
            exp = _popcount_per_stream(ref[1][:B * H * ((W + 31) // 32)], B)
            sc, acc = _rows(B)
            for rep in range(2):
                got = run((sc, acc))
                assert all(torch.equal(a, b) for a, b in zip(got, ref)), (density, clear, rep)
                assert torch.equal(sc, exp) and int(acc.abs().sum()) == 0, (density, clear, rep)


# ---- a list the layer did not build ---------------------------------------------------------------

@pytest.mark.parametrize("B", [1, 3, 8, 64])
def test_stream_bucket_counts_unsorted_lists(B):
    """cb_stream_bucket: any order, duplicates counted, empty list, count read on the device; twice and
    in a graph replayed twice."""
    from cbinfer_b200 import conv2d_cg as cg
    H, W = 7, 33
    g = torch.Generator().manual_seed(B)
    for n in (0, 1, 50, 5000, B * H * W):
        idx = torch.randint(0, B * H * W, (max(n, 1),), generator=g).int().cuda()[:n]
        ci = cg.ChangeIndexes.from_tensor(idx, (B, H, W))
        exp = _bucket(idx, B, H * W)
        sc, acc = _rows(B)
        for _ in range(2):
            cg.stream_bucket(ci, (B, H, W), (sc, acc))
            assert torch.equal(sc, exp) and int(acc.abs().sum()) == 0, n
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            cg.stream_bucket(ci, (B, H, W), (sc, acc))
        for _ in range(2):
            sc.fill_(-1)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(sc, exp) and int(acc.abs().sum()) == 0, n


# ---- models against an untracked twin ------------------------------------------------------------

def _convs(m):
    import cbinfer_b200 as cb
    return [c for c in m.modules() if type(c) is cb.CBConv2d]


def _scene(base, candidate=True, feedback=True, thr=None, tiles="auto", masked=True):
    from cbinfer_b200 import models
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                    clonePoolOutput=False, candidateDetect=candidate)
    for c, t in zip(_convs(m), thr or []):
        c.threshold = t
    for c in _convs(m):
        c.feedbackLoop = feedback
        c.tileMode = tiles
        if not masked:
            c.maskedConv = False
    return m


def _outs(o):
    return list(o) if isinstance(o, (tuple, list)) else [o]


def _layer_count(c):
    """the layer's own device count of the frame: its list's count, or, where it walked a candidate
    superset (masked contraction, either layer of the fused tail), the processed pixels the kernel wrote"""
    ci = c._lastChanges
    return int((c._scratch["count"] if ci.superset else ci.count).item())


def _check_against_twin(A, R, frames, B):
    """A tracked, R untracked with exact lists: outputs and state bit-identical, row l = R's layer-l list
    bucketed by stream, row sums = A's layer counts."""
    import cbinfer_b200 as cb
    names = cb.trackStreamChanges(A, B=B)
    assert len(names) == len(_convs(A))
    counts = cb.streamChangeCounts(A)
    with torch.no_grad():
        for t, f in enumerate(frames):
            a, r = _outs(A(f)), _outs(R(f))
            for x, y in zip(a, r):
                assert torch.equal(x, y), ("outputs", t)
            for sa, sr in zip(cb.getStateTensors(A), cb.getStateTensors(R)):
                assert torch.equal(sa, sr), ("state", t)
            for l, (ca, cr) in enumerate(zip(_convs(A), _convs(R))):
                _, _, H, W = cr.prevOutput.shape
                exp = _bucket(cr.lastChangeIndexes(), B, H * W)
                assert torch.equal(counts[l], exp), (t, l, names[l], counts[l].tolist(), exp.tolist())
                assert int(counts[l].sum()) == _layer_count(ca), (t, l)
    assert cb.streamChangeCounts(A) is counts


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 8, 0.08, seed=3)]
    thr = models.calibrateThresholds(base, _scene(base), frames[0])
    return base, frames, thr


@pytest.mark.parametrize("fuse_tail", ["0", "1"])
@pytest.mark.parametrize("fuse_pool", ["0", "1"])
@pytest.mark.parametrize("tiles", ["on", "off"])
@pytest.mark.parametrize("feedback", [True, False])
@pytest.mark.parametrize("candidate", [True, False])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_scene_rows_equal_the_twins_lists(scene, monkeypatch, dt, candidate, feedback, tiles, fuse_pool, fuse_tail):
    monkeypatch.setenv("CBINFER_FUSE_POOL", fuse_pool)
    monkeypatch.setenv("CBINFER_FUSE_TAIL", fuse_tail)
    base, frames, thr = scene
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[dt]
    base = copy.deepcopy(base).to(dtype)
    fr = [f.to(dtype) for f in frames]
    A = _scene(base, candidate, feedback, thr, tiles)
    R = _scene(base, candidate, feedback, thr, tiles, masked=False)
    _check_against_twin(A, R, fr, 4)


def test_pose_rows_equal_the_twins_lists():
    """PoseModel T=2 in bf16: small maps (one-launch detection + compaction), layers behind torch.cat."""
    from cbinfer_b200 import models, video
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    frames = [f.cuda().to(torch.bfloat16) for f in video.sequence(2, 96, 128, 6, 0.1, lo=-0.5, hi=0.5, seed=5)]

    def make(masked):
        m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
        models.calibrateThresholds(pose, m, frames[0])
        for c in _convs(m):
            c.maskedConv = c.maskedConv and masked
        return m
    _check_against_twin(make(True), make(False), frames, 2)


def test_finegrained_tensor_core_layer():
    """Fine-grained layer on the tensor cores: the first (dense) frame counts every pixel, later frames
    the touched output pixels."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import video
    torch.manual_seed(0)
    m = cb.convert(nn.Sequential(nn.Conv2d(3, 16, 3, padding=1)).cuda(), threshold=0.05)
    layer = _convs(m)[0]
    layer.finegrained = True
    B, H, W = 3, 40, 72
    cb.trackStreamChanges(m, B=B)
    counts = cb.streamChangeCounts(m)
    with torch.no_grad():
        for t, f in enumerate(video.sequence(B, H, W, 4, 0.05, seed=1)):
            m(f.cuda())
            exp = torch.full((B,), H * W, dtype=torch.int32, device="cuda") if t == 0 \
                else _bucket(layer.lastChangeIndexes(), B, H * W)
            assert torch.equal(counts[0], exp), t


def test_batch_mismatch_raises(scene):
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    m = _scene(base, thr=thr)
    cb.trackStreamChanges(m, B=3)
    with pytest.raises(CBinferError, match="3 streams"):
        m(frames[0])
    cb.trackStreamChanges(m, enable=False)
    m(frames[0])


# ---- what the contract promises -------------------------------------------------------------------

def test_skipped_refed_and_reset_streams(scene):
    """Stream 1 skipped by the mask and stream 2 fed its previous frame get 0 in every row; on the frame
    after resetStreams, stream 3 gets H_l * W_l in every row; a stream whose last row is 0 keeps its
    output rows bit for bit."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    m = _scene(base, thr=thr)
    B = 4
    with torch.no_grad():
        m(frames[0])
        names = cb.trackStreamChanges(m)
        counts = cb.streamChangeCounts(m)
        cb.setActiveStreams(m, [0, 1, 2, 3])
        last = frames[0]
        for t in range(1, len(frames)):
            f = frames[t].clone()
            f[2] = last[2]                                     # stream 2: its previous frame again
            if t == 4:
                cb.resetStreams(m, [3])
            cb.setActiveStreams(m, [0, 2, 3])                  # stream 1 skipped
            prev = _convs(m)[-1].prevOutput.clone()
            out = _outs(m(f))[0].clone()
            c = counts.clone()
            assert int(c[:, 1].abs().sum()) == 0 and int(c[:, 2].abs().sum()) == 0, (t, c.tolist())
            if t == 4:
                for l, conv in enumerate(_convs(m)):
                    _, _, H, W = conv.prevOutput.shape
                    assert int(c[l, 3]) == H * W, (names[l], c[:, 3].tolist())
            for b in range(B):
                if int(c[-1, b]) == 0:
                    assert torch.equal(out[b], prev[b]), (t, b)
            f[1] = last[1]
            last = f


# ---- graphs and the pipeline -------------------------------------------------------------------

def test_graph_ring_matches_eager(scene):
    """One graph per input slot of a ring, replayed in turn: the counts after each replay equal an eager
    tracked twin's."""
    import cbinfer_b200 as cb
    from cbinfer_b200.runtime import FrameGraph
    base, frames, thr = scene
    G, E = _scene(base, thr=thr), _scene(base, thr=thr)
    slots = [frames[0].clone() for _ in range(3)]
    with torch.no_grad():
        G(frames[0])
        cb.trackStreamChanges(G)
        graphs = [FrameGraph(G, s) for s in slots]            # warm-up runs: frames[0] three more times
        for _ in range(4):
            E(frames[0])
        cb.trackStreamChanges(E)
        cg_counts, e_counts = cb.streamChangeCounts(G), cb.streamChangeCounts(E)
        for t in range(1, len(frames)):
            slots[t % 3].copy_(frames[t])
            graphs[t % 3].replay()
            E(frames[t])
            assert torch.equal(cg_counts, e_counts), t


def test_frame_pipeline_change_counts(scene):
    """uint8 FramePipeline(trackChanges=True): changeCounts(slot) after wait(slot) equals an eager twin."""
    import cbinfer_b200 as cb
    from cbinfer_b200.runtime import FramePipeline
    base, frames, thr = scene
    u8 = [f.mul(255).round().to(torch.uint8) for f in frames]
    p_model, e = _scene(base, thr=thr), _scene(base, thr=thr)
    for m in (p_model, e):
        _convs(m)[0].inputNorm = (255.0, 0.0)
    depth = 2
    pipe = FramePipeline(p_model, u8[0], depth=depth, trackChanges=True)
    host = [f.cpu().pin_memory() for f in u8]
    with torch.no_grad():
        for _ in range(depth + 1):
            e(u8[0])
        cb.trackStreamChanges(e)
        slots, ref = [], []
        for t in range(1, len(u8)):
            slots.append(pipe.submit(host[t]))
            e(u8[t])
            ref.append(cb.streamChangeCounts(e).cpu())
            if len(slots) == depth:
                s = slots.pop(0)
                pipe.wait(s)
                assert torch.equal(pipe.changeCounts(s), ref.pop(0)), t
        pipe.drain()
        for s, r in zip(slots, ref):
            pipe.wait(s)
            assert torch.equal(pipe.changeCounts(s), r)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
            and not e.name.startswith(("Memcpy", "Memset"))]


def launch_list_main():
    """bench.py's workload (8 x 640x480, candidate path): the kernels of an untracked step and of a
    tracked one, by function name (without template arguments: the tracked ones are other
    instantiations of the same kernels)."""
    import re
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(8, 480, 640, 5, 0.05, seed=0)]
    m = _scene(base)
    models.calibrateThresholds(base, m, frames[0], factor=0.02)
    first = _convs(m)[0]

    def base_name(n):
        n = re.sub(r"\(.*$", "", n)
        while "<" in n:
            n = re.sub(r"<[^<>]*>", "", n)
        return n.split()[-1]
    with torch.no_grad():
        for f in frames[:3]:
            m(f)
        plain = Counter(base_name(n) for n in _kernel_names(lambda: m(first.detectInput(frames[3]))))
        cb.trackStreamChanges(m)
        tracked = Counter(base_name(n) for n in _kernel_names(lambda: m(first.detectInput(frames[4]))))
    print(json.dumps({"plain": plain, "tracked": tracked}))


def test_tracked_step_launches_what_an_untracked_one_does():
    """A tracked step launches the same 8 kernels as an untracked one: no launch and no memset added."""
    code = "import sys; sys.path.insert(0, %r); from tests.test_gpu_stream_counts import launch_list_main; " \
           "launch_list_main()" % REPO
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    assert res["plain"] == res["tracked"], res
    assert sum(res["plain"].values()) == 8, res
