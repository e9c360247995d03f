"""Per-stream reset (cbinfer_b200.resetStreams, cb_reset_streams): the kernel against a torch
reference at its shape edges, the reset streams against a freshly cleared model, the other streams
against a model that was never reset, and the reset inside and between CUDA graphs."""
import contextlib
import copy
import json
import os
import subprocess
import sys
from collections import Counter

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

INF = float("inf")
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


# ---- the kernel ---------------------------------------------------------------------------------

def _guarded(B, H, W, pitch_bytes, dt, shift, seed):
    """A pixel-major [B,H,W,pitch] view into random bytes with 64-byte guard regions on both sides;
    its base is 16-byte aligned plus `shift` bytes.  Returns (flat bytes, view, byte offset)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    nbytes = B * H * W * pitch_bytes
    off = 64 + shift
    flat = torch.randint(0, 256, (off + nbytes + 64,), generator=g, dtype=torch.uint8).cuda()
    view = flat[off:off + nbytes].view(dt).view(B, H, W, pitch_bytes // torch.empty(0, dtype=dt).element_size())
    return flat, view, off


def _expected(flat, off, view, channels, fill, mask):
    exp = flat.clone()
    v = exp[off:off + view.numel() * view.element_size()].view(view.dtype).view(view.shape)
    for b in range(view.shape[0]):
        if mask[b]:
            v[b, ..., :channels] = fill
            v[b, ..., channels:] = 0
    return exp


def _masks(B):
    return {"none": [0] * B, "all": [1] * B, "alternate": [1 - b % 2 for b in range(B)],
            "last": [int(b == B - 1) for b in range(B)]}


@pytest.mark.parametrize("pitch_bytes", [8, 16, 32, 272])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_reset_kernel_against_torch(dt, pitch_bytes):
    """Selected slices hold the fill in the real channels and 0 in the pad channels; every other byte,
    the guard regions included, is unchanged.  Odd H*W (slices that start and end off 16-byte
    boundaries), bases off 16-byte alignment, B = 1..5, both fills, several segments per launch."""
    from cbinfer_b200 import conv2d_cg as cg
    dtype = DTYPES[dt]
    es = torch.empty(0, dtype=dtype).element_size()
    pe = pitch_bytes // es
    seed = 0
    for B in range(1, 6):
        bufs = []
        for H, W in ((1, 1), (3, 5), (7, 9), (65, 67)):
            for channels in {pe, pe - 1, 1}:                 # no pad channel, one, all but one
                for fill, shift in ((INF, 0), (0, es)):
                    seed += 1
                    bufs.append(_guarded(B, H, W, pitch_bytes, dtype, shift, seed) + (channels, fill))
        orig = [f.clone() for f, _, _, _, _ in bufs]
        for name, m in _masks(B).items():
            for f, o in zip((b[0] for b in bufs), orig):
                f.copy_(o)
            mask = torch.tensor(m, dtype=torch.uint8, device="cuda")
            cg.reset_streams([(v, c, fill) for _, v, _, c, fill in bufs], mask)
            for (f, v, off, c, fill), o in zip(bufs, orig):
                exp = _expected(o, off, v, c, fill, m)
                assert torch.equal(f, exp), (B, name, tuple(v.shape), c, fill, off)


def test_reset_kernel_splits_many_segments_over_launches():
    """More segments than one launch's parameter block holds: every one of them is written."""
    from cbinfer_b200 import conv2d_cg as cg
    B = 3
    bufs = [_guarded(B, 5, 7, 16, torch.float32, 4 * (i % 4), 100 + i) for i in range(250)]
    orig = [f.clone() for f, _, _ in bufs]
    m = [1, 0, 1]
    cg.reset_streams([(v, 3, INF) for _, v, _ in bufs], torch.tensor(m, dtype=torch.bool, device="cuda"))
    for (f, v, off), o in zip(bufs, orig):
        assert torch.equal(f, _expected(o, off, v, 3, INF, m))


def test_reset_kernel_in_a_cuda_graph_reads_the_mask_on_the_device():
    from cbinfer_b200 import conv2d_cg as cg
    B = 5
    bufs = [_guarded(B, 7, 9, pb, dt, 0, 200 + i) + (c,)
            for i, (pb, dt, c) in enumerate(((8, torch.bfloat16, 3), (272, torch.float32, 67), (32, torch.float16, 16)))]
    orig = [f.clone() for f, _, _, _ in bufs]
    mask = torch.zeros(B, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        cg.reset_streams([(v, c, INF) for _, v, _, c in bufs], mask)      # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cg.reset_streams([(v, c, INF) for _, v, _, c in bufs], mask)
    for m in _masks(B).values():
        for (f, _, _, _), o in zip(bufs, orig):
            f.copy_(o)
        mask.copy_(torch.tensor(m, dtype=torch.uint8))
        graph.replay()
        for (f, v, off, c), o in zip(bufs, orig):
            assert torch.equal(f, _expected(o, off, v, c, INF, m)), m


# ---- models -------------------------------------------------------------------------------------

def _convs(m):
    import cbinfer_b200 as cb
    return [c for c in m.modules() if type(c) is cb.CBConv2d]


def _scene(base, candidate=True, feedback=True, thr=None):
    from cbinfer_b200 import models
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                    clonePoolOutput=False, candidateDetect=candidate)
    for c, t in zip(_convs(m), thr or []):
        c.threshold = t
    for c in _convs(m):
        c.feedbackLoop = feedback
    return m


def _thresholds(base, frame):
    from cbinfer_b200 import models
    m = _scene(base)
    return models.calibrateThresholds(base, m, frame)


@contextlib.contextmanager
def _calls():
    """Log the name of every per-frame op call in the block (as tests/test_gpu_frame_paths.py)."""
    from cbinfer_b200 import conv2d_cg as cg
    names = ("detect", "detect_u8", "detect_sparse", "detect_sparse_compact", "dilate_compact", "dilate_tiles",
             "pool_compact", "conv_update", "conv_update_tiled", "tail_update", "maxPool2d", "maxPool2d_detect")
    log = []
    orig = {n: getattr(cg, n) for n in names}

    def wrap(name):
        def w(*a, **k):
            log.append(name + ("+pool" if k.get("pool") is not None else ""))
            return orig[name](*a, **k)
        return w
    try:
        for n in names:
            setattr(cg, n, wrap(n))
        yield log
    finally:
        for n, f in orig.items():
            setattr(cg, n, f)


# the scene model's steady frame with both tile convs pooling in their epilogue and the fused 1x1 tail
FUSED_FRAME = ["detect", "dilate_tiles", "conv_update_tiled+pool", "dilate_tiles", "conv_update_tiled+pool",
               "dilate_compact", "conv_update", "tail_update"]


def _changes_of(c, streams, HW):
    """This frame's change list of layer c restricted to `streams`, indices relative to each stream;
    None for a layer whose list is only a candidate superset (the masked 1x1 layers and the fused
    tail hand one on; ChangeIndexes.tensor() refuses it with CBinferError)."""
    import cbinfer_b200 as cb
    try:
        idx = c.lastChangeIndexes().long()
    except cb._lib.CBinferError:
        return None
    return [(idx[idx // HW == b] % HW).tolist() for b in streams]


def equivalence_main(dt, candidate, feedback):
    """Run in a subprocess with CBINFER_STREAMK=0 CBINFER_KSPLIT=1 (summation order independent of
    the change count).  Prints one JSON line: the launch list of the last frame before the reset
    and those of the frames after it."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    dtype = DTYPES[dt]
    B, H, W = 4, 96, 128
    base = models.sceneLabelingBaseline().cuda().to(dtype)
    X = [f.cuda().to(dtype) for f in video.sequence(B, H, W, 9, 0.05, seed=0)]
    Y = [f.cuda().to(dtype) for f in video.sequence(B, H, W, 5, 0.05, seed=7)]
    thr = _thresholds(base, X[0])
    A, N, R = (_scene(base, candidate, feedback, thr) for _ in range(3))
    after = []
    with torch.no_grad():
        for t in range(4):
            with _calls() as steady:
                a = A(X[t])
            assert torch.equal(a, N(X[t]))
        cb.resetStreams(A, [1, 3])
        for t in range(5):
            inp = X[4 + t].clone()
            inp[[1, 3]] = Y[t][[1, 3]]
            with _calls() as log:
                a = A(inp)
            after.append(log)
            n, r = N(X[4 + t]), R(inp)
            assert torch.equal(a[[1, 3]], r[[1, 3]]), ("reset streams", t)
            assert torch.equal(a[[0, 2]], n[[0, 2]]), ("other streams", t)
            for sa, sn, sr in zip(cb.getStateTensors(A), cb.getStateTensors(N), cb.getStateTensors(R)):
                assert torch.equal(sa[[1, 3]], sr[[1, 3]]), ("state of the reset streams", t)
                assert torch.equal(sa[[0, 2]], sn[[0, 2]]), ("state of the other streams", t)
            for ca, cn, cr in zip(_convs(A), _convs(N), _convs(R)):
                HW = ca.prevOutput.shape[2] * ca.prevOutput.shape[3]
                for ref, streams in ((cr, [1, 3]), (cn, [0, 2])):
                    got, want = _changes_of(ca, streams, HW), _changes_of(ref, streams, HW)
                    assert got is None or want is None or got == want, ("change lists", streams, t)
    print(json.dumps({"steady": steady, "after": after}))


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("feedback", [True, False])
@pytest.mark.parametrize("candidate", [True, False])
def test_reset_streams_equal_a_cleared_model_and_the_others_an_untouched_one(dt, candidate, feedback):
    """Scene model, B = 4: 4 frames of X, then streams 1 and 3 start over on Y.  On every later frame
    they equal a cleared model fed Y there from Y's first frame (outputs, state, change lists), and
    streams 0 and 2 equal a model that was never reset.  Every frame after the reset launches what the
    steady frame before it did, and that frame is pinned per configuration: on the candidate path the
    first two convs take the tile path with the pool fused into their epilogue, and in fp32 the 1x1
    pair runs as the fused tail (an fp32-only kernel); without candidate detection every conv scans
    its input densely and the pools run on their own."""
    env = dict(os.environ, CBINFER_STREAMK="0", CBINFER_KSPLIT="1")
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_stream_reset import equivalence_main; "
            "equivalence_main(%r, %r, %r)" % (REPO, dt, candidate, feedback))
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    res = json.loads(p.stdout.strip().splitlines()[-1])
    steady = res["steady"]
    assert all(log == steady for log in res["after"]), res
    if candidate and dt == "f32":
        assert steady == FUSED_FRAME, steady
    elif candidate:
        assert steady.count("conv_update_tiled+pool") == 2 and "tail_update" not in steady, steady
        assert not any(op in steady for op in ("maxPool2d", "maxPool2d_detect", "pool_compact")), steady
    else:
        assert steady.count("detect") == 5 and steady.count("maxPool2d") == 2, steady
        assert not any(op.startswith("detect_sparse") or op.endswith("+pool") or op == "tail_update"
                       for op in steady), steady


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(8, 120, 160, 10, 0.05, seed=0)]
    return base, frames, _thresholds(base, frames[0])


@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_whole_batch_reset_equals_clear_memory_scene(scene, dt):
    """Default settings: resetStreams(net, range(B)) then a sequence == clearMemory then the same."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    dtype = DTYPES[dt]
    base = copy.deepcopy(base).to(dtype)
    fr = [f.to(dtype) for f in frames]
    a, c = _scene(base, thr=thr), _scene(base, thr=thr)
    with torch.no_grad():
        for f in fr[:4]:
            a(f), c(f)
        cb.resetStreams(a, range(8))
        cb.clearMemory(c)
        for f in reversed(fr[4:]):
            assert torch.equal(a(f), c(f))


def test_whole_batch_reset_equals_clear_memory_pose():
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    frames = [f.cuda().to(torch.bfloat16) for f in video.sequence(2, 96, 128, 7, 0.1, lo=-0.5, hi=0.5)]
    ms = []
    for _ in range(2):
        m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
        models.calibrateThresholds(pose, m, frames[0])
        m.parallelBranches = True
        ms.append(m)
    a, c = ms
    with torch.no_grad():
        for f in frames[:3]:
            a(f), c(f)
        cb.resetStreams(a, [0, 1])
        cb.clearMemory(c)
        for f in reversed(frames[3:]):
            (la, sa), (lc, sc) = a(f), c(f)
            assert torch.equal(la, lc) and torch.equal(sa, sc)


def test_graphs_survive_eager_and_captured_resets(scene):
    """A FrameGraph captured once keeps replaying correctly across eager resets; a graph holding
    resetStreams(net, mask) + the forward follows the mask written between replays.  Both equal the
    same schedule run eagerly."""
    import cbinfer_b200 as cb
    from cbinfer_b200.runtime import FrameGraph
    base, frames, thr = scene
    g, e = _scene(base, thr=thr), _scene(base, thr=thr)
    schedule = {5: [2], 7: [0, 7], 8: [3]}
    with torch.no_grad():
        for f in frames[:3]:
            g(f), e(f)
        static = frames[2].clone()
        fg = FrameGraph(g, static, warmup=False)
        for t in range(3, 10):
            if t in schedule:
                cb.resetStreams(g, schedule[t])
                cb.resetStreams(e, schedule[t])
            static.copy_(frames[t])
            assert torch.equal(fg.replay(), e(frames[t])), t

        g2, e2 = _scene(base, thr=thr), _scene(base, thr=thr)
        for f in frames[:3]:
            g2(f), e2(f)
        mask = torch.zeros(8, dtype=torch.bool, device="cuda")
        static2 = frames[2].clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            cb.resetStreams(g2, mask)                       # no stream selected: a no-op
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            cb.resetStreams(g2, mask)
            out = g2(static2)
        for t in range(3, 10):
            sel = schedule.get(t, [])
            mask.zero_()
            mask[sel] = True
            static2.copy_(frames[t])
            graph.replay()
            if sel:
                cb.resetStreams(e2, sel)
            assert torch.equal(out, e2(frames[t])), t


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                   and not e.name.startswith(("Memcpy", "Memset")))


def test_other_streams_stay_on_the_candidate_path(scene):
    """The frame after a one-stream reset launches the kernels of a steady frame plus the reset
    kernel: no layer falls back to a dense scan."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    m = _scene(base, thr=thr)
    mask = torch.zeros(8, dtype=torch.uint8, device="cuda")
    mask[4] = 1
    with torch.no_grad():
        for f in frames[:4]:
            m(f)
        steady = _kernel_names(lambda: m(frames[4]))

        def reset_and_frame():
            cb.resetStreams(m, mask)
            m(frames[5])
        after = _kernel_names(reset_and_frame)
    extra = after - steady
    assert not steady - after, (steady, after)
    assert len(extra) == 1 and sum(extra.values()) == 1 and "reset_streams_kernel" in next(iter(extra)), extra


def test_uint8_ingest_with_detect_input_and_the_pipeline_reset(scene):
    """uint8 frames through CBConv2d.detectInput, and FramePipeline.reset between submits: the same
    results as the eager model with the reset at the same frame."""
    import cbinfer_b200 as cb
    from cbinfer_b200.runtime import FramePipeline
    base, frames, thr = scene
    u8 = [f.mul(255).round().to(torch.uint8) for f in frames]
    a, e = _scene(base, thr=thr), _scene(base, thr=thr)
    for m in (a, e):
        _convs(m)[0].inputNorm = (255.0, 0.0)
    first = _convs(a)[0]
    with torch.no_grad():
        for t, f in enumerate(u8):
            if t == 5:
                cb.resetStreams(a, [6])
                cb.resetStreams(e, [6])
            assert torch.equal(a(first.detectInput(f)) if t >= 2 else a(f), e(f)), t

    p_model, e = _scene(base, thr=thr), _scene(base, thr=thr)
    depth = 2
    pipe = FramePipeline(p_model, frames[0], depth=depth)
    host = [f.cpu().pin_memory() for f in frames]
    with torch.no_grad():
        for _ in range(depth + 1):                          # what the pipeline ran while capturing
            e(frames[0])
        slots, ref = [], []
        for t in range(1, 10):
            if t == 6:
                pipe.reset([1, 2])
                cb.resetStreams(e, [1, 2])
            slots.append(pipe.submit(host[t]))
            ref.append(e(frames[t]).cpu())
            if len(slots) == depth:
                assert torch.equal(pipe.wait(slots[0]).clone(), ref[0])
                slots.pop(0), ref.pop(0)
        pipe.drain()
        for s, r in zip(slots, ref):
            assert torch.equal(pipe.wait(s), r)


def test_errors_and_the_no_op_before_the_first_frame(scene):
    import cbinfer_b200 as cb
    from cbinfer_b200 import models
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    m, twin = _scene(base, thr=thr), _scene(base, thr=thr)
    with torch.no_grad():
        cb.resetStreams(m, [0, 3])                          # nothing allocated yet: no-op
        cb.resetStreams(m, torch.ones(8, dtype=torch.bool, device="cuda"))
        assert torch.equal(m(frames[0]), twin(frames[0]))
        for bad in ([8], [-1]):
            with pytest.raises(CBinferError):
                cb.resetStreams(m, bad)
        with pytest.raises(CBinferError):
            cb.resetStreams(m, torch.ones(9, dtype=torch.bool, device="cuda"))
        with pytest.raises(CBinferError):
            cb.resetStreams(m, torch.ones(8, dtype=torch.bool))
        with pytest.raises(CBinferError):
            cb.resetStreams(m, torch.ones(8, dtype=torch.float32, device="cuda"))
        assert torch.equal(m(frames[1]), twin(frames[1]))  # the refused calls changed nothing
        fg = models.sceneLabelingCBinfer(base, experimentIdx=7)
        cb.resetStreams(fg, [0])                            # no state yet
        fg(frames[0])
        with pytest.raises(CBinferError):
            cb.resetStreams(fg, [0])
