"""Active-stream mask (cbinfer_b200.setActiveStreams, cb_change_detect_streams): every dense detection
kernel against its unmasked launch at its shape edges, masked models against re-feeding the skipped
streams their previous frame, the edge cases of fresh and reset streams, CUDA graphs, the launch list
and FramePipeline's partial uploads."""
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

INF = float("inf")
GUARD = 64


# ---- the kernels --------------------------------------------------------------------------------

def _masks(B):
    return {"all": [1] * B, "none": [0] * B, "alternate": [1 - b % 2 for b in range(B)],
            "first": [int(b == 0) for b in range(B)], "last": [int(b == B - 1) for b in range(B)]}


class Guarded(object):
    """A [B, ...] tensor view inside a flat byte buffer with GUARD random bytes on both sides; the
    view's per-stream slices are contiguous byte ranges of `slice_bytes` each."""

    def __init__(self, B, inner_shape, dtype, values, g):
        es = torch.empty(0, dtype=dtype).element_size()
        n = 1
        for d in inner_shape:
            n *= d
        self.slice_bytes = n * es
        self.B = B
        flat = torch.randint(0, 256, (2 * GUARD + B * n * es,), generator=g, dtype=torch.uint8)
        body = flat[GUARD:GUARD + B * n * es].view(dtype)
        body.copy_(values(B * n).to(dtype))
        self.flat = flat.cuda()
        self.buf = self.flat[GUARD:GUARD + B * n * es].view(dtype).view((B,) + tuple(inner_shape))

    def expected(self, ref_flat, orig_flat, mask):
        """ref's bytes in the active streams' slices, orig's everywhere else (guards included)."""
        exp = orig_flat.clone()
        for b in range(self.B):
            if mask[b]:
                lo = GUARD + b * self.slice_bytes
                exp[lo:lo + self.slice_bytes] = ref_flat[lo:lo + self.slice_bytes]
        exp[:GUARD] = ref_flat[:GUARD]
        exp[-GUARD:] = ref_flat[-GUARD:]
        return exp


def _pitch(dtype, C):
    v = 16 // torch.empty(0, dtype=dtype).element_size()
    return (C + v - 1) // v * v


# variant -> (x dtype, state dtype, C, H, W, x layout, state layout, kernel name)
#   layouts: 'pm' pixel-major [B,H,W,pitch], 'nchw' planar, 'hwc' uint8 interleaved (x only)
VARIANTS = {
    "vec_wlog0_f32": (torch.float32, torch.float32, 4, 3, 37, "pm", "pm", "detect_vec_kernel"),
    "vec_wlog0_c20_f32": (torch.float32, torch.float32, 20, 3, 37, "pm", "pm", "detect_vec_kernel"),
    "vec_wlog1_f32": (torch.float32, torch.float32, 128, 2, 33, "pm", "pm", "detect_vec_kernel"),
    "vec_wlog2_f32": (torch.float32, torch.float32, 256, 2, 33, "pm", "pm", "detect_vec_kernel"),
    "vec_wlog3_f32": (torch.float32, torch.float32, 512, 1, 33, "pm", "pm", "detect_vec_kernel"),
    "vec_bf16": (torch.bfloat16, torch.bfloat16, 24, 3, 37, "pm", "pm", "detect_vec_kernel"),
    "vec_wlog1_f16": (torch.float16, torch.float16, 256, 1, 40, "pm", "pm", "detect_vec_kernel"),
    "narrow_f32": (torch.float32, torch.float32, 3, 5, 45, "nchw", "pm", "detect_narrow_kernel"),
    "narrow_f16": (torch.float16, torch.float16, 3, 5, 45, "nchw", "pm", "detect_narrow_kernel"),
    "narrow_bf16": (torch.bfloat16, torch.bfloat16, 7, 5, 45, "nchw", "pm", "detect_narrow_kernel"),
    "u8_hwc": (torch.uint8, torch.float32, 3, 5, 45, "hwc", "pm", "detect_narrow_kernel"),
    "u8_planar": (torch.uint8, torch.float32, 3, 5, 45, "nchw", "pm", "detect_narrow_kernel"),
    # H*Wd = 5*2 = 10 words per stream, 4 words per block: blocks straddle stream boundaries
    "planar_f32_straddle": (torch.float32, torch.float32, 16, 5, 40, "nchw", "pm", "detect_planar_kernel"),
    "planar_bf16_straddle": (torch.bfloat16, torch.bfloat16, 24, 3, 37, "nchw", "pm", "detect_planar_kernel"),
    "planar_f32_c64": (torch.float32, torch.float32, 64, 3, 50, "nchw", "pm", "detect_planar_kernel"),
    "generic_f32": (torch.float32, torch.float32, 5, 3, 37, "nchw", "nchw", "detect_generic_kernel"),
    "generic_f16": (torch.float16, torch.float16, 3, 3, 33, "nchw", "nchw", "detect_generic_kernel"),
}


def _x(B, C, H, W, dtype, layout, active, g):
    """The input frame; the slices of inactive streams hold values that would flag every pixel and be
    written into the state if they were read (far from every state value, never NaN)."""
    if dtype == torch.uint8:
        v = torch.randint(0, 256, (B, C, H, W), generator=g, dtype=torch.uint8)
        far = 255
    else:
        v = torch.rand(B, C, H, W, generator=g).to(dtype)
        far = 1e4 if dtype == torch.float16 else 1e30
    for b in range(B):
        if not active[b]:
            v[b] = far
    if layout == "nchw":
        return v.cuda()
    if layout == "hwc":
        return v.permute(0, 2, 3, 1).contiguous().cuda().permute(0, 3, 1, 2)
    p = _pitch(dtype, C) + (_pitch(dtype, 1) if C % 8 == 4 else 0)   # a pitch wider than needed on some shapes
    buf = torch.zeros(B, H, W, p, dtype=dtype)
    buf[..., :C] = v.permute(0, 2, 3, 1)
    return buf.cuda().permute(0, 3, 1, 2)[:, :C]


def _state(B, C, H, W, dtype, layout, g):
    # in [0, 0.5): a skipped uint8 stream's x (255/255 = 1) would flag every pixel at threshold 0.3
    vals = lambda n: torch.rand(n, generator=g) * 0.5                 # noqa: E731
    if layout == "nchw":
        st = Guarded(B, (C, H, W), dtype, vals, g)
        return st, st.buf
    p = _pitch(dtype, C)
    st = Guarded(B, (H, W, p), dtype, vals, g)
    return st, st.buf.permute(0, 3, 1, 2)[:, :C]


def _aux_planes(kind, state_view, st, B, C, H, W, g):
    """Guarded operand planes in the format conv2d_cg.detect takes (see conv2d_cg._aux_args)."""
    from cbinfer_b200 import _lib
    if kind is None:
        return None, []
    if kind == "tf32":                                  # the remainder plane has the state's strides
        lo = Guarded(B, tuple(st.buf.shape[1:]), torch.float32, lambda n: torch.rand(n, generator=g), g)
        return ("tf32", lo.buf.as_strided(state_view.shape, state_view.stride())), [lo]
    p16 = _lib.C.cb_plane_pitch16(C)
    hi = Guarded(B, (H, W, p16), torch.bfloat16, lambda n: torch.rand(n, generator=g), g)
    lo = Guarded(B, (H, W, p16), torch.bfloat16, lambda n: torch.rand(n, generator=g), g)
    return ("bf16", hi.buf, lo.buf), [hi, lo]


def _old_entry_point(x, state, bits, thr, mode, aux, u8):
    """The pre-mask entry points cb_change_detect / cb_change_detect_u8, called directly."""
    from cbinfer_b200 import _lib
    from cbinfer_b200 import conv2d_cg as cg
    B, C, H, W = x.shape
    am, hi, lo = cg._aux_args(aux, state)
    s = torch.cuda.current_stream().cuda_stream
    if u8:
        rc = _lib.C.cb_change_detect_u8(s, x.data_ptr(), *x.stride(), state.data_ptr(), *state.stride(), am, hi, lo,
                                        bits.data_ptr(), B, C, H, W, 255.0, 0.0, float(thr), mode)
    else:
        rc = _lib.C.cb_change_detect(s, _lib.dtype_code(x), x.data_ptr(), *x.stride(), state.data_ptr(),
                                     *state.stride(), am, hi, lo, bits.data_ptr(), B, C, H, W, float(thr), mode)
    _lib.check(rc)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                   and not e.name.startswith(("Memcpy", "Memset")))


def _run_main(name, env=None):
    """Run `name()` of this module in a fresh interpreter and return its last stdout line as JSON.
    The checks that read the profiler run this way: once torch's profiler has been started in a
    process, CUDA-graph kernels that replay between two later profiling sessions can be reported in
    the next one, which would disturb the launch lists other test modules take in this process."""
    code = "import sys; sys.path.insert(0, %r); from tests.test_gpu_active_streams import %s; %s()" % (REPO, name, name)
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    return json.loads(p.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("mode", ["changed", "all"])
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_masked_kernel_against_the_unmasked_launch(variant, mode):
    """Active streams: bitmap words, state and operand planes bit-identical to the unmasked launch.
    Inactive streams: bitmap words 0, state and planes unchanged byte for byte, although their x
    slices would flag every pixel.  Guard regions around bitmap, state and planes stay untouched.
    A null mask is bit-identical to the entry point without one.  B = 1..9, five masks, with and
    without operand planes (fp32 states)."""
    from cbinfer_b200 import _lib
    from cbinfer_b200 import conv2d_cg as cg
    xdt, sdt, C, H, W, xl, sl, kname = VARIANTS[variant]
    umode = {"changed": _lib.UPDATE_CHANGED, "all": _lib.UPDATE_ALL}[mode]
    u8 = xdt == torch.uint8
    thr = 0.3
    auxes = [None, "tf32", "bf16"] if sdt == torch.float32 else [None]
    g = torch.Generator().manual_seed(2 * list(VARIANTS).index(variant) + (mode == "all"))
    Wd = (W + 31) // 32
    for B in range(1, 10):
        for aux_kind in auxes:
            for mname, m in _masks(B).items():
                x = _x(B, C, H, W, xdt, xl, m, g)
                st, state = _state(B, C, H, W, sdt, sl, g)
                aux, planes = _aux_planes(aux_kind, state, st, B, C, H, W, g)
                bits = Guarded(B, (H * Wd,), torch.int32,
                               lambda n: torch.randint(-2 ** 31, 2 ** 31 - 1, (n,), generator=g), g)
                owned = [st, bits] + planes
                orig = [o.flat.clone() for o in owned]

                def run(active):
                    for o, f in zip(owned, orig):
                        o.flat.copy_(f)
                    if active == "old":
                        _old_entry_point(x, state, bits.buf, thr, umode, aux, u8)
                    elif u8:
                        cg.detect_u8(x, state, bits.buf, thr, umode, 255.0, 0.0, aux=aux, active=active)
                    else:
                        cg.detect(x, state, bits.buf, thr, umode, aux=aux, active=active)
                    return [o.flat.clone() for o in owned]

                ref = run("old")
                assert all(torch.equal(a, b) for a, b in zip(run(None), ref)), (B, mname, aux_kind, "null mask")
                mask = torch.tensor(m, dtype=torch.uint8, device="cuda")
                got = run(mask)
                for o, r, f, gt in zip(owned, ref, orig, got):
                    exp = o.expected(r, f, m)
                    if o is bits:
                        for b in range(B):                         # inactive words are written as 0
                            if not m[b]:
                                lo = GUARD + b * o.slice_bytes
                                exp[lo:lo + o.slice_bytes] = 0
                    assert torch.equal(gt, exp), (B, mname, aux_kind, "bits" if o is bits else "state/planes")
                # the bool form of the mask is read the same way
                assert all(torch.equal(a, b) for a, b in zip(run(mask.bool()), got))


def kernels_main():
    """The kernel each variant of the kernel test reaches, as the profiler names it (B = 9, every
    other stream skipped)."""
    from cbinfer_b200 import conv2d_cg as cg
    g = torch.Generator().manual_seed(0)
    hits = {}
    for variant, (xdt, sdt, C, H, W, xl, sl, kname) in VARIANTS.items():
        B, m = 9, _masks(9)["alternate"]
        x = _x(B, C, H, W, xdt, xl, m, g)
        _, state = _state(B, C, H, W, sdt, sl, g)
        bits = torch.empty(B * H * ((W + 31) // 32), dtype=torch.int32, device="cuda")
        mask = torch.tensor(m, dtype=torch.uint8, device="cuda")
        if xdt == torch.uint8:
            names = _kernel_names(lambda: cg.detect_u8(x, state, bits, 0.3, 2, 255.0, 0.0, active=mask))
        else:
            names = _kernel_names(lambda: cg.detect(x, state, bits, 0.3, 2, active=mask))
        hits[variant] = [n for n in names if kname in n]
    print(json.dumps(hits))


def test_each_variant_reaches_its_kernel():
    hits = _run_main("kernels_main")
    assert all(len(v) == 1 for v in hits.values()), hits


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


def _pose(pose, frame):
    from cbinfer_b200 import models
    m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
    models.calibrateThresholds(pose, m, frame)
    m.parallelBranches = True
    return m


# which streams have a new frame at step t (t >= 1; step 0 feeds every stream)
SCHEDULE = [None, [0, 2, 3], [1, 2], [], [0, 1, 2, 3], [3], [0, 3], [1], [0, 1, 2], [2, 3], [0], [1, 2, 3]]


def _outs(o):
    return list(o) if isinstance(o, (tuple, list)) else [o]


def _run_equivalence(make, frames, B):
    """Masked run (garbage in the skipped streams' slices) against the re-feed run (skipped streams
    get their last frame again): outputs and state bit for bit, every stream, every step."""
    import cbinfer_b200 as cb
    A, R = make(), make()
    last = frames[0].clone()
    with torch.no_grad():
        for t, f in enumerate(frames[:len(SCHEDULE)]):
            act = list(range(B)) if t == 0 else SCHEDULE[t]
            keep = torch.zeros(B, dtype=torch.bool)
            keep[act] = True
            refeed = torch.where(keep.cuda().view(B, 1, 1, 1), f, last)
            masked = refeed.clone()
            masked[~keep.cuda()] = 1e6 if f.dtype == torch.float32 else 1e4     # never read
            if t > 0:
                cb.setActiveStreams(A, act)
            a, r = _outs(A(masked)), _outs(R(refeed))
            for x, y in zip(a, r):
                assert torch.equal(x, y), ("outputs", t, act)
            for sa, sr in zip(cb.getStateTensors(A), cb.getStateTensors(R)):
                assert torch.equal(sa, sr), ("state", t, act)
            last = refeed


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 12, 0.08, seed=3)]
    thr = models.calibrateThresholds(base, _scene(base), frames[0])
    return base, frames, thr


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("feedback", [True, False])
@pytest.mark.parametrize("candidate", [True, False])
def test_masked_scene_equals_refeeding_the_previous_frame(scene, dt, candidate, feedback):
    base, frames, thr = scene
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[dt]
    base = copy.deepcopy(base).to(dtype)
    fr = [f.to(dtype) for f in frames]
    _run_equivalence(lambda: _scene(base, candidate, feedback, thr), fr, 4)


def test_masked_pose_equals_refeeding_the_previous_frame():
    """PoseModel T=2: the stage-2 inputs come out of torch.cat, so the first layers of both stage-2
    branches are plain-input layers that honour the mask too."""
    from cbinfer_b200 import models, video
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    frames = [f.cuda().to(torch.bfloat16) for f in video.sequence(4, 96, 128, 12, 0.1, lo=-0.5, hi=0.5, seed=5)]
    _run_equivalence(lambda: _pose(pose, frames[0]), frames, 4)


def edge_main():
    """Run in a subprocess with CBINFER_STREAMK=0 CBINFER_KSPLIT=1: the first active step of a fresh
    stream is compared with a cleared model that sees different change counts in the other streams,
    so the summation order must not depend on them."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    B, H, W = 4, 96, 128
    base = models.sceneLabelingBaseline().cuda()
    X = [f.cuda() for f in video.sequence(B, H, W, 8, 0.05, seed=0)]
    thr = models.calibrateThresholds(base, _scene(base), X[0])
    A = _scene(base, thr=thr)
    with torch.no_grad():
        # stream 3 inactive from the very first frame (a tensor: the model has not run yet)
        cb.setActiveStreams(A, torch.tensor([1, 1, 1, 0], dtype=torch.bool, device="cuda"))
        for t in range(3):
            g = X[t].clone()
            g[3] = 7.0
            A(g)
            assert all(bool(torch.isinf(s[3]).all()) for s in cb.getStateTensors(A)), t
        # stream 1 reset, then skipped for two frames: +inf too
        cb.resetStreams(A, [1])
        cb.setActiveStreams(A, [0, 2])
        for t in range(3, 5):
            g = X[t].clone()
            g[[1, 3]] = 7.0
            A(g)
            assert all(bool(torch.isinf(s[[1, 3]]).all()) for s in cb.getStateTensors(A)), t
        # their first active step equals a freshly cleared model
        cb.setActiveStreams(A, range(B))
        a = A(X[5])
        c = _scene(base, thr=thr)(X[5])
        assert torch.equal(a[[1, 3]], c[[1, 3]])
    print(json.dumps({"ok": True}))


def test_fresh_and_reset_streams_keep_inf_until_their_first_active_step():
    env = dict(os.environ, CBINFER_STREAMK="0", CBINFER_KSPLIT="1")
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_active_streams import edge_main; edge_main()"
            % REPO)
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


def test_threshold_lowered_while_a_stream_is_skipped(scene):
    """The candidate layers ignore the mask: the full scan that follows a lowered threshold still tests
    every pixel of the skipped stream (a layer that skipped it would never test those pixels again),
    so the masked model equals the model fed the previous frame in that stream, whose full scans do
    find new changes in it."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    A, R = _scene(base, thr=thr), _scene(base, thr=thr)
    found = 0
    with torch.no_grad():
        for f in frames[:3]:
            assert torch.equal(A(f), R(f))
        prev = frames[2]
        for t in range(3, 8):
            if t == 4:
                for m in (A, R):
                    for c in _convs(m)[1:]:
                        c.threshold *= 0.25
            cb.setActiveStreams(A, [0, 1, 3] if t < 6 else range(4))
            refeed = frames[t].clone()
            if t < 6:
                refeed[2] = prev[2]
            masked = refeed.clone()
            if t < 6:
                masked[2] = 1e6
            assert torch.equal(A(masked), R(refeed)), t
            for sa, sr in zip(cb.getStateTensors(A), cb.getStateTensors(R)):
                assert torch.equal(sa, sr), t
            if t == 4:
                for c in _convs(R)[1:]:
                    try:
                        idx = c.lastChangeIndexes().long()
                    except cb._lib.CBinferError:          # a candidate superset (masked 1x1 layers)
                        continue
                    HW = c.prevOutput.shape[2] * c.prevOutput.shape[3]
                    found += int((idx // HW == 2).sum())
            prev = refeed
    assert found > 0            # the lowered threshold did catch pixels of the skipped stream


def test_graphs_follow_the_mask_written_between_replays(scene):
    """A graph captured with the mask set follows whatever is written into it before each replay,
    and a graph that holds setActiveStreams(net, tensor) + the forward follows the tensor; both equal
    the same schedule run eagerly."""
    import cbinfer_b200 as cb
    from cbinfer_b200.runtime import FrameGraph
    base, frames, thr = scene
    for captured_call in (False, True):
        g, e = _scene(base, thr=thr), _scene(base, thr=thr)
        with torch.no_grad():
            for f in frames[:2]:
                g(f), e(f)
            cb.setActiveStreams(g, range(4))
            static = frames[1].clone()
            src = torch.ones(4, dtype=torch.bool, device="cuda")
            if captured_call:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    cb.setActiveStreams(g, src)
                    g(static)
                torch.cuda.current_stream().wait_stream(side)
                e(frames[1])
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    cb.setActiveStreams(g, src)
                    out = g(static)
                replay = graph.replay
            else:
                fg = FrameGraph(g, static, warmup=True)
                e(frames[1])
                out, replay = fg.static_output, fg.graph.replay
            last = frames[1].clone()
            for t in range(2, 12):
                act = SCHEDULE[t]
                keep = torch.zeros(4, dtype=torch.bool, device="cuda")
                keep[act] = True
                refeed = torch.where(keep.view(4, 1, 1, 1), frames[t], last)
                static.copy_(refeed)
                static[~keep] = 5.0
                if captured_call:
                    src.copy_(keep)
                else:
                    cb.setActiveStreams(g, act)
                replay()
                assert torch.equal(out, e(refeed)), (captured_call, t)
                last = refeed


def launch_list_main():
    """bench.py's workload (8 x 640x480, candidate path): the kernels of a step without a mask and of
    one with half the streams skipped."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(8, 480, 640, 5, 0.05, seed=0)]
    m = _scene(base)
    models.calibrateThresholds(base, m, frames[0], factor=0.02)
    first = _convs(m)[0]
    with torch.no_grad():
        for f in frames[:3]:
            m(f)
        plain = _kernel_names(lambda: m(first.detectInput(frames[3])))
        cb.setActiveStreams(m, [0, 2, 5, 7])
        masked = _kernel_names(lambda: m(first.detectInput(frames[4])))
    print(json.dumps({"plain": plain, "masked": masked}))


def test_masked_step_launches_what_an_unmasked_one_does():
    """A step with half the streams skipped launches the same 8 kernels as a step without a mask."""
    res = _run_main("launch_list_main")
    assert res["plain"] == res["masked"], res
    assert sum(res["plain"].values()) == 8, res


def _pipeline_setup(base, frames, thr):
    """A uint8 FramePipeline with activeStreams=True and an eager twin that has run what the pipeline
    ran while capturing its graphs."""
    from cbinfer_b200.runtime import FramePipeline
    u8 = [f.mul(255).round().to(torch.uint8) for f in frames]
    p_model, e = _scene(base, thr=thr), _scene(base, thr=thr)
    for m in (p_model, e):
        _convs(m)[0].inputNorm = (255.0, 0.0)
    depth = 2
    pipe = FramePipeline(p_model, u8[0], depth=depth, activeStreams=True)
    with torch.no_grad():
        for _ in range(depth + 1):
            e(u8[0])
    return pipe, e, u8, [f.cpu().pin_memory() for f in u8]


def test_frame_pipeline_equals_eager_refeeding(scene):
    """uint8 ingest through FramePipeline(activeStreams=True) with partial uploads: results equal the
    eager model fed the skipped streams' previous frame again; a dense module in front of the first
    CB layer is refused."""
    from cbinfer_b200.runtime import FramePipeline
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    pipe, e, u8, host = _pipeline_setup(base, frames, thr)
    depth = pipe.depth
    with torch.no_grad():
        last = u8[0].clone()
        slots, ref = [], []
        for t in range(1, 12):
            act = SCHEDULE[t]
            keep = torch.zeros(4, dtype=torch.bool, device="cuda")
            keep[act] = True
            refeed = torch.where(keep.view(4, 1, 1, 1), u8[t], last)
            slots.append(pipe.submit(host[t], active=act))
            ref.append(e(refeed).cpu())
            last = refeed
            if len(slots) == depth:
                assert torch.equal(pipe.wait(slots[0]).clone(), ref[0]), t
                slots.pop(0), ref.pop(0)
        pipe.drain()
        for s, r in zip(slots, ref):
            assert torch.equal(pipe.wait(s), r)

    class Dense(nn.Module):
        def __init__(self, m):
            super().__init__()
            self.pre = nn.Identity()
            self.m = m

        def forward(self, x):
            return self.m(self.pre(x))

    with pytest.raises(CBinferError, match="Identity"):
        FramePipeline(Dense(_scene(base, thr=thr)), frames[0], depth=2, activeStreams=True)


def pipeline_h2d_main():
    """The host-to-device copies of one FramePipeline step per active set, from the profiler's trace:
    {active set: sorted byte counts}, plus the bytes of one stream's slice."""
    import tempfile
    from torch.profiler import ProfilerActivity, profile
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 3, 0.08, seed=3)]
    thr = models.calibrateThresholds(base, _scene(base), frames[0])
    pipe, _, u8, host = _pipeline_setup(base, frames, thr)
    out = {"slice_bytes": u8[0][0].numel()}
    with tempfile.TemporaryDirectory() as tmp:
        for act in ([0, 1, 3], [2], [], None):
            pipe.drain()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                pipe.wait(pipe.submit(host[1], active=act))
                pipe.drain()
            trace = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(trace)
            with open(trace) as f:
                events = json.load(f)["traceEvents"]
            out[str(act)] = sorted(int(ev.get("args", {}).get("bytes", 0)) for ev in events
                                   if ev.get("cat") == "gpu_memcpy" and "HtoD" in ev.get("name", ""))
    print(json.dumps(out))


def test_frame_pipeline_uploads_only_the_active_streams():
    """The H2D copies of a partial step carry the active slices only, one copy per contiguous run of
    active streams (the only other upload is the few-byte mask)."""
    res = _run_main("pipeline_h2d_main")
    slice_bytes = res["slice_bytes"]
    for act, runs in (([0, 1, 3], 2), ([2], 1), ([], 0), (None, 1)):
        sizes = res[str(act)]
        big = [s for s in sizes if s >= slice_bytes]
        n = 4 if act is None else len(act)
        assert len(big) == runs and sum(big) == n * slice_bytes, (act, sizes)
        assert len(sizes) - len(big) <= 1, (act, sizes)


def test_errors(scene):
    import cbinfer_b200 as cb
    from cbinfer_b200 import models
    from cbinfer_b200.runtime import FramePipeline
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    m, twin = _scene(base, thr=thr), _scene(base, thr=thr)
    with torch.no_grad():
        m(frames[0]), twin(frames[0])
        cb.setActiveStreams(m, torch.ones(5, dtype=torch.bool, device="cuda"))
        with pytest.raises(CBinferError, match="mask of 5 streams"):
            m(frames[1])
        cb.setActiveStreams(m, torch.ones(4, dtype=torch.uint8, device="cuda"))
        for bad in ([4], [-1]):
            with pytest.raises(CBinferError, match="out of range"):
                cb.setActiveStreams(m, bad)
        with pytest.raises(CBinferError, match="CUDA tensor"):
            cb.setActiveStreams(m, torch.ones(4, dtype=torch.bool))
        with pytest.raises(CBinferError):
            cb.setActiveStreams(m, torch.ones(4, dtype=torch.float32, device="cuda"))
        _convs(m)[0].gatherComputationStats = True
        with pytest.raises(CBinferError, match="gatherComputationStats"):
            m(frames[1])
        _convs(m)[0].gatherComputationStats = False
        cb.setActiveStreams(m, None)
        assert all(c._activeMask is None for c in _convs(m))
        assert torch.equal(m(frames[1]), twin(frames[1]))     # the refused calls changed nothing
        fg = models.sceneLabelingCBinfer(base, experimentIdx=7)
        with pytest.raises(CBinferError, match="fine-grained"):
            cb.setActiveStreams(fg, [0])
        pipe = FramePipeline(_scene(base, thr=thr), frames[0], depth=2)
        with pytest.raises(CBinferError, match="activeStreams=True"):
            pipe.submit(frames[1].cpu().pin_memory(), active=[0])
        pipe.drain()
