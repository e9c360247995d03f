"""Watched-pixel zones (cbinfer_b200.setStreamZones, cb_change_detect_zone / cb_change_detect_u8_zone):
each zone launch against the launch without a zone on the substituted frame x' (x at watched pixels and at
pixels whose state holds +inf, the state elsewhere), at the narrow kernel's shape edges; the model-level rule
(a zone model equals a twin without a zone fed the substituted frames) on the scene and pose models; the
overlay use case; uint8 ingest, graphs, the pipeline and the refusals."""
import copy

import pytest
import torch

from tests.test_gpu_stream_reset import FUSED_FRAME, _calls
from tests.test_gpu_stream_thresholds import _convs, _scene

DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
BITS = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}

pytestmark = pytest.mark.gpu


def _bits(t):
    """bitwise view for comparisons (NaN-safe)"""
    return t.contiguous().view(BITS.get(t.dtype, t.dtype))


def _zone_bits(mask):
    from cbinfer_b200 import conv2d_cg as cg
    bits, _ = cg._map_to_bits(mask.to(torch.int8).cuda())
    return bits


def _pattern(kind, B, H, W, g):
    if kind == "all":
        return torch.ones(B, H, W, dtype=torch.bool)
    if kind == "none":
        return torch.zeros(B, H, W, dtype=torch.bool)
    if kind == "random":
        return torch.rand(B, H, W, generator=g) < 0.5
    if kind == "stripes":                       # 7-pixel stripes: edges at 28, 35, ... cross word boundaries
        return ((torch.arange(W) // 7) % 2 == 0).expand(B, H, W).clone()
    assert kind == "per_stream"
    kinds = ("all", "none", "random", "stripes")
    return torch.stack([_pattern(kinds[b % 4], 1, H, W, g)[0] for b in range(B)])


PATTERNS = ["all", "none", "random", "stripes", "per_stream"]
SHAPES = [(1, 1), (2, 31), (3, 32), (4, 33), (5, 160), (1, 160), (5, 1)]      # (B, W), H = 3


def _unaccepted(state):
    """[B, H, W]: +inf in one of the real channels of the state view [B, C, H, W]"""
    return torch.isinf(state.float()).logical_and(state.float() > 0).any(1)


def _case(dt, B, C, H, W, layout, aux, seed):
    """x in `layout` ('planar' NCHW or 'hwc' pixel-major of pitch C), a pixel-major state of pitch 16 bytes with
    guard elements around it (near x, some pixels +inf in one channel, some in all), optional operand planes"""
    from cbinfer_b200 import conv2d_cg as cg
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, C, H, W, generator=g)
    s = x + (torch.rand(B, C, H, W, generator=g) - 0.5) * 0.4
    s = torch.where(torch.rand(B, 1, H, W, generator=g) < 0.35, x, s)           # some pixels unchanged
    one = torch.rand(B, 1, H, W, generator=g) < 0.1
    ch = torch.randint(0, C, (B, 1, H, W), generator=g)
    s = torch.where(one & (torch.arange(C).view(1, C, 1, 1) == ch), torch.tensor(float("inf")), s)
    s = torch.where(torch.rand(B, 1, H, W, generator=g) < 0.05, torch.tensor(float("inf")), s)
    pitch = 16 // torch.empty(0, dtype=dt).element_size()
    G = 64
    flat = torch.full((B * H * W * pitch + 2 * G,), 7.25, dtype=dt, device="cuda")
    core = flat[G:G + B * H * W * pitch].view(B, H, W, pitch)
    core.zero_()
    state = core[..., :C].permute(0, 3, 1, 2)
    state.copy_(s.to(dt))
    if layout == "planar":
        xv = x.to(dt).cuda().contiguous()
    else:
        xv = torch.empty(B, H, W, C, dtype=dt, device="cuda").permute(0, 3, 1, 2)
        xv.copy_(x.to(dt))
    d = dict(x=xv, state=state, flat=flat)
    fin = torch.isfinite(state)
    if aux == "tf32":
        lo_flat = torch.full_like(flat, -3.5)
        lo_core = lo_flat[G:G + B * H * W * pitch].view(B, H, W, pitch)
        lo_core.zero_()
        lo = lo_core[..., :C].permute(0, 3, 1, 2)
        lo.copy_(torch.where(fin, cg.tf32_lo(torch.where(fin, state, 0)), 0))
        d.update(aux=("tf32", lo), planes=[lo_flat])
    elif aux == "bf16":
        planes = cg.bf16_planes(torch.nan_to_num(core, posinf=0.0, neginf=0.0), C)
        d.update(aux=("bf16",) + tuple(planes), planes=list(planes))
    d["bits"] = torch.full((B * H * ((W + 31) // 32),), -1, dtype=torch.int32, device="cuda")
    return d


def _normalise(u8, divisor, bias):
    """u8 / divisor + bias with IEEE division, as the kernel computes it (torch divides by a scalar through
    its reciprocal, which is not always correctly rounded; a tensor divisor is)"""
    x = u8.float()
    return x / torch.full_like(x, divisor) + bias


def _substituted(d, zone, u8=None):
    """x' of the rule: x (or the normalised uint8 frame) where watched or never accepted, else the state"""
    x = d["x"] if u8 is None else u8
    keep = (zone.cuda() | _unaccepted(d["state"])).unsqueeze(1)
    xs = torch.empty_like(d["x"]) if u8 is None else torch.empty(d["state"].shape, device="cuda").contiguous()
    xs.copy_(torch.where(keep, x.to(d["state"].dtype), d["state"]))
    return xs


def _compare(got, ref):
    assert torch.equal(got["bits"], ref["bits"]), "bits"
    assert torch.equal(_bits(got["flat"]), _bits(ref["flat"])), "state (with guards)"
    for a, b in zip(got.get("planes", []), ref.get("planes", [])):
        assert torch.equal(_bits(a), _bits(b)), "operand planes"


def _run_pair(dt, C, layout, update, aux, B, W, kind, seed, active=None, thr_b=None, H=3):
    from cbinfer_b200 import conv2d_cg as cg
    g = torch.Generator().manual_seed(seed + 1)
    zone = _pattern(kind, B, H, W, g)
    got = _case(dt, B, C, H, W, layout, aux, seed)
    ref = _case(dt, B, C, H, W, layout, aux, seed)
    xs = _substituted(ref, zone)
    cg.detect(got["x"], got["state"], got["bits"], 0.1, update, aux=got.get("aux"), active=active, thr_b=thr_b,
              zone=_zone_bits(zone))
    cg.detect(xs, ref["state"], ref["bits"], 0.1, update, aux=ref.get("aux"), active=active, thr_b=thr_b)
    _compare(got, ref)
    if kind == "all":                                    # all watched: the plain call on x itself
        plain = _case(dt, B, C, H, W, layout, aux, seed)
        cg.detect(plain["x"], plain["state"], plain["bits"], 0.1, update, aux=plain.get("aux"), active=active,
                  thr_b=thr_b)
        _compare(got, plain)


@pytest.mark.parametrize("dt,C", [("f32", 1), ("f32", 3), ("f32", 4), ("f16", 3), ("f16", 8), ("bf16", 3),
                                  ("bf16", 8)])
@pytest.mark.parametrize("layout", ["planar", "hwc"])
@pytest.mark.parametrize("update", [0, 1, 2])
def test_zone_detect_equals_substituted_frame(dt, C, layout, update):
    auxes = [None, "tf32", "bf16"] if dt == "f32" else [None]
    for aux in auxes:
        for k, (B, W) in enumerate(SHAPES):
            for kind in PATTERNS:
                _run_pair(DTYPES[dt], C, layout, update, aux, B, W, kind, seed=100 * k + len(kind) + C)


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("update", [0, 1, 2])
def test_zone_with_active_mask_and_thresholds(dt, update):
    B = 5
    active = torch.tensor([1, 0, 1, 1, 0], dtype=torch.uint8, device="cuda")
    thr_b = torch.tensor([0.05, 0.1, 0.2, 0.0, 0.15], dtype=torch.float32, device="cuda")
    for kind in ("random", "per_stream", "none"):
        for W in (33, 160):
            _run_pair(DTYPES[dt], 3, "planar", update, None, B, W, kind, seed=W, active=active, thr_b=thr_b)
            _run_pair(DTYPES[dt], 3, "hwc", update, None, B, W, kind, seed=W + 1, active=active)


@pytest.mark.parametrize("update", [0, 1, 2])
@pytest.mark.parametrize("layout", ["planar", "hwc"])
def test_zone_detect_u8_equals_normalised_substituted_frame(update, layout):
    """the uint8 zone launch against the fp32 launch without a zone on the normalised substituted frame"""
    from cbinfer_b200 import conv2d_cg as cg
    H = 3
    for k, (B, W) in enumerate(SHAPES):
        for kind in PATTERNS:
            for aux in (None, "bf16"):
                g = torch.Generator().manual_seed(k + 7)
                zone = _pattern(kind, B, H, W, g)
                got = _case(torch.float32, B, 3, H, W, layout, aux, seed=k)
                ref = _case(torch.float32, B, 3, H, W, layout, aux, seed=k)
                u8 = torch.randint(0, 256, (B, 3, H, W), generator=g, dtype=torch.uint8)
                x8 = torch.empty(B, 3, H, W, dtype=torch.uint8, device="cuda") if layout == "planar" else \
                    torch.empty(B, H, W, 3, dtype=torch.uint8, device="cuda").permute(0, 3, 1, 2)
                x8.copy_(u8)
                norm = _normalise(u8.cuda(), 255.0, -0.5)
                xs = _substituted(ref, zone, u8=norm)
                cg.detect_u8(x8, got["state"], got["bits"], 0.1, update, 255.0, -0.5, aux=got.get("aux"),
                             zone=_zone_bits(zone))
                cg.detect(xs, ref["state"], ref["bits"], 0.1, update, aux=ref.get("aux"))
                _compare(got, ref)


# ---- models --------------------------------------------------------------------------------------------

def _first(m):
    return _convs(m)[0]


def _substitute_frame(zone_model, frame, zone):
    """the frame the twin without a zone gets: x where watched or where the zone model's first-layer state
    is +inf (or not allocated yet), the state elsewhere"""
    st = _first(zone_model).prevInput
    if st.numel() == 0 or tuple(st.shape) != tuple(frame.shape):
        return frame.clone()
    keep = (zone.cuda() | _unaccepted(st)).unsqueeze(1)
    return torch.where(keep, frame, st.to(frame.dtype)).contiguous()


def _flat(o):
    return o if isinstance(o, torch.Tensor) else torch.cat([t.reshape(t.shape[0], -1) for t in o], 1)


def _assert_twins(a, r, out_a, out_r, where):
    import cbinfer_b200 as cb
    assert torch.equal(_bits(_flat(out_a)), _bits(_flat(out_r))), ("output", where)
    for sa, sr in zip(cb.getStateTensors(a), cb.getStateTensors(r)):
        assert torch.equal(_bits(sa), _bits(sr)), ("state", where)
    assert torch.equal(cb.streamChangeCounts(a), cb.streamChangeCounts(r)), ("counts", where)
    for la, lr in zip(_convs(a), _convs(r)):
        try:
            ia = la.lastChangeIndexes()
        except cb._lib.CBinferError:
            continue
        assert torch.equal(ia, lr.lastChangeIndexes()), ("list", where)


def _overlay(frames, y0=10, x0=20, h=12, w=40, seed=5):
    """a box redrawn with new content on every frame, in every stream"""
    g = torch.Generator().manual_seed(seed)
    out = []
    for f in frames:
        f = f.clone()
        f[:, :, y0:y0 + h, x0:x0 + w] = torch.rand(f.shape[0], f.shape[1], h, w, generator=g).to(f.dtype).to(f.device)
        out.append(f)
    return out


def _box(B, H, W, y0, x0, h, w, watched_streams=()):
    z = torch.ones(B, H, W, dtype=torch.bool)
    z[:, y0:y0 + h, x0:x0 + w] = False
    for b in watched_streams:
        z[b] = True
    return z


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 8, 0.05, seed=0)]
    thr = models.calibrateThresholds(base, _scene(base, [0.1] * 5), frames[0])
    return base, frames, thr


SCENE_CONFIGS = [dict(candidate=c, feedback=f) for c in (True, False) for f in (True, False)]


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("cfg", range(len(SCENE_CONFIGS)))
def test_scene_zone_model_equals_substituted_twin(scene, dt, cfg):
    """B = 4: stream 3 watches everything, the others exclude the overlay box; the zone is widened at frame 3
    and narrowed at frame 5, stream 1 is reset before frame 4.  The twin without a zone, fed the substituted
    frames, computes the same outputs, states, per-stream counts and change lists on every frame, with the
    same launch list."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    dtype = DTYPES[dt]
    base = copy.deepcopy(base).to(dtype)
    fr = _overlay([f.to(dtype) for f in frames])
    B, _, H, W = fr[0].shape
    a, r = _scene(base, thr, **SCENE_CONFIGS[cfg]), _scene(base, thr, **SCENE_CONFIGS[cfg])
    zones = {0: _box(B, H, W, 10, 20, 12, 40, watched_streams=(3,)),
             3: _box(B, H, W, 5, 10, 40, 70, watched_streams=(3,)),           # widened
             5: _box(B, H, W, 12, 24, 8, 30, watched_streams=(3,))}           # narrowed
    for m in (a, r):
        cb.trackStreamChanges(m, B=B)
    zone = None
    with torch.no_grad():
        for t, f in enumerate(fr):
            if t in zones:
                zone = zones[t]
                assert cb.setStreamZones(a, zone) == "0"
            if t == 4:
                cb.resetStreams(a, [1])
                cb.resetStreams(r, [1])
            fs = _substitute_frame(a, f, zone)
            with _calls() as la:
                oa = a(f)
            with _calls() as lr:
                orr = r(fs)
            assert la == lr, (t, la, lr)
            if t == 2 and cfg == 0 and dt == "f32":
                assert la == FUSED_FRAME, la
            _assert_twins(a, r, oa, orr, t)


def test_pose_zone_model_equals_substituted_twin():
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    B = 4
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    fr = _overlay([f.cuda().to(torch.bfloat16) for f in video.sequence(B, 96, 128, 6, 0.1, lo=-0.5, hi=0.5)])
    probe = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
    models.calibrateThresholds(pose, probe, fr[0])
    thr = [c.threshold for c in _convs(probe)]

    def mk():
        m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
        for c, t in zip(_convs(m), thr):
            c.threshold = t
        cb.trackStreamChanges(m, B=B)
        return m
    a, r = mk(), mk()
    _, _, H, W = fr[0].shape
    zone = _box(B, H, W, 10, 20, 12, 40, watched_streams=(2,))
    name = cb.setStreamZones(a, zone)
    assert name == "model0.0" == next(n for n, c in a.named_modules() if type(c) is cb.CBConv2d)
    with torch.no_grad():
        for t, f in enumerate(fr):
            fs = _substitute_frame(a, f, zone)
            _assert_twins(a, r, a(f), r(fs), t)


def test_overlay_stream_reports_no_change():
    """A stream whose only change is a redrawn overlay box: with the box excluded its last-layer count is 0 on
    every frame after the first and its output equals the previous frame's; without the zone it is not 0."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    still = video.sequence(2, 96, 128, 1, 0.0, seed=2)[0].cuda()
    fr = _overlay([still] * 6, seed=9)
    thr = models.calibrateThresholds(base, _scene(base, [0.1] * 5), fr[0])
    a, n = _scene(base, thr), _scene(base, thr)
    for m in (a, n):
        cb.trackStreamChanges(m, B=2)
    cb.setStreamZones(a, _box(2, 96, 128, 10, 20, 12, 40))
    prev = None
    with torch.no_grad():
        for t, f in enumerate(fr):
            oa = a(f).clone()
            n(f)
            if t > 0:
                assert int(cb.streamChangeCounts(a)[-1, 0]) == 0, t
                assert torch.equal(oa, prev), t
                assert int(cb.streamChangeCounts(n)[-1, 0]) > 0, t
            prev = oa


def test_u8_ingest_through_detect_input(scene):
    """uint8 frames with inputNorm through detectInput with a zone, against the twin fed the normalised
    substituted fp32 frames"""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    fr = _overlay(frames)
    u8 = [f.mul(255.0).round().clamp(0, 255).to(torch.uint8) for f in fr]
    B, _, H, W = fr[0].shape
    a, r = _scene(base, thr), _scene(base, thr)
    for m in (a, r):
        _first(m).inputNorm = (255.0, 0.0)
        cb.trackStreamChanges(m, B=B)
    zone = _box(B, H, W, 10, 20, 12, 40, watched_streams=(0,))
    cb.setStreamZones(a, zone)
    with torch.no_grad():
        for t, f in enumerate(u8):
            norm = _normalise(f, 255.0, 0.0)
            fs = _substitute_frame(a, norm, zone)
            oa = a(f) if t == 0 else a(_first(a).detectInput(f))
            _assert_twins(a, r, oa, r(fs), t)


def test_graph_replays_the_updated_zone(scene):
    """A FrameGraph captured before a zone update reads the zone buffer: after setStreamZones (host zone) and a
    captured CUDA-zone call, replays equal the eager substituted twin."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import runtime
    base, frames, thr = scene
    fr = _overlay(frames)
    B, _, H, W = fr[0].shape
    a, r = _scene(base, thr), _scene(base, thr)
    z0 = _box(B, H, W, 10, 20, 12, 40)
    cb.setStreamZones(a, z0)
    static = fr[0].clone()
    with torch.no_grad():
        a(static)
        r(_substitute_frame(a, static, z0))      # (the twin sees what a saw: frame 0 is all tested)
        fg = runtime.FrameGraph(a, static, warmup=True)
        r(_substitute_frame(a, static, z0))      # the capture's warm-up frame
        zones = [z0, _box(B, H, W, 5, 10, 40, 70), _box(B, H, W, 0, 0, 96, 64)]
        for t, f in enumerate(fr[1:]):
            z = zones[t % 3]
            cb.setStreamZones(a, z if t % 2 else z.cuda().to(torch.uint8))
            fs = _substitute_frame(a, f, z)
            static.copy_(f)
            out = fg.replay()
            assert torch.equal(out, r(fs)), t
            for sa, sr in zip(cb.getStateTensors(a), cb.getStateTensors(r)):
                assert torch.equal(sa, sr), t
    # a capturable call: a CUDA zone written inside the captured region
    src = torch.ones(B, H, W, dtype=torch.uint8, device="cuda")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cb.setStreamZones(a, src)
    src.copy_(_box(B, H, W, 30, 30, 20, 20).to(torch.uint8))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(_first(a)._zone[0], _zone_bits(_box(B, H, W, 30, 30, 20, 20)))


def test_pipeline_zone_updates_between_submits(scene):
    import cbinfer_b200 as cb
    from cbinfer_b200 import runtime
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    fr = _overlay(frames)
    B, _, H, W = fr[0].shape
    z0, z1 = _box(B, H, W, 10, 20, 12, 40), _box(B, H, W, 5, 10, 40, 70, watched_streams=(1,))
    m = _scene(base, thr)
    with pytest.raises(CBinferError, match="captured without a zone"):
        runtime.FramePipeline(m, fr[0], depth=2).setStreamZones(z0)
    m, ref = _scene(base, thr), _scene(base, thr)
    cb.setStreamZones(m, z0)
    cb.setStreamZones(ref, z0)
    host = [f.cpu().pin_memory() for f in fr]
    pipe = runtime.FramePipeline(m, fr[0], depth=2)
    with torch.no_grad():
        ref(fr[0])
        for i, f in enumerate(host[1:5]):
            if i == 2:
                pipe.setStreamZones(z1)
                cb.setStreamZones(ref, z1)
            s = pipe.submit(f)
            got = pipe.wait(s)
            assert torch.equal(got, ref(fr[1 + i]).cpu()), i
    with pytest.raises(CBinferError, match="cannot be detached"):
        pipe.setStreamZones(None)
    with pytest.raises(CBinferError, match="zone"):
        pipe.setStreamZones(torch.ones(B, H, W + 1, dtype=torch.bool))
    pipe.drain()


def test_refusals(scene):
    import torch.nn as nn
    import cbinfer_b200 as cb
    from cbinfer_b200 import conv2d_cg as cg
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    B, _, H, W = frames[0].shape
    a = _scene(base, thr)
    cb.setStreamZones(a, _box(B, H, W, 10, 20, 12, 40))
    bits = _first(a)._zone[0]
    cb.clearMemory(a)
    assert _first(a)._zone[0] is bits                       # the zone survives clearMemory
    with torch.no_grad():
        a(frames[0])
        for bad in (frames[1][:2], frames[1][:, :, :64], frames[1][:, :, :, :96]):
            with pytest.raises(CBinferError, match="zone"):
                a(bad)                                      # B, H or W differs from the zone's
        idx = cg.ChangeIndexes.from_tensor(torch.arange(10, dtype=torch.int32, device="cuda"), (B, H, W))
        with pytest.raises(CBinferError, match="change set"):
            _first(a)(('changeIndexes', frames[1], idx))   # the zone layer handed a change set
        _first(a).gatherComputationStats = True
        with pytest.raises(CBinferError, match="gatherComputationStats"):
            a(frames[1])
        _first(a).gatherComputationStats = False
        # a frame wider than one 16-byte state pixel (5 fp32 channels)
        wide = cb.convert(nn.Sequential(nn.Conv2d(5, 8, 3, padding=1)).cuda(), threshold=0.1)
        cb.setStreamZones(wide, torch.ones(2, 8, 8, dtype=torch.bool))
        with pytest.raises(CBinferError, match="16-byte"):
            wide(torch.rand(2, 5, 8, 8, device="cuda"))
        fg = cb.convert(nn.Sequential(nn.Conv2d(3, 8, 3, padding=1)).cuda(), threshold=0.1)
        cb.setStreamZones(fg, torch.ones(2, 8, 8, dtype=torch.bool, device="cuda"))
        fg[0].finegrained = True
        with pytest.raises(CBinferError, match="fine-grained"):
            fg(torch.rand(2, 3, 8, 8, device="cuda"))
        with pytest.raises(CBinferError, match="bool or uint8"):
            cb.setStreamZones(a, torch.ones(B, H, W, device="cuda"))
        # detaching: the model computes as without a zone again
        cb.setStreamZones(a, None)
        assert _first(a)._zone is None
        a(frames[1])
