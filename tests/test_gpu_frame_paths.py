"""Which kernels each frame launches, pinned call by call.

bench.py reports its launch count from the module attributes that select the fused paths, not by
counting calls, and a model whose host logic quietly stops taking a fused path still computes the
same outputs.  These tests wrap the `conv2d_cg` ops the way bench.py's kernels_in_step does and
check the sequence (scene model) or the per-op counts (pose CPM) of every steady-state frame."""
import contextlib
import copy
from collections import Counter

import pytest
import torch

pytestmark = pytest.mark.gpu

# every op of the per-frame path that launches a kernel (bench.py, kernels_in_step)
OPS = ("detect", "detect_u8", "detect_sparse", "detect_sparse_compact", "dilate_compact", "dilate_tiles",
       "pool_compact", "conv_update", "conv_update_tiled", "tail_update", "maxPool2d", "maxPool2d_detect")

# DESIGN.md section 1: the scene model's frame on the candidate path
SCENE_FRAME = ["detect", "dilate_tiles", "conv_update_tiled", "dilate_tiles", "conv_update_tiled",
               "dilate_compact", "conv_update", "tail_update"]

# the frame after prevInput of the conv behind the second pool was rewritten from outside: that conv
# scans densely (maxPool2d + detect instead of the tile epilogue), so the conv before the pool keeps
# its ordered index list (dilate_compact instead of dilate_tiles)
REARM_FRAME = ["detect", "dilate_tiles", "conv_update_tiled", "dilate_compact", "conv_update_tiled",
               "maxPool2d", "pool_compact", "detect", "dilate_compact", "conv_update", "tail_update"]
# frames until SCENE_FRAME is back, the rewritten frame included (recorded at the commit that added
# this test)
REARM_FRAMES = 1

# Regression record, not a design statement: the per-op launch counts of one steady-state frame of
# the pose CPM (T=2, bf16, 368x368, batch 1, candidate path) as recorded at the commit that added
# this test.  A change of host logic that alters them has to say why.
POSE_FRAME = {"conv_update": 21, "conv_update_tiled": 15, "detect": 5, "detect_sparse": 18,
              "detect_sparse_compact": 10, "dilate_compact": 17, "dilate_tiles": 1, "maxPool2d_detect": 2}


@contextlib.contextmanager
def _calls():
    """Log the name of every op call in the block (bench.py, kernels_in_step)."""
    from cbinfer_b200 import conv2d_cg as cg
    log = []
    orig = {n: getattr(cg, n) for n in OPS}

    def wrap(name):
        fn = orig[name]

        def w(*a, **k):
            log.append(name)
            return fn(*a, **k)
        return w
    try:
        for n in OPS:
            setattr(cg, n, wrap(n))
        yield log
    finally:
        for n, f in orig.items():
            setattr(cg, n, f)


def _scene_frames(n):
    from cbinfer_b200 import video
    # bench.py's default workload: 8 streams of 480x640, 5% block change per frame
    return [f.cuda() for f in video.sequence(8, 480, 640, n, 0.05, "block", seed=0)]


def _scene_model(base, frame0=None):
    """bench.py's model (build_model) on the candidate path; thresholds calibrated on frame0."""
    from cbinfer_b200 import models
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                    clonePoolOutput=False, candidateDetect=True)
    if frame0 is not None:
        models.calibrateThresholds(base, m, frame0)
    return m


def _with_thresholds(m, thr):
    import cbinfer_b200 as cb
    for c, t in zip([c for c in m.modules() if type(c) is cb.CBConv2d], thr):
        c.threshold = t
    return m


def _convs(m):
    import cbinfer_b200 as cb
    return [c for c in m.modules() if type(c) is cb.CBConv2d]


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models
    return models.sceneLabelingBaseline().cuda(), _scene_frames(8)


@pytest.mark.parametrize("detect_input", [False, True])
def test_scene_candidate_frame_is_eight_launches(scene, detect_input):
    """After warm-up every frame of the benchmarked model is exactly the 8 launches of DESIGN.md
    section 1, run eagerly and through CBConv2d.detectInput + forward."""
    base, frames = scene
    m = _scene_model(base, frames[0])
    first = _convs(m)[0]
    with torch.no_grad():
        for t, f in enumerate(frames):
            with _calls() as log:
                m(first.detectInput(f)) if detect_input and t > 0 else m(f)
            if t >= 2:
                assert log == SCENE_FRAME, (t, log)


def test_rewritten_state_rearms_the_candidate_path(scene):
    """A prevInput rewritten from outside (same values, new tensor version) makes its layer scan
    densely on the next frame instead of trusting its candidates; the outputs stay those of an
    untouched twin, and the fused 8-launch frame comes back."""
    base, frames = scene
    a, b = _scene_model(base, frames[0]), _scene_model(base, frames[0])
    seqs = []
    with torch.no_grad():
        for f in frames[:3]:
            assert torch.equal(a(f), b(f))
        p = _convs(a)[2].prevInput                  # the conv after the second pool
        p.copy_(p.clone())
        for f in frames[3:]:
            with _calls() as log:
                out = a(f)
            seqs.append(log)
            assert torch.equal(out, b(f))
    assert seqs[0] == REARM_FRAME, seqs[0]
    back = next(i for i, s in enumerate(seqs) if s == SCENE_FRAME)
    assert back == REARM_FRAMES, seqs
    assert all(s == SCENE_FRAME for s in seqs[back:]), seqs


def test_pose_cpm_launch_counts_regression_record():
    """Per-op launch counts of the pose CPM's steady-state frames (POSE_FRAME, a recorded baseline)."""
    from cbinfer_b200 import models, video
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    frames = [f.cuda().to(torch.bfloat16) for f in video.sequence(1, 368, 368, 6, 0.05, lo=-0.5, hi=0.5)]
    m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
    models.calibrateThresholds(pose, m, frames[0])
    with torch.no_grad():
        for t, f in enumerate(frames):
            with _calls() as log:
                m(f)
            if t >= 2:
                assert dict(Counter(log)) == POSE_FRAME, (t, dict(Counter(log)))


def test_warm_cast_on_the_candidate_path_starts_over(scene):
    """model.half() / .float() on a warm model running the fused pool, tile epilogue and tail: from
    the cast on, the outputs are bit-identical to a fresh model of the new dtype fed the same frames,
    and every layer's state aliases its pixel-major storage again."""
    base, frames = scene
    m = _scene_model(base, frames[0])
    thr = [c.threshold for c in _convs(m)]
    convs = _convs(m)
    assert convs[0]._fusedPool and convs[1]._fusedPool and convs[3]._fusedTail
    with torch.no_grad():
        for f in frames[:3]:
            with _calls() as log:
                m(f)
        assert log == SCENE_FRAME, log             # all three fused paths ran
        for dt, fr in ((torch.float16, frames[3:6]), (torch.float32, frames[6:])):
            m.to(dt)
            # the weights the warm model has now: rounded to fp16 by the first cast
            ref = _with_thresholds(_scene_model(copy.deepcopy(base).half().to(dt)), thr)
            for f in fr:
                assert torch.equal(m(f.to(dt)), ref(f.to(dt)))
            for c in _convs(m):
                assert c.prevInput.data_ptr() == c._inBuf.data_ptr()
                assert c.prevOutput.data_ptr() == c._outBuf.data_ptr()

