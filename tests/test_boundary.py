"""CPU: the C-ABI library loads and exports every symbol include/cbinfer_b200.h declares, the
host-side size helpers agree with their definition, and the python surface mirrors the
reference's (no GPU compute calls here)."""
import os
import re

import pytest
import torch
import torch.nn as nn

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(REPO, "include", "cbinfer_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(cb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from cbinfer_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 18
    assert sorted(_lib.SYMBOLS) == syms
    for s in syms:
        assert hasattr(_lib.C, s), s
    assert _lib.C.cb_version() >= 100


def test_library_and_module_read_only_the_kept_environment_variables():
    """A setting measured worse is removed, not kept behind a variable (DESIGN.md §6 says why each
    of these stays)."""
    pkg = os.path.join(REPO, "cbinfer_b200")
    files = [os.path.join(pkg, f) for f in os.listdir(pkg) if f.endswith(".py")]
    files += [os.path.join(pkg, "csrc", f) for f in os.listdir(os.path.join(pkg, "csrc"))]
    names = set()
    for f in files:
        names |= set(re.findall(r"CBINFER_[A-Z0-9_]+", open(f).read()))
    assert names == {"CBINFER_" + n for n in ("LIB", "STREAMK", "KSPLIT", "TILES", "FUSE_POOL", "FUSE_TAIL")}


def test_size_helpers():
    from cbinfer_b200._lib import C
    assert C.cb_bitmap_row_words(640) == 20 and C.cb_bitmap_row_words(46) == 2
    assert C.cb_bitmap_words(2, 480, 640) == 2 * 480 * 20
    assert C.cb_channel_pitch(0, 3) == 4 and C.cb_channel_pitch(0, 185) == 188
    assert C.cb_channel_pitch(1, 3) == 8 and C.cb_channel_pitch(2, 185) == 192
    assert C.cb_compact_ws_bytes(1, 480, 640) >= 16 + 8 * ((9600 + 1023) // 1024)   # header + one status word per 1024-word tile
    # simt packing: fp32 [Kp][CoutP]
    assert C.cb_packed_weight_bytes(0, 0, 16, 3, 7, 7) == 49 * 4 * 16 * 4
    # tc3x packing: 2 planes x CoutPad(64) x KpPad(196->224) fp32
    assert C.cb_packed_weight_bytes(0, 2, 16, 3, 7, 7) == 2 * 16 * 224 * 4
    assert C.cb_packed_weight_bytes(2, 1, 256, 64, 7, 7) == 256 * 3136 * 2


def test_no_cpu_path():
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    m = cb.convert(nn.Sequential(nn.Conv2d(3, 4, 3, padding=1)))
    with pytest.raises(CBinferError):
        m(torch.zeros(1, 3, 8, 8))


def test_convert_surface_matches_reference_semantics():
    import cbinfer_b200 as cb
    import pycbinfer
    assert pycbinfer.CBConv2d is cb.CBConv2d
    base = nn.Sequential(
        nn.Conv2d(3, 8, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2), nn.Dropout(),
        nn.Sequential(nn.Conv2d(8, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 4, 1)),
        nn.Tanh())
    m = cb.convert(base, threshold=0.25)
    assert isinstance(m, nn.Sequential)
    names = [n for n, _ in m.named_children()]
    assert names == ["0", "2", "4", "5"]              # ReLU merged, Dropout removed, names kept
    c0 = m[0]
    assert type(c0) is cb.CBConv2d and c0.withReLU and c0.threshold == 0.25
    assert c0.weight is base[0].weight and c0.bias is base[0].bias     # parameters are shared
    inner = m[2]
    assert type(inner[0]) is cb.CBConv2d and inner[0].withReLU and not inner[1].withReLU
    assert inner[0].threshold == 0.25  # threshold is passed down the recursion (__init__.py:28)
    assert not c0.feedbackLoop and c0.copyInput and not c0.finegrained and not c0.propChangeIndexes
    assert "CBConv2d (th=0.25, 3->8, k=(7, 7), s=(1, 1), copyInput=True, pad=(3, 3), withReLU=True, propChgIdxs=False)" == repr(c0)
    assert cb.getStateTensors(m)[0].numel() == 0
    cb.clearMemory(m)
    m2 = cb.convertPools(m)
    assert type(m2[1]) is cb.CBPoolMax2d and m2[0].propChangeIndexes
    assert repr(m2[1]) == "CBPoolMax2d (k=(2, 2), s=(2, 2), ceil_mode=False, propChgIdxs=False)"
    # unsupported convs are rejected exactly like the reference (conv2d.py:91-93,104)
    for bad in (nn.Conv2d(3, 4, 3), nn.Conv2d(3, 4, 3, padding=1, stride=2),
                nn.Conv2d(4, 4, 3, padding=1, groups=2), nn.Conv2d(3, 4, 3, padding=1, bias=False)):
        with pytest.raises(AssertionError):
            cb.CBConv2d(bad, 0.1)


def test_models_build():
    from cbinfer_b200 import models
    import cbinfer_b200 as cb
    b = models.sceneLabelingBaseline()
    c = models.sceneLabelingCBinfer(b, experimentIdx=6)
    kinds = [type(m).__name__ for m in c.children()]
    assert kinds == ["CBConv2d", "CBPoolMax2d", "CBConv2d", "CBPoolMax2d", "CBConv2d", "CBConv2d", "CBConv2d"]
    assert all(m.feedbackLoop for m in c.modules() if type(m) is cb.CBConv2d)
    c2 = models.sceneLabelingCBinfer(b, experimentIdx=6, convertAll=False)
    assert [type(m).__name__ for m in c2.children()][-3:] == ["Conv2d", "ReLU", "Conv2d"]
    p = models.PoseModel(T=2)
    assert sum(1 for m in p.modules() if isinstance(m, nn.Conv2d)) == 36
    pc = models.poseModelCBinfer(p)
    assert sum(1 for m in pc.modules() if type(m) is cb.CBConv2d) == 36
    assert sum(1 for m in pc.modules() if type(m) is cb.CBPoolMax2d) == 3


def test_synthetic_video_change_rate():
    from cbinfer_b200 import video
    fr = video.sequence(2, 48, 64, 4, 0.05)
    for t in range(1, 4):
        rate = (fr[t] != fr[t - 1]).any(1).float().mean().item()
        assert abs(rate - 0.05) < 0.01
    fr = video.sequence(1, 48, 64, 3, 0.2, mode="iid")
    assert 0.1 < (fr[1] != fr[0]).any(1).float().mean().item() < 0.3


def test_hierarchical_tuner_and_pickle_roundtrip(tmp_path):
    """host logic of the reference's pose experiment 11 (poseDetection/modelConverter.py:107-168):
    trunk + first branch together, then per stage branch 1 / branch 2 with the stash-zero-restore
    dance; and the deployment flow clearMemory + torch.save / torch.load of a converted model."""
    import torch
    import cbinfer_b200 as cb
    from cbinfer_b200 import models
    pose = models.poseModelCBinfer(models.PoseModel(T=3), threshold=0.5)
    calls = []

    def fake_tune(mods, tols):
        assert len(mods) == len(tols)
        # everything outside the modules being tuned is either untuned (0) or already restored
        others = [m.threshold for m in models.getCBModuleList(pose) if m not in mods]
        calls.append((len(mods), tols[0], sorted(set(others))))
        for i, m in enumerate(mods):
            m.threshold = 0.01 * (len(calls) + i / 100.0)

    out = models.tuneHierarchical(pose, fake_tune)
    assert list(out) == ['model0', 'model1_1', 'model1_2', 'model2_1', 'model2_2', 'model3_1', 'model3_2']
    assert calls[0][1] == 5e-5 and all(c[1] == 2e-6 for c in calls[1:])
    assert calls[0][2] == [0]                                  # first call: everything else at 0
    # while model1_2 is tuned, model1_1 is zeroed: the only non-zero thresholds are model0's
    kids = dict(pose.named_children())
    n0 = len(models.getCBModuleList(kids['model0']))
    assert all(m.threshold > 0 for m in models.getCBModuleList(pose))
    assert len(calls) == 6 and calls[0][0] == n0 + len(models.getCBModuleList(kids['model1_1']))
    cb.clearMemory(pose)
    path = str(tmp_path / "pose.net")
    torch.save(pose, path)
    back = torch.load(path, weights_only=False)
    assert [m.threshold for m in models.getCBModuleList(back)] == \
        [m.threshold for m in models.getCBModuleList(pose)]
    assert repr(back) == repr(pose)


def test_pickle_of_an_older_version_gets_the_attributes_added_since(tmp_path):
    """a module pickled before a flag or a piece of private state existed loads with the flag's
    default, no fused neighbours and no version record (its state counts as written from outside)."""
    import cbinfer_b200 as cb
    conv = cb.CBConv2d(nn.Conv2d(3, 4, 3, padding=1), 0.1)
    pool = cb.CBPoolMax2d(nn.MaxPool2d(2, 2))
    for name in ('candidateDetect', 'tileMode', '_fusedPool', '_fusedTail', '_inVersion', '_outVersion'):
        del conv.__dict__[name]
    for name in ('_fusedNext', '_outVersion'):
        del pool.__dict__[name]
    path = str(tmp_path / "old.net")
    torch.save(nn.Sequential(conv, pool), path)
    conv, pool = torch.load(path, weights_only=False)
    assert conv.candidateDetect is False and conv.tileMode == 'auto'
    assert conv._fusedPool is None and conv._fusedTail is None and pool._fusedNext is None
    assert conv._inVersion is None and conv._outVersion is None and pool._outVersion is None


def test_bench_reference_arm_is_product_free():
    """bench.py's reference arm rebuilds the dense model and the synthetic video in plain torch
    (it must not load libcbinfer_sm100.so): both must equal the package's builders bit for bit, and
    running the arm must not import the product."""
    import subprocess
    import sys
    import torch
    import bench
    from cbinfer_b200 import models, video
    a, b = bench.dense_scene_cnn(), models.sceneLabelingBaseline()
    for pa, pb in zip(a.parameters(), b.parameters()):
        assert torch.equal(pa, pb)
    for mode in ("block", "iid"):
        fa = bench.synth_sequence(2, 24, 32, 4, 0.1, mode, seed=3)
        fb = video.sequence(2, 24, 32, 4, 0.1, mode, seed=3)
        assert all(torch.equal(x, y) for x, y in zip(fa, fb))
    code = ("import sys; sys.argv=['bench.py','--impl','reference','--steps','3','--warmup','1','--height','48',"
            "'--width','64','--streams','2']; import bench; bench.main(); "
            "assert 'cbinfer_b200' not in sys.modules; assert not any('libcbinfer' in l for l in open('/proc/self/maps'))")
    r = subprocess.run([sys.executable, "-c", code], cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["config"]["streams_per_gpu"] == 2 and line["gpu_launches"] == 0


def test_compat_shim_exports_the_reference_symbols():
    """the three libraries the unmodified reference dlopens (pycbinfer/conv2d_cg.py:44,50,
    conv2d_fg.py:31), built from csrc/compat_shim.cu: every symbol of the reference's cdef headers
    (conv2d_cg.py:6-38, conv2d_fg.py:13-24; conv2d_fg_cpu is the reference's CPU path: not built) resolves"""
    import ctypes
    from cbinfer_b200 import build
    libs = build.build_compat()
    cg = ["changeDetection", "changePropagation", "genXMatrix", "updateOutput", "maxPool2d"]
    for name, syms in (("cbconv2d_cg_backend", cg), ("cbconv2d_cg_half_backend", cg),
                       ("cbconv2d_fg_backend", ["changeDetectionFG", "updateOutputFG"])):
        lib = ctypes.CDLL(libs[name])
        for sname in syms:
            assert getattr(lib, sname) is not None


def test_resize_workspace_sizing_on_the_host():
    """host-side sizing of the resizer's workspace (no GPU compute)."""
    from cbinfer_b200 import _lib
    C = _lib.C
    # resize workspace: tables for both axes + the horizontally resized 8-bit intermediate
    ws = C.cb_resize_ws_bytes(720, 1280, 368, 654, 3)
    import math
    kx = math.ceil(2.0 * 1280 / 654) * 2 + 1                                   # Pillow: ceil(support * scale) * 2 + 1
    assert ws >= 32 + 8 * 654 + 4 * 654 * kx + 8 * 368 + 720 * 654 * 3 and ws % 16 == 0
    assert C.cb_resize_ws_bytes(0, 10, 10, 10, 3) == 0
