"""GPU parity tests, module level: CBConv2d / CBPoolMax2d / converted models against the oracle's
restatement of the reference flow (oracle.OracleCBConv2d / OracleCBPoolMax2d), against dense
nn.Conv2d at threshold 0, and against the UNMODIFIED reference kernels (oracle/_ref, JIT-compiled
from their compute_52/61 PTX) run on the same GPU where they are built.  The ops those tests run are
also checked, always, against their own recorded outputs (tests/golden/compat_ops_golden.npz)."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.util import ORC_DT, TORCH_DT, compare_outputs, perturb, rand_tensor, to_np, to_val, vp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _no_tf32():
    # the dense arbiter must be true fp32 (SURVEY section 8c)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


def _frames(shape, dt, n, frac, seed):
    f = [rand_tensor(shape, dt, seed)]
    for t in range(1, n):
        f.append(perturb(f[-1], frac, seed + t))
    return f


def _rel(got, exp):
    return float(np.abs(got - exp).max() / (np.abs(exp).max() + 1e-30))


# ---------------------------------------------------------------------------------------------
# CBConv2d vs the oracle flow, frame by frame
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dt,mode,tol", [("f32", "auto", 1e-4), ("f32", "tc3x", 1e-4), ("f32", "simt", 2e-5),
                                         ("bf16", "auto", 1e-2), ("f16", "auto", 2e-3)])
@pytest.mark.parametrize("feedback", [False, True])
@pytest.mark.parametrize("cfg", [(3, 16, 7, 20, 27), (16, 24, 3, 13, 18), (8, 8, 1, 9, 9)])
def test_cbconv_sequence_vs_oracle(orc, dt, mode, tol, feedback, cfg):
    import cbinfer_b200 as cb
    Cin, Cout, k, H, W = cfg
    torch.manual_seed(1)
    conv = nn.Conv2d(Cin, Cout, k, padding=k // 2).cuda().to(TORCH_DT[dt])
    m = cb.CBConv2d(conv, 0.3)
    m.withReLU = True
    m.feedbackLoop = feedback
    m.saveChangeMap = True
    m.gemmMode = mode
    o = orc.OracleCBConv2d(to_np(conv.weight), to_np(conv.bias), 0.3, dtype=ORC_DT[dt],
                           withReLU=True, feedbackLoop=feedback)
    frames = _frames((1, Cin, H, W), dt, 5, 0.06, seed=Cin)
    frames.insert(3, frames[2].clone())          # an unchanged frame: n == 0 must be a no-op
    for t, f in enumerate(frames):
        out = m(f)
        exp = o.forward(to_np(f))
        assert out is m.prevOutput                 # aliased, as in the reference (conv2d.py:259)
        assert np.array_equal(m.changeMap.cpu().numpy().astype(np.uint8), o.changeMap), t
        assert np.array_equal(to_np(m.prevInput), o.prevInput), t      # state is bit-exact
        assert _rel(to_val(out), orc.from_bits(exp, ORC_DT[dt])) <= tol, t
    assert int(m._scratch["count"].item()) > 0
    m(frames[-1])
    assert int(m._scratch["count"].item()) == 0


def test_threshold_zero_equals_dense_conv():
    """north star: with threshold 0, outputs must match dense nn.Conv2d."""
    import cbinfer_b200 as cb
    torch.manual_seed(2)
    conv = nn.Conv2d(16, 32, 7, padding=3).cuda()
    for fb in (False, True):
        m = cb.CBConv2d(conv, 0.0)
        m.feedbackLoop = fb
        for f in _frames((2, 16, 24, 31), "f32", 4, 0.1, seed=5):
            out = m(f)
            ref = F.conv2d(f, conv.weight, conv.bias, padding=3)
            assert _rel(to_val(out), to_val(ref)) <= 1e-4


def test_tuple_protocol_pool_and_graph(orc):
    """conv (propChangeIndexes) -> CBPoolMax2d -> conv, eager vs oracle chain, then the same
    frames replayed through a CUDA graph."""
    import cbinfer_b200 as cb
    torch.manual_seed(3)
    base = nn.Sequential(nn.Conv2d(3, 8, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(8, 12, 3, padding=1), nn.ReLU(), nn.Conv2d(12, 5, 1)).cuda().eval()
    m = cb.convertPools(cb.convert(base, threshold=0.05))
    for c in m.modules():
        if type(c) is cb.CBConv2d:
            c.feedbackLoop = True
    o1 = orc.OracleCBConv2d(to_np(base[0].weight), to_np(base[0].bias), 0.05, withReLU=True,
                            feedbackLoop=True, propChangeIndexes=True)
    op = orc.OracleCBPoolMax2d()
    o2 = orc.OracleCBConv2d(to_np(base[3].weight), to_np(base[3].bias), 0.05, withReLU=True,
                            feedbackLoop=True)
    o3 = orc.OracleCBConv2d(to_np(base[5].weight), to_np(base[5].bias), 0.05, feedbackLoop=True)
    frames = _frames((1, 3, 22, 30), "f32", 6, 0.05, seed=8)
    outs = []
    for f in frames:
        out = m(f)
        exp = o3.forward(o2.forward(op.forward(o1.forward(to_np(f)))))
        assert _rel(to_val(out), exp.astype(np.float64)) <= 2e-4
        outs.append(out.clone())
    r = m[0](frames[-1])
    assert type(r) is tuple and r[0] == 'changeIndexes' and isinstance(r[2], cb.ChangeIndexes)
    assert len(r[2]) == 0
    # CUDA graph: reset, warm up on frame 0, capture one step, replay the rest
    cb.clearMemory(m)
    static_in = frames[0].clone()
    m(static_in)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m(static_in)                                  # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        static_out = m(static_in)
    for t in range(1, len(frames)):
        static_in.copy_(frames[t])
        g.replay()
        assert _rel(to_val(static_out), to_val(outs[t])) <= 1e-6


def test_frame_pipeline_matches_eager():
    """runtime.FramePipeline (graphs + overlapped copies) returns what eager per-frame calls do."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, runtime, video
    base = models.sceneLabelingBaseline().cuda()
    host = [f.pin_memory() for f in video.sequence(2, 48, 64, 9, 0.06)]
    eager = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=True)
    ref = [eager(f.cuda()).clone() for f in host]
    piped = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=True,
                                        clonePoolOutput=False)
    pipe = runtime.FramePipeline(piped, host[0].cuda(), depth=2)
    # the pipeline's constructor already consumed frame 0 (state allocation + graph warm-up), so a
    # re-submission of frame 0 is an unchanged frame and the sequence continues from there
    got = []
    for f in host:
        s = pipe.submit(f)
        got.append(pipe.wait(s).clone())
    pipe.drain()
    for t in range(len(host)):
        assert _rel(to_val(got[t]), to_val(ref[t])) <= 1e-6, t


def test_user_supplied_index_tensor(orc):
    """reference-style callers hand in a plain int32 index tensor (conv2d.py:180-187)."""
    import cbinfer_b200 as cb
    x = rand_tensor((1, 6, 10, 12), "f32", 1)
    pool = cb.CBPoolMax2d(nn.MaxPool2d(2, 2))
    full = torch.arange(120, dtype=torch.int32, device="cuda")
    y = pool(('changeIndexes', x, full))
    assert torch.equal(y, F.max_pool2d(x, 2, 2))
    x2 = x.clone()
    x2[0, :, 4, 7] += 3.0
    y2 = pool(('changeIndexes', x2, torch.tensor([4 * 12 + 7], dtype=torch.int32, device="cuda")))
    assert torch.equal(y2, F.max_pool2d(x2, 2, 2))
    assert y2.data_ptr() != pool.outputState.data_ptr()       # clone, conv2d.py:73


@pytest.mark.parametrize("mode", ["auto", "simt"])
@pytest.mark.parametrize("shape", [(1, 4, 11, 13, 6, 3), (2, 16, 24, 40, 24, 7), (1, 5, 9, 70, 8, 5)])
def test_fine_grained_module(orc, mode, shape):
    """finegrained=True (conv2d.py:160-176): 'auto' = thresholded delta planes + accumulating tcgen05
    contraction, 'simt' = scattered red.global.add on planar tensors; both against the oracle's FG flow."""
    import cbinfer_b200 as cb
    B, Cin, H, W, Cout, k = shape
    torch.manual_seed(4)
    conv = nn.Conv2d(Cin, Cout, k, padding=k // 2).cuda()
    m = cb.CBConv2d(conv, 0.2)
    m.finegrained = True
    m.withReLU = True
    m.gemmMode = mode
    os_ = [orc.OracleCBConv2d(to_np(conv.weight), to_np(conv.bias), 0.2, withReLU=True, finegrained=True)
           for _ in range(B)]
    for f in _frames((B, Cin, H, W), "f32", 4, 0.1, seed=2):
        out = m(f)
        exp = np.concatenate([o.forward(to_np(f[b:b + 1])) for b, o in enumerate(os_)])
        np.testing.assert_allclose(out.cpu().numpy(), exp, rtol=1e-4, atol=1e-4)
        assert torch.equal(m.prevInput, f)                      # conv2d.py:175
    assert len(m.getStateTensors()) == 2 and tuple(m.getStateTensors()[1].shape) == (B, Cout, H, W)


def test_scene_model_small_vs_dense_and_oracle(orc):
    """the whole scene-labeling CBinfer model (all convs + pools converted, feedback loop):
    threshold 0 == dense model; threshold > 0 == oracle chain."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(1, 48, 64, 4, 0.05)]
    m0 = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.0)
    for f in frames:
        out = m0(f)
        with torch.no_grad():
            ref = base(f)
        assert _rel(to_val(out), to_val(ref)) <= 2e-4
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.05)
    cbs = [mm for mm in m.children()]
    chain = []
    for mm in cbs:
        if type(mm) is cb.CBConv2d:
            chain.append(orc.OracleCBConv2d(to_np(mm.weight), to_np(mm.bias), 0.05,
                                            withReLU=mm.withReLU, feedbackLoop=True,
                                            propChangeIndexes=mm.propChangeIndexes))
        else:
            chain.append(orc.OracleCBPoolMax2d())
    for f in frames:
        out = m(f)
        e = to_np(f)
        for o in chain:
            e = o.forward(e)
        assert _rel(to_val(out), e.astype(np.float64)) <= 5e-4


@pytest.mark.parametrize("save_maps", [True, False])
@pytest.mark.parametrize("feedback", [True, False])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_candidate_detection_equals_dense_scan(feedback, dt, save_maps):
    """B200 extension: thresholding only the pixels the upstream CB layer rewrote gives exactly
    the change maps, index lists, states and outputs of the reference's full re-scan."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda().to(TORCH_DT[dt])
    frames = [f.cuda().to(TORCH_DT[dt]) for f in video.sequence(2, 50, 78, 7, 0.08)]
    frames.insert(4, frames[3].clone())
    ms = []
    for cand in (False, True):
        m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.03, candidateDetect=cand)
        for c in m.modules():
            if type(c) is cb.CBConv2d:
                c.feedbackLoop = feedback
                # 1x1 layers: masked contraction without any compaction and, in fp32, the fused tail
                # (no maps), plain candidate path (maps saved)
                c.saveChangeMap = save_maps
        ms.append(m)
    for t, f in enumerate(frames):
        outs = [m(f) for m in ms]
        if t == 5:      # raising a threshold keeps the candidate path exact, lowering falls back
            for m in ms:
                kids = dict(m.named_children())
                kids['3'].threshold *= 2.0
                kids['6'].threshold *= 0.5
        assert torch.equal(outs[0], outs[1]), t
        for a, b in zip(ms[0].children(), ms[1].children()):
            if type(a) is cb.CBConv2d:
                if save_maps:
                    assert torch.equal(a.changeMap, b.changeMap), t
                assert torch.equal(a.prevInput, b.prevInput), t
                na, nb = int(a._scratch["count"].item()), int(b._scratch["count"].item())
                assert na == nb, t
                if not (b.maskedConv and not save_maps and t > 0):
                    # (a masked 1x1 layer never materialises its own list: its count is compared and,
                    #  with feedback, its state, which is rewritten at exactly the changed pixels)
                    assert torch.equal(a.lastChangeIndexes(), b.lastChangeIndexes()), t
            else:
                assert torch.equal(a.outputState, b.outputState), t


@pytest.mark.parametrize("dt", ["f32", "f16"])
@pytest.mark.parametrize("case", [(2, 40, 13, 37, 3), (1, 128, 46, 46, 7), (8, 16, 46, 46, 7), (1, 8, 368, 368, 3),
                                  (3, 5, 9, 70, 1), (1, 4, 1, 1, 3)])
def test_fused_small_map_detect_compact_equals_two_launches(dt, case):
    """cb_change_detect_sparse_compact (the last block of the candidate detection dilates and compacts a
    small bitmap) == cb_change_detect_sparse + cb_dilate_compact: raw / dilated bitmaps, ascending index
    list, count, feedback state; with and without clearing the raw bitmap; repeated calls (self-cleaning)."""
    from cbinfer_b200 import _lib, conv2d_cg as cg
    B, C, H, W, k = case
    shape = (B, C, H, W)
    prev = rand_tensor(shape, dt, 1)
    x = perturb(prev, 0.1, 2)
    g = torch.Generator().manual_seed(4)
    cmask = (torch.rand(B, H, W, generator=g) < 0.4).to(torch.int8).cuda()      # candidates: a subset of the pixels
    for update in (_lib.UPDATE_CHANGED, _lib.UPDATE_ALL, _lib.UPDATE_NONE):
        for clear in (False, True):
            res = []
            for fused in (False, True):
                st, _ = cg.pixel_major(shape, TORCH_DT[dt], "cuda", 0)
                st.copy_(prev)
                xv, _ = cg.pixel_major(shape, TORCH_DT[dt], "cuda", 0)
                xv.copy_(x)
                s = cg.alloc_scratch((B, H, W), "cuda")
                cand = cg.changeIndexesExtr(cmask, lazy=True)
                sync = torch.zeros(1, dtype=torch.int32, device="cuda")
                for rep in range(2):
                    if rep == 1 and update != _lib.UPDATE_NONE:
                        break                                   # (the state moved: a second pass differs by design)
                    if fused:
                        cg.detect_sparse_compact(xv, st, s["raw_bits"], 0.3, update, cand, (k, k), s["idx"], s["count"],
                                                 sync, bits_are_clear=(rep == 0 or clear), dil_bits=s["dil_bits"],
                                                 clear_raw=clear)
                    else:
                        cg.detect_sparse(xv, st, s["raw_bits"], 0.3, update, cand, bits_are_clear=(rep == 0 or clear))
                        cg.dilate_compact(s["raw_bits"], (B, H, W), (k, k), s["idx"], s["count"], s["ws"],
                                          dil_bits=s["dil_bits"], clear_raw=clear)
                n = int(s["count"].item())
                res.append((n, s["idx"][:n].clone(), s["dil_bits"].clone(), s["raw_bits"].clone(), st.clone()))
                assert int(sync.item()) == 0
            assert res[0][0] == res[1][0], (update, clear)
            for a, b in zip(res[0][1:], res[1][1:]):
                assert torch.equal(a, b), (update, clear)
            assert res[0][0] > 0 or H * W == 1
            if clear:
                assert int(res[1][3].abs().sum()) == 0


def test_pool_compact_and_sparse_detect_ops():
    from cbinfer_b200 import _lib, conv2d_cg as cg
    g = torch.Generator().manual_seed(3)
    for (B, H, W, ceil) in ((2, 9, 70, True), (1, 8, 64, False), (3, 5, 33, False), (1, 1, 1, True)):
        oH, oW = ((H - 1) // 2 + 1, (W - 1) // 2 + 1) if ceil else (H // 2, W // 2)
        m = (torch.rand(B, H, W, generator=g) < 0.15).to(torch.int8).cuda()
        bits, _ = cg._map_to_bits(m)
        s = cg.alloc_scratch((B, max(oH, 1), max(oW, 1)), "cuda")
        cg.pool_compact(bits, (B, H, W), (B, oH, oW), s["idx"], s["count"], s["ws"], out_bits=s["dil_bits"])
        pm = torch.nn.functional.max_pool2d(m.float().unsqueeze(1), 2, 2, ceil_mode=ceil).squeeze(1)
        ref = torch.nonzero(pm.reshape(-1)).view(-1).int()
        n = int(s["count"].item())
        assert n == ref.numel() and torch.equal(s["idx"][:n], ref)
    # sparse detect == dense detect when the candidates cover every difference
    for dt in ("f32", "f16"):
        shape = (2, 40, 13, 37)
        prev = rand_tensor(shape, dt, 1)
        x = perturb(prev, 0.1, 2)
        diff = (x != prev).any(1)
        extra = torch.rand(diff.shape, generator=g).cuda() < 0.05
        cand = cg.changeIndexesExtr((diff | extra).to(torch.int8), lazy=True)
        for layout in ("planar", "pixel"):
            for mode in (_lib.UPDATE_CHANGED, _lib.UPDATE_ALL, _lib.UPDATE_NONE):
                res = []
                for sparse in (False, True):
                    if layout == "pixel":
                        st = cg.pixel_major(shape, TORCH_DT[dt], "cuda", 0)[0].copy_(prev)
                        xin = cg.pixel_major(shape, TORCH_DT[dt], "cuda", 0)[0].copy_(x)
                    else:
                        st, xin = prev.clone(), x
                    sc = cg.alloc_scratch((2, 13, 37), "cuda")
                    if sparse:
                        cg.detect_sparse(xin, st, sc["raw_bits"], 0.4, mode, cand)
                    else:
                        cg.detect(xin, st, sc["raw_bits"], 0.4, mode)
                    res.append((sc["raw_bits"].clone(), st.contiguous().clone()))
                assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


@pytest.mark.parametrize("res", [(480, 640)])
def test_full_size_properties(res):
    """BASELINE config 2 size (640x480): size-independent properties instead of the slow oracle:
    threshold 0 == dense; an unchanged frame yields zero changes everywhere and leaves the output
    bit-identical; index lists are sorted, unique and match the bitmap popcount."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    H, W = res
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(1, H, W, 3, 0.05)]
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.0)
    for f in frames:
        out = m(f)
    with torch.no_grad():
        ref = base(frames[-1])
    assert _rel(to_val(out), to_val(ref)) <= 2e-4
    convs = [mm for mm in m.modules() if type(mm) is cb.CBConv2d]
    n1 = int(convs[0]._scratch["count"].item())
    assert 0.05 * H * W <= n1 <= 0.08 * H * W          # 5 % block + 3-pixel dilation ring
    idx = convs[0].lastChangeIndexes()
    assert bool((idx[1:] > idx[:-1]).all())
    bits = convs[0]._scratch["dil_bits"].cpu().numpy().view(np.uint32)
    assert int(np.unpackbits(bits.view(np.uint8)).sum()) == n1
    before = out.clone()
    out2 = m(frames[-1])
    assert all(int(c._scratch["count"].item()) == 0 for c in convs)
    assert torch.equal(out2, before)


# ---------------------------------------------------------------------------------------------
# the UNMODIFIED reference kernels on the same GPU (oracle/_ref, PTX JIT) where they are built; the
# ops' own recorded outputs always
# ---------------------------------------------------------------------------------------------

CD_CASES = ((16, 400, 300, 3, 0.1), (3, 97, 131, 7, 0.3), (64, 30, 40, 1, 0.5))


def _cd_inputs(C, H, W, dt):
    prev = rand_tensor((1, C, H, W), dt, C)
    return prev, perturb(prev, 0.05, C + 1, scale=0.7)


def reference_change_detection_outputs(lib, half):
    outs = {}
    for (C, H, W, k, thr) in CD_CASES:
        prev, x = _cd_inputs(C, H, W, "f16" if half else "f32")
        for update in (False, True):
            st_ref = prev.clone()
            cmap_ref = torch.zeros(H, W, dtype=torch.int8, device="cuda")
            grid = (H * W - 1) // 128 + 1
            lib.changeDetection(1, 1, grid, 1, 1, 128, vp(x), vp(st_ref), vp(cmap_ref), W, H, C,
                                (k - 1) // 2, (k - 1) // 2, ctypes.c_float(thr), ctypes.c_bool(update))
            torch.cuda.synchronize()
            outs["map_%d_%d" % (C, update)] = cmap_ref
            outs["state_%d_%d" % (C, update)] = st_ref
    return outs


def ops_change_detection_outputs(half):
    from cbinfer_b200 import conv2d_cg as cg
    outs = {}
    for (C, H, W, k, thr) in CD_CASES:
        prev, x = _cd_inputs(C, H, W, "f16" if half else "f32")
        for update in (False, True):
            st = prev.clone()
            cmap = cg.changeDetection(x, st, (k, k), thr, updateInputState=update)
            idx = cg.changeIndexesExtr(cmap)
            assert torch.equal(idx, torch.nonzero(cmap.view(-1)).int().view(-1))
            outs["map_%d_%d" % (C, update)] = cmap
            outs["state_%d_%d" % (C, update)] = st
    return outs


@pytest.mark.parametrize("half", [False, True])
def test_reference_cuda_kernels_change_detection(half):
    """bit-exact masks + feedback state vs cbconv2d_cg[_half]_backend.cu."""
    compare_outputs("ops_change_detection.%s" % ("f16" if half else "f32"),
             "cbconv2d_cg_half_backend" if half else "cbconv2d_cg_backend",
             ops_change_detection_outputs(half), lambda L: reference_change_detection_outputs(L, half))


def _gsp_inputs():
    C, H, W, k, Cout = 8, 37, 53, 7, 12
    x = rand_tensor((1, C, H, W), "f32", 1)
    g = torch.Generator().manual_seed(2)
    idx = torch.nonzero(torch.rand(H * W, generator=g) < 0.2).view(-1).int().cuda()
    Yt = rand_tensor((Cout, idx.numel()), "f32", 3)
    po = rand_tensor((1, Cout, H, W), "f32", 4)
    # maxPool2d (even sizes: the reference kernel has no bounds guard for odd ones)
    xe = rand_tensor((1, C, 36, 52), "f32", 5)
    idx2 = torch.nonzero(torch.rand(36 * 52, generator=g) < 0.2).view(-1).int().cuda()
    st = torch.full((1, C, 18, 26), float("inf"), device="cuda")
    return (C, H, W, k, Cout), x, idx, Yt, po, xe, idx2, st


def reference_gather_scatter_pool_outputs(lib):
    (C, H, W, k, Cout), x, idx, Yt, po_ref, xe, idx2, st_ref = _gsp_inputs()
    n = idx.numel()
    X_ref = torch.zeros(n, C * k * k, device="cuda")
    tz = 128 // (k * k)
    lib.genXMatrix(1, 1, (n - 1) // tz + 1, k, tz, k, vp(X_ref), vp(x), vp(idx), k, k, C, W, H, n)
    lib.updateOutput(1, 1, (n * Cout - 1) // 1024 + 1, 1, 1, 1024, vp(Yt), vp(po_ref), vp(idx),
                     H * W, n, Cout, ctypes.c_bool(True))
    lib.maxPool2d((idx2.numel() - 1) // 64 + 1, 64, vp(xe), vp(st_ref), vp(idx2), idx2.numel(), C,
                  36, 52, 18, 26, 2, 2)
    torch.cuda.synchronize()
    return {"xmatrix": X_ref, "output": po_ref, "pooled": st_ref}


def ops_gather_scatter_pool_outputs():
    from cbinfer_b200 import conv2d_cg as cg
    (C, H, W, k, Cout), x, idx, Yt, po, xe, idx2, st = _gsp_inputs()
    X = cg.genXMatrix(x, idx, (k, k))
    cg.updateOutput(Yt, idx, po, withReLU=True)
    cg.maxPool2d(xe, st, idx2)
    torch.cuda.synchronize()
    return {"xmatrix": X, "output": po, "pooled": st}


def test_reference_cuda_kernels_gather_scatter_pool():
    compare_outputs("ops_gather_scatter_pool", "cbconv2d_cg_backend", ops_gather_scatter_pool_outputs(),
             reference_gather_scatter_pool_outputs)


def _fg_inputs():
    Cin, Cout, H, W, k = 5, 7, 21, 26, 3
    prev = rand_tensor((1, Cin, H, W), "f32", 1)
    x = perturb(prev, 0.1, 2)
    w = rand_tensor((Cout, Cin, k, k), "f32", 3, scale=0.3)
    out = rand_tensor((1, Cout, H, W), "f32", 4)
    return (Cin, Cout, H, W, k), prev, x, w, out


def reference_fg_outputs(lib):
    (Cin, Cout, H, W, k), prev, x, w, out_ref = _fg_inputs()
    diffs = torch.zeros_like(x)
    cmap = torch.zeros(x.shape, dtype=torch.int8, device="cuda")
    lib.changeDetectionFG(vp(x), vp(prev), vp(diffs), vp(cmap), x.numel(), ctypes.c_float(0.2))
    coords = torch.nonzero(cmap.view(-1)).view(-1).contiguous()
    nchg = coords.numel()
    lib.updateOutputFG(1, 1, (nchg - 1) // 128 + 1, 1, 1, 128, vp(diffs), vp(w), vp(out_ref),
                       vp(coords), Cout, Cin, H, W, k, k, nchg)
    torch.cuda.synchronize()
    return {"changed": torch.tensor([nchg], dtype=torch.int32), "output": out_ref}


def ops_fg_outputs():
    from cbinfer_b200 import conv2d_fg as fg
    _, prev, x, w, out = _fg_inputs()
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    fg.cbconvFG(x, prev.clone(), out, w, 0.2, cnt)
    torch.cuda.synchronize()
    return {"changed": cnt, "output": out}


def test_reference_cuda_fg_kernels():
    compare_outputs("ops_fg", "cbconv2d_fg_backend", ops_fg_outputs(), reference_fg_outputs, tol={"output": (1e-5, 1e-4)})


def test_eval_tools_and_threshold_tuner(tmp_path):
    """reference harness surface: inferFrameset / inferFramesetBenchmark (evalTools.py:7-49) and the
    greedy threshold search (pycbinfer/__init__.py:98-144) run end to end on the CUDA backend."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import evalTools, models, video
    base = models.sceneLabelingBaseline().cuda()
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.0)
    frames = video.sequence(1, 48, 64, 5, 0.1)
    out = evalTools.inferFrameset(m, frames)
    with torch.no_grad():
        ref = base(frames[-1].cuda())
    assert _rel(to_val(out), to_val(ref)) <= 2e-4
    wall, dev = evalTools.inferFramesetBenchmark(m, frames)
    assert wall > 0 and dev > 0 and len(evalTools.changeStatistics(m)) == 5
    assert os.path.exists(evalTools.writeTable("t", [[1, 2]], header=["a", "b"], directory=str(tmp_path)))

    class Reader(object):
        def getDataFrames(self, seqName, numFrames):
            return frames[:numFrames + 1], None

    mods = evalTools.getCBconvLayers(m)
    cb.tuneThresholdParameters(Reader(), ["s0"], 3, lambda f: base(f.cuda()), lambda f: f, base, m,
                               lambda o, t: float((o - t).abs().mean()), mods[:2], 1e-3,
                               initThreshold=1e-3, thresholdIncrFactor=2.0)
    assert all(c.threshold >= 1e-3 for c in mods[:2])


@pytest.mark.parametrize("layout", ["hwc", "planar"])
@pytest.mark.parametrize("norm", [(255.0, 0.0), (256.0, -0.5)])
def test_uint8_ingest_bit_identical_to_normalised_fp32(layout, norm):
    """uint8 frames normalised inside the detection kernel (the readers' /255 resp. /256 - 0.5,
    sceneLabeling/videoSequenceReader.py:65, openPose/PoseDetector.py:72) give bit-identical change
    maps, states and outputs to feeding the host-normalised fp32 frame."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models
    base = models.sceneLabelingBaseline().cuda()
    g = torch.Generator().manual_seed(3)
    B, H, W = 2, 40, 70
    f8 = [torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8)]
    for t in range(4):
        nxt = f8[-1].clone()
        y0, x0 = 5 + 3 * t, 11 + 7 * t
        nxt[:, y0:y0 + 9, x0:x0 + 13] = torch.randint(0, 256, (B, 9, 13, 3), generator=g, dtype=torch.uint8)
        nxt[0, 0, 0, 1] = (int(nxt[0, 0, 0, 1]) + 1) % 256      # a one-level change, below threshold
        f8.append(nxt)
    ms = [models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=True)
          for _ in range(2)]
    first = [c for c in ms[1].modules() if type(c) is cb.CBConv2d][0]
    first.inputNorm = norm
    for c in ms[0].modules():
        if type(c) is cb.CBConv2d:
            c.saveChangeMap = True
    for c in ms[1].modules():
        if type(c) is cb.CBConv2d:
            c.saveChangeMap = True
    for t, f in enumerate(f8):
        nchw = f.permute(0, 3, 1, 2)                       # HWC memory seen as NCHW (strided view)
        if layout == "planar":
            nchw = nchw.contiguous()
        ref = ms[0](nchw.float().div(norm[0]).add(norm[1]).cuda())
        got = ms[1](nchw.cuda() if layout == "planar" else f.cuda().permute(0, 3, 1, 2))
        assert torch.equal(ref, got), t
        a = [c for c in ms[0].modules() if type(c) is cb.CBConv2d][0]
        assert torch.equal(a.prevInput, first.prevInput) and torch.equal(a.changeMap, first.changeMap), t
    m3 = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02)
    with pytest.raises(cb._lib.CBinferError):
        m3(f8[0].permute(0, 3, 1, 2).cuda())               # no inputNorm: refuse uint8


def test_save_load_converted_model_roundtrip(tmp_path):
    """the reference's deployment flow: clearMemory(model); torch.save(model, path); torch.load
    (pycbinfer/__init__.py:144, sceneLabeling/modelLoader.py:28-33)."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.03, candidateDetect=True)
    frames = [f.cuda() for f in video.sequence(1, 48, 64, 4, 0.1)]
    outs = [m(f).clone() for f in frames]
    cb.clearMemory(m)
    assert all(t.numel() == 0 for t in cb.getStateTensors(m))
    path = str(tmp_path / "model.net")
    torch.save(m, path)
    m2 = torch.load(path, weights_only=False)
    assert repr(m2) == repr(m)
    for f, o in zip(frames, outs):
        assert torch.equal(m2(f), o)


@pytest.mark.parametrize("cand", [True, False])
def test_state_snapshot_restore_like_eval03(cand):
    """the reference's per-frame timing restores getStateTensors() snapshots with copy_
    (poseDetection/eval03.py:87-95): hidden operand planes and the candidate-detection shortcuts must
    not go stale when the state is written from outside the kernels."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import evalTools, models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(2, 48, 72, 6, 0.1)]
    ms = [models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=cand)
          for _ in range(2)]
    for f in frames[:3]:
        for m in ms:
            m(f)
    snap = [t.clone() for t in cb.getStateTensors(ms[0])]
    a = ms[0](frames[3]).clone()
    ref3 = ms[1](frames[3]).clone()
    assert torch.equal(a, ref3)
    for now, prev in zip(cb.getStateTensors(ms[0]), snap):      # back to the state before frame 3
        now.copy_(prev)
    b = ms[0](frames[3]).clone()
    assert torch.equal(b, ref3)
    # and the sequence continues identically afterwards (candidate path re-armed)
    for f in frames[4:]:
        assert torch.equal(ms[0](f), ms[1](f))
    # a restore to a much older state followed by a different frame: still equal to a model that
    # really was in that state
    m3 = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=cand)
    for f in frames[:3]:
        m3(f)
    for now, prev in zip(cb.getStateTensors(ms[0]), snap):
        now.copy_(prev)
    assert torch.equal(ms[0](frames[5]), m3(frames[5]))
    wall, dev = evalTools.inferNextFrameBenchmark(ms[0], frames[4])
    assert wall > 0 and dev > 0


@pytest.mark.parametrize("u8", [False, True])
def test_detect_input_then_forward_equals_forward(u8):
    """CBConv2d.detectInput(frame) + model(token) == model(frame): the split that lets a pipeline
    read frames in place and replay the rest of the model as one CUDA graph."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(2, 40, 64, 6, 0.1)]
    if u8:
        frames = [f.mul(255).round().to(torch.uint8) for f in frames]
    ms = [models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, candidateDetect=True)
          for _ in range(2)]
    firsts = [[c for c in m.modules() if type(c) is cb.CBConv2d][0] for m in ms]
    if u8:
        for f in firsts:
            f.inputNorm = (255.0, 0.0)
    with pytest.raises(cb._lib.CBinferError):
        firsts[1].detectInput(frames[0])                       # not warmed up yet
    for t, f in enumerate(frames):
        a = ms[0](f)
        b = ms[1](f) if t < 2 else ms[1](firsts[1].detectInput(f))
        assert torch.equal(a, b), t
        assert torch.equal(firsts[0].prevInput, firsts[1].prevInput), t


def test_pose_model_cb_vs_dense_and_parallel_branches():
    """CPM (T=2) converted: threshold 0 equals the dense model within the bf16 bar; running branch 2
    of every stage on a side stream (also inside a CUDA graph) gives identical results."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    from cbinfer_b200.runtime import FrameGraph
    pose = models.PoseModel(T=2).cuda().to(torch.bfloat16)
    frames = [f.cuda().to(torch.bfloat16) for f in video.sequence(1, 96, 128, 5, 0.1, lo=-0.5, hi=0.5)]
    seq = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
    par = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
    par.parallelBranches = True
    with torch.no_grad():
        for f in frames[:3]:
            a, b = seq(f), par(f)
            for u, v in zip(a, b):
                assert torch.equal(u, v)
        ref = pose(frames[2])
        for u, v in zip(a, ref):
            assert _rel(to_val(u), to_val(v)) <= 1e-2
        x = frames[3].clone()
        g = FrameGraph(par, x)
        for f in frames[3:]:
            x.copy_(f)
            got = g.replay()
            exp = seq(f)
            for u, v in zip(got, exp):
                assert torch.equal(u, v)


def test_computation_stats():
    """gatherComputationStats (reference conv2d.py:201-218): op counts of the CG / FG variants from
    the thresholded difference and its un-padded per-channel dilation, recomputed here in numpy."""
    import cbinfer_b200 as cb
    Cin, Cout, k, H, W, thr = 5, 7, 3, 12, 17, 0.2
    conv = nn.Conv2d(Cin, Cout, k, padding=1).cuda()
    m = cb.CBConv2d(conv, thr)
    m.gatherComputationStats = True
    f0 = rand_tensor((1, Cin, H, W), "f32", 1).cuda()
    f1 = perturb(f0.cpu(), 0.15, 2).cuda()
    m(f0)
    m(f1)
    st = {kk: int(v) for kk, v in m.compStats.items()}
    a, b = to_np(f0)[0], to_np(f1)[0]
    chg = np.abs(b - a) > np.float32(thr)
    ops = Cout * k * k * 2
    prop = np.zeros((Cin, H - k + 1, W - k + 1), bool)
    for dy in range(k):
        for dx in range(k):
            prop |= chg[:, dy:dy + H - k + 1, dx:dx + W - k + 1]
    assert st["numInputChangesPerFeatureMap"] == int(chg.sum()) * ops
    assert st["numInputChanges"] == int(chg.any(0).sum()) * Cin * ops
    assert st["numInputPropedChangesPerFeatureMap"] == int(prop.sum()) * ops
    assert st["numInputPropedChanges"] == int(prop.any(0).sum()) * Cin * ops
    assert st["totalInputValues"] == W * H * Cin * ops


def test_warm_model_cast_resets_state():
    """nn.Module._apply (model.half(), .to(...)) replaces the registered state buffers with tensors
    that no longer alias the pixel-major storage the kernels write: the modules must notice and
    start from fresh state instead of returning a stale prevOutput."""
    import cbinfer_b200 as cb
    torch.manual_seed(4)
    base = nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(8, 6, 3, padding=1)).cuda().eval()
    m = cb.convertPools(cb.convert(base, threshold=0.0))
    frames = _frames((1, 3, 16, 20), "f32", 3, 0.2, seed=1)
    for f in frames[:2]:
        m(f)
    m.half()                                        # warm model, new dtype
    base_h = base.half()
    x = frames[2].half()
    out = m(x)
    ref = base_h(x)
    assert out.dtype == torch.float16
    assert _rel(to_val(out), to_val(ref)) <= 5e-3
    m.float()                                       # and back (weights were rounded to fp16 meanwhile)
    base.float()
    out = m(frames[2])
    assert _rel(to_val(out), to_val(base(frames[2]))) <= 1e-4
    c0 = [c for c in m.modules() if type(c) is cb.CBConv2d][0]
    assert c0.prevInput.data_ptr() == c0._inBuf.data_ptr()


def test_change_indexes_of_wrong_grid_are_rejected():
    """the reference's CBPoolMax2d(propChangeIndexes) forwards INPUT-resolution indices
    (conv2d.py:75-76); a following CBConv2d must not scatter with them."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import _lib
    torch.manual_seed(5)
    conv0 = cb.CBConv2d(nn.Conv2d(3, 4, 3, padding=1).cuda(), 0.1)
    conv0.propChangeIndexes = True
    pool = cb.CBPoolMax2d(nn.MaxPool2d(2, 2))
    pool.propChangeIndexes = True
    conv1 = cb.CBConv2d(nn.Conv2d(4, 4, 3, padding=1).cuda(), 0.1)
    x = rand_tensor((1, 3, 12, 16), "f32", 1)
    with pytest.raises(_lib.CBinferError):
        conv1(pool(conv0(x)))


def test_marker_for_another_module_is_rejected():
    """A DetectionDone / FrameDone in the tuple tells its owner that an upstream kernel already did
    part of the owner's frame; any other module taking it would skip work nobody did."""
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    from cbinfer_b200.conv2d import DetectionDone, FrameDone
    a, b = (cb.CBConv2d(nn.Conv2d(4, 4, 3, padding=1).cuda(), 0.1) for _ in range(2))
    pool = cb.CBPoolMax2d(nn.MaxPool2d(2, 2))
    x = rand_tensor((1, 4, 12, 16), "f32", 1)
    for module, marker in ((b, DetectionDone(a)), (b, FrameDone(a)), (pool, FrameDone(a))):
        with pytest.raises(CBinferError):
            module(('changeIndexes', x, marker))
    assert b._fresh and b._lastThr is None           # nothing was recorded for b
