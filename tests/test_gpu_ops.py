"""GPU parity tests, op level: every kernel of libcbinfer_sm100.so (called through the C ABI via
the python wrappers) against the CPU oracle on the same seeded inputs.

Bars: bit-exact for change masks, bitmaps, index lists, im2col copies, scatters and pooling;
stated tolerances for the contraction.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import (ORC_DT, TORCH_DT, bits_to_map, perturb, rand_tensor, to_np, to_val)

pytestmark = pytest.mark.gpu

# tolerance of the fused contraction vs the fp64-accumulated oracle, relative to max|ref| of the
# compared tensor: (gemm mode, dtype) -> rel
CONV_TOL = {
    ("simt", "f32"): 2e-5,     # fp32 FFMA, fp32 accumulation
    ("tc3x", "f32"): 1e-4,     # 3xTF32 split: north-star bar "rel 1e-4 fp32" (measured ~2e-6)
    ("bf16x3", "f32"): 1e-4,   # 3xBF16 split (the fp32 default): same bar (measured ~2e-5)
    ("tc", "f32"): 4e-3,       # single-pass TF32 (10-bit mantissa), opt-in fast mode
    ("simt", "f16"): 2e-3, ("tc", "f16"): 2e-3,      # output rounding to fp16 dominates
    ("simt", "bf16"): 1e-2, ("tc", "bf16"): 1e-2,    # north-star bar "1e-2 bf16"
}


@pytest.fixture(scope="module")
def cbm():
    import cbinfer_b200 as cb
    from cbinfer_b200 import _lib, conv2d_cg, conv2d_fg
    assert torch.cuda.is_available()
    return dict(cb=cb, lib=_lib, cg=conv2d_cg, fg=conv2d_fg)


def kat_input(seed=1234):
    rs = np.random.RandomState(seed)
    inp = rs.randn(1, 16, 400, 300).astype(np.float32)
    prev = inp.copy()
    for (c, y, x, d) in ((0, 0, 4, 1.00), (1, 6, 9, 0.05), (2, 10, 4, -11.00), (1, 6, 19, -0.05)):
        prev[0, c, y, x] += np.float32(d)
    return inp, prev, 0.1, (3, 3)


# ---------------------------------------------------------------------------------------------
# change detection + propagation + compaction
# ---------------------------------------------------------------------------------------------

def test_kat1_reference_gentestdata(cbm, orc, golden):
    """conv2d_cg.py:84-97,136-142: the reference's own KAT -- 15 dilated pixels."""
    cg = cbm["cg"]
    inp, prev, thr, fs = kat_input(int(golden["kat1_seed"]))
    x = torch.from_numpy(inp).cuda()
    for layout in ("planar", "pixel"):
        st = torch.from_numpy(prev).cuda()
        xx = x
        if layout == "pixel":
            xx = x.contiguous(memory_format=torch.channels_last)
            st = st.contiguous(memory_format=torch.channels_last)
        cmap = cg.changeDetection(xx, st, fs, thr)
        idx = cg.changeIndexesExtr(cmap)
        assert idx.dtype == torch.int32
        assert idx.cpu().tolist() == golden["kat1_map_idx"].tolist()
        assert np.array_equal(cmap.cpu().numpy().astype(np.uint8),
                              orc.changeDetection(inp, prev.copy(), fs, thr))
        X = cg.genXMatrix(x, idx, fs)
        assert np.array_equal(X.cpu().numpy(), golden["kat1_X"])


def test_kat2_change_indexes(cbm):
    """conv2d_cg.py:215-236."""
    cm = torch.zeros(129, 254, dtype=torch.int8)
    for (y, x) in ((3, 3), (7, 5), (5, 7), (7, 1), (1, 5), (24, 31)):
        cm[y][x] = 1
    idx = cbm["cg"].changeIndexesExtr(cm.cuda())
    assert idx.cpu().tolist() == [259, 765, 1277, 1779, 1783, 6127]


@pytest.mark.parametrize("tag", ["a", "b", "c", "d"])
def test_golden_twins(cbm, golden, tag):
    """every staged op against the outputs of the reference's python twins."""
    cg = cbm["cg"]
    C, H, W, kH, kW, Cout, relu = [int(v) for v in golden[f"{tag}_params"]]
    thr = float(golden[f"{tag}_thr"])
    f0 = torch.from_numpy(golden[f"{tag}_f0"]).cuda()
    f1 = torch.from_numpy(golden[f"{tag}_f1"]).cuda()
    cmap = cg.changeDetection(f1, f0.clone(), (kH, kW), thr)
    assert np.array_equal(cmap.cpu().numpy().astype(np.uint8), golden[f"{tag}_map"])
    raw = cg.changeDetection(f1, f0.clone(), (1, 1), thr)
    assert np.array_equal(raw.cpu().numpy().astype(np.uint8), golden[f"{tag}_raw"])
    prop = cg.changePropagation(raw, (kH, kW))
    assert np.array_equal(prop.cpu().numpy().astype(np.uint8), golden[f"{tag}_prop"])
    idx = cg.changeIndexesExtr(cmap)
    assert np.array_equal(idx.cpu().numpy(), golden[f"{tag}_idx"])
    X = cg.genXMatrix(f1, idx, (kH, kW))
    assert np.array_equal(X.cpu().numpy(), golden[f"{tag}_X"])
    Y = cg.matrixMult(X, torch.from_numpy(golden[f"{tag}_w"]).cuda(),
                      torch.from_numpy(golden[f"{tag}_b"]).cuda())
    np.testing.assert_allclose(Y.cpu().numpy(), golden[f"{tag}_Y"], rtol=1e-5, atol=1e-5)
    po = torch.from_numpy(golden[f"{tag}_prevOut"].copy()).cuda()
    Yt = torch.from_numpy(np.ascontiguousarray(golden[f"{tag}_Y"].T)).cuda()
    out = cg.updateOutput(Yt, idx, po, withReLU=bool(relu))
    assert np.array_equal(out.cpu().numpy(), golden[f"{tag}_out"])


DET_CASES = [  # B, C, H, W, kH, kW, thr
    (1, 3, 15, 20, 3, 3, 0.4), (1, 16, 33, 65, 7, 7, 0.6), (2, 5, 9, 14, 5, 3, 0.5),
    (1, 64, 12, 31, 1, 1, 0.3), (3, 8, 7, 96, 3, 7, 0.7), (1, 38, 10, 46, 7, 7, 0.5),
    (1, 185, 6, 9, 7, 7, 0.9), (1, 4, 1, 1, 3, 3, 0.1), (1, 2, 40, 300, 9, 9, 0.8),
]


@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout", ["planar", "pixel", "mixed"])
@pytest.mark.parametrize("case", DET_CASES)
def test_detect_dilate_compact(cbm, orc, dt, layout, case):
    """bit-exact mask, feedback-updated state and index list; planar = generic-stride kernel,
    pixel = vectorised pixel-major kernel (incl. padded pitch for C % vec != 0), mixed = planar NCHW
    frame against a pixel-major state (narrow kernel for one-chunk pixels, shared-memory transposing
    kernel for wide ones)."""
    cg, lib = cbm["cg"], cbm["lib"]
    B, C, H, W, kH, kW, thr = case
    prev = rand_tensor((B, C, H, W), dt, seed=sum(case[:4]) + 1)
    x = perturb(prev, 0.08, seed=B * 7 + C, scale=1.0)
    if layout == "pixel":
        xv, _ = cg.pixel_major((B, C, H, W), TORCH_DT[dt], "cuda", 0)
        xv.copy_(x)
        sv, _ = cg.pixel_major((B, C, H, W), TORCH_DT[dt], "cuda", 0)
        sv.copy_(prev)
    elif layout == "mixed":
        xv, sv = x.contiguous(), None
    else:
        xv, sv = x.contiguous(), prev.clone().contiguous()
    for update in (False, True):
        st = sv.clone() if layout == "planar" else cg.pixel_major((B, C, H, W), TORCH_DT[dt], "cuda", 0)[0]
        st.copy_(prev)
        s = cg.alloc_scratch((B, H, W), "cuda", want_map=True)
        cg.detect(xv, st, s["raw_bits"], thr, lib.UPDATE_CHANGED if update else lib.UPDATE_NONE)
        cg.dilate_compact(s["raw_bits"], (B, H, W), (kH, kW), s["idx"], s["count"], s["ws"],
                          dil_bits=s["dil_bits"], dil_map=s["dil_map"])
        n = int(s["count"].item())
        got_idx = s["idx"][:n].cpu().numpy()
        exp_maps, exp_idx, exp_state = [], [], []
        for b in range(B):
            xb, pb = to_np(x[b:b + 1]), to_np(prev[b:b + 1])
            m, raw = orc.changeDetection(xb, pb, (kH, kW), thr, updateInputState=update,
                                         dtype=ORC_DT[dt], return_raw=True)
            exp_maps.append(m)
            exp_idx.append(orc.changeIndexesExtr(m) + b * H * W)
            exp_state.append(pb)
            assert np.array_equal(bits_to_map(s["raw_bits"], B, H, W)[b], raw)
        assert np.array_equal(s["dil_map"].cpu().numpy().astype(np.uint8), np.stack(exp_maps))
        assert np.array_equal(bits_to_map(s["dil_bits"], B, H, W), np.stack(exp_maps))
        assert np.array_equal(got_idx, np.concatenate(exp_idx))
        assert np.array_equal(to_np(st), np.concatenate(exp_state))           # feedback writes
        # workspace self-cleans: a second call gives the same answer
        cg.dilate_compact(s["raw_bits"], (B, H, W), (kH, kW), s["idx"], s["count"], s["ws"])
        assert int(s["count"].item()) == n


def test_detect_update_all_and_special_values(cbm, orc):
    cg, lib = cbm["cg"], cbm["lib"]
    x = torch.zeros(1, 1, 2, 4, device="cuda")
    st = torch.tensor([[[[0.5, 1e-40, float("nan"), float("inf")],
                         [-0.5, 0.6, -0.6, float("-inf")]]]], device="cuda")
    for thr, expect in ((0.5, [[0, 0, 0, 1], [0, 1, 1, 1]]), (0.0, [[1, 0, 0, 1], [1, 1, 1, 1]])):
        m = cg.changeDetection(x, st.clone(), (1, 1), thr)
        assert m.cpu().tolist() == expect
        assert orc.changeDetection(to_np(x), to_np(st), (1, 1), thr).tolist() == expect
    # fresh state (+inf) marks everything; UPDATE_ALL copies the whole frame (conv2d.py:236)
    xx = rand_tensor((2, 6, 5, 37), "f32", 3)
    view, _ = cg.pixel_major(xx.shape, torch.float32, "cuda", float("inf"))
    s = cg.alloc_scratch((2, 5, 37), "cuda")
    cg.detect(xx, view, s["raw_bits"], 0.1, lib.UPDATE_ALL)
    assert bits_to_map(s["raw_bits"], 2, 5, 37).all()
    assert torch.equal(view, xx)
    # tf32 remainder plane: written wherever the state is written, lo = v - trunc_tf32(v), exact
    for shape, layout in (((2, 6, 5, 37), "pixel"), ((1, 3, 9, 40), "narrow"), ((1, 5, 7, 33), "planar"),
                          ((2, 19, 6, 45), "narrow"), ((1, 64, 5, 70), "narrow")):
        x0, x1 = rand_tensor(shape, "f32", 5), None
        x1 = perturb(x0, 0.2, 6)
        if layout == "planar":
            st, lo = x0.clone(), torch.zeros_like(x0)
            xin = x1
        else:
            st, _ = cg.pixel_major(shape, torch.float32, "cuda", 0)
            lo, _ = cg.pixel_major(shape, torch.float32, "cuda", 0)
            st.copy_(x0)
            xin = x1 if layout == "narrow" else cg.pixel_major(shape, torch.float32, "cuda", 0)[0].copy_(x1)
        lo.copy_(cg.tf32_lo(x0))
        s = cg.alloc_scratch((shape[0], shape[2], shape[3]), "cuda")
        p16 = cbm['lib'].C.cb_plane_pitch16(shape[1])
        h16 = torch.zeros(shape[0], shape[2], shape[3], p16, dtype=torch.bfloat16, device="cuda")
        l16 = torch.zeros_like(h16)
        eh, el = cg.bf16_pair(x0.permute(0, 2, 3, 1))
        h16[..., :shape[1]], l16[..., :shape[1]] = eh, el
        st2 = st.clone() if layout == "planar" else cg.pixel_major(shape, torch.float32, "cuda", 0)[0].copy_(st)
        cg.detect(xin, st, s["raw_bits"], 0.3, lib.UPDATE_CHANGED, aux=('tf32', lo))
        assert torch.equal(lo, cg.tf32_lo(st.contiguous()))
        hi = (st.contiguous().view(torch.int32) & -8192).view(torch.float32)
        assert torch.equal(hi + lo.contiguous(), st.contiguous())
        cg.detect(xin, st2, s["raw_bits"], 0.3, lib.UPDATE_CHANGED, aux=('bf16', h16, l16))
        eh, el = cg.bf16_pair(st2.permute(0, 2, 3, 1))
        assert torch.equal(h16[..., :shape[1]], eh) and torch.equal(l16[..., :shape[1]], el)
        assert float(h16[..., shape[1]:].abs().sum()) == 0.0
        cg.detect(xin, st, s["raw_bits"], 0.3, lib.UPDATE_ALL, aux=('tf32', lo))
        assert torch.equal(st.contiguous(), x1) and torch.equal(lo.contiguous(), cg.tf32_lo(x1))
        cg.detect(xin, st2, s["raw_bits"], 0.3, lib.UPDATE_ALL, aux=('bf16', h16, l16))
        eh, el = cg.bf16_pair(x1.permute(0, 2, 3, 1))
        assert torch.equal(h16[..., :shape[1]], eh) and torch.equal(l16[..., :shape[1]], el)


def test_large_compaction_chained_scan(cbm):
    """many tiles -> exercises the decoupled look-back; checksum + sortedness properties."""
    cg = cbm["cg"]
    B, H, W = 3, 1080, 1920
    g = torch.Generator().manual_seed(9)
    m = (torch.rand(B, H, W, generator=g) < 0.07).to(torch.int8).cuda()
    ci = cg.changeIndexesExtr(m, lazy=True)
    n = len(ci)
    idx = ci.tensor()
    ref = torch.nonzero(m.view(-1)).int().view(-1)
    assert n == ref.numel() and torch.equal(idx, ref)
    d = cg.changePropagation(m, (7, 7))
    ref_d = torch.nn.functional.max_pool2d(m.float().unsqueeze(1), 7, 1, 3).squeeze(1).to(torch.int8)
    assert torch.equal(d, ref_d)


# ---------------------------------------------------------------------------------------------
# fused gather + contraction + scatter
# ---------------------------------------------------------------------------------------------

CONV_CASES = [  # B, Cin, Cout, H, W, kH, kW, frac, relu
    (1, 3, 16, 24, 40, 7, 7, 0.10, True),
    (1, 16, 64, 20, 33, 7, 7, 0.15, True),
    (2, 64, 256, 9, 12, 7, 7, 0.30, True),
    (1, 256, 64, 10, 16, 1, 1, 0.40, True),
    (1, 64, 8, 10, 16, 1, 1, 1.00, False),
    (1, 185, 38, 8, 11, 7, 7, 0.50, False),
    (1, 128, 19, 6, 7, 3, 3, 1.00, True),
    (1, 5, 6, 9, 14, 5, 3, 0.60, True),
    (1, 40, 130, 6, 5, 3, 3, 1.00, False),
    (1, 64, 64, 46, 46, 7, 7, 0.50, True),      # split-K clusters, one tile per cluster
    (1, 128, 128, 46, 46, 7, 7, 1.00, True),    # split-K clusters, several tiles per cluster
    (1, 128, 96, 30, 40, 3, 3, 0.70, False),    # 2-way split-K
]


def _oracle_conv(orc, state_np, idx_np, w_np, b_np, out_np, filt, relu, dtype, B, H, W):
    """per-image reference: genXMatrix -> matrixMult (fp64 acc) -> updateOutput."""
    for b in range(B):
        sel = idx_np[(idx_np >= b * H * W) & (idx_np < (b + 1) * H * W)] - b * H * W
        X = orc.genXMatrix(state_np[b:b + 1], sel.astype(np.int32), filt, dtype)
        Y = orc.matrixMult(X, w_np, b_np, dtype)
        ob = np.ascontiguousarray(out_np[b:b + 1])
        orc.updateOutput(np.ascontiguousarray(Y.T), sel.astype(np.int32), ob, relu, dtype)
        out_np[b:b + 1] = ob
    return out_np


@pytest.mark.parametrize("mode,dt", [("simt", "f32"), ("tc3x", "f32"), ("bf16x3", "f32"), ("tc", "f32"),
                                     ("tc", "bf16"), ("tc", "f16"), ("simt", "bf16")])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_update(cbm, orc, mode, dt, case):
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    B, Cin, Cout, H, W, kH, kW, frac, relu = case
    tdt = TORCH_DT[dt]
    gemm = cb.CBConv2d.GEMM_MODES[mode]
    state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
    state.copy_(rand_tensor((B, Cin, H, W), dt, seed=Cin + H))
    out, obuf = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
    out.copy_(rand_tensor((B, Cout, H, W), dt, seed=Cout + W))
    w = rand_tensor((Cout, Cin, kH, kW), dt, seed=11, scale=(Cin * kH * kW) ** -0.5)
    bias = rand_tensor((Cout,), dt, seed=12)
    g = torch.Generator().manual_seed(5)
    sel = torch.nonzero(torch.rand(B * H * W, generator=g) < frac).view(-1).int().cuda()
    ci = cg.ChangeIndexes.from_tensor(sel, (B, H, W))
    out_before = to_np(out).copy()
    packed = cg.pack_weights(w, gemm)
    cg.conv_update(sbuf, ci, packed, bias.float().contiguous(), obuf, Cin, Cout, (kH, kW), relu, gemm)
    torch.cuda.synchronize()
    exp = _oracle_conv(orc, to_np(state), sel.cpu().numpy(), to_np(w), to_np(bias), out_before,
                       (kH, kW), relu, ORC_DT[dt], B, H, W)
    got_v, exp_v = to_val(out), orc.from_bits(exp, ORC_DT[dt])
    # untouched pixels must be bit-identical; touched ones within tolerance
    touched = np.zeros(B * H * W, bool)
    touched[sel.cpu().numpy()] = True
    tm = np.broadcast_to(touched.reshape(B, 1, H, W), got_v.shape)
    assert np.array_equal(to_np(out)[~tm], exp[~tm])
    if touched.any():
        scale = np.abs(exp_v[tm]).max() + 1e-30
        err = np.abs(got_v[tm] - exp_v[tm]).max() / scale
        assert err <= CONV_TOL[(mode, dt)], (err, mode, dt)
    # pad channels of the pixel-major buffer stay zero
    assert float(obuf[..., Cout:].abs().sum()) == 0.0


SK_CASES = [  # mode, dt, B, Cin, Cout, H, W, k, frac   (all reach the coarse tiling: stream-K applies)
    ("bf16x3", "f32", 8, 64, 256, 60, 80, 7, 0.60),
    ("bf16x3", "f32", 4, 16, 64, 120, 160, 7, 0.50),
    ("bf16x3", "f32", 1, 128, 128, 120, 160, 3, 1.00),
    ("tc3x", "f32", 2, 64, 64, 120, 160, 3, 0.90),
    ("tc", "f32", 2, 64, 96, 120, 160, 3, 0.80),
    ("tc", "bf16", 1, 64, 64, 120, 160, 3, 1.00),
    ("tc", "f16", 2, 32, 256, 100, 120, 5, 0.70),
]


@pytest.mark.parametrize("case", SK_CASES)
def test_conv_update_stream_k(cbm, case):
    """stream-K (equal shares of the (tile, K block) space per CTA, partial tiles summed through the
    workspace) against whole tiles per CTA and against dense F.conv2d; the workspace is left clean."""
    import torch.nn.functional as F
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    mode, dt, B, Cin, Cout, H, W, k, frac = case
    tdt = TORCH_DT[dt]
    gemm = cb.CBConv2d.GEMM_MODES[mode]
    torch.backends.cudnn.allow_tf32 = False
    state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
    state.copy_(rand_tensor((B, Cin, H, W), dt, seed=Cin + H))
    w = rand_tensor((Cout, Cin, k, k), dt, seed=11, scale=(Cin * k * k) ** -0.5).cuda()
    bias = rand_tensor((Cout,), dt, seed=12).cuda()
    g = torch.Generator().manual_seed(5)
    sel = torch.nonzero(torch.rand(B * H * W, generator=g) < frac).view(-1).int().cuda()
    ci = cg.ChangeIndexes.from_tensor(sel, (B, H, W))
    packed = cg.pack_weights(w, gemm)
    ws = torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
    outs = []
    for use_ws in (None, ws, ws):
        out, obuf = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
        out.fill_(3.0)
        cg.conv_update(sbuf, ci, packed, bias.float().contiguous(), obuf, Cin, Cout, (k, k), True, gemm,
                       ws=use_ws)
        torch.cuda.synchronize()
        outs.append(out.float())
    assert int(ws.view(torch.int32)[:1024].abs().sum()) == 0          # flags left clean
    assert torch.equal(outs[1], outs[2])                                # deterministic, reusable
    ref = F.relu(F.conv2d(state.float(), w.float(), bias.float(), padding=k // 2))
    touched = torch.zeros(B * H * W, dtype=torch.bool, device="cuda")
    touched[sel.long()] = True
    tm = touched.view(B, 1, H, W).expand(B, Cout, H, W)
    scale = float(ref.abs().max())
    for o in outs[:2]:
        if not bool(touched.all()):
            assert float((o[~tm] - 3.0).abs().max()) == 0.0              # untouched pixels untouched
        assert float((o[tm] - ref[tm]).abs().max()) / scale <= CONV_TOL[(mode, dt)]


@pytest.mark.parametrize("seed", range(6))
def test_conv_update_random_shapes(cbm, seed):
    """seeded sweep over odd shapes, change counts and tilings (fine / coarse variant, cluster
    split-K widths, stream-K cuts) against dense F.conv2d; unchanged pixels must stay untouched."""
    import random
    import torch.nn.functional as F
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    rnd = random.Random(1234 + seed)
    torch.backends.cudnn.allow_tf32 = False
    ws = torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
    for case in range(8):
        mode, dt = rnd.choice([("bf16x3", "f32"), ("bf16x3", "f32"), ("tc3x", "f32"), ("tc", "bf16"), ("tc", "f16")])
        B = rnd.choice([1, 1, 2, 5])
        Cin = rnd.choice([3, 4, 8, 16, 24, 40, 64, 128, 185])
        Cout = rnd.choice([8, 16, 19, 38, 64, 96, 128, 130, 256])
        k = rnd.choice([1, 3, 3, 5, 7])
        H, W = rnd.randint(5, 70), rnd.randint(5, 90)
        frac = rnd.choice([0.02, 0.1, 0.3, 0.6, 1.0])
        tdt, gemm = TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode]
        g = torch.Generator().manual_seed(seed * 100 + case)
        state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
        state.copy_((torch.rand(B, Cin, H, W, generator=g) - 0.5).to(tdt))
        w = ((torch.rand(Cout, Cin, k, k, generator=g) - 0.5) * 2 * (Cin * k * k) ** -0.5).to(tdt).cuda()
        bias = (torch.rand(Cout, generator=g) - 0.5).to(tdt).cuda()
        sel = torch.nonzero(torch.rand(B * H * W, generator=g) < frac).view(-1).int().cuda()
        ci = cg.ChangeIndexes.from_tensor(sel, (B, H, W))
        out, obuf = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
        out.fill_(2.0)
        cg.conv_update(sbuf, ci, cg.pack_weights(w, gemm), bias.float().contiguous(), obuf, Cin, Cout,
                       (k, k), False, gemm, ws=ws if case % 4 else None)
        torch.cuda.synchronize()
        ref = F.conv2d(state.float(), w.float(), bias.float(), padding=k // 2)
        touched = torch.zeros(B * H * W, dtype=torch.bool, device="cuda")
        touched[sel.long()] = True
        tm = touched.view(B, 1, H, W).expand(B, Cout, H, W)
        o = out.float()
        info = (seed, case, mode, dt, B, Cin, Cout, H, W, k, frac, int(sel.numel()))
        if not bool(touched.all()):
            assert float((o[~tm] - 2.0).abs().max()) == 0.0, info
        if bool(touched.any()):
            err = float((o[tm] - ref[tm]).abs().max()) / (float(ref.abs().max()) + 1e-30)
            assert err <= CONV_TOL[(mode, dt)], (err,) + info
        assert float(obuf[..., Cout:].abs().sum()) == 0.0, info
    assert int(ws.view(torch.int32)[:1024].abs().sum()) == 0


@pytest.mark.parametrize("mode,dt", [("bf16x3", "f32"), ("tc", "bf16")])
def test_conv_update_masked_superset_list(cbm, mode, dt):
    """cb_conv_update_masked: the index list is a superset, the raw bitmap decides which pixels are
    updated; equals cb_conv_update on the exact list, reports the count, clears the bitmap."""
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    tdt, gemm = TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode]
    for (B, Cin, Cout, H, W, fs, fm) in [(2, 64, 48, 30, 45, 0.5, 0.6), (8, 256, 64, 60, 80, 0.4, 0.9),
                                          (1, 16, 8, 9, 70, 1.0, 0.0), (1, 32, 256, 40, 40, 0.7, 1.0)]:
        g = torch.Generator().manual_seed(B * 7 + Cin)
        state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
        state.copy_((torch.rand(B, Cin, H, W, generator=g) - 0.5).to(tdt))
        w = ((torch.rand(Cout, Cin, 1, 1, generator=g) - 0.5) * 2 * Cin ** -0.5).to(tdt).cuda()
        bias = (torch.rand(Cout, generator=g) - 0.5).float().cuda()
        sup = torch.rand(B * H * W, generator=g) < fs                      # superset (candidates)
        keep = sup & (torch.rand(B * H * W, generator=g) < fm)             # flagged subset
        sup_idx = torch.nonzero(sup).view(-1).int().cuda()
        exact_idx = torch.nonzero(keep).view(-1).int().cuda()
        bits = torch.zeros(lib.C.cb_bitmap_words(B, H, W), dtype=torch.int32, device="cuda")
        lib.check(lib.C.cb_map_to_bits(lib.stream_ptr(torch.device("cuda")), keep.view(B, H, W).to(torch.int8).cuda().data_ptr(),
                                       bits.data_ptr(), B, H, W))
        packed = cg.pack_weights(w, gemm)
        ws = torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
        outs = []
        for masked in (False, True):
            out, obuf = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
            out.fill_(1.5)
            if masked:
                cnt = torch.full((1,), -1, dtype=torch.int32, device="cuda")
                sync = torch.zeros(2, dtype=torch.int32, device="cuda")
                cg.conv_update(sbuf, cg.ChangeIndexes.from_tensor(sup_idx, (B, H, W)), packed, bias, obuf,
                               Cin, Cout, (1, 1), True, gemm, ws=ws,
                               mask=dict(bits=bits, clear=True, count=cnt, sync=sync))
                torch.cuda.synchronize()
                assert int(cnt.item()) == int(exact_idx.numel())
                assert int(bits.abs().sum()) == 0 and int(sync.abs().sum()) == 0
            else:
                cg.conv_update(sbuf, cg.ChangeIndexes.from_tensor(exact_idx, (B, H, W)), packed, bias, obuf,
                               Cin, Cout, (1, 1), True, gemm, ws=ws)
            torch.cuda.synchronize()
            outs.append(out.clone())
        assert torch.equal(outs[0], outs[1])


def test_conv_update_zero_changes_is_noop(cbm):
    cg, lib = cbm["cg"], cbm["lib"]
    state, sbuf = cg.pixel_major((1, 16, 8, 8), torch.float32, "cuda", 1.0)
    out, obuf = cg.pixel_major((1, 32, 8, 8), torch.float32, "cuda", 7.0)
    w = rand_tensor((32, 16, 3, 3), "f32", 1)
    ci = cg.ChangeIndexes.from_tensor(torch.zeros(0, dtype=torch.int32, device="cuda"), (1, 8, 8))
    for gemm in (lib.GEMM_SIMT_F32, lib.GEMM_TC, lib.GEMM_TC_3X, lib.GEMM_TC_BF16X3):
        cg.conv_update(sbuf, ci, cg.pack_weights(w, gemm), torch.zeros(32, device="cuda"), obuf,
                       16, 32, (3, 3), True, gemm)
    torch.cuda.synchronize()
    assert float((out - 7.0).abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------
# pooling
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout", ["planar", "pixel"])
@pytest.mark.parametrize("shape,ceil", [((1, 16, 8, 10), False), ((2, 5, 9, 13), True),
                                        ((1, 64, 7, 7), False), ((1, 3, 1, 2), True)])
def test_maxpool(cbm, orc, dt, layout, shape, ceil):
    cg = cbm["cg"]
    B, C, H, W = shape
    oH, oW = ((H - 1) // 2 + 1, (W - 1) // 2 + 1) if ceil else (H // 2, W // 2)
    x0 = rand_tensor(shape, dt, 21)
    if layout == "pixel":
        xv, _ = cg.pixel_major(shape, TORCH_DT[dt], "cuda", 0)
        xv.copy_(x0)
        st, _ = cg.pixel_major((B, C, oH, oW), TORCH_DT[dt], "cuda", float("inf"))
    else:
        xv = x0
        st = torch.full((B, C, oH, oW), float("inf"), dtype=TORCH_DT[dt], device="cuda")
    g = torch.Generator().manual_seed(4)
    m = (torch.rand(B, H, W, generator=g) < 0.3).to(torch.int8).cuda()
    for with_bits in (False, True):
        ci = cg.changeIndexesExtr(m, lazy=True)
        if with_bits:
            ci.bits = cg._map_to_bits(m)[0]
        stc = st.clone() if layout == "planar" else cg.pixel_major((B, C, oH, oW), TORCH_DT[dt], "cuda", float("inf"))[0]
        cg.maxPool2d(xv, stc, ci)
        exp = []
        for b in range(B):
            eb = orc.inf_like((1, C, oH, oW), ORC_DT[dt])
            sel = orc.changeIndexesExtr(m[b].cpu().numpy())
            orc.maxPool2d(to_np(x0[b:b + 1]), eb, sel, dtype=ORC_DT[dt])
            exp.append(eb)
        assert np.array_equal(to_np(stc), np.concatenate(exp))


# ---------------------------------------------------------------------------------------------
# fine-grained path
# ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tag", ["fg1", "fg2"])
def test_fg_golden(cbm, golden, tag):
    """cbconvFG_test1 (conv2d_fg.py:98-150) data through the fused FG kernel vs the reference's
    native conv2d_fg_cpu output; tolerance 1e-4 abs (atomics reorder fp32 sums)."""
    fg = cbm["fg"]
    out = torch.from_numpy(golden[f"{tag}_prevOut"].copy()).cuda()
    prev = torch.from_numpy(golden[f"{tag}_prev"].copy()).cuda()
    x = torch.from_numpy(golden[f"{tag}_in"]).cuda()
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    fg.cbconvFG(x, prev, out, torch.from_numpy(golden[f"{tag}_w"]).cuda(), float(golden[f"{tag}_thr"]), cnt)
    np.testing.assert_allclose(out.cpu().numpy(), golden[f"{tag}_out"], rtol=1e-5, atol=1e-4)
    assert torch.equal(prev, x)
    d = np.abs(golden[f"{tag}_in"] - golden[f"{tag}_prev"])
    assert int(cnt.item()) == int((d > float(golden[f"{tag}_thr"])).sum())


@pytest.mark.parametrize("layout", ["planar", "pixel"])
@pytest.mark.parametrize("case", [(2, 6, 10, 17, 23, 7, 3), (1, 16, 64, 20, 70, 7, 7), (3, 4, 5, 9, 33, 3, 3),
                                  (1, 3, 16, 31, 40, 5, 5), (1, 64, 32, 6, 37, 3, 3)])
def test_fg_tensor_core_path_vs_oracle(cbm, orc, golden, layout, case):
    """cb_fg_detect + cb_dilate_compact + cb_conv_accumulate == the per-value scatter of the
    reference (oracle cbconvFG, pinned to conv2d_fg_cpu by the golden vectors): delta planes, bitmap,
    changed-value count and state exact, output within 1e-4 of max|out| (3xBF16 products)."""
    cg, lib = cbm["cg"], cbm["lib"]
    B, Cin, Cout, H, W, kH, kW = case
    thr = 0.25
    prev = rand_tensor((B, Cin, H, W), "f32", 31 + Cin)
    x = perturb(prev, 0.1, 32 + Cout)
    w = rand_tensor((Cout, Cin, kH, kW), "f32", 33, scale=0.2)
    out0 = rand_tensor((B, Cout, H, W), "f32", 34)
    pv, pbuf = cg.pixel_major((B, Cin, H, W), torch.float32, "cuda", 0)
    pv.copy_(prev)
    ov, obuf = cg.pixel_major((B, Cout, H, W), torch.float32, "cuda", 0)
    ov.copy_(out0)
    xin = x.contiguous() if layout == "planar" else cg.pixel_major((B, Cin, H, W), torch.float32, "cuda", 0)[0].copy_(x)
    p16 = lib.C.cb_plane_pitch16(Cin)
    hi = torch.zeros(B, H, W, p16, dtype=torch.bfloat16, device="cuda")
    lo = torch.zeros_like(hi)
    s = cg.alloc_scratch((B, H, W), "cuda")
    nval = torch.zeros(1, dtype=torch.int32, device="cuda")
    packed = cg.pack_weights(w, lib.GEMM_TC_BF16X3)
    for rep in range(2):                 # second pass: nothing changes any more, planes go back to zero
        cg.fg_detect(xin, pv, pbuf, (hi, lo), s["raw_bits"], thr, count=nval)
        d = (x - prev) if rep == 0 else torch.zeros_like(x)
        chg = d.abs() > thr
        dm = torch.where(chg, d, torch.zeros_like(d)).permute(0, 2, 3, 1)
        eh, el = cg.bf16_pair(dm)
        assert torch.equal(hi[..., :Cin], eh) and torch.equal(lo[..., :Cin], el)
        assert float(hi[..., Cin:].abs().sum()) == 0.0
        assert int(nval.item()) == int(chg.sum())
        assert np.array_equal(bits_to_map(s["raw_bits"], B, H, W), chg.any(1).cpu().numpy().astype(np.uint8))
        assert torch.equal(pv, x)
        cg.dilate_compact(s["raw_bits"], (B, H, W), (kH, kW), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"])
        ch = cg.ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])
        ws = torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
        cg.conv_accumulate((hi, lo), ch, packed, obuf, Cin, Cout, (kH, kW), lib.GEMM_TC_BF16X3, ws=ws)
    for b in range(B):
        e = to_np(out0[b:b + 1])
        orc.cbconvFG(to_np(x[b:b + 1]), to_np(prev[b:b + 1]), e, to_np(w), thr)
        got = ov[b:b + 1].cpu().numpy()
        assert np.abs(got - e).max() <= 1e-4 * max(1.0, np.abs(e).max())


def test_fg_random_vs_oracle(cbm, orc):
    fg = cbm["fg"]
    B, Cin, Cout, H, W, kH, kW = 2, 6, 10, 17, 23, 7, 3
    prev = rand_tensor((B, Cin, H, W), "f32", 31)
    x = perturb(prev, 0.1, 32)
    w = rand_tensor((Cout, Cin, kH, kW), "f32", 33, scale=0.2)
    out0 = rand_tensor((B, Cout, H, W), "f32", 34)
    out = out0.clone()
    p = prev.clone()
    fg.cbconvFG(x, p, out, w, 0.25)
    for b in range(B):
        e = to_np(out0[b:b + 1])
        orc.cbconvFG(to_np(x[b:b + 1]), to_np(prev[b:b + 1]), e, to_np(w), 0.25)
        np.testing.assert_allclose(out[b:b + 1].cpu().numpy(), e, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("n", [1, 100, 300, 5000])
def test_conv_update_stream_k_tiny_change_set(cbm, n):
    """A near-static frame on a large map with the stream-K workspace: fewer (tile, K block) units
    than CTAs.  CTAs with an empty share must drop out (they would never raise their flag and the
    tile owner would wait for them until the trap)."""
    import torch.nn.functional as F
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    B, Cin, Cout, H, W, k = 8, 64, 256, 120, 160, 7
    gemm = lib.GEMM_TC_BF16X3
    torch.backends.cudnn.allow_tf32 = False
    state, sbuf = cg.pixel_major((B, Cin, H, W), torch.float32, "cuda", 0)
    state.copy_(rand_tensor((B, Cin, H, W), "f32", seed=3))
    w = rand_tensor((Cout, Cin, k, k), "f32", seed=11, scale=(Cin * k * k) ** -0.5)
    bias = rand_tensor((Cout,), "f32", seed=12)
    g = torch.Generator().manual_seed(n)
    sel = torch.randperm(B * H * W, generator=g)[:n].sort().values.int().cuda()
    ci = cg.ChangeIndexes.from_tensor(sel, (B, H, W))
    ws = torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
    out, obuf = cg.pixel_major((B, Cout, H, W), torch.float32, "cuda", 0)
    out.fill_(3.0)
    for _ in range(2):
        cg.conv_update(sbuf, ci, cg.pack_weights(w, gemm), bias, obuf, Cin, Cout, (k, k), True, gemm, ws=ws)
    torch.cuda.synchronize()
    assert int(ws.view(torch.int32)[:1024].abs().sum()) == 0
    ref = F.relu(F.conv2d(state, w, bias, padding=k // 2))
    touched = torch.zeros(B * H * W, dtype=torch.bool, device="cuda")
    touched[sel.long()] = True
    tm = touched.view(B, 1, H, W).expand(B, Cout, H, W)
    assert float((out[~tm] - 3.0).abs().max()) == 0.0
    assert float((out[tm] - ref[tm]).abs().max()) / float(ref.abs().max()) <= CONV_TOL[("bf16x3", "f32")]


def test_stream_k_grids_on_concurrent_streams(cbm):
    """Two stream-K contractions (each with its own workspace) on two CUDA streams, 200 rounds: the
    finisher CTAs spin on their contributors' flags, so every grid must be resident as a whole
    (cooperative launch) -- two half-resident grids would wait for each other until the trap."""
    import torch.nn.functional as F
    cg, lib = cbm["cg"], cbm["lib"]
    gemm = lib.GEMM_TC_BF16X3
    torch.backends.cudnn.allow_tf32 = False
    B, Cin, Cout, H, W, k = 4, 64, 256, 120, 160, 7
    jobs = []
    for j in range(2):
        state, sbuf = cg.pixel_major((B, Cin, H, W), torch.float32, "cuda", 0)
        state.copy_(rand_tensor((B, Cin, H, W), "f32", seed=3 + j))
        w = rand_tensor((Cout, Cin, k, k), "f32", seed=11 + j, scale=(Cin * k * k) ** -0.5)
        bias = rand_tensor((Cout,), "f32", seed=12 + j)
        g = torch.Generator().manual_seed(j)
        sel = torch.nonzero(torch.rand(B * H * W, generator=g) < 0.4).view(-1).int().cuda()
        out, obuf = cg.pixel_major((B, Cout, H, W), torch.float32, "cuda", 0)
        jobs.append(dict(state=state, sbuf=sbuf, w=w, bias=bias, sel=sel, out=out, obuf=obuf,
                         ci=cg.ChangeIndexes.from_tensor(sel, (B, H, W)), packed=cg.pack_weights(w, gemm),
                         ws=torch.zeros(lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda"),
                         stream=torch.cuda.Stream()))
    torch.cuda.synchronize()
    for _ in range(200):
        for jb in jobs:
            with torch.cuda.stream(jb["stream"]):
                cg.conv_update(jb["sbuf"], jb["ci"], jb["packed"], jb["bias"], jb["obuf"], Cin, Cout, (k, k), True,
                               gemm, ws=jb["ws"])
    torch.cuda.synchronize()
    for jb in jobs:
        ref = F.relu(F.conv2d(jb["state"], jb["w"], jb["bias"], padding=k // 2))
        touched = torch.zeros(B * H * W, dtype=torch.bool, device="cuda")
        touched[jb["sel"].long()] = True
        tm = touched.view(B, 1, H, W).expand(B, Cout, H, W)
        assert float((jb["out"][tm] - ref[tm]).abs().max()) / float(ref.abs().max()) <= CONV_TOL[("bf16x3", "f32")]
        assert int(jb["ws"].view(torch.int32)[:1024].abs().sum()) == 0
