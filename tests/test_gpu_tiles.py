"""GPU parity tests of the spatially tiled contraction (cb_dilate_compact_tiles +
cb_conv_update_tiled, csrc/conv_tile.cuh): same results as the index-list kernel (cb_conv_update)
and dense F.conv2d, untouched pixels bit-identical, tile list == the set of 8x16 tiles that hold a
dilated change bit.  Reference stages replaced: genXMatrix (cbconv2d_cg_backend.cu:138-161), the
GEMM (conv2d_cg.py:342-349), updateOutput (cbconv2d_cg_backend.cu:175-189).
"""
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import TORCH_DT, bits_to_map
from tests.test_gpu_ops import CONV_TOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cbm():
    import cbinfer_b200 as cb
    from cbinfer_b200 import _lib, conv2d_cg
    assert torch.cuda.is_available()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return dict(cb=cb, lib=_lib, cg=conv2d_cg)


def _change_mask(B, H, W, kind, frac, gen):
    """raw (un-dilated) change mask: iid pixels or one rectangle per image."""
    if kind == "iid":
        return (torch.rand(B, H, W, generator=gen) < frac)
    m = torch.zeros(B, H, W, dtype=torch.bool)
    for b in range(B):
        h = max(1, int(round((frac * H * W * 0.75) ** 0.5)))
        w = max(1, int(round(h / 0.75)))
        h, w = min(h, H), min(w, W)
        y0 = int(torch.randint(0, H - h + 1, (1,), generator=gen))
        x0 = int(torch.randint(0, W - w + 1, (1,), generator=gen))
        m[b, y0:y0 + h, x0:x0 + w] = True
    return m


def _tile_set(dil_map):
    """expected dirty tiles {(b, ty, tx)} of a [B,H,W] uint8 map."""
    B, H, W = dil_map.shape
    out = set()
    for b, y, x in zip(*np.nonzero(dil_map)):
        out.add((int(b), int(y) // 16, int(x) // 8))
    return out


def _run_both(cbm, mode, dt, B, Cin, Cout, H, W, k, kind, frac, seed, relu=False):
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    tdt, gemm = TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode]
    gen = torch.Generator().manual_seed(seed)
    state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
    state.copy_((torch.rand(B, Cin, H, W, generator=gen) - 0.5).to(tdt))
    w = ((torch.rand(Cout, Cin, k, k, generator=gen) - 0.5) * 2 * (Cin * k * k) ** -0.5).to(tdt).cuda()
    bias = (torch.rand(Cout, generator=gen) - 0.5).to(tdt).cuda()
    raw = _change_mask(B, H, W, kind, frac, gen).to(torch.int8).cuda()
    raw_bits, shape = cg._map_to_bits(raw)
    s = cg.alloc_scratch(shape, "cuda")
    tile_ws = cg.alloc_tile_ws(shape, "cuda")
    packed = cg.pack_weights(w, gemm)
    outs = []
    for rep in range(2):        # twice: the tile workspace must be reusable (stamps / counter)
        cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"],
                          tile_ws=tile_ws)
        out_t, obuf_t = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
        out_t.fill_(2.0)
        cg.conv_update_tiled(sbuf, tile_ws, s["dil_bits"], packed, bias.float().contiguous(), obuf_t, Cin,
                             Cout, (k, k), relu, gemm)
        torch.cuda.synchronize()
        outs.append(out_t.float().clone())
        assert float(obuf_t[..., Cout:].abs().sum()) == 0.0
    assert torch.equal(outs[0], outs[1])
    ci = cg.ChangeIndexes(s["idx"], s["count"], shape, bits=s["dil_bits"])
    out_g, obuf_g = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
    out_g.fill_(2.0)
    cg.conv_update(sbuf, ci, packed, bias.float().contiguous(), obuf_g, Cin, Cout, (k, k), relu, gemm)
    torch.cuda.synchronize()
    dil = bits_to_map(s["dil_bits"], B, H, W)
    # tile list == tiles holding a dilated bit
    ntl = int(tile_ws[1])
    NT = (tile_ws.numel() - 4) // 2
    TY, TXp = (H + 15) // 16, ((W + 31) // 32) * 4
    lst = tile_ws[4 + NT: 4 + NT + ntl].cpu().numpy()
    got_tiles = set((int(t) // (TY * TXp), (int(t) % (TY * TXp)) // TXp, int(t) % TXp) for t in lst)
    assert len(got_tiles) == ntl, "duplicate tiles in the list"
    assert got_tiles == _tile_set(dil)
    assert int(tile_ws[0]) == 0                      # append counter left clean
    ref = F.conv2d(state.float(), w.float(), bias.float(), padding=k // 2)
    if relu:
        ref = F.relu(ref)
    tm = torch.from_numpy(dil.astype(bool)).cuda().view(B, 1, H, W).expand(B, Cout, H, W)
    return outs[0], out_g.float(), ref, tm


TILE_CASES = [  # mode, dt, B, Cin, Cout, H, W, k, kind, frac, relu
    ("bf16x3", "f32", 2, 3, 16, 48, 64, 7, "block", 0.10, True),     # 16-byte pixels, two taps per MMA
    ("bf16x3", "f32", 1, 16, 64, 37, 53, 7, "block", 0.20, True),    # 32-byte pixels (SWIZZLE_32B)
    ("bf16x3", "f32", 2, 32, 32, 33, 41, 5, "iid", 0.02, False),     # 64-byte pixels (SWIZZLE_64B)
    ("bf16x3", "f32", 1, 64, 96, 30, 40, 3, "block", 0.30, False),   # 128-byte pixels (SWIZZLE_128B)
    ("bf16x3", "f32", 1, 128, 64, 20, 24, 3, "iid", 0.05, True),     # two 128-byte channel blocks
    ("bf16x3", "f32", 1, 64, 256, 24, 40, 7, "block", 0.50, True),   # N tile 256, streamed weights
    ("bf16x3", "f32", 1, 64, 512, 17, 23, 3, "block", 0.40, False),  # two N tiles
    ("tc3x", "f32", 2, 3, 16, 40, 56, 7, "block", 0.10, True),       # fp32 operands, 16-byte pixels
    ("tc3x", "f32", 1, 16, 32, 30, 44, 3, "iid", 0.05, False),
    ("tc", "f32", 1, 32, 64, 25, 33, 3, "block", 0.20, False),
    ("tc", "bf16", 2, 64, 64, 46, 46, 3, "block", 0.30, True),
    ("tc", "bf16", 1, 3, 64, 50, 70, 3, "block", 0.20, True),
    ("tc", "f16", 1, 185, 128, 23, 23, 7, "block", 0.50, True),      # three channel blocks, K = 9408
    ("tc", "f16", 1, 16, 19, 31, 9, 5, "iid", 0.10, False),          # W < 32, ragged Cout
    ("bf16x3", "f32", 3, 16, 64, 16, 8, 7, "iid", 1.00, True),       # exactly one tile per image, all dirty
    ("bf16x3", "f32", 1, 16, 64, 40, 40, 7, "iid", 0.00, True),      # nothing changed
]


@pytest.mark.parametrize("case", TILE_CASES)
def test_conv_update_tiled(cbm, case):
    mode, dt, B, Cin, Cout, H, W, k, kind, frac, relu = case
    cg, cb = cbm["cg"], cbm["cb"]
    sup = cg.tiled_supported(TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode], (B, H, W), Cin, Cout, (k, k))
    assert sup >= 1, "case must be supported by the tile path"
    o_t, o_g, ref, tm = _run_both(cbm, mode, dt, B, Cin, Cout, H, W, k, kind, frac, seed=Cin + 7 * H, relu=relu)
    if not bool(tm.all()):
        assert float((o_t[~tm] - 2.0).abs().max()) == 0.0           # untouched pixels untouched
        assert float((o_g[~tm] - 2.0).abs().max()) == 0.0
    if bool(tm.any()):
        scale = float(ref.abs().max()) + 1e-30
        assert float((o_t[tm] - ref[tm]).abs().max()) / scale <= CONV_TOL[(mode, dt)]
        # tile path vs index-list path: same operands, same products, different summation order only
        assert float((o_t[tm] - o_g[tm]).abs().max()) / scale <= CONV_TOL[(mode, dt)] * 0.5


@pytest.mark.parametrize("seed", range(4))
def test_conv_update_tiled_random_shapes(cbm, seed):
    cg, cb = cbm["cg"], cbm["cb"]
    rnd = random.Random(4321 + seed)
    ran = 0
    for case in range(10):
        mode, dt = rnd.choice([("bf16x3", "f32"), ("bf16x3", "f32"), ("tc3x", "f32"), ("tc", "bf16"), ("tc", "f16")])
        B = rnd.choice([1, 1, 2, 4])
        Cin = rnd.choice([3, 4, 8, 16, 32, 64, 128])
        Cout = rnd.choice([8, 16, 19, 38, 64, 96, 128, 130])
        k = rnd.choice([3, 3, 5, 7])
        H, W = rnd.randint(5, 70), rnd.randint(5, 90)
        kind, frac = rnd.choice([("block", 0.05), ("block", 0.3), ("iid", 0.01), ("iid", 0.2), ("iid", 1.0)])
        if not cg.tiled_supported(TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode], (B, H, W), Cin, Cout, (k, k)):
            continue
        ran += 1
        o_t, o_g, ref, tm = _run_both(cbm, mode, dt, B, Cin, Cout, H, W, k, kind, frac, seed * 100 + case)
        info = (seed, case, mode, dt, B, Cin, Cout, H, W, k, kind, frac)
        if not bool(tm.all()):
            assert float((o_t[~tm] - 2.0).abs().max()) == 0.0, info
        if bool(tm.any()):
            scale = float(ref.abs().max()) + 1e-30
            assert float((o_t[tm] - ref[tm]).abs().max()) / scale <= CONV_TOL[(mode, dt)], info
    assert ran >= 5


def test_unsupported_shapes_are_reported(cbm):
    cg, cb, lib = cbm["cg"], cbm["cb"], cbm["lib"]
    # 1x1 filters: nothing to reuse; 24 channels of bf16 planes = 48-byte pixels: no swizzle mode
    assert cg.tiled_supported(torch.float32, lib.GEMM_TC_BF16X3, (1, 32, 32), 64, 64, (1, 1)) == 0
    assert cg.tiled_supported(torch.float32, lib.GEMM_TC_BF16X3, (1, 32, 32), 24, 64, (3, 3)) == 0
    assert cg.tiled_supported(torch.float32, lib.GEMM_SIMT_F32, (1, 32, 32), 16, 64, (3, 3)) == 0
    # the scene net: L1 / L2 recommended, L3 (64 -> 256, 7x7) possible but too heavy per tile
    assert cg.tiled_supported(torch.float32, lib.GEMM_TC_BF16X3, (8, 480, 640), 3, 16, (7, 7)) == 1
    assert cg.tiled_supported(torch.float32, lib.GEMM_TC_BF16X3, (8, 240, 320), 16, 64, (7, 7)) == 1
    assert cg.tiled_supported(torch.float32, lib.GEMM_TC_BF16X3, (8, 120, 160), 64, 256, (7, 7)) == 2


@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_module_tile_path_equals_index_path(cbm, dt, monkeypatch):
    """CBConv2d with tileMode 'on' vs 'off' over a short video: identical change sets (bit-exact),
    outputs within the contraction tolerance.  Stream-K is off for the index path so that both
    paths add the same products in the same K order (they are then bit-identical on this hardware,
    which rules out threshold flips in the deeper layers)."""
    import torch.nn as nn
    cb = cbm["cb"]
    from cbinfer_b200 import models, video
    monkeypatch.setenv("CBINFER_STREAMK", "0")
    monkeypatch.setenv("CBINFER_TILES", "1")             # (the test is about the tile path: ignore an outer knob)
    tdt = TORCH_DT[dt]
    torch.manual_seed(3)
    base = nn.Sequential(nn.Conv2d(3, 16, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(16, 64, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(64, 32, 3, padding=1)).cuda().to(tdt).eval()
    frames = [f.cuda().to(tdt) for f in video.sequence(2, 96, 128, 6, 0.08, "block", seed=5)]
    ms = []
    for mode in ("on", "off"):
        m = cb.convertPools(cb.convert(base, threshold=0.05))
        for c in m.modules():
            if type(c) is cb.CBConv2d:
                c.feedbackLoop = True
                c.tileMode = mode
        models.enableCandidateDetection(m)
        ms.append(m)
    tol = 1e-4 if dt == "f32" else 2e-2
    convs = [[c for c in m.modules() if type(c) is cb.CBConv2d] for m in ms]
    for f in frames:
        oa, ob = ms[0](f), ms[1](f)
        torch.cuda.synchronize()
        scale = float(ob.float().abs().max()) + 1e-30
        assert float((oa.float() - ob.float()).abs().max()) / scale <= tol
        for ca, cbb in zip(*convs):
            assert int(ca._scratch["count"]) == int(cbb._scratch["count"])
            assert torch.equal(ca._scratch["dil_bits"], cbb._scratch["dil_bits"])
    assert all("tile_ws" in c._scratch for c in convs[0])
    assert not any("tile_ws" in c._scratch for c in convs[1])


@pytest.mark.parametrize("dt,feedback", [("f32", True), ("f32", False), ("bf16", True), ("f16", True)])
def test_fused_pool_in_tile_epilogue_is_bit_identical(cbm, dt, feedback, monkeypatch):
    """conv (tile path) -> CBPoolMax2d -> conv on the candidate path: with the pooling and the next
    layer's detection fused into the tile kernel's epilogue (cb_conv_update_tiled_pool) every
    pooled map, state, change bitmap, index list and output is bit-identical to the three-kernel
    sequence conv, cb_maxpool2x2_detect."""
    import torch.nn as nn
    cb = cbm["cb"]
    from cbinfer_b200 import models, video
    tdt = TORCH_DT[dt]
    torch.manual_seed(7)
    base = nn.Sequential(nn.Conv2d(3, 16, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(16, 64, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
                         nn.Conv2d(64, 32, 3, padding=1)).cuda().to(tdt).eval()
    frames = [f.cuda().to(tdt) for f in video.sequence(2, 100, 136, 7, 0.08, "block", seed=9)]
    frames.insert(4, frames[3].clone())            # an unchanged frame
    runs = []
    for fuse in ("1", "0"):
        monkeypatch.setenv("CBINFER_FUSE_POOL", fuse)
        m = cb.convertPools(cb.convert(base, threshold=0.04))
        for c in m.modules():
            if type(c) is cb.CBConv2d:
                c.feedbackLoop = feedback
            if type(c) is cb.CBPoolMax2d:
                c.cloneOutput = False
        models.enableCandidateDetection(m)
        outs = []
        for f in frames:
            o = m(f)
            torch.cuda.synchronize()
            convs = [c for c in m.modules() if type(c) is cb.CBConv2d]
            pools = [c for c in m.modules() if type(c) is cb.CBPoolMax2d]
            outs.append(dict(out=o.clone(), counts=[int(c._scratch["count"]) for c in convs],
                             dil=[c._scratch["dil_bits"].clone() for c in convs],
                             states=[c.prevInput.clone() for c in convs],
                             pooled=[p.outputState.clone() for p in pools]))
        runs.append(outs)
        if fuse == "1":
            assert all(getattr(c, '_fusedPool', None) for c in convs[:2])
    for t, (a, b) in enumerate(zip(*runs)):
        assert a["counts"] == b["counts"], t
        assert torch.equal(a["out"], b["out"]), t
        for k in ("dil", "states", "pooled"):
            for x, y in zip(a[k], b[k]):
                assert torch.equal(x, y), (t, k)
    assert sum(runs[0][-1]["counts"]) > 0


@pytest.mark.parametrize("shape,k,frac", [((2, 97, 131), 7, 0.02), ((1, 480, 640), 7, 0.3), ((3, 16, 8), 3, 1.0),
                                          ((1, 40, 40), 5, 0.0), ((2, 33, 65), 17, 0.01), ((1, 50, 300), 19, 0.01),
                                          ((8, 240, 320), 7, 0.05), ((1, 7, 9000), 3, 0.05), ((2, 31, 70), 1, 0.2)])
def test_dilate_tiles_equals_dilate_compact(cbm, shape, k, frac):
    """cb_dilate_tiles (no ordered list) yields the same dilated bitmap, change count and tile set as
    cb_dilate_compact_tiles; the list compacted on demand from the bitmap equals the eager one."""
    cg = cbm["cg"]
    B, H, W = shape
    g = torch.Generator().manual_seed(H + k)
    raw = (torch.rand(B, H, W, generator=g) < frac).to(torch.int8).cuda()
    raw_bits, _ = cg._map_to_bits(raw)
    s1, s2 = cg.alloc_scratch(shape, "cuda"), cg.alloc_scratch(shape, "cuda")
    t1, t2 = cg.alloc_tile_ws(shape, "cuda"), cg.alloc_tile_ws(shape, "cuda")
    for _ in range(2):
        cg.dilate_compact(raw_bits, shape, (k, k), s1["idx"], s1["count"], s1["ws"], dil_bits=s1["dil_bits"], tile_ws=t1)
        cg.dilate_tiles(raw_bits, shape, (k, k), s2["count"], s2["ws"], s2["dil_bits"], t2)
    torch.cuda.synchronize()
    n = int(s1["count"])
    assert int(s2["count"]) == n
    assert torch.equal(s1["dil_bits"], s2["dil_bits"])
    assert int(t1[1]) == int(t2[1])
    NT = (t1.numel() - 4) // 2
    assert sorted(t1[4 + NT: 4 + NT + int(t1[1])].tolist()) == sorted(t2[4 + NT: 4 + NT + int(t2[1])].tolist())
    assert int(t2[0]) == 0
    lazy = cg.ChangeIndexes(s2["idx"], s2["count"], shape, bits=s2["dil_bits"], ws=s2["ws"], listed=False)
    assert len(lazy) == n
    assert torch.equal(lazy.tensor(), s1["idx"][:n])
    # clear_raw: same results, and the raw bitmap comes back zeroed; the workspace is left clean
    rb = raw_bits.clone()
    cg.dilate_tiles(rb, shape, (k, k), s2["count"], s2["ws"], s2["dil_bits"], t2, clear_raw=True)
    assert int(s2["count"]) == n and torch.equal(s1["dil_bits"], s2["dil_bits"]) and int(t2[1]) == int(t1[1])
    assert int(rb.abs().sum()) == 0
    cg.dilate_compact(raw_bits, shape, (k, k), s2["idx"], s2["count"], s2["ws"], dil_bits=s2["dil_bits"], tile_ws=t2)
    assert int(s2["count"]) == n and torch.equal(s2["idx"][:n], s1["idx"][:n])


@pytest.mark.parametrize("feedback", [True, False])
def test_fused_tail_is_bit_identical(cbm, feedback, monkeypatch):
    """conv 7x7 -> 1x1 (ReLU) -> 1x1 on the candidate path: the two trailing 1x1 layers as ONE
    launch (cb_tail_update) against sparse detect + masked contraction twice: outputs, states and
    change counts bit-identical on every frame (same K order, same 3xBF16 split)."""
    import torch.nn as nn
    cb = cbm["cb"]
    from cbinfer_b200 import models, video
    torch.manual_seed(11)
    base = nn.Sequential(nn.Conv2d(3, 64, 7, padding=3), nn.ReLU(), nn.Conv2d(64, 64, 1), nn.ReLU(),
                         nn.Conv2d(64, 8, 1)).cuda().eval()
    base2 = nn.Sequential(nn.Conv2d(16, 256, 3, padding=1), nn.ReLU(), nn.Conv2d(256, 32, 1), nn.ReLU(),
                          nn.Conv2d(32, 16, 1), nn.ReLU()).cuda().eval()
    for net, cin in ((base, 3), (base2, 16)):
        g = torch.Generator().manual_seed(3)
        f0 = torch.rand(2, cin, 60, 88, generator=g)
        frames = [f0]
        for t in range(1, 7):
            f = frames[-1].clone()
            y0, x0 = 5 * t, 9 * t
            f[:, :, y0:y0 + 20, x0:x0 + 30] = torch.rand(2, cin, 20, 30, generator=g)
            frames.append(f)
        frames.insert(3, frames[2].clone())          # an unchanged frame
        frames = [f.cuda() for f in frames]
        runs = []
        for fuse in ("1", "0"):
            monkeypatch.setenv("CBINFER_FUSE_TAIL", fuse)
            m = cb.convert(net, threshold=0.05)
            for c in m.modules():
                if type(c) is cb.CBConv2d:
                    c.feedbackLoop = feedback
            models.enableCandidateDetection(m)
            convs = [c for c in m.modules() if type(c) is cb.CBConv2d]
            assert getattr(convs[1], '_fusedTail', None)
            outs = []
            for f in frames:
                o = m(f)
                torch.cuda.synchronize()
                outs.append(dict(out=o.clone(), counts=[int(c._scratch["count"]) for c in convs],
                                 states=[c.prevInput.clone() for c in convs],
                                 outs=[c.prevOutput.clone() for c in convs]))
            runs.append(outs)
        for t, (a, b) in enumerate(zip(*runs)):
            assert a["counts"] == b["counts"], (t, a["counts"], b["counts"])
            assert torch.equal(a["out"], b["out"]), t
            for k in ("states", "outs"):
                for x, y in zip(a[k], b[k]):
                    assert torch.equal(x, y), (t, k)
        assert sum(runs[0][-1]["counts"]) > 0
        # and against the dense model at the end (thresholded, so only loosely)
        ref = net(frames[-1])
        assert float((runs[0][-1]["out"] - ref).abs().max()) <= 0.2 * float(ref.abs().max()) + 0.05
