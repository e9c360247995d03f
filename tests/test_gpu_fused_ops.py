"""GPU tests of the fused kernels against a float64 reference, each op called directly on pixel-major
buffers: cb_tail_update (two chained 1x1 layers in one launch), cb_conv_update_tiled_pool (conv ->
2x2 pool -> next layer's detection in the tile epilogue) and cb_maxpool2x2_detect.

Teacher-forced, as in test_gpu_parity_baseline.py: a contraction's stored output is compared with
the fp64 reference within CONV_TOL on the pixels it wrote, every other pixel bit-identical to its
value before the call; everything downstream of it (pooled values, change bits, counts, states,
operand planes) is computed exactly from the kernel's own stored output and compared bit for bit, so
no threshold decision can flip on contraction rounding.  Detection is the oracle's changeDetection
(strict '>', the fp16 / bf16 rounded-difference rule) on the candidate or re-pooled pixels only.

The model-level bit-identity tests (test_gpu_tiles.py) check that fusing changes nothing; these check
that the fused kernels compute the right thing, at the shape edges the models never reach.
"""
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_ops import CONV_TOL
from tests.util import ORC_DT, TORCH_DT, bits_to_map

pytestmark = pytest.mark.gpu

UPDATES = ("CHANGED", "ALL", "NONE")

# worst relative contraction error seen per (gemm mode, dtype), printed when the module finishes
WORST = {}


@pytest.fixture(scope="module")
def cbm():
    import cbinfer_b200 as cb
    from cbinfer_b200 import _lib, conv2d_cg
    assert torch.cuda.is_available()
    return dict(cb=cb, lib=_lib, cg=conv2d_cg)


@pytest.fixture(scope="module", autouse=True)
def _report_errors():
    yield
    for key in sorted(WORST):
        print("fused ops: worst contraction error %s/%s %.2e of max|ref| (bar %.0e)"
              % (key[0], key[1], WORST[key], CONV_TOL[key]))


def _rel_err(got, ref, key):
    """max |got - ref| / max |ref| over the compared values (float64 tensors)"""
    if got.numel() == 0:
        return 0.0
    err = float((got - ref).abs().max()) / (float(ref.abs().max()) + 1e-30)
    WORST[key] = max(WORST.get(key, 0.0), err)
    return err


def _bits(t):
    """the stored bits of a floating-point tensor, as integers of the same width"""
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


def _detect_ref(orc, new, old, thr, dt):
    """the oracle's raw change map [B,H,W] (bool) of `new` against `old`, both [B,C,H,W]"""
    new, old = orc.from_torch(new)[0], orc.from_torch(old)[0]
    maps = []
    for b in range(new.shape[0]):
        _, raw = orc.changeDetection(new[b:b + 1], old[b:b + 1], (1, 1), thr, dtype=ORC_DT[dt], return_raw=True)
        maps.append(raw.astype(bool))
    return torch.from_numpy(np.stack(maps))


def _update(lib, name):
    return getattr(lib, "UPDATE_" + name)


# ---------------------------------------------------------------------------------------------
# cb_tail_update: two chained 1x1 layers, fp32 data, 3xBF16 contraction
# ---------------------------------------------------------------------------------------------

THR1, THR2 = 0.25, 0.05
C2S = (1, 3, 8, 13, 16)
# candidate counts by the grid size SMs (one CTA per SM, tiles of up to 128 rows): rows per tile go
# from 8 to 16 above 8*SMs; above 128*SMs CTA 0 takes a second tile (of one row at 128*SMs + 1)
COUNTS = ("0", "1", "7", "9", "8SM", "8SM+1", "128SM-1", "128SM", "128SM+1", "3x128SM+5")


def _count(label, sms):
    return {"0": 0, "1": 1, "7": 7, "9": 9, "8SM": 8 * sms, "8SM+1": 8 * sms + 1, "128SM-1": 128 * sms - 1,
            "128SM": 128 * sms, "128SM+1": 128 * sms + 1, "3x128SM+5": 3 * 128 * sms + 5}[label]


def _tail_cases():
    base = []
    # every (C0, C1) pair, C2 and the candidate count cycling along
    for i, (c0, c1) in enumerate([(c0, c1) for c0 in (64, 128, 192, 256) for c1 in (16, 32, 64)]):
        base.append((c0, c1, C2S[i % 5], COUNTS[i % len(COUNTS)]))
    # every count with C0 = 64 (layer 1's lo operand plane right after its single hi K block) and
    # with 256 -> 64 (the largest shared-memory footprint)
    for j, n in enumerate(COUNTS):
        base.append((64, (16, 32, 64)[j % 3], C2S[(j + 2) % 5], n))
        base.append((256, 64, C2S[(j + 4) % 5], n))
    relus = ((True, False), (False, True), (True, True), (False, False))
    return [c + (UPDATES[k % 3], relus[k % 4], ("asc", "shuffled")[k % 2], (2, 3, 1)[(k // 3) % 3])
            for k, c in enumerate(base)]


TAIL_CASES = _tail_cases()


def _tail_id(c):
    c0, c1, c2, n, upd, (r1, r2), order, B = c
    return "C0=%d-C1=%d-C2=%d-n=%s-%s-relu%d%d-%s-B%d" % (c0, c1, c2, n, upd, r1, r2, order, B)


def _tail_inputs(rng, n, B, C0, C1, C2, relu1):
    """maps of B images holding n candidate pixels and as many non-candidates again (a quarter);
    candidate rows cycle through: changed, changed, unchanged, largest |x - state1| exactly thr1 (not
    changed), one ulp above thr1 (changed).  Layer 2's state is set near the expected layer 1 output:
    within thr2 / 5, off by 0.12 in one channel (changed at thr2, not at thr1), or far."""
    W = 64
    H = max(2, -(-(n + n // 4 + 64) // (B * W)))
    P = B * H * W
    x = rng.standard_normal((P, C0)).astype(np.float32)
    cand = rng.choice(P, n, replace=False).astype(np.int64)
    st1 = x.copy()
    far = rng.random(P) < 0.5                       # differences outside the list: to be ignored
    far[cand] = False
    st1[far] += rng.standard_normal((int(far.sum()), C0)).astype(np.float32)
    cls = np.arange(n) % 5
    r = cand[cls < 2]
    st1[r] += rng.standard_normal((r.size, C0)).astype(np.float32)
    r = cand[cls == 2]
    st1[r] += rng.uniform(-THR1 / 2, THR1 / 2, (r.size, C0)).astype(np.float32)
    for c, ulp in ((3, False), (4, True)):
        r = cand[cls == c]
        ch = rng.integers(0, C0, r.size)
        a = (1 + rng.integers(0, 8, r.size) / 8).astype(np.float32)
        sgn = np.where(rng.random(r.size) < 0.5, -1, 1).astype(np.float32)
        s = (a + sgn * np.float32(THR1)).astype(np.float32)
        if ulp:
            s = np.nextafter(s, s + sgn).astype(np.float32)
        x[r, ch] = a
        st1[r, ch] = s
    w1 = (rng.standard_normal((C1, C0)) * C0 ** -0.5).astype(np.float32)
    b1 = (rng.standard_normal(C1) * 0.5).astype(np.float32)
    w2 = (rng.standard_normal((C2, C1)) * C1 ** -0.5).astype(np.float32)
    b2 = (rng.standard_normal(C2) * 0.5).astype(np.float32)
    out1 = rng.standard_normal((P, C1)).astype(np.float32)
    st2 = rng.standard_normal((P, C1)).astype(np.float32)
    approx = x[cand].astype(np.float64) @ w1.T.astype(np.float64) + b1
    if relu1:
        approx = np.maximum(approx, 0)
    cls2 = rng.integers(0, 3, n)
    near = approx + rng.uniform(-THR2 / 5, THR2 / 5, approx.shape)
    near[np.arange(n), rng.integers(0, C1, n)] += np.where(cls2 == 1, 0.12, 0.0)
    st2[cand] = np.where((cls2 == 2)[:, None], rng.standard_normal(approx.shape), near).astype(np.float32)
    p2 = -(-C2 // 4) * 4
    out2 = np.zeros((P, p2), dtype=np.float32)
    out2[:, :C2] = rng.standard_normal((P, C2))
    return (H, W), x, cand, cls, st1, w1, b1, out1, st2, w2, b2, out2


@pytest.mark.parametrize("case", TAIL_CASES, ids=_tail_id)
def test_tail_update_vs_fp64(cbm, orc, case):
    C0, C1, C2, nlabel, upd, (relu1, relu2), order, B = case
    cg, lib = cbm["cg"], cbm["lib"]
    assert lib.C.cb_tail_supported(lib.F32, lib.GEMM_TC_BF16X3, C0, C1, C2)
    n = _count(nlabel, torch.cuda.get_device_properties(0).multi_processor_count)
    umode = _update(lib, upd)
    rng = np.random.default_rng([C0, C1, C2, n, B])
    (H, W), x, cand, cls, st1, w1, b1, out1, st2, w2, b2, out2 = _tail_inputs(rng, n, B, C0, C1, C2, relu1)
    if order == "asc":
        order_idx = np.argsort(cand)
        cand, cls = cand[order_idx], cls[order_idx]
    dev = "cuda"

    def buf(a):
        return torch.from_numpy(a).to(dev).view(B, H, W, a.shape[1])

    x_b, st1_b, out1_b, st2_b, out2_b = buf(x), buf(st1), buf(out1), buf(st2), buf(out2)
    w1_t, w2_t = torch.from_numpy(w1).to(dev), torch.from_numpy(w2).to(dev)
    packed1 = cg.pack_weights(w1_t.view(C1, C0, 1, 1), lib.GEMM_TC_BF16X3)
    packed2 = cg.pack_weights(w2_t.view(C2, C1, 1, 1), lib.GEMM_TC_BF16X3)
    b1_t, b2_t = torch.from_numpy(b1).to(dev), torch.from_numpy(b2).to(dev)
    ci = cg.ChangeIndexes.from_tensor(torch.from_numpy(cand.astype(np.int32)).to(dev), (B, H, W))
    cand_t = torch.from_numpy(cand).to(dev)
    sync = torch.zeros(4, dtype=torch.int32, device=dev)
    key = ("bf16x3", "f32")
    for rep in range(2):                 # the second call reuses the sync words the first left behind
        if rep:
            moved = cand_t[torch.from_numpy(rng.random(n) < 0.5).to(dev)]
            x_b.view(-1, C0)[moved] += torch.randn(moved.numel(), C0, device=dev)
        before = [t.clone() for t in (x_b, st1_b, out1_b, st2_b, out2_b)]
        xs, s1, o1, s2, o2 = [t.view(-1, t.shape[3]) for t in before]
        count1 = torch.full((1,), -1, dtype=torch.int32, device=dev)
        count2 = torch.full((1,), -1, dtype=torch.int32, device=dev)
        cg.tail_update(x_b, st1_b, packed1, b1_t, out1_b, relu1, THR1, st2_b, packed2, b2_t, out2_b, relu2,
                       THR2, ci, C0, C1, C2, umode, count1, count2, sync)
        torch.cuda.synchronize()
        info = (rep, n)
        # layer 1: the oracle's detection at the candidate rows
        raw1 = _detect_ref(orc, before[0].permute(0, 3, 1, 2), before[1].permute(0, 3, 1, 2), THR1, "f32")
        chg1 = raw1.view(-1).to(dev)[cand_t]
        if rep == 0:                     # the threshold edge is really there: == thr1 unchanged, one ulp above changed
            cls_t = torch.from_numpy(cls).to(dev)
            assert not bool(chg1[cls_t == 3].any()) and bool(chg1[cls_t == 4].all()), info
        rows1 = cand_t[chg1]
        assert int(count1) == rows1.numel(), info
        exp = s1.clone()
        if upd == "CHANGED":
            exp[rows1] = xs[rows1]
        elif upd == "ALL":
            exp[cand_t] = xs[cand_t]
        assert torch.equal(_bits(st1_b.view(-1, C0)), _bits(exp)), info
        o1a = out1_b.view(-1, C1)
        ref1 = xs[rows1].double() @ w1_t.double().t() + b1_t.double()
        if relu1:
            ref1 = ref1.clamp_min(0)
        assert _rel_err(o1a[rows1].double(), ref1, key) <= CONV_TOL[key], info
        kept = torch.ones(o1a.shape[0], dtype=torch.bool, device=dev)
        kept[rows1] = False
        assert torch.equal(_bits(o1a[kept]), _bits(o1[kept])), info
        # layer 2, teacher-forced: detection of the kernel's own layer 1 output against state2
        raw2 = _detect_ref(orc, out1_b.permute(0, 3, 1, 2), before[3].permute(0, 3, 1, 2), THR2, "f32")
        rows2 = rows1[raw2.view(-1).to(dev)[rows1]]
        assert int(count2) == rows2.numel(), info
        exp = s2.clone()
        if upd == "CHANGED":
            exp[rows2] = o1a[rows2]
        elif upd == "ALL":
            exp[rows1] = o1a[rows1]
        assert torch.equal(_bits(st2_b.view(-1, C1)), _bits(exp)), info
        o2a = out2_b.view(-1, out2_b.shape[3])
        ref2 = o1a[rows2].double() @ w2_t.double().t() + b2_t.double()
        if relu2:
            ref2 = ref2.clamp_min(0)
        assert _rel_err(o2a[rows2, :C2].double(), ref2, key) <= CONV_TOL[key], info
        kept = torch.ones(o2a.shape[0], dtype=torch.bool, device=dev)
        kept[rows2] = False
        assert torch.equal(_bits(o2a[kept]), _bits(o2[kept])), info
        assert int((o2a[:, C2:] != 0).sum()) == 0, info                    # pad channels stay zero
        assert int(sync.abs().sum()) == 0, info


# ---------------------------------------------------------------------------------------------
# cb_conv_update_tiled_pool: the conv, then 2x2 pool + the next layer's detection in the epilogue
# ---------------------------------------------------------------------------------------------

TILE_MODES = (("bf16x3", "f32"), ("tc3x", "f32"), ("tc", "bf16"), ("tc", "f16"))
TILE_CINS = (3, 16, 32, 64, 128)
TILE_COUTS = (16, 32, 48, 64)
TILE_KS = (3, 5, 7)
TILE_SIZES = (  # label, H, W, ceil-mode pooling
    ("even", 20, 32, False), ("even", 18, 70, False),     # (70: two words of the pooled bitmap)
    ("oddH", 21, 24, False), ("oddH", 21, 24, True),
    ("oddW", 16, 35, False), ("oddW", 16, 35, True),
    ("odd", 23, 37, False), ("odd", 23, 37, True),
    ("Wlt8", 20, 6, False), ("Wlt8", 19, 7, True),
    ("Hlt16", 10, 40, False), ("Hlt16", 13, 41, True),
)
TILE_MASKS = ("none", "all", "block", "iid", "corners")


def _tile_cases(n=48, seed=2024):
    """every value of every axis n / len(axis) times, combined at random"""
    rnd = random.Random(seed)
    axes = []
    for vals in (TILE_MODES, TILE_CINS, TILE_COUTS, TILE_KS, TILE_SIZES, (1, 3), (True, False), UPDATES,
                 TILE_MASKS):
        col = [vals[i % len(vals)] for i in range(n)]
        rnd.shuffle(col)
        axes.append(col)
    return list(zip(*axes))


TILE_CASES = _tile_cases()


def _tile_id(c):
    (mode, dt), cin, cout, k, (label, H, W, ceil), B, relu, upd, mask = c
    return "%s-%s-Cin%d-Cout%d-k%d-%s-%dx%d-%s-B%d-%s-%s-%s" % (
        mode, dt, cin, cout, k, label, H, W, "ceil" if ceil else "floor", B, "relu" if relu else "norelu", upd, mask)


def _tile_pool_runs(cbm, c):
    (mode, dt), cin, cout, k, (_, H, W, _), B = c[:6]
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    gemm = cb.CBConv2d.GEMM_MODES[mode]
    return bool(cg.tiled_supported(TORCH_DT[dt], gemm, (B, H, W), cin, cout, (k, k))) \
        and bool(lib.C.cb_conv_tiled_pool_supported(lib.dtype_code(TORCH_DT[dt]), gemm, cout))


def test_tile_pool_cases_reach_every_edge(cbm):
    """the combinations the tile path rejects are skipped; every listed value still runs"""
    ran = [c for c in TILE_CASES if _tile_pool_runs(cbm, c)]
    for i, vals in enumerate((TILE_MODES, TILE_CINS, TILE_COUTS, TILE_KS, TILE_SIZES, (1, 3), (True, False),
                              UPDATES, TILE_MASKS)):
        assert set(vals) <= set(c[i] for c in ran), vals


def _change_mask(B, H, W, kind, gen):
    m = torch.zeros(B, H, W, dtype=torch.bool)
    if kind == "all":
        m[:] = True
    elif kind == "iid":
        m = torch.rand(B, H, W, generator=gen) < 0.08
    elif kind == "block":
        h, w = max(1, H // 3), max(1, W // 3)
        for b in range(B):
            y0 = int(torch.randint(0, H - h + 1, (1,), generator=gen))
            x0 = int(torch.randint(0, W - w + 1, (1,), generator=gen))
            m[b, y0:y0 + h, x0:x0 + w] = True
    elif kind == "corners":
        for y, x in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)):
            m[:, y, x] = True
    elif kind == "windows":
        # every non-empty subset of a 2x2 window's four pixels, cycling over the whole windows
        s = 0
        for b in range(B):
            for yo in range(H // 2):
                for xo in range(W // 2):
                    sub, s = s % 15 + 1, s + 1
                    for bit, (dy, dx) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
                        if (sub >> bit) & 1:
                            m[b, 2 * yo + dy, 2 * xo + dx] = True
    else:
        assert kind == "none"
    return m


def _pooled_shape(H, W, ceil):
    return ((H - 1) // 2 + 1, (W - 1) // 2 + 1) if ceil else (H // 2, W // 2)


def _next_state(cg, near, thr, tdt, gen):
    """the next layer's previous-input state [B,C,oH,oW]: per pooled pixel equal to `near` (the
    expected pooled value), within thr / 4 of it, or far from it"""
    B, C, oH, oW = near.shape
    cls = torch.randint(0, 3, (B, 1, oH, oW), generator=gen).to(near.device)
    small = (torch.rand(B, C, oH, oW, generator=gen) - 0.5).to(near.device) * (thr / 2)
    far = torch.randn(B, C, oH, oW, generator=gen).to(near.device)
    val = torch.where(cls == 0, near, torch.where(cls == 1, near + small, far))
    view, buf = cg.pixel_major((B, C, oH, oW), tdt, near.device, 0)
    view.copy_(val.to(tdt))
    return view, buf


def _next_aux(cg, kind, nst, nbuf, C):
    """the next layer's operand planes, consistent with its state: ('bf16', hi, lo) / ('tf32', lo)"""
    if kind == "bf16":
        return ("bf16",) + cg.bf16_planes(nbuf, C)
    if kind == "tf32":
        lo, _ = cg.pixel_major(tuple(nst.shape), torch.float32, nst.device, 0)
        lo.copy_(cg.tf32_lo(nst))
        return ("tf32", lo)
    return None


def _check_pool_detect(cg, orc, dt, upd, thr, touched, pooled, pooled_exp, nst, nst_before, nbits, aux, nbuf, C):
    """pooled map, next layer's raw bits, its state and operand planes after a pool + detect kernel;
    `touched` [B,oH,oW] = the re-pooled windows, `pooled_exp` = their expected values"""
    B, _, oH, oW = pooled.shape
    tm = touched[:, None].expand_as(pooled)
    assert torch.equal(_bits(pooled), _bits(pooled_exp)), "pooled map"
    # the next layer's detection on the re-pooled pixels only (not a dense scan), from the stored pool
    det = _detect_ref(orc, pooled, nst_before, thr, dt).to(pooled.device) & touched
    got = torch.from_numpy(bits_to_map(nbits, B, oH, oW).astype(bool)).to(pooled.device)
    assert torch.equal(got, det), ("next raw bits", int((got != det).sum()))
    if upd == "CHANGED":
        exp = torch.where(det[:, None].expand_as(pooled), pooled, nst_before)
    elif upd == "ALL":
        exp = torch.where(tm, pooled, nst_before)
    else:
        exp = nst_before
    assert torch.equal(_bits(nst), _bits(exp)), "next state"
    if aux is not None and aux[0] == "bf16":
        hi, lo = cg.bf16_planes(nbuf, C)
        assert torch.equal(_bits(aux[1]), _bits(hi)) and torch.equal(_bits(aux[2]), _bits(lo)), "bf16 planes"
    elif aux is not None:
        assert torch.equal(_bits(aux[1]), _bits(cg.tf32_lo(nst))), "tf32 remainder plane"


@pytest.mark.parametrize("case", TILE_CASES, ids=_tile_id)
def test_conv_tiled_pool_vs_fp64(cbm, orc, case):
    (mode, dt), Cin, Cout, k, (label, H, W, ceil), B, relu, upd, mask = case
    if not _tile_pool_runs(cbm, case):
        pytest.skip("the tile path does not take this layer")
    cg, lib, cb = cbm["cg"], cbm["lib"], cbm["cb"]
    tdt, gemm = TORCH_DT[dt], cb.CBConv2d.GEMM_MODES[mode]
    dev = "cuda"
    gen = torch.Generator().manual_seed(TILE_CASES.index(case))
    state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, dev, 0)
    state.copy_((torch.rand(B, Cin, H, W, generator=gen) - 0.5).to(tdt))
    w = ((torch.rand(Cout, Cin, k, k, generator=gen) - 0.5) * 2 * (Cin * k * k) ** -0.5).to(tdt).to(dev)
    bias = (torch.rand(Cout, generator=gen) - 0.5).to(dev)
    out, obuf = cg.pixel_major((B, Cout, H, W), tdt, dev, 0)
    out.copy_((torch.randn(B, Cout, H, W, generator=gen) * 0.5).to(tdt))
    oH, oW = _pooled_shape(H, W, ceil)
    pooled, pbuf = cg.pixel_major((B, Cout, oH, oW), tdt, dev, 0)
    pooled.copy_(torch.randn(B, Cout, oH, oW, generator=gen).to(tdt))
    raw = _change_mask(B, H, W, mask, gen)
    raw_bits, shape = cg._map_to_bits(raw.to(torch.int8).to(dev))
    s = cg.alloc_scratch(shape, dev)
    tile_ws = cg.alloc_tile_ws(shape, dev)
    cg.dilate_tiles(raw_bits, shape, (k, k), s["count"], s["ws"], s["dil_bits"], tile_ws)   # as the product does
    dil = torch.from_numpy(bits_to_map(s["dil_bits"], B, H, W).astype(bool)).to(dev)
    ref = F.conv2d(state.double(), w.double(), bias.double(), padding=k // 2)
    if relu:
        ref = ref.clamp_min(0)
    dm = dil[:, None].expand_as(ref)
    thr = {"f32": 0.05, "bf16": 0.1, "f16": 0.05}[dt]
    near = F.max_pool2d(torch.where(dm, ref, out.double()), 2, 2, ceil_mode=ceil)
    nst, nbuf = _next_state(cg, near, thr, tdt, gen)
    aux = _next_aux(cg, {"bf16x3": "bf16", "tc3x": "tf32"}.get(mode), nst, nbuf, Cout)
    nbits = torch.zeros(max(lib.C.cb_bitmap_words(B, oH, oW), 1), dtype=torch.int32, device=dev)
    out_before, pooled_before, nst_before = out.clone(), pooled.clone(), nst.clone()
    cg.conv_update_tiled(sbuf, tile_ws, s["dil_bits"], cg.pack_weights(w, gemm), bias, obuf, Cin, Cout, (k, k),
                         relu, gemm, pool=dict(out=pooled, next_state=nst, next_raw_bits=nbits, threshold=thr,
                                               mode=_update(lib, upd), aux=aux))
    torch.cuda.synchronize()
    # the contraction: within tolerance at the dilated pixels, bit-identical elsewhere
    assert _rel_err(out.double()[dm], ref[dm], (mode, dt)) <= CONV_TOL[(mode, dt)]
    assert torch.equal(_bits(out)[~dm], _bits(out_before)[~dm])
    # re-pooled: the windows holding a dilated in-image pixel, from the stored conv outputs
    touched = F.max_pool2d(dil[:, None].double(), 2, 2, ceil_mode=ceil)[:, 0] > 0
    exp = F.max_pool2d(out.double(), 2, 2, ceil_mode=ceil).to(tdt)
    exp = torch.where(touched[:, None].expand_as(exp), exp, pooled_before)
    _check_pool_detect(cg, orc, dt, upd, thr, touched, pooled, exp, nst, nst_before, nbits, aux, nbuf, Cout)
    assert int(tile_ws[0]) == 0                      # append counter left clean


# ---------------------------------------------------------------------------------------------
# cb_maxpool2x2_detect: no contraction, every check exact
# ---------------------------------------------------------------------------------------------

MP_CASES = [  # dt, C, B, H, W, ceil, update, next-layer planes, change mask, dilation
    ("f32", 5, 2, 7, 13, True, "CHANGED", "bf16", "windows", 1),      # pitch 8
    ("f32", 5, 1, 1, 9, True, "ALL", "tf32", "iid", 3),               # H = 1
    ("f32", 5, 1, 12, 66, False, "NONE", None, "none", 3),
    ("bf16", 3, 3, 6, 10, False, "NONE", None, "windows", 1),         # pitch 8
    ("bf16", 3, 1, 9, 1, True, "CHANGED", None, "iid", 1),            # W = 1
    ("f32", 64, 2, 8, 33, False, "ALL", "bf16", "windows", 1),
    ("f32", 64, 1, 13, 70, True, "CHANGED", "tf32", "iid", 3),
    ("bf16", 64, 2, 5, 40, True, "ALL", None, "corners", 1),
    ("f16", 64, 1, 7, 7, False, "CHANGED", None, "all", 1),
    ("f16", 185, 2, 9, 11, True, "CHANGED", None, "windows", 1),      # pitch 192: 24 chunks per pixel
    ("f16", 185, 1, 6, 12, False, "ALL", None, "iid", 3),
    ("f16", 185, 1, 1, 1, True, "NONE", None, "all", 1),
    ("f32", 256, 3, 6, 8, False, "CHANGED", "bf16", "windows", 1),    # 64 chunks per pixel
    ("f32", 256, 1, 11, 5, True, "NONE", "tf32", "iid", 3),
    ("f32", 256, 2, 7, 1, True, "ALL", "bf16", "corners", 1),
    ("bf16", 256, 2, 9, 9, False, "ALL", None, "windows", 1),
]


def _mp_id(c):
    dt, C, B, H, W, ceil, upd, aux, mask, k = c
    return "%s-C%d-B%d-%dx%d-%s-%s-aux_%s-%s-k%d" % (dt, C, B, H, W, "ceil" if ceil else "floor", upd, aux, mask, k)


@pytest.mark.parametrize("case", MP_CASES, ids=_mp_id)
def test_maxpool2x2_detect_vs_fp64(cbm, orc, case):
    dt, C, B, H, W, ceil, upd, aux_kind, mask, k = case
    cg, lib = cbm["cg"], cbm["lib"]
    tdt, dev = TORCH_DT[dt], "cuda"
    gen = torch.Generator().manual_seed(MP_CASES.index(case))
    x, _ = cg.pixel_major((B, C, H, W), tdt, dev, 0)
    x.copy_(torch.randn(B, C, H, W, generator=gen).to(tdt))
    oH, oW = _pooled_shape(H, W, ceil)
    pooled, pbuf = cg.pixel_major((B, C, oH, oW), tdt, dev, 0)
    pooled.copy_(torch.randn(B, C, oH, oW, generator=gen).to(tdt))
    thr = {"f32": 0.05, "bf16": 0.1, "f16": 0.05}[dt]
    full = F.max_pool2d(x.double(), 2, 2, ceil_mode=ceil)
    nst, nbuf = _next_state(cg, full, thr, tdt, gen)
    aux = _next_aux(cg, aux_kind, nst, nbuf, C)
    raw = _change_mask(B, H, W, mask, gen)
    raw_bits, shape = cg._map_to_bits(raw.to(torch.int8).to(dev))
    s = cg.alloc_scratch(shape, dev)
    # the list and the bitmap the window ownership reads come from the same compaction
    cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"])
    ci = cg.ChangeIndexes(s["idx"], s["count"], shape, bits=s["dil_bits"])
    nbits = torch.zeros(max(lib.C.cb_bitmap_words(B, oH, oW), 1), dtype=torch.int32, device=dev)
    pooled_before, nst_before = pooled.clone(), nst.clone()
    cg.maxPool2d_detect(x, pooled, ci, nst, nbits, thr, _update(lib, upd), aux=aux)
    torch.cuda.synchronize()
    dil = torch.from_numpy(bits_to_map(s["dil_bits"], B, H, W).astype(bool)).to(dev)
    touched = F.max_pool2d(dil[:, None].double(), 2, 2, ceil_mode=ceil)[:, 0] > 0
    exp = torch.where(touched[:, None].expand_as(full), full.to(tdt), pooled_before)
    _check_pool_detect(cg, orc, dt, upd, thr, touched, pooled, exp, nst, nst_before, nbits, aux, nbuf, C)
    assert int((pbuf[..., C:] != 0).sum()) == 0 and int((nbuf[..., C:] != 0).sum()) == 0   # pad channels
