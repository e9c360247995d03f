"""Per-stream thresholds (cbinfer_b200.setStreamThresholds, the cb_*_thr entry points): each
threshold-taking launch with a table against one scalar launch per stream, a table equal to the scalars
against no table, the model-level rule (stream b with table T computes what the model computes with the
scalars T[:, b]), graphs, lowering (which restarts a stream), composition with the other per-stream
controls, refusals and pickles."""
import copy
import json
import os
import pickle
import subprocess
import sys

import pytest
import torch

from tests.test_gpu_stream_reset import FUSED_FRAME, _calls

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}

pytestmark = pytest.mark.gpu

# 0, values that round differently to fp16 and to bf16, and ordinary ones
VALUES = [0.0, 0.1, 1.0 / 3.0, 0.0999, 0.05, 0.30078125, 0.2, 0.015, 0.07]


def _table(B, device="cuda"):
    """the per-stream values with guard words around them (a kernel reading past [0, B) sees NaN)"""
    g = torch.full((B + 8,), float("nan"), dtype=torch.float32, device=device)
    g[4:4 + B] = torch.tensor(VALUES[:B], dtype=torch.float32)
    return g[4:4 + B]


def _per_stream(make, run, B, slicers):
    """`make()` -> fresh inputs/outputs (same content every call), `run(t, thr_b, scalar)` launches on them.
    One launch with the table against B launches of the plain entry point with t[b]; stream b's slice of
    every output (slicers: name -> fn(tensors, b)) must be bit-identical."""
    t = _table(B)
    got = make()
    run(got, t, 0.0)
    for b in range(B):
        ref = make()
        run(ref, None, float(t[b]))
        for name, sl in slicers.items():
            assert torch.equal(sl(got, b), sl(ref, b)), (name, b)


def _stream_bits(key, B):
    return lambda d, b: d[key].view(B, -1)[b]


# ---- dense detection: the four kernel choices and uint8 --------------------------------------------

def _dense_case(layout, dt, B, C, H, W, aux, seed):
    from cbinfer_b200 import conv2d_cg as cg
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(B, C, H, W, generator=g, device="cuda").to(dt)
    s = (x.float() + (torch.rand(B, C, H, W, generator=g, device="cuda") - 0.5) * 0.5).to(dt)
    if layout == "vec":                          # pixel-major both sides
        xv, _ = cg.pixel_major(x.shape, dt, "cuda", 0)
        xv.copy_(x)
        sv, _ = cg.pixel_major(x.shape, dt, "cuda", 0)
    elif layout in ("narrow", "planar"):        # planar x, pixel-major state (one chunk / several chunks)
        xv = x.contiguous()
        sv, _ = cg.pixel_major(x.shape, dt, "cuda", 0)
    else:                                       # generic: planar on both sides
        xv = x.contiguous()
        sv = torch.empty_like(x).contiguous()
    sv.copy_(s)
    d = dict(x=xv, state=sv, bits=torch.zeros(B * H * ((W + 31) // 32), dtype=torch.int32, device="cuda"))
    if aux == "tf32":
        lo, _ = cg.pixel_major(x.shape, dt, "cuda", 0)
        d["aux"] = ("tf32", lo)
    elif aux == "bf16":
        d["aux"] = ("bf16",) + cg.bf16_planes(torch.zeros(B, H, W, C, device="cuda"), C)
    return d


DENSE = [("vec", 16), ("narrow", 3), ("planar", 16), ("generic", 5)]


@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout,C", DENSE)
@pytest.mark.parametrize("B,W", [(1, 33), (4, 31), (9, 7), (3, 100)])
@pytest.mark.parametrize("update", [1, 2])
def test_dense_detect_per_stream(dt, layout, C, B, W, update):
    from cbinfer_b200 import conv2d_cg as cg
    dtype, H = DTYPES[dt], 5
    auxes = [None, "tf32", "bf16"] if dt == "f32" and layout in ("vec", "planar") else [None]
    for aux in auxes:
        make = lambda: _dense_case(layout, dtype, B, C, H, W, aux, seed=B * 100 + W)

        def run(d, thr_b, thr):
            cg.detect(d["x"], d["state"], d["bits"], thr, update, aux=d.get("aux"), thr_b=thr_b)
        sl = {"bits": _stream_bits("bits", B), "state": lambda d, b: d["state"][b]}
        if aux:
            sl["aux"] = lambda d, b: torch.cat([p[b].reshape(-1).float() for p in d["aux"][1:]])
        _per_stream(make, run, B, sl)


@pytest.mark.parametrize("B,W", [(1, 33), (5, 31), (9, 64)])
def test_u8_detect_per_stream(B, W):
    from cbinfer_b200 import conv2d_cg as cg
    H, C = 6, 3

    def make():
        g = torch.Generator(device="cuda").manual_seed(B + W)
        x = torch.randint(0, 256, (B, C, H, W), generator=g, device="cuda", dtype=torch.uint8)
        st, _ = cg.pixel_major((B, C, H, W), torch.float32, "cuda", 0)
        st.copy_(torch.rand(B, C, H, W, generator=g, device="cuda"))
        return dict(x=x, state=st, bits=torch.zeros(B * H * ((W + 31) // 32), dtype=torch.int32, device="cuda"))

    def run(d, thr_b, thr):
        cg.detect_u8(d["x"], d["state"], d["bits"], thr, 2, 255.0, 0.0, thr_b=thr_b)
    _per_stream(make, run, B, {"bits": _stream_bits("bits", B), "state": lambda d, b: d["state"][b]})


# ---- candidate detection: vec / generic, + compaction tracked and untracked ---------------------

def _cand_case(dt, B, C, H, W, planar, seed):
    from cbinfer_b200 import conv2d_cg as cg
    d = _dense_case("generic" if planar else "vec", DTYPES[dt], B, C, H, W, None, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    idx = torch.nonzero(torch.rand(B * H * W, generator=g, device="cuda") < 0.4)[:, 0].int()
    d["cand"] = cg.ChangeIndexes.from_tensor(idx, (B, H, W))
    return d


@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("B,W", [(1, 33), (4, 31), (9, 17)])
@pytest.mark.parametrize("update", [1, 2])
def test_sparse_detect_per_stream(dt, planar, B, W, update):
    from cbinfer_b200 import conv2d_cg as cg
    H, C = 5, 16
    make = lambda: _cand_case(dt, B, C, H, W, planar, seed=B * 7 + W)

    def run(d, thr_b, thr):
        cg.detect_sparse(d["x"], d["state"], d["bits"], thr, update, d["cand"], thr_b=thr_b)
    _per_stream(make, run, B, {"bits": _stream_bits("bits", B), "state": lambda d, b: d["state"][b]})


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("tracked", [False, True])
@pytest.mark.parametrize("B,W", [(1, 33), (4, 31), (9, 17)])
def test_sparse_compact_per_stream(dt, tracked, B, W):
    from cbinfer_b200 import conv2d_cg as cg
    H, C, HW = 5, 16, 5 * W

    def make():
        d = _cand_case(dt, B, C, H, W, False, seed=B * 3 + W)
        d.update(dil=torch.zeros_like(d["bits"]), idx=torch.zeros(B * HW, dtype=torch.int32, device="cuda"),
                 count=torch.zeros(1, dtype=torch.int32, device="cuda"),
                 sync=torch.zeros(1, dtype=torch.int32, device="cuda"),
                 rows=(torch.zeros(B, dtype=torch.int32, device="cuda"),
                       torch.zeros(B + 1, dtype=torch.int32, device="cuda")))
        return d

    def run(d, thr_b, thr):
        cg.detect_sparse_compact(d["x"], d["state"], d["bits"], thr, 2, d["cand"], (3, 3), d["idx"], d["count"],
                                 d["sync"], dil_bits=d["dil"], streams=d["rows"] if tracked else None, thr_b=thr_b)

    def lst(d, b):
        idx = d["idx"][: int(d["count"].item())].long()
        return idx[idx // HW == b]
    sl = {"bits": _stream_bits("bits", B), "dil": _stream_bits("dil", B), "state": lambda d, b: d["state"][b],
          "list": lst}
    if tracked:
        sl["counts"] = lambda d, b: d["rows"][0][b]
    _per_stream(make, run, B, sl)


# ---- pool + detect -----------------------------------------------------------------------------------

@pytest.mark.parametrize("dt", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("B,W", [(1, 34), (4, 31), (9, 17)])
def test_pool_detect_per_stream(dt, B, W):
    from cbinfer_b200 import conv2d_cg as cg
    dtype, H, C = DTYPES[dt], 6, 16
    oH, oW = H // 2, W // 2

    def make():
        g = torch.Generator(device="cuda").manual_seed(B * 11 + W)
        x, _ = cg.pixel_major((B, C, H, W), dtype, "cuda", 0)
        x.copy_(torch.rand(B, C, H, W, generator=g, device="cuda"))
        out, _ = cg.pixel_major((B, C, oH, oW), dtype, "cuda", 0)
        out.copy_(torch.rand(B, C, oH, oW, generator=g, device="cuda"))
        ns, _ = cg.pixel_major((B, C, oH, oW), dtype, "cuda", 0)
        ns.copy_(torch.rand(B, C, oH, oW, generator=g, device="cuda"))
        s = cg.alloc_scratch((B, H, W), "cuda")
        raw = (torch.rand(B, H, W, generator=g, device="cuda") < 0.3).to(torch.int8)
        cg._lib.check(cg.C.cb_map_to_bits(cg.stream_ptr(), raw.data_ptr(), s["raw_bits"].data_ptr(), B, H, W))
        cg.dilate_compact(s["raw_bits"], (B, H, W), (1, 1), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"])
        ci = cg.ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])
        return dict(x=x, out=out, ns=ns, ci=ci,
                    nbits=torch.zeros(B * oH * ((oW + 31) // 32), dtype=torch.int32, device="cuda"))

    def run(d, thr_b, thr):
        cg.maxPool2d_detect(d["x"], d["out"], d["ci"], d["ns"], d["nbits"], thr, 2, thr_b=thr_b)
    _per_stream(make, run, B, {"out": lambda d, b: d["out"][b], "ns": lambda d, b: d["ns"][b],
                               "nbits": _stream_bits("nbits", B)})


# ---- the fused tail: both tables, one of them, tracked and untracked ------------------------------

FACTORS = [1.0, 0.5, 2.0, 0.0, 1.5, 0.25, 1.0, 3.0, 0.75]      # per stream, times the kernels' base values


def _guarded(vals):
    g = torch.full((len(vals) + 8,), float("nan"), dtype=torch.float32, device="cuda")
    g[4:4 + len(vals)] = torch.tensor(vals, dtype=torch.float32)
    return g[4:4 + len(vals)]


TAIL_CHANNELS = [(64, 16, 3), (128, 32, 8), (256, 64, 13)]
TAIL_THR_CASES = [(B, TAIL_CHANNELS[k % 3], ("CHANGED", "ALL")[k % 2], which, tracked)
                  for k, (B, which, tracked) in enumerate((B, w, t) for B in (1, 3, 9)
                                                          for w in ("both", "thr1", "thr2") for t in (False, True))]


@pytest.mark.parametrize("case", TAIL_THR_CASES, ids=lambda c: "B%d-C%d-%d-%d-%s-%s-%s" % (
    (c[0],) + c[1] + (c[2], c[3], "tracked" if c[4] else "untracked")))
def test_tail_per_stream(case):
    """cb_tail_update_thr with thr1_b and / or thr2_b against one scalar launch per stream: stream b's rows
    of both states and outputs and its per-stream counts are bit-identical.  The inputs are those of the
    fp64 tests (tests/test_gpu_fused_ops.py): rows at exactly the base threshold, one ulp above it, and
    layer-2 states near layer 1's output, so factor 1.0 keeps those edges."""
    import numpy as np
    from cbinfer_b200 import _lib
    from cbinfer_b200 import conv2d_cg as cg
    from tests.test_gpu_fused_ops import THR1, THR2, _tail_inputs
    B, (C0, C1, C2), upd, which, tracked = case
    n = 150 * B + 37
    rng = np.random.default_rng([B, C0, C1, C2])
    (H, W), x, cand, _, st1, w1, b1, out1, st2, w2, b2, out2 = _tail_inputs(rng, n, B, C0, C1, C2, True)
    packed1 = cg.pack_weights(torch.from_numpy(w1).cuda().view(C1, C0, 1, 1), _lib.GEMM_TC_BF16X3)
    packed2 = cg.pack_weights(torch.from_numpy(w2).cuda().view(C2, C1, 1, 1), _lib.GEMM_TC_BF16X3)
    b1_t, b2_t = torch.from_numpy(b1).cuda(), torch.from_numpy(b2).cuda()
    ci = cg.ChangeIndexes.from_tensor(torch.from_numpy(cand.astype(np.int32)).cuda(), (B, H, W))
    t1 = _guarded([THR1 * f for f in FACTORS[:B]])
    t2 = _guarded([THR2 * f for f in FACTORS[:B]])
    mode = getattr(_lib, "UPDATE_" + upd)

    def make():
        buf = lambda a: torch.from_numpy(a).cuda().view(B, H, W, a.shape[1])
        z = lambda k: torch.zeros(k, dtype=torch.int32, device="cuda")
        return dict(x=buf(x), st1=buf(st1), out1=buf(out1), st2=buf(st2), out2=buf(out2), c1=z(1), c2=z(1),
                    sync=z(4), r1=(z(B), z(B + 1)), r2=(z(B), z(B + 1)))

    def run(d, tables, s1, s2):
        cg.tail_update(d["x"], d["st1"], packed1, b1_t, d["out1"], True, s1, d["st2"], packed2, b2_t, d["out2"],
                       False, s2, ci, C0, C1, C2, mode, d["c1"], d["c2"], d["sync"],
                       streams1=d["r1"] if tracked else None, streams2=d["r2"] if tracked else None,
                       thr1_b=tables[0], thr2_b=tables[1])

    got = make()
    run(got, (t1 if which != "thr2" else None, t2 if which != "thr1" else None), THR1, THR2)
    for b in range(B):
        ref = make()
        run(ref, (None, None), float(t1[b]) if which != "thr2" else THR1, float(t2[b]) if which != "thr1" else THR2)
        for k in ("x", "st1", "out1", "st2", "out2"):
            assert torch.equal(got[k][b], ref[k][b]), (k, b)
        if tracked:
            for k in ("r1", "r2"):
                assert torch.equal(got[k][0][b], ref[k][0][b]), (k, b)
    assert int(got["sync"].abs().sum()) == 0


# ---- the tile contraction's pooling epilogue --------------------------------------------------------

TILE_THR_CASES = [  # (mode, dt), Cout, (H, W), B, update, change mask
    (("bf16x3", "f32"), 16, (21, 37), 1, "CHANGED", "block"),
    (("bf16x3", "f32"), 64, (16, 35), 3, "ALL", "iid"),
    (("bf16x3", "f32"), 32, (20, 32), 9, "CHANGED", "iid"),
    (("tc", "bf16"), 32, (21, 37), 3, "ALL", "block"),
    (("tc", "bf16"), 64, (20, 32), 9, "CHANGED", "iid"),
    (("tc", "f16"), 16, (16, 35), 9, "ALL", "block"),
    (("tc", "f16"), 48, (21, 37), 1, "CHANGED", "iid"),
    (("tc3x", "f32"), 32, (23, 37), 4, "ALL", "iid"),
]


@pytest.mark.parametrize("case", TILE_THR_CASES, ids=lambda c: "%s-%s-Cout%d-%dx%d-B%d-%s-%s" % (
    c[0] + (c[1],) + c[2] + (c[3], c[4], c[5])))
def test_tile_pool_per_stream(case):
    """cb_conv_update_tiled_pool_thr against one scalar launch per stream: stream b's conv output, pooled
    map, next-layer raw bits, state and operand planes are bit-identical."""
    import torch.nn.functional as F
    import cbinfer_b200 as cb
    from cbinfer_b200 import _lib
    from cbinfer_b200 import conv2d_cg as cg
    from tests.test_gpu_fused_ops import _change_mask, _next_aux, _next_state
    (mode, dt), Cout, (H, W), B, upd, mask = case
    tdt, gemm = DTYPES[dt], cb.CBConv2d.GEMM_MODES[mode]
    Cin, k = 16, 3
    assert cg.tiled_supported(tdt, gemm, (B, H, W), Cin, Cout, (k, k))
    assert _lib.C.cb_conv_tiled_pool_supported(_lib.dtype_code(tdt), gemm, Cout)
    oH, oW = H // 2, W // 2
    base_thr = {"f32": 0.05, "bf16": 0.1, "f16": 0.05}[dt]
    table = _guarded([base_thr * f for f in FACTORS[:B]])
    g0 = torch.Generator().manual_seed(B * 100 + Cout)
    w = ((torch.rand(Cout, Cin, k, k, generator=g0) - 0.5) * 2 * (Cin * k * k) ** -0.5).to(tdt).cuda()
    bias = (torch.rand(Cout, generator=g0) - 0.5).cuda()
    packed = cg.pack_weights(w, gemm)

    def make():
        gen = torch.Generator().manual_seed(B * 10 + Cout)
        state, sbuf = cg.pixel_major((B, Cin, H, W), tdt, "cuda", 0)
        state.copy_((torch.rand(B, Cin, H, W, generator=gen) - 0.5).to(tdt))
        out, obuf = cg.pixel_major((B, Cout, H, W), tdt, "cuda", 0)
        out.copy_((torch.randn(B, Cout, H, W, generator=gen) * 0.5).to(tdt))
        pooled, _ = cg.pixel_major((B, Cout, oH, oW), tdt, "cuda", 0)
        pooled.copy_(torch.randn(B, Cout, oH, oW, generator=gen).to(tdt))
        raw_bits, shape = cg._map_to_bits(_change_mask(B, H, W, mask, gen).to(torch.int8).cuda())
        s = cg.alloc_scratch(shape, "cuda")
        tile_ws = cg.alloc_tile_ws(shape, "cuda")
        cg.dilate_tiles(raw_bits, shape, (k, k), s["count"], s["ws"], s["dil_bits"], tile_ws)
        ref = F.conv2d(state.double(), w.double(), bias.double(), padding=k // 2).clamp_min(0)
        near = F.max_pool2d(ref, 2, 2)
        nst, nbuf = _next_state(cg, near, base_thr, tdt, gen)
        aux = _next_aux(cg, {"bf16x3": "bf16", "tc3x": "tf32"}.get(mode), nst, nbuf, Cout)
        nbits = torch.zeros(max(_lib.C.cb_bitmap_words(B, oH, oW), 1), dtype=torch.int32, device="cuda")
        return dict(sbuf=sbuf, obuf=obuf, out=out, pooled=pooled, nst=nst, aux=aux, nbits=nbits, tile_ws=tile_ws,
                    dil=s["dil_bits"])

    def run(d, thr_b, thr):
        cg.conv_update_tiled(d["sbuf"], d["tile_ws"], d["dil"], packed, bias, d["obuf"], Cin, Cout, (k, k), True,
                             gemm, pool=dict(out=d["pooled"], next_state=d["nst"], next_raw_bits=d["nbits"],
                                             threshold=thr, mode=getattr(_lib, "UPDATE_" + upd), aux=d["aux"],
                                             thr_b=thr_b))
    sl = {"out": lambda d, b: d["out"][b], "pooled": lambda d, b: d["pooled"][b], "nst": lambda d, b: d["nst"][b],
          "nbits": _stream_bits("nbits", B),
          "aux": lambda d, b: torch.cat([p[b].reshape(-1).float() for p in d["aux"][1:]]) if d["aux"] else
          torch.zeros(1)}
    t = table
    got = make()
    run(got, t, 0.0)
    for b in range(B):
        ref = make()
        run(ref, None, float(t[b]))
        for name, f in sl.items():
            assert torch.equal(f(got, b), f(ref, b)), (name, b)


# ---- models ------------------------------------------------------------------------------------------

def _convs(m):
    import cbinfer_b200 as cb
    return [c for c in m.modules() if type(c) is cb.CBConv2d]


def _scene(base, thr, candidate=True, feedback=True, tiles="auto", fuse=True):
    from cbinfer_b200 import models
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                    clonePoolOutput=False, candidateDetect=candidate)
    for c, t in zip(_convs(m), thr):
        c.threshold = t
        c.feedbackLoop = feedback
        c.tileMode = tiles
    return m


CONFIGS = [dict(candidate=True, feedback=True), dict(candidate=True, feedback=False),
           dict(candidate=False, feedback=True), dict(candidate=True, feedback=True, tiles="off")]


@pytest.fixture(scope="module")
def scene():
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 8, 0.05, seed=0)]
    m = _scene(base, [0.1] * 5)
    thr = models.calibrateThresholds(base, m, frames[0])
    return base, frames, thr


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("cfg", range(len(CONFIGS)))
def test_scalar_table_equals_no_table(scene, dt, cfg):
    """A table equal to the scalars is bit-identical to no table on every frame and stream, eager and in
    graphs, with the same launch list per frame."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    dtype = DTYPES[dt]
    base = copy.deepcopy(base).to(dtype)
    fr = [f.to(dtype) for f in frames]
    a, n = _scene(base, thr, **CONFIGS[cfg]), _scene(base, thr, **CONFIGS[cfg])
    B = fr[0].shape[0]
    cb.setStreamThresholds(a, [[float(torch.tensor(t, dtype=torch.float32))] * B for t in thr])
    with torch.no_grad():
        for f in fr[:4]:
            with _calls() as la:
                oa = a(f)
            with _calls() as ln:
                on = n(f)
            assert la == ln, (la, ln)
            assert torch.equal(oa, on)
            for sa, sn in zip(cb.getStateTensors(a), cb.getStateTensors(n)):
                assert torch.equal(sa, sn)
        if cfg == 0 and dt == "f32":              # the fused pool-detect epilogues and the tail ran with the table
            assert la == FUSED_FRAME, la
        elif cfg == 0:
            assert la.count("conv_update_tiled+pool") == 2, la
        static = fr[4].clone()
        graphs = []
        for m in (a, n):
            m(static)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = m(static)
            graphs.append((g, out))
        for f in fr[5:]:
            static.copy_(f)
            for g, _ in graphs:
                g.replay()
            assert torch.equal(graphs[0][1], graphs[1][1])


def equivalence_main(model, dt, cfg):
    """Run in a subprocess with CBINFER_STREAMK=0 CBINFER_KSPLIT=1.  A model with a table T of distinct
    columns against, per stream b, the same model with the scalars T[:, b]: outputs, states, change lists
    and per-stream counts of stream b are equal on every frame."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    dtype = DTYPES[dt]
    B = 4
    if model == "scene":
        base = models.sceneLabelingBaseline().cuda().to(dtype)
        fr = [f.cuda().to(dtype) for f in video.sequence(B, 96, 128, 7, 0.05, seed=1)]
        thr = models.calibrateThresholds(base, _scene(base, [0.1] * 5, **CONFIGS[cfg]), fr[0])
        mk = lambda scal: _scene(base, scal, **CONFIGS[cfg])
    else:
        pose = models.PoseModel(T=2).cuda().to(dtype)
        fr = [f.cuda().to(dtype) for f in video.sequence(B, 96, 128, 7, 0.1, lo=-0.5, hi=0.5)]
        probe = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
        models.calibrateThresholds(pose, probe, fr[0])
        thr = [c.threshold for c in _convs(probe)]

        def mk(scal):
            m = models.enableCandidateDetection(models.poseModelCBinfer(pose, threshold=0.0))
            for c, t in zip(_convs(m), scal):
                c.threshold = t
            return m
    L = len(thr)
    T = torch.tensor([[t * (0.5, 1.0, 1.7, 3.0)[b] for b in range(B)] for t in thr], dtype=torch.float32)
    a = mk(thr)
    cb.setStreamThresholds(a, T)
    cb.trackStreamChanges(a, B=B)
    refs = []
    for b in range(B):
        r = mk([float(v) for v in T[:, b]])
        cb.trackStreamChanges(r, B=B)
        refs.append(r)
    flat = lambda o: o if isinstance(o, torch.Tensor) else torch.cat([t.reshape(t.shape[0], -1) for t in o], 1)
    with torch.no_grad():
        for t, f in enumerate(fr):
            out = flat(a(f))
            ca = cb.streamChangeCounts(a).clone()
            for b, r in enumerate(refs):
                ro = flat(r(f))
                assert torch.equal(out[b], ro[b]), ("output", t, b)
                assert torch.equal(ca[:, b], cb.streamChangeCounts(r)[:, b]), ("counts", t, b)
                for sa, sr in zip(cb.getStateTensors(a), cb.getStateTensors(r)):
                    if sa.numel():
                        assert torch.equal(sa[b], sr[b]), ("state", t, b)
                for la, lr in zip(_convs(a), _convs(r)):
                    try:
                        ia, ir = la.lastChangeIndexes().long(), lr.lastChangeIndexes().long()
                    except cb._lib.CBinferError:
                        continue
                    HW = la.prevOutput.shape[2] * la.prevOutput.shape[3]
                    assert torch.equal(ia[ia // HW == b], ir[ir // HW == b]), ("list", t, b)
    print(json.dumps({"ok": True, "layers": L}))


MODEL_CASES = [("scene", dt, cfg) for dt in ("f32", "bf16") for cfg in range(len(CONFIGS))] + [("pose", "bf16", 0)]


@pytest.mark.parametrize("model,dt,cfg", MODEL_CASES)
def test_stream_b_equals_the_scalars_of_column_b(model, dt, cfg):
    env = dict(os.environ, CBINFER_STREAMK="0", CBINFER_KSPLIT="1")
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_stream_thresholds import equivalence_main; "
            "equivalence_main(%r, %r, %r)" % (REPO, model, dt, cfg))
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


# ---- graphs and lowering -----------------------------------------------------------------------------

def test_captured_raise_takes_effect_on_replay(scene):
    """Raising values through a captured CUDA-tensor call: the replay computes what an eager model with the
    raised scalars computes."""
    import cbinfer_b200 as cb
    base, frames, thr = scene
    B = frames[0].shape[0]
    a = _scene(base, thr)
    cb.setStreamThresholds(a, [[t] * B for t in thr])
    hi = torch.tensor([[t * 2.0] * B for t in thr], dtype=torch.float32, device="cuda")
    r = _scene(base, thr)
    static = frames[0].clone()
    with torch.no_grad():
        for f in frames[:3]:
            a(f), r(f)
        a(static)
        g = torch.cuda.CUDAGraph()
        src = torch.empty_like(hi)
        with torch.cuda.graph(g):
            cb.setStreamThresholds(a, src)
            out = a(static)
        # the reference sees the same frames: run the frame the capture warm-up ran, raise, then replay
        r(static)
        src.copy_(hi)
        for c, t in zip(_convs(r), hi[:, 0].tolist()):
            c.threshold = t                               # raised scalars: the candidate path stays exact
        for f in frames[3:]:
            static.copy_(f)
            g.replay()
            assert torch.equal(out, r(f))


def lowering_main():
    """Run in a subprocess with CBINFER_STREAMK=0 CBINFER_KSPLIT=1 (a restarted stream changes the batch's
    change count, which must not change the summation order of the others)."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 8, 0.05, seed=0)]
    thr = models.calibrateThresholds(base, _scene(base, [0.1] * 5), frames[0])
    B = frames[0].shape[0]
    a, n = _scene(base, thr), _scene(base, thr)
    T = torch.tensor([[t] * B for t in thr], dtype=torch.float32)
    cb.setStreamThresholds(a, T)
    cb.trackStreamChanges(a, B=B)
    with torch.no_grad():
        for f in frames[:3]:
            a(f), n(f)
        low = T.clone()
        low[0, :] *= 0.5                          # first layer only: plain input, no reset
        cb.setStreamThresholds(a, low)
        for sa, sn in zip(cb.getStateTensors(a), cb.getStateTensors(n)):
            assert torch.equal(sa, sn)                       # nothing was reset
        _convs(n)[0].threshold = float(low[0, 0])            # (the dense first layer may lower its scalar)
        low2 = low.clone()
        low2[2, 1] *= 0.5                         # a candidate-fed row of stream 1
        cb.setStreamThresholds(a, low2)
        cleared = _scene(base, [float(v) for v in low2[:, 1]])
        f = frames[3]
        out, want = a(f), n(f)
        counts = cb.streamChangeCounts(a)[:, 1].tolist()
        assert torch.equal(out[1], cleared(f)[1]), "restarted stream"
        assert counts == [c.prevOutput.shape[2] * c.prevOutput.shape[3] for c in _convs(a)], counts
        others = [0, 2, 3]
        assert torch.equal(out[others], want[others]), "other streams"
    print("ok")


def test_lowering_restarts_only_that_stream():
    """Lowering a candidate-fed row of stream b: on b's next frame its output equals a cleared model's with
    the new thresholds and its counts are H_l * W_l; the other streams equal a run without the call.
    Lowering only the first (plain-input) layer's row resets nothing."""
    env = dict(os.environ, CBINFER_STREAMK="0", CBINFER_KSPLIT="1")
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_stream_thresholds import lowering_main; "
            "lowering_main()" % REPO)
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


def composition_main():
    """Run in a subprocess with CBINFER_STREAMK=0 CBINFER_KSPLIT=1.  A model with a table of distinct
    columns, tracked, under resetStreams and setActiveStreams, against per-column scalar models under the
    same calls: stream b equals stream b of the model with the scalars of column b, outputs and counts.
    After detaching, the stream whose column equals the scalars still equals its reference."""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    base = models.sceneLabelingBaseline().cuda()
    frames = [f.cuda() for f in video.sequence(4, 96, 128, 8, 0.05, seed=3)]
    thr = models.calibrateThresholds(base, _scene(base, [0.1] * 5), frames[0])
    B = frames[0].shape[0]
    T = torch.tensor([[t * (1.0, 0.5, 2.0, 1.5)[b] for b in range(B)] for t in thr], dtype=torch.float32)
    a = _scene(base, thr)
    cb.setStreamThresholds(a, T)
    refs = [_scene(base, [float(v) for v in T[:, b]]) for b in range(B)]
    models_ = [a] + refs
    for m in models_:
        cb.trackStreamChanges(m, B=B)

    def frame(f, check=range(B)):
        outs = [m(f) for m in models_]
        for b in check:
            assert torch.equal(outs[0][b], outs[1 + b][b]), b
            assert torch.equal(cb.streamChangeCounts(a)[:, b], cb.streamChangeCounts(refs[b])[:, b]), b
    with torch.no_grad():
        for f in frames[:2]:
            frame(f)
        for m in models_:
            cb.resetStreams(m, [0])
        frame(frames[2])
        for m in models_:
            cb.setActiveStreams(m, [0, 1, 2])
        frame(frames[3])
        frame(frames[4])
        for m in models_:
            cb.setActiveStreams(m, None)
        frame(frames[5])
        # detaching: a's next eager frame scans densely with the scalars (column 0's values)
        cb.setStreamThresholds(a, None)
        assert all(c._thrRow is None and c._lastThr is None for c in _convs(a))
        frame(frames[6], check=[0])
        frame(frames[7], check=[0])
    print("ok")


def test_composition_with_reset_active_streams_counts_and_detach():
    env = dict(os.environ, CBINFER_STREAMK="0", CBINFER_KSPLIT="1")
    code = ("import sys; sys.path.insert(0, %r); from tests.test_gpu_stream_thresholds import composition_main; "
            "composition_main()" % REPO)
    p = subprocess.run([sys.executable, "-c", code], cwd=REPO, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


def test_refusals_pickles_and_the_pipeline(scene):
    import cbinfer_b200 as cb
    from cbinfer_b200 import runtime
    from cbinfer_b200._lib import CBinferError
    base, frames, thr = scene
    B = frames[0].shape[0]
    a = _scene(base, thr)
    cb.setStreamThresholds(a, [[t * (1.0 + 0.5 * (b % 2)) for b in range(B)] for t in thr])
    assert cb.streamThresholds(a) is cb.streamThresholds(a)
    with torch.no_grad():
        a(frames[0])
        with pytest.raises(CBinferError, match="frame has"):
            a(frames[1][:2])
        with pytest.raises(CBinferError, match="CUDA fp32 table"):
            cb.setStreamThresholds(a, torch.zeros(len(thr), B + 1, device="cuda"))
        with pytest.raises(CBinferError, match="CUDA fp32 table"):
            cb.setStreamThresholds(a, torch.zeros(len(thr), B, dtype=torch.float64, device="cuda"))
        _convs(a)[1].threshold = 123.0
        with pytest.raises(CBinferError, match="assigned"):
            a(frames[1])
        # an older pickle loads with no table
        c = copy.deepcopy(_convs(a)[0])
        del c.__dict__["_thrRow"]
        assert pickle.loads(pickle.dumps(c))._thrRow is None
    # a scalar lowered after a frame, then a table of the new scalars attached: the table starts from the
    # threshold the state was built with, so the lowered candidate-fed rows restart their streams
    m, r = _scene(base, thr), _scene(base, thr)
    with torch.no_grad():
        m(frames[0]), r(frames[0])
        _convs(m)[2].threshold = _convs(r)[2].threshold = thr[2] * 0.5
        cb.setStreamThresholds(m, [[float(c.threshold)] * B for c in _convs(m)])
        assert torch.equal(cb.streamThresholds(m)[2].cpu(), torch.full((B,), thr[2] * 0.5, dtype=torch.float32))
        cleared = _scene(base, [c.threshold for c in _convs(m)])
        assert torch.equal(m(frames[1]), cleared(frames[1]))
    # FramePipeline: the table is attached before the graphs are captured, then written between submits
    m = _scene(base, thr)
    cb.setStreamThresholds(m, [[t] * B for t in thr])
    host = [f.cpu().pin_memory() for f in frames]
    pipe = runtime.FramePipeline(m, frames[0], depth=2)
    ref = _scene(base, thr)
    with torch.no_grad():
        ref(frames[0])
        for i, f in enumerate(host[1:4]):
            if i == 1:
                pipe.setStreamThresholds([[t * 2.0] * B for t in thr])
                for c, t in zip(_convs(ref), thr):
                    c.threshold = float(torch.tensor(t * 2.0, dtype=torch.float32))
            s = pipe.submit(f)
            got = pipe.wait(s)
            want = ref(frames[1 + i])
            assert torch.equal(got, want.cpu())
    pipe.drain()
