#!/usr/bin/env python
"""Per-CTA timeline of conv_tile_kernel (trace build: nvcc -DCB_TILE_TRACE -> build/libcbinfer_trace.so, run
with CBINFER_LIB pointing at it): where a tile kernel's 20-35 us go at 5 % change when its steady state
costs ~2.5 us per tile and CTA.  Times are clock64 cycles since kernel entry of each CTA, printed in us at
the measured SM clock; 'gt' is the CTA's entry on the global timer relative to the first CTA."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cbinfer_b200 as cb
from cbinfer_b200 import conv2d_cg as cg, _lib, video

C = _lib.C
if not hasattr(C, "cb_debug_tile_trace"):
    raise SystemExit("load a trace build: CBINFER_LIB=build/libcbinfer_trace.so")
C.cb_debug_tile_trace.restype = ctypes.c_int
C.cb_debug_tile_trace.argtypes = [ctypes.c_void_p, ctypes.c_int]
MHZ = 1965.0


def run(B, Cin, Cout, H, W, k, rate, cold, pool=False):
    gemm = _lib.GEMM_TC_BF16X3
    torch.manual_seed(0)
    state, sbuf = cg.pixel_major((B, Cin, H, W), torch.float32, "cuda", 0)
    state.copy_(torch.rand(B, Cin, H, W))
    out, obuf = cg.pixel_major((B, Cout, H, W), torch.float32, "cuda", 0)
    w = (torch.randn(Cout, Cin, k, k) * (Cin * k * k) ** -0.5).cuda()
    bias = torch.zeros(Cout, device="cuda")
    f0 = video.base_frame(B, H, W)
    f1 = video.next_frame(f0, 1, rate, "block")
    raw = (f0 != f1).any(1).to(torch.int8).cuda()
    raw_bits, shape = cg._map_to_bits(raw)
    s = cg.alloc_scratch(shape, "cuda")
    tws = cg.alloc_tile_ws(shape, "cuda")
    packed = cg.pack_weights(w, gemm)
    planes = ('bf16',) + cg.bf16_planes(sbuf, Cin)
    cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"], tile_ws=tws)
    ntl = int(tws[1])
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    pargs = None
    if pool:                                               # conv -> 2x2 pool -> next layer's detection in the epilogue
        pv, _ = cg.pixel_major((B, Cout, H // 2, W // 2), torch.float32, "cuda", 0)
        nv, nbuf = cg.pixel_major((B, Cout, H // 2, W // 2), torch.float32, "cuda", 0)
        s2 = cg.alloc_scratch((B, H // 2, W // 2), "cuda")
        nh, nl = cg.bf16_planes(nbuf, Cout)
        pargs = dict(out=pv, next_state=nv, next_raw_bits=s2["raw_bits"], threshold=0.05, mode=_lib.UPDATE_CHANGED,
                     aux=('bf16', nh, nl))
    for _ in range(3):
        cg.conv_update_tiled(sbuf, tws, s["dil_bits"], packed, bias, obuf, Cin, Cout, (k, k), True, gemm, aux=planes,
                             pool=pargs)
    torch.cuda.synchronize()
    buf = (ctypes.c_longlong * (2048 * 32))()
    C.cb_debug_tile_trace(buf, 2048)                       # clear
    if cold:
        flush.zero_()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    cg.conv_update_tiled(sbuf, tws, s["dil_bits"], packed, bias, obuf, Cin, Cout, (k, k), True, gemm, aux=planes,
                         pool=pargs)
    e1.record()
    torch.cuda.synchronize()
    nev = C.cb_debug_tile_trace(buf, 2048)
    print("\n== %d->%d %dx%d k%d B%d %.0f%%%s: %d tiles, %s caches, kernel %.1f us (event pair, incl. launch)"
          % (Cin, Cout, H, W, k, B, rate * 100, " + fused pool/detect" if pool else "", ntl, "COLD" if cold else "warm",
             e0.elapsed_time(e1) * 1e3))
    rows = []
    for cta in range(2048):
        ev = [buf[cta * nev + i] for i in range(nev)]
        if ev[31] == 0:
            continue
        rows.append((cta, ev))
    gt0 = min(ev[31] for _, ev in rows)
    names = ["halo issued", "halo landed", "mmas issued", "acc complete", "epilogue done", "weights landed"]
    us = lambda c: c / MHZ
    print("CTAs that ran: %d; entry spread on the global timer: %.1f us" % (len(rows), (max(ev[31] for _, ev in rows) - gt0) / 1e3))
    # co-residency: CTAs of one SM (%smid) whose [entry, exit] intervals on the global timer overlap
    by_sm = {}
    for _, ev in rows:
        if ev[29] and ev[28]:
            by_sm.setdefault(ev[29] - 1, []).append((ev[31], ev[28]))
    peak = []
    for iv in by_sm.values():
        pts = sorted([(a, 1) for a, _ in iv] + [(b, -1) for _, b in iv])
        cur = best = 0
        for _, d in pts:
            cur += d
            best = max(best, cur)
        peak.append(best)
    if peak:
        print("SMs used: %d; CTAs per SM: %d..%d; peak CO-RESIDENT CTAs per SM (overlapping lifetimes): min %d  median %d  max %d"
              % (len(by_sm), min(len(v) for v in by_sm.values()), max(len(v) for v in by_sm.values()),
                 min(peak), sorted(peak)[len(peak) // 2], max(peak)))
    ends = sorted(us(ev[30]) for _, ev in rows if ev[30])
    print("CTA lifetime (entry -> all roles done): min %.1f  median %.1f  max %.1f us; prologue median %.2f us"
          % (ends[0], ends[len(ends) // 2], ends[-1], sorted(us(ev[0]) for _, ev in rows)[len(rows) // 2]))
    for cta, ev in rows[:2] + rows[len(rows) // 2: len(rows) // 2 + 2] + rows[-2:]:
        line = "cta %4d gt+%.1f  prologue %.2f |" % (cta, (ev[31] - gt0) / 1e3, us(ev[0]))
        for it in range(4):
            t = [ev[1 + it * 6 + j] for j in range(6)]
            if not any(t):
                break
            line += " tile%d: halo %.1f->%.1f  w %.1f  mma-issued %.1f  acc %.1f  epi-done %.1f |" % (
                it, us(t[0]), us(t[1]), us(t[5]), us(t[2]), us(t[3]), us(t[4]))
        line += " end %.1f" % us(ev[30])
        print(line)


for cold in ((False,) if "--quick" in sys.argv else (False, True)):
    for pool in ((False,) if "--quick" in sys.argv else (False, True)):
        run(8, 16, 64, 240, 320, 7, 0.05, cold, pool)
        run(8, 3, 16, 480, 640, 7, 0.05, cold, pool)
