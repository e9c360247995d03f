#!/usr/bin/env python
"""Tiled vs index-list contraction on one layer shape with a block change set (default: the scene
net's L1 / L2 / L3 at 8 streams, 5 % block): CUDA-event timing over graph replays."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cbinfer_b200 as cb
from cbinfer_b200 import conv2d_cg as cg, _lib, video


def timed(fn, rep=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(rep):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (3 * rep)


def one(B, Cin, Cout, H, W, k, rate, mode, dt, kind="block"):
    gemm = cb.CBConv2d.GEMM_MODES[mode]
    torch.manual_seed(0)
    state, sbuf = cg.pixel_major((B, Cin, H, W), dt, "cuda", 0)
    state.copy_(torch.rand(B, Cin, H, W).to(dt))
    out, obuf = cg.pixel_major((B, Cout, H, W), dt, "cuda", 0)
    w = (torch.randn(Cout, Cin, k, k) * (Cin * k * k) ** -0.5).to(dt).cuda()
    bias = torch.zeros(Cout, device="cuda")
    f0 = video.base_frame(B, H, W)
    f1 = video.next_frame(f0, 1, rate, kind)
    raw = (f0 != f1).any(1).to(torch.int8).cuda()
    raw_bits, shape = cg._map_to_bits(raw)
    s = cg.alloc_scratch(shape, "cuda")
    tws = cg.alloc_tile_ws(shape, "cuda")
    packed = cg.pack_weights(w, gemm)
    planes = ('bf16',) + cg.bf16_planes(sbuf, Cin) if gemm == _lib.GEMM_TC_BF16X3 else None
    ws = torch.zeros(_lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")
    cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"], tile_ws=tws)
    ci = cg.ChangeIndexes(s["idx"], s["count"], shape, bits=s["dil_bits"])
    n, ntl = int(s["count"]), int(tws[1])
    t_dc = timed(lambda: cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"], tile_ws=tws))
    t_dc0 = timed(lambda: cg.dilate_compact(raw_bits, shape, (k, k), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"]))
    t_g = timed(lambda: cg.conv_update(sbuf, ci, packed, bias, obuf, Cin, Cout, (k, k), True, gemm, aux=planes, ws=ws))
    sup = cg.tiled_supported(dt, gemm, shape, Cin, Cout, (k, k))
    t_t = float("nan")
    if sup:
        t_t = timed(lambda: cg.conv_update_tiled(sbuf, tws, s["dil_bits"], packed, bias, obuf, Cin, Cout, (k, k), True, gemm, aux=planes))
    fl = 2.0 * n * Cin * k * k * Cout
    print("B%d %3d->%-3d %4dx%-4d k%d %s %.0f%% %s: n=%d tiles=%d (eff %.2f) | compact %.2f us (+tiles %.2f) | gather %.2f us | tiled %.2f us (%.1f TFLOP/s alg, sup=%d)"
          % (B, Cin, Cout, H, W, k, kind, rate * 100, mode, n, ntl, n / max(ntl * 128, 1), t_dc0, t_dc, t_g, t_t, fl / t_t * 1e-6, sup), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--set", default="scene")
    a = ap.parse_args()
    f32, bf = torch.float32, torch.bfloat16
    if a.set == "scene":
        for rate in (0.05, 0.2, 1.0):
            one(8, 3, 16, 480, 640, 7, rate, "bf16x3", f32)
            one(8, 16, 64, 240, 320, 7, rate, "bf16x3", f32)
            one(8, 64, 256, 120, 160, 7, rate, "bf16x3", f32)
        one(8, 3, 16, 480, 640, 7, 0.05, "tc3x", f32)
        one(8, 16, 64, 240, 320, 7, 0.05, "bf16x3", f32, kind="iid")
        one(1, 3, 16, 480, 640, 7, 0.05, "bf16x3", f32)
        one(1, 16, 64, 240, 320, 7, 0.05, "bf16x3", f32)
    elif a.set == "dense":
        for rate in (0.5, 1.0):
            one(8, 64, 256, 120, 160, 7, rate, "tc", bf)
            one(8, 64, 256, 120, 160, 7, rate, "bf16x3", f32)
            one(8, 64, 64, 368, 368, 3, rate, "tc", bf)
            one(8, 512, 512, 46, 46, 3, rate, "tc", bf)
            one(8, 128, 128, 46, 46, 7, rate, "tc", bf)
    elif a.set == "policy":
        # long-K layers the static policy keeps on the index-list kernel: where does the tile kernel win?
        for rate in (0.01, 0.05, 0.2, 1.0):
            one(8, 64, 256, 120, 160, 7, rate, "tc", bf)
            one(8, 128, 128, 46, 46, 7, rate, "tc", bf)
            one(8, 128, 128, 46, 46, 7, rate, "bf16x3", f32)
            one(1, 128, 128, 46, 46, 7, rate, "tc", bf)
    else:
        for rate in (0.05, 1.0):
            one(8, 64, 64, 368, 368, 3, rate, "tc", bf)
            one(8, 128, 128, 184, 184, 3, rate, "tc", bf)
            one(8, 256, 256, 92, 92, 3, rate, "tc", bf)
            one(8, 512, 512, 46, 46, 3, rate, "tc", bf)
            one(8, 128, 128, 46, 46, 7, rate, "tc", bf)
