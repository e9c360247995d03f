#!/usr/bin/env python
"""One conv_update shape in isolation (default: scene L3 at 8 streams, ~5 % change): CUDA-event
timing over graph replays; small enough to wrap in ncu.  Env knob: CBINFER_STREAMK."""
import argparse, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cbinfer_b200 as cb
from cbinfer_b200 import conv2d_cg as cg, _lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="8,64,256,120,160,7")
    ap.add_argument("--n", type=int, default=13913)
    ap.add_argument("--dtype", default="f32")
    ap.add_argument("--gemm", default="bf16x3")
    ap.add_argument("--rep", type=int, default=20)
    ap.add_argument("--no-ws", action="store_true")
    a = ap.parse_args()
    B, Cin, Cout, H, W, k = [int(v) for v in a.shape.split(",")]
    dt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[a.dtype]
    gemm = cb.CBConv2d.GEMM_MODES[a.gemm]
    torch.manual_seed(0)
    state, sbuf = cg.pixel_major((B, Cin, H, W), dt, "cuda", 0)
    state.copy_(torch.rand(B, Cin, H, W).to(dt))
    out, obuf = cg.pixel_major((B, Cout, H, W), dt, "cuda", 0)
    w = (torch.randn(Cout, Cin, k, k) * (Cin * k * k) ** -0.5).to(dt).cuda()
    bias = torch.zeros(Cout, device="cuda")
    # clustered change set: whole rows blocks per image, n pixels in total
    per = a.n // B
    sel = torch.cat([torch.arange(per, dtype=torch.int32) + b * H * W + (H // 3) * W for b in range(B)]).cuda()
    ci = cg.ChangeIndexes.from_tensor(sel, (B, H, W))
    packed = cg.pack_weights(w, gemm)
    planes = ('bf16',) + cg.bf16_planes(sbuf, Cin) if gemm == _lib.GEMM_TC_BF16X3 else None
    ws = None if a.no_ws else torch.zeros(_lib.C.cb_conv_ws_bytes(), dtype=torch.uint8, device="cuda")

    def run():
        cg.conv_update(sbuf, ci, packed, bias, obuf, Cin, Cout, (k, k), True, gemm, aux=planes, ws=ws)

    for _ in range(3):
        run()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(a.rep):
            run()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / a.rep
    flops = 2.0 * sel.numel() * Cin * k * k * Cout
    print("shape %s n=%d %s/%s ws=%s SK=%s: %.2f us  %.1f TFLOP/s (algorithmic)" % (
        a.shape, sel.numel(), a.dtype, a.gemm, ws is not None,
        os.environ.get("CBINFER_STREAMK", "1"), us, flops / us * 1e-6))


if __name__ == "__main__":
    main()
