#!/usr/bin/env python
"""detect_planar_kernel / fg_detect_kernel timing (CUDA events, L2 flushed between launches):
planar NCHW frame vs pixel-major state, C = 64 (8x368x368) and C = 16 (8x240x320), fp32 + bf16."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cbinfer_b200 import _lib, conv2d_cg as cg

dev = "cuda"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timeit(fn, n=10):
    ts = []
    for _ in range(n):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


for (B, C, H, W) in ((8, 64, 368, 368), (8, 16, 240, 320), (8, 512, 46, 46)):
    for dt in (torch.float32, torch.bfloat16):
        x0 = torch.rand(B, C, H, W, device=dev).to(dt)
        st, _ = cg.pixel_major((B, C, H, W), dt, dev, 0)
        st.copy_(x0)
        x1 = x0.clone()
        x1[:, :, 3:3 + H // 5, 5:5 + W // 4] += 1.0
        s = cg.alloc_scratch((B, H, W), dev)
        xp, _ = cg.pixel_major((B, C, H, W), dt, dev, 0)
        xp.copy_(x1)
        nbytes = 2 * x0.numel() * x0.element_size()
        t_pl = timeit(lambda: cg.detect(x1, st, s["raw_bits"], 0.5, _lib.UPDATE_NONE))
        t_pm = timeit(lambda: cg.detect(xp, st, s["raw_bits"], 0.5, _lib.UPDATE_NONE))
        print("C=%d %dx%d %s: planar x %.1f us (%.2f TB/s)   pixel-major x %.1f us (%.2f TB/s)" % (
            C, H, W, str(dt).split(".")[-1], t_pl, nbytes / t_pl / 1e6, t_pm, nbytes / t_pm / 1e6), flush=True)
