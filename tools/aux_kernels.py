#!/usr/bin/env python
"""Launch the small HBM-side kernels once or twice each at bench sizes (for `ncu --set full`):
detect_planar (C=64, 8x368x368, fp32 + bf16), fg_detect (C=16, 8x240x320), dilate_tiles / dilate_compact
(8x480x640, 5 % block), detect_sparse_vec + maxpool2x2_detect (scene layer-2 sizes)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cbinfer_b200 import _lib, conv2d_cg as cg

dev = "cuda"
torch.manual_seed(0)


def block_change(x, rate):
    B, C, H, W = x.shape
    bh, bw = int((rate * H * W * 3 / 4) ** 0.5), 0
    bw = int(rate * H * W / max(bh, 1))
    y = x.clone()
    y[:, :, 5:5 + bh, 7:7 + bw] = torch.rand(B, C, bh, bw, device=x.device).to(x.dtype)
    return y


for dt in (torch.float32, torch.bfloat16):
    B, C, H, W = 8, 64, 368, 368
    x0 = torch.rand(B, C, H, W, device=dev).to(dt)
    st, _ = cg.pixel_major((B, C, H, W), dt, dev, 0)
    st.copy_(x0)
    s = cg.alloc_scratch((B, H, W), dev)
    x1 = block_change(x0, 0.05)
    for _ in range(2):
        cg.detect(x1, st, s["raw_bits"], 0.1, _lib.UPDATE_CHANGED)          # detect_planar_kernel
    xp, _ = cg.pixel_major((B, C, H, W), dt, dev, 0)
    xp.copy_(x1)
    for _ in range(2):
        cg.detect(xp, st, s["raw_bits"], 0.1, _lib.UPDATE_CHANGED)          # detect_vec_kernel (pixel-major x)
    torch.cuda.synchronize()
    del x0, x1, xp, st

B, C, H, W = 8, 16, 240, 320
x0 = torch.rand(B, C, H, W, device=dev)
pv, pb = cg.pixel_major((B, C, H, W), torch.float32, dev, 0)
pv.copy_(x0)
p16 = _lib.C.cb_plane_pitch16(C)
hi = torch.zeros(B, H, W, p16, dtype=torch.bfloat16, device=dev)
lo = torch.zeros_like(hi)
s = cg.alloc_scratch((B, H, W), dev)
cnt = torch.zeros(1, dtype=torch.int32, device=dev)
for _ in range(2):
    cg.fg_detect(block_change(x0, 0.05), pv, pb, (hi, lo), s["raw_bits"], 0.1, count=cnt)   # fg_detect_kernel

shape = (8, 480, 640)
m = torch.zeros(shape, dtype=torch.int8, device=dev)
m[:, 100:207, 200:343] = 1
bits, _ = cg._map_to_bits(m)
s = cg.alloc_scratch(shape, dev)
tw = cg.alloc_tile_ws(shape, dev)
for _ in range(2):
    cg.dilate_tiles(bits, shape, (7, 7), s["count"], s["ws"], s["dil_bits"], tw)            # dilate_compact_kernel, tiles only
    cg.dilate_compact(bits, shape, (7, 7), s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"])  # dilate_compact_kernel

# scene layer 2 sizes: 8 x 16ch x 480x640 conv output -> pool -> 240x320 state; ~135k changed pixels
B, C, H, W = 8, 16, 480, 640
xv, _ = cg.pixel_major((B, C, H, W), torch.float32, dev, 0)
xv.copy_(torch.rand(B, C, H, W, device=dev))
ov, _ = cg.pixel_major((B, C, H // 2, W // 2), torch.float32, dev, 0)
nv, _ = cg.pixel_major((B, C, H // 2, W // 2), torch.float32, dev, 0)
ch = cg.ChangeIndexes(s["idx"], s["count"], shape, bits=s["dil_bits"])
s2 = cg.alloc_scratch((B, H // 2, W // 2), dev)
for _ in range(2):
    cg.maxPool2d_detect(xv, ov, ch, nv, s2["raw_bits"], 0.05, _lib.UPDATE_CHANGED)          # maxpool2x2_detect_kernel
    s2["raw_bits"].zero_()
    cg.pool_compact(s["dil_bits"], shape, (B, H // 2, W // 2), s2["idx"], s2["count"], s2["ws"], out_bits=s2["dil_bits"])
    cand = cg.ChangeIndexes(s2["idx"], s2["count"], (B, H // 2, W // 2), bits=s2["dil_bits"])
    cg.detect_sparse(ov, nv, s2["raw_bits"], 0.05, _lib.UPDATE_CHANGED, cand, bits_are_clear=True)  # detect_sparse_vec
    s2["raw_bits"].zero_()
torch.cuda.synchronize()
print("aux kernels done")
