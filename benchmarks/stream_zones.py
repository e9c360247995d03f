#!/usr/bin/env python
"""What a watched-pixel zone saves and costs (cbinfer_b200.setStreamZones), on bench.py's workload (scene
model, 8 streams of 640x480, 5 % block change, candidate path, one graph replay per step from a ring of
per-slot graphs), with a synthetic overlay drawn here: a 200 x 24 box at a fixed position in every stream
(a burned-in timestamp), redrawn with new content on every frame.  Arms, alternated in one run, best of
several runs with their spread:
  (a) the block change alone;
  (b) block + overlay;
  (c) block + overlay, with a zone that excludes the box;
  (d) the overlay alone, without and with the zone.
Also per-layer change counts summed over the frame window per arm, the last layer's per-stream counts of
arm (d), and the first layer's detection with and without a zone (fp32 and uint8 frames), 50 launches in
one graph.  One JSON line; the GPU name and power limit are read in the same run."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cbinfer_b200 as cb
from cbinfer_b200 import _lib
from cbinfer_b200 import conv2d_cg as cg
from cbinfer_b200 import models, video
from bench import SceneStep
from benchmarks.stream_counts import build, graph_us, timed
from benchmarks.stream_reset import gpu_identity
from benchmarks.stream_thresholds import stepper

BOX = (16, 420, 24, 200)            # y0, x0, height, width of the overlay (scaled to the frame if smaller)


def box_of(H, W):
    y0, x0, h, w = BOX
    return min(y0, H - 1), min(x0, max(0, W - w)), min(h, H), min(w, W)


def with_overlay(frames, seed=7):
    """every frame with the box redrawn (new content every frame, every stream)"""
    B, C, H, W = frames[0].shape
    y0, x0, h, w = box_of(H, W)
    g = torch.Generator().manual_seed(seed)
    out = []
    for f in frames:
        f = f.clone()
        f[:, :, y0:y0 + h, x0:x0 + w] = torch.rand(B, C, h, w, generator=g).to(f.device, f.dtype)
        out.append(f)
    return out


def zone_of(B, H, W):
    y0, x0, h, w = box_of(H, W)
    z = torch.ones(B, H, W, dtype=torch.bool)
    z[:, y0:y0 + h, x0:x0 + w] = False
    return z


def ring(base, frames, zone=None, track=False):
    m = build(base, frames[0])
    B = frames[0].shape[0]
    if zone is not None:
        cb.setStreamZones(m, zone)
    if track:
        cb.trackStreamChanges(m, B=B)
    st = SceneStep(m, frames[0], frames[1])
    return [st, [st.capture_slot(f) for f in frames], 2]


def counts(base, frames, zone):
    """per-layer counts (summed over streams) summed over one pass of the window, and the last layer's
    per-stream counts summed likewise"""
    r = ring(base, frames, zone, track=True)
    N = len(frames)
    step = stepper(r, N)
    tot = None
    for _ in range(N - 1):
        step()
        c = cb.streamChangeCounts(r[0].model).long()
        tot = c.clone() if tot is None else tot + c
    torch.cuda.synchronize()
    return {"per_layer": tot.sum(1).tolist(), "last_layer_per_stream": tot[-1].tolist()}


def kernels(model, frame, zone):
    """the first layer's dense detection on the model's own state, without and with the zone (and with an
    all-watched zone), fp32 and uint8 frames; UPDATE_NONE leaves the state alone"""
    first = [c for c in model.modules() if type(c) is cb.CBConv2d][0]
    B, _, H, W = frame.shape
    bits = torch.zeros(_lib.C.cb_bitmap_words(B, H, W), dtype=torch.int32, device="cuda")
    zb, _ = cg._map_to_bits(zone.to(torch.int8).cuda())
    allw, _ = cg._map_to_bits(torch.ones(B, H, W, dtype=torch.int8, device="cuda"))
    x8 = frame.mul(255.0).round().clamp(0, 255).to(torch.uint8)
    out = {}
    for z, tag in ((None, "no_zone"), (allw, "zone_all_watched"), (zb, "zone_box_excluded")):
        out.setdefault("detect_f32", {})[tag] = graph_us(
            lambda: cg.detect(frame, first.prevInput, bits, first.threshold, _lib.UPDATE_NONE, zone=z))
        out.setdefault("detect_u8", {})[tag] = graph_us(
            lambda: cg.detect_u8(x8, first.prevInput, bits, first.threshold, _lib.UPDATE_NONE, 255.0, 0.0, zone=z))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--rate", type=float, default=0.05)
    ap.add_argument("--frames", type=int, default=24, help="frame window, played forwards and backwards")
    ap.add_argument("--steps", type=int, default=400, help="timed steps per graph-replay measurement")
    ap.add_argument("--runs", type=int, default=4, help="alternated runs per arm (best of)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_zones.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, W = args.streams, args.height, args.width
    base = models.sceneLabelingBaseline().to(dev)
    block = video.sequence(S, H, W, args.frames, args.rate, "block", seed=0, device=dev)
    still = [block[0]] * args.frames
    zone = zone_of(S, H, W)
    arms = {"a_block": (block, None), "b_block_overlay": (with_overlay(block), None),
            "c_block_overlay_zone": (with_overlay(block), zone), "d_overlay": (with_overlay(still), None),
            "d_overlay_zone": (with_overlay(still), zone)}
    N = args.frames

    rings = {k: ring(base, fr, z) for k, (fr, z) in arms.items()}
    runs = {k: [] for k in rings}
    for _ in range(args.runs):
        for k, r in rings.items():
            runs[k].append(round(timed(stepper(r, N), args.steps), 4))
    best = {k: min(v) for k, v in runs.items()}
    spread = {k: round(max(v) - min(v), 4) for k, v in runs.items()}
    kern = kernels(rings["a_block"][0].model, block[1], zone)
    del rings

    cnt = {k: counts(base, fr, z) for k, (fr, z) in arms.items()}

    name, power = gpu_identity(dev.index)
    print(json.dumps({
        "benchmark": "stream_zones", "gpu": name, "power_limit_w": power,
        "config": {"streams": S, "height": H, "width": W, "change_rate": args.rate, "change_mode": "block",
                   "overlay_box_yxhw": list(box_of(H, W)),
                   "model": "sceneLabeling CBinfer, experimentIdx 6, candidate path, thresholds 0.02 x range",
                   "frames": args.frames, "steps": args.steps, "runs": args.runs},
        "step_ms_best": best, "step_ms_runs": runs, "step_ms_spread": spread,
        "counts_window_sum": {k: v["per_layer"] for k, v in cnt.items()},
        "last_layer_per_stream_d": {k: cnt[k]["last_layer_per_stream"] for k in ("d_overlay", "d_overlay_zone")},
        "kernel_us": kern,
    }))


if __name__ == "__main__":
    main()
