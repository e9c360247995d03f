#!/usr/bin/env python
"""What skipping the streams without a new frame saves: bench.py's workload (scene model, 8 streams of
640x480, 5 % block change, candidate path, one graph replay per step from a ring of per-slot graphs)
with k of the streams active through cbinfer_b200.setActiveStreams, against the status quo in which
the other streams are fed their previous frame again.  Also the first layer's detection kernel with
and without the mask, and the uint8 host-fed FramePipeline with partial uploads against full ones.
One JSON line; the GPU name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cbinfer_b200 as cb
from cbinfer_b200 import conv2d_cg as cg
from cbinfer_b200 import models, runtime, video
from bench import SceneStep
from benchmarks.stream_reset import gpu_identity


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--rate", type=float, default=0.05)
    ap.add_argument("--frames", type=int, default=24, help="frame window, played forwards and backwards")
    ap.add_argument("--steps", type=int, default=400, help="timed steps per graph-replay measurement")
    ap.add_argument("--pipe-steps", type=int, default=200, help="timed steps per FramePipeline measurement")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("active_streams.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, W, N = args.streams, args.height, args.width, args.frames
    ks = [k for k in (8, 6, 4, 2, 1) if k <= S]
    frames = [f.to(dev) for f in video.sequence(S, H, W, N, args.rate, "block", seed=0)]
    base = models.sceneLabelingBaseline().to(dev)

    def build():
        m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                        clonePoolOutput=False, candidateDetect=True)
        models.calibrateThresholds(base, m, frames[0], factor=0.02)
        return m

    def fidx(t):
        period = 2 * (N - 1)
        r = t % period
        return r if r < N else period - r

    def fill_slots(slots, k, src):
        """streams < k see the video, the others keep frame 0 (a re-fed, unchanged frame)"""
        for i, s in enumerate(slots):
            s[:k].copy_(src[i][:k])
            s[k:].copy_(src[0][k:])

    def timed(fn, steps):
        for _ in range(20):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    # ---- one graph replay per step: masked model vs re-feed model, over the same slot buffers ---------
    slots = [f.clone() for f in frames]
    masked, refeed = build(), build()
    cb.setActiveStreams(masked, torch.ones(S, dtype=torch.uint8, device=dev))
    rings = {}
    for name, m in (("masked", masked), ("refeed", refeed)):
        st = SceneStep(m, frames[0], frames[1])
        rings[name] = (st, [st.capture_slot(s) for s in slots])
    t = [2]

    def step(name):
        rings[name][1][fidx(t[0])].replay()
        t[0] += 1

    step_ms = {}
    for k in ks:
        fill_slots(slots, k, frames)
        cb.setActiveStreams(masked, list(range(k)))
        for name in ("refeed", "masked", "refeed", "masked"):      # alternated, best of two
            ms = timed(lambda: step(name), args.steps)
            key = "k%d" % k
            step_ms.setdefault(key, {}).setdefault(name, []).append(ms)
    step_ms = {k: {n: round(min(v), 4) for n, v in d.items()} for k, d in step_ms.items()}

    # ---- the first layer's detection kernel alone: 50 launches in one graph, with and without a mask ----
    first = rings["masked"][0].first
    s = first._scratch
    mode = cb._lib.UPDATE_CHANGED if first.feedbackLoop else cb._lib.UPDATE_ALL
    aux = first._auxPlanes
    kernel_us = {}
    reps = 50
    for k in [None] + ks:
        mask = None
        if k is not None:
            mask = torch.zeros(S, dtype=torch.uint8, device=dev)
            mask[:k] = 1
        cg.detect(slots[1], first.prevInput, s["raw_bits"], first.threshold, mode, aux=aux, active=mask)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                cg.detect(slots[1], first.prevInput, s["raw_bits"], first.threshold, mode, aux=aux, active=mask)
        best = None
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / reps
            best = us if best is None else min(best, us)
        kernel_us["no_mask" if k is None else "k%d" % k] = round(best, 2)
        del g
    del rings, masked, refeed

    # ---- uint8 host-fed FramePipeline: partial uploads vs the full upload of re-fed frames ------------
    host = [f.mul(255.0).round().to(torch.uint8).pin_memory() for f in (x.cpu() for x in frames)]
    ring = [h.clone().pin_memory() for h in host]
    slice_bytes = host[0][0].numel()

    def pipe_rate(pipe, frames_host, active):
        for i in range(1, 11):
            pipe.submit(frames_host[fidx(i)], active=active)
        pipe.drain()
        t0 = time.perf_counter()
        last = None
        for i in range(11, 11 + args.pipe_steps):
            last = pipe.submit(frames_host[fidx(i)], active=active)
        pipe.wait(last)
        pipe.drain()
        return args.pipe_steps / (time.perf_counter() - t0)

    pipe_res = {}
    for k in ks:
        for i in range(N):
            ring[i][:k].copy_(host[i][:k])
            ring[i][k:].copy_(host[0][k:])
        row = {}
        for name in ("full_upload", "partial_upload"):
            m = build()
            [c for c in m.modules() if type(c) is cb.CBConv2d][0].inputNorm = (255.0, 0.0)
            partial = name == "partial_upload"
            pipe = runtime.FramePipeline(m, ring[0].to(dev), depth=2, activeStreams=partial)
            rate = pipe_rate(pipe, ring, list(range(k)) if partial else None)
            row[name] = {"steps_s": round(rate, 1), "h2d_bytes_per_step": (k if partial else S) * slice_bytes}
            del pipe, m
        pipe_res["k%d" % k] = row

    name, power = gpu_identity(dev.index)
    print(json.dumps({
        "benchmark": "active_streams", "gpu": name, "power_limit_w": power,
        "config": {"streams": S, "height": H, "width": W, "change_rate": args.rate, "change_mode": "block",
                   "model": "sceneLabeling CBinfer, experimentIdx 6, candidate path, thresholds 0.02 x range",
                   "frames": N, "steps": args.steps, "pipe_steps": args.pipe_steps,
                   "status_quo": "inactive streams re-fed their previous frame (unchanged), no mask"},
        "step_ms": step_ms,
        "first_layer_detect_us": kernel_us,
        "pipeline_u8": pipe_res,
    }))


if __name__ == "__main__":
    main()
