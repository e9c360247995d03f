#!/usr/bin/env python
"""What per-stream change counts cost (cbinfer_b200.trackStreamChanges): bench.py's workload (scene model,
8 streams of 640x480, 5 % block change, candidate path, one graph replay per step from a ring of per-slot
graphs), tracked against untracked, alternated, best of several runs; each kernel that gains a counting
variant (dilate_tiles, dilate_compact, the fused tail), 50 launches in one graph, with and without
counting; the uint8 host-fed FramePipeline with and without trackChanges; and the same step at 64
streams of 1080p.  One JSON line; the GPU name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cbinfer_b200 as cb
from cbinfer_b200 import _lib
from cbinfer_b200 import conv2d_cg as cg
from cbinfer_b200 import models, runtime, video
from bench import SceneStep
from benchmarks.stream_reset import gpu_identity


def build(base, frame0):
    m = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                    clonePoolOutput=False, candidateDetect=True)
    models.calibrateThresholds(base, m, frame0, factor=0.02)
    return m


def timed(fn, steps, warm=20):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def step_pair(base, frames, steps, runs):
    """ms per step of the graph ring, untracked and tracked models over the same slot buffers, alternated"""
    N = len(frames)
    rings = {}
    for name in ("untracked", "tracked"):
        m = build(base, frames[0])
        if name == "tracked":
            cb.trackStreamChanges(m, B=frames[0].shape[0])
        st = SceneStep(m, frames[0], frames[1])
        rings[name] = [st, [st.capture_slot(f) for f in frames], 2]

    def step(name):
        r = rings[name]
        period = 2 * (N - 1)
        k = r[2] % period
        r[1][k if k < N else period - k].replay()
        r[2] += 1

    res = {"untracked": [], "tracked": []}
    for _ in range(runs):
        for name in ("untracked", "tracked"):
            res[name].append(timed(lambda: step(name), steps))
    return {n: round(min(v), 4) for n, v in res.items()}, {n: [round(x, 4) for x in v] for n, v in res.items()}, rings


def graph_us(fn, reps=50, tries=5):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    best = None
    for _ in range(tries):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        best = us if best is None else min(best, us)
    return round(best, 2)


def kernels(model, B):
    """the counting kernels on the model's own buffers after a frame, with and without a counts row"""
    convs = [c for c in model.modules() if type(c) is cb.CBConv2d]
    first = convs[0]
    s = first._scratch
    _, _, H, W = first.prevOutput.shape
    shape, k = (B, H, W), first.kernel_size
    tw = cg.alloc_tile_ws(shape, s["raw_bits"].device)
    row = (torch.zeros(B, dtype=torch.int32, device="cuda"), torch.zeros(B + 1, dtype=torch.int32, device="cuda"))
    out = {}
    for streams, tag in ((None, "untracked"), (row, "tracked")):
        out.setdefault("dilate_tiles", {})[tag] = graph_us(
            lambda: cg.dilate_tiles(s["raw_bits"], shape, k, s["count"], s["ws"], s["dil_bits"], tw, streams=streams))
        out.setdefault("dilate_compact", {})[tag] = graph_us(
            lambda: cg.dilate_compact(s["raw_bits"], shape, k, s["idx"], s["count"], s["ws"], dil_bits=s["dil_bits"],
                                      streams=streams))
    # the fused tail on the candidates layer 3 handed it last frame, without accepting anything into the
    # states (UPDATE_NONE), so that every launch does the same work
    l3, l4, l5 = convs[2], convs[3], convs[4]
    cand = l3._lastChanges
    _, p4, b4 = l4._weights(torch.float32, l4.prevInput.device)
    _, p5, b5 = l5._weights(torch.float32, l5.prevInput.device)
    sync = torch.zeros(4, dtype=torch.int32, device="cuda")
    c1, c2 = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    row2 = (torch.zeros(B, dtype=torch.int32, device="cuda"), torch.zeros(B + 1, dtype=torch.int32, device="cuda"))
    x_buf = l3._outBuf
    for rows, tag in (((None, None), "untracked"), ((row, row2), "tracked")):
        out.setdefault("tail", {})[tag] = graph_us(
            lambda: cg.tail_update(x_buf, l4._inBuf, p4, b4, l4._outBuf, l4.withReLU, l4.threshold, l5._inBuf, p5, b5,
                                   l5._outBuf, l5.withReLU, l5.threshold, cand, l4.in_channels, l4.out_channels,
                                   l5.out_channels, _lib.UPDATE_NONE, c1, c2, sync, streams1=rows[0], streams2=rows[1]))
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
    ap.add_argument("--pipe-steps", type=int, default=200, help="timed steps per FramePipeline measurement")
    ap.add_argument("--big-streams", type=int, default=64, help="streams of the 1080p leg (0 skips it)")
    ap.add_argument("--big-frames", type=int, default=6)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_counts.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, W = args.streams, args.height, args.width
    base = models.sceneLabelingBaseline().to(dev)
    frames = video.sequence(S, H, W, args.frames, args.rate, "block", seed=0, device=dev)

    best, runs, rings = step_pair(base, frames, args.steps, args.runs)
    kern = kernels(rings["tracked"][0].model, S)
    del rings

    # ---- uint8 host-fed FramePipeline, with and without trackChanges --------------------------------
    host = [f.mul(255.0).round().to(torch.uint8).cpu().pin_memory() for f in frames]
    N = len(host)

    def pipe_rate(pipe):
        period = 2 * (N - 1)
        idx = [(i % period if i % period < N else period - i % period) for i in range(11 + args.pipe_steps)]
        for i in range(1, 11):
            pipe.submit(host[idx[i]])
        pipe.drain()
        t0 = time.perf_counter()
        last = None
        for i in range(11, 11 + args.pipe_steps):
            last = pipe.submit(host[idx[i]])
        pipe.wait(last)
        pipe.drain()
        return args.pipe_steps / (time.perf_counter() - t0)

    pipe_res = {}
    for _ in range(2):
        for tag in ("untracked", "tracked"):
            m = build(base, frames[0])
            [c for c in m.modules() if type(c) is cb.CBConv2d][0].inputNorm = (255.0, 0.0)
            pipe = runtime.FramePipeline(m, host[0].to(dev), depth=2, trackChanges=tag == "tracked")
            pipe_res.setdefault(tag, []).append(round(pipe_rate(pipe), 1))
            del pipe, m
    del frames

    # ---- 64 streams of 1080p (BASELINE configs[4] on one GPU) --------------------------------------------
    big = None
    if args.big_streams:
        torch.cuda.empty_cache()
        bf = video.sequence(args.big_streams, 1080, 1920, args.big_frames, args.rate, "block", seed=0, device=dev)
        b_best, b_runs, _ = step_pair(base, bf, max(args.steps // 8, 20), args.runs)
        big = {"streams": args.big_streams, "frames": args.big_frames, "step_ms_best": b_best, "step_ms_runs": b_runs}
        del bf

    name, power = gpu_identity(dev.index)
    print(json.dumps({
        "benchmark": "stream_counts", "gpu": name, "power_limit_w": power,
        "config": {"streams": S, "height": H, "width": W, "change_rate": args.rate, "change_mode": "block",
                   "model": "sceneLabeling CBinfer, experimentIdx 6, candidate path, thresholds 0.02 x range",
                   "frames": args.frames, "steps": args.steps, "runs": args.runs, "pipe_steps": args.pipe_steps},
        "step_ms_best": best, "step_ms_runs": runs,
        "tracked_overhead_pct": round(100.0 * (best["tracked"] / best["untracked"] - 1.0), 2),
        "kernel_us": kern,
        "pipeline_u8_steps_s": pipe_res,
        "streams1080p": big,
    }))


if __name__ == "__main__":
    main()
