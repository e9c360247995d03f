#!/usr/bin/env python
"""What starting a new sequence in some streams costs: bench.py's workload (scene model, 8 streams
of 640x480, 5 % block change, candidate path, one graph replay per step from a ring of per-slot
graphs) with cbinfer_b200.resetStreams against the status quo, clearMemory + a warm-up frame + a
graph recapture.  One JSON line; the GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import cbinfer_b200 as cb
from cbinfer_b200 import models, video
from bench import SceneStep


def gpu_identity(index):
    name = torch.cuda.get_device_name(index)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        power = float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        power = None
    return name, power


def median(v):
    s = sorted(v)
    return s[len(s) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--rate", type=float, default=0.05)
    ap.add_argument("--steps", type=int, default=400, help="steps of the steady-state timing")
    ap.add_argument("--reps", type=int, default=30, help="repetitions of each reset timing")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_reset.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, W = args.streams, args.height, args.width
    nframes = 48
    frames = [f.to(dev) for f in video.sequence(S, H, W, nframes, args.rate, "block", seed=0)]
    base = models.sceneLabelingBaseline().to(dev)
    model = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                        clonePoolOutput=False, candidateDetect=True)
    models.calibrateThresholds(base, model, frames[0], factor=0.02)
    step_obj = SceneStep(model, frames[0], frames[1])
    slots = [step_obj.capture_slot(f) for f in frames]

    def fidx(t):                                   # the video played forwards and backwards (bench.py)
        period = 2 * (nframes - 1)
        r = t % period
        return r if r < nframes else period - r

    t = 2

    def step():
        nonlocal t
        slots[fidx(t)].replay()
        t += 1

    def event_pair():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    for _ in range(20):
        step()
    torch.cuda.synchronize()

    # steady state: K steps between two events
    e0, e1 = event_pair()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    steady_ms = e0.elapsed_time(e1) / args.steps

    masks = {}
    for n in (1, S):
        m = torch.zeros(S, dtype=torch.uint8, device=dev)
        m[:n] = 1
        masks[n] = m

    def one_step_ms(reset_mask):
        """median over reps of one step (the reset launch included), each after 3 steady steps"""
        ms = []
        for _ in range(args.reps):
            for _ in range(3):
                step()
            a, b = event_pair()
            a.record()
            if reset_mask is not None:
                cb.resetStreams(model, reset_mask)
            step()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return median(ms)

    single_ms = one_step_ms(None)
    after_ms = {n: one_step_ms(masks[n]) for n in masks}

    # the reset kernel alone, over the segments resetStreams hands it: `reps` launches captured in one
    # graph, so the time is the kernel's and not that of the python calls building the segment array
    segments = [seg for layer in cb._cb_layers(model) for seg in layer._resetSegments()]
    kernel = {}
    reps = 50
    for n, m in masks.items():
        nbytes = n * sum(buf.shape[1] * buf.shape[2] * buf.stride(2) * buf.element_size() for buf, _, _ in segments)
        cb._cg.reset_streams(segments, m)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                cb._cg.reset_streams(segments, m)
        g.replay()
        a, b = event_pair()
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / reps
        kernel["streams_%d" % n] = {"us": round(us, 2), "bytes": nbytes, "gb_s": round(nbytes / us / 1e3, 1)}
        del g
    for _ in range(3):
        step()                                     # the state is +inf after the kernel loop: recompute once

    # status quo: clearMemory, one (dense) warm-up frame and a recapture of one slot graph (first-layer
    # detection on the slot + the rest of the model, as SceneStep.capture_slot); the graphs captured
    # before point at freed buffers afterwards, so this runs last
    del slots
    first = step_obj.first
    quo = []
    for r in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cb.clearMemory(model)
        with torch.no_grad():
            model(frames[fidx(t)])
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                model(first.detectInput(frames[fidx(t + 1)]))
        torch.cuda.synchronize()
        quo.append((time.perf_counter() - t0) * 1e3)
        del g
        t += 1
    name, power = gpu_identity(dev.index)
    print(json.dumps({
        "benchmark": "stream_reset", "gpu": name, "power_limit_w": power,
        "config": {"streams": S, "height": H, "width": W, "change_rate": args.rate, "change_mode": "block",
                   "model": "sceneLabeling CBinfer, experimentIdx 6, candidate path, thresholds 0.02 x range",
                   "steps": args.steps, "reps": args.reps, "reset_kernel_launches_timed": reps},
        "steady_step_ms": round(steady_ms, 4),
        "single_step_ms": round(single_ms, 4),
        "step_after_reset_1_stream_ms": round(after_ms[1], 4),
        "step_after_reset_%d_streams_ms" % S: round(after_ms[S], 4),
        "reset_kernel": kernel,
        "reset_segments": len(segments),
        "status_quo_clear_frame_recapture_ms": round(median(quo), 3),
    }))


if __name__ == "__main__":
    main()
