#!/usr/bin/env python
"""Steady-state latency of every kernel of one scene-model frame: the arguments of each C-ABI call
of a real frame are recorded, then each call is replayed REP times inside one CUDA graph and timed
with CUDA events (per-launch time incl. the dependent-launch gap, warm caches for small layers)."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cbinfer_b200 as cb
from cbinfer_b200 import models, video, conv2d_cg as cg

OPS = ("detect", "detect_sparse", "dilate_compact", "pool_compact", "conv_update", "maxPool2d",
       "maxPool2d_detect")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--rate", type=float, default=0.05)
    ap.add_argument("--dtype", default="f32")
    ap.add_argument("--gemm", default="auto")
    ap.add_argument("--rep", type=int, default=20)
    args = ap.parse_args()
    dt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[args.dtype]
    base = models.sceneLabelingBaseline().cuda().to(dt)
    model = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, clonePoolOutput=False,
                                        candidateDetect=True)
    for m in model.modules():
        if type(m) is cb.CBConv2d:
            m.gemmMode = args.gemm
    fr = [f.cuda().to(dt) for f in video.sequence(args.streams, args.height, args.width, 4, args.rate)]
    models.calibrateThresholds(base, model, fr[0], factor=0.02)
    with torch.no_grad():
        for f in fr[:3]:
            model(f)
    calls = []
    cur = {"layer": None}
    orig = {n: getattr(cg, n) for n in OPS}
    hooks = [m.register_forward_pre_hook(lambda mod, inp, n=n: cur.__setitem__("layer", n))
             for n, m in model.named_children()]
    for n in OPS:
        def w(*a, _n=n, **k):
            if _n == "dilate_compact":
                k = dict(k, clear_raw=False)   # keep the raw bitmap so the replays see the real input
            calls.append((cur["layer"], _n, a, k))
            return orig[_n](*a, **k)
        setattr(cg, n, w)
    with torch.no_grad():
        model(fr[3])
    for n in OPS:
        setattr(cg, n, orig[n])
    for h in hooks:
        h.remove()
    torch.cuda.synchronize()
    counts = {n: int(m._scratch["count"].item()) for n, m in model.named_children() if type(m) is cb.CBConv2d}
    total = 0.0
    rows = []
    # reverse order: a producer's repetitions (e.g. a second feedback detection finds no change)
    # must not wipe the inputs of its consumers before those are timed
    for layer, name, a, k in reversed(calls):
        k = dict(k)
        if name == "dilate_compact":
            k["clear_raw"] = False          # keep the input intact across repetitions
        if name == "detect_sparse":
            k["bits_are_clear"] = False
        fn = orig[name]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn(*a, **k)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(args.rep):
                fn(*a, **k)
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (5 * args.rep)
        total += us
        rows.append((layer, name, us))
        print("%-3s %-15s %8.2f us   n=%s" % (layer, name, us, counts.get(layer, "")), flush=True)
    print("sum %.1f us" % total)


if __name__ == "__main__":
    main()
