#!/usr/bin/env python
"""In-step kernel times of the bench workload: one CUDA graph per frame slot as in bench.py, with
EXTERNAL timing events recorded as graph nodes before and after every C-ABI call, so every kernel is
timed in the cache state and on the inputs it really sees inside a step (the back-to-back replays of
bench.py's kernel table run warm; ncu runs cold and serialised).  The event nodes cost a little
themselves: the instrumented step is printed next to the plain one."""
import argparse, os, sys, types
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench as B
import cbinfer_b200 as cb
from cbinfer_b200 import models, video, conv2d_cg as cg

ap = argparse.ArgumentParser()
ap.add_argument("--streams", type=int, default=8)
ap.add_argument("--rate", type=float, default=0.05)
ap.add_argument("--frames", type=int, default=8)
ap.add_argument("--reps", type=int, default=30)
a = ap.parse_args()
dev = torch.device("cuda", 0)
S, H, W = a.streams, 480, 640
base = models.sceneLabelingBaseline().to(dev)
frames = [f.to(dev) for f in video.sequence(S, H, W, a.frames, a.rate, "block", seed=0)]
args = types.SimpleNamespace(gemm="auto", dense_scan=False, threshold_factor=0.02)
model, _ = B.build_model(args, base, frames[0])
so = B.SceneStep(model, frames[0], frames[1])
plain = [so.capture_slot(f) for f in frames]

names = ("detect", "detect_u8", "detect_sparse", "dilate_compact", "dilate_tiles", "pool_compact", "conv_update",
         "conv_update_tiled", "tail_update", "maxPool2d", "maxPool2d_detect")
orig = {n: getattr(cg, n) for n in names}
log = None


def wrap(name):
    fn = orig[name]

    def w(*x, **k):
        e0 = torch.cuda.Event(enable_timing=True, external=True)
        e1 = torch.cuda.Event(enable_timing=True, external=True)
        e0.record()
        r = fn(*x, **k)
        e1.record()
        log.append((name, e0, e1))
        return r
    return w


inst = []
for n in names:
    setattr(cg, n, wrap(n))
try:
    for f in frames:
        log = []
        inst.append((so.capture_slot(f), log))
finally:
    for n, f in orig.items():
        setattr(cg, n, f)

nf = len(frames)
period = 2 * (nf - 1)


def fidx(t):
    r = t % period
    return r if r < nf else period - r


def run(graphs, reps):
    t = 2
    for _ in range(20):
        graphs[fidx(t)].replay(); t += 1
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps * period):
        graphs[fidx(t)].replay(); t += 1
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * period)


print("plain step        %.1f us" % run(plain, a.reps))
print("instrumented step %.1f us" % run([g for g, _ in inst], a.reps))
# per-kernel times: replay each slot's instrumented graph in ring order, read its events after each replay
acc = {}
t = 2
for rep in range(a.reps * period):
    g, lg = inst[fidx(t)]
    g.replay()
    torch.cuda.synchronize()
    prev_end = None
    for i, (name, e0, e1) in enumerate(lg):
        d = e0.elapsed_time(e1) * 1e3
        gap = prev_end.elapsed_time(e0) * 1e3 if prev_end is not None else 0.0
        acc.setdefault((i, name), []).append((d, gap))
        prev_end = e1
    t += 1
tot = 0.0
for (i, name), v in sorted(acc.items()):
    ds = sorted(x[0] for x in v)
    gs = sorted(x[1] for x in v)
    med, gmed = ds[len(ds) // 2], gs[len(gs) // 2]
    tot += med + gmed
    print("%d %-20s %7.2f us  (min %.2f max %.2f)   gap before %5.2f us" % (i, name, med, ds[0], ds[-1], gmed))
print("sum of medians (kernels + gaps) %.1f us" % tot)
