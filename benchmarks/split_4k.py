#!/usr/bin/env python
"""BASELINE config 5 (second half): one 3840x2160 stream split in G row bands over G GPUs with a
one-off 24-row input halo exchange (NCCL send/recv) and an all_gather of the output bands.
Launch: torchrun --nproc-per-node G benchmarks/split_4k.py     (G=1 works too: the full frame).
Rank 0 prints one JSON line; with --check the gathered result is compared with the full-frame CB
model run on rank 0."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
import cbinfer_b200 as cb
from cbinfer_b200 import models, video, spatial, streams
from cbinfer_b200.runtime import FrameGraph


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--rate", type=float, default=0.05)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the gathered output of the last timed frame to DIR/output.npy (float32, rank 0)")
    args = ap.parse_args()
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", 1), ("RANK", 0), ("LOCAL_RANK", 0)))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    H, W = args.height, args.width
    base = models.sceneLabelingBaseline().to(dev)
    frames = [f.to(dev) for f in video.sequence(1, H, W, args.frames, args.rate)]   # same on all ranks
    model = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, clonePoolOutput=False,
                                        candidateDetect=True)
    models.calibrateThresholds(base, model, frames[0][:, :, :480, :640].contiguous(), factor=0.02)
    sp = spatial.SpatialSplit(model, H, world, rank, halo=24, stride=4)
    lo, hi = sp.band
    bands = [f[:, :, lo:hi].contiguous() for f in frames]
    # warm-up: two frames eagerly, then the model part of every later frame is one graph replay
    with torch.no_grad():
        slab = sp.exchange_halo(bands[0])
        sp.forward_slab(slab)
        slab.copy_(sp.exchange_halo(bands[1]))
        sp.forward_slab(slab)
    g = FrameGraph(model, slab)
    o0 = (lo - sp.slab[0]) // 4
    ms, out = [], None
    for t in range(2, args.frames):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        slab.copy_(sp.exchange_halo(bands[t]))
        y = g.replay()
        out = sp.gather(y[:, :, o0:o0 + (hi - lo) // 4])
        b.record()
        torch.cuda.synchronize()
        ms.append(streams.max_over_ranks(a.elapsed_time(b), dev))
    ms = sorted(ms[2:])
    res = {"workload": "%dx%d scene CBinfer, %d row bands, 24-row input halo" % (W, H, world),
           "n_gpus": world, "band_rows": hi - lo, "slab_rows": sp.slab[1] - sp.slab[0],
           "ms_per_frame_median": round(ms[len(ms) // 2], 3), "frames_per_s": round(1000.0 / ms[len(ms) // 2], 1)}
    if args.dump_outputs and rank == 0:
        from bench import DUMP_BYTES, dump_outputs
        dump_outputs(args.dump_outputs, out, "output", DUMP_BYTES)
    if args.check and rank == 0:
        full = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.02, clonePoolOutput=False,
                                           candidateDetect=True)
        for c, c2 in zip([m for m in full.modules() if type(m) is cb.CBConv2d],
                         [m for m in model.modules() if type(m) is cb.CBConv2d]):
            c.threshold = c2.threshold
        with torch.no_grad():
            for f in frames:
                ref = full(f)
        res["max_abs_diff_vs_full_frame"] = float((out - ref).abs().max())
        res["ref_max_abs"] = float(ref.abs().max())
    if rank == 0:
        print(json.dumps(res))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
