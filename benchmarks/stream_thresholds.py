#!/usr/bin/env python
"""What per-stream thresholds cost and what they change (cbinfer_b200.setStreamThresholds), on bench.py's
workload (scene model, 8 streams of 640x480, 5 % block change, candidate path, one graph replay per step
from a ring of per-slot graphs):
  1. the step without a table against a table equal to the scalars, alternated, best of several runs;
  2. each threshold-taking kernel with and without a table, 50 launches in one graph: those of the step
     (dense detection, the tile contraction with the pool and the next detection in its epilogue, the
     fused tail) and the others (uint8 and candidate detection, detection + compaction, pool + detection);
  3. a heterogeneous table (streams at 0.5x / 1x / 2x / 4x the scalars): per-stream counts of every layer
     and the step time;
  4. a call that lowers one stream's values (which restarts that stream), plus the next step.
One JSON line; the GPU name and power limit are read in the same run."""
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
from cbinfer_b200 import models, video
from bench import SceneStep
from benchmarks.stream_counts import build, graph_us, timed
from benchmarks.stream_reset import gpu_identity


def convs(m):
    return [c for c in m.modules() if type(c) is cb.CBConv2d]


def scalars(m, B):
    return torch.tensor([[float(c.threshold)] * B for c in convs(m)], dtype=torch.float32)


def ring(base, frames, table=None, track=False):
    m = build(base, frames[0])
    B = frames[0].shape[0]
    if table is not None:
        cb.setStreamThresholds(m, table(m, B))
    if track:
        cb.trackStreamChanges(m, B=B)
    st = SceneStep(m, frames[0], frames[1])
    return [st, [st.capture_slot(f) for f in frames], 2]


def stepper(r, N):
    def step():
        period = 2 * (N - 1)
        k = r[2] % period
        r[1][k if k < N else period - k].replay()
        r[2] += 1
    return step


def kernels(model, B):
    """the threshold-taking kernels of the step on the model's own buffers after a frame, with and without
    a table (all launches leave the states alone: UPDATE_NONE, scratch bitmaps)"""
    cs = convs(model)
    table = scalars(model, B).cuda()
    out = {}
    first = cs[0]
    _, _, H, W = first.prevOutput.shape
    bits = torch.zeros(cb._lib.C.cb_bitmap_words(B, H, W), dtype=torch.int32, device="cuda")
    x = first.prevInput.clone()
    for thr_b, tag in ((None, "no_table"), (table[0], "table")):
        out.setdefault("detect", {})[tag] = graph_us(
            lambda: cg.detect(x, first.prevInput, bits, first.threshold, _lib.UPDATE_NONE, thr_b=thr_b))
    # candidate detection of layer 3 on the candidates layer 2 handed it (its last list), scratch bitmap
    l2, l3 = cs[1], cs[2]
    _, _, H3, W3 = l3.prevInput.shape
    bits3 = torch.zeros(cb._lib.C.cb_bitmap_words(B, H3, W3), dtype=torch.int32, device="cuda")
    cand = cg.ChangeIndexes.from_tensor(torch.nonzero(torch.ones(B * H3 * W3, device="cuda"))[::20, 0].int(),
                                        (B, H3, W3))
    x3 = l3.prevInput.clone()
    for thr_b, tag in ((None, "no_table"), (table[2], "table")):
        out.setdefault("detect_sparse", {})[tag] = graph_us(
            lambda: cg.detect_sparse(x3, l3.prevInput, bits3, l3.threshold, _lib.UPDATE_NONE, cand,
                                     bits_are_clear=True, thr_b=thr_b))
    # uint8 dense detection of L1 (the ingest path), on a uint8 copy of the frame it last saw
    x8 = first.prevInput.mul(255.0).round().clamp(0, 255).to(torch.uint8)
    for thr_b, tag in ((None, "no_table"), (table[0], "table")):
        out.setdefault("detect_u8", {})[tag] = graph_us(
            lambda: cg.detect_u8(x8, first.prevInput, bits, first.threshold, _lib.UPDATE_NONE, 255.0, 0.0,
                                 thr_b=thr_b))
    # candidate detection + compaction in one launch (small maps): L3 of as many streams as fit
    nb = max(1, min(B, _lib.C.cb_compact_small_max_words() // _lib.C.cb_bitmap_words(1, H3, W3)))
    sub = cg.ChangeIndexes.from_tensor(torch.nonzero(torch.ones(nb * H3 * W3, device="cuda"))[::20, 0].int(),
                                       (nb, H3, W3))
    sc = cg.alloc_scratch((nb, H3, W3), "cuda")
    sync = torch.zeros(1, dtype=torch.int32, device="cuda")
    x3s, st3s = x3[:nb], l3.prevInput[:nb]
    for thr_b, tag in ((None, "no_table"), (table[2][:nb], "table")):
        out.setdefault("detect_sparse_compact", {})[tag] = graph_us(
            lambda: cg.detect_sparse_compact(x3s, st3s, sc["raw_bits"], l3.threshold, _lib.UPDATE_NONE, sub,
                                             l3.kernel_size, sc["idx"], sc["count"], sync, dil_bits=sc["dil_bits"],
                                             thr_b=thr_b))
    # L1's conv with the pool and L2's detection in its epilogue, on L1's last dilated bitmap (the conv and
    # pooled maps are rewritten with the values they hold; the next layer's bits go to a scratch bitmap and
    # its state is left alone)
    s = first._scratch
    pool = first._fusedPool[0]
    gemm, packed, bias32 = first._weights(torch.float32, first.prevInput.device)
    oH, oW = l2.prevInput.shape[2:]
    nbits = torch.zeros(cb._lib.C.cb_bitmap_words(B, oH, oW), dtype=torch.int32, device="cuda")
    aux = first._aux(gemm)
    for thr_b, tag in ((None, "no_table"), (table[1], "table")):
        def tile():                               # (the tile list of the last frame: the kernel only reads it)
            cg.conv_update_tiled(first._inBuf, s["tile_ws"], s["dil_bits"], packed, bias32, first._outBuf,
                                 first.in_channels, first.out_channels, first.kernel_size, first.withReLU, gemm,
                                 aux=aux, pool=dict(out=pool.outputState, next_state=l2.prevInput,
                                                    next_raw_bits=nbits, threshold=l2.threshold,
                                                    mode=_lib.UPDATE_NONE, aux=None, thr_b=thr_b))
        out.setdefault("conv_tiled_pool", {})[tag] = graph_us(tile)
    # 2x2 pool + L2's detection (cb_maxpool2x2_detect) on L1's last dilated pixels
    ci = cg.ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])
    cg.dilate_compact(s["dil_bits"], (B, H, W), (1, 1), s["idx"], s["count"], s["ws"])
    pooled = pool.outputState.clone()
    for thr_b, tag in ((None, "no_table"), (table[1], "table")):
        out.setdefault("maxpool2x2_detect", {})[tag] = graph_us(
            lambda: cg.maxPool2d_detect(first.prevOutput, pooled, ci, l2.prevInput, nbits, l2.threshold,
                                        _lib.UPDATE_NONE, thr_b=thr_b))
    # the fused tail on the candidates layer 3 handed it last frame, without accepting anything
    l4, l5 = cs[3], cs[4]
    cand = l3._lastChanges
    _, p4, b4 = l4._weights(torch.float32, l4.prevInput.device)
    _, p5, b5 = l5._weights(torch.float32, l5.prevInput.device)
    sync = torch.zeros(4, dtype=torch.int32, device="cuda")
    c1, c2 = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    for rows, tag in (((None, None), "no_table"), ((table[3], table[4]), "table")):
        out.setdefault("tail", {})[tag] = graph_us(
            lambda: cg.tail_update(l3._outBuf, l4._inBuf, p4, b4, l4._outBuf, l4.withReLU, l4.threshold, l5._inBuf, p5,
                                   b5, l5._outBuf, l5.withReLU, l5.threshold, cand, l4.in_channels, l4.out_channels,
                                   l5.out_channels, _lib.UPDATE_NONE, c1, c2, sync, thr1_b=rows[0], thr2_b=rows[1]))
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
        raise SystemExit("stream_thresholds.py: no CUDA device (there is no CPU path)")
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, W = args.streams, args.height, args.width
    base = models.sceneLabelingBaseline().to(dev)
    frames = video.sequence(S, H, W, args.frames, args.rate, "block", seed=0, device=dev)
    N = len(frames)

    # ---- 1. no table against a table equal to the scalars ---------------------------------------------
    rings = {"no_table": ring(base, frames), "scalar_table": ring(base, frames, table=scalars)}
    runs = {k: [] for k in rings}
    for _ in range(args.runs):
        for k, r in rings.items():
            runs[k].append(round(timed(stepper(r, N), args.steps), 4))
    best = {k: min(v) for k, v in runs.items()}
    spread = {k: round(max(v) - min(v), 4) for k, v in runs.items()}

    # ---- 2. the kernels -------------------------------------------------------------------------------
    kern = kernels(rings["no_table"][0].model, S)
    del rings

    # ---- 3. heterogeneous table: per-stream counts and step time -------------------------------------
    factors = [(0.5, 1.0, 2.0, 4.0)[b % 4] for b in range(S)]

    def hetero(m, B):
        return scalars(m, B) * torch.tensor(factors, dtype=torch.float32)

    het = {}
    for name, table in (("scalar_table", scalars), ("heterogeneous", hetero)):
        r = ring(base, frames, table=table, track=True)
        step = stepper(r, N)
        ms = min(timed(step, args.steps) for _ in range(2))
        step()
        torch.cuda.synchronize()
        het[name] = {"step_ms_best": round(ms, 4),
                     "counts_last_step": cb.streamChangeCounts(r[0].model).cpu().tolist()}
        del r

    # ---- 4. lowering one stream: the call, then the next step ---------------------------------------
    r = ring(base, frames, table=scalars)
    m = r[0].model
    step = stepper(r, N)
    low = scalars(m, S)
    low[:, S - 1] *= 0.5
    high = scalars(m, S)
    timed(step, 20)
    call_ms, next_ms, plain_ms = [], [], []
    for i in range(10):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cb.setStreamThresholds(m, low if i % 2 == 0 else high)     # raising back resets nothing
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        step()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        step()
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if i % 2 == 0:
            call_ms.append((t1 - t0) * 1e3)
            next_ms.append((t2 - t1) * 1e3)
            plain_ms.append((t3 - t2) * 1e3)
    lower = {"call_ms_median": round(sorted(call_ms)[len(call_ms) // 2], 4),
             "next_step_ms_median": round(sorted(next_ms)[len(next_ms) // 2], 4),
             "step_after_ms_median": round(sorted(plain_ms)[len(plain_ms) // 2], 4),
             "note": "host clock around device-synchronised work; the call copies a host table"}
    del r, m

    name, power = gpu_identity(dev.index)
    print(json.dumps({
        "benchmark": "stream_thresholds", "gpu": name, "power_limit_w": power,
        "config": {"streams": S, "height": H, "width": W, "change_rate": args.rate, "change_mode": "block",
                   "model": "sceneLabeling CBinfer, experimentIdx 6, candidate path, thresholds 0.02 x range",
                   "frames": args.frames, "steps": args.steps, "runs": args.runs},
        "step_ms_best": best, "step_ms_runs": runs, "step_ms_spread": spread,
        "table_overhead_pct": round(100.0 * (best["scalar_table"] / best["no_table"] - 1.0), 2),
        "kernel_us": kern,
        "heterogeneous": dict(het, factors=factors),
        "lower_one_stream": lower,
    }))


if __name__ == "__main__":
    main()
