#!/usr/bin/env python
"""bench.py -- frames/s of the CBinfer change-based conv/pool path on B200 (BASELINE.json metric).

Workload (config.workload): BASELINE.json configs[1] -- the scene-labeling CBinfer model (all five
convs + both max-pools converted, feedback loop, fp32) on synthetic 640x480 video with 5 % block
change per frame, `streams_per_gpu` independent video streams batched per GPU.  `--workload
streams1080p` = configs[4] (64 x 1080p streams in total, sharded 64/N per GPU, strong scaling),
`--workload split4k` = one 3840x2160 stream in N row bands; `--rate` sets the change rate.

A "step" is one frame of every resident stream through the whole model: the first layer's change
detection is launched on the frame where it lies in HBM, the other launches replay as one CUDA graph.
  value : frames/s with the frames already resident in HBM: exactly K = --steps steps after
          max(W, 3) warm-up steps (W = --warmup), bracketed by barrier + synchronize and device-timed
          (max over ranks)
  e2e   : frames/s through the public module call with HOST (pinned) frames: per step one H2D copy
          of the step's frames and one D2H read of the step's logits inside the timed region (K steps)
  e2e_u8_ingest : the same with uint8 host frames, normalised inside the detection kernel
  parity_max_rel: the benchmarked configuration against the reference flow (unmodified reference
          CUDA kernels of oracle/_ref + fp32 torch.matmul, tests/ref_flow.py), outside the timed region
  roofline      : dominant kernel vs its HBM / tensor roofline (per-kernel CUDA-event timing)
  cpu_baseline  : the reference's dense PyTorch CPU inference path on this box's host cores
`--impl reference` times that CPU path alone on the same config; it never imports the product.

Launch: python bench.py --gpus N --steps K --warmup W      (N>1: via torch.distributed.run)

`--dump-outputs DIR` writes what the timed path returned in its last timed step -- the logits
[streams, 8, H/4, W/4] -- as DIR/output.npy (float32; DIR/output_rank<r>.npy per rank when N > 1;
split4k: the stitched [1, 8, H/4, W/4] of its last timed frame, written by rank 0).
The model, the video and the thresholds are seeded, so the same arguments give the same inputs and
two builds can be compared output for output.  Above 64 MB in all the file holds a fixed sample: every
s-th element of the flattened logits, s the smallest stride that fits.
"""
import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)


WORKLOADS = {
    # name: (height, width, streams per GPU at N GPUs, scaling)
    "scene640": dict(h=480, w=640, streams=lambda n: 8, scaling="weak",
                     note="BASELINE configs[1]: 8 independent 640x480 streams per GPU"),
    "streams1080p": dict(h=1080, w=1920, streams=lambda n: max(1, 64 // n), scaling="strong",
                         note="BASELINE configs[4]: 64 independent 1080p streams in total, sharded 64/N per GPU"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="scene640", choices=list(WORKLOADS) + ["split4k"],
                    help="scene640 (default, BASELINE configs[1]); streams1080p = 64 x 1080p streams sharded "
                         "64/N per GPU (strong scaling); split4k = one 3840x2160 stream in N row bands "
                         "(delegates to benchmarks/split_4k.py)")
    ap.add_argument("--streams", type=int, default=0, help="video streams per GPU (0 = the workload's own)")
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--rate", type=float, default=0.05, help="fraction of pixels changed per frame")
    ap.add_argument("--mode", default="block", choices=["block", "iid"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "bf16", "f16"])
    ap.add_argument("--gemm", default="auto", choices=["auto", "simt", "tc", "tc3x", "bf16x3"])
    ap.add_argument("--threshold-factor", type=float, default=0.02)
    ap.add_argument("--dense-scan", action="store_true",
                    help="re-scan every layer's whole input like the reference (default: candidate detection)")
    ap.add_argument("--eager-detect", action="store_true",
                    help="first-layer detection launched eagerly per frame + one graph for the rest (default: one "
                         "graph per input slot of the frame ring, detection included)")
    ap.add_argument("--profile", type=int, default=0, metavar="N",
                    help="profiling aid: after the warm-up run N steps between cudaProfilerStart/Stop and exit "
                         "(ncu --profile-from-start off); prints no bench line")
    ap.add_argument("--no-extras", action="store_true", help="skip dense/latency/kernel/cpu/check legs")
    ap.add_argument("--no-check", action="store_true", help="skip the parity leg against the reference flow")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits of the last timed step to DIR/output.npy (float32)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.profile):
        ap.error("--dump-outputs needs --impl ours and a timed run (no --profile)")
    if args.workload in WORKLOADS:
        wl = WORKLOADS[args.workload]
        args.height = args.height or wl["h"]
        args.width = args.width or wl["w"]
        args.streams = args.streams or wl["streams"](max(args.gpus, int(os.environ.get("WORLD_SIZE", "1"))))
        args.scaling = wl["scaling"]
    return args


# ---------------------------------------------------------------------------------------------
# pure-torch restatement of the dense model and the synthetic video for the REFERENCE arm: that arm
# must not load anything of the product (importing cbinfer_b200 dlopens libcbinfer_sm100.so).
# tests/test_boundary.py checks these against cbinfer_b200.models / .video bit for bit.
# ---------------------------------------------------------------------------------------------
def dense_scene_cnn(seed=0):
    """the dense scene-labeling CNN (topology: sceneLabeling/modelLoader.py:9-10,47,72-78)"""
    import torch
    import torch.nn as nn
    g = torch.random.get_rng_state()
    torch.manual_seed(seed)
    m = nn.Sequential(
        nn.Conv2d(3, 16, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
        nn.Conv2d(16, 64, 7, padding=3), nn.ReLU(), nn.MaxPool2d(2, 2),
        nn.Conv2d(64, 256, 7, padding=3), nn.ReLU(),
        nn.Conv2d(256, 64, 1), nn.ReLU(),
        nn.Conv2d(64, 8, 1),
    ).eval()
    torch.random.set_rng_state(g)
    return m


def synth_sequence(B, H, W, n, rate, mode="block", seed=0):
    """static-camera synthetic video (SURVEY section 8d): frame t = frame t-1 with one re-drawn
    rectangle of area rate*H*W (block) or Bernoulli(rate) pixels (iid) per stream"""
    import math
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    frames = [torch.rand(B, 3, H, W, generator=g)]
    for t in range(1, n):
        f = frames[-1].clone()
        if rate > 0:
            g = torch.Generator(device="cpu").manual_seed(1000 + t)
            if mode == "block":
                area = rate * H * W
                bh = min(H, max(1, int(round(math.sqrt(area * 3.0 / 4.0)))))
                bw = min(W, max(1, int(round(area / bh))))
                for b in range(B):
                    y0 = int(torch.randint(0, H - bh + 1, (1,), generator=g))
                    x0 = int(torch.randint(0, W - bw + 1, (1,), generator=g))
                    f[b, :, y0:y0 + bh, x0:x0 + bw] = torch.rand(3, bh, bw, generator=g)
            else:
                m = torch.rand(B, 1, H, W, generator=g) < rate
                f = torch.where(m, torch.rand(B, 3, H, W, generator=g), f)
        frames.append(f)
    return frames


# ---------------------------------------------------------------------------------------------
# clocks sampler (runs during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.004)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# the reference arm / cpu baseline: dense PyTorch CPU inference (the reference's dense path)
# ---------------------------------------------------------------------------------------------
def cpu_dense_fps(args, seconds, warm=2, max_steps=200):
    """the reference's dense inference path (evalTools.inferFrameset on the unconverted model) on
    the host cores, on the SAME batch as our arm: one step = one frame of all `streams` streams."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)            # reference: sceneLabeling/modelConverter.py:4
    base = dense_scene_cnn().float()
    S = args.streams
    frames = synth_sequence(S, args.height, args.width, 4, args.rate, args.mode)
    times = []
    with torch.no_grad():
        for i in range(warm):
            base(frames[i % 4])
        t_end = time.perf_counter() + seconds
        i = 0
        while (time.perf_counter() < t_end and len(times) < max_steps) or len(times) < 3:
            t0 = time.perf_counter()
            base(frames[i % 4])
            times.append(time.perf_counter() - t0)
            i += 1
    mean = sum(times) / len(times)
    return {"value": S / mean, "best": S / min(times), "unit": "frames/s", "cores": cores,
            "kind": "reference", "steps": len(times), "ms_per_step": mean * 1e3,
            "sample": "%d steps of %d frames %dx%d (one frame of each of the %d streams, batched) through the "
                      "dense nn.Conv2d/ReLU/MaxPool2d scene CNN on torch CPU (the reference's dense inference "
                      "path, evalTools.inferFrameset), fp32, %d threads; BASELINE configs[0] is the same model "
                      "on a 10-frame 320x240 sequence, this is the bench workload's size"
                      % (len(times), S, args.width, args.height, S, cores)}


def cpu_cb_oracle_fps(args, frames_cpu, thresholds, base, max_seconds=10.0):
    """the oracle's C port of the CB path (OpenMP) on a bounded sample -- reported, not a target."""
    import numpy as np
    import torch.nn as nn
    from oracle import oracle as orc
    L = orc.lib()
    convs = [m for m in base.modules() if isinstance(m, nn.Conv2d)]
    H, W = args.height, args.width
    dims = [(H, W), (H // 2, W // 2), (H // 4, W // 4), (H // 4, W // 4), (H // 4, W // 4)]
    st = []
    for c, (h, w) in zip(convs, dims):
        st.append(dict(
            wt=np.ascontiguousarray(c.weight.detach().cpu().numpy()), b=c.bias.detach().cpu().numpy().copy(),
            sin=np.full((c.in_channels, h, w), np.inf, np.float32),
            sout=np.full((c.out_channels, h, w), np.inf, np.float32),
            idx=np.zeros(h * w, np.int32), map=np.zeros(h * w, np.uint8), h=h, w=w))

    def frame(x):
        cur = x
        for i, (c, s) in enumerate(zip(convs, st)):
            k = c.kernel_size[0]
            L.orc_cbconv_frame_fast_f32(orc._p(cur), orc._p(s["sin"]), orc._p(s["sout"]), orc._p(s["wt"]),
                                        orc._p(s["b"]), orc._p(s["idx"]), orc._p(s["map"]), s["w"], s["h"],
                                        c.in_channels, c.out_channels, k, k, float(thresholds[i]), 1,
                                        int(i < 4))
            cur = s["sout"]
            if i < 2:      # dense 2x2 pool on the CPU side keeps the port simple
                cur = np.ascontiguousarray(cur.reshape(cur.shape[0], s["h"] // 2, 2, s["w"] // 2, 2).max(axis=(2, 4)))
        return cur

    xs = [np.ascontiguousarray(f[0].numpy()) for f in frames_cpu]
    frame(xs[0])
    times = []
    t_end = time.perf_counter() + max_seconds
    i = 1
    while time.perf_counter() < t_end and i < len(xs):
        t0 = time.perf_counter()
        frame(xs[i])
        times.append(time.perf_counter() - t0)
        i += 1
    if not times:
        return None
    return {"value": len(times) / sum(times), "unit": "frames/s", "cores": os.cpu_count(), "kind": "port",
            "sample": "%d frames through oracle/cbinfer_oracle.c orc_cbconv_frame_fast_f32 (OpenMP)" % len(times)}


def run_reference(args):
    """--impl reference: the reference's own CPU inference path, same config, nothing of the product
    loaded (no `import cbinfer_b200`).  Each step = one frame of every stream of one GPU's batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    budget = min(150.0, max(5.0, 0.6 * (args.steps + args.warmup)))
    r = cpu_dense_fps(args, seconds=budget, warm=max(min(args.warmup, 3), 1), max_steps=max(args.steps, 3))
    assert "cbinfer_b200" not in sys.modules
    out = {
        "impl": "reference", "metric": "frames/s", "value": r["value"], "unit": "frames/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": getattr(args, "scaling", "weak"),
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, streams=args.streams),
        "cpu_baseline": r,
        "e2e": {"value": r["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(out))


def workload_config(args, streams):
    return {"workload": "sceneLabeling CBinfer CNN (5 CBConv2d + 2 CBPoolMax2d, feedback loop) on synthetic "
                        "%dx%d video, %.0f%% %s change per frame" % (args.width, args.height, args.rate * 100, args.mode),
            "workload_name": args.workload,
            "streams_per_gpu": streams, "height": args.height, "width": args.width,
            "change_rate": args.rate, "change_mode": args.mode, "threshold_factor": args.threshold_factor,
            "gemm": args.gemm, "detection": "dense re-scan per layer" if args.dense_scan else
            "dense scan on the input frame, candidate detection on CB-fed layers", "parallelism": "independent video streams sharded per GPU, no collective"}


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
class SceneStep(object):
    """One step of the bench: the first layer's change detection runs eagerly on each frame WHERE
    IT LIES in HBM (CBConv2d.detectInput); everything after it replays as one CUDA graph captured
    on the "detection done" tuple -- no copy of the frame into a static graph input."""

    def __init__(self, model, frame0, frame1):
        import torch
        import cbinfer_b200 as cb
        from cbinfer_b200.conv2d import DetectionDone
        self.model = model
        self.first = [m for m in model.modules() if type(m) is cb.CBConv2d][0]
        self.static_in = frame0.clone()
        with torch.no_grad():
            model(self.static_in)                 # first frame: everything changed
            self.static_in.copy_(frame1)
            model(self.static_in)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            model(self.static_in)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self.out = model(('changeIndexes', self.static_in, DetectionDone(self.first)))

    def __call__(self, frame):
        import torch
        with torch.no_grad():
            self.first.detectInput(frame)
        self.graph.replay()
        return self.out

    def capture_slot(self, frame):
        """A graph of the WHOLE step for one input slot (a frame buffer at a fixed address, as in a
        decoder's surface pool): first-layer detection on that slot + the rest of the model.  One
        graph launch per step instead of an eager launch + a graph launch."""
        import torch
        from cbinfer_b200.conv2d import DetectionDone
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g), torch.no_grad():
            tup = self.first.detectInput(frame)
            out = self.model(tup)
        assert out.data_ptr() == self.out.data_ptr()
        return g


def build_model(args, base, first_frame):
    """the benchmarked model: scene CBinfer net, all convs + pools converted, feedback loop,
    thresholds = threshold_factor * range of each layer's dense input on the first frame"""
    import cbinfer_b200 as cb
    from cbinfer_b200 import models
    mdl = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                      clonePoolOutput=False, candidateDetect=not args.dense_scan)
    for m in mdl.modules():
        if type(m) is cb.CBConv2d:
            m.gemmMode = args.gemm
    thresholds = models.calibrateThresholds(base, mdl, first_frame, factor=args.threshold_factor)
    return mdl, thresholds


def parity_check(args, base, thresholds, frames_cpu, dev, nstreams=2, nframes=6):
    """--check leg (outside every timed region): the benchmarked configuration (candidate path,
    masked 1x1 layers, detectInput + graph) against the reference FLOW -- the unmodified reference
    CUDA kernels of oracle/_ref driven by tests/ref_flow.py with fp32 torch.matmul -- on the first
    `nstreams` streams.  Returns None when oracle/_ref was not built."""
    import torch
    import cbinfer_b200 as cb
    from tests import ref_flow
    if ref_flow.libs() is None:
        return None
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    S = min(nstreams, frames_cpu[0].shape[0])
    fr = [f[:S].to(dev) for f in frames_cpu[:nframes]]
    mdl, _ = build_model(args, base, fr[0])
    for c, th in zip([m for m in mdl.modules() if type(m) is cb.CBConv2d], thresholds):
        c.threshold = th
    step = SceneStep(mdl, fr[0], fr[1])
    refs = [ref_flow.convert_sequential(base, thresholds) for _ in range(S)]
    for s_ in range(S):
        for t in (0, 1, 1):                       # the same frames the warm-up of SceneStep saw
            ref_flow.run(refs[s_], fr[t][s_:s_ + 1].contiguous())
    worst, l1_equal, flips = 0.0, True, 0
    convs = [m for m in mdl.modules() if type(m) is cb.CBConv2d]
    for t in range(2, len(fr)):
        out = step(fr[t])
        torch.cuda.synchronize()
        mine = convs[0].lastChangeIndexes()
        for s_ in range(S):
            ro, _ = ref_flow.run(refs[s_], fr[t][s_:s_ + 1].contiguous())
            scale = float(ro.abs().max()) + 1e-30
            worst = max(worst, float((out[s_:s_ + 1].float() - ro).abs().max()) / scale)
            P = fr[t].shape[2] * fr[t].shape[3]
            sel = mine[(mine >= s_ * P) & (mine < (s_ + 1) * P)] - s_ * P
            l1_equal &= bool(torch.equal(sel, refs[s_][0].changeIndexes))
    for s_ in range(S):
        for li, ci in ((2, 1), (4, 2)):           # deeper 7x7 layers: differing change pixels (threshold flips)
            ref_idx = refs[s_][li].changeIndexes
            c = convs[ci]
            P = c.prevInput.shape[2] * c.prevInput.shape[3]
            mi = c.lastChangeIndexes()
            sel = mi[(mi >= s_ * P) & (mi < (s_ + 1) * P)] - s_ * P
            a = torch.zeros(P, dtype=torch.bool, device=dev)
            b = torch.zeros(P, dtype=torch.bool, device=dev)
            a[sel.long()] = True
            b[ref_idx.long()] = True
            flips += int((a ^ b).sum())
    return {"parity_max_rel": worst, "layer1_index_lists_bit_exact": l1_equal,
            "deeper_layer_mask_bits_differing_last_frame": flips, "streams": S, "frames": len(fr) - 2,
            "against": "unmodified reference kernels (oracle/_ref) + fp32 torch.matmul, tests/ref_flow.py"}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "split4k":
        sys.argv = [sys.argv[0], "--rate", str(args.rate), "--check"] + (
            ["--dump-outputs", args.dump_outputs] if args.dump_outputs else [])
        from benchmarks import split_4k
        return split_4k.main()

    import torch
    import torch.distributed as dist
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video, streams, conv2d_cg as cg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tdt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[args.dtype]
    S, H, W, K, Wm = args.streams, args.height, args.width, args.steps, max(args.warmup, 3)
    torch.backends.cudnn.benchmark = True

    # ---- model + synthetic video (each rank: its own streams, seeds offset by rank) ----------
    base = models.sceneLabelingBaseline().to(dev).to(tdt)
    # the video is played forwards and backwards over a window of <= 48 frames (walking back undoes
    # the same block change, so every step still sees one block change): long timed regions
    # without holding hundreds of frames; large workloads keep the window under ~6 GB
    frame_bytes = S * 3 * H * W * 4
    nframes = max(4, min(K + Wm + 2, 48, int(6e9 // frame_bytes)))

    def fidx(t):
        period = 2 * (nframes - 1)
        r = t % period
        return r if r < nframes else period - r

    my_streams = streams.shard_streams(S * world, world, rank)      # global stream ids of this rank
    frames_cpu = video.sequence(S, H, W, nframes, args.rate, args.mode, seed=my_streams[0])
    pinned = [f.to(tdt).pin_memory() for f in frames_cpu]
    frames = [f.to(dev, non_blocking=True) for f in pinned]
    torch.cuda.synchronize()
    model, thresholds = build_model(args, base, frames[0])          # the timed model
    step_obj = SceneStep(model, frames[0], frames[1])
    # my kernels per step: dense scan: 5 x (detect, compact, conv) + 2 pools = 17; candidate path: the two
    # pools also run the next conv's detection (15), the two trailing 1x1 layers skip the compaction (their
    # contraction masks the candidate list: 13) and the two tiled convs pool in their epilogue (11)
    fused_pools = sum(1 for m in model.modules() if type(m) is cb.CBConv2d and getattr(m, '_fusedPool', None)
                      and os.environ.get("CBINFER_FUSE_POOL", "1") != "0" and os.environ.get("CBINFER_TILES", "1") != "0")
    fused_tail = sum(1 for m in model.modules() if type(m) is cb.CBConv2d and getattr(m, '_fusedTail', None)
                     and os.environ.get("CBINFER_FUSE_TAIL", "1") != "0")
    # (... and derive their dilated bitmap + tile list themselves, cb_conv_update_tiled_self: 6 with the tail fused)
    self_tiles = sum(1 for m in model.modules() if type(m) is cb.CBConv2d and getattr(m, '_fusedPool', None)
                     and m._inBuf is not None and m._selfTiles(*m._inBuf.shape[:3])) if fused_pools else 0
    my_launches_per_step = 17 if args.dense_scan else 13 - fused_pools - 3 * fused_tail - self_tiles

    # one captured graph per input slot of the frame ring (the bench cycles over `nframes` device
    # buffers): a step is ONE graph launch -- first-layer detection on the slot where the frame lies
    # + the rest of the model.  --eager-detect: detection launched eagerly on arbitrary frame addresses
    # + one graph for the rest (what CBConv2d.detectInput offers to callers without a fixed ring).
    slot_graphs = None
    if not args.eager_detect:
        slot_graphs = [step_obj.capture_slot(f) for f in frames]

    def step(t):
        if slot_graphs is not None:
            slot_graphs[fidx(t)].replay()
        else:
            step_obj(frames[fidx(t)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    t = 2
    for _ in range(Wm):
        step(t)
        t += 1
    if args.profile:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for _ in range(args.profile):
            step(t)
            t += 1
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled_steps": args.profile, "launches_per_step": my_launches_per_step}))
        return
    # ---- timed region: EXACTLY K steps, bracketed by barrier + synchronize and timed on the device
    #      (max over ranks) ----------------------------------------------------------------------------
    sampler = ClockSampler(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.start()
    e0.record()
    for _ in range(K):
        step(t)
        t += 1
    e1.record()
    barrier()
    # whole-job rate: frames of all ranks / slowest rank's device time
    fps, elapsed_ms = streams.whole_job_rate(S * K, e0.elapsed_time(e1), dev)
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, step_obj.out, "output" if world == 1 else "output_rank%d" % rank,
                     DUMP_BYTES // world)
    counts = [int(m._scratch["count"].item()) for m in model.modules() if type(m) is cb.CBConv2d]
    state_mb = sum(x.numel() * x.element_size() for x in cb.getStateTensors(model)) / 1e6

    # ---- e2e: the public per-frame API with HOST frames: every step copies its frames from pinned
    #      host memory (H2D) and reads its logits back (D2H).  runtime.FramePipeline = one graph
    #      replay per frame with the copies of neighbouring frames overlapped on their own streams.
    from cbinfer_b200 import runtime
    del step_obj, slot_graphs
    cb.clearMemory(model)

    def copy_only_gbs(pin, first_frame_dev, n=60):
        """host-side ceiling of the e2e legs: the same pinned buffers copied H2D on ALL ranks at once,
        no compute (PCIe + host memory fabric of the box; per GPU, GB/s)"""
        dst = torch.empty_like(first_frame_dev)
        wall = 0.0
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            for i in range(n):
                dst.copy_(pin[fidx(i)], non_blocking=True)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            barrier()
        worst = streams.max_over_ranks(wall, dev)
        return pin[0].numel() * pin[0].element_size() * n / worst / 1e9

    def e2e_leg(pin, first_frame_dev, mdl=None):
        pipe = runtime.FramePipeline(mdl if mdl is not None else model, first_frame_dev, depth=2)
        for i in range(1, Wm + 1):
            pipe.submit(pin[fidx(i)])
        pipe.drain()
        last = None
        barrier()
        t0 = time.perf_counter()
        for i in range(Wm + 1, Wm + 1 + K):
            last = pipe.submit(pin[fidx(i)])
        pipe.wait(last)
        pipe.drain()
        wall_ms = (time.perf_counter() - t0) * 1e3
        barrier()
        # host wall clock from first submit to last result on the host (a device event pair on
        # the default stream does not see the side streams)
        f_, ms_ = streams.whole_job_rate(S * K, wall_ms, dev)
        d2h_ = pipe.out_host[0].numel() * pipe.out_host[0].element_size()
        chk = float(pipe.out_host[last].float().abs().sum())
        del pipe
        return f_, ms_, d2h_, chk

    h2d = pinned[0].numel() * pinned[0].element_size()
    ceiling_gbs = copy_only_gbs(pinned, frames[0])
    e2e_fps, e2e_ms, d2h, e2e_checksum = e2e_leg(pinned, frames[0])

    # ---- e2e with uint8 host frames (what a camera / decoder delivers): the first layer's detection
    #      kernel normalises u8/255 on the fly (cb_change_detect_u8), so a quarter of the bytes cross
    #      PCIe.  Same pipeline, same change pattern; reported beside `e2e`, never instead of it.
    e2e_u8 = None
    if args.dtype == "f32":
        cb.clearMemory(model)
        first = [m for m in model.modules() if type(m) is cb.CBConv2d][0]
        first.inputNorm = (255.0, 0.0)
        pinned8 = [f.mul(255.0).round().to(torch.uint8).pin_memory() for f in frames_cpu]
        u8_fps, u8_ms, _, u8_chk = e2e_leg(pinned8, pinned8[0].to(dev))
        e2e_u8 = {"value": u8_fps, "unit": "frames/s", "ms_per_step": u8_ms / K,
                  "h2d_gbs": pinned8[0].numel() / (u8_ms / K * 1e-3) / 1e9,
                  "h2d_bytes_per_step": pinned8[0].numel(), "d2h_bytes_per_step": d2h,
                  "checksum": u8_chk,
                  "path": "as e2e, but the pinned host frames are uint8 and are normalised (u8/255) inside "
                          "the first layer's detection kernel (cb_change_detect_u8)"}
        # ... and with the task's result instead of the logits coming back: the label map (argmax over the
        # classes, one byte per pixel) is computed on the device inside the same graph, so 1/32 of the
        # D2H bytes cross the host fabric -- what bounds the multi-GPU e2e rate (see host_h2d_copy_only_gbs)
        cb.clearMemory(model)

        class LabelHead(torch.nn.Module):
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, x):
                return self.m(x).argmax(1).to(torch.uint8)

        lb_fps, lb_ms, lb_d2h, lb_chk = e2e_leg(pinned8, pinned8[0].to(dev), LabelHead(model))
        e2e_u8["labels_out"] = {"value": lb_fps, "unit": "frames/s", "ms_per_step": lb_ms / K,
                                "h2d_bytes_per_step": pinned8[0].numel(), "d2h_bytes_per_step": lb_d2h,
                                "checksum": lb_chk,
                                "path": "as e2e_u8_ingest, D2H = uint8 label map (argmax over the 8 classes on the "
                                        "device) instead of the fp32 logits"}
        del pinned8
        first.inputNorm = None
        cb.clearMemory(model)

    result = {
        "metric": "frames/s", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": dict(workload_config(args, S),
                       note=WORKLOADS[args.workload]["note"],
                       l2="no flush: per-step working set = persistent state maps of %d streams = %.0f MB %s 126 MB L2"
                          % (S, state_mb, ">" if state_mb > 126 else "<= (L2-resident!)"),
                       launch=("per step: first-layer detection launched eagerly on the frame where it lies in "
                               "HBM, the other launches replayed as one CUDA graph") if args.eager_detect else
                              ("per step ONE CUDA-graph launch: a graph per input slot of the %d-frame ring holds the "
                               "first-layer detection on that slot (read in place) and the rest of the model" % nframes),
                       timing="one device-timed block of %d steps after %d warm-up steps" % (K, Wm),
                       thresholds=[round(x, 5) for x in thresholds],
                       changed_pixels_last_frame=counts),
        "timed_region_s": elapsed_ms * 1e-3,
        "clocks": clocks,
        "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / K, "checksum": e2e_checksum,
                "h2d_gbs": h2d / (e2e_ms / K * 1e-3) / 1e9,     # PCIe roofline of this leg (Gen5 x16 ~ 55 GB/s)
                # the box's host-side ceiling at this N: the same pinned frames copied H2D by all ranks
                # at once without any compute (one GPU alone ~55 GB/s; 8 GPUs share ~190 GB/s)
                "host_h2d_copy_only_gbs_per_gpu": ceiling_gbs,
                "path": "runtime.FramePipeline: per step pinned H2D of the frames, one graph replay, D2H of the "
                        "logits; copies of neighbouring steps overlap compute (3 streams); host wall clock"},
        "gpu_launches": my_launches_per_step * K,
    }
    if e2e_u8 is not None:
        result["e2e_u8_ingest"] = e2e_u8

    # ---- extras on rank 0: parity leg, kernel table / roofline, dense cuDNN, single-stream latency, CPU ----
    if rank == 0 and not args.no_extras:
        if not args.no_check and args.dtype == "f32":
            try:
                chk = parity_check(args, base, thresholds, frames_cpu, dev)
                if chk is not None:
                    result["parity_max_rel"] = chk["parity_max_rel"]
                    result["parity"] = chk
            except Exception as e:
                result["parity_error"] = repr(e)
        try:
            result.update(kernel_roofline(args, model, frames, dev, tdt, elapsed_ms / K * 1e3))
        except Exception as e:                                   # never lose the headline line
            result["roofline_error"] = repr(e)
        try:
            ins = kernels_in_step(args, model, frames)
            result["kernels_in_step"] = ins
            rf = result.get("roofline")
            if rf and rf.get("bound") == "tensor":
                # the dominant kernel as it runs INSIDE a step (cold data), next to the warm replay figure
                us = next((r["us"] for r in ins["launches"] if "%s[%s]" % (r["kernel"], r["layer"]) == rf["kernel"]), None)
                if us:
                    flops = next(r["flops"] for r in result["kernels"]
                                 if "%s[%s]" % (r["kernel"], r["layer"]) == rf["kernel"])
                    rf["in_step"] = {"us": us, "achieved": round(flops / (us * 1e-6) / 1e12, 2),
                                     "frac": flops / (us * 1e-6) / 1e12 / rf["peak"],
                                     "note": "timed by external event nodes inside the step's graph; includes ~%.0f us of "
                                             "event-node overhead per launch" % ins["event_overhead_us_per_launch"]}
        except Exception as e:
            result["kernels_in_step_error"] = repr(e)
        try:
            result["dense_cudnn"] = dense_gpu(args, base, frames, dev)
        except Exception as e:
            result["dense_cudnn_error"] = repr(e)
        if world == 1:
            try:
                result["single_stream"] = single_stream_latency(args, base, dev, tdt)
            except Exception as e:
                result["single_stream_error"] = repr(e)
            try:
                result["cpu_baseline"] = cpu_dense_fps(args, seconds=args.cpu_seconds)
                if args.dtype == "f32" and args.workload == "scene640":
                    r = cpu_cb_oracle_fps(args, [f[:1].float() for f in frames_cpu[:12]], thresholds, base.float().cpu())
                    base.to(dev)
                    if r:
                        result["cpu_cb_port"] = r
            except Exception as e:
                result["cpu_baseline_error"] = repr(e)
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 64_000_000       # all files of one --dump-outputs run together


def dump_outputs(directory, out, name, budget):
    """DIR/<name>.npy: `out` as float32; if it exceeds `budget` bytes, every s-th element of the
    flattened array with the smallest stride s that fits"""
    import numpy as np
    a = out.detach().float().cpu().numpy()
    stride = -(-a.size // ((budget - 4096) // a.itemsize))          # 4 KB for the .npy header
    if stride > 1:
        a = np.ascontiguousarray(a.reshape(-1)[::stride])
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, name + ".npy"), a)


def kernels_in_step(args, model, frames, reps=40):
    """Every launch of a step timed INSIDE the step: the step's CUDA graph is captured with external
    timing events recorded as graph nodes around each C-ABI call, so each kernel runs on the inputs and in
    the cache state it really sees (the back-to-back replays of kernel_roofline run warm).  The event nodes
    cost a few microseconds per launch: the instrumented step is reported next to the plain one."""
    import torch
    import cbinfer_b200 as cb
    from cbinfer_b200 import conv2d_cg as cg
    cb.clearMemory(model)
    fr = frames[:8]
    so = SceneStep(model, fr[0], fr[1])
    plain = [so.capture_slot(f) for f in fr]
    names = ("detect", "detect_u8", "detect_sparse", "detect_sparse_compact", "dilate_compact", "dilate_tiles",
             "pool_compact", "conv_update", "conv_update_tiled", "tail_update", "maxPool2d", "maxPool2d_detect",
             "detect_compact_sparse")
    orig = {n: getattr(cg, n) for n in names}
    cur = {"layer": None, "log": None}

    def wrap(name):
        fn = orig[name]

        def w(*a, **k):
            e0 = torch.cuda.Event(enable_timing=True, external=True)
            e1 = torch.cuda.Event(enable_timing=True, external=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            cur["log"].append((cur["layer"], name, e0, e1))
            return r
        return w

    hooks = [m.register_forward_pre_hook(lambda mod, inp, ln=ln: cur.__setitem__("layer", ln))
             for ln, m in model.named_children()]
    inst = []
    try:
        for n in names:
            setattr(cg, n, wrap(n))
        for f in fr:
            cur["log"] = []
            cur["layer"] = next(iter(dict(model.named_children())))
            inst.append((so.capture_slot(f), cur["log"]))
    finally:
        for n, f in orig.items():
            setattr(cg, n, f)
        for h in hooks:
            h.remove()
    nf = len(fr)
    period = 2 * (nf - 1)

    def fidx(t):
        r = t % period
        return r if r < nf else period - r

    def run(graphs):
        t = 2
        for _ in range(20):
            graphs[fidx(t)].replay()
            t += 1
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps * period):
            graphs[fidx(t)].replay()
            t += 1
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (reps * period)

    plain_us = run(plain)
    inst_us = run([g for g, _ in inst])
    acc = {}
    t = 2
    for _ in range(reps):
        g, lg = inst[fidx(t)]
        g.replay()
        torch.cuda.synchronize()
        for i, (ln, name, e0, e1) in enumerate(lg):
            acc.setdefault((i, ln, name), []).append(e0.elapsed_time(e1) * 1e3)
        t += 1
    rows = []
    for (i, ln, name), v in sorted(acc.items()):
        v.sort()
        rows.append({"layer": ln, "kernel": name, "us": round(v[len(v) // 2], 2)})
    del plain, inst, so
    cb.clearMemory(model)
    n = max(len(rows), 1)
    return {"launches": rows, "plain_step_us": round(plain_us, 1), "instrumented_step_us": round(inst_us, 1),
            "event_overhead_us_per_launch": round((inst_us - plain_us) / n, 1)}


def kernel_roofline(args, model, frames, dev, tdt, step_us):
    """Per-kernel CUDA-event timing of one steady-state frame (graph replays of each recorded launch)
    and the roofline of the dominant kernel.  Algorithmic bytes / FLOPs per launch: DESIGN.md 3."""
    import torch
    import cbinfer_b200 as cb
    from cbinfer_b200 import conv2d_cg as cg
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    bf16 = float(peaks.get("bf16_tflops", 1590.0))
    src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    es = 4 if args.dtype == "f32" else 2
    # Steady-state time of every launch of one frame: the arguments of each C-ABI call of a real
    # frame are recorded, then each call is replayed REP times inside one CUDA graph and timed with
    # CUDA events on the launching stream (per-launch time incl. the dependent-launch gap; an event
    # pair around a single eager launch would include the host's launch latency).  Replays run in
    # reverse order so a producer's repetitions do not wipe its consumers' inputs.
    REP = 20
    cur = {"layer": None}
    calls = []
    names = ("detect", "detect_sparse", "dilate_compact", "dilate_tiles", "pool_compact", "conv_update", "conv_update_tiled", "tail_update",
             "maxPool2d", "maxPool2d_detect", "detect_compact_sparse")
    orig = {n: getattr(cg, n) for n in names}

    def recorder(name):
        fn = orig[name]

        def w(*a, **k):
            if name in ("dilate_compact", "dilate_tiles"):
                k = dict(k, clear_raw=False)  # keep the raw bitmap: the replays must see the real input
            if name == "conv_update_tiled" and k.get("self_list"):
                k = dict(k, self_list=dict(k["self_list"], clear_raw=False))
            calls.append((cur["layer"], name, a, k))
            return fn(*a, **k)
        return w

    hooks = []
    for lname, m in model.named_children():
        hooks.append(m.register_forward_pre_hook(lambda mod, inp, lname=lname: cur.__setitem__("layer", lname)))
    try:
        cb.clearMemory(model)
        with torch.no_grad():
            for i in range(0, 4):
                model(frames[i])
            for n in orig:
                setattr(cg, n, recorder(n))
            model(frames[4])
        torch.cuda.synchronize()
        counts = {ln: int(m._scratch["count"].item()) for ln, m in model.named_children()
                  if type(m) is cb.CBConv2d}
    finally:
        for n, f in orig.items():
            setattr(cg, n, f)
        for h in hooks:
            h.remove()
    rec = {}
    for lname, kname, a, k in reversed(calls):
        k = dict(k)
        if kname in ("dilate_compact", "dilate_tiles"):
            k["clear_raw"] = False           # keep the input bitmap intact across repetitions
        if kname == "detect_sparse":
            k["bits_are_clear"] = False
        if kname == "tail_update":
            a = a[:17] + (0,) + a[18:]       # update_mode NONE: every repetition sees the same changes
        fn = orig[kname]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn(*a, **k)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(REP):
                fn(*a, **k)
        g.replay()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(3):
            g.replay()
        a1.record()
        torch.cuda.synchronize()
        rec[(lname, kname)] = (a0.elapsed_time(a1) * 1e3 / (3 * REP), 3 * REP)
        del g
    mods = dict(model.named_children())
    table = []
    for (lname, kname), (us, nl) in rec.items():
        m = mods[lname]
        row = {"layer": lname, "kernel": kname, "us": round(us, 2), "launches": nl}
        if type(m) is cb.CBConv2d:
            B, Cin, Hh, Ww = m.prevInput.shape
            P = B * Hh * Ww
            n = counts[lname]
            k2 = m.kernel_size[0] * m.kernel_size[1]
            if kname == "detect_sparse":
                row.update(bound="hbm")
            elif kname == "detect":
                by = 2 * Cin * P * es + P // 8
                row.update(bound="hbm", bytes=by, achieved=by / (us * 1e-6) / 1e9, peak=hbm, unit="GB/s")
            elif kname in ("dilate_compact", "dilate_tiles"):
                by = P // 8 + (4 * n if kname == "dilate_compact" else P // 8)
                row.update(bound="hbm", bytes=by, achieved=by / (us * 1e-6) / 1e9, peak=hbm, unit="GB/s")
            elif kname in ("conv_update", "conv_update_tiled"):
                fl = 2.0 * n * Cin * k2 * m.out_channels
                by = min(n * k2, P) * Cin * es + m.out_channels * Cin * k2 * es + 4 * n + n * m.out_channels * es
                pk = bf16 / 2 if (args.dtype == "f32" and args.gemm in ("tc", "tc3x")) else bf16
                row.update(bound="tensor", flops=fl, bytes=by, achieved=fl / (us * 1e-6) / 1e12, peak=pk,
                           unit="TFLOP/s", n=n, hbm_gbs=by / (us * 1e-6) / 1e9)
                if kname == "conv_update_tiled":
                    row["tiles"] = int(m._scratch["tile_ws"][1])
        else:
            row.update(bound="hbm")
        if "achieved" in row:
            row["frac"] = row["achieved"] / row["peak"]
            row["achieved"] = round(row["achieved"], 2)
        table.append(row)
    cb.clearMemory(model)                     # the recorded frame left raw bitmaps uncleared
    table.sort(key=lambda r: -r["us"])
    total = sum(r["us"] for r in table)
    top = next((r for r in table if "achieved" in r), None)
    out = {"kernels": table, "kernel_us_per_step": round(total, 1), "peaks_source": src}
    if top:
        key = "%s[%s]" % (top["kernel"], top["layer"])
        traffic = None
        try:
            traffic = json.load(open(os.path.join(REPO, "profiles", "r02_traffic.json"))).get(key, {}).get("bytes")
        except Exception:
            pass
        out["roofline"] = {"kernel": key, "bound": top["bound"],
                           "achieved": top["achieved"], "peak": top["peak"], "unit": top["unit"],
                           "frac": top["frac"], "traffic": traffic,
                           "tensor_work_frac": (3.0 * top["frac"] if top["bound"] == "tensor" and args.dtype == "f32"
                                                and args.gemm in ("auto", "bf16x3", "tc3x") else top["frac"]),
                           # share of the timed (graph-replay) step; the eager per-launch timings of the
                           # small kernels include launch gaps, so their sum is not the denominator
                           "share_of_step": top["us"] / step_us if step_us else None,
                           "note": ("fp32 data: %s split, 3 tensor-core MMAs per product; peak = %s; `achieved` counts the "
                                    "algorithmic FLOPs 2*n*K*Cout once, tensor_work_frac counts the 3x MMA work"
                                    % (("3xTF32", "bf16 burst / 2") if args.gemm == "tc3x" else ("3xBF16", "bf16 burst")))
                           if top["bound"] == "tensor" and args.dtype == "f32" and args.gemm in ("auto", "bf16x3", "tc3x") else ""}
    return out


def dense_gpu(args, base, frames, dev):
    """dense cuDNN comparator on the same GPU, same batch: fp32 (TF32 off / on) and bf16."""
    import torch
    res = {}
    S = frames[0].shape[0]
    for name, tf32, dt, cl in (("fp32", False, torch.float32, False), ("tf32", True, torch.float32, False),
                               ("tf32_channels_last", True, torch.float32, True),
                               ("bf16_channels_last", True, torch.bfloat16, True)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        m = base.to(dt)
        xs = [f.to(dt) for f in frames[:4]]
        if cl:
            m = m.to(memory_format=torch.channels_last)
            xs = [x.contiguous(memory_format=torch.channels_last) for x in xs]
        with torch.no_grad():
            for i in range(5):
                m(xs[i % 4])
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(20):
                m(xs[i % 4])
            b.record()
            torch.cuda.synchronize()
        res[name] = round(S * 20 / (a.elapsed_time(b) * 1e-3), 1)
        base.to(frames[0].dtype).to(memory_format=torch.contiguous_format)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res["unit"] = "frames/s"
    res["batch"] = S
    return res


def single_stream_latency(args, base, dev, tdt):
    """one stream (batch 1, the reference's own operating point): per-frame latency through a CUDA
    graph with an L2 flush (256 MB write) before every timed frame."""
    import torch
    import cbinfer_b200 as cb
    from cbinfer_b200 import models, video
    model = models.sceneLabelingCBinfer(base, experimentIdx=6, threshold=0.1, convertAll=True,
                                        clonePoolOutput=False, candidateDetect=not args.dense_scan)
    for m in model.modules():
        if type(m) is cb.CBConv2d:
            m.gemmMode = args.gemm
    fr = [f.to(dev).to(tdt) for f in video.sequence(1, args.height, args.width, 24, args.rate, args.mode, seed=77)]
    models.calibrateThresholds(base, model, fr[0], factor=args.threshold_factor)
    x = fr[0].clone()
    with torch.no_grad():
        model(x)
        x.copy_(fr[1])
        model(x)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        model(x)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g), torch.no_grad():
        model(x)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ms = []
    for i in range(3, 24):
        x.copy_(fr[i])
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ms = ms[3:]
    ms.sort()
    med = ms[len(ms) // 2]
    return {"streams": 1, "ms_per_frame_median": round(med, 4), "frames_per_s": round(1000.0 / med, 1),
            "l2_flush": "256 MB write before each timed frame", "frames": len(ms)}


if __name__ == "__main__":
    main()
