"""Per-frame runtime around a converted model: CUDA-graph replay and a copy/compute pipeline.

The reference drives its model with one python call per frame (`poseDetection/evalTools.py:37-49`:
``model(frame.cuda())``), paying ~10 launches and a host sync per layer.  Here a frame of the whole
model is ONE CUDA-graph replay (no host work between kernels), and `FramePipeline` overlaps the
host->device copy of frame t+1 and the device->host copy of result t-1 with the compute of frame t
on separate streams (H2D, compute, D2H), which is what bounds end-to-end throughput once the
kernels are fast: a 640x480 fp32 frame is 3.7 MB of PCIe traffic.
"""
import torch

from ._lib import CBinferError


class FrameGraph(object):
    """Capture ``model(static_input)`` once; ``replay()`` re-runs it on whatever the caller copied
    into ``static_input``.  The model must have seen at least one frame (state allocated)."""

    def __init__(self, model, static_input, warmup=True):
        self.model = model
        self.static_input = static_input
        if warmup:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side), torch.no_grad():
                model(static_input)
            torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph), torch.no_grad():
            self.static_output = model(static_input)

    def replay(self):
        self.graph.replay()
        return self.static_output


class FramePipeline(object):
    """Feed pinned host frames through a converted model with copies overlapped with compute.

    depth input slots, each with its own captured graph of the same model (the model's state is
    shared, so graphs replay strictly in submission order on the compute stream).

    activeStreams=True: ``submit(frame, active)`` may name the streams that have a new frame; only
    their slices cross PCIe and the others are skipped by the model (cbinfer_b200.setActiveStreams).
    The constructor sets an all-active mask on the model before capturing the graphs, and refuses a
    model in which a module other than a CB layer reads the input frame directly: the input slot of
    a skipped stream holds a stale frame, which only the mask-honouring CB layers may be given.

    trackChanges=True: the model's per-stream change counts (cbinfer_b200.trackStreamChanges, enabled
    here if it is not yet) travel with each slot's output: ``changeCounts(slot)`` is the int32 [L, B]
    host copy of the frame's counts, valid after ``wait(slot)``."""

    def __init__(self, model, example_frame, depth=2, activeStreams=False, trackChanges=False):
        from . import CBConv2d, CBPoolMax2d, setActiveStreams, streamChangeCounts, trackStreamChanges
        dev = example_frame.device
        assert dev.type == "cuda"
        self.model = model
        self.depth = depth
        self.compute = torch.cuda.Stream(dev)
        self.h2d = torch.cuda.Stream(dev)
        self.d2h = torch.cuda.Stream(dev)
        self.inputs = [example_frame.clone() for _ in range(depth)]
        B = example_frame.shape[0]
        self._mask = None
        cur = torch.cuda.current_stream(dev)
        self.compute.wait_stream(cur)
        readers, hooks = [], []
        if activeStreams:
            def pre_hook(mod, args):
                if any(isinstance(a, torch.Tensor) and a.data_ptr() == self.inputs[0].data_ptr() for a in args):
                    readers.append(type(mod).__name__)
            hooks = [m.register_forward_pre_hook(pre_hook) for m in model.modules()
                     if not list(m.children()) and type(m) not in (CBConv2d, CBPoolMax2d)]
        with torch.cuda.stream(self.compute), torch.no_grad():
            if activeStreams:
                setActiveStreams(model, torch.ones(B, dtype=torch.uint8, device=dev))
                self._mask = next(c._activeMask for c in model.modules() if type(c) is CBConv2d)
            if trackChanges and not any(type(c) is CBConv2d and c._streamRow is not None for c in model.modules()):
                trackStreamChanges(model, B=B)
            try:
                probe = model(self.inputs[0])                 # allocates state on first use
            finally:
                for h in hooks:
                    h.remove()
            if readers:
                raise CBinferError("FramePipeline(activeStreams=True): %s read the input frame directly; a "
                                   "skipped stream's slice of it is stale" % sorted(set(readers)))
            if isinstance(probe, tuple) and probe and probe[0] == 'changeIndexes':
                probe = probe[1]
            self.graphs = [FrameGraph(model, x, warmup=True) for x in self.inputs]
        self.compute.synchronize()
        outs = self.graphs[0].static_output
        self._multi = isinstance(outs, (tuple, list))
        first = outs[0] if self._multi else outs
        self.out_dev = [torch.empty_like(first, memory_format=torch.contiguous_format)
                        for _ in range(depth)]
        self.out_host = [torch.empty(first.shape, dtype=first.dtype).pin_memory() for _ in range(depth)]
        self.in_free = [torch.cuda.Event() for _ in range(depth)]     # slot's graph has consumed it
        self.in_ready = [torch.cuda.Event() for _ in range(depth)]
        self.out_ready = [torch.cuda.Event() for _ in range(depth)]   # device-side result copied
        self.out_done = [torch.cuda.Event() for _ in range(depth)]    # host buffer filled
        if activeStreams:
            # per-slot staging of the mask in pinned host and in device memory: it travels with the
            # slot's frame on the copy stream, and the device mask that every graph reads is written
            # from it on the compute stream right before the slot's replay (writing the shared
            # buffer on the copy stream would race with the previous slot's replay)
            self.mask_host = [torch.ones(B, dtype=torch.uint8).pin_memory() for _ in range(depth)]
            self.mask_dev = [torch.ones(B, dtype=torch.uint8, device=dev) for _ in range(depth)]
        self._counts = None
        if trackChanges:
            # the model's buffer is rewritten by every replay: copied per slot on the compute stream right
            # after the replay (as the output), then to pinned host memory on the copy stream
            self._counts = streamChangeCounts(model)
            self.counts_dev = [torch.empty_like(self._counts) for _ in range(depth)]
            self.counts_host = [torch.empty(self._counts.shape, dtype=torch.int32).pin_memory() for _ in range(depth)]
        self.t = 0
        for e in self.in_free + self.out_done:
            e.record(self.compute)

    def submit(self, host_frame, active=None):
        """Queue one frame (pinned host tensor); returns the slot whose host result buffer will
        hold this frame's output once `wait(slot)` returns.

        `active` (activeStreams=True only): the indices of the streams that have a new frame, None =
        all.  Only their slices of `host_frame` are copied (one copy per contiguous run); the other
        streams are skipped and their rows of the result hold their previous output."""
        B = self.inputs[0].shape[0]
        if active is None:
            keep = [True] * B
        else:
            if self._mask is None:
                raise CBinferError("FramePipeline.submit(active=...) needs FramePipeline(activeStreams=True)")
            idx = [int(i) for i in active]
            if any(not 0 <= i < B for i in idx):
                raise CBinferError("FramePipeline.submit: stream indices %s out of range for %d streams" % (idx, B))
            keep = [False] * B
            for i in idx:
                keep[i] = True
        s = self.t % self.depth
        self.t += 1
        if self._mask is not None:
            self.in_ready[s].synchronize()                 # the slot's last upload has read the staging
            self.mask_host[s].copy_(torch.tensor(keep, dtype=torch.uint8))
        with torch.cuda.stream(self.h2d):
            self.h2d.wait_event(self.in_free[s])
            b = 0
            while b < B:                                   # one copy per contiguous run of active streams
                if not keep[b]:
                    b += 1
                    continue
                e = b
                while e < B and keep[e]:
                    e += 1
                self.inputs[s][b:e].copy_(host_frame[b:e], non_blocking=True)
                b = e
            if self._mask is not None:
                self.mask_dev[s].copy_(self.mask_host[s], non_blocking=True)
            self.in_ready[s].record(self.h2d)
        with torch.cuda.stream(self.compute):
            self.compute.wait_event(self.in_ready[s])
            self.compute.wait_event(self.out_done[s])      # previous D2H of this slot finished
            if self._mask is not None:
                self._mask.copy_(self.mask_dev[s])
            out = self.graphs[s].replay()
            self.in_free[s].record(self.compute)
            self.out_dev[s].copy_(out[0] if self._multi else out)
            if self._counts is not None:
                self.counts_dev[s].copy_(self._counts)
            self.out_ready[s].record(self.compute)
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(self.out_ready[s])
            self.out_host[s].copy_(self.out_dev[s], non_blocking=True)
            if self._counts is not None:
                self.counts_host[s].copy_(self.counts_dev[s], non_blocking=True)
            self.out_done[s].record(self.d2h)
        return s

    def reset(self, streams):
        """Start a new sequence in `streams` (see cbinfer_b200.resetStreams): enqueued on the compute
        stream, so it applies from the next `submit`ted frame on; frames already submitted are
        computed without it.  The captured graphs stay valid."""
        from . import resetStreams
        with torch.cuda.stream(self.compute):
            resetStreams(self.model, streams)

    def setStreamThresholds(self, table):
        """Write new per-stream thresholds (see cbinfer_b200.setStreamThresholds, including which streams
        restart): enqueued on the compute stream, so they apply from the next `submit`ted frame on; frames
        already submitted are computed with the old values.  The captured graphs stay valid: they read the
        table the model had when they were captured, so one must be attached before the pipeline is built."""
        from . import setStreamThresholds, streamThresholds
        streamThresholds(self.model)                 # raises if the graphs were captured without a table
        if table is None:
            raise CBinferError("FramePipeline.setStreamThresholds: the graphs read the table; it cannot be detached")
        with torch.cuda.stream(self.compute):
            setStreamThresholds(self.model, table)

    def setStreamZones(self, zones):
        """Write a new watched-pixel zone of the same [B, H, W] (see cbinfer_b200.setStreamZones): enqueued on
        the compute stream, so it applies from the next `submit`ted frame on.  The captured graphs read the
        zone buffer the model had when they were captured, so one must be attached before the pipeline is
        built, and it cannot be detached or reshaped through the pipeline."""
        from . import CBConv2d, setStreamZones
        first = next(c for c in self.model.modules() if type(c) is CBConv2d)
        if first._zone is None:
            raise CBinferError("FramePipeline.setStreamZones: the graphs were captured without a zone; attach one "
                               "(cbinfer_b200.setStreamZones) before building the pipeline")
        if zones is None:
            raise CBinferError("FramePipeline.setStreamZones: the graphs read the zone; it cannot be detached")
        if not isinstance(zones, torch.Tensor) or tuple(zones.shape) != first._zone[1]:
            raise CBinferError("FramePipeline.setStreamZones: the graphs read a zone [B, H, W] = %s"
                               % (list(first._zone[1]),))
        with torch.cuda.stream(self.compute):
            setStreamZones(self.model, zones)

    def wait(self, slot):
        self.out_done[slot].synchronize()
        return self.out_host[slot]

    def changeCounts(self, slot):
        """The per-stream change counts (int32 [L, B] host tensor, see trackStreamChanges) of the frame
        last submitted to `slot`; valid after ``wait(slot)``.  Needs FramePipeline(trackChanges=True)."""
        if self._counts is None:
            raise CBinferError("FramePipeline.changeCounts needs FramePipeline(trackChanges=True)")
        return self.counts_host[slot]

    def drain(self):
        self.h2d.synchronize()
        self.compute.synchronize()
        self.d2h.synchronize()


def _cpulist(text):
    cpus = []
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus += list(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_host_cores(local_rank, local_world, min_cores=2):
    """Pin this feeder process to its own slice of the host cores, taken from the NUMA node its GPU
    hangs off when the box exposes one (sysfs), so that the pinned frame buffers it allocates
    afterwards are node-local and N feeders do not migrate over each other's cores.  Returns the
    cores chosen (or None when the host gives every rank fewer than `min_cores`).  Call before the
    first CUDA / pinned allocation."""
    import os
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return None
    def node_of(i):
        try:
            p = torch.cuda.get_device_properties(i)
            bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
            return int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        except Exception:                          # noqa: BLE001 - no sysfs / no such attribute
            return -1

    cpus, index, peers = allowed, local_rank, max(local_world, 1)
    node = node_of(local_rank)
    if node >= 0:
        try:
            local = set(_cpulist(open("/sys/devices/system/node/node%d/cpulist" % node).read())) & set(allowed)
        except OSError:
            local = set()
        same = [i for i in range(peers) if node_of(i) == node]     # the feeders sharing this node
        if len(local) >= min_cores * max(len(same), 1) and local_rank in same:
            cpus, index, peers = sorted(local), same.index(local_rank), len(same)
    per = len(cpus) // peers
    if per < min_cores:
        return None
    mine = cpus[index * per:(index + 1) * per]
    os.sched_setaffinity(0, mine)
    return mine
