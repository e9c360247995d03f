"""Per-frame runtime around a converted model: CUDA-graph replay and a copy/compute pipeline.

The reference drives its model with one python call per frame (`poseDetection/evalTools.py:37-49`:
``model(frame.cuda())``), paying ~10 launches and a host sync per layer.  Here a frame of the whole
model is ONE CUDA-graph replay (no host work between kernels), and `FramePipeline` overlaps the
host->device copy of frame t+1 and the device->host copy of result t-1 with the compute of frame t
on separate streams (H2D, compute, D2H), which is what bounds end-to-end throughput once the
kernels are fast: a 640x480 fp32 frame is 3.7 MB of PCIe traffic.
"""
import torch


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
    shared, so graphs replay strictly in submission order on the compute stream)."""

    def __init__(self, model, example_frame, depth=2):
        dev = example_frame.device
        assert dev.type == "cuda"
        self.model = model
        self.depth = depth
        self.compute = torch.cuda.Stream(dev)
        self.h2d = torch.cuda.Stream(dev)
        self.d2h = torch.cuda.Stream(dev)
        self.inputs = [example_frame.clone() for _ in range(depth)]
        cur = torch.cuda.current_stream(dev)
        self.compute.wait_stream(cur)
        with torch.cuda.stream(self.compute), torch.no_grad():
            probe = model(self.inputs[0])                 # allocates state on first use
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
        self.t = 0
        for e in self.in_free + self.out_done:
            e.record(self.compute)

    def submit(self, host_frame):
        """Queue one frame (pinned host tensor); returns the slot whose host result buffer will
        hold this frame's output once `wait(slot)` returns."""
        s = self.t % self.depth
        self.t += 1
        with torch.cuda.stream(self.h2d):
            self.h2d.wait_event(self.in_free[s])
            self.inputs[s].copy_(host_frame, non_blocking=True)
            self.in_ready[s].record(self.h2d)
        with torch.cuda.stream(self.compute):
            self.compute.wait_event(self.in_ready[s])
            self.compute.wait_event(self.out_done[s])      # previous D2H of this slot finished
            out = self.graphs[s].replay()
            self.in_free[s].record(self.compute)
            self.out_dev[s].copy_(out[0] if self._multi else out)
            self.out_ready[s].record(self.compute)
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(self.out_ready[s])
            self.out_host[s].copy_(self.out_dev[s], non_blocking=True)
            self.out_done[s].record(self.d2h)
        return s

    def reset(self, streams):
        """Start a new sequence in `streams` (see cbinfer_b200.resetStreams): enqueued on the compute
        stream, so it applies from the next `submit`ted frame on; frames already submitted are
        computed without it.  The captured graphs stay valid."""
        from . import resetStreams
        with torch.cuda.stream(self.compute):
            resetStreams(self.model, streams)

    def wait(self, slot):
        self.out_done[slot].synchronize()
        return self.out_host[slot]

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
