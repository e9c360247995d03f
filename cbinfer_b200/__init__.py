"""cbinfer_b200 -- the pycbinfer surface on a B200-native (sm_100a) backend.

Mirrors the reference's ``pycbinfer/__init__.py``: ``convert`` (:91-94), ``convertRecur``
(:20-45), ``subsitute`` (:10-17), ``mergeReLURecur`` (:47-66), ``propChangeIndexesOf1x1``
(:68-77), ``clearMemory`` (:79-82), ``getStateTensors`` (:84-89), ``tuneThresholdParameters``
(:98-144) and the classes ``CBConv2d`` / ``CBPoolMax2d``.  Same names, argument meaning and
return types; the per-frame work runs in ``libcbinfer_sm100.so`` (include/cbinfer_b200.h).
"""
import torch
import torch.nn as nn

from . import conv2d_cg as _cg
from ._lib import CBinferError
from .conv2d import CBConv2d
from .conv2d import CBPoolMax2d
from .conv2d_cg import ChangeIndexes

__all__ = ['CBConv2d', 'CBPoolMax2d', 'ChangeIndexes', 'subsitute', 'convertRecur', 'mergeReLURecur',
           'propChangeIndexesOf1x1', 'clearMemory', 'getStateTensors', 'convert',
           'tuneThresholdParameters', 'convertPools', 'shareWorkspace', 'resetStreams',
           'setActiveStreams', 'trackStreamChanges', 'streamChangeCounts', 'setStreamThresholds',
           'streamThresholds', 'setStreamZones']

verbose = False


def _log(fmt, *args):
    if verbose:
        print(fmt % args if args else fmt)


def _is(node, cls):
    """exact-type test, as the reference does (subclasses of nn.Conv2d / nn.ReLU are left alone)"""
    return type(node) is cls


def subsitute(node, threshold=1e-1, finegrained=False):
    """(node, replaced?) - an exact nn.Conv2d becomes a CBConv2d sharing its parameters
    (reference __init__.py:10-17; the misspelt name is the reference's)."""
    if not _is(node, nn.Conv2d):
        return node, False
    _log('replacing conv2d')
    cb = CBConv2d(node, threshold)
    cb.finegrained = finegrained
    return cb, True


def convertRecur(m, ignoreList=[], threshold=1e-1, finegrained=False):
    """One conversion pass over the children of `m` (reference __init__.py:20-45): containers
    recurse, Dropout and every type in `ignoreList` disappear, convolutions are substituted; the
    result is a fresh nn.Sequential with the surviving child names.  Returns (model, changed?)."""
    dropped = tuple(ignoreList) + (nn.Dropout,)
    out, changed = nn.Sequential(), False
    for name, child in m.named_children():
        if _is(child, nn.Sequential):
            # (like the reference, the recursion does not forward `finegrained`, __init__.py:28)
            child, hit = convertRecur(child, ignoreList, threshold)
        elif type(child) in dropped:
            _log('removing node %s', type(child))
            changed = True
            continue
        else:
            child, hit = subsitute(child, threshold=threshold, finegrained=finegrained)
        out.add_module(name, child)
        changed = changed or hit
    if changed:
        # the reference converts again until nothing changes (__init__.py:43-44); the second
        # pass only ever merges ReLUs
        out = convert(out, ignoreList)
    return out, changed


def mergeReLURecur(m):
    """Fold an nn.ReLU that directly follows a CBConv2d into that layer's `withReLU` flag and drop
    it from the container (reference __init__.py:47-66)."""
    kids = list(m.named_children())
    out = nn.Sequential()
    for pos, (name, child) in enumerate(kids):
        if _is(child, nn.Sequential):
            out.add_module(name, mergeReLURecur(child))
            continue
        if _is(child, CBConv2d):
            follower = kids[pos + 1][1] if pos + 1 < len(kids) else None
            if _is(follower, nn.ReLU):
                child.withReLU = True
        elif _is(child, nn.ReLU) and pos > 0 and _is(kids[pos - 1][1], CBConv2d):
            _log('merging ReLU layer')
            continue
        out.add_module(name, child)
    return out


def propChangeIndexesOf1x1(rootModule):
    """reference __init__.py:68-77.  Its test `m.kernel_size == [1,1]` compares a tuple with a list
    and therefore never holds; the behaviour (nothing is enabled) is kept on purpose."""
    for seq in [c for c in rootModule.modules() if _is(c, nn.Sequential)]:
        before = None
        for layer in seq:
            if _is(layer, CBConv2d) and _is(before, CBConv2d) and layer.kernel_size == [1, 1]:
                _log('enabling propagation of change indexes for 1x1')
                before.propChangeIndexes = True
            before = layer
    return rootModule


def _cb_layers(net):
    return [c for c in net.modules() if type(c) in (CBConv2d, CBPoolMax2d)]


def clearMemory(net):
    """drop the per-layer state of every CB layer (reference __init__.py:79-82)"""
    for layer in _cb_layers(net):
        layer.clearMemory()


def resetStreams(net, streams):
    """Start a new sequence in some streams of a batched model, in place: every CB layer under `net`
    gets those streams' slices of its state set to what a cleared model starts from (+inf state,
    zero operand planes).  Their next frame is then computed exactly as by a freshly cleared model,
    while the other streams stay on the candidate path with their own change sets; nothing is freed,
    so captured CUDA graphs stay valid (DESIGN.md section 3.12).

    `net` must be the whole model the caller runs per frame: the argument needs every CB layer to
    start over together.  The first layer then sees every pixel of a reset stream change, and each
    layer after it receives all of them as candidates from the layer before; a layer left out would
    keep its state for those streams and, being on the candidate path, would never test the pixels
    its upstream neighbour does not hand on.

    `streams`: an iterable of stream indices (the mask is built on the host and copied with an
    ordinary asynchronous copy), or a bool / uint8 CUDA tensor [B] read on the device, which makes
    the call capturable in a CUDA graph.  Work is enqueued on the current stream.  A model that has
    not run yet has nothing to reset.  Fine-grained layers with state are not supported."""
    if isinstance(streams, torch.Tensor) and not streams.is_cuda:
        raise CBinferError("resetStreams: the stream mask must be a CUDA tensor (got one on %s)" % streams.device)
    segments = [seg for layer in _cb_layers(net) for seg in layer._resetSegments()]
    if not segments:
        return
    counts = set(buf.shape[0] for buf, _, _ in segments)
    if len(counts) != 1:
        raise CBinferError("resetStreams: the layers hold state of different batch sizes %s" % sorted(counts))
    B = counts.pop()
    dev = segments[0][0].device
    if isinstance(streams, torch.Tensor):
        mask = streams
        if mask.dim() != 1 or mask.numel() != B:
            raise CBinferError("resetStreams: a mask of shape %s for %d streams" % (tuple(mask.shape), B))
    else:
        idx = [int(i) for i in streams]
        bad = [i for i in idx if not 0 <= i < B]
        if bad:
            raise CBinferError("resetStreams: stream indices %s out of range for %d streams" % (bad, B))
        host = torch.zeros(B, dtype=torch.uint8)
        host[idx] = 1
        mask = host.to(dev, non_blocking=True)
    _cg.reset_streams(segments, mask)


def setActiveStreams(net, streams):
    """Select the streams of a batched model that have a new frame: from the next frame on, a stream
    that is not active is skipped.  The dense change scan of every plain-input CB layer (the first
    layer, and layers behind dense modules such as a torch.cat) neither reads its input slice nor
    writes its state and reports no change for it, so every later kernel leaves it alone too: its
    state and outputs stay exactly as they were, and its slice of the input frame may hold anything
    (need not be uploaded).  Layers fed a change set by an upstream CB layer ignore the mask.  With
    fixed thresholds, the result equals feeding the skipped streams their previous frame again
    (DESIGN.md section 3.13).

    `streams`: an iterable of active stream indices, a bool / uint8 CUDA tensor [B] (non-zero =
    active), or None.  The first call allocates one device uint8 [B] mask and hands it to every
    CBConv2d under `net`; later calls write into that same buffer on the current stream (a host
    index list is built on the host and copied asynchronously; a tensor is copied on the device, so
    that call can be captured in a CUDA graph), so graphs captured with the mask read what was last
    written before each replay.  An index list needs B: from the mask already set or from the
    layers' state, so the first call on a model that has not run takes a tensor.  None detaches the
    mask (every stream active again): graphs captured without a mask never see one, and graphs
    captured with it must not be replayed after detaching.  The mask's length must equal the
    frames' batch size (checked at forward).  Fine-grained layers and gatherComputationStats are
    not supported."""
    convs = [c for c in _cb_layers(net) if type(c) is CBConv2d]
    for c in convs:
        if c.finegrained or (c._auxPlanes is not None and c._auxPlanes[0] == 'fg'):
            raise CBinferError("setActiveStreams: a fine-grained layer's dense scan (cb_fg_detect) cannot "
                               "skip streams")
        if c.gatherComputationStats and streams is not None:
            raise CBinferError("setActiveStreams: gatherComputationStats reads the whole input")
    if streams is None:
        for c in convs:
            c._activeMask = None
        return
    buf = next((c._activeMask for c in convs if c._activeMask is not None), None)
    if isinstance(streams, torch.Tensor):
        if not streams.is_cuda:
            raise CBinferError("setActiveStreams: the stream mask must be a CUDA tensor (got one on %s)"
                               % streams.device)
        if streams.dim() != 1 or streams.dtype not in (torch.bool, torch.uint8):
            raise CBinferError("setActiveStreams: the mask must be a bool or uint8 tensor [B], got %s %s"
                               % (streams.dtype, tuple(streams.shape)))
        if buf is None or buf.numel() != streams.numel() or buf.device != streams.device:
            buf = torch.empty(streams.numel(), dtype=torch.uint8, device=streams.device)
        buf.copy_(streams)
    else:
        if buf is None:
            state = [c._inBuf for c in convs if c._inBuf is not None]
            if not state:
                raise CBinferError("setActiveStreams: the model has not run yet, so the number of streams is "
                                   "unknown; pass a CUDA mask tensor [B]")
            buf = torch.empty(state[0].shape[0], dtype=torch.uint8, device=state[0].device)
        B = buf.numel()
        idx = [int(i) for i in streams]
        bad = [i for i in idx if not 0 <= i < B]
        if bad:
            raise CBinferError("setActiveStreams: stream indices %s out of range for %d streams" % (bad, B))
        host = torch.zeros(B, dtype=torch.uint8)
        host[idx] = 1
        buf.copy_(host, non_blocking=True)
    for c in convs:
        c._activeMask = buf


def trackStreamChanges(net, enable=True, B=None):
    """Count, per video stream, the output pixels each CBConv2d under `net` recomputes.  After this,
    every frame writes ``counts[l, b]``: the number of output pixels of stream b that layer l (in
    ``net.modules()`` order) recomputed in that frame -- the layer's change count split by stream,
    written by the kernels that already produce that count, so no launch is added (DESIGN.md section
    3.14).  A stream skipped by the active-stream mask, or fed its previous frame again, gets 0 in
    every row; a stream started over by resetStreams gets H*W of each layer on its next frame.  If the
    last layer's count of stream b is 0, b's output is bit-identical to its previous frame.

    Allocates one device int32 [L, B] buffer (plus the kernels' accumulators) and hands each CBConv2d
    its row; returns the layers' qualified names in row order.  B comes from the argument or from the
    layers' state (as setActiveStreams takes it); a frame of another batch size raises at forward.
    The buffer (streamChangeCounts) is the same tensor every frame, so CUDA graphs captured after this
    call keep writing it.  enable=False detaches it.  Pools get no row; fine-grained layers on the
    planar path (gemmMode='simt') are not supported."""
    named = [(name, c) for name, c in net.named_modules() if type(c) is CBConv2d]
    convs = [c for _, c in named]
    if not enable:
        for c in convs:
            c._streamRow = None
        return []
    for c in convs:
        if c.finegrained and c.gemmMode == 'simt':
            raise CBinferError("trackStreamChanges: the planar fine-grained path (gemmMode='simt') does not "
                               "count changes per stream")
    state = [c._inBuf for c in convs if c._inBuf is not None]
    if B is None:
        if not state:
            raise CBinferError("trackStreamChanges: the model has not run yet, so the number of streams is "
                               "unknown; pass B")
        B = state[0].shape[0]
    B = int(B)
    if B < 1:
        raise CBinferError("trackStreamChanges: B = %d streams" % B)
    dev = state[0].device if state else next(net.parameters()).device
    if dev.type != "cuda":
        raise CBinferError("trackStreamChanges: the model is on %s; the counts live on a CUDA device" % dev)
    counts = torch.zeros(len(convs), B, dtype=torch.int32, device=dev)
    acc = torch.zeros(len(convs), B + 1, dtype=torch.int32, device=dev)    # zero at rest (the kernels keep it so)
    for l, c in enumerate(convs):
        c._streamRow = (counts, l, acc)
    return [name for name, _ in named]


def streamChangeCounts(net):
    """The device int32 [L, B] buffer of per-stream change counts of a model set up with
    trackStreamChanges: row l holds layer l's counts of the last frame.  Always the same tensor; read
    it after the frame's work (it is written on the stream the frame ran on)."""
    for c in net.modules():
        if type(c) is CBConv2d and c._streamRow is not None:
            return c._streamRow[0]
    raise CBinferError("streamChangeCounts: the model is not tracked (trackStreamChanges)")


def setStreamThresholds(net, table):
    """Give each video stream of a batched model its own change thresholds.  `table[l, b]` is the threshold
    of CBConv2d l (every CBConv2d under `net` in named_modules() order, the row order of
    trackStreamChanges) for stream b: wherever layer l's change detection runs -- its own kernel, an
    upstream pool or tile epilogue, the fused tail -- stream b's pixels are tested against it, rounded to
    the layer's data type as the scalar `threshold` is.  Stream b then computes exactly what the model
    computes with the scalar thresholds ``table[:, b]`` (DESIGN.md section 3.15).  Returns the layers'
    qualified names in row order.

    The first call allocates one device fp32 [L, B] table, starting from the threshold each layer's last
    detection used (its scalar before any frame), and hands every CBConv2d its row; later calls write into it on the current stream, so CUDA graphs
    captured with the table read the values it holds at each replay.  Raising a value, or writing the same
    value, takes effect in place.  LOWERING A VALUE RESTARTS THE STREAM when that row belongs to a layer
    that thresholds only the candidates an upstream layer hands on (candidateDetect, fed a change set in
    its last frame): pixels that no upstream change touches could now exceed the threshold, and only a
    full rescan would find them.  The call therefore decides on the device which streams had such a value
    lowered and resets them as resetStreams does, in the same enqueued work: their next frame is computed
    as by a freshly cleared model with the new thresholds, and the other streams are not touched.  Layers
    that scan their input densely every frame (plain input, no candidateDetect) never need this.

    `table`: host values (nested lists, a numpy array or a CPU tensor [L, B]; checked for shape and for
    NaN and infinite values, then copied asynchronously), or a CUDA fp32 tensor [L, B], copied on the
    device so that the call can be captured in a CUDA graph; a CUDA table is not checked for its values.
    B comes from the table attached already, else from the layers' state, else from `table`.  While a
    table is attached the scalar `threshold` is not read: a frame raises CBinferError if it was assigned
    since.  None detaches the table: each layer's next eager frame scans densely (the scalar threshold may
    have been lowered), and graphs captured with the table must not be replayed after detaching.
    Fine-grained layers and gatherComputationStats are not supported."""
    named = [(name, c) for name, c in net.named_modules() if type(c) is CBConv2d]
    convs = [c for _, c in named]
    if table is None:
        for c in convs:
            if c._thrRow is not None:
                c._thrRow = None
                c._lastThr = None
        return []
    for c in convs:
        if c.finegrained or (c._auxPlanes is not None and c._auxPlanes[0] == 'fg'):
            raise CBinferError("setStreamThresholds: fine-grained layers (cb_fg_detect) take one scalar threshold")
        if c.gatherComputationStats:
            raise CBinferError("setStreamThresholds: gatherComputationStats thresholds with the scalar threshold")
    L = len(convs)
    cur = next((c._thrRow[0] for c in convs if c._thrRow is not None), None)
    state = [c._inBuf for c in convs if c._inBuf is not None]
    if cur is not None:
        B, dev = cur.shape[1], cur.device
    elif state:
        B, dev = state[0].shape[0], state[0].device
    else:
        B, dev = None, next(net.parameters()).device
    if isinstance(table, torch.Tensor) and table.is_cuda:
        if table.dtype != torch.float32 or table.dim() != 2 or table.shape[0] != L \
                or (B is not None and table.shape[1] != B) or (dev.type == "cuda" and table.device != dev):
            raise CBinferError("setStreamThresholds: a CUDA fp32 table [%d, %s] on %s is needed, got %s %s on %s"
                               % (L, B if B is not None else "B", dev, table.dtype, tuple(table.shape), table.device))
        new, dev = table, table.device
    else:
        host = torch.as_tensor(table, dtype=torch.float32)
        if host.dim() != 2 or host.shape[0] != L or (B is not None and host.shape[1] != B):
            raise CBinferError("setStreamThresholds: a table [%d, %s] is needed, got %s"
                               % (L, B if B is not None else "B", tuple(host.shape)))
        if not bool(torch.isfinite(host).all()):
            raise CBinferError("setStreamThresholds: the table holds NaN or infinite values")
        new = None
    B = new.shape[1] if new is not None else host.shape[1]
    if B < 1:
        raise CBinferError("setStreamThresholds: B = %d streams" % B)
    if dev.type != "cuda":
        raise CBinferError("setStreamThresholds: the model is on %s; the table lives on a CUDA device" % dev)
    if new is None:
        new = host.to(dev, non_blocking=True)
    if cur is None:
        # the thresholds the layers' state was built with: the one each layer's last detection used, or
        # its scalar before any detection (then there is no state the table could make inexact)
        built = [c._lastThr if c._lastThr is not None else c.threshold for c in convs]
        cur = torch.tensor([float(t) for t in built], dtype=torch.float32).to(dev).unsqueeze(1) \
            .repeat(1, B).contiguous()
        for l, c in enumerate(convs):
            c._thrRow = (cur, l, c.threshold)
    # a stream restarts if a layer that tests only the candidates handed to it got a lower value
    fed = [l for l, c in enumerate(convs) if c.candidateDetect and c._lastPlain is False]
    segments = [seg for layer in _cb_layers(net) for seg in layer._resetSegments()]
    lowered = None
    if fed and segments and new is not cur:
        lowered = torch.stack([new[l] < cur[l] for l in fed]).any(0)
    if new is not cur:
        cur.copy_(new)
    if lowered is not None:
        _cg.reset_streams(segments, lowered)
    return [name for name, _ in named]


def streamThresholds(net):
    """The device fp32 [L, B] table of per-stream thresholds attached by setStreamThresholds: the same tensor
    until it is detached.  Write it through setStreamThresholds: a value lowered by writing into the tensor
    directly does not restart the streams that need it."""
    for c in net.modules():
        if type(c) is CBConv2d and c._thrRow is not None:
            return c._thrRow[0]
    raise CBinferError("streamThresholds: no per-stream thresholds are attached (setStreamThresholds)")


def setStreamZones(net, zones):
    """Exclude regions of each video stream's frame from change detection: a burned-in clock, a waving
    tree, a privacy mask.  The zone belongs to the frame-taking layer, the first CBConv2d under `net` in
    named_modules() order; its qualified name is returned.  `zones` is a bool or uint8 tensor [B, H, W]
    (non-zero = watched) on the host or on the model's CUDA device; None detaches it.

    While a zone is attached, that layer's dense change scan treats every pixel of stream b outside
    zones[b] as unchanged: it is not compared, and its state and operand planes are not written.  A pixel
    whose state holds +inf (never accepted: a fresh model, or a stream reset by resetStreams and not run
    since) is tested as usual.  Stream b then computes exactly what the model without a zone computes
    when each excluded pixel with a finite state is replaced by the value the first layer's state holds
    for it (DESIGN.md section 3.16).  Every later layer is driven by the first layer's change bits, so
    nothing else changes; a zone may be widened or narrowed between any two frames without a restart.

    The first call allocates one device bitmap (plus an int8 staging map); later calls with the same
    [B, H, W] rewrite that buffer on the current stream, so CUDA graphs captured after the first call read
    the zone as it is at each replay.  A host zone is uploaded with an ordinary asynchronous copy; a CUDA
    zone is converted on the device, which makes the call capturable.  The zone survives clearMemory.
    Frames of another B, H or W, frames wider than one 16-byte state pixel (> 4 fp32 or > 8 fp16 / bf16
    channels) and change sets handed to the zone layer raise at forward.  Fine-grained layers,
    gatherComputationStats and CPU models are not supported."""
    named = [(name, c) for name, c in net.named_modules() if type(c) is CBConv2d]
    if not named:
        raise CBinferError("setStreamZones: the model has no CBConv2d")
    name, first = named[0]
    if zones is None:
        first._zone = None
        return name
    if first.finegrained or (first._auxPlanes is not None and first._auxPlanes[0] == 'fg'):
        raise CBinferError("setStreamZones: a fine-grained layer's detection (cb_fg_detect) takes no zone")
    if first.gatherComputationStats:
        raise CBinferError("setStreamZones: gatherComputationStats reads the whole input")
    if not isinstance(zones, torch.Tensor) or zones.dim() != 3 or zones.dtype not in (torch.bool, torch.uint8):
        raise CBinferError("setStreamZones: a bool or uint8 tensor [B, H, W] is needed, got %s"
                           % ("%s %s" % (zones.dtype, tuple(zones.shape)) if isinstance(zones, torch.Tensor)
                              else type(zones).__name__))
    dev = first.weight.device
    if dev.type != "cuda":
        raise CBinferError("setStreamZones: the model is on %s; the zone lives on a CUDA device" % dev)
    if zones.is_cuda and zones.device != dev:
        raise CBinferError("setStreamZones: the zone is on %s, the model on %s" % (zones.device, dev))
    shape = tuple(zones.shape)
    if min(shape) < 1:
        raise CBinferError("setStreamZones: an empty zone %s" % (shape,))
    if first._zone is not None and first._zone[1] == shape:
        bits, _, stage = first._zone
    else:
        bits = torch.zeros(_cg.C.cb_bitmap_words(*shape), dtype=torch.int32, device=dev)
        stage = torch.empty(shape, dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        if zones.is_cuda:
            stage.copy_(zones)
        else:
            stage.copy_(zones.to(torch.int8), non_blocking=True)
        _cg.check(_cg.C.cb_map_to_bits(_cg.stream_ptr(dev), stage.data_ptr(), bits.data_ptr(), *shape))
    first._zone = (bits, shape, stage)
    return name


def getStateTensors(net):
    """all state tensors of the CB layers in forward order (reference __init__.py:84-89)"""
    return [t for layer in _cb_layers(net) for t in layer.getStateTensors()]


def shareWorkspace(net):
    """Let all CBConv2d layers of one model instance share one stream-K workspace (their launches
    are ordered).  Models that may run concurrently must not share: call this per instance."""
    holder = None
    for m in net.modules():
        if type(m) == CBConv2d:
            if holder is None:
                holder = m._wsHolder
            m._wsHolder = holder
    return net


def convert(m, ignoreList=[], threshold=1e-1):
    """nn.Conv2d -> CBConv2d, Dropout removed, ReLUs folded (reference __init__.py:91-94); returns an
    nn.Sequential with the original child names."""
    converted, _ = convertRecur(m, ignoreList=ignoreList, threshold=threshold)
    return shareWorkspace(mergeReLURecur(converted))


def convertPools(m):
    """Helper for the hand-written recipe of the reference (sceneLabeling/modelLoader.py:72-78):
    wrap every 2x2/stride-2 nn.MaxPool2d that directly follows a CBConv2d in CBPoolMax2d and let
    that conv propagate its change indexes.  Not part of the reference API (it does this by
    hand); returns a new nn.Sequential with the same child names."""
    mout = nn.Sequential()
    prev = None
    for name, node in m.named_children():
        if type(node) is nn.Sequential:
            node = convertPools(node)
        elif type(node) is nn.MaxPool2d and type(prev) is CBConv2d and not prev.finegrained:
            ks = node.kernel_size if isinstance(node.kernel_size, tuple) else (node.kernel_size,) * 2
            st = node.stride if isinstance(node.stride, tuple) else (node.stride,) * 2
            if ks == (2, 2) and st == (2, 2) and node.padding in (0, (0, 0)):
                prev.propChangeIndexes = True
                node = CBPoolMax2d(node)
        mout.add_module(name, node)
        prev = node
    return mout


def tuneThresholdParameters(vidSeqReader, evalSequences, numFramesPerSeq,
                            targetGenerator, preprocessor,
                            modelBaseline, modelTest, evaluator,
                            cbModuleList, lossToleranceList, initThreshold=1e-2, thresholdIncrFactor=1.2):
    """Greedy front-to-back threshold search (reference __init__.py:98-144).  Layer by layer: start
    at `initThreshold`, multiply by `thresholdIncrFactor` for as long as the summed loss over the
    evaluation sequences stays within that layer's tolerance of the loss before the layer was
    touched, then undo the last step.  A scalar tolerance applies to every layer."""
    tolerances = lossToleranceList if type(lossToleranceList) is list \
        else [lossToleranceList] * len(cbModuleList)
    assert len(tolerances) == len(cbModuleList)

    def summed_loss():
        clearMemory(modelTest)
        total = 0
        with torch.no_grad():
            for seq in evalSequences:
                frames, target = vidSeqReader.getDataFrames(seqName=seq, numFrames=numFramesPerSeq)
                if target is None:
                    target = targetGenerator(frames[-1])
                out = None
                for frame in frames:
                    out = modelTest(preprocessor(frame).cuda())
                total += evaluator(out, target)
        return total

    reference_loss = summed_loss()
    for pos, layer in enumerate(cbModuleList):
        _log('adjusting threshold for module %d of %d', pos + 1, len(cbModuleList))
        layer.threshold = initThreshold
        while True:
            layer.threshold *= thresholdIncrFactor
            loss = summed_loss()
            _log('. (%f < %f + %f)', loss, reference_loss, tolerances[pos])
            if loss - reference_loss > tolerances[pos]:
                layer.threshold /= thresholdIncrFactor
                break
        reference_loss = summed_loss()
    return modelTest
