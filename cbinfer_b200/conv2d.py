"""CBConv2d / CBPoolMax2d -- the nn.Modules of the pycbinfer surface on the sm_100a backend.

Mirrors the reference's ``pycbinfer/conv2d.py``: class ``CBPoolMax2d`` (:24-84) and class
``CBConv2d`` (:87-304) with the same constructor arguments, flags (``withReLU``,
``saveChangeMap``, ``propChangeIndexes``, ``gatherComputationStats``, ``finegrained``,
``copyInput``, ``feedbackLoop``; :112-118), ``threshold`` attribute, state buffers
(``prevInput``, ``prevOutput``, ``outputState``), ``clearMemory()`` / ``getStateTensors()``,
``('changeIndexes', tensor, indices)`` tuple protocol (:180-187, :256-257) and ``__repr__``.

What is different underneath (B200-first, not a translation):
  * state lives pixel-major ([B,H,W,pitch], exposed as channels-last [B,C,H,W] views) so a changed
    pixel's channels are one contiguous run for detection, gather, scatter and pooling;
  * one frame of a layer is three launches -- detect, dilate+compact, fused gather/tcgen05
    contraction/bias/ReLU/scatter -- with the change count kept on the device: no torch.nonzero,
    no host sync, no X / Y / Y^T matrices (reference: ~10 launches + 1 sync, conv2d.py:222-251);
  * batch > 1 = independent video streams (the reference is batch 1);
  * CUDA only: the reference's CPU branches (conv2d.py:225-227,244-245,252-253) do not exist.
"""
import functools
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from . import conv2d_cg as cg
from .conv2d_cg import ChangeIndexes
from .conv2d_fg import cbconvFG

_INF = float("inf")


class DetectionDone(object):
    """Marker in the index slot of the ('changeIndexes', x, idx) tuple: the change detection of the
    CBConv2d `owner` already ran on x -- in CBConv2d.detectInput, or fused into the kernel of an
    upstream CBPoolMax2d or tile epilogue; its raw bitmap, state and operand planes are up to date.
    The owner records the detection when it takes the marker."""

    def __init__(self, owner, dense=False):
        self.owner = owner
        self.dense = dense        # True: a dense scan wrote every bitmap word (CBConv2d.detectInput)


class FrameDone(object):
    """Marker in the index slot of the tuple: the frame of `owner` already ran inside an upstream
    kernel.  For a CBPoolMax2d: the CBConv2d before it pooled in its tile epilogue and ran the
    detection of the layer after the pool there (cb_conv_update_tiled_pool).  For a CBConv2d: the
    1x1 layer before it ran its detection and contraction (cb_tail_update); `candidates` is the
    superset list both layers walked."""

    def __init__(self, owner, candidates=None):
        self.owner = owner
        self.candidates = candidates


def _checkOwner(marker, module):
    if marker.owner is not module:      # the work it reports was done for that module, not this one
        raise _lib.CBinferError("%s got a %s for another module" % (type(module).__name__, type(marker).__name__))


@functools.lru_cache(maxsize=None)
def _tiles_ok(dt, gemm, shape, Cin, Cout, filtSize, mode):
    sup = cg.tiled_supported(dt, gemm, shape, Cin, Cout, filtSize)
    return sup >= 1 if mode == 'on' else sup == 1


def _parse_input(inp):
    """tensor, or ('changeIndexes', tensor, indices) from an upstream CB layer (conv2d.py:180-187)."""
    if type(inp) == tuple:
        assert inp[0] == 'changeIndexes'
        return inp[1].detach(), inp[2]
    return inp.detach(), None


class CBPoolMax2d(nn.Module):
    def __init__(self, m):
        super(CBPoolMax2d, self).__init__()
        ks = m.kernel_size if isinstance(m.kernel_size, tuple) else (m.kernel_size,) * 2
        st = m.stride if isinstance(m.stride, tuple) else (m.stride,) * 2
        assert(ks == (2, 2) and st == (2, 2))
        self.stride = st
        self.kernel_size = ks
        self.ceil_mode = m.ceil_mode
        self.propChangeIndexes = False
        self.propPooledIndexes = False  # extension: hand pooled-resolution change candidates on
        self._fusedNext = None          # extension: [downstream CBConv2d] whose detection is fused in
        self.cloneOutput = True   # reference returns outputState.clone() (conv2d.py:73)
        self._outVersion = None   # outputState._version as the kernels last left it
        self.register_buffer('outputState', torch.empty(0))
        self.clearMemory()

    def __setstate__(self, state):
        # pickles of older versions may lack these: no fused neighbour, and the state counts as touched
        super(CBPoolMax2d, self).__setstate__(state)
        for name in ('_fusedNext', '_outVersion'):
            self.__dict__.setdefault(name, None)

    def clearMemory(self):
        self.outputState = self.outputState.new_empty(0)
        self._stateBuf = None
        self._scratch = None

    def getStateTensors(self):
        return [self.outputState]

    def _resetSegments(self):
        """The pooled map as a cg.reset_streams segment (+inf), if allocated."""
        if self._stateBuf is None:
            return []
        return [(self._stateBuf, self.outputState.shape[1], _INF)]

    def _pooled_size(self, h, w):
        if self.ceil_mode:
            return (h - 1) // 2 + 1, (w - 1) // 2 + 1
        return h // 2, w // 2

    def _stateAllocated(self, input_shape, dtype, device):
        """outputState is the pixel-major pooled map the kernels own for an input of `input_shape`
        (see CBConv2d._stateAllocated)."""
        B, nc, h, w = input_shape
        st = self.outputState
        return self._stateBuf is not None and tuple(st.shape) == (B, nc) + self._pooled_size(h, w) \
            and st.dtype == dtype and st.device == device and st.data_ptr() == self._stateBuf.data_ptr()

    def _stateTouched(self):
        """outputState written from outside the kernels since this pool last ran?"""
        return self._outVersion != self.outputState._version

    def _fusedPoolTarget(self, input_shape, dtype, device):
        """What an upstream CBConv2d on the tile path needs to pool inside its own epilogue and run the
        next layer's detection there (cb_conv_update_tiled_pool), or None when this pool's state is
        not allocated yet / was touched from outside, or the next layer's candidate-detection
        conditions do not hold (then the ordinary path runs and sets everything up)."""
        if not self._fusedNext or not self._stateAllocated(input_shape, dtype, device) or self._stateTouched():
            return None
        tgt = self._fusedNext[0]._fusedDetectTarget(tuple(self.outputState.shape), dtype, device)
        return None if tgt is None else dict(tgt, out=self.outputState)

    def forward(self, inp):
        assert(type(inp) == tuple and inp[0] == 'changeIndexes')
        input, handed = inp[1].detach(), inp[2]
        assert input.dim() == 4
        _lib.require_cuda(input)
        nxt = self._fusedNext[0] if self._fusedNext else None
        if isinstance(handed, FrameDone):
            # the producing CBConv2d already pooled its tiles and ran the next layer's detection inside
            # its epilogue (cb_conv_update_tiled_pool); that layer records it on taking the DetectionDone
            _checkOwner(handed, self)
            handOn = DetectionDone(nxt)
        else:
            handOn = self._pool(input, handed, nxt)
        output = self.outputState.clone() if self.cloneOutput else self.outputState
        return output if handOn is None else ('changeIndexes', output, handOn)

    def _pool(self, input, changeIndexes, nxt):
        """Pool the touched windows; returns what the output tuple hands on, or None (plain output)."""
        B, nc, h, w = input.shape
        oh, ow = self._pooled_size(h, w)
        if not isinstance(changeIndexes, ChangeIndexes):
            assert(changeIndexes.dim() == 1)
            changeIndexes = ChangeIndexes.from_tensor(changeIndexes, (B, h, w))
        if not self._stateAllocated(input.shape, input.dtype, input.device):
            # deviation (stated): the reference allocates only once a non-empty index list arrives
            # (conv2d.py:53-62); deciding that needs a host sync, so the state is allocated up front.
            self.outputState, self._stateBuf = cg.pixel_major((B, nc, oh, ow), input.dtype,
                                                              input.device, _INF)
            self._scratch = None
        # candidates handed downstream are complete only if neither the producer's output nor this
        # pool's state was written from outside the kernels (see CBConv2d.forward_normal)
        complete = changeIndexes.complete and not self._stateTouched()
        self._outVersion = self.outputState._version
        tgt = None
        if nxt is not None and complete and changeIndexes.bits is not None and input.stride(1) == 1:
            tgt = nxt._fusedDetectTarget((B, nc, oh, ow), input.dtype, input.device)
        if tgt is not None:
            # pooling + the next layer's detection in one kernel (cb_maxpool2x2_detect)
            cg.maxPool2d_detect(input, self.outputState, changeIndexes, tgt['next_state'], tgt['next_raw_bits'],
                                tgt['threshold'], tgt['mode'], aux=tgt['aux'], thr_b=tgt['thr_b'])
            return DetectionDone(nxt)
        cg.maxPool2d(input, self.outputState, changeIndexes, self.kernel_size, self.stride)
        if self.propPooledIndexes and changeIndexes.bits is not None:
            # extension (no reference counterpart): change candidates at the pooled resolution for
            # a downstream CBConv2d with candidateDetect=True
            if self._scratch is None:
                self._scratch = cg.alloc_scratch((B, oh, ow), input.device)
            s = self._scratch
            cg.pool_compact(changeIndexes.bits, (B, h, w), (B, oh, ow), s["idx"], s["count"], s["ws"],
                            out_bits=s["dil_bits"])
            pooled = ChangeIndexes(s["idx"], s["count"], (B, oh, ow), bits=s["dil_bits"])
            pooled.complete = complete
            return pooled
        if self.propChangeIndexes:
            # reference behaviour: the *input-resolution* indices are forwarded (conv2d.py:75-76)
            return changeIndexes
        return None

    def __repr__(self):
        s = ('{name} (k={kernel_size}, s={stride}, ceil_mode={ceil_mode}')
        s += ', propChgIdxs={propChangeIndexes}'
        s += ')'
        return s.format(name=self.__class__.__name__, **self.__dict__)


class CBConv2d(nn.Module):
    #: contraction arithmetic (see include/cbinfer_b200.h).  gemmMode 'auto': fp32 data -> 3xBF16
    #: split on the tensor cores (max rel. error ~2e-5, bar 1e-4), 16-bit data -> kind::f16 with
    #: fp32 accumulation.  'tc3x' = 3xTF32 (~2e-6), 'tc' = single-pass TF32, 'simt' = fp32 FFMA.
    GEMM_MODES = {'simt': _lib.GEMM_SIMT_F32, 'tc': _lib.GEMM_TC, 'tc3x': _lib.GEMM_TC_3X,
                  'bf16x3': _lib.GEMM_TC_BF16X3}

    def __init__(self, m, threshold):
        super(CBConv2d, self).__init__()

        assert(m.groups == 1 and m.transposed == False)
        assert(m.output_padding == (0, 0) and m.padding == (m.kernel_size[-2] // 2, m.kernel_size[-1] // 2))
        assert(m.dilation == (1, 1) and m.stride == (1, 1))
        self.groups = m.groups
        self.transposed = m.transposed
        self.output_padding = m.output_padding
        self.padding = m.padding
        self.dilation = m.dilation
        self.stride = m.stride
        self.kernel_size = m.kernel_size
        self.in_channels = m.in_channels
        self.out_channels = m.out_channels

        assert(m.weight is not None and m.bias is not None)
        self.weight = m.weight
        self.bias = m.bias

        self.threshold = threshold
        self._setDefaultValues()

        # neighbours whose work runs inside this layer's kernels (models.enableCandidateDetection):
        # [CBPoolMax2d] pooled in the tile epilogue, [CBConv2d] whose frame cb_tail_update runs too
        self._fusedPool = None
        self._fusedTail = None
        self._inVersion = None    # prevInput._version / prevOutput._version as the kernels last left them
        self._outVersion = None
        self._activeMask = None   # active-stream mask (cbinfer_b200.setActiveStreams), None = all
        # per-stream change counts (cbinfer_b200.trackStreamChanges): (counts int32 [L,B], this layer's
        # row l, accumulators int32 [L,B+1] zeroed once), or None = not tracked
        self._streamRow = None
        # per-stream thresholds (cbinfer_b200.setStreamThresholds): (table fp32 [L,B], this layer's row l, the
        # scalar threshold when the table was attached), or None = the scalar threshold for every stream
        self._thrRow = None
        # watched-pixel zone of the frame-taking layer (cbinfer_b200.setStreamZones): (bitmap int32
        # [B*H*Wd], (B, H, W), int8 staging map [B, H, W]), or None = every pixel watched
        self._zone = None
        self._lastPlain = None    # was the last frame's input plain (not a change set)?  None: no frame yet
        self._wsHolder = cg.ConvWorkspace()    # shared per model by pycbinfer.convert()
        self.register_buffer('prevInput', self.weight.data.new_empty(0))
        self.register_buffer('prevOutput', self.weight.data.new_empty(0))
        self.clearMemory()

    def _setDefaultValues(self):
        """The public flags and their defaults; sets those missing (pickles of older versions)."""
        for name, val in (('withReLU', False), ('saveChangeMap', False), ('propChangeIndexes', False),
                          ('gatherComputationStats', False), ('finegrained', False),
                          ('copyInput', True), ('feedbackLoop', False), ('gemmMode', 'auto'),
                          # extension: treat indices received from upstream as *candidates* for the
                          # thresholded detection instead of as the final change set (exact, see
                          # cb_change_detect_sparse)
                          ('candidateDetect', False),
                          # extension: (divisor, bias) applied to uint8 input frames inside the
                          # detection kernel
                          ('inputNorm', None),
                          # extension: 1x1 layer on the candidate path without any compaction (see
                          # forward_normal)
                          ('maskedConv', False),
                          # extension: contraction over dirty 8x16 output tiles (TMA-staged halo,
                          # implicit im2col) instead of the per-pixel gather: 'auto' = where the
                          # library recommends it (cb_conv_tiled_supported == 1; CBINFER_TILES=0
                          # disables), 'on' = wherever supported, 'off'
                          ('tileMode', 'auto')):
            if not(hasattr(self, name)):
                setattr(self, name, val)

    def __setstate__(self, state):
        # pickles of older versions lack what was added since: flags take their defaults, there are
        # no fused neighbours, and without a version record the state counts as touched
        super(CBConv2d, self).__setstate__(state)
        self._setDefaultValues()
        for name in ('_fusedPool', '_fusedTail', '_inVersion', '_outVersion', '_activeMask', '_streamRow', '_thrRow',
                     '_zone', '_lastPlain'):
            self.__dict__.setdefault(name, None)

    # ---- state ---------------------------------------------------------------------------
    def clearMemory(self):
        # reference: fill_(-1e100).resize_(0) (conv2d.py:147-148; raises on torch >= 1.x)
        self.prevInput = self.weight.data.new_empty(0)
        self.prevOutput = self.weight.data.new_empty(0)
        self._inBuf = None        # pixel-major storage behind prevInput / prevOutput
        self._outBuf = None
        self._auxPlanes = None    # fp32 only: operand planes of prevInput for the 3x modes
        self._scratch = None      # bitmaps, index list, count, compaction workspace
        self._packed = None       # (key, packed weights, fp32 bias)
        self._fresh = True        # state holds +inf: the next detection must be a full scan
        self._lastThr = None
        self._lastChanges = None
        self.changeMap = None
        self.compStats = None
        self._wsHolder.clear()

    def getStateTensors(self):
        return [self.prevInput, self.prevOutput]

    def _resetSegments(self):
        """The pixel-major state as cg.reset_streams segments: prevInput / prevOutput (+inf) and the
        operand planes of prevInput (0, what _aux builds from a +inf state), where allocated."""
        if (self.finegrained and self.prevInput.numel() > 0) or \
                (self._auxPlanes is not None and self._auxPlanes[0] == 'fg'):
            raise _lib.CBinferError("resetStreams: a fine-grained layer's first frame is a dense convolution "
                                    "of the whole batch; it cannot start one stream over")
        if self._inBuf is None:
            return []
        segs = [(self._inBuf, self.in_channels, _INF), (self._outBuf, self.out_channels, _INF)]
        if self._auxPlanes is not None and self._auxPlanes[0] == 'tf32':
            segs.append((self._auxPlanes[1].permute(0, 2, 3, 1), self.in_channels, 0))
        elif self._auxPlanes is not None and self._auxPlanes[0] == 'bf16':
            segs += [(plane, self.in_channels, 0) for plane in self._auxPlanes[1:]]
        return segs

    def _stateAllocated(self, shape, dtype, device):
        """Rule 1, first half: are prevInput / prevOutput the state the kernels own for an input of
        `shape`, allocated for it and still aliasing _inBuf / _outBuf?  (model.half() / .to() on a
        warm model replace the registered buffers with tensors that do not.)  Else: reallocate."""
        B, _, H, W = shape
        for t, buf, want in ((self.prevInput, self._inBuf, tuple(shape)),
                             (self.prevOutput, self._outBuf, (B, self.out_channels, H, W))):
            if buf is None or tuple(t.shape) != want or t.dtype != dtype or t.device != device \
                    or t.data_ptr() != buf.data_ptr():
                return False
        return True

    def _stateTouched(self):
        """Rule 1, second half: (prevInput, prevOutput) written from outside the kernels since this
        layer last ran?  The reference's eval scripts snapshot and restore getStateTensors() with
        copy_ (poseDetection/eval03.py:87-95): torch bumps the tensor version, the kernels do not."""
        return self._inVersion != self.prevInput._version, self._outVersion != self.prevOutput._version

    def _candidatesExact(self, shape, dtype, device):
        """Rule 2: may this frame threshold only the candidate pixels (cb_change_detect_sparse)?  Exact
        while the state is the kernels' own, untouched, not fresh, and the threshold not lowered:
        every other pixel then still lies within the threshold of the state.  With per-stream
        thresholds attached, a stream whose value was lowered is started over by setStreamThresholds
        itself, so the scalar comparison does not apply."""
        return self.candidateDetect and not self.finegrained and not self._fresh \
            and self._lastThr is not None and (self._thrRow is not None or self.threshold >= self._lastThr) \
            and self._stateAllocated(shape, dtype, device) and not any(self._stateTouched())

    def _recordDetection(self):
        """This layer's detection ran with its threshold (here or inside an upstream kernel).  The
        state's version is recorded where a frame ends (_frameDone, detectInput)."""
        self._fresh = False
        self._lastThr = self.threshold

    def _frameDone(self, changes, handOn):
        """Record the versions the kernels left and the frame's change list; return the output."""
        self._inVersion = self.prevInput._version
        self._outVersion = self.prevOutput._version
        self._lastChanges = changes
        if handOn is None:
            return self.prevOutput
        return 'changeIndexes', self.prevOutput, handOn

    def _gemm(self, dtype):
        if self.gemmMode == 'auto':
            return _lib.GEMM_TC_BF16X3 if dtype == torch.float32 else _lib.GEMM_TC
        g = self.GEMM_MODES[self.gemmMode]
        if g in (_lib.GEMM_TC_3X, _lib.GEMM_TC_BF16X3) and dtype != torch.float32:
            g = _lib.GEMM_TC
        return g

    def _aux(self, gemm):
        """Auxiliary operand planes of prevInput for the 3x modes, in the ops' `aux` format (kept in
        step by the detection kernel); (re)built from prevInput when the mode changes or after a
        plain copy."""
        want = {_lib.GEMM_TC_3X: 'tf32', _lib.GEMM_TC_BF16X3: 'bf16'}.get(gemm) \
            if self.prevInput.dtype == torch.float32 else None
        if want is None:
            self._auxPlanes = None
        elif self._auxPlanes is None or self._auxPlanes[0] != want:
            if want == 'tf32':
                lo, _ = cg.pixel_major(self.prevInput.shape, torch.float32, self.prevInput.device, 0)
                fin = torch.isfinite(self.prevInput)
                lo.copy_(torch.where(fin, cg.tf32_lo(torch.where(fin, self.prevInput, 0)), 0))
                self._auxPlanes = ('tf32', lo)
            else:
                self._auxPlanes = ('bf16',) + cg.bf16_planes(
                    torch.nan_to_num(self._inBuf, posinf=0.0, neginf=0.0), self.in_channels)
        return self._auxPlanes

    def _fusedDetectTarget(self, shape, dtype, device):
        """What an upstream CBPoolMax2d needs to run this layer's detection inside its own kernel,
        or None when candidate detection is not exact for this layer this frame."""
        if not self._candidatesExact(shape, dtype, device) or not self._scratch.get("raw_clear", False):
            return None
        gemm, _, _ = self._weights(dtype, device)
        return dict(next_state=self.prevInput, next_raw_bits=self._scratch["raw_bits"],
                    threshold=self.threshold, thr_b=self._thrB(shape[0]),
                    mode=_lib.UPDATE_CHANGED if self.feedbackLoop else _lib.UPDATE_ALL,
                    aux=self._aux(gemm))

    def _weights(self, dtype, device):
        gemm = self._gemm(dtype)
        key = (self.weight.data_ptr(), self.weight._version, self.bias.data_ptr(),
               self.bias._version, dtype, gemm, str(device))
        if self._packed is None or self._packed[0] != key:
            w = self.weight.detach().to(device=device, dtype=dtype)
            self._packed = (key, cg.pack_weights(w, gemm),
                            self.bias.detach().to(device=device, dtype=torch.float32).contiguous())
        return gemm, self._packed[1], self._packed[2]

    # ---- fine-grained path (conv2d.py:160-176) ---------------------------------------------
    def forward_fg(self, inp):
        """Reference flow: the first frame is a dense convolution (:163-167); afterwards every input
        VALUE whose change exceeds the threshold pushes W*delta into (a clone of) prevOutput
        (cbconvFG, :169-170) and prevInput = input (:175).  Here: per-value thresholded delta planes
        (cb_fg_detect) -> touched output pixels (cb_dilate_compact) -> accumulating tcgen05
        contraction over them (cb_conv_accumulate); gemmMode='simt' keeps the scattered
        red.global.add kernel on planar tensors (cb_fg_update, exact fp32 products)."""
        input = inp.detach()
        _lib.require_cuda(input)
        if input.dtype != torch.float32:
            raise _lib.CBinferError("the fine-grained path is fp32 only (as in the reference)")
        if self.gemmMode == 'simt':
            if self._streamRow is not None:
                raise _lib.CBinferError("per-stream change counts are not supported on the planar fine-grained "
                                        "path (gemmMode='simt')")
            return self._forward_fg_planar(input.contiguous())
        B, _, H, W = input.shape
        rows = self._streams(B)
        dev = input.device
        outpSize = (B, self.out_channels, H, W)
        gemm = _lib.GEMM_TC_BF16X3
        key = (self.weight.data_ptr(), self.weight._version, 'fg', str(dev))
        if self._packed is None or self._packed[0] != key:
            self._packed = (key, cg.pack_weights(self.weight.detach().to(device=dev, dtype=torch.float32), gemm),
                            None)
        if not self._stateAllocated(input.shape, torch.float32, dev) \
                or self._auxPlanes is None or self._auxPlanes[0] != 'fg':
            self.prevOutput, self._outBuf = cg.pixel_major(outpSize, torch.float32, dev, 0)
            self.prevOutput.copy_(F.conv2d(input, self.weight.detach(),
                                           padding=tuple(s // 2 for s in self.weight.size()[2:]),
                                           bias=self.bias.detach()))
            self.prevInput, self._inBuf = cg.pixel_major(input.shape, torch.float32, dev, 0)
            self.prevInput.copy_(input)
            p16 = _lib.C.cb_plane_pitch16(self.in_channels)
            # the thresholded delta planes (hi, lo) of the last frame
            self._auxPlanes = ('fg', (torch.zeros(B, H, W, p16, dtype=torch.bfloat16, device=dev),
                                      torch.zeros(B, H, W, p16, dtype=torch.bfloat16, device=dev)))
            self._scratch = cg.alloc_scratch((B, H, W), dev)
            self._scratch["nvalues"] = torch.zeros(1, dtype=torch.int32, device=dev)
            if rows is not None:
                rows[0].fill_(H * W)              # the dense first frame computes every output pixel
        else:
            s = self._scratch
            _, planes = self._auxPlanes
            cg.fg_detect(input, self.prevInput, self._inBuf, planes, s["raw_bits"], self.threshold,
                         count=s["nvalues"])
            cg.dilate_compact(s["raw_bits"], (B, H, W), self.kernel_size, s["idx"], s["count"], s["ws"],
                              dil_bits=s["dil_bits"], streams=rows)
            changes = ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])
            cg.conv_accumulate(planes, changes, self._packed[1], self._outBuf, self.in_channels,
                               self.out_channels, self.kernel_size, gemm, ws=self._wsHolder.get(dev))
            self._lastChanges = changes
        # the reference updates a clone (:169), so outputs handed out earlier stay as they were
        return F.relu(self.prevOutput) if self.withReLU else self.prevOutput.clone()

    def _forward_fg_planar(self, input):
        if self.prevInput.size() != input.size() or not self.prevInput.is_contiguous() \
                or not self.prevOutput.is_contiguous():
            # init prevOutput with a dense convolution, as the reference does (conv2d.py:163-167)
            self.prevOutput = F.conv2d(input, self.weight.detach(),
                                       padding=tuple(s // 2 for s in self.weight.size()[2:]),
                                       bias=self.bias.detach()).contiguous()
            self.prevInput = input.clone()
            self._inBuf = self._outBuf = None
        else:
            po = self.prevOutput.clone()                     # conv2d.py:169
            # also performs prevInput = input (conv2d.py:175) in the same pass
            self.prevOutput = cbconvFG(input, self.prevInput, po, self.weight, self.threshold)
        outp = self.prevOutput
        if self.withReLU:
            outp = F.relu(outp)
        return outp

    # ---- coarse-grained path (conv2d.py:178-259) ---------------------------------------------
    def forward_normal(self, inp):
        input, handed = _parse_input(inp)
        assert(input.dim() == 4)
        assert(input.size(-3) == self.in_channels)
        _lib.require_cuda(input)
        # `handed`: nothing (a plain frame), the upstream layer's change list, or a marker that an
        # upstream kernel already ran part of this frame.  This layer records that work itself: the
        # upstream module read its state (_fusedDetectTarget, _tailTarget) right before the launch,
        # nothing since reads _fresh or _lastThr, and kernels bump no tensor versions.
        # (a DetectionDone for the zone layer reports its own dense scan: nothing runs upstream of it)
        if self._zone is not None and handed is not None and not isinstance(handed, DetectionDone):
            raise _lib.CBinferError("the zone layer (setStreamZones) takes plain frames; it was handed a change set")
        if isinstance(handed, (DetectionDone, FrameDone)):
            _checkOwner(handed, self)
            self._recordDetection()
        if isinstance(handed, FrameDone):
            # cb_tail_update ran this layer's detection and contraction too; it split the operands on
            # the fly, so this layer's operand planes are stale
            self._auxPlanes = None
            self._lastPlain = False
            return self._frameDone(handed.candidates, handed.candidates if self.propChangeIndexes else None)
        B, _, H, W = input.shape
        dev, dt = input.device, input.dtype
        rows = self._streams(B)
        self._thrB(B)             # (a table of another batch size raises before any state is touched)
        detected = isinstance(handed, DetectionDone)
        upstream = None           # the upstream layer's change list
        if handed is not None and not detected:
            assert(handed.dim() == 1)
            upstream = handed if isinstance(handed, ChangeIndexes) \
                else ChangeIndexes.from_tensor(handed.detach(), (B, H, W))
        # a layer fed with plain frames re-scans them densely every frame, which rewrites every word of
        # its raw bitmap: nothing ever ORs bits into it, so its compaction need not zero it afterwards
        plain_input = handed is None or (detected and handed.dense)
        self._lastPlain = plain_input
        # uint8 frames (decoder output) are normalised inside the detection kernel:
        # value = u8 / divisor + bias with inputNorm = (divisor, bias); the layer computes in fp32
        u8norm = None
        if dt == torch.uint8:
            u8norm = self.inputNorm
            if u8norm is None:
                raise _lib.CBinferError("uint8 input needs CBConv2d.inputNorm = (divisor, bias), e.g. "
                                        "(255.0, 0.0) for the scene reader's frame/255")
            if upstream is not None or self.gatherComputationStats or self.in_channels > 4:
                input = input.float().div(u8norm[0]).add(u8norm[1])     # rare paths: plain fp32
                u8norm = None
            dt = torch.float32
        self._zoneBits(input.shape, dt)  # (a frame the zone does not fit raises before any state is touched)

        if not self._stateAllocated(input.shape, dt, dev):
            # a fresh output map needs every pixel recomputed: the input state goes too
            self.prevInput, self._inBuf = cg.pixel_major(input.shape, dt, dev, _INF)                 # :192-194
            self.prevOutput, self._outBuf = cg.pixel_major((B, self.out_channels, H, W), dt, dev, _INF)  # :195-199
            self._auxPlanes = None
            self._scratch = None
            self._fresh = True
        # a touched prevInput is treated as fresh (dense scan, operand planes rebuilt); a touched
        # prevOutput makes this frame's index list an incomplete candidate set for the next layer
        in_touched, ext_out = self._stateTouched()
        if in_touched:
            self._fresh = True
            self._auxPlanes = None
        if self._scratch is None:
            self._scratch = cg.alloc_scratch((B, H, W), dev, want_map=self.saveChangeMap)
        if self.saveChangeMap and "dil_map" not in self._scratch:
            self._scratch["dil_map"] = torch.zeros(B, H, W, dtype=torch.int8, device=dev)
        s = self._scratch

        if self.gatherComputationStats:
            if self._zone is not None:
                raise _lib.CBinferError("gatherComputationStats reads the whole input: it cannot be combined "
                                        "with a zone (setStreamZones)")
            if self._activeMask is not None:
                raise _lib.CBinferError("gatherComputationStats reads the whole input: it cannot be combined "
                                        "with an active-stream mask (setActiveStreams)")
            self._gatherStats(input)

        gemm, packed, bias32 = self._weights(dt, dev)
        tail = self._tryTail(input, upstream, gemm, packed, bias32)
        if tail is not None:
            return tail
        aux = self._aux(gemm)

        use_tiles = self._useTiles(dt, gemm, (B, H, W))
        # a directly following CBPoolMax2d (+ the detection of the layer after it) rides along in the
        # tile kernel's epilogue when everything is warmed up (cb_conv_update_tiled_pool); nobody
        # then needs this layer's ordered index list, so it is only compacted on demand
        pool_args = None
        if use_tiles and self._fusedPool and self.propChangeIndexes and not ext_out \
                and os.environ.get("CBINFER_FUSE_POOL", "1") != "0" \
                and _lib.C.cb_conv_tiled_pool_supported(_lib.dtype_code(dt), gemm, self.out_channels):
            pool_args = self._fusedPool[0]._fusedPoolTarget((B, self.out_channels, H, W), dt, dev)
        # the upstream list as this frame's detection candidates, where that is exact
        candidates = upstream if self.candidateDetect and upstream is not None \
            and tuple(upstream.shape) == (B, H, W) and upstream.complete \
            and self._candidatesExact(input.shape, dt, dev) else None

        mask = None
        tiled = False             # this frame's contraction walks the dirty-tile list
        if upstream is None or self.candidateDetect:
            # reference: detect (feedback updates prevInput at changed pixels, :222-224), nonzero
            # (:232), then prevInput.copy_(input) when not in feedback mode (:234-238).  Here the
            # copy is part of the detection pass; copyInput=False (alias the input as state) is
            # honoured as a copy -- the state always owns its memory.
            sparse_next = self.candidateDetect and not plain_input
            changes, mask = (None, None) if detected else \
                self._detect(input, candidates, u8norm, aux, gemm, use_tiles, sparse_next)
            if changes is None:
                changes = self._compact(s, B, H, W, sparse_next, tiles=use_tiles,
                                        lazy=pool_args is not None and not self.saveChangeMap)
                tiled = use_tiles
        else:
            # the upstream list is this frame's change set (reference behaviour)
            if tuple(upstream.shape) != (B, H, W):
                # e.g. a CBPoolMax2d with the reference's propChangeIndexes forwards INPUT-resolution
                # indices (conv2d.py:75-76): using them here would scatter out of bounds
                raise _lib.CBinferError("change indexes refer to a %s grid, this layer's map is %s"
                                        % (tuple(upstream.shape), (B, H, W)))
            changes = upstream
            if rows is not None:
                cg.stream_bucket(changes, (B, H, W), rows)
            if not self.feedbackLoop:
                self.prevInput.copy_(input)                                            # :234-236
                self._auxPlanes = None
                aux = self._aux(gemm)
            # (with feedbackLoop the reference never refreshes prevInput here either, :220,234)

        if tiled:
            # spatially clustered change sets: contraction over the dirty 8x16 tiles (TMA-staged
            # halo, implicit im2col through the UMMA descriptors), rows masked by the dilated bitmap
            cg.conv_update_tiled(self._inBuf, s["tile_ws"], s["dil_bits"], packed, bias32, self._outBuf,
                                 self.in_channels, self.out_channels, self.kernel_size, self.withReLU,
                                 gemm, aux=aux, pool=pool_args)                             # :242-251
        else:
            cg.conv_update(self._inBuf, changes, packed, bias32, self._outBuf, self.in_channels,
                           self.out_channels, self.kernel_size, self.withReLU, gemm,
                           aux=aux, ws=self._wsHolder.get(dev), mask=mask)                 # :242-251
        changes.complete = not ext_out
        if tiled and pool_args is not None:
            return self._frameDone(changes, FrameDone(self._fusedPool[0]))     # the epilogue did its frame
        return self._frameDone(changes, changes if self.propChangeIndexes else None)

    def _detect(self, input, candidates, u8norm, aux, gemm, use_tiles, sparse_next):
        """Dense scan, or the test of the `candidates` only.  Returns (change list if the launch
        built one, mask of the masked contraction), each or both None.  `sparse_next`: this layer
        is fed change sets, so its bitmap is left clear for the next candidate test, and a dense scan
        covers every stream (see setActiveStreams); else the dense scan skips inactive streams."""
        B, _, H, W = input.shape
        s = self._scratch
        mode = _lib.UPDATE_CHANGED if self.feedbackLoop else _lib.UPDATE_ALL
        active = None if sparse_next else self._streamMask(B)
        thr_b = self._thrB(B)
        # extension: no compaction at all for a 1x1 layer on the candidate path - the
        # contraction walks the candidate list and skips pixels whose raw bit is not set
        # (cb_conv_update_masked); this layer's own index list is then never materialised
        masked = (candidates is not None and tuple(self.kernel_size) == (1, 1) and self.maskedConv
                  and not self.saveChangeMap and gemm != _lib.GEMM_SIMT_F32)
        changes = mask = None
        if candidates is not None and not masked and not use_tiles and not self.saveChangeMap \
                and input.stride(1) == 1 and self._smallMap(B, H, W):
            # small map: candidate detection + dilation + ordered compaction in ONE launch (the
            # last block of the detection kernel compacts), cb_change_detect_sparse_compact
            if "sdc_sync" not in s:
                s["sdc_sync"] = torch.zeros(1, dtype=torch.int32, device=input.device)
            cg.detect_sparse_compact(input, self.prevInput, s["raw_bits"], self.threshold, mode, candidates,
                                     self.kernel_size, s["idx"], s["count"], s["sdc_sync"], aux=aux,
                                     bits_are_clear=s.get("raw_clear", False), dil_bits=s["dil_bits"],
                                     clear_raw=sparse_next, streams=self._streams(B), thr_b=thr_b)
            s["raw_clear"] = sparse_next
            changes = ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])
        elif candidates is not None:
            cg.detect_sparse(input, self.prevInput, s["raw_bits"], self.threshold, mode,
                             candidates, aux=aux,
                             bits_are_clear=s.get("raw_clear", False), thr_b=thr_b)
            if masked:
                if "mask_sync" not in s:
                    s["mask_sync"] = torch.zeros(2, dtype=torch.int32, device=input.device)
                mask = dict(bits=s["raw_bits"], clear=True, count=s["count"], sync=s["mask_sync"],
                            streams=self._streams(B))
                s["raw_clear"] = True                # the masked contraction clears the bitmap
                changes = ChangeIndexes(candidates.buffer, candidates.count, (B, H, W), bits=None)
                changes.superset = True
        elif u8norm is not None:
            cg.detect_u8(input, self.prevInput, s["raw_bits"], self.threshold, mode,
                         u8norm[0], u8norm[1], aux=aux, active=active, thr_b=thr_b,
                         zone=self._zoneBits(input.shape, torch.float32))
        else:
            cg.detect(input, self.prevInput, s["raw_bits"], self.threshold, mode, aux=aux, active=active, thr_b=thr_b,
                      zone=self._zoneBits(input.shape, input.dtype))
        self._recordDetection()
        return changes, mask

    def _streams(self, B):
        """This layer's per-stream counts row for a frame of B streams, as (counts int32 [B], accumulator
        int32 [B+1]), or None when the model is not tracked (cbinfer_b200.trackStreamChanges)."""
        if self._streamRow is None:
            return None
        counts, l, acc = self._streamRow
        if counts.shape[1] != B:
            raise _lib.CBinferError("per-stream change counts of %d streams, the frame has %d (trackStreamChanges)"
                                    % (counts.shape[1], B))
        return counts[l], acc[l]

    def _thrB(self, B):
        """This layer's row of per-stream thresholds (fp32 [B] on the device) for a frame of B streams, or
        None when no table is attached (cbinfer_b200.setStreamThresholds)."""
        if self._thrRow is None:
            return None
        table, l, _ = self._thrRow
        if table.shape[1] != B:
            raise _lib.CBinferError("per-stream thresholds of %d streams, the frame has %d (setStreamThresholds)"
                                    % (table.shape[1], B))
        return table[l]

    def _zoneBits(self, shape, dtype):
        """The zone bitmap for a frame of `shape` whose state has `dtype`, or None when no zone is attached
        (cbinfer_b200.setStreamZones).  A frame the zone does not fit raises."""
        if self._zone is None:
            return None
        bits, zshape, _ = self._zone
        B, C_, H, W = shape
        if (B, H, W) != zshape:
            raise _lib.CBinferError("the zone (setStreamZones) is [B, H, W] = %s, the frame is %s" % (list(zshape), [B, H, W]))
        if C_ * torch.empty(0, dtype=dtype).element_size() > 16:
            raise _lib.CBinferError("a zone (setStreamZones) needs a frame of at most one 16-byte state pixel; "
                                    "this one has %d %s channels" % (C_, dtype))
        return bits

    def _checkThresholds(self):
        """Refuse what a frame with per-stream thresholds attached cannot honour."""
        if self._thrRow is None:
            return
        if self.finegrained:
            raise _lib.CBinferError("per-stream thresholds are not supported on a fine-grained layer")
        if self.gatherComputationStats:
            raise _lib.CBinferError("gatherComputationStats thresholds the whole input with the scalar threshold: "
                                    "it cannot be combined with per-stream thresholds (setStreamThresholds)")
        if self.threshold != self._thrRow[2]:
            raise _lib.CBinferError("CBConv2d.threshold was assigned while per-stream thresholds are attached; the "
                                    "kernels read the table (setStreamThresholds), so the assignment would do nothing")

    def _streamMask(self, B):
        """The active-stream mask for a frame of B streams, or None when none is set."""
        m = self._activeMask
        if m is not None and m.numel() != B:
            raise _lib.CBinferError("active-stream mask of %d streams, the frame has %d (setActiveStreams)"
                                    % (m.numel(), B))
        return m

    # ---- two chained 1x1 layers in one launch (extension) ------------------------------------------
    def _tailReady(self, shape, dtype, device):
        """May this masked 1x1 layer's frame run inside cb_tail_update?"""
        return self.maskedConv and tuple(self.kernel_size) == (1, 1) and not self.saveChangeMap \
            and not self.gatherComputationStats and self._candidatesExact(shape, dtype, device) \
            and self._scratch.get("raw_clear", False)

    def _tailTarget(self, shape, dt, dev, feedback):
        """What the 1x1 layer feeding this one needs to run this layer's frame inside its own kernel
        (cb_tail_update), or None when that does not apply to this layer this frame."""
        if self.feedbackLoop != feedback or not self._tailReady(shape, dt, dev):
            return None
        gemm, packed, bias32 = self._weights(dt, dev)
        return dict(gemm=gemm, packed=packed, bias=bias32, state=self._inBuf, out=self._outBuf,
                    thr=self.threshold, thr_b=self._thrB(shape[0]), relu=self.withReLU, count=self._scratch["count"])

    def _tryTail(self, input, changeIndexes, gemm, packed, bias32):
        if not self._fusedTail or os.environ.get("CBINFER_FUSE_TAIL", "1") == "0" \
                or not isinstance(changeIndexes, ChangeIndexes) or input.dtype != torch.float32:
            return None
        B, C0, H, W = input.shape
        if tuple(changeIndexes.shape) != (B, H, W) or not changeIndexes.complete \
                or not self._tailReady(input.shape, input.dtype, input.device):
            return None
        nxt = self._fusedTail[0]
        C1, C2 = self.out_channels, nxt.out_channels
        if not _lib.C.cb_tail_supported(_lib.dtype_code(input.dtype), gemm, C0, C1, C2):
            return None
        # the input must be the upstream layer's pixel-major map itself (pitch == channels)
        if input.stride() != (H * W * C0, 1, W * C0, C0) or self._inBuf.shape[3] != C0 \
                or self._outBuf.shape[3] != C1:
            return None
        tgt = nxt._tailTarget((B, C1, H, W), input.dtype, input.device, self.feedbackLoop)
        if tgt is None or tgt['gemm'] != gemm:
            return None
        rows1, rows2 = self._streams(B), nxt._streams(B)
        if (rows1 is None) != (rows2 is None):      # one kernel writes both rows or neither
            return None
        s = self._scratch
        if "tail_sync" not in s:
            s["tail_sync"] = torch.zeros(4, dtype=torch.int32, device=input.device)
        x_buf = input.permute(0, 2, 3, 1)
        cg.tail_update(x_buf, self._inBuf, packed, bias32, self._outBuf, self.withReLU, self.threshold,
                       tgt['state'], tgt['packed'], tgt['bias'], tgt['out'], tgt['relu'], tgt['thr'],
                       changeIndexes, C0, C1, C2,
                       _lib.UPDATE_CHANGED if self.feedbackLoop else _lib.UPDATE_ALL,
                       s["count"], tgt['count'], s["tail_sync"], streams1=rows1, streams2=rows2,
                       thr1_b=self._thrB(B), thr2_b=tgt['thr_b'])
        # the kernel splits its operands on the fly: this layer's operand planes are stale now
        self._auxPlanes = None
        self._recordDetection()
        sup = ChangeIndexes(changeIndexes._buffer, changeIndexes.count, (B, H, W), bits=changeIndexes.bits,
                            ws=changeIndexes._ws, listed=changeIndexes.listed)
        sup.superset = True
        return self._frameDone(sup, FrameDone(nxt, sup))

    def lastChangeIndexes(self):
        """This frame's change indexes as an int32 tensor (ascending b*H*W + y*W + x): what the
        reference hands on as ``changeIndexes`` (conv2d.py:256-257).  The list of a layer on the
        tile path is compacted only now, on demand."""
        ci = self._lastChanges
        if ci is None:
            raise _lib.CBinferError("no frame processed yet")
        return ci.tensor() if isinstance(ci, ChangeIndexes) else ci

    def detectInput(self, input):
        """Run only this layer's (dense) change detection on `input` and return the tuple that makes
        the following ``forward`` skip it: ``model(first.detectInput(frame))``.  Lets a pipeline read
        every frame where it lies (e.g. straight from a decoder's output buffer) while the rest of
        the model replays as one CUDA graph captured on that tuple - no copy into a static input
        tensor.  Needs a warmed-up layer (state allocated by an ordinary forward of this shape)."""
        input = input.detach()
        _lib.require_cuda(input)
        dt = torch.float32 if input.dtype == torch.uint8 else input.dtype
        if self.finegrained or self.gatherComputationStats \
                or not self._stateAllocated(input.shape, dt, input.device):
            raise _lib.CBinferError("detectInput: run one ordinary forward of this input shape first")
        if self._stateTouched()[0]:
            self._auxPlanes = None       # rebuilt from the touched state; the scan below is dense anyway
        gemm, _, _ = self._weights(dt, input.device)
        norm = None
        if input.dtype == torch.uint8:
            norm = self.inputNorm
            if norm is None or self.in_channels > 4:
                raise _lib.CBinferError("detectInput: uint8 input needs inputNorm and <= 4 channels")
        self._detect(input, None, norm, self._aux(gemm), gemm, False, False)
        self._inVersion = self.prevInput._version
        return 'changeIndexes', input, DetectionDone(self, dense=True)

    def _smallMap(self, B, H, W):
        """bitmap small enough for the one-launch detection + compaction (cb_change_detect_sparse_compact)?"""
        return 0 < _lib.C.cb_bitmap_words(B, H, W) <= _lib.C.cb_compact_small_max_words()

    def _useTiles(self, dt, gemm, shape):
        """tile path for this layer / shape?  (tileMode 'auto': where the library recommends it)"""
        if self.tileMode == 'off' or os.environ.get("CBINFER_TILES", "1") == "0" or gemm == _lib.GEMM_SIMT_F32:
            return False
        return _tiles_ok(dt, gemm, tuple(shape), self.in_channels, self.out_channels, tuple(self.kernel_size),
                         self.tileMode)

    def _selfTiles(self, B, H, W):
        """Always False: no kernel lists its own tiles.  bench.py reads it to count launches."""
        return False

    def _compact(self, s, B, H, W, sparse_next, tiles=False, lazy=False):
        """dilate the raw bitmap by the filter footprint and compact it to the index list."""
        if tiles and "tile_ws" not in s:
            s["tile_ws"] = cg.alloc_tile_ws((B, H, W), s["idx"].device)
        if tiles and lazy:
            # tiles + dilated bitmap + count only; the ordered list is compacted if somebody asks
            cg.dilate_tiles(s["raw_bits"], (B, H, W), self.kernel_size, s["count"], s["ws"], s["dil_bits"],
                            s["tile_ws"], clear_raw=sparse_next, streams=self._streams(B))
            s["raw_clear"] = sparse_next
            return ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"], ws=s["ws"], listed=False)
        dil_map = s.get("dil_map") if self.saveChangeMap else None
        # a layer on the candidate path lets the compaction zero the raw bitmap once it has been
        # consumed, so the next frame's candidate detection needs no memset
        cg.dilate_compact(s["raw_bits"], (B, H, W), self.kernel_size, s["idx"], s["count"],
                          s["ws"], dil_bits=s["dil_bits"], dil_map=dil_map, clear_raw=sparse_next,
                          tile_ws=s["tile_ws"] if tiles else None, streams=self._streams(B))
        s["raw_clear"] = sparse_next
        if self.saveChangeMap:
            self.changeMap = dil_map[0] if B == 1 else dil_map
        return ChangeIndexes(s["idx"], s["count"], (B, H, W), bits=s["dil_bits"])

    def _gatherStats(self, input):
        """op-count bookkeeping of conv2d.py:201-218 (dense torch ops, only when enabled)."""
        changeTensor = (input - self.prevInput).abs().gt(self.threshold)
        ones = torch.ones(changeTensor.size(-3), 1, self.weight.size(2), self.weight.size(3),
                          device=input.device)
        proped = F.conv2d(changeTensor.float(), ones, groups=changeTensor.size(-3)).gt(0)
        opsPerValue = self.weight.size(0) * self.weight.size(2) * self.weight.size(3) * 2
        nC = changeTensor.size(-3)
        self.compStats = dict(
            numInputChangesPerFeatureMap=changeTensor.sum() * opsPerValue,
            numInputChanges=changeTensor.sum(-3).gt(0).sum() * nC * opsPerValue,
            numInputPropedChangesPerFeatureMap=proped.sum() * opsPerValue,
            numInputPropedChanges=proped.sum(-3).gt(0).sum() * nC * opsPerValue,
            totalInputValues=changeTensor.size(-1) * changeTensor.size(-2) * nC * opsPerValue,
        )

    def forward(self, inp):
        with torch.no_grad():
            self._checkThresholds()
            if self.finegrained:
                assert(self.feedbackLoop == False)
                if self._zone is not None:
                    raise _lib.CBinferError("a zone (setStreamZones) is not supported on a fine-grained layer")
                if self._activeMask is not None:
                    raise _lib.CBinferError("an active-stream mask is not supported on a fine-grained layer")
                return self.forward_fg(inp)
            else:
                return self.forward_normal(inp)

    def __repr__(self):
        s = ('{name} (th={threshold}, {in_channels}->{out_channels}, k={kernel_size}'
             ', s={stride}, copyInput={copyInput}')
        if self.padding != (0,) * len(self.padding):
            s += ', pad={padding}'
        if self.dilation != (1,) * len(self.dilation):
            s += ', dilation={dilation}'
        if self.output_padding != (0,) * len(self.output_padding):
            s += ', outpad={output_padding}'
        if self.groups != 1:
            s += ', grp={groups}'
        if self.bias is None:
            s += ', bias=False'
        if self.withReLU:
            s += ', withReLU={withReLU}'
        s += ', propChgIdxs={propChangeIndexes}'
        s += ')'
        return s.format(name=self.__class__.__name__, **self.__dict__)
