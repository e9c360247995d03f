"""Coarse-grained change-based ops: python wrappers over the sm_100a C ABI.

Mirrors the op surface of the reference's ``pycbinfer/conv2d_cg.py`` -- same function names,
argument meaning and tensor layouts (planar NCHW, batch 1, int8 change maps, ascending int32
indices) -- so code and tests written against the reference read the same here:

    changeDetection      conv2d_cg.py:100-122      changePropagation   conv2d_cg.py:159-177
    changeIndexesExtr    conv2d_cg.py:200-213      genXMatrix          conv2d_cg.py:239-261
    matrixMult           conv2d_cg.py:342-349      updateOutput        conv2d_cg.py:292-313
    maxPool2d            conv2d_cg.py:58-82

Differences, all deliberate: no ``useHalf`` flag (the dtype is taken from the tensor), launch
geometry lives in the library, the change count never has to visit the host
(:class:`ChangeIndexes`), and every op is CUDA-only -- the reference's ``*_python`` CPU twins
exist in this repo only inside ``oracle/`` as the parity checker.

The fused per-frame path used by ``CBConv2d`` (``detect`` -> ``dilate_compact`` ->
``conv_update``) is exposed as well.
"""
import os

import torch

from . import _lib
from ._lib import C, check, dtype_code, require_cuda, stream_ptr


def _strides4(t):
    """(sb, sc, sy, sx) element strides of a [B,C,H,W] tensor."""
    assert t.dim() == 4
    return t.stride(0), t.stride(1), t.stride(2), t.stride(3)


class ChangeIndexes(object):
    """Device-resident change-index list: ``buffer[:count]`` holds ascending int32 pixel indices
    ``b*H*W + y*W + x``.  It stands in for the exact-length tensor the reference passes between
    layers (conv2d.py:256-257) without forcing the device->host sync ``torch.nonzero`` implies
    (conv2d_cg.py:202): consumers in this package read ``count`` on the device; anything that
    needs a real tensor (``len``, ``.tensor()``, indexing) synchronises on demand."""

    def __init__(self, buffer, count, shape, bits=None, ws=None, listed=True):
        self._buffer = buffer         # int32 [capacity]
        # listed=False: only the dilated bitmap, the tile list and the count exist so far (cb_dilate_tiles);
        # the ordered list is compacted from `bits` the first time somebody asks for it
        self.listed = listed
        self._ws = ws                 # compaction workspace for that
        self.count = count            # int32 [1] on the device
        self.shape = shape            # (B, H, W) the indices refer to
        self.bits = bits              # optional dilated bitmap the list was compacted from
        # False when the producer's output was also modified outside its own kernels (e.g. a state
        # snapshot restored with copy_): the list is then not a complete candidate set downstream
        self.complete = True
        # True when the list is only a superset of the changed pixels (a masked 1x1 layer hands its
        # own candidates on instead of compacting): fine as detection candidates, not an exact list
        self.superset = False

    @property
    def buffer(self):
        if not self.listed:
            # compacted on every access, never cached: under CUDA-graph replay this python object
            # outlives the frame it was created for, while `bits` always holds the current frame
            assert self.bits is not None and self._ws is not None
            dilate_compact(self.bits, self.shape, (1, 1), self._buffer, self.count, self._ws)
        return self._buffer

    @classmethod
    def from_tensor(cls, idx, shape):
        idx = idx.to(torch.int32).contiguous()
        count = torch.full((1,), idx.numel(), dtype=torch.int32, device=idx.device)
        if idx.numel() == 0:                  # keep a valid device pointer for the C ABI
            idx = torch.zeros(1, dtype=torch.int32, device=idx.device)
        return cls(idx, count, shape)

    def tensor(self):
        if self.superset:
            raise _lib.CBinferError("this change list is a candidate superset (producer ran with "
                                    "maskedConv=True); set maskedConv=False on it for exact lists")
        buf = self.buffer
        return buf[: int(self.count.item())]

    # tensor-like conveniences (all synchronise)
    def __len__(self):
        return int(self.count.item())

    def numel(self):
        return len(self)

    def dim(self):
        return 1

    def size(self, d=None):
        return torch.Size([len(self)]) if d is None else len(self)

    def contiguous(self):
        return self

    @property
    def data(self):
        return self

    @property
    def is_cuda(self):
        return self._buffer.is_cuda

    def cpu(self):
        return self.tensor().cpu()

    def __getitem__(self, i):
        return self.tensor()[i]


# ---------------------------------------------------------------------------------------------
# fused-path primitives (native pixel-major layout, batch-capable, no host sync)
# ---------------------------------------------------------------------------------------------

def _aux_args(aux, state):
    """aux: None | ('tf32', lo_view) | ('bf16', hi16_buf, lo16_buf) -> (mode, hi_ptr, lo_ptr)."""
    if aux is None:
        return _lib.AUX_NONE, None, None
    if aux[0] == 'tf32':
        assert aux[1].stride() == state.stride() and aux[1].dtype == state.dtype
        return _lib.AUX_TF32_LO, None, aux[1].data_ptr()
    assert aux[0] == 'bf16' and aux[1].dtype == torch.bfloat16 and aux[2].dtype == torch.bfloat16
    return _lib.AUX_BF16_PAIR, aux[1].data_ptr(), aux[2].data_ptr()


def _active_ptr(active, B, device):
    """Device pointer of an active-stream mask (a contiguous bool / uint8 CUDA tensor [B] on x's
    device), or None for no mask (every stream active)."""
    if active is None:
        return None
    require_cuda(active)
    if active.dim() != 1 or active.dtype not in (torch.bool, torch.uint8) or not active.is_contiguous():
        raise _lib.CBinferError("active-stream mask: a contiguous bool or uint8 tensor [B] is needed, got %s %s"
                                % (active.dtype, tuple(active.shape)))
    if active.numel() != B or active.device != device:
        raise _lib.CBinferError("active-stream mask: %d entries on %s for %d streams on %s"
                                % (active.numel(), active.device, B, device))
    return active.data_ptr()


def _thr_ptr(thr_b, B, device):
    """Device pointer of a per-stream threshold table (a contiguous fp32 CUDA tensor [B] on the data's
    device), or None for none (the scalar threshold for every stream)."""
    if thr_b is None:
        return None
    require_cuda(thr_b)
    if thr_b.dim() != 1 or thr_b.dtype != torch.float32 or not thr_b.is_contiguous() \
            or thr_b.numel() != B or thr_b.device != device:
        raise _lib.CBinferError("per-stream thresholds: a contiguous fp32 tensor [%d] on %s is needed, got %s %s on %s"
                                % (B, device, thr_b.dtype, tuple(thr_b.shape), thr_b.device))
    return thr_b.data_ptr()


def _zone_ptr(zone, B, H, W, device):
    """Device pointer of a watched-pixel zone (a contiguous int32 CUDA bitmap [B, H, ceil(W/32)] on the
    data's device, as cb_map_to_bits writes it), or None for none (every pixel watched)."""
    if zone is None:
        return None
    require_cuda(zone)
    words = C.cb_bitmap_words(B, H, W)
    if zone.dtype != torch.int32 or not zone.is_contiguous() or zone.numel() != words or zone.device != device:
        raise _lib.CBinferError("zone: a contiguous int32 bitmap of %d words on %s is needed, got %s %s on %s"
                                % (words, device, zone.dtype, tuple(zone.shape), zone.device))
    return zone.data_ptr()


def detect(x, state, raw_bits, threshold, update_mode, aux=None, active=None, thr_b=None, zone=None):
    """cb_change_detect: raw (un-dilated) change bitmap of x vs state; updates state and, when
    given, the auxiliary operand planes `aux` (see _aux_args).  `active`: optional bool / uint8
    CUDA tensor [B], read on the device; a stream with active[b] == 0 is skipped (its bitmap words
    0, its x not read, its state and planes untouched: cb_change_detect_streams).  `thr_b`: optional
    fp32 CUDA tensor [B] of per-stream thresholds, read on the device instead of `threshold`
    (cb_change_detect_thr); the same holds for every wrapper below that takes it.  `zone`: optional
    int32 bitmap of watched pixels (see _zone_ptr); an excluded pixel whose state is finite counts as
    unchanged and is neither read nor written (cb_change_detect_zone)."""
    require_cuda(x, state, raw_bits)
    B, Cc, H, W = x.shape
    assert state.shape == x.shape and state.dtype == x.dtype
    act = _active_ptr(active, B, x.device)
    mode, hi, lo = _aux_args(aux, state)
    check(C.cb_change_detect_zone(stream_ptr(x.device), dtype_code(x), x.data_ptr(), *_strides4(x),
                                  state.data_ptr(), *_strides4(state), mode, hi, lo,
                                  raw_bits.data_ptr(), B, Cc, H, W, float(threshold), int(update_mode), act,
                                  _thr_ptr(thr_b, B, x.device), _zone_ptr(zone, B, H, W, x.device)))


def detect_u8(x, state, raw_bits, threshold, update_mode, divisor, bias, aux=None, active=None, thr_b=None,
              zone=None):
    """cb_change_detect_u8: detection on a uint8 frame normalised on the fly as u8/divisor + bias
    (the readers' /255 resp. /256 - 0.5); `state` is the fp32 pixel-major state.  Bit-identical to
    :func:`detect` on ``x.float() / divisor + bias``.  `active`, `thr_b` and `zone` as in :func:`detect`."""
    require_cuda(x, state, raw_bits)
    B, Cc, H, W = x.shape
    assert x.dtype == torch.uint8 and state.dtype == torch.float32 and state.shape == x.shape
    act = _active_ptr(active, B, x.device)
    mode, hi, lo = _aux_args(aux, state)
    check(C.cb_change_detect_u8_zone(stream_ptr(x.device), x.data_ptr(), *_strides4(x),
                                     state.data_ptr(), *_strides4(state), mode, hi, lo,
                                     raw_bits.data_ptr(), B, Cc, H, W, float(divisor), float(bias),
                                     float(threshold), int(update_mode), act, _thr_ptr(thr_b, B, x.device),
                                     _zone_ptr(zone, B, H, W, x.device)))


def detect_sparse(x, state, raw_bits, threshold, update_mode, candidates, aux=None,
                  bits_are_clear=False, thr_b=None):
    """cb_change_detect_sparse: the detection test at the candidate pixels only (see the header
    for the exactness conditions).  `candidates` is a :class:`ChangeIndexes` at x's resolution."""
    require_cuda(x, state, raw_bits)
    B, Cc, H, W = x.shape
    assert state.shape == x.shape and state.dtype == x.dtype
    assert tuple(candidates.shape) == (B, H, W)
    mode, hi, lo = _aux_args(aux, state)
    check(C.cb_change_detect_sparse_thr(stream_ptr(x.device), dtype_code(x), x.data_ptr(), *_strides4(x),
                                        state.data_ptr(), *_strides4(state), mode, hi, lo,
                                        candidates.buffer.data_ptr(), candidates.count.data_ptr(),
                                        raw_bits.data_ptr(), B, Cc, H, W, float(threshold),
                                        int(update_mode), int(bool(bits_are_clear)), _thr_ptr(thr_b, B, x.device)))


def _streams_args(streams, B):
    """(stream_counts, stream_acc) pointers of a per-stream counts row: `streams` = (counts, acc), int32 CUDA
    tensors of at least B (counts) and B (acc) entries, or None = (None, None)."""
    if streams is None:
        return None, None
    counts, acc = streams
    require_cuda(counts, acc)
    if counts.dtype != torch.int32 or acc.dtype != torch.int32 or counts.numel() < B or acc.numel() < B \
            or not counts.is_contiguous() or not acc.is_contiguous():
        raise _lib.CBinferError("per-stream counts: contiguous int32 tensors of >= %d entries are needed" % B)
    return counts.data_ptr(), acc.data_ptr()


def stream_bucket(changes, shape, streams):
    """cb_stream_bucket: counts[b] = number of entries of the index list `changes` (a
    :class:`ChangeIndexes`, any order) in stream b of a [B,H,W] grid; `streams` = (counts int32 [B],
    accumulator int32 [B+1] zeroed once)."""
    B, H, W = shape
    sc, acc = _streams_args(streams, B)
    if streams[1].numel() < B + 1:
        raise _lib.CBinferError("stream_bucket: the accumulator needs B + 1 = %d entries" % (B + 1))
    check(C.cb_stream_bucket(stream_ptr(changes.count.device), changes.buffer.data_ptr(), changes.count.data_ptr(),
                             B, H * W, sc, acc))


def detect_sparse_compact(x, state, raw_bits, threshold, update_mode, candidates, filtSize, idx, count, sync,
                          aux=None, bits_are_clear=False, dil_bits=None, clear_raw=False, streams=None, thr_b=None):
    """cb_change_detect_sparse_compact: candidate detection + dilation + ordered compaction in one launch
    (small maps: at most cb_compact_small_max_words() bitmap words).  `sync` = int32[1], zeroed once.
    `streams`: optional (counts int32 [B], accumulator int32 [B] zeroed once): the count split by stream
    (cb_change_detect_sparse_compact_streams)."""
    require_cuda(x, state, raw_bits)
    B, Cc, H, W = x.shape
    assert state.shape == x.shape and state.dtype == x.dtype
    assert tuple(candidates.shape) == (B, H, W)
    mode, hi, lo = _aux_args(aux, state)
    check(C.cb_change_detect_sparse_compact_thr(
        stream_ptr(x.device), dtype_code(x), x.data_ptr(), *_strides4(x), state.data_ptr(), *_strides4(state),
        mode, hi, lo, candidates.buffer.data_ptr(), candidates.count.data_ptr(), raw_bits.data_ptr(), B, Cc, H, W,
        float(threshold), int(update_mode), int(bool(bits_are_clear)),
        dil_bits.data_ptr() if dil_bits is not None else None, idx.data_ptr(), count.data_ptr(), sync.data_ptr(),
        (filtSize[0] - 1) // 2, (filtSize[1] - 1) // 2, int(bool(clear_raw)), *_streams_args(streams, B),
        _thr_ptr(thr_b, B, x.device)))


def detect_compact_sparse(*args, **kwargs):
    """Removed kernel; the name stays only because bench.py looks it up to build its kernel tables."""
    raise _lib.CBinferError("detect_compact_sparse was removed")


def pool_compact(in_bits, in_shape, out_shape, idx, count, ws, out_bits=None):
    """cb_pool_compact: change candidates at the 2x2-pooled resolution from an input bitmap."""
    B, H, W = in_shape
    B2, oH, oW = out_shape
    assert B == B2
    check(C.cb_pool_compact(stream_ptr(in_bits.device), in_bits.data_ptr(),
                            out_bits.data_ptr() if out_bits is not None else None,
                            idx.data_ptr(), count.data_ptr(), ws.data_ptr(), B, H, W, oH, oW))


def dilate_tiles(raw_bits, shape, filtSize, count, ws, dil_bits, tile_ws, clear_raw=False, streams=None):
    """cb_dilate_tiles: dilation + dirty-tile list + change count, no ordered index list.  `streams` as in
    :func:`detect_sparse_compact`."""
    B, H, W = shape
    check(C.cb_dilate_tiles_streams(stream_ptr(raw_bits.device), raw_bits.data_ptr(), dil_bits.data_ptr(),
                                    count.data_ptr(), ws.data_ptr(), tile_ws.data_ptr(), B, H, W,
                                    (filtSize[0] - 1) // 2, (filtSize[1] - 1) // 2, int(bool(clear_raw)),
                                    *_streams_args(streams, B)))


def dilate_compact(raw_bits, shape, filtSize, idx, count, ws, dil_bits=None, dil_map=None,
                   clear_raw=False, tile_ws=None, streams=None):
    """cb_dilate_compact: dilation by the filter footprint + ordered compaction.  With `tile_ws`
    (cb_tile_ws_bytes of zeroed int32 device memory) the dirty 8x16 output tiles are listed as well
    (cb_dilate_compact_tiles), for :func:`conv_update_tiled`.  `streams` as in
    :func:`detect_sparse_compact`."""
    B, H, W = shape
    sc, acc = _streams_args(streams, B)
    if tile_ws is not None:
        check(C.cb_dilate_compact_tiles_streams(stream_ptr(raw_bits.device), raw_bits.data_ptr(),
                                                dil_bits.data_ptr() if dil_bits is not None else None,
                                                dil_map.data_ptr() if dil_map is not None else None,
                                                idx.data_ptr(), count.data_ptr(), ws.data_ptr(),
                                                tile_ws.data_ptr(), B, H, W, (filtSize[0] - 1) // 2,
                                                (filtSize[1] - 1) // 2, int(bool(clear_raw)), sc, acc))
        return
    check(C.cb_dilate_compact_streams(stream_ptr(raw_bits.device), raw_bits.data_ptr(),
                                      dil_bits.data_ptr() if dil_bits is not None else None,
                                      dil_map.data_ptr() if dil_map is not None else None,
                                      idx.data_ptr(), count.data_ptr(), ws.data_ptr(), B, H, W,
                                      (filtSize[0] - 1) // 2, (filtSize[1] - 1) // 2, int(bool(clear_raw)), sc, acc))


def alloc_tile_ws(shape, device):
    """tile workspace of cb_dilate_compact_tiles / cb_conv_update_tiled for a [B,H,W] pixel grid."""
    B, H, W = shape
    return torch.zeros(C.cb_tile_ws_bytes(B, H, W) // 4, dtype=torch.int32, device=device)


def tiled_supported(dtype, gemm, shape, Cin, Cout, filtSize):
    """cb_conv_tiled_supported: 1 = run the tile path, 2 = possible but not recommended, 0 = no."""
    B, H, W = shape
    return C.cb_conv_tiled_supported(dtype_code(dtype), gemm, B, H, W, Cin, Cout, filtSize[0], filtSize[1])


def alloc_scratch(shape, device, want_map=False):
    """bitmaps / index buffer / count / compaction workspace for a [B,H,W] pixel grid."""
    B, H, W = shape
    nwords = C.cb_bitmap_words(B, H, W)
    s = dict(
        raw_bits=torch.zeros(max(nwords, 1), dtype=torch.int32, device=device),
        dil_bits=torch.zeros(max(nwords, 1), dtype=torch.int32, device=device),
        idx=torch.zeros(max(B * H * W, 1), dtype=torch.int32, device=device),
        count=torch.zeros(1, dtype=torch.int32, device=device),
        ws=torch.zeros(C.cb_compact_ws_bytes(B, H, W), dtype=torch.uint8, device=device),
    )
    if want_map:
        s["dil_map"] = torch.zeros(B, H, W, dtype=torch.int8, device=device)
    return s


def pack_weights(weight, gemm):
    """cb_pack_weights: [Cout,Cin,kH,kW] -> the layout cb_conv_update expects for `gemm`."""
    require_cuda(weight)
    Cout, Cin, kH, kW = weight.shape
    w = weight.detach().contiguous()
    nbytes = C.cb_packed_weight_bytes(dtype_code(w), gemm, Cout, Cin, kH, kW)
    packed = torch.empty(nbytes + 256, dtype=torch.uint8, device=w.device)
    off = (-packed.data_ptr()) % 256                       # TMA wants >=128-byte alignment
    packed = packed[off: off + nbytes]
    check(C.cb_pack_weights(stream_ptr(w.device), dtype_code(w), gemm, w.data_ptr(),
                            packed.data_ptr(), Cout, Cin, kH, kW))
    return packed


def tf32_lo(x):
    """v - trunc_tf32(v): the remainder plane the 3xTF32 contraction consumes (exact in fp32)."""
    hi = (x.contiguous().view(torch.int32) & -8192).view(torch.float32)
    return x - hi


def bf16_pair(x):
    """(bf16(v), bf16(v - bf16(v))): the operand planes of the 3xBF16 contraction."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def bf16_planes(state_buf, C_):
    """pixel-major bf16 hi/lo planes [B,H,W,pitch16] of a pixel-major fp32 buffer."""
    B, H, W, _ = state_buf.shape
    p16 = C.cb_plane_pitch16(C_)
    hi = torch.zeros(B, H, W, p16, dtype=torch.bfloat16, device=state_buf.device)
    lo = torch.zeros_like(hi)
    h, l = bf16_pair(state_buf[..., :C_])
    hi[..., :C_] = h
    lo[..., :C_] = l
    return hi, lo


class ConvWorkspace(object):
    """Stream-K workspace of cb_conv_update (cb_conv_ws_bytes() of zeroed device memory; the kernel
    leaves it clean).  Launches that may overlap need their own: one holder per model instance,
    shared by its layers (a model's layers run in order).  Not pickled."""

    def __init__(self):
        self.buf = None

    def get(self, device):
        if os.environ.get("CBINFER_STREAMK", "1") == "0":
            return None
        if self.buf is None or self.buf.device != device:
            self.buf = torch.zeros(C.cb_conv_ws_bytes(), dtype=torch.uint8, device=device)
        return self.buf

    def clear(self):
        self.buf = None

    def __getstate__(self):
        return {}

    def __setstate__(self, state):
        self.buf = None


def _conv_operands(state_buf, Cin, gemm, aux):
    """(source, remainder plane or None, pitch) the contraction reads: the bf16 hi/lo planes for
    GEMM_TC_BF16X3, else the state with, for GEMM_TC_3X on fp32 data, its tf32 remainder plane.
    `aux` holds the planes in the format of :func:`_aux_args`; without it they are derived from
    the state on the fly."""
    if gemm == _lib.GEMM_TC_BF16X3:
        assert state_buf.dtype == torch.float32
        _, hi, lo = aux if aux is not None else ('bf16',) + bf16_planes(state_buf, Cin)
        return hi, lo, hi.shape[3]
    lo = None
    if gemm == _lib.GEMM_TC_3X and state_buf.dtype == torch.float32:
        lo = aux[1] if aux is not None else tf32_lo(state_buf)
    return state_buf, lo, state_buf.shape[3]


def conv_update(state_buf, changes, packed_w, bias_f32, out_buf, Cin, Cout, filtSize, relu, gemm,
                aux=None, ws=None, mask=None):
    """cb_conv_update on pixel-major buffers [B,H,W,pitch].  GEMM_TC_3X (fp32) consumes the tf32
    remainder plane, GEMM_TC_BF16X3 the bf16 hi/lo planes, passed as `aux` (see _aux_args: what
    cb_change_detect keeps in step) or derived on the fly."""
    B, H, W, _ = state_buf.shape
    assert out_buf.shape[:3] == state_buf.shape[:3]
    src, src_lo, pitch = _conv_operands(state_buf, Cin, gemm, aux)
    if mask is not None:
        # `changes` is a superset list; mask = dict(bits=raw bitmap, clear=bool, count=int32[1] out,
        # sync=int32[2] zeroed once, optional streams as in detect_sparse_compact): only pixels whose bit
        # is set are processed (cb_conv_update_masked[_streams])
        check(C.cb_conv_update_masked_streams(stream_ptr(state_buf.device), dtype_code(state_buf), gemm,
                                      src.data_ptr(), src_lo.data_ptr() if src_lo is not None else None,
                                      pitch, changes.buffer.data_ptr(), changes.count.data_ptr(),
                                      packed_w.data_ptr(), bias_f32.data_ptr(), out_buf.data_ptr(),
                                      out_buf.shape[3], B, H, W, Cin, Cout, filtSize[0], filtSize[1],
                                      int(bool(relu)), ws.data_ptr() if ws is not None else None,
                                      ws.numel() if ws is not None else 0,
                                      mask['bits'].data_ptr(), int(bool(mask.get('clear', False))),
                                      mask['count'].data_ptr(), mask['sync'].data_ptr(),
                                      *_streams_args(mask.get('streams'), B)))
        return
    check(C.cb_conv_update(stream_ptr(state_buf.device), dtype_code(state_buf), gemm,
                           src.data_ptr(), src_lo.data_ptr() if src_lo is not None else None,
                           pitch, changes.buffer.data_ptr(),
                           changes.count.data_ptr(), packed_w.data_ptr(), bias_f32.data_ptr(),
                           out_buf.data_ptr(), out_buf.shape[3], B, H, W, Cin, Cout,
                           filtSize[0], filtSize[1], int(bool(relu)),
                           ws.data_ptr() if ws is not None else None,
                           ws.numel() if ws is not None else 0))


def fg_detect(x, prev_view, prev_buf, planes16, raw_bits, threshold, count=None):
    """cb_fg_detect: per-VALUE thresholded delta of x against the pixel-major fp32 state (`prev_view` =
    the [B,C,H,W] view of `prev_buf` [B,H,W,pitch]) -> bf16 hi/lo delta planes `planes16`, raw pixel
    bitmap, changed-value count; the state is overwritten with x."""
    require_cuda(x, prev_buf, raw_bits)
    B, Cc, H, W = x.shape
    assert x.dtype == torch.float32 and prev_buf.dtype == torch.float32
    assert tuple(prev_view.shape) == tuple(x.shape) and prev_view.stride(1) == 1
    hi, lo = planes16
    assert hi.dtype == torch.bfloat16 and hi.shape == (B, H, W, C.cb_plane_pitch16(Cc)) and lo.shape == hi.shape
    check(C.cb_fg_detect(stream_ptr(x.device), x.data_ptr(), *_strides4(x), prev_view.data_ptr(),
                         prev_view.stride(0), prev_view.stride(2), prev_view.stride(3),
                         hi.data_ptr(), lo.data_ptr(), raw_bits.data_ptr(),
                         count.data_ptr() if count is not None else None, B, Cc, H, W, float(threshold)))


def conv_accumulate(planes16, changes, packed_w, out_buf, Cin, Cout, filtSize, gemm, ws=None):
    """cb_conv_accumulate: out_buf[pix, :] += contraction of the operand planes around pix with the
    packed weights, for the listed pixels (no bias, no ReLU) - the fine-grained update."""
    src, src_lo = planes16
    B, H, W, pitch = src.shape
    assert gemm == _lib.GEMM_TC_BF16X3 and out_buf.dtype == torch.float32
    assert out_buf.shape[:3] == src.shape[:3]
    check(C.cb_conv_accumulate(stream_ptr(src.device), _lib.F32, gemm, src.data_ptr(), src_lo.data_ptr(),
                               pitch, changes.buffer.data_ptr(), changes.count.data_ptr(),
                               packed_w.data_ptr(), out_buf.data_ptr(), out_buf.shape[3], B, H, W, Cin,
                               Cout, filtSize[0], filtSize[1],
                               ws.data_ptr() if ws is not None else None,
                               ws.numel() if ws is not None else 0))


def conv_update_tiled(state_buf, tile_ws, dil_bits, packed_w, bias_f32, out_buf, Cin, Cout, filtSize,
                      relu, gemm, aux=None, pool=None):
    """cb_conv_update_tiled on pixel-major buffers: the contraction over the dirty 8x16 tiles listed
    in `tile_ws` (TMA-staged halo tiles, implicit im2col), writing the pixels set in `dil_bits`.
    Operand conventions as :func:`conv_update`."""
    B, H, W, _ = state_buf.shape
    assert out_buf.shape[:3] == state_buf.shape[:3]
    src, src_lo, pitch = _conv_operands(state_buf, Cin, gemm, aux)
    if pool is not None:
        # pool = dict(out=pooled map view, next_state=view, next_raw_bits, threshold, mode, aux, optional
        # thr_b): the epilogue also re-pools the touched 2x2 windows and runs the next layer's detection on them
        po, ns = pool["out"], pool["next_state"]
        assert po.stride(1) == 1 and ns.stride(1) == 1 and po.shape == ns.shape, "pixel-major maps only"
        mode, hi, lo = _aux_args(pool.get("aux"), ns)
        check(C.cb_conv_update_tiled_pool_thr(stream_ptr(state_buf.device), dtype_code(state_buf), gemm,
                                          src.data_ptr(), src_lo.data_ptr() if src_lo is not None else None,
                                          pitch, tile_ws.data_ptr(), dil_bits.data_ptr(), packed_w.data_ptr(),
                                          bias_f32.data_ptr(), out_buf.data_ptr(), out_buf.shape[3], B, H, W,
                                          Cin, Cout, filtSize[0], filtSize[1], int(bool(relu)),
                                          po.data_ptr(), po.stride(0), po.stride(2), po.stride(3),
                                          po.size(2), po.size(3), ns.data_ptr(), ns.stride(0), ns.stride(2),
                                          ns.stride(3), mode, hi, lo, pool["next_raw_bits"].data_ptr(),
                                          float(pool["threshold"]), int(pool["mode"]),
                                          _thr_ptr(pool.get("thr_b"), B, state_buf.device)))
        return
    check(C.cb_conv_update_tiled(stream_ptr(state_buf.device), dtype_code(state_buf), gemm,
                                 src.data_ptr(), src_lo.data_ptr() if src_lo is not None else None,
                                 pitch, tile_ws.data_ptr(), dil_bits.data_ptr(), packed_w.data_ptr(),
                                 bias_f32.data_ptr(), out_buf.data_ptr(), out_buf.shape[3], B, H, W,
                                 Cin, Cout, filtSize[0], filtSize[1], int(bool(relu))))


def tail_update(x_buf, state1_buf, packed1, bias1, out1_buf, relu1, thr1, state2_buf, packed2, bias2,
                out2_buf, relu2, thr2, candidates, C0, C1, C2, update_mode, count1, count2, sync,
                streams1=None, streams2=None, thr1_b=None, thr2_b=None):
    """cb_tail_update: two chained 1x1 change-based layers (detect, contraction, detect,
    contraction) for the candidate pixels in one launch; pixel-major fp32 buffers [B,H,W,pitch].
    `streams1` / `streams2`: optional per-stream counts rows of the two layers, as in
    :func:`detect_sparse_compact` (both or neither).  `thr1_b` / `thr2_b`: the layers' per-stream thresholds."""
    assert x_buf.dtype == torch.float32 and x_buf.shape[3] == C0 and state1_buf.shape == x_buf.shape
    assert out1_buf.shape[3] == C1 and state2_buf.shape == out1_buf.shape
    B, H, W, _ = x_buf.shape
    check(C.cb_tail_update_thr(stream_ptr(x_buf.device), x_buf.data_ptr(), state1_buf.data_ptr(),
                           packed1.data_ptr(), bias1.data_ptr(), out1_buf.data_ptr(), int(bool(relu1)),
                           float(thr1), state2_buf.data_ptr(), packed2.data_ptr(), bias2.data_ptr(),
                           out2_buf.data_ptr(), out2_buf.shape[3], int(bool(relu2)), float(thr2),
                           candidates.buffer.data_ptr(), candidates.count.data_ptr(), C0, C1, C2,
                           int(update_mode), count1.data_ptr(), count2.data_ptr(), sync.data_ptr(), B, H * W,
                           *_streams_args(streams1, B), *_streams_args(streams2, B),
                           _thr_ptr(thr1_b, B, x_buf.device), _thr_ptr(thr2_b, B, x_buf.device)))


def reset_streams(segments, mask):
    """cb_reset_streams: for every stream b with ``mask[b] != 0`` rewrite stream b's slice of each
    segment.  A segment is ``(buf, channels, fill)``: ``buf`` a pixel-major [B,H,W,*] tensor whose
    pixel stride (``buf.stride(2)``) is the pitch and whose first ``channels`` channels are real;
    those are set to ``fill`` (``inf`` or 0), the pad channels up to the pitch to 0.  ``mask`` is a
    bool / uint8 CUDA tensor [B]; it is read on the device, so the call can be captured in a graph."""
    require_cuda(mask)
    if mask.dim() != 1 or mask.dtype not in (torch.bool, torch.uint8) or not mask.is_contiguous():
        raise _lib.CBinferError("reset_streams: the mask must be a contiguous bool or uint8 tensor [B]")
    B = mask.numel()
    segs = (_lib.ResetSegment * max(len(segments), 1))()
    for i, (buf, channels, fill) in enumerate(segments):
        require_cuda(buf)
        Bb, H, W, _ = buf.shape
        pitch = buf.stride(2)
        if Bb != B or buf.device != mask.device:
            raise _lib.CBinferError("reset_streams: a buffer of %d streams on %s, a mask of %d on %s"
                                    % (Bb, buf.device, B, mask.device))
        assert buf.stride(3) == 1 and buf.stride(1) == W * pitch and buf.stride(0) == H * W * pitch \
            and channels <= pitch, "pixel-major buffers only"
        es = buf.element_size()
        segs[i] = _lib.ResetSegment(buf.data_ptr(), H * W, pitch * es, channels * es, dtype_code(buf),
                                    _lib.RESET_FILL_INF if fill != 0 else _lib.RESET_FILL_ZERO)
    with torch.cuda.device(mask.device):
        check(C.cb_reset_streams(stream_ptr(mask.device), mask.data_ptr(), B, segs, len(segments)))


def pixel_major(shape, dtype, device, fill):
    """Allocate a [B,C,H,W]-shaped *view* over a pixel-major [B,H,W,pitch] buffer whose pitch is
    C rounded up to 16 bytes.  Real channels are set to `fill`, pad channels to 0 (they meet zero
    weights in the contraction).  Returns (view, buffer)."""
    B, Cc, H, W = shape
    pitch = _lib.channel_pitch(dtype, Cc)
    buf = torch.zeros(B, H, W, pitch, dtype=dtype, device=device)
    view = buf[..., :Cc].permute(0, 3, 1, 2)
    if fill != 0:
        view.fill_(fill)
    return view, buf


# ---------------------------------------------------------------------------------------------
# reference-named ops (planar layout, batch 1 unless noted)
# ---------------------------------------------------------------------------------------------

def changeDetection(input, prevInput, filtSize, threshold, updateInputState=False):
    """conv2d_cg.py:100-122: int8 change map [H,W] (batch 1) / [B,H,W], dilated by filtSize;
    with updateInputState the changed pixels of prevInput are overwritten in place."""
    assert input.size() == prevInput.size() and input.dim() == 4
    require_cuda(input, prevInput)
    B, _, H, W = input.shape
    s = alloc_scratch((B, H, W), input.device, want_map=True)
    detect(input, prevInput, s["raw_bits"], threshold,
           _lib.UPDATE_CHANGED if updateInputState else _lib.UPDATE_NONE)
    dilate_compact(s["raw_bits"], (B, H, W), filtSize, s["idx"], s["count"], s["ws"],
                   dil_map=s["dil_map"])
    return s["dil_map"][0] if B == 1 else s["dil_map"]


def _map_to_bits(changeMap):
    H, W = changeMap.shape[-2:]
    B = changeMap.numel() // (H * W)
    m = changeMap.reshape(B, H, W).to(torch.int8).contiguous()
    require_cuda(m)
    bits = torch.zeros(max(C.cb_bitmap_words(B, H, W), 1), dtype=torch.int32, device=m.device)
    check(C.cb_map_to_bits(stream_ptr(m.device), m.data_ptr(), bits.data_ptr(), B, H, W))
    return bits, (B, H, W)


def changePropagation(changeMap, filtSize):
    """conv2d_cg.py:159-177: gather-dilate an int8/bool change map by filtSize."""
    assert len(filtSize) == 2
    if filtSize[0] == 1 and filtSize[1] == 1:
        return changeMap
    bits, shape = _map_to_bits(changeMap)
    s = alloc_scratch(shape, changeMap.device, want_map=True)
    dilate_compact(bits, shape, filtSize, s["idx"], s["count"], s["ws"], dil_map=s["dil_map"])
    return s["dil_map"].reshape(changeMap.shape).to(changeMap.dtype)


def changeIndexesExtr(changeMap, lazy=False):
    """conv2d_cg.py:200-213: ascending int32 indices of the non-zero map cells.  With
    ``lazy=True`` returns a :class:`ChangeIndexes` (no host sync)."""
    bits, shape = _map_to_bits(changeMap)
    s = alloc_scratch(shape, changeMap.device)
    dilate_compact(bits, shape, (1, 1), s["idx"], s["count"], s["ws"])
    ci = ChangeIndexes(s["idx"], s["count"], shape)
    return ci if lazy else ci.tensor()


changeIndexesExtr_python = changeIndexesExtr     # the reference's forward calls the *_python name


def genXMatrix(input, changeIndexes, filtSize):
    """conv2d_cg.py:239-261: im2col of the changed pixels, X[n, Cin*kH*kW] (planar input)."""
    require_cuda(input)
    inC, inH, inW = input.size(-3), input.size(-2), input.size(-1)
    kH, kW = filtSize
    idx = changeIndexes.tensor() if isinstance(changeIndexes, ChangeIndexes) else changeIndexes
    idx = idx.to(torch.int32).contiguous()
    n = idx.numel()
    X = input.new_empty(n, inC * kH * kW)
    if n > 0:
        inp = input.contiguous()
        check(C.cb_gen_xmatrix(stream_ptr(input.device), dtype_code(input), X.data_ptr(),
                               inp.data_ptr(), idx.data_ptr(), kW, kH, inC, inW, inH, n))
    return X


def matrixMult(Xmatrix, weights, bias, activFun=None):
    """conv2d_cg.py:342-349: Y = X . W.view(Cout,-1)^T + bias (fp32 accumulation)."""
    if Xmatrix.numel() == 0:
        return Xmatrix.clone()
    require_cuda(Xmatrix, weights, bias)
    n, K = Xmatrix.shape
    Cout = weights.size(0)
    Y = Xmatrix.new_empty(n, Cout)
    w = weights.detach().contiguous().view(Cout, -1)
    assert w.size(1) == K
    check(C.cb_matrix_mult(stream_ptr(Xmatrix.device), dtype_code(Xmatrix),
                           Xmatrix.contiguous().data_ptr(), w.data_ptr(),
                           bias.detach().contiguous().data_ptr(), Y.data_ptr(), n, K, Cout))
    if activFun is not None:
        Y = activFun(Y)
    return Y


matrixMult_python = matrixMult


def updateOutput(YMatrix, changeIndexes, prevOutput, withReLU=False):
    """conv2d_cg.py:292-313: scatter Y^T[Cout,n] into the planar prevOutput (in place)."""
    require_cuda(YMatrix, prevOutput)
    outC, outH, outW = prevOutput.size(-3), prevOutput.size(-2), prevOutput.size(-1)
    idx = changeIndexes.tensor() if isinstance(changeIndexes, ChangeIndexes) else changeIndexes
    idx = idx.to(torch.int32).contiguous()
    n = idx.numel()
    if n > 0:
        assert prevOutput.is_contiguous()
        Yt = YMatrix.contiguous()
        check(C.cb_update_output(stream_ptr(prevOutput.device), dtype_code(prevOutput),
                                 Yt.data_ptr(), prevOutput.data_ptr(), idx.data_ptr(),
                                 outW * outH, n, outC, int(bool(withReLU))))
    return prevOutput


def maxPool2d(input, outputState, changeIndexes, kernelSize=(2, 2), stride=(2, 2)):
    """conv2d_cg.py:58-82: recompute the 2x2/stride-2 windows touched by the changed input
    pixels into outputState (in place).  Any strides, batch >= 1."""
    assert tuple(kernelSize) == (2, 2) and tuple(stride) == (2, 2)
    require_cuda(input, outputState)
    assert input.dim() == 4 and outputState.dim() == 4
    B, Cc, H, W = input.shape
    oH, oW = outputState.size(-2), outputState.size(-1)
    if not isinstance(changeIndexes, ChangeIndexes):
        changeIndexes = ChangeIndexes.from_tensor(changeIndexes, (B, H, W))
    bits = changeIndexes.bits
    check(C.cb_maxpool2x2(stream_ptr(input.device), dtype_code(input), input.data_ptr(),
                          *_strides4(input), changeIndexes.buffer.data_ptr(),
                          changeIndexes.count.data_ptr(),
                          bits.data_ptr() if bits is not None else None,
                          outputState.data_ptr(), *_strides4(outputState), B, Cc, H, W, oH, oW))
    return outputState


def maxPool2d_detect(input, outputState, changeIndexes, next_state, next_raw_bits, threshold,
                     update_mode, aux=None, thr_b=None):
    """cb_maxpool2x2_detect: change-based pooling fused with the next layer's detection (pixel-major
    tensors only; `changeIndexes.bits` required; `next_raw_bits` must be clear)."""
    require_cuda(input, outputState, next_state)
    B, Cc, H, W = input.shape
    oH, oW = outputState.size(-2), outputState.size(-1)
    assert changeIndexes.bits is not None and next_state.shape == outputState.shape
    for t in (input, outputState, next_state):
        assert t.stride(1) == 1, "pixel-major tensors only"
    mode, hi, lo = _aux_args(aux, next_state)
    check(C.cb_maxpool2x2_detect_thr(stream_ptr(input.device), dtype_code(input), input.data_ptr(),
                                 input.stride(0), input.stride(2), input.stride(3),
                                 changeIndexes.buffer.data_ptr(), changeIndexes.count.data_ptr(),
                                 changeIndexes.bits.data_ptr(), outputState.data_ptr(),
                                 outputState.stride(0), outputState.stride(2), outputState.stride(3),
                                 B, Cc, H, W, oH, oW, next_state.data_ptr(), next_state.stride(0),
                                 next_state.stride(2), next_state.stride(3), mode, hi, lo,
                                 next_raw_bits.data_ptr(), float(threshold), int(update_mode),
                                 _thr_ptr(thr_b, B, input.device)))
    return outputState
