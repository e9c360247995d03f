"""CPU: cb_reset_streams checks its arguments on the host and refuses bad ones with a status code
before anything reaches the device (no GPU needed: nothing is launched)."""
import ctypes

import pytest


def _seg(**kw):
    from cbinfer_b200 import _lib
    a = dict(base=4096, pixels=15, pitch_bytes=16, channel_bytes=12, dtype=_lib.F32, fill=_lib.RESET_FILL_INF)
    a.update(kw)
    return _lib.ResetSegment(**a)


@pytest.mark.parametrize("bad", [
    dict(base=4098),                                  # not aligned to the 4-byte elements
    dict(dtype=7),                                    # unknown dtype
    dict(pitch_bytes=0), dict(pitch_bytes=18),        # empty pitch, pitch not a multiple of the element
    dict(channel_bytes=20),                           # channels beyond the pitch
    dict(channel_bytes=6),                            # channel bytes not a multiple of the element
    dict(pixels=-1), dict(fill=2), dict(base=0),
    dict(dtype=1, base=4097),                         # fp16: 2-byte alignment
])
def test_bad_segments_are_refused(bad):
    from cbinfer_b200 import _lib
    segs = (_lib.ResetSegment * 2)(_seg(), _seg(**bad))
    assert _lib.C.cb_reset_streams(None, ctypes.c_void_p(4096), 3, segs, 2) == 2
    assert b"reset_streams: segment 1" in _lib.C.cb_last_error()


def test_bad_calls_are_refused():
    from cbinfer_b200 import _lib
    segs = (_lib.ResetSegment * 1)(_seg())
    mask = ctypes.c_void_p(4096)
    assert _lib.C.cb_reset_streams(None, mask, 0, segs, 1) == 2          # B = 0
    assert _lib.C.cb_reset_streams(None, mask, 3, segs, -1) == 2         # negative segment count
    assert _lib.C.cb_reset_streams(None, None, 3, segs, 1) == 2          # no mask
    assert _lib.C.cb_reset_streams(None, mask, 3, None, 1) == 2          # no segments
    assert _lib.C.cb_reset_streams(None, mask, 3, None, 0) == 0          # nothing to do
    # an empty segment (no pixels) needs no base and launches nothing
    empty = (_lib.ResetSegment * 1)(_seg(base=0, pixels=0))
    assert _lib.C.cb_reset_streams(None, mask, 3, empty, 1) == 0
