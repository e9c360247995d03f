"""CPU: the host-side argument checks of the per-stream change counts -- the *_streams C entry points
refuse bad arguments with a status code before anything reaches the device, and
cbinfer_b200.trackStreamChanges refuses what it cannot honour (no GPU needed: nothing is launched)."""
import ctypes

import pytest
import torch
import torch.nn as nn

P = ctypes.c_void_p(4096)            # stand-in device pointers (never dereferenced: the calls fail first)
SC = ctypes.c_void_p(8192)
ACC = ctypes.c_void_p(12288)


def _calls(sc, acc):
    """Every *_streams entry point with valid arguments except the counts row (sc, acc)."""
    from cbinfer_b200 import _lib
    C = _lib.C
    return {
        "dilate_compact": lambda: C.cb_dilate_compact_streams(None, P, None, None, P, P, P, 2, 5, 7, 1, 1, 0, sc, acc),
        "dilate_compact_tiles": lambda: C.cb_dilate_compact_tiles_streams(None, P, P, None, P, P, P, P, 2, 5, 7, 1, 1,
                                                                          0, sc, acc),
        "dilate_tiles": lambda: C.cb_dilate_tiles_streams(None, P, P, P, P, P, 2, 5, 7, 1, 1, 0, sc, acc),
        "sparse_compact": lambda: C.cb_change_detect_sparse_compact_streams(
            None, _lib.F32, P, 140, 1, 28, 4, P, 140, 1, 28, 4, _lib.AUX_NONE, None, None, P, P, P, 2, 4, 5, 7, 0.1,
            _lib.UPDATE_ALL, 0, P, P, P, P, 1, 1, 0, sc, acc),
        "masked": lambda: C.cb_conv_update_masked_streams(
            None, _lib.F32, _lib.GEMM_TC_BF16X3, P, P, 8, P, P, P, P, P, 16, 2, 5, 7, 8, 16, 1, 1, 0, None, 0,
            P, 1, P, P, sc, acc),
        "tail": lambda: C.cb_tail_update_streams(
            None, P, P, P, P, P, 1, 0.1, P, P, P, P, 8, 0, 0.1, P, P, 64, 16, 8, _lib.UPDATE_ALL, P, P, P, 2, 35,
            sc, acc, sc, acc),
        "bucket": lambda: C.cb_stream_bucket(None, P, P, 2, 35, sc, acc),
    }


@pytest.mark.parametrize("name", sorted(_calls(None, None)))
@pytest.mark.parametrize("row", ["no_acc", "aliased"])
def test_streams_entry_points_refuse_a_row_without_its_own_accumulator(name, row):
    from cbinfer_b200 import _lib
    sc, acc = (SC, None) if row == "no_acc" else (SC, SC)
    assert _calls(sc, acc)[name]() == 2
    assert b"stream_acc" in _lib.C.cb_last_error()


def test_tail_counts_both_layers_or_neither():
    from cbinfer_b200 import _lib
    C = _lib.C
    args = (None, P, P, P, P, P, 1, 0.1, P, P, P, P, 8, 0, 0.1, P, P, 64, 16, 8, _lib.UPDATE_ALL, P, P, P)
    assert C.cb_tail_update_streams(*args, 2, 35, SC, ACC, None, None) == 2
    assert C.cb_tail_update_streams(*args, 0, 35, SC, ACC, SC, ACC) == 2      # B needed with counts


@pytest.mark.parametrize("bad", [dict(idx=None), dict(count=None), dict(sc=None), dict(B=0), dict(B=-3),
                                 dict(hw=-1), dict(B=1 << 20, hw=1 << 12)])
def test_stream_bucket_refuses_bad_arguments(bad):
    from cbinfer_b200 import _lib
    a = dict(idx=P, count=P, sc=SC, acc=ACC, B=2, hw=35)
    a.update(bad)
    assert _lib.C.cb_stream_bucket(None, a["idx"], a["count"], a["B"], a["hw"], a["sc"], a["acc"]) == 2
    assert _lib.C.cb_last_error()


def test_masked_streams_refuses_the_simt_mode():
    from cbinfer_b200 import _lib
    rc = _lib.C.cb_conv_update_masked_streams(None, _lib.F32, _lib.GEMM_SIMT_F32, P, None, 8, P, P, P, P, P, 16,
                                              2, 5, 7, 8, 16, 1, 1, 0, None, 0, P, 1, P, P, SC, ACC)
    assert rc == 2


def test_plain_entry_points_still_check_their_own_arguments():
    """The entry points without counts forward with NULL and keep refusing what they refused."""
    from cbinfer_b200 import _lib
    assert _lib.C.cb_dilate_compact(None, None, None, None, P, P, P, 2, 5, 7, 1, 1, 0) == 2
    assert _lib.C.cb_dilate_tiles(None, P, None, P, P, P, 2, 5, 7, 1, 1, 0) == 2


def _model(**flags):
    import cbinfer_b200 as cb
    torch.manual_seed(0)
    m = cb.convert(nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 4, 1)), threshold=0.1)
    for c in m.modules():
        if type(c) is cb.CBConv2d:
            for k, v in flags.items():
                setattr(c, k, v)
    return m


def test_track_stream_changes_refuses_what_it_cannot_honour():
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    with pytest.raises(CBinferError, match="not run yet"):
        cb.trackStreamChanges(_model())                       # no state, no B
    with pytest.raises(CBinferError, match="simt"):
        cb.trackStreamChanges(_model(finegrained=True, gemmMode='simt'), B=2)
    with pytest.raises(CBinferError, match="B = 0"):
        cb.trackStreamChanges(_model(), B=0)
    with pytest.raises(CBinferError, match="not tracked"):
        cb.streamChangeCounts(_model())
    m = _model()
    assert cb.trackStreamChanges(m, enable=False) == []      # detaching an untracked model: a no-op
    assert all(c._streamRow is None for c in m.modules() if type(c) is cb.CBConv2d)


def test_old_pickles_load_untracked():
    """A CBConv2d pickled before per-stream counts existed loads without a counts row."""
    import pickle
    c = _model()[0]
    del c.__dict__["_streamRow"]
    c2 = pickle.loads(pickle.dumps(c))
    assert c2._streamRow is None
