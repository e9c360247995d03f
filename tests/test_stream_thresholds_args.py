"""CPU: the host-side argument checks of the per-stream thresholds -- every *_thr C entry point refuses
bad arguments with status 2 before anything reaches the device, and cbinfer_b200.setStreamThresholds
refuses tables and models it cannot honour (no GPU needed: nothing is launched)."""
import ctypes
import math

import pytest
import torch
import torch.nn as nn

P = ctypes.c_void_p(4096)            # a stand-in device pointer (never dereferenced: the calls fail first)
THR = ctypes.c_void_p(8192)          # a stand-in threshold table
ODD = ctypes.c_void_p(8194)          # not 4-byte aligned


def _lib():
    from cbinfer_b200 import _lib
    return _lib


def _detect(**kw):
    L = _lib()
    a = dict(dtype=L.F32, x=P, state=P, bits=P, B=2, C=3, H=5, W=7, aux=L.AUX_NONE, hi=None, lo=None,
             update=L.UPDATE_ALL, thr=THR)
    a.update(kw)
    return L.C.cb_change_detect_thr(None, a["dtype"], a["x"], 105, 35, 7, 1, a["state"], 140, 1, 28, 4,
                                    a["aux"], a["hi"], a["lo"], a["bits"], a["B"], a["C"], a["H"], a["W"],
                                    0.1, a["update"], None, a["thr"])


def _detect_u8(**kw):
    L = _lib()
    a = dict(x=P, state=P, bits=P, B=2, C=3, H=5, W=7, s_sx=4, divisor=255.0, update=L.UPDATE_ALL, thr=THR)
    a.update(kw)
    return L.C.cb_change_detect_u8_thr(None, a["x"], 105, 35, 7, 1, a["state"], 140, 1, 28, a["s_sx"],
                                       L.AUX_NONE, None, None, a["bits"], a["B"], a["C"], a["H"], a["W"],
                                       a["divisor"], 0.0, 0.1, a["update"], None, a["thr"])


def _sparse(**kw):
    L = _lib()
    a = dict(dtype=L.F32, x=P, state=P, bits=P, cand=P, ncand=P, B=2, C=3, H=5, W=7, update=L.UPDATE_ALL,
             thr=THR)
    a.update(kw)
    return L.C.cb_change_detect_sparse_thr(None, a["dtype"], a["x"], 140, 1, 28, 4, a["state"], 140, 1, 28, 4,
                                           L.AUX_NONE, None, None, a["cand"], a["ncand"], a["bits"], a["B"],
                                           a["C"], a["H"], a["W"], 0.1, a["update"], 1, a["thr"])


def _sparse_compact(**kw):
    L = _lib()
    a = dict(x=P, state=P, bits=P, cand=P, ncand=P, idx=P, count=P, sync=P, dil=P, B=2, C=3, H=5, W=7,
             kw_half=1, sc=None, acc=None, thr=THR)
    a.update(kw)
    return L.C.cb_change_detect_sparse_compact_thr(
        None, L.F32, a["x"], 140, 1, 28, 4, a["state"], 140, 1, 28, 4, L.AUX_NONE, None, None, a["cand"],
        a["ncand"], a["bits"], a["B"], a["C"], a["H"], a["W"], 0.1, L.UPDATE_ALL, 1, a["dil"], a["idx"],
        a["count"], a["sync"], 1, a["kw_half"], 1, a["sc"], a["acc"], a["thr"])


def _pool_detect(**kw):
    L = _lib()
    a = dict(x=P, idx=P, count=P, bits=P, out=P, nst=P, nbits=P, pitch=4, update=L.UPDATE_ALL, thr=THR)
    a.update(kw)
    return L.C.cb_maxpool2x2_detect_thr(None, L.F32, a["x"], 140, 28, a["pitch"], a["idx"], a["count"], a["bits"],
                                        a["out"], 48, 12, 4, 2, 3, 5, 7, 2, 3, a["nst"], 48, 12, 4, L.AUX_NONE, None,
                                        None, a["nbits"], 0.1, a["update"], a["thr"])


def _tiled_pool(**kw):
    L = _lib()
    a = dict(pool=P, nst=P, nbits=P, o_pitch=16, update=L.UPDATE_ALL, thr=THR)
    a.update(kw)
    return L.C.cb_conv_update_tiled_pool_thr(None, L.F32, L.GEMM_TC_BF16X3, P, P, 16, P, P, P, P, P, 16, 2, 16, 16,
                                             16, 16, 3, 3, 1, a["pool"], 1024, 128, a["o_pitch"], 8, 8, a["nst"], 1024,
                                             128, 16, L.AUX_NONE, None, None, a["nbits"], 0.1, a["update"], a["thr"])


def _tail(**kw):
    L = _lib()
    a = dict(x=P, cand=P, B=2, hw=35, update=L.UPDATE_ALL, t1=THR, t2=THR)
    a.update(kw)
    return L.C.cb_tail_update_thr(None, a["x"], P, P, P, P, 1, 0.1, P, P, P, P, 8, 0, 0.1, a["cand"], P, 64, 64, 8,
                                  a["update"], P, P, P, a["B"], a["hw"], None, None, None, None, a["t1"], a["t2"])


@pytest.mark.parametrize("bad", [
    dict(x=None), dict(state=None), dict(bits=None),          # null pointers
    dict(B=-1), dict(C=0), dict(H=-1), dict(W=-2),            # bad shapes
    dict(dtype=7),                                            # unknown dtype
    dict(aux=3), dict(aux=1, lo=None),                        # bad operand-plane mode / missing plane
    dict(dtype=1, aux=2, hi=P, lo=P),                         # operand planes of 16-bit data
    dict(update=5),                                           # unknown update mode
    dict(thr=ODD),                                            # misaligned threshold table
])
def test_detect_thr_refuses_bad_arguments(bad):
    assert _detect(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(x=None), dict(state=None), dict(bits=None), dict(B=-1), dict(C=0),
                                 dict(C=5), dict(s_sx=8), dict(divisor=0.0), dict(update=5), dict(thr=ODD)])
def test_detect_u8_thr_refuses_bad_arguments(bad):
    assert _detect_u8(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(x=None), dict(state=None), dict(bits=None), dict(cand=None), dict(ncand=None),
                                 dict(B=-1), dict(C=0), dict(dtype=7), dict(thr=ODD)])
def test_detect_sparse_thr_refuses_bad_arguments(bad):
    assert _sparse(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(idx=None), dict(count=None), dict(sync=None), dict(cand=None), dict(B=-1),
                                 dict(kw_half=32), dict(dil=P, bits=P), dict(sc=P, acc=None), dict(thr=ODD)])
def test_detect_sparse_compact_thr_refuses_bad_arguments(bad):
    assert _sparse_compact(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(x=None), dict(idx=None), dict(bits=None), dict(out=None), dict(nst=None),
                                 dict(nbits=None), dict(pitch=6), dict(update=5), dict(thr=ODD)])
def test_pool_detect_thr_refuses_bad_arguments(bad):
    assert _pool_detect(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(pool=None), dict(nst=None), dict(nbits=None), dict(update=5), dict(o_pitch=12),
                                 dict(thr=ODD)])
def test_tiled_pool_thr_refuses_bad_arguments(bad):
    assert _tiled_pool(**bad) == 2
    assert _lib().C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(x=None), dict(cand=None), dict(update=5), dict(B=0), dict(hw=0),
                                 dict(t1=None, hw=0), dict(t1=ODD), dict(t2=ODD)])
def test_tail_thr_refuses_bad_arguments(bad):
    assert _tail(**bad) == 2
    assert _lib().C.cb_last_error()


def test_empty_frame_launches_nothing():
    assert _detect(B=0) == 0 and _detect(H=0) == 0
    assert _detect_u8(B=0) == 0 and _detect_u8(W=0) == 0


def _model(**flags):
    import cbinfer_b200 as cb
    torch.manual_seed(0)
    m = cb.convert(nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 4, 1)), threshold=0.1)
    for c in m.modules():
        if type(c) is cb.CBConv2d:
            for k, v in flags.items():
                setattr(c, k, v)
    return m


def test_set_stream_thresholds_refuses_what_it_cannot_honour():
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    m = _model()
    with pytest.raises(CBinferError, match="fine-grained"):
        cb.setStreamThresholds(_model(finegrained=True), [[0.1, 0.1], [0.1, 0.1]])
    with pytest.raises(CBinferError, match="gatherComputationStats"):
        cb.setStreamThresholds(_model(gatherComputationStats=True), [[0.1, 0.1], [0.1, 0.1]])
    for bad in ([0.1, 0.1], [[0.1, 0.1]], [[0.1, 0.1], [0.1, 0.1], [0.1, 0.1]]):
        with pytest.raises(CBinferError, match="table"):
            cb.setStreamThresholds(m, bad)                    # not [L = 2, B]
    for v in (math.nan, math.inf, -math.inf, 1e40):          # (1e40 is infinite in fp32)
        with pytest.raises(CBinferError, match="NaN or infinite"):
            cb.setStreamThresholds(m, [[0.1, v], [0.1, 0.1]])
    # B known from the layers' (here host-side) state: a table of another width is refused
    convs = [c for c in m.modules() if type(c) is cb.CBConv2d]
    convs[0]._inBuf = torch.zeros(4, 5, 7, 4)
    with pytest.raises(CBinferError, match="table"):
        cb.setStreamThresholds(m, [[0.1] * 3, [0.1] * 3])
    with pytest.raises(CBinferError, match="CUDA device"):
        cb.setStreamThresholds(m, [[0.1] * 4, [0.1] * 4])   # a CPU model: the table cannot live there
    assert all(c._thrRow is None for c in convs)             # refused calls attach nothing
    assert cb.setStreamThresholds(m, None) == []              # detaching without a table: a no-op
    with pytest.raises(CBinferError, match="no per-stream thresholds"):
        cb.streamThresholds(m)


def test_thr_wrapper_refuses_a_host_table():
    from cbinfer_b200 import conv2d_cg as cg
    from cbinfer_b200._lib import CBinferError
    with pytest.raises(CBinferError):
        cg._thr_ptr(torch.ones(2), 2, torch.device("cuda", 0))


def test_old_pickles_load_without_a_table():
    """A CBConv2d pickled before per-stream thresholds existed loads with none."""
    import pickle
    c = _model()[0]
    del c.__dict__["_thrRow"]
    del c.__dict__["_lastPlain"]
    c2 = pickle.loads(pickle.dumps(c))
    assert c2._thrRow is None and c2._lastPlain is None
