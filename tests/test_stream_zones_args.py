"""CPU: the host-side argument checks of watched-pixel zones -- cb_change_detect_zone and
cb_change_detect_u8_zone refuse a misaligned zone and a zone on a layout the narrow kernel cannot take
with status 2, and with a NULL zone behave as the *_thr entry points; cbinfer_b200.setStreamZones refuses
zones and models it cannot honour (no GPU needed: nothing is launched)."""
import ctypes

import pytest
import torch
import torch.nn as nn

P = ctypes.c_void_p(4096)            # a stand-in device pointer (never dereferenced: the calls fail first)
THR = ctypes.c_void_p(8192)          # a stand-in threshold table
ZONE = ctypes.c_void_p(12288)        # a stand-in zone bitmap
ODD = ctypes.c_void_p(12290)         # not 4-byte aligned


def _lib():
    from cbinfer_b200 import _lib
    return _lib


def _detect(fn, **kw):
    """cb_change_detect_{thr,zone}: planar fp32 x [2, C, 5, 7]; the state pixel-major of pitch s_sx"""
    L = _lib()
    a = dict(dtype=L.F32, x=P, state=P, bits=P, B=2, C=3, H=5, W=7, aux=L.AUX_NONE, hi=None, lo=None,
             update=L.UPDATE_ALL, thr=THR, s_sc=1, s_sx=4, zone=ZONE)
    a.update(kw)
    C_, s_sx = a["C"], a["s_sx"]
    args = [None, a["dtype"], a["x"], C_ * 35, 35, 7, 1, a["state"], 35 * s_sx, a["s_sc"], 7 * s_sx, s_sx,
            a["aux"], a["hi"], a["lo"], a["bits"], a["B"], C_, a["H"], a["W"], 0.1, a["update"], None, a["thr"]]
    if fn == "zone":
        return L.C.cb_change_detect_zone(*args, a["zone"])
    return L.C.cb_change_detect_thr(*args)


def _detect_u8(fn, **kw):
    L = _lib()
    a = dict(x=P, state=P, bits=P, B=2, C=3, H=5, W=7, s_sx=4, divisor=255.0, update=L.UPDATE_ALL, thr=THR,
             zone=ZONE)
    a.update(kw)
    args = [None, a["x"], 105, 35, 7, 1, a["state"], 140, 1, 28, a["s_sx"], L.AUX_NONE, None, None, a["bits"],
            a["B"], a["C"], a["H"], a["W"], a["divisor"], 0.0, 0.1, a["update"], None, a["thr"]]
    if fn == "zone":
        return L.C.cb_change_detect_u8_zone(*args, a["zone"])
    return L.C.cb_change_detect_u8_thr(*args)


def _outcome(call):
    status = call()
    return status, _lib().C.cb_last_error() if status else None


# argument sets the *_thr entry points refuse (and one they accept: an empty frame launches nothing)
THR_CASES = [dict(x=None), dict(state=None), dict(bits=None), dict(B=-1), dict(C=0), dict(W=-2), dict(dtype=7),
             dict(aux=3), dict(update=5), dict(thr=ctypes.c_void_p(8194)), dict(B=0), dict(H=0)]
U8_CASES = [dict(x=None), dict(state=None), dict(B=-1), dict(C=5), dict(s_sx=8), dict(divisor=0.0), dict(update=5),
            dict(thr=ctypes.c_void_p(8194)), dict(B=0), dict(W=0)]


@pytest.mark.parametrize("case", THR_CASES)
def test_null_zone_is_the_thr_call(case):
    assert _outcome(lambda: _detect("zone", zone=None, **case)) == _outcome(lambda: _detect("thr", **case))


@pytest.mark.parametrize("case", U8_CASES)
def test_null_zone_is_the_thr_call_u8(case):
    assert _outcome(lambda: _detect_u8("zone", zone=None, **case)) == _outcome(lambda: _detect_u8("thr", **case))


@pytest.mark.parametrize("dtype_name", ["F32", "F16", "BF16"])
def test_misaligned_zone_is_refused(dtype_name):
    dt = getattr(_lib(), dtype_name)
    assert _detect("zone", dtype=dt, s_sx=4 if dt == _lib().F32 else 8, zone=ODD) == 2
    assert b"zone" in _lib().C.cb_last_error()
    assert _detect_u8("zone", zone=ODD) == 2
    assert b"zone" in _lib().C.cb_last_error()


@pytest.mark.parametrize("case", [
    dict(C=5, s_sx=8),                   # fp32: two 16-byte chunks per pixel (vec / planar kernels)
    dict(C=16, s_sx=16),                 # fp32, planar x: the planar kernel
    dict(dtype=2, C=9, s_sx=16),         # bf16: more than 8 channels
    dict(C=3, s_sc=35, s_sx=1),          # planar state: the generic kernel
    dict(C=3, s_sx=8),                   # fp32 state of pitch 8 (not one chunk per pixel)
])
def test_zone_without_the_narrow_kernel_is_refused(case):
    assert _detect("zone", **case) == 2
    assert b"zone" in _lib().C.cb_last_error()


def test_zone_of_an_empty_frame_launches_nothing():
    assert _detect("zone", B=0) == 0 and _detect("zone", W=0) == 0
    assert _detect_u8("zone", B=0) == 0 and _detect_u8("zone", H=0) == 0


def _model(**flags):
    import cbinfer_b200 as cb
    torch.manual_seed(0)
    m = cb.convert(nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU(), nn.Conv2d(8, 4, 1)), threshold=0.1)
    for c in m.modules():
        if type(c) is cb.CBConv2d:
            for k, v in flags.items():
                setattr(c, k, v)
    return m


def test_set_stream_zones_refuses_what_it_cannot_honour():
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    ok = torch.ones(2, 5, 7, dtype=torch.bool)
    with pytest.raises(CBinferError, match="fine-grained"):
        cb.setStreamZones(_model(finegrained=True), ok)
    with pytest.raises(CBinferError, match="gatherComputationStats"):
        cb.setStreamZones(_model(gatherComputationStats=True), ok)
    with pytest.raises(CBinferError, match="no CBConv2d"):
        cb.setStreamZones(nn.Sequential(nn.ReLU()), ok)
    m = _model()
    for bad in (torch.ones(5, 7, dtype=torch.bool), torch.ones(1, 2, 5, 7, dtype=torch.bool),
                torch.ones(2, 5, 7), torch.ones(2, 5, 7, dtype=torch.int32), [[[1]]]):
        with pytest.raises(CBinferError, match="bool or uint8 tensor"):
            cb.setStreamZones(m, bad)
    with pytest.raises(CBinferError, match="CUDA device"):
        cb.setStreamZones(m, ok)                             # a CPU model: the zone cannot live there
    assert all(c._zone is None for c in m.modules() if type(c) is cb.CBConv2d)   # refused calls attach nothing
    assert cb.setStreamZones(m, None) == "0"                 # detaching: the zone layer's name


def test_zone_wrapper_refuses_a_host_bitmap():
    from cbinfer_b200 import conv2d_cg as cg
    from cbinfer_b200._lib import CBinferError
    with pytest.raises(CBinferError):
        cg._zone_ptr(torch.ones(2 * 5, dtype=torch.int32), 2, 5, 7, torch.device("cuda", 0))


def test_old_pickles_load_without_a_zone():
    """A CBConv2d pickled before zones existed loads with none; clearMemory keeps an attached one."""
    import pickle
    c = _model()[0]
    del c.__dict__["_zone"]
    c2 = pickle.loads(pickle.dumps(c))
    assert c2._zone is None
    c2._zone = ("bits", (2, 5, 7), "stage")
    c2.clearMemory()
    assert c2._zone == ("bits", (2, 5, 7), "stage")
