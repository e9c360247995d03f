"""CPU: the host-side argument checks of the active-stream mask -- the C entry points
cb_change_detect_streams / cb_change_detect_u8_streams refuse bad arguments with a status code
before anything reaches the device, and cbinfer_b200.setActiveStreams refuses what it cannot honour
(no GPU needed: nothing is launched)."""
import ctypes

import pytest
import torch
import torch.nn as nn

P = ctypes.c_void_p(4096)            # a stand-in device pointer (never dereferenced: the calls fail first)
MASK = ctypes.c_void_p(8192)


def _detect(**kw):
    from cbinfer_b200 import _lib
    a = dict(dtype=_lib.F32, x=P, state=P, bits=P, B=2, C=3, H=5, W=7, aux=_lib.AUX_NONE, hi=None, lo=None,
             update=_lib.UPDATE_ALL)
    a.update(kw)
    return _lib.C.cb_change_detect_streams(None, a["dtype"], a["x"], 105, 35, 7, 1, a["state"], 140, 1, 28, 4,
                                           a["aux"], a["hi"], a["lo"], a["bits"], a["B"], a["C"], a["H"], a["W"],
                                           0.1, a["update"], MASK)


def _detect_u8(**kw):
    from cbinfer_b200 import _lib
    a = dict(x=P, state=P, bits=P, B=2, C=3, H=5, W=7, s_sx=4, divisor=255.0, update=_lib.UPDATE_ALL)
    a.update(kw)
    return _lib.C.cb_change_detect_u8_streams(None, a["x"], 105, 35, 7, 1, a["state"], 140, 1, 28, a["s_sx"],
                                              _lib.AUX_NONE, None, None, a["bits"], a["B"], a["C"], a["H"], a["W"],
                                              a["divisor"], 0.0, 0.1, a["update"], MASK)


@pytest.mark.parametrize("bad", [
    dict(x=None), dict(state=None), dict(bits=None),          # null pointers
    dict(B=-1), dict(C=0), dict(H=-1), dict(W=-2),            # bad shapes
    dict(dtype=7),                                            # unknown dtype
    dict(aux=3), dict(aux=1, lo=None),                        # bad operand-plane mode / missing plane
    dict(dtype=1, aux=2, hi=P, lo=P),                         # operand planes of 16-bit data
    dict(update=5),                                           # unknown update mode
])
def test_detect_streams_refuses_bad_arguments(bad):
    from cbinfer_b200 import _lib
    assert _detect(**bad) == 2
    assert _lib.C.cb_last_error()


@pytest.mark.parametrize("bad", [dict(x=None), dict(state=None), dict(bits=None), dict(B=-1), dict(C=0),
                                 dict(C=5), dict(s_sx=8), dict(divisor=0.0), dict(update=5)])
def test_detect_u8_streams_refuses_bad_arguments(bad):
    from cbinfer_b200 import _lib
    assert _detect_u8(**bad) == 2
    assert _lib.C.cb_last_error()


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


def test_set_active_streams_refuses_what_it_cannot_honour():
    import cbinfer_b200 as cb
    from cbinfer_b200._lib import CBinferError
    m = _model()
    with pytest.raises(CBinferError, match="CUDA tensor"):
        cb.setActiveStreams(m, torch.ones(4, dtype=torch.bool))
    with pytest.raises(CBinferError, match="not run yet"):
        cb.setActiveStreams(m, [0, 1])                      # no mask yet, no state: B unknown
    with pytest.raises(CBinferError, match="fine-grained"):
        cb.setActiveStreams(_model(finegrained=True), None)
    with pytest.raises(CBinferError, match="gatherComputationStats"):
        cb.setActiveStreams(_model(gatherComputationStats=True), [0])
    # out-of-range indices, with B known from the layers' (here host-side) state
    convs = [c for c in m.modules() if type(c) is cb.CBConv2d]
    convs[0]._inBuf = torch.zeros(4, 5, 7, 4)
    for bad in ([4], [-1], [0, 9]):
        with pytest.raises(CBinferError, match="out of range"):
            cb.setActiveStreams(m, bad)
    assert all(c._activeMask is None for c in convs)         # refused calls set nothing
    cb.setActiveStreams(m, None)                             # detaching without a mask: a no-op


def test_detect_refuses_a_host_mask():
    from cbinfer_b200 import conv2d_cg as cg
    from cbinfer_b200._lib import CBinferError
    with pytest.raises(CBinferError):
        cg._active_ptr(torch.ones(2, dtype=torch.uint8), 2, torch.device("cuda", 0))


def test_old_pickles_load_without_a_mask():
    """A CBConv2d pickled before the mask existed loads with none (every stream active)."""
    import pickle
    m = _model()
    c = m[0]
    del c.__dict__["_activeMask"]
    c2 = pickle.loads(pickle.dumps(c))
    assert c2._activeMask is None
