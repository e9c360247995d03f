"""The reference's own FFI symbols, bound the way the reference binds them (cdef prototypes of
pycbinfer/conv2d_cg.py:6-38 and conv2d_fg.py:13-29, launch geometry of its wrappers), exported by the
compatibility shim built from cbinfer_b200/csrc/compat_shim.cu on top of libcbinfer_sm100.so
(cbinfer_b200/compat/).  Identical call sequences, identical inputs, checked against
  * the UNMODIFIED reference libraries (oracle/_ref, compiled from the reference's sources by
    oracle/Makefile) where they are built: this is the evidence that the unmodified reference python
    files can run on the sm_100a kernels by swapping the three .so files;
  * always, the shim's own outputs as tests/golden/make_compat_ops_golden.py recorded them
    (tests/golden/compat_ops_golden.npz): a regression record of this project, not reference output.
Change maps, feedback state, im2col matrix, scattered output and pooled map must be bit-identical, the
fine-grained update within 1e-4 (atomic summation order)."""
import ctypes

import pytest
import torch

from tests.util import compare_outputs, rand_tensor, perturb, shim_lib, vp

pytestmark = pytest.mark.gpu


def _change_detection(lib, x, prev, k, thr, update):
    """conv2d_cg.py:100-122"""
    H, W = x.shape[-2:]
    cmap = torch.zeros(H, W, dtype=torch.int8, device="cuda")
    st = prev.clone()
    lib.changeDetection(1, 1, (H * W - 1) // 128 + 1, 1, 1, 128, vp(x), vp(st), vp(cmap), W, H, x.shape[1],
                        (k - 1) // 2, (k - 1) // 2, ctypes.c_float(thr), ctypes.c_bool(update))
    torch.cuda.synchronize()
    return cmap, st


def change_detection_outputs(lib, half):
    dt = "f16" if half else "f32"
    outs = {}
    for (C, H, W, k, thr) in ((16, 40, 30, 3, 0.1), (3, 15, 20, 7, 0.4), (64, 33, 65, 1, 0.6), (5, 9, 130, 5, 0.5)):
        prev = rand_tensor((1, C, H, W), dt, C + H)
        x = perturb(prev, 0.08, C + 3)
        for update in (False, True):
            cmap, st = _change_detection(lib, x, prev, k, thr, update)
            outs["map_%d_%d_%d_%d" % (C, H, W, update)] = cmap
            outs["state_%d_%d_%d_%d" % (C, H, W, update)] = st
    return outs


@pytest.mark.parametrize("half", [False, True])
def test_shim_change_detection_equals_reference_library(half):
    name = "cbconv2d_cg_half_backend" if half else "cbconv2d_cg_backend"
    outs = change_detection_outputs(shim_lib(name), half)
    assert all(int(m.sum()) > 0 for n, m in outs.items() if n.startswith("map_"))
    compare_outputs("shim_change_detection.%s" % name, name, outs, lambda L: change_detection_outputs(L, half))


def test_shim_reference_kat_15_pixels():
    """genTestData + changeDetection_test1 (conv2d_cg.py:84-98,136-142): two of the four perturbed points
    exceed the threshold; with a 3x3 filter the dilated map holds 6 + 9 pixels (one point sits on the border)"""
    shim = shim_lib("cbconv2d_cg_backend")
    torch.manual_seed(10)
    x = torch.randn(1, 16, 400, 300, device="cuda")
    prev = x.clone()
    for c, y, xx, d in ((0, 0, 4, 1.00), (1, 6, 9, 0.05), (2, 10, 4, -11.00), (1, 6, 19, -0.05)):
        prev[0, c, y, xx] += d
    cmap, _ = _change_detection(shim, x, prev, 3, 0.1, False)
    assert int(cmap.sum()) == 15
    assert sorted(torch.nonzero(cmap.view(-1)).view(-1).tolist())[:3] == [3, 4, 5]


def propagation_gather_scatter_pool_outputs(lib):
    g = torch.Generator().manual_seed(5)
    C, Cout, H, W, k = 6, 10, 37, 45, 5
    # changePropagation (conv2d_cg.py:159-177)
    raw = (torch.rand(H, W, generator=g) < 0.03).to(torch.int8).cuda()
    prop = torch.zeros(H, W, dtype=torch.int8, device="cuda")
    lib.changePropagation(1, 1, (H * W - 1) // 128 + 1, 1, 1, 128, vp(raw), vp(prop), W, H,
                          (k - 1) // 2, (k - 1) // 2)                          # geometry of conv2d_cg.py:166-170
    torch.cuda.synchronize()
    # genXMatrix (conv2d_cg.py:239-261), updateOutput (:292-313), maxPool2d (:58-82); the index list is
    # the one of the propagated map the reference returns
    x = rand_tensor((1, C, H, W), "f32", 1)
    idx = torch.nonzero(prop.view(-1)).view(-1).int().cuda()
    n = idx.numel()
    tz = 128 // (k * k)
    Yt = rand_tensor((Cout, n), "f32", 3)
    po = rand_tensor((1, Cout, H, W), "f32", 4)
    xe = rand_tensor((1, C, 36, 52), "f32", 5)
    idx2 = torch.nonzero(torch.rand(36 * 52, generator=g) < 0.2).view(-1).int().cuda()
    X = torch.zeros(n, C * k * k, device="cuda")
    lib.genXMatrix(1, 1, (n - 1) // tz + 1, k, tz, k, vp(X), vp(x), vp(idx), k, k, C, W, H, n)
    lib.updateOutput(1, 1, (n * Cout - 1) // 1024 + 1, 1, 1, 1024, vp(Yt), vp(po), vp(idx), H * W, n, Cout,
                     ctypes.c_bool(True))
    st = torch.full((1, C, 18, 26), float("inf"), device="cuda")
    lib.maxPool2d((idx2.numel() - 1) // 64 + 1, 64, vp(xe), vp(st), vp(idx2), idx2.numel(), C, 36, 52, 18, 26, 2, 2)
    torch.cuda.synchronize()
    return {"propagated": prop, "xmatrix": X, "output": po, "pooled": st}, raw


def test_shim_propagation_gather_scatter_pool_equal_reference_library():
    outs, raw = propagation_gather_scatter_pool_outputs(shim_lib("cbconv2d_cg_backend"))
    assert int(outs["propagated"].sum()) > int(raw.sum())
    compare_outputs("shim_propagation_gather_scatter_pool", "cbconv2d_cg_backend", outs,
             lambda L: propagation_gather_scatter_pool_outputs(L)[0])


def half_gather_scatter_pool_outputs(lib):
    g = torch.Generator().manual_seed(6)
    C, Cout, H, W, k = 8, 12, 30, 44, 3
    x = rand_tensor((1, C, H, W), "f16", 1)
    idx = torch.nonzero(torch.rand(H * W, generator=g) < 0.2).view(-1).int().cuda()
    n = idx.numel()
    tz = 128 // (k * k)
    Yt = rand_tensor((Cout, n), "f16", 3)
    po = rand_tensor((1, Cout, H, W), "f16", 4)
    idx2 = torch.nonzero(torch.rand(H * W, generator=g) < 0.2).view(-1).int().cuda()
    X = torch.zeros(n, C * k * k, device="cuda", dtype=torch.float16)
    lib.genXMatrix(1, 1, (n - 1) // tz + 1, k, tz, k, vp(X), vp(x), vp(idx), k, k, C, W, H, n)
    lib.updateOutput(1, 1, (n * Cout - 1) // 1024 + 1, 1, 1, 1024, vp(Yt), vp(po), vp(idx), H * W, n, Cout,
                     ctypes.c_bool(False))
    st = torch.full((1, C, H // 2, W // 2), float("inf"), device="cuda", dtype=torch.float16)
    lib.maxPool2d((idx2.numel() - 1) // 64 + 1, 64, vp(x), vp(st), vp(idx2), idx2.numel(), C, H, W, H // 2, W // 2, 2, 2)
    torch.cuda.synchronize()
    return {"xmatrix": X, "output": po, "pooled": st}


def test_shim_half_gather_scatter_pool_equal_reference_library():
    outs = half_gather_scatter_pool_outputs(shim_lib("cbconv2d_cg_half_backend"))
    compare_outputs("shim_half_gather_scatter_pool", "cbconv2d_cg_half_backend", outs, half_gather_scatter_pool_outputs)


def fine_grained_outputs(lib):
    Cin, Cout, H, W, k = 5, 7, 21, 26, 3
    prev = rand_tensor((1, Cin, H, W), "f32", 1)
    x = perturb(prev, 0.1, 2)
    w = rand_tensor((Cout, Cin, k, k), "f32", 3, scale=0.3)
    out = rand_tensor((1, Cout, H, W), "f32", 4)
    diffs = torch.zeros_like(x)
    cmap = torch.zeros(x.shape, dtype=torch.int8, device="cuda")
    lib.changeDetectionFG(vp(x), vp(prev), vp(diffs), vp(cmap), x.numel(), ctypes.c_float(0.2))
    torch.cuda.synchronize()
    coords = torch.nonzero(cmap.view(-1)).view(-1).contiguous()          # conv2d_fg.py:82
    lib.updateOutputFG(1, 1, (coords.numel() - 1) // 128 + 1, 1, 1, 128, vp(diffs), vp(w), vp(out), vp(coords),
                       Cout, Cin, H, W, k, k, coords.numel())
    torch.cuda.synchronize()
    return {"map": cmap, "diffs": diffs, "output": out}


def test_shim_fine_grained_equals_reference_library():
    outs = fine_grained_outputs(shim_lib("cbconv2d_fg_backend"))
    assert int(outs["map"].sum()) > 0
    compare_outputs("shim_fine_grained", "cbconv2d_fg_backend", outs, fine_grained_outputs, tol={"output": (1e-5, 1e-4)})
