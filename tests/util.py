"""helpers shared by the GPU parity tests: torch <-> oracle (numpy) plumbing."""
import ctypes
import hashlib
import os
import platform

import numpy as np
import torch

from oracle import oracle as orc

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TORCH_DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
ORC_DT = {"f32": orc.F32, "f16": orc.F16, "bf16": orc.BF16}


def to_np(t):
    """torch tensor (any device / layout) -> oracle storage array in planar NCHW order."""
    return orc.from_torch(t.detach().cpu().contiguous())[0]


def to_val(t):
    return t.detach().cpu().contiguous().double().numpy()


def bits_to_map(bits, B, H, W):
    """int32 bitmap tensor -> uint8 [B,H,W] numpy map."""
    Wd = (W + 31) // 32
    words = bits.detach().cpu().numpy().view(np.uint32)[: B * H * Wd].reshape(B * H, Wd)
    m = ((words[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).astype(np.uint8)
    return m.reshape(B * H, Wd * 32)[:, :W].reshape(B, H, W)


def rand_tensor(shape, dt, seed, scale=1.0, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(TORCH_DT[dt]).to(device)


def perturb(x, frac, seed, scale=1.0):
    """copy of x with ~frac of the *pixels* changed in a random subset of channels."""
    g = torch.Generator().manual_seed(seed)
    B, C, H, W = x.shape
    pm = (torch.rand(B, 1, H, W, generator=g) < frac)
    cm = (torch.rand(B, C, H, W, generator=g) < 0.5)
    d = torch.randn(B, C, H, W, generator=g) * scale
    y = x.detach().cpu().float() + (pm & cm).float() * d
    return y.to(x.dtype).to(x.device)


def ref_lib(name):
    """ctypes handle of an UNMODIFIED reference library compiled into oracle/_ref (or None)."""
    p = os.path.join(REPO, "oracle", "_ref", "%s_%s.so" % (name, platform.machine()))
    if not os.path.exists(p):
        return None
    return ctypes.CDLL(p)


def shim_lib(name):
    """ctypes handle of the compatibility shim that exports the reference library `name`'s symbols
    on top of libcbinfer_sm100.so (cbinfer_b200/compat, built by build_compat)."""
    p = os.path.join(REPO, "cbinfer_b200", "compat", "%s_%s.so" % (name, platform.machine()))
    if not os.path.exists(p):
        from cbinfer_b200 import build
        build.build_compat()
    return ctypes.CDLL(p)


OUTPUTS_GOLDEN = os.path.join(REPO, "tests", "golden", "compat_ops_golden.npz")


def digest(t):
    """SHA-256 of a tensor's dtype, shape and bytes: bit-exact comparison with a recorded output."""
    a = t.detach().contiguous().cpu()
    h = hashlib.sha256(("%s %s " % (a.dtype, tuple(a.shape))).encode())
    h.update(a.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def recorded_outputs():
    """this project's own outputs (compat shim and ops) on the inputs of the tests that compare with
    the reference libraries, as tests/golden/make_compat_ops_golden.py recorded them"""
    return np.load(OUTPUTS_GOLDEN)


def record(prefix, outs, tol=()):
    """{prefix.name: digest} of the tensors in `outs`, an array instead for the names in `tol`"""
    return {"%s.%s" % (prefix, n): (t.detach().float().cpu().numpy() if n in tol else np.array(digest(t)))
            for n, t in outs.items()}


def check_outputs(expected, prefix, outs, tol={}):
    """`outs` ({name: tensor}) against `expected` (a record() of other outputs): bit-exact by digest,
    or within (rtol, atol) for the names in `tol`"""
    for name, t in outs.items():
        key = "%s.%s" % (prefix, name)
        if name in tol:
            np.testing.assert_allclose(t.detach().float().cpu().numpy(), expected[key], *tol[name], err_msg=key)
        else:
            assert digest(t) == str(expected[key]), key


def compare_outputs(prefix, name, outs, outputs_of, tol={}):
    """`outs` against this project's recorded outputs and, where oracle/_ref holds the reference
    library `name`, against `outputs_of(that library)` for the same calls"""
    check_outputs(recorded_outputs(), prefix, outs, tol)
    ref = ref_lib(name)
    if ref is not None:
        check_outputs(record(prefix, outputs_of(ref), tol), prefix, outs, tol)


def vp(t):
    return ctypes.c_void_p(t.data_ptr())
