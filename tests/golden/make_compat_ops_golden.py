#!/usr/bin/env python
"""Record tests/golden/compat_ops_golden.npz: THIS PROJECT's own outputs -- the compat shim's
(tests/test_gpu_compat_shim.py) and the ops' (the reference kernel tests of tests/test_gpu_modules.py)
-- for the call sequences and inputs of the tests that compare with the reference libraries.  Those
tests check against this record always, and against the unmodified reference libraries only where
oracle/_ref is built; the record is not reference output.  Needs a GPU.

Exact outputs are stored as SHA-256 digests (tests.util.digest), the fine-grained update (atomic
summation order) as arrays.

  python tests/golden/make_compat_ops_golden.py [--out PATH]     (default: next to this file)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests import test_gpu_compat_shim as shim_tests  # noqa: E402
from tests import test_gpu_modules as module_tests  # noqa: E402
from tests.util import OUTPUTS_GOLDEN, record, shim_lib  # noqa: E402


def main():
    cg, half, fg = (shim_lib(n) for n in ("cbconv2d_cg_backend", "cbconv2d_cg_half_backend", "cbconv2d_fg_backend"))
    tol = ("output",)
    g = {}
    g.update(record("shim_change_detection.cbconv2d_cg_backend", shim_tests.change_detection_outputs(cg, False)))
    g.update(record("shim_change_detection.cbconv2d_cg_half_backend", shim_tests.change_detection_outputs(half, True)))
    g.update(record("shim_propagation_gather_scatter_pool", shim_tests.propagation_gather_scatter_pool_outputs(cg)[0]))
    g.update(record("shim_half_gather_scatter_pool", shim_tests.half_gather_scatter_pool_outputs(half)))
    g.update(record("shim_fine_grained", shim_tests.fine_grained_outputs(fg), tol))
    g.update(record("ops_change_detection.f32", module_tests.ops_change_detection_outputs(False)))
    g.update(record("ops_change_detection.f16", module_tests.ops_change_detection_outputs(True)))
    g.update(record("ops_gather_scatter_pool", module_tests.ops_gather_scatter_pool_outputs()))
    g.update(record("ops_fg", module_tests.ops_fg_outputs(), tol))
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else OUTPUTS_GOLDEN
    np.savez_compressed(out, **g)
    print("wrote %s: %d entries, %d bytes" % (out, len(g), os.path.getsize(out)))


if __name__ == "__main__":
    main()
