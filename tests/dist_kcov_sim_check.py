"""Run under torchrun on 2 GPUs (tests/test_gpu_kcov_sim.py::test_two_ranks_unsupported): simulation needs the dense
factor of the joint matrix, which is single-GPU, so gsi_kernelcov_chol_diag on a context of two ranks is refused with
GSI_ERR_UNSUPPORTED; writes the status to <outdir>/sim_rank<r>.txt."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import gsi_b200 as gsi            # noqa: E402
from gsi_b200 import dist as gdist  # noqa: E402


def main():
    outdir = sys.argv[1]
    ctx = gdist.context_from_torch_distributed()
    assert ctx.world == 2
    n = 500
    coords = np.random.default_rng(3).uniform(0, 10, (2, n))
    r0, ml = gsi.partition_rows(n, ctx.world, ctx.rank)
    op = gsi.KernelCovMatrix("exponential", coords, [2.0, 2.0], ctx=ctx, row0=r0, mloc=ml)
    d = np.full(n, 0.1)
    h, col = C.c_void_p(), C.c_int64(-1)
    status = ctx._lib.gsi_kernelcov_chol_diag(op._h, d.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h), C.byref(col))
    with open(os.path.join(outdir, f"sim_rank{ctx.rank}.txt"), "w") as f:
        f.write(f"{status} {int(bool(h))}\n")
    ctx.sync()


if __name__ == "__main__":
    main()
