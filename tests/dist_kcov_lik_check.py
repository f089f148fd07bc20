"""Run under torchrun on 2 GPUs (tests/test_gpu_kcov_lik.py::test_two_ranks_unsupported): the likelihood needs the dense
factor, which is single-GPU, so gsi_kernelcov_loglik on a context of two ranks is refused with GSI_ERR_UNSUPPORTED;
writes the status to <outdir>/lik_rank<r>.txt."""
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
    op = gsi.KernelCovMatrix("exponential", coords, [2.0, 2.0], nugget=0.1, ctx=ctx, row0=r0, mloc=ml)
    y = np.ones(n)
    pd = C.POINTER(C.c_double)
    val, col = C.c_double(0.0), C.c_int64(-1)
    status = ctx._lib.gsi_kernelcov_loglik(op._h, y.ctypes.data_as(pd), None, 0, 0, C.byref(val), None, None,
                                           C.byref(col))
    with open(os.path.join(outdir, f"lik_rank{ctx.rank}.txt"), "w") as f:
        f.write(f"{status}\n")
    ctx.sync()


if __name__ == "__main__":
    main()
