"""Run under torchrun on 2 GPUs (tests/test_gpu_kcov_cross.py::test_two_ranks): the targets of a cross-covariance operator
are split unevenly and not 64-aligned (rank 1 starts at an odd row); each rank saves its rows of C X, the all-reduced
C' X and its (replicated) randsvd Z to <outdir>/cross_rank<r>.npz for the test to compare with one rank and the oracle."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gsi_b200 as gsi            # noqa: E402
from gsi_b200 import dist as gdist  # noqa: E402
from test_gpu_kcov_cross import DIST_SPLIT, dist_case  # noqa: E402


def main():
    outdir = sys.argv[1]
    ctx = gdist.context_from_torch_distributed()
    assert ctx.world == 2
    structures, T, S, X, Xt = dist_case()
    m, n = T.shape[1], S.shape[1]
    r0, ml = (0, DIST_SPLIT) if ctx.rank == 0 else (DIST_SPLIT, m - DIST_SPLIT)
    op = gsi.KernelCrossCovMatrix(structures, T, S, ctx=ctx, row0=r0, mloc=ml)
    Y = op.apply(gsi.DeviceMatrix.from_host(ctx, X)).numpy()
    Yt = op.apply(gsi.DeviceMatrix.from_host(ctx, Xt), trans=True).numpy()
    K, p, q = 20, 10, 1
    Omega = np.random.default_rng(5).standard_normal((n, K + p))
    Z = gsi.randsvd(op, K, p, q, Omega=Omega, normaliser=gsi.NORMALISER_LU_REF)
    np.savez(os.path.join(outdir, f"cross_rank{ctx.rank}.npz"), row0=r0, Y=Y, Yt=Yt, Z=Z)
    ctx.sync()


if __name__ == "__main__":
    main()
