"""Run under torchrun on 2 GPUs (tests/test_gpu_kcov_model.py::test_two_ranks_row_sharded): each rank applies its row
block of a nested-model operator (fused kernel and signed lattice table) and saves it to <outdir>/<path>_rank<r>.npz
for the test to compare with the one-rank product."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gsi_b200 as gsi            # noqa: E402
from gsi_b200 import dist as gdist  # noqa: E402
import oracle                     # noqa: E402
from test_gpu_kcov_model import models  # noqa: E402


def main():
    outdir = sys.argv[1]
    ctx = gdist.context_from_torch_distributed()
    shape = (70, 60)
    structures = models(2, shape)["three"]
    coords = oracle.grid_coords(shape)
    n = coords.shape[1]
    X = np.random.default_rng(1).standard_normal((n, 33))
    r0, ml = gsi.partition_rows(n, ctx.world, ctx.rank)
    for path in ("fused", "signed"):
        if path == "fused":
            op = gsi.KernelCovModelMatrix(structures, coords, ctx=ctx, row0=r0, mloc=ml)
        else:
            op = gsi.GridKernelCovModelMatrix(structures, shape, ctx=ctx, row0=r0, mloc=ml)
        Xd = gsi.DeviceMatrix.from_host(ctx, X)
        Y = op.apply(Xd).numpy()
        np.savez(os.path.join(outdir, f"{path}_rank{ctx.rank}.npz"), row0=r0, Y=Y)
    ctx.sync()


if __name__ == "__main__":
    main()
