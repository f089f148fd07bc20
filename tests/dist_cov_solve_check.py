"""Run under torchrun on 2 GPUs (tests/test_gpu_cov_solve.py::test_two_ranks): each rank owns its row block of a nested-
model covariance operator and solves A X = B with and without the Nystrom preconditioner, X delivered as this rank's
rows and as all rows; saves X, the iteration counts and the residuals to <outdir>/solve_rank<r>.npz for the test to
compare with the one-rank solve."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gsi_b200 as gsi            # noqa: E402
from gsi_b200 import dist as gdist  # noqa: E402
from test_gpu_cov_solve import DIST_N, RTOL, dist_case  # noqa: E402


def main():
    outdir = sys.argv[1]
    ctx = gdist.context_from_torch_distributed()
    assert ctx.world == 2
    st, coords, nugget, B, Omega = dist_case()
    r0, ml = gsi.partition_rows(DIST_N, ctx.world, ctx.rank)
    op = gsi.KernelCovModelMatrix(st, coords, nugget, ctx=ctx, row0=r0, mloc=ml)
    out = {}
    for name, Om in (("plain", None), ("nys", Omega)):
        Xl, info = gsi.cov_solve(op, B, rtol=RTOL, Omega=Om)
        Xa, info_a = gsi.cov_solve(op, B, rtol=RTOL, Omega=Om, full=True)
        assert np.array_equal(info["iterations"], info_a["iterations"])
        out.update({f"{name}_local": Xl, f"{name}_all": Xa, f"{name}_iters": info["iterations"],
                    f"{name}_relres": info["relres"]})
    np.savez(os.path.join(outdir, f"solve_rank{ctx.rank}.npz"), **out)
    ctx.sync()


if __name__ == "__main__":
    main()
