#!/usr/bin/env python
"""Times single launches of the matrix-free product kernel (csrc/kcov_gemm.cu) on a structured grid.

    python tools/kcov_probe.py --grid 64,56,56 [--generation table|arithmetic] [--reps 3] [--l 210]
    python tools/kcov_probe.py --grid 32,28,28      # 25088 rows = the row schedule of one rank of C3 at 8 GPUs
    python tools/kcov_probe.py --model spherical,exponential --angle 30 [--generation table] [--separate]

--model KIND,KIND,...: a nested model (KernelCovModelMatrix / GridKernelCovModelMatrix) of one structure per kind,
structure s with sill 1/S, ranges ell * 2^s and a rotation by (-1)^s * angle degrees about the z axis (a rotated model
on the grid uses the signed lattice table).  --separate times what a user without nested models runs instead: one
single-structure operator per structure, S products (the host-side sum of their results is not counted, so the fused
speed-up over it is a lower bound).
--cross N: a cross-covariance operator C(grid, sources) of the same kernel or model (KernelCrossCovMatrix /
GridKernelCrossCovMatrix) whose targets are the grid's nodes and whose N sources are --sources grid (distinct nodes
drawn from the grid; both generation paths) or random (uniform points in the grid's box; arithmetic only).  One line
per direction: "CX" (rows = the grid, k = N) and "CtX" (rows = N, k = the grid: few rows and a long k range, the
all-SM stream-K launch); --square adds a line for the square operator of the grid in the same call.
Every line carries the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as gsi      # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def model_structures(kinds, ell, angle, d):
    S = len(kinds)
    out = []
    for s, kind in enumerate(kinds):
        a = np.deg2rad(angle) * (-1) ** s
        rot = None if angle == 0 else gsi.rotation_matrix((a,) if d == 2 else (a, 0.0, 0.0))
        out.append(gsi.CovStructure(kind, 1.0 / S, np.asarray(ell) * 2.0 ** s, rot))
    return out


def time_products(ctx, ops, X, reps, trans=False):
    for op in ops:
        op.apply(X, trans=trans).free()
    ctx.sync()
    ctx.gemm_timing(enable=True)
    for _ in range(reps):
        for op in ops:
            op.apply(X, trans=trans).free()
    ctx.sync()
    ms, nl, fl = ctx.gemm_timing(enable=False)
    return ms / reps, nl, fl / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grid", default="64,56,56")
    ap.add_argument("--ell", default="9,7,5")
    ap.add_argument("--kind", default="gaussian")
    ap.add_argument("--model", default=None, help="comma-separated kinds of a nested model")
    ap.add_argument("--angle", type=float, default=30.0, help="rotation of the model's structures, degrees")
    ap.add_argument("--separate", action="store_true", help="one single-structure operator per structure")
    ap.add_argument("--cross", type=int, default=0, help="sources of a cross-covariance operator C(grid, sources)")
    ap.add_argument("--sources", default="grid", choices=["grid", "random"])
    ap.add_argument("--square", action="store_true", help="--cross: also time the square operator of the grid")
    ap.add_argument("--generation", default="table", choices=["table", "arithmetic"])
    ap.add_argument("--l", type=int, default=210)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    grid = [int(v) for v in args.grid.split(",")]
    ell = [float(v) for v in args.ell.split(",")][:len(grid)]
    n = int(np.prod(grid))
    ctx = gsi.default_context()
    axes = np.meshgrid(*[np.arange(s, dtype=np.float64) for s in grid], indexing="ij")
    coords = np.stack([g.ravel(order="F") for g in axes], axis=0)
    if args.cross:
        cross_main(args, ctx, grid, ell, coords)
        return
    if args.model:
        structures = model_structures(args.model.split(","), ell, args.angle, len(grid))
        groups = [[s] for s in structures] if args.separate else [structures]
        if args.generation == "table":
            ops = [gsi.GridKernelCovModelMatrix(g, grid, ctx=ctx) for g in groups]
        else:
            ops = [gsi.KernelCovModelMatrix(g, coords, ctx=ctx) for g in groups]
        what = {"model": args.model, "angle_deg": args.angle, "separate": args.separate}
    else:
        if args.generation == "table":
            ops = [gsi.GridKernelCovMatrix(args.kind, grid, ell, ctx=ctx)]
        else:
            ops = [gsi.KernelCovMatrix(args.kind, coords, ell, ctx=ctx)]
        what = {"kind": args.kind}
    X = gsi.DeviceMatrix.from_host(ctx, np.random.default_rng(0).standard_normal((n, args.l)))
    ms, nl, fl = time_products(ctx, ops, X, args.reps)
    one = 2.0 * n * n * args.l                  # flops of one product C X
    rg = (n + 15) // 16
    print(json.dumps({"grid": grid, "n": n, "l": args.l, "generation": args.generation, **what, "row_groups": rg,
                      "launches_per_product": nl / args.reps, "ms_per_product": ms,
                      "tflops": one / (ms * 1e-3) * 1e-12 if ms > 0 else None, "card": card()}))


def cross_main(args, ctx, grid, ell, coords):
    m = coords.shape[1]
    if args.model:
        structures = model_structures(args.model.split(","), ell, args.angle, len(grid))
        what = {"model": args.model, "angle_deg": args.angle}
    else:
        structures = [gsi.CovStructure(args.kind, 1.0, ell)]
        what = {"kind": args.kind}
    rng = np.random.default_rng(1)
    n = args.cross
    if args.sources == "grid":
        idx = np.sort(rng.choice(m, n, replace=False))
        if args.generation == "table":
            op = gsi.GridKernelCrossCovMatrix(structures, grid, sources=idx, ctx=ctx)
        else:
            op = gsi.KernelCrossCovMatrix(structures, coords, coords[:, idx], ctx=ctx)
    else:
        if args.generation == "table":
            raise SystemExit("--sources random needs --generation arithmetic (the points are not grid nodes)")
        box = np.array(grid, dtype=np.float64)[:, None] - 1.0
        op = gsi.KernelCrossCovMatrix(structures, coords, rng.uniform(0, 1, (len(grid), n)) * box, ctx=ctx)
    base = {"grid": grid, "m": m, "n": n, "l": args.l, "generation": args.generation, "sources": args.sources, **what}
    runs = [("CX", op, n, False, m), ("CtX", op, m, True, n)]
    if args.square:
        if args.generation == "table":
            sq = gsi.GridKernelCovModelMatrix(structures, grid, ctx=ctx)
        else:
            sq = gsi.KernelCovModelMatrix(structures, coords, ctx=ctx)
        runs.append(("square", sq, m, False, m))
    for name, o, k, trans, rows in runs:
        X = gsi.DeviceMatrix.from_host(ctx, np.random.default_rng(0).standard_normal((k, args.l)))
        ms, nl, fl = time_products(ctx, [o], X, args.reps, trans=trans)
        X.free()
        one = 2.0 * rows * k * args.l
        print(json.dumps({**base, "product": name, "rows": rows, "k": k, "row_groups": (rows + 15) // 16,
                          "launches_per_product": nl / args.reps, "ms_per_product": ms,
                          "tflops": one / (ms * 1e-3) * 1e-12 if ms > 0 else None, "card": card()}), flush=True)


if __name__ == "__main__":
    main()
