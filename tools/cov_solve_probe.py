#!/usr/bin/env python
"""Measures the kriging solve gsi_b200.cov_solve (csrc/cov_solve.cu) on the B200: one JSON line per case.

    python tools/cov_solve_probe.py [--out profiles/r06/cov_solve_probe.jsonl] [--maxiter 600] [--rtol 1e-8]

Cases: the C3 grid (64 x 56 x 56 = 200 704 nodes) as observations with a Gaussian lattice-table operator and with a
rotated spherical + exponential model (signed table), and 20 000 scattered points with an exponential kernel (the
arithmetic path), each with a nugget; per case k = 1, 2, 8 at r = 0, 50, 200 (--runs selects a subset).

Per line:
  iterations        per column, to rtol (rtol 1e-8); "converged": false when --maxiter stopped a column first
  solve_ms          wall time of the whole call (it ends in a device synchronisation)
  setup_ms          wall time of the same call with maxiter = 0: upload, Nystrom build, the final residual product
  build_ms          setup_ms at this r minus setup_ms at r = 0 (the Nystrom preconditioner)
  iter_ms           (solve_ms - setup_ms) / iterations of the slowest column
  product_ms        operator-product time per iteration (CUDA events, Context.gemm_timing)
  product_share     product_ms / iter_ms
  host_gap_ms       device idle time per iteration: gaps between the library's kernels and copies in a
                    torch.profiler trace of a separate run of the same solve (at most 30 iterations; the idle time of
                    a maxiter = 0 run is subtracted and the rest divided by the iterations that run made)
  product_ms_k210   one 210-column product of the same operator, for the width-1 / width-210 ratio
Every line carries the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as gsi      # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make_cases():
    shape = (64, 56, 56)
    L = np.array(shape, dtype=np.float64)
    rot = gsi.rotation_matrix((0.5, 0.0, 0.0))
    model = [gsi.CovStructure("spherical", 0.6, L / 4, rot), gsi.CovStructure("exponential", 0.4, L / 6)]
    pts = np.random.default_rng(0).uniform(0.0, 1.0, (3, 20000)) * np.array([[64.0], [56.0], [56.0]])
    return [
        ("c3_gaussian_table", lambda: gsi.GridKernelCovMatrix("gaussian", shape, L / 8, nugget=0.1)),
        ("c3_model_signed_table", lambda: gsi.GridKernelCovModelMatrix(model, shape, nugget=0.1)),
        ("scattered_20k_exponential", lambda: gsi.KernelCovMatrix("exponential", pts, L / 6, nugget=0.1)),
    ]


def solve(op, B, rtol, maxiter, Omega):
    t0 = time.perf_counter()
    try:
        X, info = gsi.cov_solve(op, B, rtol=rtol, maxiter=maxiter, Omega=Omega)
        ok = True
    except gsi.GsiError as e:
        if e.code != gsi._lib.ERR_NO_CONVERGENCE:
            raise
        info, ok = e.info, False
    return (time.perf_counter() - t0) * 1e3, info, ok


def host_gap(ctx, op, B, rtol, Omega, iters=30):
    """(device idle ms per iteration, trace events per iteration) in a profiled run of at most `iters` iterations (the
    set-up is subtracted the same way)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    def idle(maxiter):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _, info, _ = solve(op, B, rtol, maxiter, Omega)
            torch.cuda.synchronize()
        ran = int(np.max(info["iterations"]))
        iv = sorted((e.time_range.start, e.time_range.end) for e in prof.events()
                    if e.device_type.name == "CUDA" and e.time_range.end > e.time_range.start)
        if not iv:
            return None, ran
        busy, cur0, cur1 = 0.0, iv[0][0], iv[0][1]
        for a, b in iv[1:]:
            if a > cur1:
                busy += cur1 - cur0
                cur0, cur1 = a, b
            else:
                cur1 = max(cur1, b)
        busy += cur1 - cur0
        return (((iv[-1][1] - iv[0][0]) - busy) * 1e-3, len(iv)), ran

    (a, _), (b, ran) = idle(0), idle(iters)
    if a is None or b is None or ran == 0:
        return None, None
    return (b[0] - a[0]) / ran, (b[1] - a[1]) / ran


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06", "cov_solve_probe.jsonl"))
    ap.add_argument("--maxiter", type=int, default=600)
    ap.add_argument("--rtol", type=float, default=1e-8)
    ap.add_argument("--cases", default="")
    ap.add_argument("--runs", default="1:0,1:50,1:200,2:0,2:50,2:200,8:0,8:50,8:200", help="k:r pairs")
    args = ap.parse_args()
    ctx = gsi.default_context()
    cardname = card()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    runs = [tuple(int(v) for v in kr.split(":")) for kr in args.runs.split(",")]
    with open(args.out, "a") as f:
        for name, build in make_cases():
            if args.cases and name not in args.cases.split(","):
                continue
            op = build()
            n = op.shape[0]
            rng = np.random.default_rng(1)
            Bfull = rng.standard_normal((n, 8))
            X210 = gsi.DeviceMatrix.from_host(ctx, rng.standard_normal((n, 210)))
            op.apply(X210).free()
            ctx.sync()
            ctx.gemm_timing(enable=True)
            op.apply(X210).free()
            ctx.sync()
            p210 = ctx.gemm_timing(enable=False)[0]
            X210.free()
            setup0 = {}
            for k, r in runs:
                B = Bfull[:, :k]
                Omega = rng.standard_normal((n, r)) if r else None
                solve(op, B, args.rtol, 0, Omega)                          # warm-up of every shape
                ts, _, _ = solve(op, B, args.rtol, 0, Omega)
                if r == 0:
                    setup0[k] = ts
                ctx.gemm_timing(enable=True)
                _, _, _ = solve(op, B, args.rtol, 0, Omega)
                g0 = ctx.gemm_timing(enable=True)[0]
                tf, info, ok = solve(op, B, args.rtol, args.maxiter, Omega)
                g1 = ctx.gemm_timing(enable=False)[0]
                its = int(np.max(info["iterations"]))
                iter_ms = (tf - ts) / its if its else None
                prod_ms = (g1 - g0) / its if its else None
                gap, ev_per_iter = host_gap(ctx, op, B, args.rtol, Omega)
                line = {"case": name, "n": n, "k": k, "r": r, "rtol": args.rtol, "nugget": 0.1, "converged": ok,
                        "iterations": [int(x) for x in info["iterations"]], "relres_max": float(np.max(info["relres"])),
                        "solve_ms": tf, "setup_ms": ts, "build_ms": (ts - setup0[k]) if (r and k in setup0) else None,
                        "iter_ms": iter_ms, "product_ms": prod_ms,
                        "product_share": (prod_ms / iter_ms) if iter_ms else None,
                        "host_gap_ms": gap, "trace_events_per_iter": ev_per_iter, "maxiter": args.maxiter,
                        "product_ms_k210": p210, "card": cardname}
                print(json.dumps(line), flush=True)
                f.write(json.dumps(line) + "\n")
                f.flush()
            op.free()


if __name__ == "__main__":
    main()
