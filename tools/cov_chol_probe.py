#!/usr/bin/env python
"""Measures the dense Cholesky path gsi_b200.KernelCovCholesky (csrc/cov_chol.cu) on the B200: one JSON line per case.

    python tools/cov_chol_probe.py [--out profiles/r07/cov_chol_probe.jsonl] [--sizes 5000,20000,50000]

Lines ("what"):
  dgemm_peak     FP64 matrix-product rate of the card in this run (torch.matmul, 8192^3, float64), the yardstick of the
                 trailing-update kernel
  factor         per n (scattered points in the 64 x 56 x 56 box of profiles/r06, exponential kernel, nugget 0.1):
                 factor_ms (wall time of the call, which ends in a synchronisation; median of --reps after a warm-up),
                 rate_tflops = (n^3 / 3) / factor_ms, and the phases from CUDA events in a separate timed run: fill_ms
                 (materialising A), diag_ms (diagonal blocks), panel_ms (panel solves), trailing_ms and trailing_tflops
                 (the flops the trailing-update kernel executes over its time), trailing_of_peak
  solve          per n and k in {1, 200}: solve_ms of A^-1 B (wall, median)
  variance       n = 20 000, m = 100 000 simple-kriging variances: variance_ms and targets per second
  direct_vs_cg   the 20 000-point case of profiles/r06 (rtol 1e-8): factor + solve against cov_solve at r = 0 and
                 r = 200, end to end, for 1 and 200 right-hand sides
Every line carries the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import ctypes as C
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


def dgemm_peak():
    import torch
    a = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    b = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
    for _ in range(2):
        torch.matmul(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    reps = 10
    for _ in range(reps):
        torch.matmul(a, b)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * 8192 ** 3 / (ms * 1e-3) / 1e12


def points(n, seed=0):
    return np.random.default_rng(seed).uniform(0.0, 1.0, (3, n)) * np.array([[64.0], [56.0], [56.0]])


L3 = np.array([64.0, 56.0, 56.0])


def phases(ctx):
    """the eight per-phase times of gsi_ctx_phase_timing (reset afterwards): [5] fill, [6] diagonal blocks, [7] panels"""
    out = (C.c_double * 8)()
    gsi._lib.check(ctx._lib.gsi_ctx_phase_timing(ctx._h, out, 1))
    return list(out)


def timed(fn, reps):
    out, ts = None, []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07", "cov_chol_probe.jsonl"))
    ap.add_argument("--sizes", default="5000,20000,50000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--variance-m", type=int, default=100000)
    ap.add_argument("--skip-cg", action="store_true")
    args = ap.parse_args()
    ctx = gsi.default_context()
    cardname = card()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    f = open(args.out, "a")

    def emit(line):
        line["card"] = cardname
        print(json.dumps(line), flush=True)
        f.write(json.dumps(line) + "\n")
        f.flush()

    peak = dgemm_peak()
    emit({"what": "dgemm_peak", "tflops": peak, "shape": [8192, 8192, 8192]})
    for n in [int(s) for s in args.sizes.split(",") if s]:
        op = gsi.KernelCovMatrix("exponential", points(n), L3 / 6, nugget=0.1)
        gsi.KernelCovCholesky(op).free()                                     # warm-up
        ms, _ = timed(lambda: gsi.KernelCovCholesky(op).free(), args.reps)
        ctx.gemm_timing(enable=True)
        phases(ctx)
        fac = gsi.KernelCovCholesky(op)
        ph = phases(ctx)
        tr_ms, _, tr_flops = ctx.gemm_timing(enable=False)
        fl = n ** 3 / 3.0
        emit({"what": "factor", "n": n, "factor_ms": ms, "rate_tflops": fl / (ms * 1e-3) / 1e12,
              "fill_ms": ph[5], "diag_ms": ph[6], "panel_ms": ph[7], "trailing_ms": tr_ms,
              "trailing_tflops": tr_flops / (tr_ms * 1e-3) / 1e12 if tr_ms else None,
              "trailing_of_peak": (tr_flops / (tr_ms * 1e-3) / 1e12) / peak if tr_ms else None,
              "phases_note": "phase times come from a separate run with an event pair around every launch"})
        rng = np.random.default_rng(1)
        for k in (1, 200):
            B = rng.standard_normal((n, k))
            fac.solve(B)
            sms, _ = timed(lambda: fac.solve(B), args.reps)
            emit({"what": "solve", "n": n, "k": k, "solve_ms": sms})
        if n == 20000 and args.variance_m > 0:
            T = points(args.variance_m, seed=5)
            st = [gsi.CovStructure("exponential", 1.0, L3 / 6)]
            cross = gsi.KernelCrossCovMatrix(st, T, points(n), ctx=ctx)
            fac.variance(cross)
            vms, var = timed(lambda: fac.variance(cross), 1)
            emit({"what": "variance", "n": n, "m": args.variance_m, "variance_ms": vms,
                  "targets_per_s": args.variance_m / (vms * 1e-3), "var_min": float(var.min()),
                  "var_max": float(var.max())})
            cross.free()
        if n == 20000 and not args.skip_cg:
            for k in (1, 200):
                B = rng.standard_normal((n, k))

                def direct():
                    g = gsi.KernelCovCholesky(op)
                    X = g.solve(B)
                    g.free()
                    return X
                dms, Xd = timed(direct, args.reps)
                for r in (0, 200):
                    Om = rng.standard_normal((n, r)) if r else None
                    try:                                                # warm-up of the shape (set-up only)
                        gsi.cov_solve(op, B, rtol=1e-8, maxiter=0, Omega=Om)
                    except gsi.GsiError as e:
                        if e.code != gsi._lib.ERR_NO_CONVERGENCE:
                            raise
                    t0 = time.perf_counter()
                    Xc, info = gsi.cov_solve(op, B, rtol=1e-8, maxiter=2000, Omega=Om)
                    cms = (time.perf_counter() - t0) * 1e3
                    emit({"what": "direct_vs_cg", "n": n, "k": k, "r": r, "direct_ms": dms, "cg_ms": cms,
                          "cg_iterations_max": int(np.max(info["iterations"])), "speedup": cms / dms,
                          "rel_diff": float(np.linalg.norm(Xd - Xc) / np.linalg.norm(Xd))})
        fac.free()
        op.free()
    f.close()


if __name__ == "__main__":
    main()
