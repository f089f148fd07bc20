#!/usr/bin/env python
"""Measures cross-validation on the dense factor (KernelCovCholesky.crossval / cross_validate, gsi_chol_crossval;
csrc/cov_chol.cu) on the B200: one JSON line per case.

    python tools/cov_cv_probe.py [--out profiles/r10/cov_cv_probe.jsonl] [--sizes 5000,20000,50000]

Points are scattered in the 64 x 56 x 56 box of profiles/r06, nugget 0.1, constant drift (p = 1).  Models:
"exponential" (ranges L / 6) and "sph_exp" (a rotated spherical plus an exponential structure), as in
tools/cov_lik_probe.py.  Lines ("what"):
  dgemm_peak   FP64 matrix-product rate of the card in this run (torch.matmul, 8192^3, float64)
  cv           per case: loo (leave-one-out), contig16 / contig128 (consecutive indices in groups of 16 / 128),
               scattered16 (random groups of 16), all on one factor, and cv_1pct (cross_validate with 1 % of the
               points held out in random groups of 16: operator, factor and crossval in one call).
               factor_ms: KernelCovCholesky alone; cv_ms: the call, host clock around calls that end in a
               synchronisation, median of --reps, every rep in cv_ms_reps (the host is shared: the spread shows when
               another process took it); operator_ms (cv_1pct): building the operator that cross_validate builds.
               From a separate run under torch.profiler, device time by launch order: drift_ms (the [F | y] sweep, the
               drift solve and the backward sweep for alpha), sweeps_ms (the chunks' forward sweeps from the scatter
               kernel on), proj_gram_ms (from the chunk's column norms to its Gram: the projection and W'W), group_ms
               (chol_cv_group_kernel), fill_factor_ms (cv_1pct: the fill and the factor).  sweep_tflops: the forward
               sweeps' flops (from the chunks, as the device packs them) over sweeps_ms, sweep_of_peak against
               dgemm_peak.
Every line carries the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gsi_b200 as gsi                                          # noqa: E402
from cov_chol_probe import card, dgemm_peak, points, L3, timed  # noqa: E402

CS = gsi.CovStructure


def models():
    return {"exponential": [CS("exponential", 1.0, L3 / 6)],
            "sph_exp": [CS("spherical", 0.6, L3 / 3, gsi.rotation_matrix((0.5, -0.3, 0.8))),
                        CS("exponential", 0.4, L3 / 8)]}


def make_op(name, P):
    if name == "exponential":
        return gsi.KernelCovMatrix("exponential", P, L3 / 6, nugget=0.1)
    return gsi.KernelCovModelMatrix(models()[name], P, 0.1)


def sweep_flops(groups, n):
    """flops of the chunks' forward sweeps: groups by smallest index, packed whole into <= 1024 columns; a chunk of
    wp columns from block row kb0 costs 128^2 wp N (N + 1), N = nb - kb0"""
    nb = -(-n // 128)
    sized = sorted(((int(np.min(g)), len(g)) for g in groups))
    total, w, kb0 = 0.0, 0, None

    def close(w, kb0):
        wp = -(-w // 128) * 128
        N = nb - kb0
        return 128.0 ** 2 * wp * N * (N + 1)
    for mn, s in sized:
        if kb0 is not None and w + s > 1024:
            total += close(w, kb0)
            w, kb0 = 0, None
        if kb0 is None:
            kb0 = mn // 128
        w += s
    return total + close(w, kb0)


def profiled(fn):
    """device ms per stage of one call, by launch order in a torch.profiler chrome trace (in a temporary directory)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        ev = json.load(open(path))["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    out = {"factor": 0.0, "drift": 0.0, "sweeps": 0.0, "proj_gram": 0.0, "group": 0.0}
    stage = "factor" if any("chol_logdet_kernel" in e["name"] for e in kern) else "drift"
    for e in kern:
        nm = e["name"]
        if "chol_cv_scatter_kernel" in nm:
            stage = "sweeps"
        elif "cov_solve_dot_kernel" in nm and stage == "sweeps":
            stage = "proj_gram"
        out["group" if "chol_cv_group_kernel" in nm else stage] += e["dur"] / 1e3
        if "chol_logdet_kernel" in nm:
            stage = "drift"                                 # cross_validate: the fill and the factor end here
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10", "cov_cv_probe.jsonl"))
    ap.add_argument("--sizes", default="5000,20000,50000")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    gsi.default_context()
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
        P = points(n)
        y = 1.0 + np.random.default_rng(1).standard_normal(n)
        reps = args.reps
        rng = np.random.default_rng(2)
        perm = rng.permutation(n)
        held = rng.permutation(n)[:n // 100]
        cases = {"loo": [np.array([i]) for i in range(n)],
                 "contig16": [np.arange(k, min(k + 16, n)) for k in range(0, n, 16)],
                 "contig128": [np.arange(k, min(k + 128, n)) for k in range(0, n, 128)],
                 "scattered16": [perm[k:k + 16] for k in range(0, n, 16)],
                 "cv_1pct": [held[k:k + 16] for k in range(0, held.size, 16)]}
        for name in models():
            op = make_op(name, P)
            fms, _ = timed(lambda: gsi.KernelCovCholesky(op).free(), reps)
            fac = gsi.KernelCovCholesky(op)
            for case, groups in cases.items():
                if case == "cv_1pct":
                    call = lambda: gsi.cross_validate(models()[name], P, y, nugget=0.1, drift="constant",  # noqa: E731
                                                      groups=groups)
                    # cross_validate puts the held-out points last: its sweeps start at column n - m
                    m = held.size
                    fl_groups = [np.arange(n - m + k, n - m + min(k + 16, m)) for k in range(0, m, 16)]
                else:
                    call = lambda: fac.crossval(y, drift="constant", groups=None if case == "loo" else groups)  # noqa
                    fl_groups = groups
                call()                                                               # warm-up
                ts = []
                for _ in range(reps):
                    t0 = time.perf_counter()
                    res = call()
                    ts.append((time.perf_counter() - t0) * 1e3)
                cms = float(np.median(ts))
                pk = profiled(call)
                fl = sweep_flops(fl_groups, n)
                line = {"what": "cv", "n": n, "model": name, "case": case, "p": 1,
                        "held_out": int(sum(len(g) for g in groups)), "ngroups": len(groups), "factor_ms": fms,
                        "cv_ms": cms, "cv_ms_reps": ts}
                if case == "cv_1pct":                                # cross_validate builds its own operator
                    line["operator_ms"], _ = timed(lambda: gsi.KernelCovModelMatrix(models()[name], P, 0.1).free(),
                                                   reps)
                emit(line | {"drift_ms": pk["drift"], "sweeps_ms": pk["sweeps"], "proj_gram_ms": pk["proj_gram"],
                             "group_ms": pk["group"],
                             "fill_factor_ms": pk["factor"], "group_share": pk["group"] / cms,
                             "sweep_tflops": fl / (pk["sweeps"] * 1e-3) / 1e12,
                             "sweep_of_peak": fl / (pk["sweeps"] * 1e-3) / 1e12 / peak, "cv_over_factor": cms / fms,
                             "sum_logpdf": float(np.sum(res.logpdf))})
            fac.free()
            op.free()
    f.close()


if __name__ == "__main__":
    main()
