#!/usr/bin/env python
"""Measures conditional simulation on the dense factor (KernelCovCholesky.simulate, gsi_chol_simulate; csrc/cov_chol.cu)
on the B200: one JSON line per case.

    python tools/cov_sim_probe.py [--out profiles/r08/cov_sim_probe.jsonl] [--sizes 5000,20000,50000]

Each N has ns = N / 4 scattered sources and m = 3 N / 4 scattered targets (the 64 x 56 x 56 box of profiles/r06,
exponential kernel, nugget 0.1 at the sources, none at the targets).  Lines ("what"):
  dgemm_peak   FP64 matrix-product rate of the card in this run (torch.matmul, 8192^3, float64), the TRMM's yardstick
  factor       factor_ms: wall time of the joint factorisation (gsi_kernelcov_chol_diag, median of --reps)
  simulate     per p in {0, 1} (simple, ordinary kriging) and k in {1, 128, 1024}: upload_ms (Xi to the device),
               simulate_ms (the gsi_chol_simulate call, which ends in a synchronisation; median of --reps), trmm_ms (the
               triangular product chol_trmm_kernel by CUDA events, in a separate run), rest_ms = simulate_ms - trmm_ms,
               trmm_tflops = executed flops 2 * 128^3 * (k / 128 rounded up) * sum over row tiles i of (i + 1) over
               trmm_ms, trmm_of_peak against dgemm_peak, download_ms (Z to the host) and realisations_per_s = k over
               upload + simulate + download
Every line carries the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gsi_b200 as gsi                                          # noqa: E402
from cov_chol_probe import card, dgemm_peak, points, L3         # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08", "cov_sim_probe.jsonl"))
    ap.add_argument("--sizes", default="5000,20000,50000")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    ctx = gsi.default_context()
    lib = ctx._lib
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
    rng = np.random.default_rng(2)
    for N in [int(s) for s in args.sizes.split(",") if s]:
        ns, m = N // 4, N - N // 4
        P = points(N)
        st = [gsi.CovStructure("exponential", 1.0, L3 / 6)]
        op = gsi.KernelCovModelMatrix(st, P, 0.0)
        d = np.r_[np.full(ns, 0.1), np.zeros(m)]
        gsi.KernelCovCholesky(op, diag=d).free()                                 # warm-up
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fac = gsi.KernelCovCholesky(op, diag=d)
            ts.append((time.perf_counter() - t0) * 1e3)
            if len(ts) < args.reps:
                fac.free()
        emit({"what": "factor", "N": N, "ns": ns, "m": m, "factor_ms": float(np.median(ts))})
        y = np.sin(P[0, :ns] / 7) + 0.1 * rng.standard_normal(ns)
        np_, nb, i0 = -(-N // 128) * 128, -(-N // 128), ns // 128
        for p in (0, 1):
            Fs, Ft = np.ones((ns, p), order="F"), np.ones((m, p), order="F")
            for k in (1, 128, 1024):
                Xi = rng.standard_normal((N, k))
                Zd = gsi.DeviceMatrix(ctx, m, k, gsi.LAYOUT_TALL)

                def call(Xd):
                    gsi._lib.check(lib.gsi_chol_simulate(fac._h, ns, gsi.core._pd(y), gsi.core._pd(Fs) if p else None,
                                                         gsi.core._pd(Ft) if p else None, p, Xd._h, Zd._h))
                Xd = gsi.DeviceMatrix.from_host(ctx, Xi)
                call(Xd)                                                         # warm-up
                up, sim, down = [], [], []
                for _ in range(args.reps):
                    Xd.free()
                    t0 = time.perf_counter()
                    Xd = gsi.DeviceMatrix.from_host(ctx, Xi)
                    ctx.sync()
                    t1 = time.perf_counter()
                    call(Xd)
                    t2 = time.perf_counter()
                    Zd.numpy()
                    t3 = time.perf_counter()
                    up.append((t1 - t0) * 1e3)
                    sim.append((t2 - t1) * 1e3)
                    down.append((t3 - t2) * 1e3)
                ctx.gemm_timing(enable=True)
                call(Xd)
                tr_ms, _, tr_flops = ctx.gemm_timing(enable=False)
                Xd.free()
                Zd.free()
                flops = 2.0 * 128 ** 3 * (-(-k // 128)) * ((nb * (nb + 1) - i0 * (i0 + 1)) // 2)
                assert flops == tr_flops, (flops, tr_flops)
                u, s, dn = float(np.median(up)), float(np.median(sim)), float(np.median(down))
                emit({"what": "simulate", "N": N, "ns": ns, "m": m, "p": p, "k": k, "np": np_, "upload_ms": u,
                      "simulate_ms": s, "trmm_ms": tr_ms, "rest_ms": s - tr_ms, "download_ms": dn,
                      "trmm_tflops": flops / (tr_ms * 1e-3) / 1e12,
                      "trmm_of_peak": flops / (tr_ms * 1e-3) / 1e12 / peak,
                      "realisations_per_s": k / ((u + s + dn) * 1e-3),
                      "timing_note": "trmm_ms from CUDA events in a separate call; the others are wall times"})
        fac.free()
        op.free()
    f.close()


if __name__ == "__main__":
    main()
