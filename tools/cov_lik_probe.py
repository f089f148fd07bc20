#!/usr/bin/env python
"""Measures the Gaussian log-likelihood and its gradient on the dense factor (gsi_b200.loglik, gsi_kernelcov_loglik;
csrc/cov_chol.cu and kcov_grad_kernel in csrc/kcov_gemm.cu) on the B200: one JSON line per case.

    python tools/cov_lik_probe.py [--out profiles/r09/cov_lik_probe.jsonl] [--sizes 5000,20000,50000]

Points are scattered in the 64 x 56 x 56 box of profiles/r06; the drift is a constant (p = 1) and the likelihood REML.
Models: "exponential" (KernelCovMatrix, ranges L / 6, nugget 0.1) and "sph_exp" (KernelCovModelMatrix: a rotated
spherical plus an exponential structure, nugget 0.1).  Lines ("what"):
  dgemm_peak   FP64 matrix-product rate of the card in this run (torch.matmul, 8192^3, float64)
  lik          factor_ms (KernelCovCholesky alone), value_ms (loglik without gradient), grad_ms (loglik with gradient):
               host clock around calls that end in a synchronisation, median of --reps (1 at n = 50 000).
               value_sweeps_ms = value_ms - factor_ms.  From a separate run under torch.profiler (CUDA activity of one
               gradient call): contraction_ms (kcov_grad_kernel), rank_update_ms (chol_gemm_kernel<true, true, true>);
               inversion_ms = grad_ms - value_ms - contraction_ms - rank_update_ms (the chunked sweeps with their
               memsets, identity columns and partial-sum reductions).  inversion_tflops = (2 n^3 / 3) / inversion_ms,
               inversion_of_peak against dgemm_peak; contraction_gentries_per_s = n (n + 1) / 2 / contraction_ms.
  host_grad    n = 5 000 only: one host evaluation of value and gradient with NumPy / SciPy on this machine's CPU (dense A
               and dA / dtheta, Cholesky, A^-1, the contraction), host_ms.
Every line carries the card's name, power limit and maximum SM clock, read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gsi_b200 as gsi                                          # noqa: E402
from cov_chol_probe import card, dgemm_peak, points, L3, timed  # noqa: E402


def models():
    return {"exponential": None,
            "sph_exp": [gsi.CovStructure("spherical", 0.6, L3 / 3, gsi.rotation_matrix((0.5, -0.3, 0.8))),
                        gsi.CovStructure("exponential", 0.4, L3 / 8)]}


def make_op(name, P):
    if name == "exponential":
        return gsi.KernelCovMatrix("exponential", P, L3 / 6, nugget=0.1)
    return gsi.KernelCovModelMatrix(models()[name], P, 0.1)


def profiled(fn):
    """device time (ms) per kernel-name fragment of one call, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    out = {"kcov_grad_kernel": 0.0, "chol_gemm_kernel<true, true, true>": 0.0}
    for ev in prof.key_averages():
        for k in out:
            if k in ev.key:
                out[k] += ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
    return out


def host_grad(P, y):
    """value and gradient of the exponential case on the host (NumPy / SciPy)"""
    import scipy.linalg
    n = P.shape[1]
    u = P / (L3 / 6)[:, None]
    du2 = (u[:, :, None] - u[:, None, :]) ** 2
    r = np.sqrt(du2.sum(axis=0))
    K = np.exp(-r)
    A = K + 0.1 * np.eye(n)
    L = np.linalg.cholesky(A)
    F = np.ones((n, 1))
    g = scipy.linalg.solve_triangular(L, y, lower=True)
    G = scipy.linalg.solve_triangular(L, F, lower=True)
    gg = float(G[:, 0] @ G[:, 0])
    e = g - G[:, 0] * (float(G[:, 0] @ g) / gg)
    Ai = scipy.linalg.cho_solve((L, True), np.eye(n))
    alpha = scipy.linalg.solve_triangular(L.T, e, lower=False)
    H = scipy.linalg.solve_triangular(L.T, G / np.sqrt(gg), lower=False)
    W = np.outer(alpha, alpha) - Ai + H @ H.T
    kp = np.where(r > 0, -K / (2 * np.where(r > 0, r, 1.0)), 0.0)
    grad = [0.5 * np.sum(W * K)] + [np.sum(W * kp * (-2 * du2[a]) / (L3[a] / 6)) * 0.5 for a in range(3)]
    return grad + [0.5 * np.trace(W)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09", "cov_lik_probe.jsonl"))
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
        reps = 1 if n > 20000 else args.reps
        for name in models():
            op = make_op(name, P)
            value = lambda: gsi.loglik(op, y, drift="constant", reml=True)              # noqa: E731
            grad = lambda: gsi.loglik(op, y, drift="constant", reml=True, grad=True)    # noqa: E731
            grad()                                                                      # warm-up
            fms, _ = timed(lambda: gsi.KernelCovCholesky(op).free(), reps)
            vms, _ = timed(value, reps)
            gms, out = timed(grad, reps)
            pk = profiled(grad)
            con, rank = pk["kcov_grad_kernel"], pk["chol_gemm_kernel<true, true, true>"]
            inv = gms - vms - con - rank
            emit({"what": "lik", "n": n, "model": name, "p": 1, "reml": True, "factor_ms": fms, "value_ms": vms,
                  "grad_ms": gms, "value_sweeps_ms": vms - fms, "contraction_ms": con, "rank_update_ms": rank,
                  "inversion_ms": inv, "inversion_tflops": 2 * n ** 3 / 3 / (inv * 1e-3) / 1e12,
                  "inversion_of_peak": 2 * n ** 3 / 3 / (inv * 1e-3) / 1e12 / peak,
                  "contraction_gentries_per_s": n * (n + 1) / 2 / (con * 1e-3) / 1e9 if con else None,
                  "grad_over_factor": gms / fms, "loglik": out[0], "grad": [float(v) for v in out[2]]})
            op.free()
        if n == 5000:
            t0 = time.perf_counter()
            host_grad(P, y)
            emit({"what": "host_grad", "n": n, "model": "exponential", "host_ms": (time.perf_counter() - t0) * 1e3,
                  "cpu_threads": os.cpu_count()})
    f.close()


if __name__ == "__main__":
    main()
