"""Leave-one-out and leave-group-out cross-validation of kriging on the dense factor (gsi_chol_crossval,
KernelCovCholesky.crossval, cross_validate).

With A = L L', P = A^-1 - A^-1 F (F'A^-1 F)^-1 F'A^-1 and alpha = P y, for a held-out set B (Dubrule 1983):
    err_B = y_B - yhat_B = P_BB^-1 alpha_B,  var_B = diag(P_BB^-1),  logpdf_B = -1/2 (alpha_B' err_B + |B| log 2 pi - log det P_BB)
the prediction yhat_B being universal kriging (drift re-estimated by GLS) from the other points, var_B its error variance
for the observation (nugget included).

* Without a GPU: the NumPy restatement of the device algorithm (P_BB as the Gram of the projected columns
  (I - G^ G^') L^-1 E_B, G^ = L^-1 F R^-1) against brute-force refits without each group, for n in {60, 300},
  p in {0, 1, 3}, leave-one-out, mixed group sizes 1..128, scattered groups, a subset of the points and per-point noise.
* On the GPU: err, var and logpdf against the restatement on the operator's own matrix (gsi_op_kernelcov_block) within
  TOL relative (lines starting with CVREPORT carry the worst measured ratios); against krige(method="cholesky",
  return_variance=True) refitted without a group; bit equalities (reruns, NULL groups against n singletons, a group
  alone against the same group among shuffled others, cross_validate against crossval within TOL); n = 65 600 (past
  2^32 factor entries) against the closed form of a pair-block-diagonal A; every refusal.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.linalg
import scipy.stats

from gpu_util import gsi  # noqa: F401
from test_gpu_kcov_lik import CASE_IDS, CASES, drift, host_A, observations, points, total_sill

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G                                   # noqa: E402

CS = G.CovStructure
LOG2PI = np.log(2 * np.pi)
TOL = 1e-11


# ------------------------------------------------------------------ host
def host_cv(A, y, F, groups):
    """The device algorithm restated: err, var (lists per group) and logpdf per group."""
    L = np.linalg.cholesky(A)
    n, p = F.shape
    g = scipy.linalg.solve_triangular(L, y, lower=True)
    if p:
        Gm = scipy.linalg.solve_triangular(L, F, lower=True)
        R = np.linalg.cholesky(Gm.T @ Gm).T
        beta = scipy.linalg.cho_solve((R, False), Gm.T @ g)
        Gh = scipy.linalg.solve_triangular(R.T, Gm.T, lower=True).T
        e = g - Gm @ beta
    else:
        Gh, e = np.zeros((n, 0)), g
    alpha = scipy.linalg.solve_triangular(L.T, e, lower=False)
    errs, vars_, lps = [], [], []
    for B in groups:
        B = np.asarray(B)
        E = np.zeros((n, B.size))
        E[B, np.arange(B.size)] = 1.0
        W = scipy.linalg.solve_triangular(L, E, lower=True)
        W = W - Gh @ (Gh.T @ W)
        P = W.T @ W
        Lb = np.linalg.cholesky(P)
        X = scipy.linalg.solve_triangular(Lb, np.eye(B.size), lower=True)
        z = X @ alpha[B]
        errs.append(X.T @ z)
        vars_.append((X * X).sum(axis=0))
        lps.append(-0.5 * (z @ z + B.size * LOG2PI - 2 * np.log(np.diag(Lb)).sum()))
    return errs, vars_, np.array(lps)


def refit(A, y, F, B):
    """Brute force: GLS universal kriging of y_B from the other points; (prediction, error covariance, log-density)."""
    n = A.shape[0]
    B = np.asarray(B)
    Rm = np.setdiff1d(np.arange(n), B)
    Arr, Abr = A[np.ix_(Rm, Rm)], A[np.ix_(B, Rm)]
    K = Abr @ np.linalg.inv(Arr)
    C = A[np.ix_(B, B)] - K @ Abr.T
    if F.shape[1]:
        Fr, Fb = F[Rm], F[B]
        Ai_F = np.linalg.solve(Arr, Fr)
        beta = np.linalg.solve(Fr.T @ Ai_F, Ai_F.T @ y[Rm])
        yhat = Fb @ beta + K @ (y[Rm] - Fr @ beta)
        D = Fb - K @ Fr
        C = C + D @ np.linalg.solve(Fr.T @ Ai_F, D.T)
    else:
        yhat = K @ y[Rm]
    C = 0.5 * (C + C.T)
    return yhat, C, scipy.stats.multivariate_normal(mean=yhat, cov=C).logpdf(y[B])


def mixed_groups(n, seed, frac=0.8):
    """Groups of 1..128 points over about frac of the points: one across the 128-row tile boundary, one across index
    1024 (n > 1050), one of exactly 128 scattered points (n >= 200), then scattered groups of cycling sizes; the rest
    of the points stay in."""
    rng = np.random.default_rng(seed)
    out = [np.arange(124, 132)] if n > 132 else []
    if n > 1050:
        out.append(np.arange(1000, 1050))
    used = set(np.concatenate(out).tolist()) if out else set()
    rest = rng.permutation([i for i in range(n) if i not in used])
    k, sizes, s = 0, [1, 7, 32, 33, 2, 90, 1, 17, 64, 1, 5], 0
    if n >= 200:
        out.append(np.sort(rest[:128]))
        k = 128
    while k < rest.size and len(used) + k < frac * n:
        sz = sizes[s % len(sizes)]
        out.append(np.sort(rest[k:k + sz]) if s % 2 else rest[k:k + sz])
        k += sz
        s += 1
    return [np.asarray(g) for g in out if len(g)]


def host_model(n, p, seed, noise=None):
    X = points(n, 2, seed)
    sts = CASES[CASE_IDS.index("sph_exp_d2")][1]
    A, _ = host_A(sts, X, 0.1)
    if noise is not None:
        A = A + np.diag(noise)
    return A, observations(A, X, seed + 1), drift(X, p)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("p", [0, 1, 3])
@pytest.mark.parametrize("n", [60, 300])
def test_host_restatement_against_refits(n, p, noise):
    d = np.random.default_rng(3).uniform(0.0, 0.5, n) if noise else None
    A, y, F = host_model(n, p, 7, d)
    loo = [np.array([i]) for i in range(0, n, 1 if n == 60 else 23)]
    for groups in (loo, mixed_groups(n, 4, frac=0.6)):
        errs, vars_, lps = host_cv(A, y, F, groups)
        for B, e, v, lp in zip(groups, errs, vars_, lps):
            yhat, Cb, lpr = refit(A, y, F, B)
            scale = np.sqrt(np.diag(Cb))
            assert np.all(np.abs(e - (y[B] - yhat)) <= 1e-9 * (np.abs(e) + scale)), B
            assert np.allclose(v, np.diag(Cb), rtol=1e-9), B
            assert abs(lp - lpr) <= 1e-9 * (abs(lpr) + B.size), B


def test_host_loo_scalar_form():
    """Leave-one-out: e_i = alpha_i / P_ii, var_i = 1 / P_ii with P formed explicitly."""
    A, y, F = host_model(60, 1, 9)
    Ai = np.linalg.inv(A)
    P = Ai - Ai @ F @ np.linalg.solve(F.T @ Ai @ F, F.T @ Ai)
    alpha = P @ y
    errs, vars_, _ = host_cv(A, y, F, [np.array([i]) for i in range(60)])
    assert np.allclose(np.concatenate(errs), alpha / np.diag(P), rtol=1e-9, atol=1e-12)
    assert np.allclose(np.concatenate(vars_), 1 / np.diag(P), rtol=1e-9)


def test_exports():
    assert G.cross_validate is G.kriging.cross_validate
    assert G.CrossValidation._fields == ("prediction", "error", "variance", "logpdf")
    assert "gsi_chol_crossval" in G._lib.SIGNATURES


# ------------------------------------------------------------------ GPU helpers
def op_matrix(gsi, op, n):
    from test_gpu_kcov_chol import block
    return block(gsi, op, 0, 0, n, n)


WORST = {"err": 0.0, "var": 0.0, "logpdf": 0.0}


def report():
    print(f"CVREPORT worst ratios (of {TOL:g} relative): err {WORST['err']:.3e} var {WORST['var']:.3e} "
          f"logpdf {WORST['logpdf']:.3e}")


def compare(res, A, y, F, groups):
    """The device result against host_cv on the device's own A, within TOL: err against |err| + sqrt(var), var and
    logpdf relative (logpdf against |logpdf| + |B|)."""
    errs, vars_, lps = host_cv(A, y, F, groups)
    for k, B in enumerate(groups):
        re = np.abs(res.error[B] - errs[k]) / (TOL * (np.abs(errs[k]) + np.sqrt(vars_[k])))
        rv = np.abs(res.variance[B] - vars_[k]) / (TOL * vars_[k])
        rl = abs(res.logpdf[k] - lps[k]) / (TOL * (abs(lps[k]) + B.size))
        WORST["err"] = max(WORST["err"], float(re.max()))
        WORST["var"] = max(WORST["var"], float(rv.max()))
        WORST["logpdf"] = max(WORST["logpdf"], float(rl))
        assert re.max() <= 1 and rv.max() <= 1 and rl <= 1, (k, B, re.max(), rv.max(), rl)
        assert np.array_equal(res.prediction[B], y[B] - res.error[B])
    held = np.zeros(len(y), bool)
    held[np.concatenate(groups)] = True
    assert np.all(np.isnan(res.error[~held])) and np.all(np.isnan(res.variance[~held]))


def device_cv(gsi, op, y, F, groups, diag=None):
    n = op.shape[1]
    A = op_matrix(gsi, op, n)
    if diag is not None:
        A = A + np.diag(diag)
    fac = G.KernelCovCholesky(op, diag=diag)
    try:
        res = fac.crossval(y, drift=F if F.shape[1] else None, groups=groups)
    finally:
        fac.free()
    return res, A


# ------------------------------------------------------------------ GPU
GPU_CASES = [(c, p) for c in CASE_IDS for p in (0, 1, 3)
             if p == 1 or c in ("exponential_d2", "spherical_d1", "matern52_d3", "sph_exp_d2", "three_d3")]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [257, 2000])
@pytest.mark.parametrize("case,p", GPU_CASES)
def test_device_vs_host(gsi, case, p, n):
    if n == 2000 and case not in ("exponential_d2", "three_d3", "sph_exp_d2"):
        pytest.skip("n = 2000 runs the exponential and the two rotated models")
    _, sts, d = CASES[CASE_IDS.index(case)]
    X = points(n, d, 21)
    nug = 0.05 * total_sill(sts)
    A, _ = host_A(sts, X, nug)
    y = observations(A, X, 22)
    F = drift(X, p)
    op = (G.KernelCovMatrix(sts[0].kind, X, sts[0].ranges, sigma2=sts[0].sill, nugget=nug, beta=sts[0].beta)
          if len(sts) == 1 else G.KernelCovModelMatrix(sts, X, nug))
    try:
        groups = mixed_groups(n, 23)
        res, Ad = device_cv(gsi, op, y, F, groups)
        compare(res, Ad, y, F, groups)
        if n == 257:                                          # leave-one-out
            res, Ad = device_cv(gsi, op, y, F, None)
            compare(res, Ad, y, F, [np.array([i]) for i in range(n)])
    finally:
        op.free()
    report()


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0, 1])
def test_grid_operator_and_diag(gsi, p):
    """A grid operator (lattice table) and a factor with a per-point diagonal (heteroscedastic noise)."""
    shape, spacing = (23, 17), 0.5
    sts = [CS("exponential", 1.0, [3.0, 2.0], G.rotation_matrix(0.4)), CS("gaussian", 0.5, [2.0, 2.0])]
    n = shape[0] * shape[1]
    ix, iy = np.meshgrid(np.arange(shape[0]), np.arange(shape[1]), indexing="ij")
    X = np.vstack([ix.ravel(order="F"), iy.ravel(order="F")]) * spacing
    y = np.sin(X[0]) + np.cos(X[1] / 2)
    F = drift(X, p)
    gop = G.GridKernelCovModelMatrix(sts, shape, spacing=spacing, nugget=0.1)
    try:
        groups = mixed_groups(n, 31)
        res, Ad = device_cv(gsi, gop, y, F, groups)
        compare(res, Ad, y, F, groups)
    finally:
        gop.free()
    dg = np.random.default_rng(32).uniform(0.01, 0.4, n)
    op = G.KernelCovModelMatrix(sts, X, 0.0)
    try:
        res, Ad = device_cv(gsi, op, y, F, None, diag=dg)
        compare(res, Ad, y, F, [np.array([i]) for i in range(n)])
    finally:
        op.free()
    report()


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0, 1, 3])
def test_against_krige_refits(gsi, p):
    """The prediction is that of krige(method="cholesky") without the group; the variance is its kriging variance plus
    the nugget."""
    n = 600
    sts = CASES[CASE_IDS.index("sph_exp_d2")][1]
    X = points(n, 2, 41)
    nug = 0.08
    A, _ = host_A(sts, X, nug)
    y = observations(A, X, 42)
    F = drift(X, p)
    groups = [np.array([5]), np.arange(100, 140), np.array([599, 3, 211]), np.arange(256, 384)]
    res = G.cross_validate(sts, X, y, nugget=nug, drift=F if p else None, groups=groups)
    for k, B in enumerate(groups):
        Rm = np.setdiff1d(np.arange(n), B)
        dr = (F[Rm], F[B]) if p else None
        yhat, var = G.krige(sts, X[:, Rm], y[Rm], X[:, B], nugget=nug, drift=dr, method="cholesky", return_variance=True)
        assert np.all(np.abs(res.prediction[B] - yhat) <= 1e-9 * (np.abs(yhat) + np.sqrt(var + nug))), k
        assert np.allclose(res.variance[B], var + nug, rtol=1e-9), k


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0, 3])
def test_bit_equalities(gsi, p):
    n = 1500
    sts = CASES[CASE_IDS.index("three_d3")][1]
    X = points(n, 3, 51)
    A, _ = host_A(sts, X, 0.2)
    y = observations(A, X, 52)
    F = drift(X, p)
    dr = F if p else None
    op = G.KernelCovModelMatrix(sts, X, 0.2)
    fac = G.KernelCovCholesky(op)
    try:
        groups = mixed_groups(n, 53)
        a = fac.crossval(y, drift=dr, groups=groups)
        b = fac.crossval(y, drift=dr, groups=groups)
        for u, v in zip(a, b):
            assert np.array_equal(u, v, equal_nan=True)
        loo = fac.crossval(y, drift=dr)
        single = fac.crossval(y, drift=dr, groups=[[i] for i in range(n)])
        for u, v in zip(loo, single):
            assert np.array_equal(u, v, equal_nan=True)
        # a group alone, and among the others in shuffled order (its chunk and its columns move)
        order = np.random.default_rng(54).permutation(len(groups))
        shuffled = fac.crossval(y, drift=dr, groups=[groups[k] for k in order])
        for k in (0, 1, 2, len(groups) // 2, len(groups) - 1):
            B = groups[k]
            alone = fac.crossval(y, drift=dr, groups=[B])
            assert np.array_equal(alone.error[B], a.error[B]) and np.array_equal(alone.variance[B], a.variance[B])
            assert np.array_equal(alone.error[B], shuffled.error[B])
            assert np.array_equal(alone.variance[B], shuffled.variance[B])
            assert alone.logpdf[0] == a.logpdf[k] == shuffled.logpdf[int(np.where(order == k)[0][0])]
        # leave-one-out of a singleton alone gives the bits of the full leave-one-out run
        for i in (0, 700, n - 1):
            one = fac.crossval(y, drift=dr, groups=[[i]])
            assert one.error[i] == loo.error[i] and one.variance[i] == loo.variance[i]
    finally:
        fac.free()
        op.free()
    # cross_validate (points reordered, another factor) against crossval within TOL
    cv = G.cross_validate(sts, X, y, nugget=0.2, drift=dr, groups=groups)
    held = np.concatenate(groups)
    assert np.all(np.abs(cv.error[held] - a.error[held]) <= TOL * (np.abs(a.error[held]) + np.sqrt(a.variance[held])))
    assert np.allclose(cv.variance[held], a.variance[held], rtol=TOL)
    assert np.allclose(cv.logpdf, a.logpdf, rtol=TOL)
    assert np.all(np.isnan(cv.error[np.setdiff1d(np.arange(n), held)]))


@pytest.mark.gpu
def test_rows_above_a_chunk_are_not_read(gsi):
    """p = 0: a chunk's sweep starts at its first block row, and the rows above it are exact zeros of its columns.  The
    pivot scale of a group, the norm of its swept columns, must not pick up whatever the work block held there before:
    a freshly allocated block (filled with NaN here through torch and released just before the call), or the previous
    chunk's columns (1 024 singletons first).  Every call succeeds and gives the bits of the same points in
    leave-one-out."""
    import torch
    n = 2000
    sts = CASES[CASE_IDS.index("exponential_d2")][1]
    X = points(n, 2, 81)
    A, _ = host_A(sts, X, 0.05)
    y = observations(A, X, 82)
    op = G.KernelCovMatrix(sts[0].kind, X, sts[0].ranges, sigma2=sts[0].sill, nugget=0.05)
    fac = G.KernelCovCholesky(op)
    try:
        loo = fac.crossval(y)
        for groups in ([[1900]], [[1900], [1950, 1960, 1999]], [[i] for i in range(1024)] + [[1900], [1950, 1960]]):
            junk = torch.full((1 << 28,), float("nan"), dtype=torch.float64, device="cuda")   # 2 GiB of NaN
            torch.cuda.synchronize()
            del junk
            torch.cuda.empty_cache()
            res = fac.crossval(y, groups=groups)
            held = np.concatenate([np.asarray(g) for g in groups])
            singles = [g[0] for g in groups if len(g) == 1]
            assert np.array_equal(res.error[singles], loo.error[singles])
            assert np.array_equal(res.variance[singles], loo.variance[singles])
            assert np.all(np.isfinite(res.error[held])) and np.all(np.isfinite(res.logpdf))
    finally:
        fac.free()
        op.free()
    # the same through cross_validate (held-out points last: its only chunk starts far below row 0), twice
    groups = [np.array([5, 17]), np.array([400])]
    first = G.cross_validate(sts, X, y, nugget=0.05, groups=groups)
    torch.full((1 << 28,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    second = G.cross_validate(sts, X, y, nugget=0.05, groups=groups)
    for u, v in zip(first, second):
        assert np.array_equal(u, v, equal_nan=True)


@pytest.mark.gpu
def test_past_2_32_factor_entries(gsi):
    """n = 65 600 (the factor has 4.31e9 > 2^32 entries) on the pair construction of test_gpu_kcov_lik_exact: A is
    block-diagonal with 2 x 2 blocks [a c; c a], read from the device.  p = 0: e_i = y_i - (c / a) y_j and
    var_i = a - c^2 / a; p = 1 (constant): P = A^-1 - u u' / s with u = A^-1 1 (u_i = 1 / (a + c)), s = 1'u."""
    import torch
    from test_gpu_kcov_lik_exact import device_pairs, pair_case
    free = torch.cuda.mem_get_info()[0]
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory for a 34.5 GB factor, {free / 1e9:.1f} GB free")
    sts = [CS("exponential", 0.6, [1.5, 1.0]), CS("spherical", 0.4, [2.0, 1.2], G.rotation_matrix(0.5))]
    P = 32800
    n = 2 * P
    X = pair_case(sts, 2, P, 65600)
    y = np.random.default_rng(61).standard_normal(n) + 1.0
    op = G.KernelCovModelMatrix(sts, X, 2.0)
    try:
        a, c = device_pairs(gsi, op, n)
        fac = G.KernelCovCholesky(op)
        try:
            ya, yb = y[0::2], y[1::2]
            # pairs at the start, around column 2^32 / n_p = 65 408 (pair 32 704) and at the end
            sel = np.r_[0:40, 32680:32730, P - 40:P]
            pairs = [np.array([2 * q, 2 * q + 1]) for q in sel]
            det = a * a - c * c
            u = 1.0 / (a + c)
            s = 2.0 * u.sum()
            for p in (0, 1):
                loo = fac.crossval(y, drift="constant" if p else None)
                lpo = fac.crossval(y, drift="constant" if p else None, groups=pairs)
                if p == 0:
                    e = np.empty(n)
                    e[0::2], e[1::2] = ya - (c / a) * yb, yb - (c / a) * ya
                    v = np.repeat(a - c * c / a, 2)
                    assert np.allclose(loo.error, e, rtol=1e-12, atol=1e-12 * np.abs(y).max())
                    assert np.allclose(loo.variance, v, rtol=1e-12)
                    ep = np.empty(n)
                    ep[0::2], ep[1::2] = ya, yb                      # a whole pair out: the prediction is 0
                else:
                    Ay = np.empty(n)
                    Ay[0::2], Ay[1::2] = (a * ya - c * yb) / det, (a * yb - c * ya) / det
                    uy = (u * (ya + yb)).sum()
                    alpha = Ay - np.repeat(u, 2) * uy / s
                    Pii = np.repeat(a / det - u * u / s, 2)
                    assert np.allclose(loo.error, alpha / Pii, rtol=1e-9, atol=1e-9 * np.abs(y).max())
                    assert np.allclose(loo.variance, 1 / Pii, rtol=1e-9)
                for k, B in enumerate(pairs):
                    q = B[0] // 2
                    if p == 0:
                        eB, CB = y[B], np.array([[a[q], c[q]], [c[q], a[q]]])
                    else:
                        PB = np.array([[a[q], -c[q]], [-c[q], a[q]]]) / det[q] - u[q] * u[q] / s
                        CB = np.linalg.inv(PB)
                        eB = CB @ alpha[B]
                    assert np.allclose(lpo.error[B], eB, rtol=1e-9, atol=1e-9 * np.abs(y).max()), (p, q)
                    assert np.allclose(lpo.variance[B], np.diag(CB), rtol=1e-9), (p, q)
                    lp = scipy.stats.multivariate_normal(mean=y[B] - eB, cov=CB).logpdf(y[B])
                    assert abs(lpo.logpdf[k] - lp) <= 1e-9 * (abs(lp) + 2), (p, q)
        finally:
            fac.free()
    finally:
        op.free()


def raw_call(fac, y, F, p, ngroups, ptr, idx):
    pi64 = C.POINTER(C.c_int64)
    m = len(y) if ptr is None else max(int(ptr[-1]), 1)
    err, var, lpd = np.empty(max(m, len(y))), np.empty(max(m, len(y))), np.empty(max(ngroups, 1))
    failed = C.c_int64(-1)
    st = fac._lib.gsi_chol_crossval(fac._h, y.ctypes.data_as(C.POINTER(C.c_double)),
                                    None if F is None else F.ctypes.data_as(C.POINTER(C.c_double)), p, ngroups,
                                    None if ptr is None else np.ascontiguousarray(ptr, np.int64).ctypes.data_as(pi64),
                                    None if idx is None else np.ascontiguousarray(idx, np.int64).ctypes.data_as(pi64),
                                    err.ctypes.data_as(C.POINTER(C.c_double)), var.ctypes.data_as(C.POINTER(C.c_double)),
                                    lpd.ctypes.data_as(C.POINTER(C.c_double)), C.byref(failed))
    return st, failed.value


@pytest.mark.gpu
def test_refusals(gsi):
    n = 300
    X = points(n, 2, 71)
    y = np.random.default_rng(72).standard_normal(n)
    op = G.KernelCovMatrix("exponential", X, [2.0, 2.0], nugget=0.1)
    fac = G.KernelCovCholesky(op)
    ctx = op.ctx
    try:
        F1 = np.ones(n)
        ybad = y.copy()
        ybad[4] = np.nan
        Fbad = np.ones(n)
        Fbad[9] = np.inf
        ok_ptr, ok_idx = np.array([0, 2, 5]), np.array([1, 2, 10, 11, 12])
        cases = [
            ("non-monotone ptr", y, None, 0, 2, np.array([0, 3, 2]), ok_idx),
            ("ptr[0] != 0", y, None, 0, 2, np.array([1, 3, 5]), ok_idx),
            ("empty group", y, None, 0, 2, np.array([0, 0, 5]), ok_idx),
            ("129 points", y, None, 0, 1, np.array([0, 129]), np.arange(129)),
            ("index out of range", y, None, 0, 2, ok_ptr, np.array([1, 2, 10, 11, n])),
            ("negative index", y, None, 0, 2, ok_ptr, np.array([1, -2, 10, 11, 12])),
            ("duplicate in a group", y, None, 0, 2, ok_ptr, np.array([1, 1, 10, 11, 12])),
            ("duplicate across groups", y, None, 0, 2, ok_ptr, np.array([1, 2, 10, 11, 2])),
            ("no groups", y, None, 0, 0, np.array([0]), np.zeros(1, np.int64)),
            ("loo with ngroups != n", y, None, 0, n - 1, None, None),
            ("p = 33", y, np.ones((n, 33)) + np.arange(33), 33, 2, ok_ptr, ok_idx),
            ("F with p = 0", y, F1, 0, 2, ok_ptr, ok_idx),
            ("no F with p = 1", y, None, 1, 2, ok_ptr, ok_idx),
            ("non-finite y", ybad, None, 0, 2, ok_ptr, ok_idx),
            ("non-finite F", y, Fbad, 1, 2, ok_ptr, ok_idx),
        ]
        for name, yy, F, p, ng, ptr, idx in cases:
            before = ctx.launch_count()
            st, _ = raw_call(fac, np.ascontiguousarray(yy), None if F is None else np.asfortranarray(F), p, ng, ptr, idx)
            assert st == G._lib.ERR_INVALID_ARGUMENT, name
            assert ctx.launch_count() == before, name                 # refused before any device work
        with pytest.raises(G.PosDefException):                         # dependent drift columns (a zero column)
            fac.crossval(y, drift=np.column_stack([np.ones(n), np.zeros(n)]))
        # a drift column that indicates one group's points: the other points cannot identify its coefficient
        groups = [np.array([3]), np.arange(40, 60), np.array([7, 100, 250]), np.arange(200, 210)]
        for bad in (1, 2):
            Fi = np.column_stack([np.ones(n), np.zeros(n)])
            Fi[groups[bad], 1] = 1.0
            with pytest.raises(G.PosDefException) as ei:
                fac.crossval(y, drift=Fi, groups=groups)
            assert ei.value.group == bad
            st, failed = raw_call(fac, y, np.asfortranarray(Fi), 2, 4, np.cumsum([0] + [g.size for g in groups]),
                                  np.concatenate(groups))
            assert st == G._lib.ERR_NOT_POSDEF and failed == bad + 1
    finally:
        fac.free()
        op.free()
