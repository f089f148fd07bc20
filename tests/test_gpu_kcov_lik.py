"""Gaussian log-likelihood of the covariance parameters and its exact gradient (gsi_kernelcov_loglik / gsi_b200.loglik),
and maximum-likelihood fitting on it (gsi_b200.fit_covariance).

With A = C(S, S) + nugget I = L L', g = L^-1 y, G = L^-1 F, R'R = G'G, beta = (G'G)^-1 G'g, e = g - G beta, q = ||e||^2:
    ML   = -1/2 (n log 2 pi + log det A + q)
    REML = -1/2 ((n - p) log 2 pi + log det A + 2 sum log R_kk + q)
    d l / d theta = 1/2 sum_ij W_ij dA_ij / dtheta,  W = alpha alpha' - A^-1 (+ H H' for REML)

* Without a GPU: the NumPy restatement against scipy's multivariate normal (ML, p = 0) and the explicit P-matrix form of
  REML; the analytic host gradient against central differences of the host value for every kind, d = 1..3, rotated
  2-4-structure models, p in {0, 1, 3}, ML and REML.
* On the GPU: value and beta against the host within 1e-12 (n + |log det A| + q); the gradient against the host gradient
  within 1e-11 S_theta (S_theta = 1/2 sum |W| |dA / dtheta|), both 1 % of the first bounds 1e-10 and 1e-9 (largest
  measured on a B200 at 1000 W: 2.3e-15 (n + |log det A| + q) and 4.6e-14 S_theta), and against central differences of
  the device value (largest measured: 6.8e-8 S_theta against 1e-5); n = 20 000; bit equalities;
  refusals; two ranks; the fit against host L-BFGS-B on the host likelihood.  Lines starting with LIKREPORT carry the
  measured worst ratios.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import scipy.linalg
import scipy.optimize
import scipy.stats

from gpu_util import gsi  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G                                   # noqa: E402
from gsi_b200 import kriging                           # noqa: E402

KINDS = ["exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"]
CS = G.CovStructure


# ------------------------------------------------------------------ host model and its derivatives
def coords_of(st, X):
    """Unscaled principal-axis coordinates (R x) / range of one structure (d x n)."""
    d = X.shape[0]
    Y = X if st.rotation is None else st.rotation.reshape(d, d) @ X
    return Y / np.broadcast_to(st.ranges, (d,))[:, None]


def kval(kind, r2, beta):
    from test_gpu_kcov_model import kvalue
    return kvalue(kind, r2, beta)


def kder(kind, r2, beta):
    """dk / dr2 of the unscaled definitions (include/gsi_b200.h); 0 where r2 = 0 (multiplied by du^2 = 0 there)."""
    s = np.sqrt(r2)
    safe = np.where(s > 0, s, 1.0)
    if kind == 0:
        return np.where(s > 0, -np.exp(-s) / (2 * safe), 0.0)
    if kind == 1:
        return -0.5 * np.exp(-0.5 * r2)
    if kind == 2:
        return -beta * (1.0 + r2) ** (-beta - 1.0)
    if kind == 3:
        return -1.5 * np.exp(-np.sqrt(3.0 * r2))
    if kind == 4:
        t = np.sqrt(5.0 * r2)
        return -(5.0 / 6.0) * (1.0 + t) * np.exp(-t)
    return np.where((s > 0) & (s < 1), -0.75 * (1 - s) * (1 + s) / safe, 0.0)


def host_A(sts, X, nugget):
    """A and the list of dA / dtheta (per structure: sill, ranges; then the nugget)."""
    n, d = X.shape[1], X.shape[0]
    A = nugget * np.eye(n)
    dA = []
    for st in sts:
        u = coords_of(st, X)
        du2 = (u[:, :, None] - u[:, None, :]) ** 2
        r2 = du2.sum(axis=0)
        k = kval(st.kind, r2, st.beta)
        A = A + st.sill * k
        dA.append(k)
        kp = kder(st.kind, r2, st.beta)
        rng = np.broadcast_to(st.ranges, (d,))
        for a in range(d):
            dA.append(st.sill * kp * (-2.0 * du2[a]) / rng[a])
    dA.append(np.eye(n))
    return A, dA


def host_lik(A, y, F, reml):
    """(value, beta, W, q, logdet) of the Cholesky restatement."""
    n, p = F.shape
    L = np.linalg.cholesky(A)
    g = scipy.linalg.solve_triangular(L, y, lower=True)
    Gm = scipy.linalg.solve_triangular(L, F, lower=True)
    logdet = 2 * np.log(np.diag(L)).sum()
    if p:
        R = np.linalg.cholesky(Gm.T @ Gm).T
        beta = np.linalg.solve(Gm.T @ Gm, Gm.T @ g)
        ldr = np.log(np.diag(R)).sum()
    else:
        R, beta, ldr = np.zeros((0, 0)), np.zeros(0), 0.0
    e = g - Gm @ beta
    q = e @ e
    Ai = scipy.linalg.cho_solve((L, True), np.eye(n))
    alpha = scipy.linalg.solve_triangular(L.T, e, lower=False)
    W = np.outer(alpha, alpha) - Ai
    if reml and p:
        H = scipy.linalg.solve_triangular(L.T, scipy.linalg.solve_triangular(R.T, Gm.T, lower=True).T, lower=False)
        W = W + H @ H.T
    if reml:
        v = -0.5 * ((n - p) * np.log(2 * np.pi) + logdet + 2 * ldr + q)
    else:
        v = -0.5 * (n * np.log(2 * np.pi) + logdet + q)
    return v, beta, W, q, logdet


def host_grad(W, dA):
    g = np.array([0.5 * np.sum(W * D) for D in dA])
    S = np.array([0.5 * np.sum(np.abs(W) * np.abs(D)) for D in dA])
    return g, S


def drift(X, p):
    n = X.shape[1]
    return np.column_stack([np.ones(n), X.T / 10.0, (X[0] / 10.0) ** 2])[:, :p]


def perturbed(sts, nugget, idx, h):
    """The model with parameter idx (ABI order) scaled by (1 + h)."""
    d = len(sts[0].ranges)
    out, k = [], 0
    for st in sts:
        sill, rng = st.sill, np.array(np.broadcast_to(st.ranges, (d,)), dtype=np.float64)
        if idx == k:
            sill = sill * (1 + h)
        for a in range(d):
            if idx == k + 1 + a:
                rng[a] = rng[a] * (1 + h)
        k += 1 + d
        out.append(CS(st.kind, sill, rng, st.rotation, st.beta))
    return out, nugget * (1 + h) if idx == k else nugget


def base_value(sts, nugget, idx):
    if idx == len(sts) * (1 + len(sts[0].ranges)):
        return nugget
    d = len(sts[0].ranges)
    s, r = divmod(idx, 1 + d)
    return sts[s].sill if r == 0 else sts[s].ranges[r - 1]


def cases():
    """(name, structures, d): every kind at d = 1..3, and rotated nested models of 2-4 structures."""
    out = []
    for i, kind in enumerate(KINDS):
        for d in (1, 2, 3):
            ell = np.array([4.0, 2.5, 3.0][:d])
            out.append((f"{kind}_d{d}", [CS(kind, 1.3, ell, beta=0.8 if kind == "powerlaw" else 1.0)], d))
    r2a, r2b = G.rotation_matrix(0.5), G.rotation_matrix(-0.35)
    r3a, r3b = G.rotation_matrix((0.5, -0.3, 0.8)), G.rotation_matrix((-0.35, 0.2, -0.6))
    out.append(("sph_exp_d2", [CS("spherical", 0.6, [6.0, 3.0], r2a), CS("exponential", 0.4, [2.0, 3.5], r2b)], 2))
    out.append(("three_d3", [CS("spherical", 0.5, [5.0, 3.0, 4.0], r3b), CS("matern32", 0.7, [1.5, 2.0, 1.0], r3a),
                             CS("exponential", 1.3, [3.0, 3.0, 2.0])], 3))
    out.append(("four_d2", [CS("gaussian", 0.3, [2.5, 1.5], r2a), CS("matern52", 0.9, [3.0, 2.0], r2b),
                            CS("powerlaw", 0.2, [2.0, 2.0], beta=0.8), CS("matern32", 1.1, [4.0, 2.5], r2a)], 2))
    return out


CASES = cases()
CASE_IDS = [c[0] for c in CASES]


def points(n, d, seed):
    return np.random.default_rng(seed).uniform(0, 10, (d, n))


def observations(A, X, seed):
    rng = np.random.default_rng(seed)
    L = np.linalg.cholesky(A)
    return 0.7 + 0.2 * X[0] + L @ rng.standard_normal(A.shape[0])


def total_sill(sts):
    return sum(st.sill for st in sts)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("p", [0, 1, 3])
def test_host_values(p):
    X = points(60, 2, 1)
    sts = CASES[CASE_IDS.index("sph_exp_d2")][1]
    A, _ = host_A(sts, X, 0.1)
    y = observations(A, X, 2)
    F = drift(X, p)
    v_ml, beta, _, _, _ = host_lik(A, y, F, False)
    Ai = np.linalg.inv(A)
    if p == 0:
        ref = scipy.stats.multivariate_normal(mean=np.zeros(60), cov=A).logpdf(y)
        assert abs(v_ml - ref) <= 1e-10 * abs(ref)
    else:
        b = np.linalg.solve(F.T @ Ai @ F, F.T @ Ai @ y)
        assert np.allclose(beta, b, rtol=1e-10, atol=1e-12)
        r = y - F @ b
        ref = scipy.stats.multivariate_normal(mean=F @ b, cov=A).logpdf(y)
        assert abs(v_ml - ref) <= 1e-10 * abs(ref)
        assert r.shape == (60,)
    # REML: the explicit projection P = A^-1 - A^-1 F (F'A^-1 F)^-1 F'A^-1
    v_reml = host_lik(A, y, F, True)[0]
    P = Ai - (Ai @ F @ np.linalg.solve(F.T @ Ai @ F, F.T @ Ai) if p else 0.0)
    ld = np.linalg.slogdet(A)[1] + (np.linalg.slogdet(F.T @ Ai @ F)[1] if p else 0.0)
    ref = -0.5 * ((60 - p) * np.log(2 * np.pi) + ld + y @ P @ y)
    assert abs(v_reml - ref) <= 1e-10 * abs(ref)


@pytest.mark.parametrize("reml", [False, True])
@pytest.mark.parametrize("p", [0, 1, 3])
@pytest.mark.parametrize("case", CASE_IDS)
def test_host_gradient_fd(case, p, reml):
    """The analytic host gradient against central differences of the host value (h = 1e-5 relative)."""
    _, sts, d = CASES[CASE_IDS.index(case)]
    X = points(50, d, 3)
    nug = 0.1 * total_sill(sts)
    A, dA = host_A(sts, X, nug)
    y = observations(A, X, 4)
    F = drift(X, p)
    _, _, W, _, _ = host_lik(A, y, F, reml)
    g, S = host_grad(W, dA)
    h = 1e-5
    for idx in range(len(dA)):
        th = base_value(sts, nug, idx)
        vals = []
        for sgn in (1, -1):
            s2, n2 = perturbed(sts, nug, idx, sgn * h)
            vals.append(host_lik(host_A(s2, X, n2)[0], y, F, reml)[0])
        fd = (vals[0] - vals[1]) / (2 * h * th)
        assert abs(fd - g[idx]) <= 1e-7 * (S[idx] + abs(g[idx])) + 1e-9, (idx, fd, g[idx], S[idx])


def test_exports():
    assert G.loglik is kriging.loglik and G.fit_covariance is kriging.fit_covariance
    assert "gsi_kernelcov_loglik" in G._lib.SIGNATURES


# ------------------------------------------------------------------ GPU helpers
def device_op(sts, X, nug, single):
    if single:
        st = sts[0]
        return G.KernelCovMatrix(st.kind, X, st.ranges, sigma2=st.sill, nugget=nug, beta=st.beta)
    return G.KernelCovModelMatrix(sts, X, nug)


def device_lik(sts, X, nug, y, F, reml, grad, single=False):
    op = device_op(sts, X, nug, single)
    try:
        return G.loglik(op, y, drift=F if F.shape[1] else None, reml=reml, grad=grad)
    finally:
        op.free()


WORST = {"value": 0.0, "grad": 0.0, "fd": 0.0}


def report():
    print(f"LIKREPORT worst value ratio {WORST['value']:.3e} (of 1e-12 (n + |logdet| + q)), gradient ratio "
          f"{WORST['grad']:.3e} (of 1e-11 S), device central differences {WORST['fd']:.3e} (of 1e-5 S)")


# ------------------------------------------------------------------ GPU
GPU_GRID = [(c, p, reml) for c in CASE_IDS for p in (0, 1, 3) for reml in (False, True)
            if p == 1 or c in ("exponential_d2", "sph_exp_d2", "three_d3", "four_d2", "spherical_d1", "matern52_d3")]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [257, 2000])
@pytest.mark.parametrize("case,p,reml", GPU_GRID)
def test_device_vs_host(gsi, case, p, reml, n):
    if n == 2000 and not (reml and p == 1) and case not in ("sph_exp_d2", "three_d3"):
        pytest.skip("n = 2000 runs the REML p = 1 column and the two rotated models")
    _, sts, d = CASES[CASE_IDS.index(case)]
    X = points(n, d, 5)
    nug = 0.05 * total_sill(sts)
    A, dA = host_A(sts, X, nug)
    y = observations(A, X, 6)
    F = drift(X, p)
    v, beta, W, q, logdet = host_lik(A, y, F, reml)
    g_host, S = host_grad(W, dA)
    single = len(sts) == 1
    vd, bd, gd = device_lik(sts, X, nug, y, F, reml, True, single=single)
    tol_v = 1e-12 * (n + abs(logdet) + q)
    assert abs(vd - v) <= tol_v, (vd, v)
    WORST["value"] = max(WORST["value"], abs(vd - v) / tol_v)
    if p:
        assert np.allclose(bd, beta, rtol=1e-8, atol=1e-9 * np.abs(beta).max())
    assert gd.shape == g_host.shape
    ratio = np.abs(gd - g_host) / (1e-11 * S)
    WORST["grad"] = max(WORST["grad"], float(ratio.max()))
    assert np.all(ratio <= 1.0), (ratio, gd, g_host)
    report()


FD_CASES = ["exponential_d2", "matern52_d1", "spherical_d3", "powerlaw_d2", "sph_exp_d2", "three_d3"]


@pytest.mark.gpu
@pytest.mark.parametrize("reml", [False, True])
@pytest.mark.parametrize("case", FD_CASES)
def test_device_gradient_fd(gsi, case, reml):
    """The device gradient against central differences of the device value, rebuilding the operator at theta (1 +- h),
    h = 1e-4: independent of the host formula."""
    _, sts, d = CASES[CASE_IDS.index(case)]
    n = 700
    X = points(n, d, 7)
    nug = 0.05 * total_sill(sts)
    A, dA = host_A(sts, X, nug)
    y = observations(A, X, 8)
    F = drift(X, 1)
    _, _, W, _, _ = host_lik(A, y, F, reml)
    _, S = host_grad(W, dA)
    _, _, gd = device_lik(sts, X, nug, y, F, reml, True)
    h = 1e-4
    for idx in range(len(dA)):
        th = base_value(sts, nug, idx)
        vals = []
        for sgn in (1, -1):
            s2, n2 = perturbed(sts, nug, idx, sgn * h)
            vals.append(device_lik(s2, X, n2, y, F, reml, False)[0])
        fd = (vals[0] - vals[1]) / (2 * h * th)
        WORST["fd"] = max(WORST["fd"], abs(fd - gd[idx]) / (1e-5 * S[idx]))
        assert abs(fd - gd[idx]) <= 1e-5 * S[idx], (idx, fd, gd[idx], S[idx])
    report()


@pytest.mark.gpu
def test_n20000_reml(gsi):
    """A rotated two-structure model at n = 20 000 (p = 1, REML) against central differences of the device value.  The
    host cannot form S_theta at this size; n / theta, the size of 1/2 tr(A^-1 dA / dtheta) for a sill or the nugget, stands
    in for it."""
    n = 20000
    sts = [CS("spherical", 0.6, [30.0, 15.0], G.rotation_matrix(0.5)),
           CS("exponential", 0.4, [8.0, 12.0], G.rotation_matrix(-0.35))]
    X = np.random.default_rng(9).uniform(0, 100, (2, n))
    nug = 0.1
    y = 0.5 + 0.01 * X[0] + np.random.default_rng(10).standard_normal(n)
    F = np.ones((n, 1))
    v, _, gd = device_lik(sts, X, nug, y, F, True, True)
    assert np.isfinite(v) and np.all(np.isfinite(gd))
    h = 1e-4
    for idx in range(len(gd)):
        th = base_value(sts, nug, idx)
        vals = []
        for sgn in (1, -1):
            s2, n2 = perturbed(sts, nug, idx, sgn * h)
            vals.append(device_lik(s2, X, n2, y, F, True, False)[0])
        fd = (vals[0] - vals[1]) / (2 * h * th)
        assert abs(fd - gd[idx]) <= 1e-5 * (abs(gd[idx]) + n / th), (idx, fd, gd[idx])


@pytest.mark.gpu
def test_bit_equalities(gsi):
    """A single kind and the equivalent one-structure model give the same bits; the value-only call gives the bits of
    the gradient call; two identical calls agree bit for bit (n = 1000: not a multiple of 128)."""
    n = 1000
    X = points(n, 2, 11)
    st = [CS("matern32", 1.2, [2.0, 3.0])]
    A, _ = host_A(st, X, 0.1)
    y = observations(A, X, 12)
    F = drift(X, 3)
    a = device_lik(st, X, 0.1, y, F, True, True, single=True)
    b = device_lik(st, X, 0.1, y, F, True, True, single=False)
    c = device_lik(st, X, 0.1, y, F, True, False)
    e = device_lik(st, X, 0.1, y, F, True, True, single=True)
    assert a[0] == b[0] == c[0] == e[0]
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[1], c[1])
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[2], e[2])
    sts = CASES[CASE_IDS.index("three_d3")][1]
    X3 = points(n, 3, 13)
    r1 = device_lik(sts, X3, 0.2, y, F[:, :1], False, True)
    r2 = device_lik(sts, X3, 0.2, y, F[:, :1], False, True)
    assert r1[0] == r2[0] and np.array_equal(r1[2], r2[2])


@pytest.mark.gpu
def test_grid_operator(gsi):
    """A grid operator gives the value (matching the coordinate operator) and refuses the gradient."""
    shape, spacing = (23, 17), 0.5
    sts = [CS("exponential", 1.0, [3.0, 2.0], G.rotation_matrix(0.4)), CS("gaussian", 0.5, [2.0, 2.0])]
    gop = G.GridKernelCovModelMatrix(sts, shape, spacing=spacing, nugget=0.1)
    ix, iy = np.meshgrid(np.arange(shape[0]), np.arange(shape[1]), indexing="ij")
    X = np.vstack([ix.ravel(order="F"), iy.ravel(order="F")]) * spacing
    n = X.shape[1]
    y = np.sin(X[0]) + np.cos(X[1] / 2)
    try:
        vg, bg = G.loglik(gop, y, drift="constant", reml=True)
        with pytest.raises(G.GsiError) as ei:
            G.loglik(gop, y, drift="constant", reml=True, grad=True)
        assert ei.value.code == G._lib.ERR_UNSUPPORTED
    finally:
        gop.free()
    vc, bc = device_lik(sts, X, 0.1, y, np.ones((n, 1)), True, False)
    A, _ = host_A(sts, X, 0.1)
    _, _, _, q, logdet = host_lik(A, y, np.ones((n, 1)), True)
    assert abs(vg - vc) <= 1e-10 * (n + abs(logdet) + q)
    assert np.allclose(bg, bc, rtol=1e-9)


@pytest.mark.gpu
def test_refusals(gsi):
    n = 300
    X = points(n, 2, 14)
    y = np.random.default_rng(15).standard_normal(n)
    op = G.KernelCovMatrix("exponential", X, [2.0, 2.0], nugget=0.1)
    try:
        F = np.ones((n, 2))                                            # dependent drift columns
        with pytest.raises(G.PosDefException):
            G.loglik(op, y, drift=F)
        with pytest.raises(G.GsiError) as ei:
            G.loglik(op, y, drift=np.ones((n, 33)) + np.arange(33))
        assert ei.value.code == G._lib.ERR_INVALID_ARGUMENT
        yb = y.copy()
        yb[7] = np.nan
        with pytest.raises(G.GsiError) as ei:
            G.loglik(op, yb)
        assert ei.value.code == G._lib.ERR_INVALID_ARGUMENT
        Fb = np.ones((n, 1))
        Fb[3, 0] = np.inf
        with pytest.raises(G.GsiError) as ei:
            G.loglik(op, y, drift=Fb, grad=True)
        assert ei.value.code == G._lib.ERR_INVALID_ARGUMENT
    finally:
        op.free()
    Xs = points(5, 2, 16)
    small = G.KernelCovMatrix("exponential", Xs, [2.0, 2.0], nugget=0.1)
    try:
        with pytest.raises(G.GsiError) as ei:
            G.loglik(small, np.ones(5), drift=np.column_stack([np.ones(5), Xs.T, Xs[0] ** 2, Xs[1] ** 2]), reml=True)
        assert ei.value.code == G._lib.ERR_INVALID_ARGUMENT
    finally:
        small.free()
    import oracle
    Xg = oracle.grid_coords((30, 30)).astype(np.float64)               # numerically singular: Gaussian, no nugget
    bad = G.KernelCovMatrix("gaussian", Xg, [8.0, 8.0])
    try:
        with pytest.raises(G.PosDefException) as ei:
            G.loglik(bad, np.ones(900), grad=True)
        assert 1 <= ei.value.column <= 900
    finally:
        bad.free()


@pytest.mark.gpu
def test_two_ranks_unsupported(gsi):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29557", os.path.join(ROOT, "tests", "dist_kcov_lik_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        for rank in range(2):
            assert int(open(os.path.join(tmp, f"lik_rank{rank}.txt")).read()) == G._lib.ERR_UNSUPPORTED


# ------------------------------------------------------------------ fit
FIT_TRUE = [CS("spherical", 1.0, [25.0, 25.0]), CS("exponential", 0.5, [4.0, 4.0])]


def fit_data():
    n = 1500
    X = np.random.default_rng(20).uniform(0, 100, (2, n))
    y = G.simulate(FIT_TRUE, X, 1, target_nugget=0.2, rng=np.random.default_rng(21))[:, 0] + 1.0
    start = [CS("spherical", 1.4, [18.0, 18.0]), CS("exponential", 0.3, [6.0, 6.0])]
    return X, y, start, 0.3


def host_fit(X, y, start, nug0):
    """Host L-BFGS-B on the host REML likelihood, isotropic, same log parametrisation and options as fit_covariance."""
    d = X.shape[0]

    def unpack(x):
        return ([CS(st.kind, np.exp(x[2 * s]), np.full(d, np.exp(x[2 * s + 1])), st.rotation, st.beta)
                 for s, st in enumerate(start)], float(np.exp(x[-1])))

    def fun(x):
        sts, nug = unpack(x)
        A, dA = host_A(sts, X, nug)
        v, _, W, _, _ = host_lik(A, y, np.ones((X.shape[1], 1)), True)
        g, _ = host_grad(W, dA)
        lg = []
        for s, st in enumerate(sts):
            gs = g[s * (1 + d):(s + 1) * (1 + d)]
            lg += [st.sill * gs[0], (st.ranges * gs[1:]).sum()]
        lg.append(nug * g[-1])
        return -v, -np.array(lg)

    x0 = np.array(sum([[np.log(st.sill), np.log(st.ranges[0])] for st in start], []) + [np.log(nug0)])
    res = scipy.optimize.minimize(fun, x0, jac=True, method="L-BFGS-B", options=kriging.FIT_OPTIONS | {"maxiter": 200})
    return unpack(res.x), -res.fun


@pytest.mark.gpu
def test_fit_against_host(gsi):
    X, y, start, nug0 = fit_data()
    sts, nug, info = G.fit_covariance(start, X, y, nugget=nug0, drift="constant", reml=True, isotropic=True)
    (hsts, hnug), hval = host_fit(X, y, start, nug0)
    dev = np.array([p for st in sts for p in (st.sill, st.ranges[0])] + [nug])
    host = np.array([p for st in hsts for p in (st.sill, st.ranges[0])] + [hnug])
    print(f"LIKREPORT fit device {dev.tolist()} host {host.tolist()} loglik {info['loglik']!r} {hval!r} "
          f"nit {info['nit']} nfev {info['nfev']}")
    for st in sts:
        assert st.ranges[0] == st.ranges[1]                            # isotropic ties the ranges
    assert np.all(np.abs(dev - host) <= 1e-4 * np.abs(host)), (dev, host)
    assert abs(info["loglik"] - hval) <= 1e-8 * abs(hval)
    # projected gradient in log parameters at the result: small against the size of its terms (~ n)
    lg = [sts[0].sill * info["grad"][0], (sts[0].ranges * info["grad"][1:3]).sum(),
          sts[1].sill * info["grad"][3], (sts[1].ranges * info["grad"][4:6]).sum(), nug * info["grad"][6]]
    assert np.max(np.abs(lg)) <= 1e-3 * X.shape[1], lg


@pytest.mark.gpu
def test_fit_fixed_parameters(gsi):
    X, y, start, nug0 = fit_data()
    rot = [CS("spherical", 1.4, [18.0, 14.0], G.rotation_matrix(0.3)), CS("exponential", 0.3, [6.0, 6.0])]
    sts, nug, info = G.fit_covariance(rot, X[:, :600], y[:600], nugget=nug0, drift="constant", fit_nugget=False,
                                      maxiter=5)
    assert nug == nug0
    assert np.array_equal(sts[0].rotation, rot[0].rotation) and sts[1].rotation is None
    assert info["nfev"] >= 1 and info["grad"].shape == (7,)
