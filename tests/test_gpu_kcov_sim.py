"""Conditional Gaussian simulation on the dense factor of the joint source-target covariance (gsi_kernelcov_chol_diag,
gsi_chol_simulate / gsi_b200.simulate, KernelCovCholesky.simulate).

With P = [S; T] (sources first), A = C(P, P) + diag(d) = L L' and standard normals Xi = [Xi_S; Xi_T]:
    g = L_SS^-1 y,  G = L_SS^-1 F_s,  B = (G'G)^-1 G' (g 1' - Xi_S),  V = [g 1' - G B; Xi_T],  Z = F_t B + L(T, :) V.

* Without a GPU: the NumPy restatement of that formula against the residual method (unconditional sample plus dual-form
  kriging of its residual) and against the conditional mean and covariance of the bordered system.
* On the GPU: the per-point diagonal (bitwise against the nugget, residual, refusals); the leading block of the joint
  factor; Z against the host formula on the downloaded factor within an elementwise rounding bound; the estimate at
  Xi = 0 against krige; sample statistics; p = 0 ignoring Xi_S; n = 20 000; reproducibility, refusals, the Python
  column loop and two ranks.
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import scipy.linalg

import oracle
from gpu_util import gsi  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G                                   # noqa: E402
from gsi_b200 import kriging                           # noqa: E402

U = 2.0 ** -53


def model_dense(structures, coords, rows=None, nugget=0.0):
    from test_gpu_kcov_model import model_dense as md
    return md(structures, coords, rows=rows, nugget=nugget)


# ------------------------------------------------------------------ host restatement
def host_simulate(L, ns, y, Fs, Ft, Xi):
    """(Z, V, B, G) of the conditioning formula on a host factor L of the joint matrix."""
    N, k = Xi.shape
    p = Fs.shape[1]
    B = np.zeros((p, k))
    G = np.zeros((ns, p))
    VS = np.zeros((ns, k))
    if ns:
        Lss = L[:ns, :ns]
        g = scipy.linalg.solve_triangular(Lss, y, lower=True)
        if p:
            G = scipy.linalg.solve_triangular(Lss, Fs, lower=True)
            B = np.linalg.solve(G.T @ G, G.T @ (g[:, None] - Xi[:ns]))
        VS = g[:, None] - G @ B
    V = np.vstack([VS, Xi[ns:]])
    return Ft @ B + L[ns:] @ V, V, B, G


def dense_case(ns, m, p, seed, tau=0.0, nugget=0.1):
    rng = np.random.default_rng(seed)
    S, T = rng.uniform(0, 20, (2, ns)), rng.uniform(0, 20, (2, m))
    st = [G.CovStructure("spherical", 1.0, [8.0, 5.0], G.rotation_matrix(0.4)),
          G.CovStructure("exponential", 0.5, [3.0, 3.0])]
    P = np.concatenate([S, T], axis=1)
    A = model_dense(st, P) + np.diag(np.r_[np.full(ns, nugget), np.full(m, tau)])
    y = np.sin(S[0] / 5) + 0.1 * rng.standard_normal(ns)
    Fs = np.column_stack([np.ones(ns), S.T / 20, (S[0] / 20) ** 2])[:, :p]
    Ft = np.column_stack([np.ones(m), T.T / 20, (T[0] / 20) ** 2])[:, :p]
    return st, S, T, A, y, Fs, Ft


def bordered(A, ns, Fs, Ft, y):
    """Conditional mean and covariance at the targets from the bordered (KKT) system."""
    p = Fs.shape[1]
    Css, Cst, Ctt = A[:ns, :ns], A[:ns, ns:], A[ns:, ns:]
    K = np.block([[Css, Fs], [Fs.T, np.zeros((p, p))]])
    R = np.vstack([Cst, Ft.T])
    sol = np.linalg.solve(K, np.concatenate([y, np.zeros(p)]))
    return R.T @ sol, Ctt - R.T @ np.linalg.solve(K, R)


@pytest.mark.parametrize("p", [0, 1, 3])
def test_formula_is_residual_method(p):
    ns, m, k = 60, 35, 7
    _, _, _, A, y, Fs, Ft = dense_case(ns, m, p, seed=p, tau=1e-3)
    L = np.linalg.cholesky(A)
    Xi = np.random.default_rng(10 + p).standard_normal((ns + m, k))
    Z, _, _, _ = host_simulate(L, ns, y, Fs, Ft, Xi)
    u = L @ Xi                                         # unconditional sample, noise included at the sources
    solve = lambda R: scipy.linalg.cho_solve((L[:ns, :ns], True), R)          # noqa: E731
    for j in range(k):
        est, _, _ = kriging.dual_kriging(solve, lambda w: A[ns:, :ns] @ w, y - u[:ns, j], Fs, Ft)
        assert np.allclose(Z[:, j], u[ns:, j] + est, rtol=0, atol=1e-11)


@pytest.mark.parametrize("p", [0, 1, 3])
def test_formula_mean_and_covariance(p):
    ns, m = 50, 30
    _, _, _, A, y, Fs, Ft = dense_case(ns, m, p, seed=20 + p, tau=1e-2)
    L = np.linalg.cholesky(A)
    Z0, _, _, _ = host_simulate(L, ns, y, Fs, Ft, np.zeros((ns + m, 1)))
    M = host_simulate(L, ns, y, Fs, Ft, np.eye(ns + m))[0] - Z0               # Z is affine in Xi: Z = Z0 + M Xi
    mean, cov = bordered(A, ns, Fs, Ft, y)
    assert np.allclose(Z0[:, 0], mean, rtol=0, atol=1e-11)
    assert np.allclose(M @ M.T, cov, rtol=0, atol=1e-11)
    if p == 0:                                         # simple kriging never reads Xi_S
        Xi = np.random.default_rng(p).standard_normal((ns + m, 4))
        Xi2 = Xi.copy()
        Xi2[:ns] *= -3.0
        assert np.array_equal(host_simulate(L, ns, y, Fs, Ft, Xi)[0], host_simulate(L, ns, y, Fs, Ft, Xi2)[0])


# ------------------------------------------------------------------ device helpers
def raw_chol(op, diag):
    """(status, failed column, L or None) of gsi_kernelcov_chol_diag; diag None passes NULL."""
    lib = op.ctx._lib
    h, col = C.c_void_p(), C.c_int64(-1)
    d = None if diag is None else np.ascontiguousarray(diag, dtype=np.float64)
    status = lib.gsi_kernelcov_chol_diag(op._h, None if d is None else G.core._pd(d), C.byref(h), C.byref(col))
    L, ld = None, None
    if h:
        n = op.shape[1]
        L = np.empty((n, n), order="F")
        G._lib.check(lib.gsi_chol_download(h, G.core._pd(L), n))
        v = C.c_double()
        G._lib.check(lib.gsi_chol_logdet(h, C.byref(v)))
        ld = v.value
        lib.gsi_chol_free(h)
    return status, int(col.value), L, ld


def scattered(n, d=2, seed=0, box=30.0):
    return np.random.default_rng(seed).uniform(0, box, (d, n))


def rot3(L):
    ang = (0.5, -0.3, 0.8)
    R1, R2 = G.rotation_matrix(ang), G.rotation_matrix(tuple(-0.7 * a for a in ang))
    L = np.asarray(L, dtype=np.float64)
    return [G.CovStructure("spherical", 0.6, L / 3, R1), G.CovStructure("exponential", 0.4, L / 5, R2),
            G.CovStructure("matern52", 0.3, L / 4, R1)]


# ------------------------------------------------------------------ 1. the diagonal
@pytest.mark.gpu
def test_diag_constant_equals_nugget_bitwise(gsi):
    n = 700
    X = scattered(n, 2, seed=1)
    c = 0.137
    op0 = gsi.KernelCovMatrix("exponential", X, [4.0, 4.0], nugget=0.0)
    opc = gsi.KernelCovMatrix("exponential", X, [4.0, 4.0], nugget=c, ctx=op0.ctx)
    s1, _, L1, ld1 = raw_chol(op0, np.full(n, c))
    fc = gsi.KernelCovCholesky(opc)
    try:
        L2, ld2 = fc.L, fc.logdet
    finally:
        fc.free()
    assert s1 == G._lib.OK and np.array_equal(L1, L2) and ld1 == ld2
    s3, _, L3, ld3 = raw_chol(opc, None)               # NULL: exactly gsi_kernelcov_chol
    assert s3 == G._lib.OK and np.array_equal(L3, L2) and ld3 == ld2


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 127, 128, 129, 3000])
def test_diag_varying_residual(gsi, n):
    X = scattered(n, 2, seed=n, box=max(n, 8) ** 0.5)
    st = [G.CovStructure("exponential", 1.0, [2.0, 2.0])]
    A0 = model_dense(st, X)
    d = np.random.default_rng(n).uniform(0.01, 0.5, n)
    op = gsi.KernelCovModelMatrix(st, X, 0.0)
    f = gsi.KernelCovCholesky(op, diag=d)
    try:
        L = f.L
    finally:
        f.free()
    A = A0 + np.diag(d)
    assert np.linalg.norm(A - L @ L.T) / np.linalg.norm(A) <= 4 * n * U


@pytest.mark.gpu
def test_diag_refusals(gsi):
    n = 300
    X = scattered(n, 2, seed=2)
    op = gsi.KernelCovMatrix("exponential", X, [3.0, 3.0], nugget=0.0)
    for v in (np.nan, np.inf, -np.inf):
        d = np.full(n, 0.1)
        d[123] = v
        status, col, L, _ = raw_chol(op, d)
        assert status == G._lib.ERR_INVALID_ARGUMENT and col == 0 and L is None
    d = np.zeros(n)
    d[200] = -2.0                                       # pivot 201 becomes negative, the earlier ones are untouched
    status, col, L, _ = raw_chol(op, d)
    assert status == G._lib.ERR_NOT_POSDEF and col == 201 and L is None
    with pytest.raises(G.PosDefException) as e:
        gsi.KernelCovCholesky(op, diag=d)
    assert e.value.column == 201
    with pytest.raises(G.DimensionMismatch):
        gsi.KernelCovCholesky(op, diag=np.zeros(n - 1))


# ------------------------------------------------------------------ 2. the leading block
@pytest.mark.gpu
@pytest.mark.parametrize("ns,m", [(129, 300), (300, 200), (256, 77)])
def test_leading_block_is_source_factor(gsi, ns, m):
    st = rot3([20.0, 20.0, 20.0])
    S, T = scattered(ns, 3, seed=ns), scattered(m, 3, seed=ns + 1)
    nug, tau = 0.05, 1e-3
    joint = gsi.KernelCovModelMatrix(st, np.concatenate([S, T], axis=1), 0.0)
    src = gsi.KernelCovModelMatrix(st, S, nug, ctx=joint.ctx)
    fj = gsi.KernelCovCholesky(joint, diag=np.r_[np.full(ns, nug), np.full(m, tau)])
    fs = gsi.KernelCovCholesky(src)
    try:
        assert np.array_equal(fj.L[:ns, :ns], fs.L)
    finally:
        fj.free()
        fs.free()


# ------------------------------------------------------------------ 3. against the host formula
def bound(L, ns, V, B, G_, Ft):
    """Elementwise rounding bound of Z = F_t B + L(T, :) V: 4 N u (|L(T, :)| (|V| + |G||B| on the source rows) +
    |F_t||B|); the |G||B| term covers the rounding of V_S = g - G B, which enters through L_TS."""
    N = L.shape[0]
    W = np.abs(V)
    W[:ns] += np.abs(G_) @ np.abs(B)
    return 4 * N * U * (np.abs(L[ns:]) @ W + np.abs(Ft) @ np.abs(B))


def drift_pair(kind, S, T, p):
    ns, m = S.shape[1], T.shape[1]
    if p == 0:
        return np.zeros((ns, 0)), np.zeros((m, 0))
    if p == 1:
        return np.ones((ns, 1)), np.ones((m, 1))
    return (np.column_stack([np.ones(ns), S[:2].T / 20]), np.column_stack([np.ones(m), T[:2].T / 20]))


CASES = [  # (model, ns, m, k, p)
    ("exponential", 1, 128, 129, 0),
    ("exponential", 127, 129, 1, 1),
    ("exponential", 128, 500, 1024, 3),
    ("exponential", 129, 1, 1, 1),
    ("exponential", 300, 129, 129, 3),
    ("rotated", 129, 500, 129, 0),
    ("rotated", 300, 128, 1024, 1),
    ("rotated", 127, 1, 1024, 3),
    ("rotated", 1, 129, 1, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("model,ns,m,k,p", CASES)
def test_against_host_formula(gsi, model, ns, m, k, p):
    rng = np.random.default_rng(ns * 7 + m + k + p)
    d = 3 if model == "rotated" else 2
    S, T = rng.uniform(0, 20, (d, ns)), rng.uniform(0, 20, (d, m))
    st = rot3([20.0] * 3) if model == "rotated" else [G.CovStructure("exponential", 1.0, [4.0, 4.0])]
    op = gsi.KernelCovModelMatrix(st, np.concatenate([S, T], axis=1), 0.0)
    f = gsi.KernelCovCholesky(op, diag=np.r_[np.full(ns, 0.1), np.full(m, 1e-3)])
    try:
        y = np.cos(S[0] / 4) + 0.1 * rng.standard_normal(ns)
        Fs, Ft = drift_pair(model, S, T, p)
        Xi = rng.standard_normal((ns + m, k))
        spec = None if p == 0 else (Fs, Ft)
        Z = f.simulate(Xi, n_cond=ns, y=y, drift=spec)
        L = f.L
    finally:
        f.free()
    Zh, V, B, G_ = host_simulate(L, ns, y, Fs, Ft, Xi)
    assert Z.shape == (m, k)
    err = np.abs(Z - Zh)
    tol = bound(L, ns, V, B, G_, Ft)
    assert np.all(err <= tol), (np.max(err / tol))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 129])
def test_unconditional_grid_model(gsi, k):
    shape = (40, 30)
    st = [G.CovStructure("spherical", 0.6, [12.0, 8.0], G.rotation_matrix(0.5)),
          G.CovStructure("exponential", 0.4, [5.0, 5.0])]
    op = gsi.GridKernelCovModelMatrix(st, shape, nugget=0.01)
    n = op.shape[1]
    f = gsi.KernelCovCholesky(op)
    try:
        Xi = np.random.default_rng(k).standard_normal((n, k))
        Z = f.simulate(Xi)
        L = f.L
    finally:
        f.free()
    assert np.all(np.abs(Z - L @ Xi) <= 4 * n * U * (np.abs(L) @ np.abs(Xi)))


# ------------------------------------------------------------------ 4. the estimate at Xi = 0
def estimate_case(n, m, seed):
    """scattered sources and targets, the nugget rule of test_gpu_kcov_chol.square_case (kappa about 2e3 n at most)"""
    rng = np.random.default_rng(seed)
    L = np.full(2, n ** 0.5)
    S, T = rng.uniform(0, 1, (2, n)) * L[:, None], rng.uniform(0, 1, (2, m)) * L[:, None]
    st = [G.CovStructure("exponential", 1.3, L / 4)]
    A0 = model_dense(st, S)
    nugget = max(1e-3, float(np.max(np.sum(np.abs(A0), axis=1))) / 2e3)
    y = np.sin(S[0] / 3) + 0.1 * rng.standard_normal(n)
    return st, S, T, A0 + nugget * np.eye(n), nugget, y


@pytest.mark.gpu
@pytest.mark.parametrize("drift", [None, "constant", "universal"])
def test_zero_xi_gives_krige_estimate(gsi, drift):
    n, m = 700, 300
    st, S, T, A, nugget, y = estimate_case(n, m, seed=4)
    spec = (np.column_stack([np.ones(n), S.T / 26]), np.column_stack([np.ones(m), T.T / 26])) \
        if drift == "universal" else drift
    yhat = gsi.krige(st, S, y, T, nugget=nugget, drift=spec, method="cholesky")
    Z = gsi.simulate(st, T, 1, sources=S, y=y, nugget=nugget, drift=spec, Xi=np.zeros((n + m, 1)))
    kap = np.linalg.cond(A)
    assert Z.shape == (m, 1)
    assert np.max(np.abs(Z[:, 0] - yhat)) <= 10 * np.sqrt(n + m) * kap * U * np.max(np.abs(yhat)), kap


# ------------------------------------------------------------------ 5. statistics
@pytest.mark.gpu
@pytest.mark.parametrize("drift", [None, "constant"])
def test_sample_statistics(gsi, drift):
    ns, m, K, tau = 150, 40, 20000, 1e-2
    _, S, T, A, y, _, _ = dense_case(ns, m, 0, seed=5, tau=tau, nugget=0.1)
    st = [G.CovStructure("spherical", 1.0, [8.0, 5.0], G.rotation_matrix(0.4)),
          G.CovStructure("exponential", 0.5, [3.0, 3.0])]
    Z = gsi.simulate(st, T, K, sources=S, y=y, nugget=0.1, target_nugget=tau, drift=drift, rng=123)
    Fs, Ft = kriging.drift_matrices(drift, ns, m)
    yhat = gsi.krige(st, S, y, T, nugget=0.1, drift=drift, method="cholesky")
    C_ss = gsi.KernelCovModelMatrix(st, S, 0.1)
    C_ts = gsi.KernelCrossCovMatrix(st, T, S, ctx=C_ss.ctx)
    f = gsi.KernelCovCholesky(C_ss)
    try:
        var = f.variance(C_ts, drift) + tau
    finally:
        f.free()
        C_ss.free()
        C_ts.free()
    _, cov = bordered(A, ns, Fs, Ft, y)
    assert np.allclose(np.diag(cov), var, rtol=1e-10, atol=1e-12)
    mu = Z.mean(axis=1)
    assert np.all(np.abs(mu - yhat) <= 6 * np.sqrt(var / K))
    ev = Z.var(axis=1, ddof=1)
    assert np.all(np.abs(ev / var - 1) <= 6 * np.sqrt(2 / K))
    ec = np.cov(Z)
    se = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / K)
    assert np.all(np.abs(ec - cov) <= 6 * se)


@pytest.mark.gpu
def test_unconditional_statistics(gsi):
    m, K = 40, 20000
    T = scattered(m, 2, seed=6, box=20.0)
    st = [G.CovStructure("exponential", 1.0, [4.0, 4.0])]
    Z = gsi.simulate(st, T, K, target_nugget=1e-3, rng=7)
    Cm = model_dense(st, T) + 1e-3 * np.eye(m)
    ec = np.cov(Z)
    se = np.sqrt((np.outer(np.diag(Cm), np.diag(Cm)) + Cm ** 2) / K)
    assert np.all(np.abs(ec - Cm) <= 6 * se)
    assert np.all(np.abs(Z.mean(axis=1)) <= 6 * np.sqrt(np.diag(Cm) / K))
    with pytest.raises(ValueError, match="conditioning data"):
        gsi.simulate(st, T, 2, drift="constant")


# ------------------------------------------------------------------ 6. p = 0 ignores Xi_S
@pytest.mark.gpu
def test_simple_kriging_ignores_source_normals(gsi):
    ns, m, k = 300, 200, 50
    rng = np.random.default_rng(8)
    S, T = rng.uniform(0, 20, (2, ns)), rng.uniform(0, 20, (2, m))
    st = [G.CovStructure("matern32", 1.0, [5.0, 5.0])]
    Xi = rng.standard_normal((ns + m, k))
    Xi2 = Xi.copy()
    Xi2[:ns] = 1e3 * rng.standard_normal((ns, k))
    y = rng.standard_normal(ns)
    Z1 = gsi.simulate(st, T, k, sources=S, y=y, nugget=0.1, Xi=Xi)
    Z2 = gsi.simulate(st, T, k, sources=S, y=y, nugget=0.1, Xi=Xi2)
    assert np.array_equal(Z1, Z2)


# ------------------------------------------------------------------ 7. scale
@pytest.mark.gpu
def test_scale_20000(gsi):
    ns, m, k = 5000, 15000, 64
    rng = np.random.default_rng(9)
    P = rng.uniform(0, 100, (2, ns + m))
    st = [G.CovStructure("exponential", 1.0, [10.0, 10.0])]
    op = gsi.KernelCovModelMatrix(st, P, 0.0)
    f = gsi.KernelCovCholesky(op, diag=np.r_[np.full(ns, 0.1), np.zeros(m)])
    try:
        y = rng.standard_normal(ns)
        Fs, Ft = np.ones((ns, 1)), np.ones((m, 1))
        Xi = rng.standard_normal((ns + m, k))
        Z = f.simulate(Xi, n_cond=ns, y=y, drift="constant")
        L = f.L
    finally:
        f.free()
        op.free()
    Zh, V, B, G_ = host_simulate(L, ns, y, Fs, Ft, Xi)
    tol = bound(L, ns, V, B, G_, Ft)
    del L
    assert np.all(np.abs(Z - Zh) <= tol), np.max(np.abs(Z - Zh) / tol)


# ------------------------------------------------------------------ 8. reproducibility, refusals, the Python loop, ranks
def sim_case(gsi, ns=200, m=150):
    rng = np.random.default_rng(11)
    S, T = rng.uniform(0, 20, (2, ns)), rng.uniform(0, 20, (2, m))
    st = [G.CovStructure("exponential", 1.0, [4.0, 4.0])]
    op = gsi.KernelCovModelMatrix(st, np.concatenate([S, T], axis=1), 0.0)
    f = gsi.KernelCovCholesky(op, diag=np.r_[np.full(ns, 0.1), np.full(m, 1e-3)])
    return op, f, S, T, rng.standard_normal(ns)


@pytest.mark.gpu
def test_reproducible_and_column_loop(gsi):
    op, f, S, T, y = sim_case(gsi)
    try:
        n = f.n
        Xi = np.random.default_rng(12).standard_normal((n, 2500))
        Z = f.simulate(Xi, n_cond=200, y=y, drift="constant")
        assert Z.shape == (150, 2500)
        assert np.array_equal(Z, f.simulate(Xi, n_cond=200, y=y, drift="constant"))
        parts = [f.simulate(Xi[:, c0:c0 + 1024], n_cond=200, y=y, drift="constant") for c0 in (0, 1024, 2048)]
        assert np.array_equal(Z, np.concatenate(parts, axis=1))
    finally:
        f.free()
        op.free()


@pytest.mark.gpu
def test_simulate_refusals(gsi):
    L = G._lib
    ns, m = 200, 150
    op, f, S, T, y = sim_case(gsi, ns, m)
    lib = op.ctx._lib
    n = ns + m
    try:
        def raw(nsv, yv, Fs, Ft, p, xrows, xcols, zrows, zcols, xl=G.LAYOUT_TALL, zl=G.LAYOUT_TALL, Xv=None):
            Xd = gsi.DeviceMatrix(op.ctx, xrows, xcols, xl)
            Zd = gsi.DeviceMatrix(op.ctx, zrows, zcols, zl)
            try:
                if Xv is not None:
                    Xd.upload(Xv)
                pd = lambda a: None if a is None else G.core._pd(a)               # noqa: E731
                return lib.gsi_chol_simulate(f._h, nsv, pd(yv), pd(Fs), pd(Ft), p, Xd._h, Zd._h)
            finally:
                Xd.free()
                Zd.free()
        F1s, F1t = np.ones((ns, 1), order="F"), np.ones((m, 1), order="F")
        X0 = np.zeros((n, 3), order="F")
        assert raw(ns, y, F1s, F1t, 1, n, 3, m, 3, Xv=X0) == L.OK
        assert raw(n, y, None, None, 0, n, 3, 1, 3) == L.ERR_INVALID_ARGUMENT                  # ns = n
        assert raw(-1, y, None, None, 0, n, 3, m, 3) == L.ERR_INVALID_ARGUMENT
        assert raw(ns, y, F1s, F1t, 33, n, 3, m, 3) == L.ERR_INVALID_ARGUMENT                  # p > 32
        assert raw(ns, y, F1s, F1t, -1, n, 3, m, 3) == L.ERR_INVALID_ARGUMENT
        assert raw(0, None, np.ones((0, 1)), np.ones((n, 1)), 1, n, 3, n, 3) == L.ERR_INVALID_ARGUMENT   # drift, ns = 0
        assert raw(ns, None, None, None, 0, n, 3, m, 3) == L.ERR_INVALID_ARGUMENT              # y missing
        for v in (np.nan, np.inf):
            yb = y.copy()
            yb[7] = v
            assert raw(ns, yb, None, None, 0, n, 3, m, 3, Xv=X0) == L.ERR_INVALID_ARGUMENT
            Fb = F1t.copy()
            Fb[3, 0] = v
            assert raw(ns, y, F1s, Fb, 1, n, 3, m, 3, Xv=X0) == L.ERR_INVALID_ARGUMENT
            Xb = X0.copy()
            Xb[n - 1, 2] = v
            assert raw(ns, y, None, None, 0, n, 3, m, 3, Xv=Xb) == L.ERR_INVALID_ARGUMENT
        assert raw(ns, y, None, None, 0, n - 1, 3, m, 3) == L.ERR_DIMENSION_MISMATCH
        assert raw(ns, y, None, None, 0, n, 3, m + 1, 3) == L.ERR_DIMENSION_MISMATCH
        assert raw(ns, y, None, None, 0, n, 3, m, 2) == L.ERR_DIMENSION_MISMATCH
        assert raw(ns, y, None, None, 0, n, 3, m, 3, xl=G.LAYOUT_COLMAJOR) == L.ERR_DIMENSION_MISMATCH
        assert raw(ns, y, None, None, 0, n, 3, m, 3, zl=G.LAYOUT_COLMAJOR) == L.ERR_DIMENSION_MISMATCH
        Fdup = np.column_stack([np.ones(ns), np.zeros(ns)])                                     # dependent columns
        assert raw(ns, y, np.asfortranarray(Fdup), np.ones((m, 2), order="F"), 2, n, 3, m, 3, Xv=X0) == L.ERR_NOT_POSDEF
        with pytest.raises(G.PosDefException):
            f.simulate(X0, n_cond=ns, y=y, drift=(Fdup, np.ones((m, 2))))
        assert np.all(np.isfinite(f.simulate(X0, n_cond=ns, y=y)))                               # still usable
    finally:
        f.free()
        op.free()


@pytest.mark.gpu
def test_two_ranks_unsupported(gsi):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29553", os.path.join(ROOT, "tests", "dist_kcov_sim_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        for rank in range(2):
            status, made = open(os.path.join(tmp, f"sim_rank{rank}.txt")).read().split()
            assert int(status) == G._lib.ERR_UNSUPPORTED and made == "0"


def test_simulation_exports():
    assert G.simulate is kriging.simulate
    for name in ("gsi_kernelcov_chol_diag", "gsi_chol_simulate"):
        assert name in G._lib.SIGNATURES
