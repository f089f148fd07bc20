"""Kriging solve on the matrix-free covariance operator (gsi_kernelcov_solve / gsi_b200.cov_solve / gsi_b200.krige).

* CPU: a NumPy restatement of the randomized Nystrom preconditioner (Frangella, Tropp and Udell 2023, Alg. 2.1) and of
  the column-wise preconditioned CG the device runs; with a dense K its eigenvalue estimates lie below the true ones
  and match the top ones, and the preconditioned recurrence converges in fewer iterations than plain CG.  The
  dual-form kriging algebra of gsi_b200.krige equals the bordered system [C F; F' 0] for simple, ordinary and
  universal kriging.
* GPU: every square operator path (exponential, Matern 5/2 and spherical coordinates, a Gaussian lattice table, rotated
  2-4-structure models on the fused arithmetic kind and on the signed table), d = 1..3, n from 1 to a size with a
  stream-K tail, k from 1 to 300: the reported true relative residual meets rtol and agrees with the dense host
  residual.  The device preconditioner matches the host restatement (eigenvalues, iteration counts); solves are
  bit-reproducible; zero and easy columns stop early; krige matches the dense host solution; the error paths; two
  ranks.
"""
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
import gsi_b200 as G                                   # noqa: E402  (importing needs no GPU)
from gsi_b200 import kriging                           # noqa: E402

U = 2.0 ** -53
RTOL = 1e-10


# ------------------------------------------------------------------ host restatements
def nystrom_host(A, mu, Omega):
    """(U, lambda) of the randomized Nystrom approximation of K = A - mu I from the sketch Omega, step by step as the
    device builds it (FTU Alg. 2.1 with the shift nu = sqrt(n) eps ||Y||_F)."""
    n = A.shape[0]
    Om, _ = np.linalg.qr(Omega)
    Y = A @ Om - mu * Om
    nu = np.sqrt(n) * 2.0 ** -52 * np.linalg.norm(Y)
    Ynu = Y + nu * Om
    C = scipy.linalg.cholesky(Om.T @ Ynu, lower=False)          # upper triangle, as dpotrf 'U'
    F = scipy.linalg.solve_triangular(C, Ynu.T, trans="T", lower=False).T
    Uf, s, _ = np.linalg.svd(F, full_matrices=False)
    return Uf, np.maximum(0.0, s * s - nu)


def pcg_host(A, B, rtol, maxiter, Uf=None, lam=None, mu=0.0):
    """Column-wise preconditioned CG as the device runs it: column j stops when its recursive residual satisfies
    ||r_j|| <= rtol ||b_j||; P^-1 r = r + U diag((lam_r + mu) / (lam + mu) - 1) U' r.  Returns (X, iterations)."""
    n, k = B.shape
    X = np.zeros((n, k))
    R = B.copy()
    bn = np.linalg.norm(B, axis=0)
    iters = np.zeros(k, dtype=np.int64)
    active = ~(np.linalg.norm(R, axis=0) <= rtol * bn)

    def prec(R):
        if Uf is None:
            return R.copy()
        d = (lam[-1] + mu) / (lam + mu) - 1.0
        return R + Uf @ (d[:, None] * (Uf.T @ R))

    Z = prec(R)
    rz = np.sum(R * Z, axis=0)
    P = np.where(active, Z, 0.0)
    it = 0
    while active.any() and it < maxiter:
        it += 1
        Q = A @ P
        alpha = np.where(active, rz / np.where(active, np.sum(P * Q, axis=0), 1.0), 0.0)
        X += alpha * P
        R -= alpha * Q
        done = active & (np.linalg.norm(R, axis=0) <= rtol * bn)
        iters[done] = it
        active &= ~done
        Z = prec(R)
        rz_new = np.sum(R * Z, axis=0)
        P = np.where(active, Z + (rz_new / np.where(rz != 0, rz, 1.0)) * P, 0.0)
        rz = rz_new
    iters[active] = it
    return X, iters


def kernel_dense(structures, coords, nugget=0.0):
    from test_gpu_kcov_model import model_dense
    return model_dense(structures, coords, nugget=nugget)


def kappa_bound(A, nugget):
    """Upper bound of the condition number of K + nugget I (K positive semidefinite): max row sum of |A| over nugget."""
    return float(np.max(np.sum(np.abs(A), axis=1)) / nugget)


# ------------------------------------------------------------------ CPU
def _cpu_case(kind="exponential", n=500, nugget=1e-3, seed=0, ranges=(2.0, 1.5)):
    rng = np.random.default_rng(seed)
    coords = rng.uniform(0.0, 10.0, (2, n))
    A = kernel_dense([G.CovStructure(kind, 1.0, list(ranges))], coords, nugget)
    return A, rng


def test_nystrom_host_eigenvalues():
    """lambda_hat <= the eigenvalues of K (a Nystrom approximation is below K) and the top ones match."""
    A, rng = _cpu_case("gaussian", 400, 0.0, ranges=(5.0, 4.0))
    lam_true = np.linalg.eigvalsh(A)[::-1]
    Uf, lam = nystrom_host(A, 0.0, rng.standard_normal((400, 60)))
    assert np.allclose(Uf.T @ Uf, np.eye(60), atol=1e-12)
    assert np.all(lam <= lam_true[:60] + 1e-10 * lam_true[0])
    assert np.max(np.abs(lam[:10] - lam_true[:10]) / lam_true[:10]) < 1e-6


def test_pcg_host_beats_cg():
    """On a fixed seeded case the Nystrom-preconditioned recurrence reaches rtol in fewer iterations than plain CG,
    and both meet rtol on the true residual."""
    A, rng = _cpu_case("exponential", 600, 1e-3, seed=3)
    B = rng.standard_normal((600, 3))
    X0, it0 = pcg_host(A, B, 1e-8, 600)
    Uf, lam = nystrom_host(A, 1e-3, rng.standard_normal((600, 100)))
    X1, it1 = pcg_host(A, B, 1e-8, 600, Uf, lam, 1e-3)
    for X in (X0, X1):
        assert np.all(np.linalg.norm(B - A @ X, axis=0) <= 1e-7 * np.linalg.norm(B, axis=0))
    assert np.all(it1 < it0), (it0, it1)


def _kkt(C, F, y, Cts, FT):
    n, p = F.shape
    K = np.block([[C, F], [F.T, np.zeros((p, p))]])
    sol = np.linalg.solve(K, np.concatenate([y, np.zeros(p)]))
    w, beta = sol[:n], sol[n:]
    return Cts @ w + FT @ beta, beta, w


@pytest.mark.parametrize("drift", [None, "constant", "universal"])
def test_dual_kriging_equals_kkt(drift):
    rng = np.random.default_rng(11)
    n, m = 300, 120
    S, T = rng.uniform(0, 10, (2, n)), rng.uniform(0, 10, (2, m))
    st = [G.CovStructure("spherical", 1.0, [4.0, 3.0]), G.CovStructure("exponential", 0.5, [2.0, 2.0])]
    full = kernel_dense(st, np.concatenate([S, T], axis=1))
    C = full[:n, :n] + 0.05 * np.eye(n)
    Cts = full[n:, :n]
    y = rng.standard_normal(n)
    spec = (np.column_stack([np.ones(n), S.T]), np.column_stack([np.ones(m), T.T])) if drift == "universal" else drift
    F, FT = kriging.drift_matrices(spec, n, m)
    yhat, beta, w = kriging.dual_kriging(lambda R: np.linalg.solve(C, R), lambda w: Cts @ w, y, F, FT)
    y2, b2, w2 = _kkt(C, F, y, Cts, FT)
    assert F.shape[1] == {None: 0, "constant": 1, "universal": 3}[drift]
    assert np.linalg.norm(yhat - y2) <= 1e-10 * np.linalg.norm(y2)
    assert np.linalg.norm(w - w2) <= 1e-10 * np.linalg.norm(w2)
    if F.shape[1]:
        assert np.linalg.norm(beta - b2) <= 1e-10 * np.linalg.norm(b2)
        assert np.linalg.norm(F.T @ w) <= 1e-10 * np.linalg.norm(F) * np.linalg.norm(w)


def test_cov_solve_exports():
    assert G.cov_solve is kriging.cov_solve and G.krige is kriging.krige
    assert "gsi_kernelcov_solve" in G._lib.SIGNATURES


# ------------------------------------------------------------------ GPU: coverage
def _models(d, L):
    L = np.asarray(L, dtype=np.float64)
    if d == 1:
        return [G.CovStructure("spherical", 0.6, L / 3), G.CovStructure("exponential", 0.4, L / 5),
                G.CovStructure("matern32", 0.5, L / 4)]
    ang = (0.5,) if d == 2 else (0.5, -0.3, 0.8)
    R1, R2 = G.rotation_matrix(ang), G.rotation_matrix(tuple(-0.7 * a for a in ang))
    return [G.CovStructure("spherical", 0.6, L / 3, R1), G.CovStructure("exponential", 0.4, L / 5, R2),
            G.CovStructure("matern52", 0.3, L / 4, R1), G.CovStructure("gaussian", 0.2, L / 6)][:2 + d % 3]


GRIDS = {(1, 65): (65,), (2, 63): (9, 7), (2, 1000): (40, 25), (3, 5000): (25, 20, 10)}


def build_case(gsi, path, d, n, nugget=None):
    """(operator, dense matrix, nugget) of one coverage case."""
    rng = np.random.default_rng(100 * d + n % 97)
    if path in ("gauss_table", "model_table"):
        shape = GRIDS[(d, n)]
        coords = oracle.grid_coords(shape)
        L = np.array(shape, dtype=np.float64)
    else:
        L = np.full(d, max(n, 8) ** (1.0 / d))
        coords = rng.uniform(0.0, 1.0, (d, n)) * L[:, None]
    if path in ("exponential", "matern52", "spherical"):
        st = [G.CovStructure(path, 1.3, L / 4)]
    elif path == "gauss_table":
        st = [G.CovStructure("gaussian", 1.0, L / 6)]
    else:
        st = _models(d, L)
    A0 = kernel_dense(st, coords)
    if nugget is None:
        nugget = max(1e-3, float(np.max(np.sum(np.abs(A0), axis=1))) / 2e3)
    A = A0 + nugget * np.eye(A0.shape[0])
    if path in ("exponential", "matern52", "spherical"):
        op = gsi.KernelCovMatrix(path, coords, L / 4, sigma2=1.3, nugget=nugget)
    elif path == "gauss_table":
        op = gsi.GridKernelCovMatrix("gaussian", shape, L / 6, nugget=nugget)
    elif path == "model_fused":
        op = gsi.KernelCovModelMatrix(st, coords, nugget)
    else:
        op = gsi.GridKernelCovModelMatrix(st, shape, nugget=nugget)
    return op, A, nugget


COVERAGE = [("exponential", 1, 1, 1), ("exponential", 2, 63, 3), ("exponential", 3, 1000, 8),
            ("exponential", 2, 5000, 64),
            ("matern52", 1, 64, 9), ("matern52", 2, 5000, 1), ("matern52", 3, 65, 64),
            ("spherical", 2, 1000, 300), ("spherical", 3, 63, 1), ("spherical", 1, 5000, 3),
            ("gauss_table", 1, 65, 8), ("gauss_table", 2, 1000, 3), ("gauss_table", 3, 5000, 9),
            ("model_fused", 1, 1000, 3), ("model_fused", 2, 1000, 64), ("model_fused", 3, 5000, 8),
            ("model_fused", 2, 64, 300),
            ("model_table", 2, 63, 9), ("model_table", 2, 1000, 1), ("model_table", 3, 5000, 3)]


def _check_solution(A, B, X, info, rtol, tag):
    bn = np.linalg.norm(B, axis=0)
    host = np.linalg.norm(B - A @ X, axis=0) / np.where(bn > 0, bn, 1.0)
    slack = 8 * np.sqrt(A.shape[0]) * U * np.linalg.norm(np.abs(A) @ np.abs(X), axis=0) / np.where(bn > 0, bn, 1.0)
    rel = info["relres"]
    assert np.all(rel <= rtol), (tag, rel.max())
    assert np.all(np.abs(rel - host) <= 0.05 * np.maximum(rel, host) + slack), (tag, rel, host)


def _poison(gsi, op, n, k):
    """A product of the solve's shape on an all-NaN X: the pooled scratch then holds NaN."""
    Xn = gsi.DeviceMatrix.from_host(op.ctx, np.full((n, k), np.nan))
    op.apply(Xn).free()
    Xn.free()


@pytest.mark.gpu
@pytest.mark.parametrize("path,d,n,k", COVERAGE)
def test_solve_coverage(gsi, path, d, n, k):
    op, A, nugget = build_case(gsi, path, d, n)
    assert kappa_bound(A, nugget) <= 1e6
    B = np.random.default_rng(n + k).standard_normal((n, k))
    _poison(gsi, op, n, k)
    X, info = gsi.cov_solve(op, B, rtol=RTOL, maxiter=4 * n)        # small n at kappa ~ 2e3 may need a few more than n
    _check_solution(A, B, X, info, RTOL, (path, d, n, k))
    assert np.all(info["iterations"] >= 1)


@pytest.mark.gpu
def test_solve_big_shape(gsi):
    """A size whose products have one full round and a stream-K tail, preconditioned and not."""
    from test_gpu_product_exact import big_ok, grid_shape, num_sms
    shape = grid_shape(2, "big")
    n = int(np.prod(shape))
    assert big_ok(n, num_sms())
    coords = oracle.grid_coords(shape) + np.random.default_rng(7).uniform(-0.3, 0.3, (2, n))
    L = np.array(shape, dtype=np.float64)
    st = [G.CovStructure("matern32", 1.0, L / 5)]
    A0 = kernel_dense(st, coords)
    nugget = float(np.max(np.sum(A0, axis=1))) / 2e3
    A = A0 + nugget * np.eye(n)
    assert kappa_bound(A, nugget) <= 1e6
    op = gsi.KernelCovModelMatrix(st, coords, nugget)
    B = np.random.default_rng(1).standard_normal((n, 3))
    _poison(gsi, op, n, 3)
    X0, i0 = gsi.cov_solve(op, B, rtol=RTOL)
    _check_solution(A, B, X0, i0, RTOL, "big r=0")
    X1, i1 = gsi.cov_solve(op, B, rtol=RTOL, rank=100, rng=2)
    _check_solution(A, B, X1, i1, RTOL, "big r=100")
    assert np.all(i1["iterations"] < i0["iterations"])


# ------------------------------------------------------------------ GPU: the preconditioner
@pytest.mark.gpu
@pytest.mark.parametrize("path,d,n,r", [("exponential", 2, 1000, 50), ("model_table", 2, 1000, 100),
                                        ("gauss_table", 3, 5000, 200)])
def test_nystrom_matches_host(gsi, path, d, n, r):
    op, A, nugget = build_case(gsi, path, d, n)
    rng = np.random.default_rng(r)
    B = rng.standard_normal((n, 3))
    Omega = rng.standard_normal((n, r))
    Uf, lam = nystrom_host(A, nugget, Omega)
    X, info = gsi.cov_solve(op, B, rtol=RTOL, Omega=Omega)
    _check_solution(A, B, X, info, RTOL, (path, r))
    assert np.max(np.abs(info["nystrom_eigenvalues"] - lam)) <= 1e-10 * lam[0]
    _, it_host = pcg_host(A, B, RTOL, n, Uf, lam, nugget)
    assert np.all(np.abs(info["iterations"] - it_host) <= 2), (info["iterations"], it_host)
    _, info0 = gsi.cov_solve(op, B, rtol=RTOL)
    assert np.all(info["iterations"] < info0["iterations"]), (info["iterations"], info0["iterations"])


# ------------------------------------------------------------------ GPU: behaviour
@pytest.mark.gpu
def test_bit_reproducible(gsi):
    op, A, _ = build_case(gsi, "model_fused", 2, 5000)
    B = np.random.default_rng(3).standard_normal((5000, 9))
    runs = [gsi.cov_solve(op, B, rtol=RTOL, rank=50, rng=4) for _ in range(2)]
    assert np.array_equal(runs[0][0], runs[1][0])
    assert np.array_equal(runs[0][1]["iterations"], runs[1][1]["iterations"])


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [0, 40])
def test_zero_and_uneven_columns(gsi, rank):
    """A zero column gives x = 0 after 0 iterations; a column in the span of three top eigenvectors of A stops well
    before a random one, and every column meets rtol."""
    op, A, nugget = build_case(gsi, "exponential", 2, 1000)
    rng = np.random.default_rng(8)
    easy = np.linalg.eigh(A)[1][:, -3:] @ np.array([1.0, 0.5, 0.25])
    B = np.column_stack([rng.standard_normal(1000), np.zeros(1000), easy, rng.standard_normal(1000)])
    X, info = gsi.cov_solve(op, B, rtol=RTOL, rank=rank, rng=5)
    assert np.all(X[:, 1] == 0.0) and info["iterations"][1] == 0 and info["relres"][1] == 0.0
    assert info["iterations"][2] < info["iterations"][0]
    _check_solution(A, B, X, info, RTOL, "uneven")


@pytest.mark.gpu
@pytest.mark.parametrize("drift", [None, "constant", "universal"])
def test_krige_matches_dense(gsi, drift):
    rng = np.random.default_rng(21)
    n, m = 2000, 5000
    S, T = rng.uniform(0, 50, (2, n)), rng.uniform(0, 50, (2, m))
    st = [G.CovStructure("spherical", 1.0, [15.0, 10.0], G.rotation_matrix(0.4)),
          G.CovStructure("exponential", 0.5, [5.0, 5.0])]
    nugget = 0.05
    y = np.sin(S[0] / 7) + 0.1 * rng.standard_normal(n)
    spec = (np.column_stack([np.ones(n), S.T / 50]), np.column_stack([np.ones(m), T.T / 50])) \
        if drift == "universal" else drift
    yhat, beta, w = gsi.krige(st, S, y, T, nugget=nugget, drift=spec, rtol=RTOL, rank=50, rng=6, return_weights=True)
    from test_gpu_kcov_model import model_dense
    C = kernel_dense(st, S, nugget)
    Cts = model_dense(st, np.concatenate([T, S], axis=1), rows=np.arange(m))[:, m:]
    F, FT = kriging.drift_matrices(spec, n, m)
    y2, b2, w2 = _kkt(C, F, y, Cts, FT)
    ev = np.linalg.eigvalsh(C)
    kap = ev[-1] / ev[0]
    assert kap <= 1e6
    assert np.linalg.norm(yhat - y2) <= 10 * kap * RTOL * np.linalg.norm(y2)
    if F.shape[1]:
        assert np.linalg.norm(beta - b2) <= 10 * kap * RTOL * np.linalg.norm(b2)


@pytest.mark.gpu
def test_no_convergence_fills_x(gsi):
    op, A, _ = build_case(gsi, "exponential", 2, 1000)
    B = np.random.default_rng(9).standard_normal((1000, 2))
    with pytest.raises(G.GsiError) as e:
        gsi.cov_solve(op, B, rtol=RTOL, maxiter=1)
    assert e.value.code == G._lib.ERR_NO_CONVERGENCE
    X, info = e.value.X, e.value.info
    assert np.all(info["iterations"] == 1)
    host = np.linalg.norm(B - A @ X, axis=0) / np.linalg.norm(B, axis=0)
    assert np.all(np.isfinite(X)) and np.allclose(info["relres"], host, rtol=1e-8)
    assert np.all(info["relres"] > RTOL)


@pytest.mark.gpu
def test_singular_gaussian_fails_cleanly(gsi):
    """Nugget 0 on a near-singular Gaussian case: NOT_POSDEF or NO_CONVERGENCE, never a fault; the context still works."""
    coords = oracle.grid_coords((30, 30)).astype(np.float64)
    op = gsi.KernelCovMatrix("gaussian", coords, [8.0, 8.0])
    B = np.random.default_rng(10).standard_normal((900, 2))
    for rank in (0, 200):
        with pytest.raises(G.GsiError) as e:
            gsi.cov_solve(op, B, rtol=RTOL, maxiter=20, rank=rank, rng=1)
        assert e.value.code in (G._lib.ERR_NOT_POSDEF, G._lib.ERR_NO_CONVERGENCE), e.value
    op2, A2, _ = build_case(gsi, "exponential", 2, 63)
    X, info = gsi.cov_solve(op2, B[:63], rtol=RTOL, maxiter=4 * 63)
    _check_solution(A2, B[:63], X, info, RTOL, "after failure")


def _solve_raw(gsi, op, B, Omega, rtol, maxiter, xrows, xcols, layout=G.LAYOUT_TALL):
    import ctypes as C
    ctx = op.ctx
    Bd = gsi.DeviceMatrix.from_host(ctx, B)
    Od = None if Omega is None else gsi.DeviceMatrix.from_host(ctx, Omega)
    Xd = gsi.DeviceMatrix(ctx, xrows, xcols, layout)
    k = B.shape[1]
    it, rel = np.zeros(k, dtype=np.int64), np.zeros(k)
    return ctx._lib.gsi_kernelcov_solve(op._h, Bd._h, None if Od is None else Od._h, rtol, maxiter, Xd._h,
                                        it.ctypes.data_as(C.POINTER(C.c_int64)), G.core._pd(rel), None)


@pytest.mark.gpu
def test_error_paths(gsi):
    L = G._lib
    coords = np.random.default_rng(0).uniform(0, 10, (2, 300))
    n = 300
    st = [G.CovStructure("exponential", 1.0, [2.0, 2.0])]
    op = gsi.KernelCovModelMatrix(st, coords, 0.1)
    B = np.ones((n, 2))
    others = [gsi.DenseMatrix(np.eye(n)), gsi.LowRankCovMatrix(np.random.default_rng(1).standard_normal((n, 5))),
              gsi.KernelCrossCovMatrix(st, coords, coords)]
    for o in others:
        assert _solve_raw(gsi, o, B, None, RTOL, 10, n, 2) == L.ERR_UNSUPPORTED
    assert _solve_raw(gsi, op, np.ones((n - 1, 2)), None, RTOL, 10, n, 2) == L.ERR_DIMENSION_MISMATCH   # B rows
    assert _solve_raw(gsi, op, B, None, RTOL, 10, n, 3) == L.ERR_DIMENSION_MISMATCH                    # X cols
    assert _solve_raw(gsi, op, B, None, RTOL, 10, n - 1, 2) == L.ERR_DIMENSION_MISMATCH                # X rows
    assert _solve_raw(gsi, op, B, None, RTOL, 10, n, 2, G.LAYOUT_COLMAJOR) == L.ERR_DIMENSION_MISMATCH  # X layout
    assert _solve_raw(gsi, op, B, np.ones((n - 1, 4)), RTOL, 10, n, 2) == L.ERR_DIMENSION_MISMATCH     # Omega rows
    assert _solve_raw(gsi, op, B, np.ones((n, 257)), RTOL, 10, n, 2) == L.ERR_INVALID_ARGUMENT         # r > 256
    small = gsi.KernelCovModelMatrix(st, coords[:, :20], 0.1)
    assert _solve_raw(gsi, small, np.ones((20, 1)), np.ones((20, 20)), RTOL, 10, 20, 1) == L.ERR_INVALID_ARGUMENT  # r >= n
    # r = 0: no device buffer has zero columns, so a zero-column sketch is refused when it is uploaded
    with pytest.raises(G.GsiError) as e:
        gsi.cov_solve(op, B, Omega=np.ones((n, 0)))
    assert e.value.code == L.ERR_INVALID_ARGUMENT
    Obad = np.random.default_rng(2).standard_normal((n, 20))                                          # Omega not finite
    for v in (np.nan, np.inf):
        Obad[5, 3] = v
        assert _solve_raw(gsi, op, B, Obad, RTOL, 10, n, 2) == L.ERR_INVALID_ARGUMENT
    for rtol in (0.0, -1.0, np.nan, np.inf):
        assert _solve_raw(gsi, op, B, None, rtol, 10, n, 2) == L.ERR_INVALID_ARGUMENT
    assert _solve_raw(gsi, op, B, None, RTOL, -1, n, 2) == L.ERR_INVALID_ARGUMENT
    Bbad = B.copy()
    Bbad[17, 1] = np.nan
    assert _solve_raw(gsi, op, Bbad, None, RTOL, 10, n, 2) == L.ERR_INVALID_ARGUMENT
    Bbad[17, 1] = np.inf
    assert _solve_raw(gsi, op, Bbad, None, RTOL, 10, n, 2) == L.ERR_INVALID_ARGUMENT
    X, info = gsi.cov_solve(op, B, rtol=RTOL)                                                          # still usable
    assert np.all(info["relres"] <= RTOL)


# ------------------------------------------------------------------ two ranks
DIST_N = 3001


def dist_case():
    rng = np.random.default_rng(12)
    coords = rng.uniform(0, 30, (2, DIST_N))
    st = [G.CovStructure("spherical", 1.0, [8.0, 6.0], G.rotation_matrix(0.3)),
          G.CovStructure("exponential", 0.5, [3.0, 3.0])]
    B = rng.standard_normal((DIST_N, 5))
    Omega = rng.standard_normal((DIST_N, 60))
    return st, coords, 0.02, B, Omega


@pytest.mark.gpu
def test_two_ranks(gsi):
    """Row-sharded solves (plain and preconditioned, X as this rank's rows and as all rows) match one rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "dist_cov_solve_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=540, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        st, coords, nugget, B, Omega = dist_case()
        op = gsi.KernelCovModelMatrix(st, coords, nugget)
        ref = {"plain": gsi.cov_solve(op, B, rtol=RTOL), "nys": gsi.cov_solve(op, B, rtol=RTOL, Omega=Omega)}
        for rank in range(2):
            f = np.load(os.path.join(tmp, f"solve_rank{rank}.npz"))
            r0, ml = G.partition_rows(DIST_N, 2, rank)
            for name, (X1, info1) in ref.items():
                Xl, Xa, it = f[f"{name}_local"], f[f"{name}_all"], f[f"{name}_iters"]
                assert Xl.shape == (ml, 5) and Xa.shape == (DIST_N, 5)
                assert np.linalg.norm(Xa - X1) <= 1e-10 * np.linalg.norm(X1), (rank, name)
                assert np.linalg.norm(Xl - X1[r0:r0 + ml]) <= 1e-10 * np.linalg.norm(X1), (rank, name)
                assert np.all(np.abs(it - info1["iterations"]) <= 1), (rank, name, it, info1["iterations"])
                assert np.all(f[f"{name}_relres"] <= RTOL)
