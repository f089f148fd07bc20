"""Direct kriging on a dense Cholesky factor (gsi_kernelcov_chol / gsi_b200.KernelCovCholesky / krige(method="cholesky")).

* The materialised covariance blocks equal the operator product on identity columns bit for bit, for every square path
  and the cross-covariance operators; the diagonal carries the nugget.
* The factor: ||A - L L'||_F / ||A||_F against the host-built A for every square path, d = 1..3 and n around the block
  width; at n = 20 000 through the matrix-free product.  Solves against scipy's cho_solve and the CG solve, logdet
  against slogdet, the kriging variance against the bordered (KKT) dense formula, krige against CG and the dense
  solution; failures, refusals, reproducibility and two ranks.
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
import gsi_b200 as G                                   # noqa: E402  (importing needs no GPU)
from gsi_b200 import kriging                           # noqa: E402

U = 2.0 ** -53
B_W = 128                                              # block width of the factorisation


def model_dense(structures, coords, rows=None, nugget=0.0):
    from test_gpu_kcov_model import model_dense as md
    return md(structures, coords, rows=rows, nugget=nugget)


def block(gsi, op, row0, col0, rows, cols):
    """C[row0:row0+rows, col0:col0+cols] through gsi_op_kernelcov_block."""
    out = gsi.DeviceMatrix(op.ctx, rows, cols, G.LAYOUT_COLMAJOR)
    try:
        G._lib.check(op.ctx._lib.gsi_op_kernelcov_block(op._h, row0, col0, out._h))
        return out.numpy()
    finally:
        out.free()


def identity_columns(n, col0, w):
    E = np.zeros((n, w))
    E[col0 + np.arange(w), np.arange(w)] = 1.0
    return E


def grid_shape(d, n):
    if n == 3000:
        return {1: (3000,), 2: (60, 50), 3: (15, 20, 10)}[d]
    return (n,) + (1,) * (d - 1)


def rotated_models(d, L):
    L = np.asarray(L, dtype=np.float64)
    if d == 1:
        return [G.CovStructure("spherical", 0.6, L / 3), G.CovStructure("exponential", 0.4, L / 5),
                G.CovStructure("matern32", 0.5, L / 4)]
    ang = (0.5,) if d == 2 else (0.5, -0.3, 0.8)
    R1, R2 = G.rotation_matrix(ang), G.rotation_matrix(tuple(-0.7 * a for a in ang))
    return [G.CovStructure("spherical", 0.6, L / 3, R1), G.CovStructure("exponential", 0.4, L / 5, R2),
            G.CovStructure("matern52", 0.3, L / 4, R1)]


def square_case(gsi, path, d, n, nugget=None):
    """(operator, host-built dense A, nugget) of one square path; the nugget keeps kappa(A) below about 2e3 * n."""
    rng = np.random.default_rng(1000 * d + n)
    if path in ("gauss_table", "model_table"):
        shape = grid_shape(d, n)
        coords = oracle.grid_coords(shape)
        L = np.maximum(np.array(shape, dtype=np.float64), 4.0)
    else:
        L = np.full(d, max(n, 8) ** (1.0 / d))
        coords = rng.uniform(0.0, 1.0, (d, n)) * L[:, None]
    if path in ("exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"):
        st = [G.CovStructure(path, 1.3, L / 4, beta=0.7)]
    elif path == "gauss_table":
        st = [G.CovStructure("gaussian", 1.0, L / 6)]
    else:
        st = rotated_models(d, L)
    A0 = model_dense(st, coords)
    if nugget is None:
        nugget = max(1e-3, float(np.max(np.sum(np.abs(A0), axis=1))) / 2e3)
    A = A0 + nugget * np.eye(n)
    if path in ("exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"):
        op = gsi.KernelCovMatrix(path, coords, L / 4, sigma2=1.3, nugget=nugget, beta=0.7)
    elif path == "gauss_table":
        op = gsi.GridKernelCovMatrix("gaussian", shape, L / 6, nugget=nugget)
    elif path == "model_fused":
        op = gsi.KernelCovModelMatrix(st, coords, nugget)
    else:
        op = gsi.GridKernelCovModelMatrix(st, shape, nugget=nugget)
    return op, A, nugget


KINDS = ["exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"]


# ------------------------------------------------------------------ materialisation
@pytest.mark.gpu
@pytest.mark.parametrize("path", KINDS + ["model_fused", "gauss_table", "model_table"])
@pytest.mark.parametrize("d", [1, 2, 3])
def test_block_equals_product_bitwise(gsi, path, d):
    n = 300 if path not in ("gauss_table", "model_table") else 3000
    op, A, nugget = square_case(gsi, path, d, n)
    for col0, w in ((0, 1), (37, 70), (n - 9, 9)):
        P = op.apply(identity_columns(n, col0, w))
        Bk = block(gsi, op, 0, col0, n, w)
        assert np.array_equal(Bk, P), (path, d, col0, np.max(np.abs(Bk - P)))
    # the diagonal carries the nugget; the block agrees with the host-built matrix to rounding
    D = block(gsi, op, 5, 5, 40, 40)
    assert np.allclose(np.diag(D), np.diag(A)[5:45], rtol=1e-13, atol=0)
    assert np.allclose(D, A[5:45, 5:45], rtol=1e-12, atol=1e-14)
    assert nugget >= 1e-3 * np.min(np.diag(A))          # so rtol 1e-13 on the diagonal would see a missing nugget


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [False, True])
def test_cross_block_equals_product_bitwise(gsi, grid):
    rng = np.random.default_rng(5)
    if grid:
        shape = (40, 30)
        ti, si = rng.choice(1200, 333, replace=False), rng.choice(1200, 211, replace=False)
        st = rotated_models(2, shape)
        op = gsi.GridKernelCrossCovMatrix(st, shape, targets=ti, sources=si)
    else:
        T, S = rng.uniform(0, 30, (3, 333)), rng.uniform(0, 30, (3, 211))
        st = rotated_models(3, [30.0, 30.0, 30.0])
        op = gsi.KernelCrossCovMatrix(st, T, S)
    m, n = op.shape
    P = op.apply(identity_columns(n, 17, 150))
    assert np.array_equal(block(gsi, op, 0, 17, m, 150), P)
    assert np.array_equal(block(gsi, op, 100, 17, 50, 150), P[100:150])


# ------------------------------------------------------------------ factor
SQUARE_PATHS = ["exponential", "matern52", "spherical", "gauss_table", "model_fused", "model_table"]
# c of the bound ||A - L L'||_F <= c n u ||A||_F.  The Cholesky backward error is |A - L L'| <= gamma_(n+1) |L| |L'|
# (Higham, Accuracy and Stability, Thm 10.3); the panels here use the explicit inverse of the 128 x 128 diagonal blocks,
# whose error is bounded by kappa(L11) times that (Du Croz and Higham 1992), and kappa(L11) <= sqrt(kappa(A)) <= 50 for
# these nuggets.  Rounding errors of the length-n dot products add up like sqrt(n) in practice, and || |L||L'| ||_F is
# ||A||_F for these matrices (nonnegative, diagonally heavy): c = 4 leaves a wide margin over what is observed.
C_FACTOR = 4.0


@pytest.mark.gpu
@pytest.mark.parametrize("path", SQUARE_PATHS)
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 2, B_W - 1, B_W, B_W + 1, 3 * B_W + 17, 3000])
def test_factor_residual(gsi, path, d, n):
    op, A, _ = square_case(gsi, path, d, n)
    f = gsi.KernelCovCholesky(op)
    try:
        L = f.L
        assert f.n == n and np.all(np.triu(L, 1) == 0.0) and np.all(np.diag(L) > 0)
        err = np.linalg.norm(A - L @ L.T) / np.linalg.norm(A)
        assert err <= C_FACTOR * n * U, (path, d, n, err / (n * U))
    finally:
        f.free()


@pytest.mark.gpu
def test_factor_big_matrix_free_residual(gsi):
    """n = 20 000 scattered points: ||A v - L (L' v)|| / (||A|| ||v||) through the matrix-free product (||A|| bounded below
    by ||A v|| / ||v||, which makes the ratio an upper bound)."""
    n = 20000
    rng = np.random.default_rng(20)
    coords = rng.uniform(0, 100, (2, n))
    op = gsi.KernelCovMatrix("exponential", coords, [10.0, 10.0], nugget=0.05)
    f = gsi.KernelCovCholesky(op)
    try:
        V = rng.standard_normal((n, 3))
        AV = op.apply(V)
        L = f.L
        LLV = L @ (L.T @ V)
        del L
        for j in range(3):
            nrm_a = np.linalg.norm(AV[:, j]) / np.linalg.norm(V[:, j])
            err = np.linalg.norm(AV[:, j] - LLV[:, j]) / (nrm_a * np.linalg.norm(V[:, j]))
            assert err <= n * U, (j, err)
    finally:
        f.free()


# ------------------------------------------------------------------ solve / logdet
def kappa_bound(A, nugget):
    return float(np.max(np.sum(np.abs(A), axis=1)) / nugget)


@pytest.mark.gpu
@pytest.mark.parametrize("path,d,n", [("exponential", 2, 3000), ("model_table", 2, 3000), ("matern52", 3, 401),
                                      ("model_fused", 1, 129)])
@pytest.mark.parametrize("k", [1, 7, 1024, 1500])
def test_solve(gsi, path, d, n, k):
    op, A, nugget = square_case(gsi, path, d, n)
    kap = kappa_bound(A, nugget)
    B = np.random.default_rng(k).standard_normal((n, k))
    f = gsi.KernelCovCholesky(op)
    try:
        X = f.solve(B)
        ref = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), B)
        # forward error <= kappa x backward error, the backward error bounded as in test_factor_residual
        err = np.linalg.norm(X - ref, axis=0) / np.linalg.norm(ref, axis=0)
        assert np.all(err <= kap * C_FACTOR * n * U), (err.max(), kap)
        Y = f.solve_lower(B)                                # the half solve by its residual
        L = f.L
        res = np.linalg.norm(L @ Y - B, axis=0) / (np.linalg.norm(L, 2) * np.linalg.norm(Y, axis=0))
        assert np.all(res <= n * U), res.max()
        if k == 7:
            Xcg, info = gsi.cov_solve(op, B, rtol=1e-10, maxiter=4 * n)
            assert np.linalg.norm(X - Xcg) <= 10 * kap * 1e-10 * np.linalg.norm(X)
            ld = f.logdet
            s, ref_ld = np.linalg.slogdet(A)
            assert s > 0 and abs(ld - ref_ld) <= 1e-9 * n, (ld, ref_ld)
    finally:
        f.free()


# ------------------------------------------------------------------ variance
def kkt_variance(C, F, Cts, FT, ctt):
    n, p = F.shape
    K = np.block([[C, F], [F.T, np.zeros((p, p))]])
    R = np.vstack([Cts.T, FT.T])
    return ctt - np.sum(R * np.linalg.solve(K, R), axis=0)


def variance_case(gsi, m, nugget=0.05, seed=31):
    rng = np.random.default_rng(seed)
    n = 1500
    S, T = rng.uniform(0, 40, (2, n)), rng.uniform(0, 40, (2, m))
    st = [G.CovStructure("spherical", 1.0, [15.0, 10.0], G.rotation_matrix(0.4)),
          G.CovStructure("exponential", 0.5, [5.0, 5.0])]
    return st, S, T, nugget


@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 1023, 1024, 1025])
@pytest.mark.parametrize("drift", [None, "constant", "universal"])
def test_variance_matches_kkt(gsi, m, drift):
    st, S, T, nugget = variance_case(gsi, m)
    n = S.shape[1]
    op = gsi.KernelCovModelMatrix(st, S, nugget)
    cross = gsi.KernelCrossCovMatrix(st, T, S, ctx=op.ctx)
    spec = (np.column_stack([np.ones(n), S.T / 40]), np.column_stack([np.ones(m), T.T / 40])) \
        if drift == "universal" else drift
    F, FT = kriging.drift_matrices(spec, n, m)
    f = gsi.KernelCovCholesky(op)
    try:
        var = f.variance(cross, spec)
    finally:
        f.free()
    C = model_dense(st, S, nugget=nugget)
    Cts = model_dense(st, np.concatenate([T, S], axis=1), rows=np.arange(m))[:, m:]
    ref = kkt_variance(C, F, Cts, FT, 1.5)
    kap = np.linalg.cond(C)
    assert np.max(np.abs(var - ref)) <= 10 * kap * np.sqrt(n) * U * 1.5, (np.max(np.abs(var - ref)), kap)
    assert np.all(var > 0)


@pytest.mark.gpu
def test_variance_special_targets(gsi):
    """Zero nugget: a target that is a source has variance about 0; a target beyond every range has the total sill
    (simple kriging); targets on the nodes of a grid (the cross-grid operator) match the dense formula."""
    st, S, _, _ = variance_case(gsi, 1)
    S = S[:, :800]
    n = S.shape[1]
    st0 = [G.CovStructure("spherical", 1.0, [15.0, 10.0], G.rotation_matrix(0.4)),
           G.CovStructure("exponential", 0.5, [5.0, 5.0])]
    op = gsi.KernelCovModelMatrix(st0, S, 0.0)
    T = np.column_stack([S[:, 3], S[:, 500], [1e4, 1e4]])
    cross = gsi.KernelCrossCovMatrix(st0, T, S, ctx=op.ctx)
    f = gsi.KernelCovCholesky(op)
    try:
        var = f.variance(cross)
    finally:
        f.free()
    assert abs(var[0]) <= 1e-7 and abs(var[1]) <= 1e-7, var
    assert var[2] == 1.5
    # grid nodes: sources and targets of one 50 x 40 grid
    shape = (50, 40)
    rng = np.random.default_rng(4)
    si, ti = rng.choice(2000, 700, replace=False), rng.choice(2000, 1100, replace=False)
    stg = rotated_models(2, shape)
    opg = gsi.KernelCovModelMatrix(stg, oracle.grid_coords(shape)[:, si], 0.01)
    cg = gsi.GridKernelCrossCovMatrix(stg, shape, targets=ti, sources=si)
    f = gsi.KernelCovCholesky(opg)
    try:
        var = f.variance(cg, "constant")
    finally:
        f.free()
    X = oracle.grid_coords(shape)
    C = model_dense(stg, X[:, si], nugget=0.01)
    Cts = model_dense(stg, np.concatenate([X[:, ti], X[:, si]], axis=1), rows=np.arange(ti.size))[:, ti.size:]
    ref = kkt_variance(C, np.ones((si.size, 1)), Cts, np.ones((ti.size, 1)), sum(s.sill for s in stg))
    assert np.max(np.abs(var - ref)) <= 1e-9, np.max(np.abs(var - ref))


@pytest.mark.gpu
@pytest.mark.parametrize("drift", [None, "constant", "universal"])
def test_krige_cholesky_matches_cg_and_dense(gsi, drift):
    rng = np.random.default_rng(21)
    n, m = 2000, 5000
    S, T = rng.uniform(0, 50, (2, n)), rng.uniform(0, 50, (2, m))
    st = [G.CovStructure("spherical", 1.0, [15.0, 10.0], G.rotation_matrix(0.4)),
          G.CovStructure("exponential", 0.5, [5.0, 5.0])]
    nugget = 0.05
    y = np.sin(S[0] / 7) + 0.1 * rng.standard_normal(n)
    spec = (np.column_stack([np.ones(n), S.T / 50]), np.column_stack([np.ones(m), T.T / 50])) \
        if drift == "universal" else drift
    yc, bc, wc, var = gsi.krige(st, S, y, T, nugget=nugget, drift=spec, method="cholesky", return_weights=True,
                                return_variance=True)
    yg = gsi.krige(st, S, y, T, nugget=nugget, drift=spec, rtol=1e-10, rank=50, rng=6)
    C = model_dense(st, S, nugget=nugget)
    Cts = model_dense(st, np.concatenate([T, S], axis=1), rows=np.arange(m))[:, m:]
    F, FT = kriging.drift_matrices(spec, n, m)
    p = F.shape[1]
    K = np.block([[C, F], [F.T, np.zeros((p, p))]])
    sol = np.linalg.solve(K, np.concatenate([y, np.zeros(p)]))
    y2 = Cts @ sol[:n] + FT @ sol[n:]
    kap = np.linalg.cond(C)
    assert np.linalg.norm(yc - y2) <= 10 * kap * np.sqrt(n) * U * np.linalg.norm(y2)
    assert np.linalg.norm(yc - yg) <= 10 * kap * 1e-10 * np.linalg.norm(y2)
    assert var.shape == (m,) and np.all(var > 0)
    assert np.max(np.abs(var - kkt_variance(C, F, Cts, FT, 1.5))) <= 1e-9
    assert gsi.krige(st, S, y, T, nugget=nugget, drift=spec, method="cholesky").shape == (m,)
    with pytest.raises(ValueError, match="one iterative solve per target"):
        gsi.krige(st, S, y, T, nugget=nugget, drift=spec, return_variance=True)


# ------------------------------------------------------------------ failures, refusals, reproducibility
def _chol_raw(op):
    h, col = C.c_void_p(), C.c_int64(-1)
    status = op.ctx._lib.gsi_kernelcov_chol(op._h, C.byref(h), C.byref(col))
    if h:
        op.ctx._lib.gsi_chol_free(h)
    return status, int(col.value), bool(h)


@pytest.mark.gpu
def test_singular_gaussian_raises_posdef(gsi):
    """The near-singular Gaussian case of the CG tests (nugget 0): PosDefException with the failing column; the failure
    path frees what it allocated and the context factors the next operator."""
    coords = oracle.grid_coords((30, 30)).astype(np.float64)
    op = gsi.KernelCovMatrix("gaussian", coords, [8.0, 8.0])
    with pytest.raises(G.PosDefException) as e:
        gsi.KernelCovCholesky(op)
    assert 1 <= e.value.column <= 900 and str(e.value.column) in e.value.message
    status, col, made = _chol_raw(op)
    assert status == G._lib.ERR_NOT_POSDEF and col == e.value.column and not made
    op2, A2, _ = square_case(gsi, "exponential", 2, 3 * B_W + 17)
    f = gsi.KernelCovCholesky(op2)
    L = f.L
    f.free()
    assert np.linalg.norm(A2 - L @ L.T) <= C_FACTOR * A2.shape[0] * U * np.linalg.norm(A2)


@pytest.mark.gpu
def test_refusals(gsi):
    L = G._lib
    big = gsi.GridKernelCovMatrix("exponential", (1000, 1000), [50.0, 50.0], nugget=0.1)
    with pytest.raises(G.GsiError) as e:
        gsi.KernelCovCholesky(big)
    assert e.value.code == L.ERR_UNSUPPORTED and "bytes" in e.value.message
    n = 300
    coords = np.random.default_rng(0).uniform(0, 10, (2, n))
    st = [G.CovStructure("exponential", 1.0, [2.0, 2.0])]
    for o in (gsi.DenseMatrix(np.eye(n)), gsi.LowRankCovMatrix(np.random.default_rng(1).standard_normal((n, 5))),
              gsi.KernelCrossCovMatrix(st, coords, coords)):
        assert _chol_raw(o)[0] == L.ERR_UNSUPPORTED
    op = gsi.KernelCovModelMatrix(st, coords, 0.1)
    f = gsi.KernelCovCholesky(op)
    try:
        lib = op.ctx._lib

        def raw_solve(B, xrows, xcols, half=0, layout=G.LAYOUT_TALL):
            Bd = gsi.DeviceMatrix.from_host(op.ctx, B)
            Xd = gsi.DeviceMatrix(op.ctx, xrows, xcols, layout)
            try:
                return lib.gsi_chol_solve(f._h, half, Bd._h, Xd._h)
            finally:
                Bd.free()
                Xd.free()
        B = np.ones((n, 2))
        assert raw_solve(np.ones((n - 1, 2)), n, 2) == L.ERR_DIMENSION_MISMATCH
        assert raw_solve(B, n, 3) == L.ERR_DIMENSION_MISMATCH
        assert raw_solve(B, n, 2, layout=G.LAYOUT_COLMAJOR) == L.ERR_DIMENSION_MISMATCH
        assert raw_solve(B, n, 2, half=2) == L.ERR_INVALID_ARGUMENT
        for v in (np.nan, np.inf):
            Bb = B.copy()
            Bb[17, 1] = v
            assert raw_solve(Bb, n, 2) == L.ERR_INVALID_ARGUMENT
        other = gsi.KernelCrossCovMatrix(st, coords[:, :50], coords[:, :299], ctx=op.ctx)
        var = np.empty(50)
        assert lib.gsi_chol_krige_variance(f._h, other._h, None, None, 0, G.core._pd(var)) == L.ERR_DIMENSION_MISMATCH
        assert lib.gsi_chol_krige_variance(f._h, op._h, None, None, 0, G.core._pd(var)) == L.ERR_INVALID_ARGUMENT
        assert np.all(np.isfinite(f.solve(B)))                                      # still usable
    finally:
        f.free()
    assert lib.gsi_chol_free(None) == L.OK


@pytest.mark.gpu
def test_bit_reproducible(gsi):
    op, _, _ = square_case(gsi, "model_fused", 2, 3000)
    B = np.random.default_rng(3).standard_normal((3000, 9))
    runs = []
    for _ in range(2):
        f = gsi.KernelCovCholesky(op)
        runs.append((f.L, f.solve(B), f.logdet))
        f.free()
    assert np.array_equal(runs[0][0], runs[1][0])
    assert np.array_equal(runs[0][1], runs[1][1])
    assert runs[0][2] == runs[1][2]


@pytest.mark.gpu
def test_two_ranks_unsupported(gsi):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29551", os.path.join(ROOT, "tests", "dist_kcov_chol_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        for rank in range(2):
            status, made, _ = open(os.path.join(tmp, f"chol_rank{rank}.txt")).read().split()
            assert int(status) == G._lib.ERR_UNSUPPORTED and made == "0"


def test_cholesky_exports():
    assert G.KernelCovCholesky is kriging.KernelCovCholesky
    for name in ("gsi_kernelcov_chol", "gsi_chol_solve", "gsi_chol_logdet", "gsi_chol_krige_variance",
                 "gsi_op_kernelcov_block"):
        assert name in G._lib.SIGNATURES


def test_krige_rejects_variance_on_cg():
    with pytest.raises(ValueError, match="method='cholesky'"):
        G.krige([], np.zeros((2, 1)), [0.0], np.zeros((2, 1)), return_variance=True)
    with pytest.raises(ValueError, match="unknown method"):
        G.krige([], np.zeros((2, 1)), [0.0], np.zeros((2, 1)), method="lu")
