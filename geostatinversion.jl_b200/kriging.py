"""Kriging on the kernel-covariance operator: the solve A X = B by preconditioned CG on the matrix-free operator
(gsi_kernelcov_solve; the n x n covariance matrix is never formed, a solve costs one operator product of width k per
iteration) or on a dense Cholesky factor (KernelCovCholesky, gsi_kernelcov_chol: n^3 / 3 flops once, then any number of
solves, the kriging variance and log det A), and simple / ordinary / universal kriging in dual form on top of either;
conditional and unconditional Gaussian simulation on the dense factor of the joint source-target covariance
(simulate, gsi_chol_simulate); the ML / REML log-likelihood of the covariance parameters with its exact gradient
(loglik, gsi_kernelcov_loglik) and maximum-likelihood fitting of a nested model on it (fit_covariance); leave-one-out
and leave-group-out cross-validation on the dense factor (KernelCovCholesky.crossval, cross_validate, gsi_chol_crossval)."""
import ctypes as C
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import check, LAYOUT_TALL
from .core import (CovStructure, DeviceMatrix, KernelCovModelMatrix, KernelCrossCovMatrix, _f64_colmajor, _pd,
                   as_operator)
from .randmatfact import _rng


def cov_solve(A, B, *, rtol=1e-10, maxiter=None, rank=0, Omega=None, rng=None, full=False):
    """X = A^-1 B for a square kernel-covariance operator A (KernelCovMatrix, GridKernelCovMatrix, KernelCovModelMatrix
    or GridKernelCovModelMatrix; A exactly as built, nugget included).  B: n or n x k (k <= 1024).

    The k columns run independent preconditioned CG recurrences that share one operator product per iteration; column
    j stops when ||r_j|| <= rtol ||b_j||.  rank > 0 draws an n x rank Gaussian sketch from `rng` (or pass `Omega`) for
    the randomized Nystrom preconditioner (1 <= rank <= 256, rank < n).  maxiter=None means n.  On a multi-rank context
    each rank gets its own row block of X unless full=True.

    Returns (X, info) with info["iterations"] (per column), info["relres"] (the true ||b - A x|| / ||b|| of the returned
    X) and info["nystrom_eigenvalues"].  A column that does not converge raises GsiError (ERR_NO_CONVERGENCE) carrying
    the same X and info as attributes; p'Ap <= 0 or a failed preconditioner raises PosDefException."""
    op = as_operator(A)
    ctx = op.ctx
    n = op.shape[1]
    Bh = np.asarray(B, dtype=np.float64)
    vector = Bh.ndim == 1
    Bh = Bh.reshape(n, -1) if vector else Bh
    if Bh.shape[0] != n:
        raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH, f"cov_solve: B has {Bh.shape[0]} rows, A is {n} x {n}")
    k = Bh.shape[1]
    if Omega is None and rank > 0:
        Omega = _rng(rng).standard_normal((n, int(rank)))
    r = 0 if Omega is None else np.shape(Omega)[1]
    maxiter = n if maxiter is None else int(maxiter)
    xrows = op.mloc if (ctx.world > 1 and not full) else n
    iters = np.zeros(k, dtype=np.int64)
    relres = np.zeros(k, dtype=np.float64)
    lam = np.zeros(max(r, 1), dtype=np.float64)
    Bd = DeviceMatrix.from_host(ctx, Bh)
    Om = None
    Xd = None
    try:
        if Omega is not None:
            Om = Omega if isinstance(Omega, DeviceMatrix) else DeviceMatrix.from_host(ctx, Omega)
        Xd = DeviceMatrix(ctx, xrows, k, LAYOUT_TALL)
        status = ctx._lib.gsi_kernelcov_solve(op._h, Bd._h, None if Om is None else Om._h, float(rtol), maxiter, Xd._h,
                                              iters.ctypes.data_as(C.POINTER(C.c_int64)), _pd(relres), _pd(lam))
        X = Xd.numpy() if status in (_lib.OK, _lib.ERR_NO_CONVERGENCE) else None
    finally:
        Bd.free()
        if Om is not None and Om is not Omega:
            Om.free()
        if Xd is not None:
            Xd.free()
    info = {"iterations": iters, "relres": relres, "nystrom_eigenvalues": lam[:r]}
    if X is not None and vector:
        X = X[:, 0]
    try:
        check(status)
    except _lib.GsiError as e:
        e.X, e.info = X, info
        raise
    return X, info


def drift_matrices(drift, n, m):
    """(F_sources n x p, F_targets m x p) of a drift specification: None (p = 0), "constant" or a pair of arrays."""
    if drift is None:
        return np.zeros((n, 0)), np.zeros((m, 0))
    if isinstance(drift, str):
        if drift != "constant":
            raise ValueError(f"krige: unknown drift {drift!r} (None, 'constant' or (F_sources, F_targets))")
        return np.ones((n, 1)), np.ones((m, 1))
    Fs, Ft = (np.asarray(f, dtype=np.float64) for f in drift)
    Fs, Ft = Fs.reshape(n, -1), Ft.reshape(m, -1)
    if Fs.shape[1] != Ft.shape[1]:
        raise ValueError(f"krige: drift has {Fs.shape[1]} columns at the sources and {Ft.shape[1]} at the targets")
    return Fs, Ft


def dual_kriging(solve, cross, y, F, FT):
    """Dual-form kriging given solve(R) = C^-1 R and cross(w) = C(T, S) w: one solve C [alpha | B_F] = [y | F], then
    beta = (F' B_F)^-1 F' alpha (p x p), w = alpha - B_F beta and yhat = F_T beta + C(T, S) w.  This is the solution
    of the bordered system [C F; F' 0] [w; beta] = [y; 0]; p = 0 is simple kriging."""
    p = F.shape[1]
    Xs = solve(np.column_stack([y, F]))
    alpha, BF = Xs[:, 0], Xs[:, 1:]
    if p:
        beta = np.linalg.solve(F.T @ BF, F.T @ alpha)
        w = alpha - BF @ beta
    else:
        beta = np.zeros(0)
        w = alpha
    return FT @ beta + cross(w), beta, w


def krige(structures, sources, y, targets, *, nugget=0.0, drift=None, rtol=1e-10, rank=0, rng=None,
          return_weights=False, method="cg", return_variance=False):
    """Kriging estimate at the targets (d x m) from observations y at the sources (d x n) under the nested covariance
    model `structures` (CovStructure list) plus `nugget` on the observations, in dual form.

    drift=None: simple kriging (known zero mean); "constant": ordinary kriging; (F_sources n x p, F_targets m x p):
    universal kriging / kriging with external drift.  method="cg": the n x (1 + p) right-hand side is one matrix-free
    cov_solve (rank > 0: with a Nystrom preconditioner of that rank; rtol, rank and rng apply to it).  method="cholesky":
    one dense factorisation (KernelCovCholesky; about 8 n^2 bytes of device memory) whose solve replaces cov_solve.
    Returns yhat (m), or (yhat, beta, w) with return_weights=True; return_variance=True appends the kriging variance of
    the noise-free value at every target (KernelCovCholesky.variance; method="cholesky" only)."""
    if method not in ("cg", "cholesky"):
        raise ValueError(f"krige: unknown method {method!r} ('cg' or 'cholesky')")
    if return_variance and method == "cg":
        raise ValueError("krige: return_variance needs method='cholesky' -- on the CG path the variance costs one "
                         "iterative solve per target")
    S, T = _f64_colmajor(sources), _f64_colmajor(targets)
    n, m = S.shape[1], T.shape[1]
    y = np.asarray(y, dtype=np.float64).reshape(n)
    F, FT = drift_matrices(drift, n, m)
    C_ss = KernelCovModelMatrix(structures, S, nugget)
    C_ts = KernelCrossCovMatrix(structures, T, S, ctx=C_ss.ctx)
    fac = None
    var = None
    try:
        cross = lambda w: C_ts.apply(w.reshape(n, 1))[:, 0]          # noqa: E731
        if method == "cg":
            yhat, beta, w = dual_kriging(lambda R: cov_solve(C_ss, R, rtol=rtol, rank=rank, rng=rng)[0], cross, y, F, FT)
        else:
            fac = KernelCovCholesky(C_ss)
            yhat, beta, w = dual_kriging(fac.solve, cross, y, F, FT)
            if return_variance:
                var = fac.variance(C_ts, (F, FT) if F.shape[1] else None)
    finally:
        if fac is not None:
            fac.free()
        C_ss.free()
        C_ts.free()
    out = (yhat, beta, w) if return_weights else (yhat,)
    if return_variance:
        out = out + (var,)
    return out if len(out) > 1 else out[0]


def simulate(structures, targets, nreal, *, sources=None, y=None, nugget=0.0, target_nugget=0.0, drift=None, rng=None,
             Xi=None):
    """nreal Gaussian realisations (m x nreal) at the targets (d x m) under the nested covariance model `structures`,
    conditioned on observations y at the sources (d x ns, observation noise `nugget`) or unconditional (sources=None).

    LU simulation on one dense factor of the joint matrix C([S T], [S T]) + diag(nugget at the sources, target_nugget at
    the targets) (KernelCovCholesky.simulate; about 8 (ns + m)^2 bytes of device memory).  target_nugget = 0 simulates
    the noise-free field that krige estimates; a small target_nugget > 0 is the jitter smooth kernels need when targets
    lie close together.  drift: None (simple kriging, known zero mean), "constant" or (F_sources ns x p, F_targets m x p)
    as in krige; conditional simulation only.  The standard normals are drawn on the host from `rng`, 1024 columns at a
    time; pass Xi ((ns + m) x nreal) to make a run exact."""
    T = _f64_colmajor(targets)
    m = T.shape[1]
    if sources is None:
        if drift is not None:
            raise ValueError("simulate: a drift needs conditioning data (sources and y)")
        S = np.zeros((T.shape[0], 0))
    else:
        S = _f64_colmajor(sources)
    ns = S.shape[1]
    nreal = int(nreal)
    if Xi is None:
        g = _rng(rng)
        Xi = np.empty((ns + m, nreal), dtype=np.float64, order="F")
        for c0 in range(0, nreal, 1024):
            Xi[:, c0:c0 + 1024] = g.standard_normal((ns + m, min(1024, nreal - c0)))
    elif np.shape(Xi) != (ns + m, nreal):
        raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                     f"simulate: Xi has shape {np.shape(Xi)}, expected {(ns + m, nreal)}")
    P = np.concatenate([S, T], axis=1)
    d = np.concatenate([np.full(ns, float(nugget)), np.full(m, float(target_nugget))])
    A = KernelCovModelMatrix(structures, P, 0.0)
    fac = None
    try:
        fac = KernelCovCholesky(A, diag=d)
        return fac.simulate(Xi, n_cond=ns, y=None if ns == 0 else y, drift=drift)
    finally:
        if fac is not None:
            fac.free()
        A.free()


def _drift_columns(drift, n):
    """F (n x p, column-major) of a drift specification: None (p = 0), "constant" or an n x p array."""
    if drift is None:
        return np.zeros((n, 0), order="F")
    if isinstance(drift, str):
        if drift != "constant":
            raise ValueError(f"unknown drift {drift!r} (None, 'constant' or an n x p array)")
        return np.ones((n, 1), order="F")
    return np.asfortranarray(np.asarray(drift, dtype=np.float64).reshape(n, -1))


def loglik(A, y, *, drift=None, reml=False, grad=False):
    """Gaussian log-likelihood of the observations y under the square kernel-covariance operator A (KernelCovMatrix,
    GridKernelCovMatrix, KernelCovModelMatrix or GridKernelCovModelMatrix, nugget included), the drift coefficients
    profiled out by GLS (gsi_kernelcov_loglik; one dense factorisation, about 8 n^2 bytes, single GPU).

    drift: None (known zero mean), "constant" or an n x p array F (p <= 32).  reml=False: ML,
    -1/2 (n log 2 pi + log det A + q); reml=True: REML, -1/2 ((n - p) log 2 pi + log det A + log det F'A^-1F + q) without
    the constant log det F'F (so the value depends on the scaling of F, the maximiser does not); q is the GLS residual
    (y - F beta)' A^-1 (y - F beta).

    Returns (value, beta), or (value, beta, gradient) with grad=True: d value / d theta for, per structure, the sill and
    then the d principal-axis ranges, and last the nugget (nstruct (1 + d) + 1 entries; rotations and power-law
    exponents are held fixed).  The gradient is not available on grid operators (pass the nodes' coordinates instead).
    A matrix that is not positive definite raises PosDefException with the 1-based failing column in `.column`."""
    op = as_operator(A)
    n = op.shape[1]
    yh = np.ascontiguousarray(y, dtype=np.float64).reshape(-1)
    if yh.size != n:
        raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH, f"loglik: y has {yh.size} values, A is {n} x {n}")
    F = _drift_columns(drift, n)
    p = F.shape[1]
    val = C.c_double(0.0)
    col = C.c_int64(0)
    beta = np.zeros(max(p, 1))
    g = np.zeros(op.nstruct * (1 + op.dim) + 1) if grad else None
    status = op.ctx._lib.gsi_kernelcov_loglik(op._h, _pd(yh), _pd(F) if p else None, p, 1 if reml else 0, C.byref(val),
                                              _pd(beta), None if g is None else _pd(g), C.byref(col))
    try:
        check(status)
    except _lib.PosDefException as e:
        e.column = int(col.value)
        raise
    out = (float(val.value), beta[:p])
    return out + (g,) if grad else out


# L-BFGS-B stopping rule of fit_covariance: a relative change of the likelihood below 1e-13 or a projected log-parameter
# gradient below 1e-5 (the default ftol of 2.2e-9 stops far from the optimum on likelihoods of n ~ 1e3 .. 1e4)
FIT_OPTIONS = {"ftol": 1e-13, "gtol": 1e-5}


def fit_covariance(structures, sources, y, *, nugget, drift=None, reml=True, fit_nugget=True, isotropic=False,
                   bounds=None, maxiter=200):
    """Maximum-likelihood fit of the sills and ranges of a nested covariance model (and of the nugget) to observations y
    at the sources (d x n), by L-BFGS-B on the logarithms of the parameters with the exact gradient of loglik (one
    factorisation plus about 2 n^3 / 3 flops of sweeps per evaluation).

    structures: the starting CovStructure list; rotations and power-law exponents are held at their values.  nugget:
    the starting nugget (> 0 when fitted), held fixed with fit_nugget=False.  isotropic=True ties the ranges of each
    structure to one parameter.  drift, reml: as in loglik (REML by default).  bounds: None or one (low, high) pair per
    fitted parameter in natural units, in the order sill, ranges (one with isotropic=True) per structure, then the
    nugget; None inside a pair leaves that side open.

    Returns (structures, nugget, info): the fitted CovStructure list, the nugget, and info with "loglik", "beta",
    "grad" (the natural-parameter gradient of loglik at the result), "nit", "nfev", "success" and "message"."""
    from scipy.optimize import minimize               # scipy is needed here only

    S = _f64_colmajor(sources)
    d = S.shape[0]
    yh = np.asarray(y, dtype=np.float64).reshape(-1)
    structures = list(structures)
    ranges0 = [np.broadcast_to(st.ranges, (d,)).astype(np.float64) for st in structures]
    if isotropic and any(np.any(r != r[0]) for r in ranges0):
        raise ValueError("fit_covariance: isotropic=True needs equal starting ranges in every structure")
    nr = 1 if isotropic else d
    if fit_nugget and not nugget > 0:
        raise ValueError("fit_covariance: a fitted nugget needs a positive starting value")

    def unpack(x):
        sts, k = [], 0
        for st in structures:
            sill, rng = np.exp(x[k]), np.exp(x[k + 1:k + 1 + nr])
            k += 1 + nr
            sts.append(CovStructure(st.kind, sill, np.full(d, rng[0]) if isotropic else rng, st.rotation, st.beta))
        return sts, (float(np.exp(x[k])) if fit_nugget else float(nugget))

    def log_grad(sts, nug, g):
        """d loglik / d log theta = theta d loglik / d theta over the fitted parameters (isotropic: the axis sum)"""
        out = []
        for s, st in enumerate(sts):
            gs = g[s * (1 + d):(s + 1) * (1 + d)]
            out.append(st.sill * gs[0])
            ax = st.ranges * gs[1:]
            out.extend([ax.sum()] if isotropic else list(ax))
        if fit_nugget:
            out.append(nug * g[-1])
        return np.array(out)

    x0 = []
    for st, r in zip(structures, ranges0):
        x0.append(np.log(st.sill))
        x0.extend(np.log(r[:nr]))
    if fit_nugget:
        x0.append(np.log(nugget))
    lb = None
    if bounds is not None:
        if len(bounds) != len(x0):
            raise ValueError(f"fit_covariance: {len(bounds)} bounds for {len(x0)} fitted parameters")
        lb = [(None if lo is None else np.log(lo), None if hi is None else np.log(hi)) for lo, hi in bounds]
    last = {}

    def fun(x):
        sts, nug = unpack(x)
        A = KernelCovModelMatrix(sts, S, nug)
        try:
            v, beta, g = loglik(A, yh, drift=drift, reml=reml, grad=True)
        finally:
            A.free()
        last.update(x=np.array(x), value=v, beta=beta, grad=g)
        return -v, -log_grad(sts, nug, g)

    res = minimize(fun, np.array(x0), jac=True, method="L-BFGS-B", bounds=lb, options=FIT_OPTIONS | {"maxiter": int(maxiter)})
    if not np.array_equal(last.get("x"), res.x):
        fun(res.x)
    sts, nug = unpack(res.x)
    info = {"loglik": last["value"], "beta": last["beta"], "grad": last["grad"], "nit": int(res.nit),
            "nfev": int(res.nfev), "success": bool(res.success), "message": str(res.message)}
    return sts, nug, info


CrossValidation = namedtuple("CrossValidation", ["prediction", "error", "variance", "logpdf"])
CrossValidation.__doc__ = """Cross-validation results: prediction, error = y - prediction and variance per point (n entries in
point order, NaN at points not held out), logpdf per group (the Gaussian log-density of the group's values given the
other points; their sum is the usual criterion for comparing models)."""


def _groups_csr(groups, n):
    """(ngroups, group_ptr, group_idx) of a sequence of index arrays; None: leave-one-out (NULL pointers)"""
    if groups is None:
        return n, None, None
    sizes = [np.size(g) for g in groups]
    ptr = np.zeros(len(sizes) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum(sizes)
    idx = np.concatenate([np.asarray(g, dtype=np.int64).reshape(-1) for g in groups]) if sizes else np.zeros(0, np.int64)
    return len(sizes), ptr, idx


def cross_validate(structures, sources, y, *, nugget=0.0, drift=None, groups=None):
    """Leave-one-out (groups=None) or leave-group-out cross-validation of kriging of y at the sources (d x n) under the
    nested covariance model `structures` with observation noise `nugget` (a scalar, or n per-point values), drift None
    (simple kriging), "constant" or an n x p array (universal kriging; the drift is re-estimated from the remaining
    points for every group).  groups: a sequence of index arrays of 1..128 distinct points each.

    Builds the covariance and its dense factor (about 8 n^2 bytes of device memory) and frees both.  The points are
    ordered so that the held-out points come last, group by group: the sweeps then start at the held-out columns, so
    cross-validating a few groups costs about one factorisation.  Returns a CrossValidation in the caller's point order
    (KernelCovCholesky.crossval)."""
    S = _f64_colmajor(sources)
    n = S.shape[1]
    yh = np.asarray(y, dtype=np.float64).reshape(n)
    F = _drift_columns(drift, n)
    if groups is None:
        perm = np.arange(n)
        pgroups = None
    else:
        gl = [np.asarray(g, dtype=np.int64).reshape(-1) for g in groups]
        held = np.concatenate(gl) if gl else np.zeros(0, np.int64)
        if held.size and (held.min() < 0 or held.max() >= n):
            raise ValueError(f"cross_validate: a group index lies outside 0 .. {n - 1}")
        if np.unique(held).size != held.size:
            raise ValueError("cross_validate: a point is held out twice")
        rest = np.setdiff1d(np.arange(n), held)
        perm = np.concatenate([rest, held])
        pgroups, k = [], rest.size
        for g in gl:
            pgroups.append(np.arange(k, k + g.size))
            k += g.size
    nug = np.asarray(nugget, dtype=np.float64)
    per_point = nug.ndim > 0
    A = KernelCovModelMatrix(structures, np.ascontiguousarray(S[:, perm]), 0.0 if per_point else float(nug))
    fac = None
    try:
        fac = KernelCovCholesky(A, diag=nug.reshape(n)[perm] if per_point else None)
        r = fac.crossval(yh[perm], drift=F[perm] if F.shape[1] else None, groups=pgroups)
    finally:
        if fac is not None:
            fac.free()
        A.free()
    inv = np.empty(n, dtype=np.int64)
    inv[perm] = np.arange(n)
    return CrossValidation(r.prediction[inv], r.error[inv], r.variance[inv], r.logpdf)


class KernelCovCholesky:
    """Dense Cholesky factor A = L L' of a square kernel-covariance operator A (KernelCovMatrix, GridKernelCovMatrix,
    KernelCovModelMatrix or GridKernelCovModelMatrix; exactly as built, nugget included), held on the device
    (gsi_kernelcov_chol; single GPU, about 8 n^2 bytes).  A is materialised by the product kernel's own value code and
    factored once (n^3 / 3 flops on the FP64 tensor cores); every solve after that is two triangular sweeps.

    diag (n values, optional) is added to A's diagonal before the factorisation (gsi_kernelcov_chol_diag): per-point
    nuggets, such as heteroscedastic observation noise or the joint source / target matrix of `simulate`.

    A non-positive pivot raises PosDefException with the 1-based failing column in `.column`."""

    def __init__(self, A, diag=None):
        op = as_operator(A)
        self.ctx = op.ctx
        self._lib = op.ctx._lib
        self._h = C.c_void_p()
        col = C.c_int64(0)
        if diag is None:
            status = self._lib.gsi_kernelcov_chol(op._h, C.byref(self._h), C.byref(col))
        else:
            d = np.ascontiguousarray(diag, dtype=np.float64).reshape(-1)
            if d.size != op.shape[1]:
                raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                             f"KernelCovCholesky: diag has {d.size} values, A is {op.shape[1]} x {op.shape[1]}")
            status = self._lib.gsi_kernelcov_chol_diag(op._h, _pd(d), C.byref(self._h), C.byref(col))
        try:
            check(status)
        except _lib.PosDefException as e:
            e.column = int(col.value)
            raise
        n = C.c_int64()
        check(self._lib.gsi_chol_size(self._h, C.byref(n)))
        self.n = int(n.value)

    @property
    def logdet(self):
        """log det A = 2 sum log L[i, i] (summed in a fixed order on the device)."""
        v = C.c_double()
        check(self._lib.gsi_chol_logdet(self._h, C.byref(v)))
        return float(v.value)

    @property
    def L(self):
        """The factor on the host (n x n lower triangular)."""
        out = np.empty((self.n, self.n), dtype=np.float64, order="F")
        check(self._lib.gsi_chol_download(self._h, _pd(out), max(1, self.n)))
        return out

    def _solve(self, B, half):
        Bh = np.asarray(B, dtype=np.float64)
        vector = Bh.ndim == 1
        Bh = Bh.reshape(-1, 1) if vector else Bh
        if Bh.ndim != 2 or Bh.shape[0] != self.n:
            raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                         f"KernelCovCholesky: B has shape {Bh.shape}, the factor is {self.n} x {self.n}")
        k = Bh.shape[1]
        X = np.empty((self.n, k), dtype=np.float64, order="F")
        for c0 in range(0, k, 1024):                    # the widest device iterate: 1024 columns per call
            Bd = DeviceMatrix.from_host(self.ctx, Bh[:, c0:c0 + 1024])
            try:
                check(self._lib.gsi_chol_solve(self._h, half, Bd._h, Bd._h))
                X[:, c0:c0 + 1024] = Bd.numpy()
            finally:
                Bd.free()
        return X[:, 0] if vector else X

    def solve(self, B):
        """A^-1 B (B: n or n x k, any k)."""
        return self._solve(B, 0)

    def solve_lower(self, B):
        """L^-1 B (B: n or n x k, any k)."""
        return self._solve(B, 1)

    def variance(self, cross_op, drift=None):
        """Kriging variance of the noise-free value at the m targets of cross_op = C(T, S) (KernelCrossCovMatrix or
        GridKernelCrossCovMatrix whose sources are this factor's n points, same covariance model): c(t, t) -
        ||L^-1 c_t||^2 for simple kriging (drift None), plus r' (G'G)^-1 r, G = L^-1 F_s, r = f_t - G' L^-1 c_t, with a
        drift ("constant" or (F_sources n x p, F_targets m x p), p <= 32)."""
        m = cross_op.shape[0]
        Fs, Ft = drift_matrices(drift, self.n, m)
        p = Fs.shape[1]
        Fs, Ft = np.asfortranarray(Fs, dtype=np.float64), np.asfortranarray(Ft, dtype=np.float64)
        var = np.empty(m, dtype=np.float64)
        check(self._lib.gsi_chol_krige_variance(self._h, cross_op._h, _pd(Fs) if p else None, _pd(Ft) if p else None,
                                                p, _pd(var)))
        return var

    def simulate(self, Xi, *, n_cond=0, y=None, drift=None):
        """Realisations at the last n - n_cond points of a factor of the joint matrix [sources; targets] (gsi_chol_simulate):
        Z = F_t B + L(T, :) V from the standard normals Xi (n x k, any k; 1024 columns per device call), conditioned on
        y (n_cond values) at the first n_cond points with drift None (simple kriging: known zero mean), "constant" or
        (F_sources n_cond x p, F_targets (n - n_cond) x p), p <= 32.  Xi = 0 gives the kriging estimate; n_cond = 0 gives
        unconditional samples L Xi.  Returns (n - n_cond) x k."""
        ns = int(n_cond)
        m = self.n - ns
        Xh = np.asarray(Xi, dtype=np.float64)
        Xh = Xh.reshape(-1, 1) if Xh.ndim == 1 else Xh
        if Xh.ndim != 2 or Xh.shape[0] != self.n:
            raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                         f"KernelCovCholesky.simulate: Xi has shape {Xh.shape}, the factor is {self.n} x {self.n}")
        if drift is not None and ns == 0:
            raise ValueError("simulate: a drift needs conditioning data (n_cond > 0)")
        Fs, Ft = drift_matrices(drift, ns, m)
        p = Fs.shape[1]
        yh = np.ascontiguousarray(np.zeros(0) if y is None else y, dtype=np.float64).reshape(-1)
        if yh.size != ns:
            raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                         f"KernelCovCholesky.simulate: y has {yh.size} values, n_cond is {ns}")
        Fs, Ft = np.asfortranarray(Fs, dtype=np.float64), np.asfortranarray(Ft, dtype=np.float64)
        k = Xh.shape[1]
        Z = np.empty((m, k), dtype=np.float64, order="F")
        for c0 in range(0, k, 1024):                    # the widest device iterate: 1024 columns per call
            Xd = DeviceMatrix.from_host(self.ctx, Xh[:, c0:c0 + 1024])
            Zd = None
            try:
                Zd = DeviceMatrix(self.ctx, m, Xd.shape[1], LAYOUT_TALL)
                check(self._lib.gsi_chol_simulate(self._h, ns, _pd(yh) if ns else None, _pd(Fs) if p else None,
                                                  _pd(Ft) if p else None, p, Xd._h, Zd._h))
                Z[:, c0:c0 + 1024] = Zd.numpy()
            finally:
                Xd.free()
                if Zd is not None:
                    Zd.free()
        return Z

    def crossval(self, y, *, drift=None, groups=None):
        """Leave-one-out (groups=None) or leave-group-out cross-validation of kriging on this factor
        (gsi_chol_crossval; Dubrule 1983): for every group B, the prediction of y_B from all other points with the
        drift re-estimated by GLS from them (drift None: simple kriging, "constant" or an n x p array, p <= 32), its
        error y_B - yhat_B, the error variance and the Gaussian log-density log p(y_B | y_-B).  groups: a sequence of
        index arrays of 1..128 distinct points each; points in no group are not held out.

        The variance is that of predicting the observation: the noise-free kriging variance plus the point's nugget
        (or diag entry); the noise-free variance is variance - nugget_i.  Returns a CrossValidation with prediction,
        error and variance in point order (NaN where not held out) and one logpdf per group.  A group whose drift the
        remaining points cannot identify raises PosDefException with its 0-based index in `.group`."""
        n = self.n
        yh = np.ascontiguousarray(y, dtype=np.float64).reshape(-1)
        if yh.size != n:
            raise _lib.DimensionMismatch(_lib.ERR_DIMENSION_MISMATCH,
                                         f"KernelCovCholesky.crossval: y has {yh.size} values, the factor is {n} x {n}")
        F = _drift_columns(drift, n)
        p = F.shape[1]
        ng, ptr, idx = _groups_csr(groups, n)
        m = n if ptr is None else int(ptr[-1])
        err = np.empty(max(m, 1))
        var = np.empty(max(m, 1))
        lpd = np.empty(max(ng, 1))
        failed = C.c_int64(0)
        pi64 = C.POINTER(C.c_int64)
        status = self._lib.gsi_chol_crossval(self._h, _pd(yh), _pd(F) if p else None, p, ng,
                                             None if ptr is None else ptr.ctypes.data_as(pi64),
                                             None if idx is None else idx.ctypes.data_as(pi64), _pd(err), _pd(var),
                                             _pd(lpd), C.byref(failed))
        try:
            check(status)
        except _lib.PosDefException as e:
            e.group = int(failed.value) - 1 if failed.value else None
            raise
        points = np.arange(n) if idx is None else idx
        out = [np.full(n, np.nan) for _ in range(3)]
        out[1][points] = err[:m]
        out[2][points] = var[:m]
        out[0][points] = yh[points] - err[:m]
        return CrossValidation(out[0], out[1], out[2], lpd[:ng])

    def free(self):
        if getattr(self, "_h", None) and self._h:
            self._lib.gsi_chol_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
