"""Matern (nu = 3/2, 5/2) and spherical covariance kernels of the matrix-free operator (GSI_KERNEL_MATERN32 /
MATERN52 / SPHERICAL), tested to the standard of tests/test_gpu_product_exact.py, whose helpers are reused:

* CPU: the kind codes agree across the C header, the Python host, the Julia shim and the oracle; the dense
  reference below (kernel_cov_dense: the new kinds' formulas, used by the randsvd parity tests) equals the Matern
  Bessel form, and its spherical model is 1 at 0, 0 beyond the range and C^1 there.
* GPU: kernel values in ulps against a 160-bit reference of the device's own r2 (arithmetic path) or of the
  host's scaled lattice offsets (table path); symmetry, unit diagonal, range, epilogue and width / schedule
  independence of the extracted values; element-wise product bounds at every width and schedule shape; the
  grid operator against the arithmetic one; randsvd parity (oracle.randsvd on the dense reference);
  the error paths of both constructors.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle
from gpu_util import get_gsi, gsi  # noqa: F401
from test_gpu_product_exact import (TWO_M1000, U, WIDTHS, _mp, apply_dev, big_ok, extract, extracted, fma,
                                    grid_shape, kcov_schedule, num_sms, sample_rows, ulp_err, unit_columns)
from test_gpu_randsvd import SINE_TOL, SV_TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_KINDS = ["matern32", "matern52", "spherical"]
PRE = {"matern32": 3.0 ** 0.5, "matern52": 5.0 ** 0.5, "spherical": 1.0}     # host scaling of gsi_op_kernelcov
PRE_LITERAL = {"matern32": 1.73205080756887729353, "matern52": 2.23606797749978969641, "spherical": 1.0}


# ------------------------------------------------------------------ CPU: constants and the dense reference
def _defines(path, pattern):
    with open(os.path.join(ROOT, path)) as f:
        return {m.group(1): int(m.group(2)) for m in re.finditer(pattern, f.read())}


def test_kernel_kind_codes_agree():
    """GSI_KERNEL_* in the header == _lib.py == the Julia consts == core._KINDS (and == oracle/kernels.py for the
    kinds the oracle defines)."""
    import gsi_b200
    from gsi_b200 import _lib, core
    from oracle import kernels
    hdr = _defines("include/gsi_b200.h", r"#define GSI_KERNEL_(\w+) (-?\d+)")
    jl = _defines("julia/GeostatInversionB200.jl", r"const GSI_KERNEL_(\w+) = Int32\((-?\d+)\)")
    assert set(hdr) == {"EXPONENTIAL", "GAUSSIAN", "POWERLAW", "MATERN32", "MATERN52", "SPHERICAL"}
    assert jl == hdr
    for name, code in hdr.items():
        assert getattr(_lib, "KERNEL_" + name) == code, name
        assert getattr(gsi_b200, "KERNEL_" + name) == code, name
        if hasattr(kernels, name):
            assert getattr(kernels, name) == code, name
        assert core._KINDS[name.lower()] == code and core._KINDS[code] == code, name
    assert len(set(hdr.values())) == len(hdr)


def kernel_cov_dense(kind, coords, ell, rows=None):
    """Dense reference C[rows, :] (sigma2 = 1, nugget = 0) of the new kinds, straight from the definitions in
    include/gsi_b200.h in the style of oracle.kernel_cov_dense (r2 fma-free, k = 0..d-1 in order)."""
    u = oracle.scaled_coords(coords, ell)
    ui = u if rows is None else u[:, rows]
    r2 = np.zeros((ui.shape[1], u.shape[1]))
    for k in range(u.shape[0]):
        diff = ui[k][:, None] - u[k][None, :]
        r2 += diff * diff
    if kind == "matern32":
        s = np.sqrt(3.0 * r2)
        return (1.0 + s) * np.exp(-s)
    if kind == "matern52":
        s = np.sqrt(5.0 * r2)
        return (1.0 + s + s * s / 3.0) * np.exp(-s)
    if kind == "spherical":
        r = np.sqrt(r2)
        return np.where(r < 1.0, 0.5 * (1.0 - r) ** 2 * (2.0 + r), 0.0)     # = 1 - 1.5 r + 0.5 r^3, no cancellation
    raise ValueError(kind)


def _k1d(kind, r, ell=1.0):
    """Reference kernel values k(r) at distances r (one row of the dense matrix of 1-D points)."""
    coords = np.concatenate([[0.0], np.asarray(r, dtype=np.float64)])[None, :]
    return kernel_cov_dense(kind, coords, [ell], rows=[0])[0, 1:]


@pytest.mark.parametrize("nu,kind", [(1.5, "matern32"), (2.5, "matern52")])
def test_reference_matern_equals_bessel_form(nu, kind):
    """2^(1-nu) / Gamma(nu) (sqrt(2 nu) r)^nu K_nu(sqrt(2 nu) r), the Rasmussen-Williams form, to 1e-14 (for r <= 5:
    beyond, both sides' rounding of sqrt(2 nu) r, amplified by the conditioning ~ sqrt(2 nu) r of exp, dominates)."""
    sp = pytest.importorskip("scipy.special")
    r = np.concatenate([10.0 ** np.linspace(-6, 0, 200), np.linspace(1, 5, 400)])
    x = np.sqrt(2 * nu) * r
    bessel = 2.0 ** (1 - nu) / sp.gamma(nu) * x ** nu * sp.kv(nu, x)
    k = _k1d(kind, r)
    assert np.max(np.abs(k - bessel) / bessel) <= 1e-14
    assert _k1d(kind, [0.0])[0] == 1.0


def test_reference_spherical_shape():
    """1 at r = 0, 0 at r >= 1, C^1 at r = 1 (value and slope 1.5 (r^2 - 1) both reach 0), equal to
    1 - 1.5 r + 0.5 r^3 inside the range."""
    sph = "spherical"
    assert _k1d(sph, [0.0])[0] == 1.0
    assert np.all(_k1d(sph, [1.0, 1.0 + 1e-15, 1.5, 3.0, 1e6]) == 0.0)
    r = np.linspace(0, 0.999, 1000)
    assert np.allclose(_k1d(sph, r), 1 - 1.5 * r + 0.5 * r ** 3, rtol=0, atol=1e-15)
    for h in (1e-2, 1e-4, 1e-6):
        left = _k1d(sph, [1.0 - h])[0]
        assert 0 < left <= 1.5 * h * h * (1 + h)               # k(1 - h) = 1.5 h^2 - 0.5 h^3: slope -> 0
    assert np.all(np.diff(_k1d(sph, np.linspace(0, 1, 101))) < 0)
    assert _k1d(sph, [2.0], ell=2.0)[0] == 0.0 and _k1d(sph, [1.0], ell=2.0)[0] == 0.3125   # ell is the range


# ------------------------------------------------------------------ A. kernel values against a high-precision reference
# Bounds, derived beside kern_eval (csrc/kcov_gemm.cu) from the instruction sequences: relative error
# (c0 + 2 kappa) 2^-52 with c0 = 3 / 4.25 / 2.5, where kappa = |s k'(s) / k(s)| carries fast_sqrt_pos's 2 ulp of s.
# In ulps of the reference that is at most twice as much (the value and its error may sit at opposite ends of a
# binade): c = 2 c0 and 4 kappa.  The lattice table's host sequence (libm exp <= 1 ulp, sqrt, and the same or fewer
# roundings) stays within the same constants.
C_ULP = {"matern32": 6.0, "matern52": 8.5, "spherical": 5.0}


def kappa(kind, s):
    if kind == "matern32":
        return s * s / (1 + s)
    if kind == "matern52":
        return s * s * (1 + s) / (3 + 3 * s + s * s)
    return 2 * s / (1 - s) - s / (2 + s)


def ref_value(kind, mp, R2):
    """k of the device's own argument: s = sqrt(r2) in scaled (sqrt(2 nu)-folded) coordinates."""
    s = mp.sqrt(R2)
    if kind == "matern32":
        return (1 + s) * mp.exp(-s), s
    if kind == "matern52":
        return (1 + s + R2 / 3) * mp.exp(-s), s
    return (mp.mpf(0.5) * (1 - s) ** 2 * (2 + s) if s < 1 else mp.mpf(0)), s


# s within the sqrt error of the spherical range: 1 - s and fast_sqrt_pos's 2 ulp are of the same size, so any
# value in [0, 1.5 (2^-50)^2] (the spherical value of an argument 2^-50 below 1) is accepted
SPH_BAND = 2.0 ** -50


def _targets(kind, rng):
    """Distances s (scaled coordinates, after the sqrt(2 nu) fold) the points are placed at."""
    small = 10.0 ** rng.uniform(-12, -2, 100)
    if kind == "spherical":
        near = 10.0 ** rng.uniform(-15.5, -3, 200)
        ulps = np.array([1.0 + k * 2.0 ** -52 for k in range(-8, 9)])
        return np.concatenate([rng.uniform(0, 1, 3000), small, 1 - near, 1 + near, ulps, rng.uniform(1, 3, 300)])
    return np.concatenate([rng.uniform(0, 8, 4000), small, rng.uniform(690, 700, 300), rng.uniform(1020, 1023.99, 30),
                           rng.uniform(1024, 1030, 30), [1024.0, 1023.9999999]])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_kernel_values_ulp(gsi, kind, d):
    """Arithmetic generation: every extracted value against the 160-bit kernel of the device's own r2 (rebuilt
    exactly: the host scaling, then the same subtraction and fma chain from the 1e-300 offset)."""
    mp = _mp()
    rng = np.random.default_rng(100 * d + len(kind))
    ell = np.array([1.3, 0.7, 2.1][:d])
    pre = PRE_LITERAL[kind]
    rho = _targets(kind, rng)
    dirs = rng.standard_normal((d, rho.size))
    dirs /= np.linalg.norm(dirs, axis=0)
    origin = np.array([0.37, -1.1, 0.52][:d])
    coords = np.concatenate([origin[:, None], origin[:, None] + rho * dirs * (ell / pre)[:, None]], axis=1)
    n = coords.shape[1]
    op = gsi.KernelCovMatrix(kind, coords, ell, beta=0.8)
    col = extract(gsi, op, n, [0])[:, 0]
    u = (coords / ell[:, None]) * pre
    errs, args, bounds, nflush, nzero, nband = [], [], [], 0, 0, 0
    for i in range(n):
        r2 = 1e-300
        for k in range(d):
            dk = float(u[k, i] - u[k, 0])
            r2 = fma(dk, dk, r2)
        ref, s = ref_value(kind, mp, mp.mpf(r2))
        dev = float(col[i])
        if kind == "spherical":
            if abs(1 - s) <= SPH_BAND:
                nband += 1
                assert 0.0 <= dev <= 1.5 * SPH_BAND ** 2, (float(s), dev)
                continue
            if s >= 1:
                nzero += 1
                assert dev == 0.0, (float(s), dev)
                continue
        elif mp.exp(-s) < TWO_M1000 and dev == 0.0:
            nflush += 1                                                  # flushed with the exp factor
            continue
        errs.append(ulp_err(dev, ref, mp))
        args.append(float(s))
        bounds.append(C_ULP[kind] + 4 * float(kappa(kind, s)))
    errs, args, bounds = np.array(errs), np.array(args), np.array(bounds)
    w = int(np.argmax(errs - bounds))
    small = args < 1.0 if kind != "spherical" else args < 0.5
    msg = (f"{kind} d={d}: max error {errs.max():.3f} ulp (at s < {1.0 if kind != 'spherical' else 0.5}: "
           f"{errs[small].max():.3f} ulp); worst against the bound: {errs[w]:.3f} ulp at s = {args[w]!r} "
           f"(bound {bounds[w]:.3f}); {errs.size} values, {nflush} flushed, {nzero} beyond the range, {nband} at it")
    print(msg)
    assert np.all(errs <= bounds), msg
    if kind == "spherical":
        assert nzero >= 300 and nband >= 3, msg
    else:
        assert nflush >= 60, msg


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_table_kernel_values_ulp(gsi, kind, d):
    """Structured grid: the looked-up values (host libm) against the 160-bit kernel of the host's scaled offsets."""
    mp = _mp()
    shape, spacing = {1: ((3000,), (0.003,)), 2: ((1500, 3), (0.005, 345.5)), 3: ((500, 3, 2), (0.015, 300.0, 600.0))}[d]
    ell = np.ones(d)
    op = gsi.GridKernelCovMatrix(kind, shape, ell, spacing=spacing)
    n = int(np.prod(shape))
    col = extract(gsi, op, n, [0])[:, 0]
    lat = np.array(np.unravel_index(np.arange(n), shape, order="F"))
    pre = {"matern32": mp.sqrt(3), "matern52": mp.sqrt(5), "spherical": mp.mpf(1)}[kind]
    errs, args, bounds, nzero = [], [], [], 0
    for i in range(n):
        R2 = mp.mpf(0)
        for k in range(d):
            uk = (float(lat[k, i]) * spacing[k]) / ell[k]
            R2 += mp.mpf(uk) ** 2
        ref, s = ref_value(kind, mp, R2 * pre * pre)
        dev = float(col[i])
        if kind == "spherical" and s >= 1:
            nzero += 1
            assert dev == 0.0 or s - 1 < SPH_BAND, (float(s), dev)
            continue
        errs.append(ulp_err(dev, ref, mp))
        args.append(float(s))
        bounds.append(C_ULP[kind] + 4 * float(kappa(kind, s)))
    errs, args, bounds = np.array(errs), np.array(args), np.array(bounds)
    w = int(np.argmax(errs - bounds))
    msg = (f"table {kind} d={d}: max error {errs.max():.3f} ulp; worst against the bound: {errs[w]:.3f} ulp at "
           f"s = {args[w]!r} (bound {bounds[w]:.3f}); {n} values, {nzero} beyond the range")
    print(msg)
    assert np.all(errs <= bounds), msg


# ------------------------------------------------------------------ B. extracted values on the schedule shapes
@pytest.mark.gpu
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_kernel_values_symmetry_range_and_epilogue(gsi, kind, dim):
    """Full round + ragged stream-K tail: C_hat[S, S] exactly symmetric with a unit diagonal, 0 < k <= 1 (Matern)
    or 0 <= k <= 1 (spherical, which reaches 0 inside this grid), sigma2 / nugget applied with one rounding."""
    from test_gpu_product_exact import make_op
    op, S, Cs = extracted(kind, dim, "big")
    n = op.shape[0]
    assert kcov_schedule(n, n, num_sms())["full_rounds"] == 1
    Css = Cs[:, S]
    assert np.array_equal(Css, Css.T)
    assert np.all(np.diag(Css) == 1.0)
    assert np.all(Cs <= 1.0)
    if kind == "spherical":
        assert np.all(Cs >= 0.0) and np.any(Cs == 0.0) and np.any((Cs > 0.0) & (Cs < 1.0))
    else:
        assert np.all(Cs > 0.0)
    E = unit_columns(n, S)
    unit = E.T.astype(bool)
    for sigma2 in (0.5, 1.7):
        Y = apply_dev(gsi, make_op(gsi, kind, dim, "big", sigma2=sigma2, nugget=0.3), E).T
        plain = sigma2 * Cs
        assert np.array_equal(Y[~unit], plain[~unit]), sigma2
        for c, j in zip(*np.nonzero(unit)):
            ok = (float(np.float64(sigma2 * Cs[c, j]) + 0.3), fma(sigma2, Cs[c, j], 0.3))
            assert Y[c, j] in ok, (sigma2, S[c], j, Y[c, j], ok)


@pytest.mark.gpu
def test_matern_values_near_zero_distance(gsi):
    """s from 1e-12 to 1e-4, densely around 2e-8 where (1 + s + s^2/3) e^-s rounds up to 1 + 2^-52 before the
    clamp: every value lies in (0, 1]."""
    rng = np.random.default_rng(11)
    rho = np.concatenate([10.0 ** rng.uniform(-12, -4, 2000), rng.uniform(1.5e-8, 2.5e-8, 2000)])
    coords = np.concatenate([[0.0], rho])[None, :]
    for kind in ("matern32", "matern52"):
        col = extract(gsi, gsi.KernelCovMatrix(kind, coords / PRE[kind], [1.0]), coords.shape[1], [0])[:, 0]
        assert np.all(col > 0.0) and np.all(col <= 1.0), (kind, float(col.max()).hex())


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_kernel_values_width_and_schedule_independent(gsi, kind, dim):
    """The same (i, j) through every width and through other k-sweep schedules is bit-identical."""
    op, _, _ = extracted(kind, dim, "big")
    ctx = op.ctx
    n = op.shape[0]
    R = np.random.default_rng(3).choice(n, 1024, replace=False)
    special = [0, n - 1] + [a for a, _ in kcov_schedule(n, n, num_sms())["tail_tiles"]]
    R[:len(special)] = special
    ref = extract(gsi, op, n, R)
    for w in WIDTHS[:-1]:
        assert np.array_equal(extract(gsi, op, n, R[:w]), ref[:, :w]), w
    keys = ("kcov.sweep_groups", "kcov.sweep_div", "kcov.window", "kcov.epoch_shift")
    saved = {k: ctx.get_option(k) for k in keys}
    try:
        for groups, div, window in ((1, 0, 0), (8, -3, 0), (64, 4, 0), (1, 0, 2)):
            ctx.set_option("kcov.sweep_groups", groups)
            ctx.set_option("kcov.sweep_div", div)
            ctx.set_option("kcov.epoch_shift", 2)
            ctx.set_option("kcov.window", window)
            for w in (27, 256):
                assert np.array_equal(extract(gsi, op, n, R[:w]), ref[:, :w]), (groups, div, window, w)
    finally:
        for k, v in saved.items():
            ctx.set_option(k, v)


# ------------------------------------------------------------------ C. products
def _bound_check(Y, ref, bound, what):
    err = np.abs(Y - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {bad.sum()} elements out of bound, first at {tuple(np.argwhere(bad)[0])}; "
                           f"max err/bound {np.nanmax(err / bound):.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("size", ["small", "big"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_kcov_product_bound(gsi, kind, dim, size, cols):
    """Y = C X on sampled rows within 2 gamma_n (|C_hat| |X|) of C_hat X, after a NaN-poisoned product."""
    op, S, Cs = extracted(kind, dim, size)
    n = op.shape[0]
    sched = kcov_schedule(n, n, num_sms())
    if size == "small":
        assert sched["full_rounds"] == 0 and sched["tail_tiles"]
    else:
        assert big_ok(n, num_sms())
    apply_dev(gsi, op, np.full((n, cols), np.nan))
    X = np.random.default_rng(cols).standard_normal((n, cols))
    Y = apply_dev(gsi, op, X)[S]
    gamma = n * U / (1 - n * U)
    _bound_check(Y, Cs @ X, 2 * gamma * (np.abs(Cs) @ np.abs(X)), f"{kind} dim={dim} n={n} cols={cols}")


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [1, 64, 300])
@pytest.mark.parametrize("size", ["small", "big"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_grid_operator_matches_arithmetic(gsi, kind, dim, size, cols):
    """GridKernelCovMatrix against KernelCovMatrix on the same lattice points: the products differ by no more
    than both rounding bounds plus the difference of the two extracted value sets applied to |X|."""
    shape = grid_shape(dim, size)
    ell = [s / 2.5 for s in shape]
    coords = oracle.grid_coords(shape)
    n = coords.shape[1]
    S = sample_rows(n)
    opg = gsi.GridKernelCovMatrix(kind, shape, ell)
    opa = gsi.KernelCovMatrix(kind, coords, ell)
    Cg = np.ascontiguousarray(extract(gsi, opg, n, S).T)
    Ca = np.ascontiguousarray(extract(gsi, opa, n, S).T)
    assert np.max(np.abs(Cg - Ca)) < 1e-13
    X = np.random.default_rng(cols + 5).standard_normal((n, cols))
    Yg = apply_dev(gsi, opg, X)[S]
    Ya = apply_dev(gsi, opa, X)[S]
    gamma = n * U / (1 - n * U)
    aX = np.abs(X)
    bound = 2 * gamma * ((np.abs(Cg) + np.abs(Ca)) @ aX) + np.abs(Cg - Ca) @ aX
    _bound_check(Yg, Ya, bound, f"grid vs arithmetic {kind} dim={dim} {size} cols={cols}")


# ------------------------------------------------------------------ D. randsvd parity with oracle.randsvd on the dense reference
# Anisotropic grids (SURVEY.md: degenerate spectra); the relative gap sigma_K / sigma_{K+1} - 1 of the covariance
# is >= 1e-3 in every case (checked on the host when the cases were chosen).
RSVD_CASES = {
    "matern32": ((90, 80), (12.0, 8.0), 200),
    "matern52": ((90, 80), (12.0, 8.0), 200),
    "spherical": ((90, 80), (40.0, 30.0), 200),
}


def _dense(kind, grid, ell):
    return kernel_cov_dense(kind, oracle.grid_coords(grid), ell)


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 2])
@pytest.mark.parametrize("path", ["arithmetic", "grid"])
@pytest.mark.parametrize("kind", NEW_KINDS)
def test_randsvd_parity(gsi, kind, path, q):
    """gsi.randsvd on the operator (LU_REF normaliser) against oracle.randsvd on the dense reference matrix."""
    grid, ell, K = RSVD_CASES[kind]
    p = 10
    C = _dense(kind, grid, ell)
    n = C.shape[0]
    Omega = np.random.default_rng(q).standard_normal((n, K + p))
    Zref = oracle.randsvd(C, Omega, K, p, q)
    if path == "grid":
        op = gsi.GridKernelCovMatrix(kind, grid, ell)
    else:
        op = gsi.KernelCovMatrix(kind, oracle.grid_coords(grid), ell)
    Z, S = gsi.randsvd(op, K, p, q, Omega=Omega, normaliser=gsi.NORMALISER_LU_REF, return_singular_values=True)
    c = oracle.compare_Z(Z, Zref, K)
    assert c["tail_zero"]
    assert c["sv_rel"] < SV_TOL and c["sine"] < SINE_TOL, c
    assert np.max(np.abs(S[:K] - oracle.singvals_from_Z(Zref, K)) / S[:K]) < SV_TOL


# ------------------------------------------------------------------ E. error paths
@pytest.mark.gpu
def test_unknown_kind_name_raises(gsi):
    with pytest.raises(KeyError):
        gsi.KernelCovMatrix("matern", np.zeros((2, 4)), [1.0, 1.0])
    with pytest.raises(KeyError):
        gsi.GridKernelCovMatrix("matern72", (4, 4), [1.0, 1.0])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [6, -1, 15])
def test_abi_rejects_unknown_kind(gsi, kind):
    """Kinds outside 0..5 -- including the library's internal lattice-table kind -- are invalid arguments of
    both constructors, and no operator is returned."""
    ctx = gsi.default_context()
    lib = ctx._lib
    pd = C.POINTER(C.c_double)
    coords = np.ascontiguousarray(np.arange(8, dtype=np.float64))
    ell = np.ones(2)
    dims = (C.c_int64 * 2)(2, 2)
    spacing = np.ones(2)
    h = C.c_void_p()
    st = lib.gsi_op_kernelcov(ctx._h, kind, 2, 4, coords.ctypes.data_as(pd), ell.ctypes.data_as(pd), 1.0, 0.0, 1.0,
                              0, 4, C.byref(h))
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h.value
    st = lib.gsi_op_kernelcov_grid(ctx._h, kind, 2, dims, spacing.ctypes.data_as(pd), ell.ctypes.data_as(pd), 1.0,
                                   0.0, 1.0, 0, 4, C.byref(h))
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h.value
    assert "unknown kernel kind" in lib.gsi_last_error_string().decode()
