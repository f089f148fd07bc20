"""Nested covariance models with rotated anisotropy (gsi_op_kernelcov_model / gsi_op_kernelcov_model_grid), tested to
the standard of tests/test_gpu_product_exact.py, whose helpers are reused:

* CPU: rotation_matrix is a rotation whose first row points along the angle; the dense model reference below equals the
  single-kind references for one unrotated structure; the exact 90-degree rotation equals swapping the two ranges.
* GPU, bit for bit: one unrotated structure equals KernelCovMatrix / GridKernelCovMatrix with sigma2 = its sill; two
  identical structures of sill 0.5 (the fused KC_KIND_MODEL kernel) equal the single-kind operator with sigma2 = 1,
  unrotated and rotated, at every width and both schedule shapes.
* GPU, within bounds: extracted values of 2-4-structure rotated models in ulps against a 160-bit reference of the
  device's own coordinates with the bound documented beside kern_eval; symmetry, diagonal, spherical range, width /
  schedule independence; element-wise product bounds; the signed lattice table against a 160-bit reference of the
  host's rotated offsets and against the arithmetic operator; randsvd parity with oracle.randsvd; the error paths;
  two ranks.
"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle
from gpu_util import get_gsi, gsi  # noqa: F401
from test_gpu_matern import C_ULP, SPH_BAND, kappa
from test_gpu_matern import kernel_cov_dense as matern_dense
from test_gpu_product_exact import (U, WIDTHS, _mp, apply_dev, big_ok, extract, fma, grid_shape, kcov_schedule,
                                    num_sms, sample_rows, unit_columns)
from test_gpu_randsvd import SINE_TOL, SV_TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G      # noqa: E402  (importing needs no GPU)

KINDS = ["exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"]
CODE = {k: i for i, k in enumerate(KINDS)}
NAME = {i: k for k, i in CODE.items()}
# host scaling of the coordinates (gsi_op_kernelcov): the kernel sees r2 with these factors folded in
PRE = {0: 1.0, 1: 0.70710678118654752440, 2: 1.0, 3: 1.73205080756887729353, 4: 2.23606797749978969641, 5: 1.0}
TWO52 = 2.0 ** -52


# ------------------------------------------------------------------ host model: coordinates and dense reference
def structure_coords(st, coords, pre):
    """u = ((sum_j R[k,j] x_j) / range_k) * pre, rebuilt exactly as the library's host code computes it."""
    d, n = coords.shape
    ranges = np.broadcast_to(st.ranges, (d,))
    if st.rotation is None:
        y = coords
    else:
        R = st.rotation.reshape(d, d)
        y = np.empty_like(coords)
        for k in range(d):
            acc = np.zeros(n)
            for j in range(d):
                acc = acc + R[k, j] * coords[j]
            y[k] = acc
    return (y / ranges[:, None]) * pre


def kvalue(kind, r2, beta):
    """k(r2) of unscaled coordinates (x / range), the definitions of include/gsi_b200.h."""
    if kind == 0:
        return np.exp(-np.sqrt(r2))
    if kind == 1:
        return np.exp(-0.5 * r2)
    if kind == 2:
        return np.exp(-beta * np.log1p(r2))
    if kind == 3:
        s = np.sqrt(3.0 * r2)
        return (1.0 + s) * np.exp(-s)
    if kind == 4:
        s = np.sqrt(5.0 * r2)
        return (1.0 + s + s * s / 3.0) * np.exp(-s)
    r = np.sqrt(r2)
    return np.where(r < 1.0, 0.5 * (1.0 - r) ** 2 * (2.0 + r), 0.0)


def model_dense(structures, coords, rows=None, nugget=0.0):
    """Dense reference C[rows, :] = sum_s sill_s k_s + nugget I."""
    n = coords.shape[1]
    rows = np.arange(n) if rows is None else np.asarray(rows)
    C = np.zeros((rows.size, n))
    for st in structures:
        u = structure_coords(st, coords, 1.0)
        r2 = np.zeros_like(C)
        for k in range(u.shape[0]):
            diff = u[k][rows][:, None] - u[k][None, :]
            r2 += diff * diff
        C += st.sill * kvalue(st.kind, r2, st.beta)
    C[np.arange(rows.size), rows] += nugget
    return C


def models(dim, shape):
    """Rotated models of 2..4 structures with mixed kinds, ranges scaled to the grid."""
    L = np.array(shape, dtype=np.float64)
    ang = (0.5,) if dim == 2 else (0.5, -0.3, 0.8)
    R1 = G.rotation_matrix(ang)
    R2 = G.rotation_matrix(tuple(-0.7 * a for a in ang))
    S = G.CovStructure
    return {
        "sph_exp": [S("spherical", 0.6, L / 3, R1), S("exponential", 0.4, L / 2, R2)],
        "three": [S("spherical", 0.5, L / 2, R2), S("matern32", 0.7, L / 6, R1), S("exponential", 1.3, L / 3)],
        "four": [S("gaussian", 0.3, L / 4, R1), S("matern52", 0.9, L / 3, R2), S("powerlaw", 0.2, L / 5, beta=0.8),
                 S("matern32", 1.1, L / 2.5, R1)],
        "two_sph": [S("spherical", 0.5, L / 4, R1), S("spherical", 1.5, L / 3, R2)],
    }


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("angles", [(0.0,), (0.3,), (2.0,), (-1.2,), (0.0, 0.0, 0.0), (0.4, 0.0, 0.0),
                                    (0.5, -0.3, 0.8), (2.5, 1.1, -2.0)])
def test_rotation_matrix(angles):
    """Orthonormal with det +1; in 2-D (and 3-D about z only) the first row is (cos a, sin a), so u_0 measures the
    distance along the principal axis at angle a from the x axis; in 3-D the rows are the z-y-x rotated axes."""
    R = G.rotation_matrix(angles)
    d = 2 if len(angles) == 1 else 3
    assert R.shape == (d, d)
    assert np.max(np.abs(R.T @ R - np.eye(d))) < 1e-15
    assert abs(np.linalg.det(R) - 1.0) < 1e-15
    a = angles[0]
    if d == 2 or angles[1:] == (0.0, 0.0):
        assert np.allclose(R[0, :2], [np.cos(a), np.sin(a)], rtol=0, atol=1e-16)
        x = np.zeros(d)
        x[:2] = [np.cos(a), np.sin(a)]
        assert np.allclose(R @ x, np.eye(d)[0], rtol=0, atol=1e-15)
    else:
        cz, sz, cy, sy = np.cos(a), np.sin(a), np.cos(angles[1]), np.sin(angles[1])
        assert np.allclose(R[0], [cz * cy, sz * cy, -sy], rtol=0, atol=1e-15)


@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_dense_reference_single_structure(kind, d):
    """One structure with R = I equals oracle.kernel_cov_dense (kinds 0..2) or the Matern file's reference (3..5)."""
    rng = np.random.default_rng(d)
    coords = rng.uniform(0, 10, (d, 300))
    ell = np.array([2.5, 1.5, 4.0][:d])
    rot = None if d == 1 else np.eye(d)
    C = model_dense([G.CovStructure(kind, 1.0, ell, rot, beta=0.8)], coords)
    if CODE[kind] <= 2:
        ref = oracle.kernel_cov_dense(CODE[kind], coords, ell, beta=0.8)
    else:
        ref = matern_dense(kind, coords, ell)
    assert np.allclose(C, ref, rtol=1e-13, atol=1e-300)


@pytest.mark.parametrize("kind", KINDS)
def test_rotation_90_degrees_swaps_ranges(kind):
    """R = [[0, 1], [-1, 0]] (exactly representable): u = (x_1 / a_0, -x_0 / a_1), the same r2 as ranges (a_1, a_0)
    without rotation, up to the order of the two squares."""
    coords = np.random.default_rng(5).uniform(-5, 5, (2, 200))
    rot = np.array([[0.0, 1.0], [-1.0, 0.0]])
    a = np.array([3.0, 0.7])
    Cr = model_dense([G.CovStructure(kind, 1.3, a, rot, beta=0.8)], coords)
    Cs = model_dense([G.CovStructure(kind, 1.3, a[::-1], beta=0.8)], coords)
    assert np.allclose(Cr, Cs, rtol=4e-15, atol=1e-300)


def test_cov_structure_and_exports():
    assert G.MODEL_MAX_STRUCTURES == 4
    st = G.CovStructure("matern52", 2.0, [1.0, 3.0])
    assert st.kind == G.KERNEL_MATERN52 and st.sill == 2.0 and st.rotation is None and st.beta == 1.0
    with pytest.raises(KeyError):
        G.CovStructure("matern72", 1.0, [1.0])
    with pytest.raises(ValueError):
        G.rotation_matrix((0.1, 0.2))


# ------------------------------------------------------------------ GPU helpers
def _coords(dim, size):
    shape = grid_shape(dim, size)
    c = oracle.grid_coords(shape)
    return shape, c + np.random.default_rng(7).uniform(-0.3, 0.3, c.shape)


def _ops_equal(gsi, a, b, X):
    Ya, Yb = apply_dev(gsi, a, X), apply_dev(gsi, b, X)
    return np.array_equal(Ya, Yb), Ya, Yb


# ------------------------------------------------------------------ GPU: bit-exact
@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_single_structure_equals_single_kind(gsi, kind, d):
    """R = NULL and sill c: the specialised kernel with sigma2 = c, on both paths, bit for bit (nugget included)."""
    rng = np.random.default_rng(d + 10 * CODE[kind])
    shape = {1: (700,), 2: (30, 23), 3: (9, 8, 10)}[d]
    ell = np.array([70.0, 9.0, 4.0][:d]) / (3.0 if kind == "spherical" else 1.0)
    coords = oracle.grid_coords(shape) + rng.uniform(-0.3, 0.3, (d, int(np.prod(shape))))
    st = [gsi.CovStructure(kind, 1.7, ell, beta=0.8)]
    X = rng.standard_normal((coords.shape[1], 7))
    ok, Ym, Yk = _ops_equal(gsi, gsi.KernelCovModelMatrix(st, coords, nugget=0.2),
                            gsi.KernelCovMatrix(kind, coords, ell, sigma2=1.7, nugget=0.2, beta=0.8), X)
    assert ok, np.max(np.abs(Ym - Yk))
    ok, Ym, Yk = _ops_equal(gsi, gsi.GridKernelCovModelMatrix(st, shape, spacing=0.9, nugget=0.2),
                            gsi.GridKernelCovMatrix(kind, shape, ell, spacing=0.9, sigma2=1.7, nugget=0.2, beta=0.8), X)
    assert ok, np.max(np.abs(Ym - Yk))


@pytest.mark.gpu
@pytest.mark.parametrize("rotated", [False, True])
@pytest.mark.parametrize("size", ["small", "big"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_fused_kernel_equals_single_kind(gsi, kind, dim, size, rotated):
    """Two identical structures of sill 0.5 (fused KC_KIND_MODEL kernel): 0.5 k + 0.5 k = k, so every product equals
    the single-kind operator (unrotated: KernelCovMatrix with sigma2 = 1; rotated: the one-structure rotated model) bit
    for bit, at every width (256-column chunks included) on both schedule shapes."""
    shape, coords = _coords(dim, size)
    n = coords.shape[1]
    if size == "big":
        assert big_ok(n, num_sms())
    else:
        assert kcov_schedule(n, n, num_sms())["full_rounds"] == 0
    ell = np.array(shape, dtype=np.float64) / (2.5 if kind != "powerlaw" else 8.0)
    rot = gsi.rotation_matrix((0.6,) if dim == 2 else (0.6, -0.4, 1.1)) if rotated else None
    half = gsi.CovStructure(kind, 0.5, ell, rot, beta=0.8)
    fused = gsi.KernelCovModelMatrix([half, half], coords)
    if rotated:
        single = gsi.KernelCovModelMatrix([gsi.CovStructure(kind, 1.0, ell, rot, beta=0.8)], coords)
    else:
        single = gsi.KernelCovMatrix(kind, coords, ell, beta=0.8)
    Xall = np.random.default_rng(n).standard_normal((n, max(WIDTHS)))
    for w in WIDTHS:
        ok, Yf, Ys = _ops_equal(gsi, fused, single, Xall[:, :w])
        assert ok, (w, int(np.sum(Yf != Ys)), float(np.max(np.abs(Yf - Ys))))


# ------------------------------------------------------------------ GPU: extracted values against 160-bit references
def _term_ref(mp, kind, R2, beta):
    """(k, bound in ulps of k) of the device's argument R2 (scaled coordinates, exact)."""
    if kind == 0:
        s = mp.sqrt(R2)
        return mp.exp(-s), 2.5 + 4 * float(s), s
    if kind == 1:
        return mp.exp(-R2), 2.5, None
    if kind == 2:
        z = beta * mp.log1p(R2)
        return mp.exp(-z), 2.0 + 4 * float(z), None
    s = mp.sqrt(R2)
    if kind == 3:
        return (1 + s) * mp.exp(-s), C_ULP["matern32"] + 4 * float(kappa("matern32", s)), s
    if kind == 4:
        return (1 + s + R2 / 3) * mp.exp(-s), C_ULP["matern52"] + 4 * float(kappa("matern52", s)), s
    if s >= 1:
        return mp.mpf(0), 0.0, s
    return mp.mpf(0.5) * (1 - s) ** 2 * (2 + s), C_ULP["spherical"] + 4 * float(kappa("spherical", s)), s


def _check_values(mp, vals, refs, what):
    """vals[i] against (v, allowed absolute error) pairs; returns the largest error in ulps of v."""
    worst = 0.0
    for i, (dev, (v, allow)) in enumerate(zip(vals, refs)):
        err = abs(mp.mpf(float(dev)) - v)
        assert err <= allow, f"{what}: value {i}: {float(dev)!r} vs {mp.nstr(v, 20)}, error {mp.nstr(err, 5)} > {mp.nstr(allow, 5)}"
        if v > 0:
            e = max(int(mp.floor(mp.log(v, 2))), -1022)
            worst = max(worst, float(err / mp.ldexp(1, e - 52)))
    return worst


def arithmetic_refs(mp, structures, coords, col):
    """For every row i: (exact C[i, col] of the device's own r2_s, allowed error).  Bound (kern_eval comment):
    2^-52 sum_s c_s k_s b_s + gamma_S v, plus c_s 1.5 SPH_BAND^2 for a spherical term within the sqrt error of its
    range."""
    S = len(structures)
    us = [structure_coords(st, coords, PRE[st.kind]) for st in structures]
    out, nzero_sph, nband = [], 0, 0
    for i in range(coords.shape[1]):
        v, allow = mp.mpf(0), mp.mpf(0)
        for st, u in zip(structures, us):
            r2 = 1e-300 if st.kind not in (1, 2) else 0.0
            for k in range(u.shape[0]):
                dk = float(u[k, i] - u[k, col])
                r2 = fma(dk, dk, r2)
            k_, b, s = _term_ref(mp, st.kind, mp.mpf(r2), st.beta)
            if st.kind == 5 and abs(1 - s) <= SPH_BAND:
                nband += 1
                allow += st.sill * 1.5 * SPH_BAND ** 2
            elif st.kind == 5 and s >= 1:
                nzero_sph += 1
            v += st.sill * k_
            allow += st.sill * k_ * b * TWO52
        allow += S * U * v * (1 + 1e-6)
        out.append((v, allow))
    return out, nzero_sph, nband


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["sph_exp", "three", "four", "two_sph"])
@pytest.mark.parametrize("dim", [2, 3])
def test_model_values_ulp(gsi, dim, model):
    """Fused kernel: C[:, j] for three columns j against the 160-bit value of the device's own per-structure r2 (the
    host rebuilds u and the fma chain exactly), within the documented bound; values of all-spherical models vanish
    exactly where every structure is beyond its range."""
    mp = _mp()
    shape, coords = _coords(dim, "small")
    structures = models(dim, shape)[model]
    n = coords.shape[1]
    op = gsi.KernelCovModelMatrix(structures, coords)
    cols = [0, n // 2, n - 1]
    Cx = extract(gsi, op, n, cols)
    worst, nz = 0.0, 0
    for c, j in enumerate(cols):
        refs, nzero, _ = arithmetic_refs(mp, structures, coords, j)
        worst = max(worst, _check_values(mp, Cx[:, c], refs, f"{model} dim={dim} column {j}"))
        if model == "two_sph":
            zero = np.array([v == 0 for v, _ in refs])
            assert np.all(Cx[zero, c] == 0.0)
            nz += int(zero.sum())
    print(f"{model} dim={dim}: largest error {worst:.3f} ulp over {3 * n} values")
    if model == "two_sph":
        assert nz > 100


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [2, 3])
def test_model_symmetry_diagonal_nugget(gsi, dim):
    """Full round + ragged stream-K tail: C_hat[S, S] exactly symmetric, diagonal = sills summed in order (every k is
    exactly 1 at distance 0), values in [0, sum of sills], and the nugget added on the diagonal only."""
    shape, coords = _coords(dim, "big")
    n = coords.shape[1]
    structures = models(dim, shape)["four"]
    S = sample_rows(n)
    Cs = np.ascontiguousarray(extract(gsi, gsi.KernelCovModelMatrix(structures, coords), n, S).T)
    Css = Cs[:, S]
    assert np.array_equal(Css, Css.T)
    diag = 0.0
    for st in structures:
        diag = diag + st.sill
    assert np.all(np.diag(Css) == diag)
    assert np.all(Cs >= 0.0) and np.all(Cs <= diag)
    E = unit_columns(n, S)
    Y = apply_dev(gsi, gsi.KernelCovModelMatrix(structures, coords, nugget=0.3), E).T
    unit = E.T.astype(bool)
    assert np.array_equal(Y[~unit], Cs[~unit])
    assert np.all(Y[unit] == diag + 0.3)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [2, 3])
def test_model_values_width_and_schedule_independent(gsi, dim):
    shape, coords = _coords(dim, "big")
    n = coords.shape[1]
    op = gsi.KernelCovModelMatrix(models(dim, shape)["three"], coords)
    ctx = op.ctx
    R = np.random.default_rng(3).choice(n, 1024, replace=False)
    special = [0, n - 1] + [a for a, _ in kcov_schedule(n, n, num_sms())["tail_tiles"]]
    R[:len(special)] = special
    ref = extract(gsi, op, n, R)
    for w in WIDTHS[:-1]:
        assert np.array_equal(extract(gsi, op, n, R[:w]), ref[:, :w]), w
    keys = ("kcov.sweep_groups", "kcov.sweep_div", "kcov.window", "kcov.epoch_shift")
    saved = {k: ctx.get_option(k) for k in keys}
    try:
        for groups, div, window in ((1, 0, 0), (8, -3, 0), (1, 0, 2)):
            ctx.set_option("kcov.sweep_groups", groups)
            ctx.set_option("kcov.sweep_div", div)
            ctx.set_option("kcov.epoch_shift", 2)
            ctx.set_option("kcov.window", window)
            for w in (27, 256):
                assert np.array_equal(extract(gsi, op, n, R[:w]), ref[:, :w]), (groups, div, window, w)
    finally:
        for k, v in saved.items():
            ctx.set_option(k, v)


# ------------------------------------------------------------------ GPU: products
_CACHE = {}


def model_op(path, dim, size):
    """(operator, sampled rows S, C_hat[S, :]) of the three-structure rotated model: fused kernel on jittered points or
    signed lattice table on the grid."""
    key = (path, dim, size)
    if key not in _CACHE:
        g = get_gsi()
        if path == "fused":
            shape, coords = _coords(dim, size)
            op = g.KernelCovModelMatrix(models(dim, shape)["three"], coords)
        else:
            shape = grid_shape(dim, size)
            op = g.GridKernelCovModelMatrix(models(dim, shape)["three"], shape)
        n = op.shape[0]
        S = sample_rows(n)
        _CACHE[key] = (op, S, np.ascontiguousarray(extract(g, op, n, S).T))
    return _CACHE[key]


def _bound_check(Y, ref, bound, what):
    err = np.abs(Y - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {bad.sum()} elements out of bound, first at {tuple(np.argwhere(bad)[0])}; "
                           f"max err/bound {np.nanmax(err / bound):.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("size", ["small", "big"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("path", ["fused", "signed"])
def test_model_product_bound(gsi, path, dim, size, cols):
    """Y = C X on sampled rows within 2 gamma_n (|C_hat| |X|) of C_hat X, after the same shape ran on a NaN X."""
    op, S, Cs = model_op(path, dim, size)
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
    _bound_check(Y, Cs @ X, 2 * gamma * (np.abs(Cs) @ np.abs(X)), f"{path} dim={dim} n={n} cols={cols}")


# ------------------------------------------------------------------ GPU: signed lattice table
TABLE_BOUND = {0: lambda a: 4 + 4 * a, 1: lambda a: 4 + 4 * a, 2: lambda a: 4 + 4 * a}


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["sph_exp", "three", "four"])
@pytest.mark.parametrize("dim", [2, 3])
def test_signed_table_values(gsi, dim, model):
    """Signed table: C[:, centre] (offsets of both signs on every axis) against the 160-bit model value of the host's
    rotated offsets; per term the table bounds of the single kinds (4 + 4 arg, or those of tests/test_gpu_matern.py),
    plus 2 S roundings of the host's sum.  The extracted block is exactly symmetric."""
    mp = _mp()
    shape, spacing = {2: ((41, 33), (0.7, 1.3)), 3: ((15, 13, 11), (1.1, 0.8, 1.6))}[dim]
    L = np.array(shape) * np.array(spacing)
    structures = models(dim, L)[model]
    op = gsi.GridKernelCovModelMatrix(structures, shape, spacing=spacing)
    n = int(np.prod(shape))
    lat = np.array(np.unravel_index(np.arange(n), shape, order="F"))
    centre = int(np.ravel_multi_index(tuple(s // 2 for s in shape), shape, order="F"))
    col = extract(gsi, op, n, [centre])[:, 0]
    refs = []
    for i in range(n):
        x = (lat[:, i] - lat[:, centre]).astype(np.float64) * np.array(spacing)
        v, allow = mp.mpf(0), mp.mpf(0)
        for st in structures:
            u = structure_coords(st, x[:, None], 1.0)[:, 0]
            R2 = sum(mp.mpf(float(uk)) ** 2 for uk in u)
            if st.kind in (0, 1, 2):
                arg = {0: mp.sqrt(R2), 1: R2 / 2, 2: st.beta * mp.log1p(R2)}[st.kind]
                k_, b = mp.exp(-arg), 4 + 4 * float(arg)
            else:
                k_, b, s = _term_ref(mp, st.kind, R2 * mp.mpf(PRE[st.kind]) ** 2 if st.kind != 5 else R2, st.beta)
                if st.kind == 5 and abs(1 - s) <= SPH_BAND:
                    allow += st.sill * 1.5 * SPH_BAND ** 2
            v += st.sill * k_
            allow += st.sill * k_ * b * TWO52
        allow += 2 * len(structures) * U * v * (1 + 1e-6)
        refs.append((v, allow))
    worst = _check_values(mp, col, refs, f"signed table {model} dim={dim}")
    print(f"signed table {model} dim={dim}: largest error {worst:.3f} ulp over {n} values")
    S = sample_rows(n, k=40)
    Cs = extract(gsi, op, n, S)[S]
    assert np.array_equal(Cs, Cs.T)


GRID_SHAPES = [(40, 25), (1, 60), (60, 1), (10, 10, 10), (12, 1, 9), (1, 8, 7), (9, 7, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [1, 64, 300])
@pytest.mark.parametrize("shape", GRID_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_signed_table_matches_arithmetic(gsi, shape, cols):
    """Rotated model: grid operator (signed table) against the fused kernel on the same lattice points, including axes
    of length 1: extracted values within 1e-12 and products within both rounding bounds plus their difference."""
    dim = len(shape)
    structures = models(dim, [max(s, 4) for s in shape])["three"]
    coords = oracle.grid_coords(shape)
    n = coords.shape[1]
    S = sample_rows(n, k=min(24, n - 8))
    opg = gsi.GridKernelCovModelMatrix(structures, shape)
    opa = gsi.KernelCovModelMatrix(structures, coords)
    Cg = np.ascontiguousarray(extract(gsi, opg, n, S).T)
    Ca = np.ascontiguousarray(extract(gsi, opa, n, S).T)
    assert np.max(np.abs(Cg - Ca)) < 1e-12
    X = np.random.default_rng(cols + 5).standard_normal((n, cols))
    Yg = apply_dev(gsi, opg, X)[S]
    Ya = apply_dev(gsi, opa, X)[S]
    gamma = n * U / (1 - n * U)
    aX = np.abs(X)
    _bound_check(Yg, Ya, 2 * gamma * ((np.abs(Cg) + np.abs(Ca)) @ aX) + np.abs(Cg - Ca) @ aX,
                 f"grid vs arithmetic {shape} cols={cols}")


# ------------------------------------------------------------------ GPU: randsvd parity
RSVD_GRID, RSVD_K = (60, 50), 50


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 2])
@pytest.mark.parametrize("path", ["arithmetic", "grid"])
def test_randsvd_parity(gsi, path, q):
    """gsi.randsvd on the rotated two-structure model (fused kernel or signed table) against oracle.randsvd on the
    dense reference; sigma_K / sigma_{K+1} - 1 = 0.118 for this case (host eigvalsh)."""
    structures = models(2, RSVD_GRID)["sph_exp"]
    coords = oracle.grid_coords(RSVD_GRID)
    C = model_dense(structures, coords)
    n, K, p = C.shape[0], RSVD_K, 10
    Omega = np.random.default_rng(q).standard_normal((n, K + p))
    Zref = oracle.randsvd(C, Omega, K, p, q)
    if path == "grid":
        op = gsi.GridKernelCovModelMatrix(structures, RSVD_GRID)
    else:
        op = gsi.KernelCovModelMatrix(structures, coords)
    Z, S = gsi.randsvd(op, K, p, q, Omega=Omega, normaliser=gsi.NORMALISER_LU_REF, return_singular_values=True)
    c = oracle.compare_Z(Z, Zref, K)
    assert c["tail_zero"]
    assert c["sv_rel"] < SV_TOL and c["sine"] < SINE_TOL, c
    assert np.max(np.abs(S[:K] - oracle.singvals_from_Z(Zref, K)) / S[:K]) < SV_TOL


# ------------------------------------------------------------------ GPU: error paths
def _call(gsi, grid, d=2, nstruct=1, kinds=(0,), sills=(1.0,), ranges=None, rot=None, betas=None, coords=True,
          dims=(4, 3), null=None):
    ctx = gsi.default_context()
    lib = ctx._lib
    pd = C.POINTER(C.c_double)
    kinds_a = (C.c_int32 * max(1, len(kinds)))(*kinds)
    sills_a = np.ascontiguousarray(sills, dtype=np.float64)
    ranges_a = np.ascontiguousarray(np.ones(max(1, len(sills)) * max(d, 1)) if ranges is None else ranges, dtype=np.float64)
    rot_a = None if rot is None else np.ascontiguousarray(rot, dtype=np.float64)
    xs = np.ascontiguousarray(np.arange(3.0 * 12))
    h = C.c_void_p()
    args = dict(kinds=kinds_a, sills=sills_a.ctypes.data_as(pd), ranges=ranges_a.ctypes.data_as(pd),
                rot=None if rot_a is None else rot_a.ctypes.data_as(pd), out=C.byref(h))
    if null:
        args[null] = None
    if grid:
        dims_a = (C.c_int64 * 3)(*dims, *([1] * (3 - len(dims))))
        spacing = np.ones(3)
        st = lib.gsi_op_kernelcov_model_grid(ctx._h, d, dims_a, spacing.ctypes.data_as(pd), nstruct, args["kinds"],
                                             args["sills"], args["ranges"], args["rot"], None, 0.0, 0,
                                             int(np.prod(dims)), args["out"])
    else:
        st = lib.gsi_op_kernelcov_model(ctx._h, d, 12, None if null == "coords" else xs.ctypes.data_as(pd), nstruct,
                                        args["kinds"], args["sills"], args["ranges"], args["rot"], None, 0.0, 0, 12,
                                        args["out"])
    if st == 0:
        lib.gsi_op_free(h)
    return st, h.value


BAD = {
    "nstruct_0": dict(nstruct=0),
    "nstruct_5": dict(nstruct=5, kinds=(0,) * 5, sills=(1.0,) * 5),
    "kind_6": dict(kinds=(6,)), "kind_-1": dict(kinds=(-1,)), "kind_13": dict(kinds=(13,)),
    "kind_14": dict(kinds=(14,)), "kind_15": dict(kinds=(15,)),
    "sill_0": dict(sills=(0.0,)), "sill_neg": dict(sills=(-1.0,)), "sill_nan": dict(sills=(np.nan,)),
    "sill_inf": dict(sills=(np.inf,)),
    "range_0": dict(ranges=(1.0, 0.0)), "range_neg": dict(ranges=(-2.0, 1.0)), "range_nan": dict(ranges=(1.0, np.nan)),
    "rot_nan": dict(rot=(1.0, 0.0, np.nan, 1.0)), "rot_inf": dict(rot=(np.inf, 0.0, 0.0, 1.0)),
    "rot_scaled": dict(rot=(1.0 + 1e-11, 0.0, 0.0, 1.0)), "rot_shear": dict(rot=(1.0, 0.0, 1e-6, 1.0)),
    "second_sill": dict(nstruct=2, kinds=(0, 1), sills=(1.0, -0.5), ranges=np.ones(4)),
    "null_kinds": dict(null="kinds"), "null_sills": dict(null="sills"), "null_ranges": dict(null="ranges"),
    "null_out": dict(null="out"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [False, True], ids=["arithmetic", "grid"])
@pytest.mark.parametrize("case", sorted(BAD))
def test_rejects_invalid_model(gsi, case, grid):
    st, h = _call(gsi, grid, **BAD[case])
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h, (case, st, gsi._lib.load().gsi_last_error_string())


@pytest.mark.gpu
def test_rejects_null_coords_and_unsupported(gsi):
    st, h = _call(gsi, False, null="coords")
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h
    for grid in (False, True):
        for d in (0, 4):
            st, h = _call(gsi, grid, d=d)
            assert st == gsi._lib.ERR_UNSUPPORTED and not h, (grid, d)
    rot2 = np.array([[0.0, 1.0], [-1.0, 0.0]]).ravel(order="F")
    # signed tables of 2^31 entries or more are refused before anything is allocated (the points themselves fit)
    st, h = _call(gsi, True, d=2, rot=rot2, dims=(40000, 30000))
    assert st == gsi._lib.ERR_UNSUPPORTED and not h
    R3 = gsi.rotation_matrix((0.3, 0.2, 0.1)).ravel(order="F")
    st, h = _call(gsi, True, d=3, rot=R3, ranges=np.ones(3), dims=(1300, 1300, 1200))
    assert st == gsi._lib.ERR_UNSUPPORTED and not h
    # the valid call of the same helper succeeds on both paths
    for grid in (False, True):
        st, h = _call(gsi, grid, rot=rot2)
        assert st == 0


# ------------------------------------------------------------------ GPU: two ranks
@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_two_ranks_row_sharded(gsi):
    """A row-sharded model operator (fused kernel and signed table) on two ranks gives the rows of the one-rank
    product within rounding (the stream-K split of a rank's rows differs, so the sums may be ordered differently)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29541", os.path.join(ROOT, "tests", "dist_kcov_model_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=540, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        for path in ("fused", "signed"):
            shape = (70, 60)
            structures = models(2, shape)["three"]
            coords = oracle.grid_coords(shape)
            n = coords.shape[1]
            X = np.random.default_rng(1).standard_normal((n, 33))
            op = (gsi.KernelCovModelMatrix(structures, coords) if path == "fused"
                  else gsi.GridKernelCovModelMatrix(structures, shape))
            Y1 = apply_dev(gsi, op, X)
            bound = 4 * n * U * (np.abs(model_dense(structures, coords)) @ np.abs(X)) + 1e-300
            for rank in range(2):
                f = np.load(os.path.join(tmp, f"{path}_rank{rank}.npz"))
                r0, Y2 = int(f["row0"]), f["Y"]
                _bound_check(Y2, Y1[r0:r0 + Y2.shape[0]], bound[r0:r0 + Y2.shape[0]], f"{path} rank {rank}")
