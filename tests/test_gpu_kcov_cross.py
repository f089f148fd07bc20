"""Cross-covariance operator C(T, S) between two point sets (gsi_op_kernelcov_cross / gsi_op_kernelcov_cross_grid), tested
to the standard of tests/test_gpu_product_exact.py and tests/test_gpu_kcov_model.py, whose helpers are reused:

* CPU: the dense cross reference below is the (T, S) block of the model's dense matrix on the union of the two sets;
  the all-SM launch shape of the cross products (mirrored below) keeps the stream-K tail invariants over a sweep of
  shapes: the grid, at most two segments per CTA, at most KF_MAX_PIECES pieces per tile, every k-tile unit once.
* GPU, bit for bit: every extracted C(T, S) value equals the (T, S) block of the square operator on [T S] (nugget 0), in
  both directions, for every single kind, 2-4-structure rotated models, the unsigned and signed lattice tables and
  d = 1..3; with T = S (same order) the cross products equal the square operator's at every width where both launch
  the same grid; A' X equals the product of the cross operator with the sets swapped.
* GPU, within bounds: |Y - C X| <= 2 gamma_k (|C| |X|) element by element in both directions at every width, on a full
  round with a ragged tail, short-wide all-SM tails with CTAs that own no work, m = 1, n = 1 and n not a multiple of
  32, each after the same shape ran on an all-NaN X; randsvd parity with oracle.randsvd for m > n and m < n; the error
  paths; two ranks.
"""
import ctypes as C
import functools
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import oracle
from gpu_util import gsi  # noqa: F401
from test_gpu_kcov_model import KINDS, _bound_check, model_dense, models
from test_gpu_product_exact import U, WIDTHS, _cdiv, apply_dev, big_ok, grid_shape, num_sms, unit_columns
from test_gpu_randsvd import SINE_TOL, SV_TOL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G      # noqa: E402  (importing needs no GPU)

KF_MAX_PIECES = 160       # csrc/kcov_gemm.cu


# ------------------------------------------------------------------ host references
def cross_dense(structures, targets, sources):
    """Dense reference C(T, S)[i, j] = sum_s sill_s k_s(t_i, s_j) (no nugget)."""
    return model_dense(structures, np.concatenate([targets, sources], axis=1))[:targets.shape[1], targets.shape[1]:]


def cross_schedule(rows, k, sms):
    """launch_kcov for a cross-covariance product (rows x k, all-SM grid): the persistent grid is never capped at the row
    groups; full rounds of 64-row tiles, then a stream-K tail of the leftover tiles in shares of tail_u k-tile units."""
    total_rg = _cdiv(rows, 16)
    grid = sms
    full_rounds = total_rg // (4 * grid)
    tail_rg0 = full_rounds * 4 * grid
    tail_tiles = _cdiv(total_rg - tail_rg0, 4)
    nkt = _cdiv(k, 32)
    tail_u = _cdiv(tail_tiles * nkt, grid) if tail_tiles else 0
    tiles = [(tail_rg0 * 16 + 64 * t, min(rows, tail_rg0 * 16 + 64 * t + 64)) for t in range(tail_tiles)]
    busy = _cdiv(tail_tiles * nkt, tail_u) if tail_u else 0
    return dict(grid=grid, full_rounds=full_rounds, tail_tiles=tiles, tail_u=tail_u, nkt=nkt,
                empty_ctas=grid - busy if tail_u else 0)


def tail_shares(s):
    """The kernel's split of the tail (per CTA: segments (tile, k0, len, slot)) and the fix-up's pieces per tile."""
    nkt, tail_u, grid = s["nkt"], s["tail_u"], s["grid"]
    units = len(s["tail_tiles"]) * nkt
    segs = []
    for b in range(grid):
        u0, u1 = min(b * tail_u, units), min(b * tail_u + tail_u, units)
        tA, kA = divmod(u0, nkt)
        lenA = min(u1 - u0, nkt - kA)
        lenB = (u1 - u0) - lenA
        mine = []
        if lenA > 0:
            mine.append((tA, kA, lenA, 2 * b))
        if lenB > 0:
            mine.append((tA + 1, 0, lenB, 2 * b + 1))
        segs.append(mine)
    pieces = []
    for t in range(len(s["tail_tiles"])):
        ulo, uhi = t * nkt, t * nkt + nkt
        b_first, b_last = ulo // tail_u, min((uhi - 1) // tail_u, grid - 1)
        pieces.append([2 * b + (0 if t == (b * tail_u) // nkt else 1) for b in range(b_first, b_last + 1)])
    return segs, pieces


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("model", ["single", "sph_exp", "four"])
def test_cross_dense_is_a_block_of_the_union(model, d):
    rng = np.random.default_rng(d)
    T, S = rng.uniform(0, 10, (d, 70)), rng.uniform(0, 10, (d, 45))
    L = np.full(max(d, 2), 10.0)
    if d == 1 or model == "single":
        structures = [G.CovStructure("matern52", 1.3, np.full(d, 2.5))]
    else:
        structures = models(d, L[:d])[model]
    U_ = np.concatenate([T, S], axis=1)
    full = model_dense(structures, U_)
    Cx = cross_dense(structures, T, S)
    assert Cx.shape == (70, 45)
    assert np.array_equal(Cx, full[:70, 70:])
    assert np.array_equal(cross_dense(structures, S, T), full[70:, :70])
    assert np.allclose(Cx, cross_dense(structures, S, T).T, rtol=1e-15, atol=0)


SCHED_SHAPES = [(r, k) for r in (1, 16, 17, 64, 200, 1000, 2367, 9472, 9473, 9536, 20000, 38000, 200704)
                for k in (1, 31, 32, 33, 1000, 20000, 200704)]


@pytest.mark.parametrize("sms", [148, 132, 1])
def test_cross_schedule_invariants(sms):
    """All-SM launch shape: tail tiles <= grid, shares of at most two segments, <= KF_MAX_PIECES pieces per tile, the
    fix-up's slot of every piece is the one its CTA wrote, and every (tile, k-tile) unit is covered exactly once."""
    for rows, k in SCHED_SHAPES:
        s = cross_schedule(rows, k, sms)
        assert s["grid"] == sms
        tiles, nkt = s["tail_tiles"], s["nkt"]
        assert len(tiles) <= s["grid"]
        rg = _cdiv(rows, 16)                      # a full round may end in the ragged last row group
        assert rg >= 4 * sms * s["full_rounds"]
        if not tiles:
            assert rg == 4 * sms * s["full_rounds"]
            continue
        assert tiles[0][0] == 64 * sms * s["full_rounds"] and tiles[-1][1] == rows
        assert s["tail_u"] <= nkt
        segs, pieces = tail_shares(s)
        cover = {}
        for b, mine in enumerate(segs):
            assert len(mine) <= 2
            for t, k0, ln, slot in mine:
                assert 0 <= t < len(tiles) and 0 <= k0 and k0 + ln <= nkt
                for kt in range(k0, k0 + ln):
                    assert (t, kt) not in cover
                    cover[(t, kt)] = slot
        assert len(cover) == len(tiles) * nkt
        for t, pl in enumerate(pieces):
            assert 1 <= len(pl) <= KF_MAX_PIECES
            assert sorted(pl) == sorted({cover[(t, kt)] for kt in range(nkt)})


def test_cross_exports():
    assert G.KernelCrossCovMatrix.symmetric is False and G.GridKernelCrossCovMatrix.symmetric is False
    assert "gsi_op_kernelcov_cross" in G._lib.SIGNATURES and "gsi_op_kernelcov_cross_grid" in G._lib.SIGNATURES


# ------------------------------------------------------------------ GPU helpers
def _jitter(c, seed):
    return c + np.random.default_rng(seed).uniform(-0.3, 0.3, c.shape)


def extract_cols(gsi, op, rows):
    """C(T, S)[:, rows] (unit columns of size n)."""
    return apply_dev(gsi, op, unit_columns(op.shape[1], rows))


def extract_rows(gsi, op, rows):
    """C(T, S)[rows, :] = (C' e_rows)' through the transposed product."""
    return apply_dev_t(gsi, op, unit_columns(op.shape[0], rows)).T


def apply_dev_t(gsi, op, X):
    ctx = op.ctx
    Xd = gsi.DeviceMatrix.from_host(ctx, X)
    try:
        Yd = op.apply(Xd, trans=True)
        try:
            return Yd.numpy()
        finally:
            Yd.free()
    finally:
        Xd.free()


def _point_sets(d, m, n, seed):
    """m targets on a jittered lattice and n sources scattered over the same box."""
    shape = {1: (m,), 2: (max(1, m // 20), 20), 3: (max(1, m // 64), 8, 8)}[d] if m >= 64 else (m,) + (1,) * (d - 1)
    T = _jitter(oracle.grid_coords(shape), seed)[:, :m]
    if T.shape[1] < m:
        T = np.concatenate([T, np.random.default_rng(seed).uniform(0, 8, (d, m - T.shape[1]))], axis=1)
    box = np.array(shape, dtype=np.float64)[:, None]
    S = np.random.default_rng(seed + 1).uniform(0, 1, (d, n)) * box
    return T, S, np.array(shape, dtype=np.float64)


def _check_against_square(gsi, cross, square, m, n, rng):
    """Extracted C(T, S) columns / C(S, T) columns against the square operator on [T S] (or on the whole grid through
    index maps ti / si), bit for bit."""
    sq_n = square.shape[0]
    ti, si = cross._ti, cross._si
    cols = sorted(set([0, n - 1] + rng.choice(n, min(n, 12), replace=False).tolist()))
    rows = sorted(set([0, m - 1] + rng.choice(m, min(m, 12), replace=False).tolist()))
    Cx = extract_cols(gsi, cross, cols)                             # m x |cols|
    Cs = apply_dev(gsi, square, unit_columns(sq_n, si[cols]))       # sq_n x |cols|
    assert np.array_equal(Cx, Cs[ti]), ("C(T,S)", int(np.sum(Cx != Cs[ti])))
    Ct = apply_dev_t(gsi, cross, unit_columns(m, rows))             # n x |rows| = C(S, T)[:, rows]
    Cs2 = apply_dev(gsi, square, unit_columns(sq_n, ti[rows]))
    assert np.array_equal(Ct, Cs2[si]), ("C(S,T)", int(np.sum(Ct != Cs2[si])))


def _arith_pair(gsi, structures, T, S):
    cross = gsi.KernelCrossCovMatrix(structures, T, S)
    square = gsi.KernelCovModelMatrix(structures, np.concatenate([T, S], axis=1))
    m = T.shape[1]
    cross._ti, cross._si = np.arange(m), m + np.arange(S.shape[1])
    return cross, square


# ------------------------------------------------------------------ GPU: bit-exact values
@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_values_single_kind_equal_square(gsi, kind, d):
    """Every single kind on the arithmetic path (one structure: the specialised kernel, sigma2 = the sill)."""
    T, S, L = _point_sets(d, 700, 333, 10 * d)
    ell = L / (3.0 if kind == "spherical" else 2.0)
    cross, square = _arith_pair(gsi, [gsi.CovStructure(kind, 1.7, ell, beta=0.8)], T, S)
    _check_against_square(gsi, cross, square, T.shape[1], S.shape[1], np.random.default_rng(d))


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["sph_exp", "three", "four", "two_sph"])
@pytest.mark.parametrize("d", [2, 3])
def test_values_fused_model_equal_square(gsi, d, model):
    """2-4-structure rotated models in the fused KC_KIND_MODEL kernel (row coordinates staged in shared memory)."""
    T, S, L = _point_sets(d, 900, 517, 3 + d)
    cross, square = _arith_pair(gsi, models(d, L)[model], T, S)
    _check_against_square(gsi, cross, square, T.shape[1], S.shape[1], np.random.default_rng(5))


GRID_CASES = {1: (300,), 2: (41, 33), 3: (15, 13, 11)}


@pytest.mark.gpu
@pytest.mark.parametrize("table", ["unsigned", "signed"])
@pytest.mark.parametrize("d", [1, 2, 3])
def test_values_grid_equal_square(gsi, d, table):
    """Lattice tables: targets / sources given by linear indices (unordered, repeated) against the square grid
    operator of the same model; the signed table is a rotated model (d = 1 is unsigned whatever the rotation)."""
    shape = GRID_CASES[d]
    nodes = int(np.prod(shape))
    rng = np.random.default_rng(d)
    ti = rng.permutation(nodes)[: nodes // 2]
    si = np.concatenate([rng.choice(nodes, 150, replace=False), [0, nodes - 1, 0]])
    L = np.array(shape, dtype=np.float64)
    if table == "signed" and d >= 2:
        structures = models(d, L)["three"]
    else:
        structures = [gsi.CovStructure("exponential", 0.7, L / 3), gsi.CovStructure("spherical", 1.1, L / 2)]
    cross = gsi.GridKernelCrossCovMatrix(structures, shape, targets=ti, sources=si, spacing=0.9)
    square = gsi.GridKernelCovModelMatrix(structures, shape, spacing=0.9)
    cross._ti, cross._si = ti, si
    _check_against_square(gsi, cross, square, ti.size, si.size, rng)
    # every node in order (NULL index lists) on both sides: the square operator itself
    full = gsi.GridKernelCrossCovMatrix(structures, shape, spacing=0.9)
    assert full.shape == (nodes, nodes)
    full._ti = full._si = np.arange(nodes)
    _check_against_square(gsi, full, square, nodes, nodes, rng)


# ------------------------------------------------------------------ GPU: bit-exact products
@functools.lru_cache(maxsize=None)
def _big_points(dim):
    """Jittered points of the big schedule shape (a full round plus a ragged stream-K tail) and a model."""
    shape = grid_shape(dim, "big")
    coords = _jitter(oracle.grid_coords(shape), 7)
    return shape, coords


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["single", "fused", "table"])
@pytest.mark.parametrize("dim", [2, 3])
def test_same_sets_equal_square_products(gsi, dim, path):
    """T = S in the same order, at least 4 x SMs row groups (the square and the cross launch the same grid): every product
    is the square operator's bit for bit, at every width."""
    shape, coords = _big_points(dim)
    n = coords.shape[1]
    assert big_ok(n, num_sms())
    L = np.array(shape, dtype=np.float64)
    if path == "single":
        st = [gsi.CovStructure("exponential", 1.0, L / 2.5)]
        cross, square = gsi.KernelCrossCovMatrix(st, coords, coords), gsi.KernelCovMatrix("exponential", coords, L / 2.5)
    elif path == "fused":
        st = models(dim, L)["three"]
        cross, square = gsi.KernelCrossCovMatrix(st, coords, coords), gsi.KernelCovModelMatrix(st, coords)
    else:
        st = models(dim, L)["three"]
        cross, square = gsi.GridKernelCrossCovMatrix(st, shape), gsi.GridKernelCovModelMatrix(st, shape)
    Xall = np.random.default_rng(n).standard_normal((n, max(WIDTHS)))
    for w in WIDTHS:
        X = Xall[:, :w]
        Yc, Ys = apply_dev(gsi, cross, X), apply_dev(gsi, square, X)
        assert np.array_equal(Yc, Ys), (w, int(np.sum(Yc != Ys)))
        Yt = apply_dev_t(gsi, cross, X)
        assert np.array_equal(Yt, Ys), ("transposed", w, int(np.sum(Yt != Ys)))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "table"])
def test_transpose_equals_swapped_operator(gsi, path):
    """A(T, S)' X = A(S, T) X bit for bit at every width (the same rows, columns and launch)."""
    shape = (70, 40)
    L = np.array(shape, dtype=np.float64)
    st = models(2, L)["sph_exp"]
    rng = np.random.default_rng(2)
    if path == "fused":
        T, S, _ = _point_sets(2, 2800, 1300, 9)
        A, B = gsi.KernelCrossCovMatrix(st, T, S), gsi.KernelCrossCovMatrix(st, S, T)
    else:
        nodes = int(np.prod(shape))
        ti, si = rng.choice(nodes, 2100, replace=False), rng.choice(nodes, 777, replace=False)
        A = gsi.GridKernelCrossCovMatrix(st, shape, targets=ti, sources=si)
        B = gsi.GridKernelCrossCovMatrix(st, shape, targets=si, sources=ti)
    m = A.shape[0]
    assert B.shape == A.shape[::-1]
    Xall = rng.standard_normal((m, max(WIDTHS)))
    for w in WIDTHS:
        Ya, Yb = apply_dev_t(gsi, A, Xall[:, :w]), apply_dev(gsi, B, Xall[:, :w])
        assert np.array_equal(Ya, Yb), (w, int(np.sum(Ya != Yb)))


# ------------------------------------------------------------------ GPU: element-wise product bounds
def _bound_shapes():
    sms = num_sms()
    big = 64 * sms + 97                           # a full round of row tiles plus a ragged tail
    return {
        "round_ragged": (big, 1501),              # trans = 0: full round + tail; trans = 1: 1501 rows, all-SM tail
        "short_wide": (200, 1000),                # 13 row groups over the whole grid: CTAs with no work
        "short_wide_long": (37, 160 * sms - 5),   # few rows, long k: 5 k-tiles for every CTA of the tail
        "m1": (1, 3001),
        "n1": (2999, 1),
        "n_ragged": (1200, 4129),                 # n not a multiple of 32 (k range and rows)
    }


_BOUND_CACHE = {}


def bound_case(name):
    """(operator, sampled target rows RT, C[RT, :], sampled source rows RS, C'[RS, :])."""
    if name not in _BOUND_CACHE:
        import gsi_b200 as g
        m, n = _bound_shapes()[name]
        T, S, L = _point_sets(3, m, n, 17)
        op = g.KernelCrossCovMatrix(models(3, L)["three"], T, S)
        sms = num_sms()

        def sample(rows, k):
            s = cross_schedule(rows, k, sms)
            r = {0, rows - 1, min(15, rows - 1), min(16, rows - 1)}
            for a, b in s["tail_tiles"]:
                r |= {a, b - 1}
            r |= set(np.random.default_rng(rows).choice(rows, min(rows, 20), replace=False).tolist())
            return sorted(r)
        RT, RS = sample(m, n), sample(n, m)
        _BOUND_CACHE[name] = (op, RT, extract_rows(g, op, RT), RS, np.ascontiguousarray(extract_cols(g, op, RS).T))
    return _BOUND_CACHE[name]


@pytest.mark.gpu
def test_bound_shapes_cover_the_schedules(gsi):
    sms = num_sms()
    sh = _bound_shapes()
    s = cross_schedule(*sh["round_ragged"], sms)
    assert s["full_rounds"] == 1 and s["tail_tiles"] and sh["round_ragged"][0] % 16 != 0
    s = cross_schedule(*sh["short_wide"], sms)
    assert s["full_rounds"] == 0 and s["empty_ctas"] > 0
    s = cross_schedule(*sh["short_wide_long"], sms)
    assert s["empty_ctas"] == 0 and s["tail_u"] < s["nkt"]
    assert sh["n_ragged"][1] % 32 != 0


@pytest.mark.gpu
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("trans", [False, True], ids=["CX", "CtX"])
@pytest.mark.parametrize("shape", ["round_ragged", "short_wide", "short_wide_long", "m1", "n1", "n_ragged"])
def test_cross_product_bound(gsi, shape, trans, cols):
    """Y = C X (or C' X) on sampled rows within 2 gamma_k (|C_hat| |X|) of C_hat X, after the same shape ran on a NaN X."""
    op, RT, CT, RS, CS = bound_case(shape)
    m, n = op.shape
    k, rows, Cr = (m, RS, CS) if trans else (n, RT, CT)
    run = apply_dev_t if trans else apply_dev
    run(gsi, op, np.full((k, cols), np.nan))
    X = np.random.default_rng(cols + 7 * trans).standard_normal((k, cols))
    Y = run(gsi, op, X)[rows]
    gamma = k * U / (1 - k * U)
    _bound_check(Y, Cr @ X, 2 * gamma * (np.abs(Cr) @ np.abs(X)), f"{shape} trans={trans} m={m} n={n} cols={cols}")


# ------------------------------------------------------------------ GPU: randsvd parity
RSVD_GRID, RSVD_K, RSVD_NSRC = (60, 50), 20, 400


@pytest.mark.gpu
@pytest.mark.parametrize("q", [0, 2])
@pytest.mark.parametrize("orient", ["m_gt_n", "m_lt_n"])
def test_randsvd_parity(gsi, orient, q):
    """gsi.randsvd of C(grid, scattered points) (m > n) and of C(points, grid) (m < n) against oracle.randsvd on the
    dense reference; sigma_K / sigma_{K+1} - 1 = 0.114 (host SVD)."""
    structures = models(2, RSVD_GRID)["sph_exp"]
    grid = oracle.grid_coords(RSVD_GRID)
    pts = np.random.default_rng(11).uniform(0, 1, (2, RSVD_NSRC)) * (np.array(RSVD_GRID, dtype=np.float64) - 1)[:, None]
    T, S = (grid, pts) if orient == "m_gt_n" else (pts, grid)
    A = cross_dense(structures, T, S)
    n, K, p = A.shape[1], RSVD_K, 10
    Omega = np.random.default_rng(q).standard_normal((n, K + p))
    Zref = oracle.randsvd(A, Omega, K, p, q)
    op = gsi.KernelCrossCovMatrix(structures, T, S)
    Z, Sv = gsi.randsvd(op, K, p, q, Omega=Omega, normaliser=gsi.NORMALISER_LU_REF, return_singular_values=True)
    assert Z.shape == (n, K + p)
    c = oracle.compare_Z(Z, Zref, K)
    assert c["tail_zero"]
    assert c["sv_rel"] < SV_TOL and c["sine"] < SINE_TOL, c
    assert np.max(np.abs(Sv[:K] - oracle.singvals_from_Z(Zref, K)) / Sv[:K]) < SV_TOL


# ------------------------------------------------------------------ GPU: error paths
def _call(gsi, grid, d=2, m=5, n=4, row0=0, mloc=None, tidx="ok", sidx="ok", dims=(4, 3), nstruct=1, sills=(1.0,),
          rot=None, null=None):
    ctx = gsi.default_context()
    lib = ctx._lib
    pd, pi = C.POINTER(C.c_double), C.POINTER(C.c_int64)
    mloc = m if mloc is None else mloc
    kinds = (C.c_int32 * 1)(0)
    sills_a = np.ascontiguousarray(sills, dtype=np.float64)
    ranges = np.ones(max(1, d) * max(1, nstruct))
    rot_a = None if rot is None else np.ascontiguousarray(rot, dtype=np.float64)
    pts = np.ascontiguousarray(np.arange(3.0 * 64))
    h = C.c_void_p()
    a = dict(kinds=kinds, sills=sills_a.ctypes.data_as(pd), ranges=ranges.ctypes.data_as(pd), out=C.byref(h),
             targets=pts.ctypes.data_as(pd), sources=pts.ctypes.data_as(pd))
    rotp = None if rot_a is None else rot_a.ctypes.data_as(pd)
    if grid:
        nodes = max(1, int(np.prod(dims)))

        def index_list(idx, count):
            """"ok": valid node indices; None: a NULL list; otherwise the given indices."""
            if idx is None:
                return None
            return np.ascontiguousarray(np.arange(max(count, 0)) % nodes if isinstance(idx, str) else idx, dtype=np.int64)
        ti, si = index_list(tidx, m), index_list(sidx, n)
        dims_a = (C.c_int64 * 3)(*dims, *([1] * (3 - len(dims))))
        spacing = np.ones(3)
        a.update(dims=dims_a, spacing=spacing.ctypes.data_as(pd), target_idx=None if ti is None else ti.ctypes.data_as(pi),
                 source_idx=None if si is None else si.ctypes.data_as(pi))
        if null:
            a[null] = None
        st = lib.gsi_op_kernelcov_cross_grid(ctx._h, d, a["dims"], a["spacing"], m, a["target_idx"], n, a["source_idx"],
                                             nstruct, a["kinds"], a["sills"], a["ranges"], rotp, None, row0, mloc, a["out"])
    else:
        if null:
            a[null] = None
        st = lib.gsi_op_kernelcov_cross(ctx._h, d, m, a["targets"], n, a["sources"], nstruct, a["kinds"], a["sills"],
                                        a["ranges"], rotp, None, row0, mloc, a["out"])
    if st == 0:
        lib.gsi_op_free(h)
    return st, h.value


BAD_BOTH = {
    "m_0": dict(m=0), "n_0": dict(n=0), "m_neg": dict(m=-3), "row0_neg": dict(row0=-1, mloc=5),
    "mloc_over": dict(mloc=6), "block_over": dict(row0=2, mloc=4), "mloc_partial": dict(mloc=3),
    "nstruct_0": dict(nstruct=0), "sill_0": dict(sills=(0.0,)),
    "null_kinds": dict(null="kinds"), "null_sills": dict(null="sills"), "null_ranges": dict(null="ranges"),
    "null_out": dict(null="out"),
}
BAD_ARITH = {"null_targets": dict(null="targets"), "null_sources": dict(null="sources")}
BAD_GRID = {
    "null_dims": dict(null="dims"), "null_spacing": dict(null="spacing"),
    "target_idx_neg": dict(tidx=[0, 1, -1, 2, 3]), "target_idx_over": dict(tidx=[0, 1, 12, 2, 3]),
    "source_idx_neg": dict(sidx=[0, -5, 1, 2]), "source_idx_over": dict(sidx=[0, 1, 2, 100]),
    "target_null_m": dict(tidx=None), "source_null_n": dict(sidx=None), "dims_0": dict(dims=(4, 0)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", [False, True], ids=["arithmetic", "grid"])
@pytest.mark.parametrize("case", sorted(BAD_BOTH))
def test_rejects_invalid_cross(gsi, case, grid):
    st, h = _call(gsi, grid, **BAD_BOTH[case])
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h, (case, st, gsi._lib.load().gsi_last_error_string())


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(BAD_ARITH) + sorted(BAD_GRID))
def test_rejects_invalid_cross_path(gsi, case):
    grid = case in BAD_GRID
    st, h = _call(gsi, grid, **(BAD_GRID if grid else BAD_ARITH)[case])
    assert st == gsi._lib.ERR_INVALID_ARGUMENT and not h, (case, st, gsi._lib.load().gsi_last_error_string())


@pytest.mark.gpu
def test_rejects_unsupported_cross(gsi):
    for grid in (False, True):
        for d in (0, 4):
            st, h = _call(gsi, grid, d=d)
            assert st == gsi._lib.ERR_UNSUPPORTED and not h, (grid, d)
    rot2 = np.array([[0.0, 1.0], [-1.0, 0.0]]).ravel(order="F")
    # a signed table of 2^31 entries or more is refused before anything is allocated (the two points themselves fit)
    st, h = _call(gsi, True, d=2, m=1, n=1, tidx=[0], sidx=[7], rot=rot2, dims=(40000, 30000))
    assert st == gsi._lib.ERR_UNSUPPORTED and not h
    # NULL index lists with m, n = prod(dims) and the valid calls succeed; gsi_op_size reports (m, n)
    for grid, kw in ((False, {}), (True, {}), (True, dict(m=12, n=12, tidx=None, sidx=None)), (True, dict(rot=rot2))):
        st, _ = _call(gsi, grid, **kw)
        assert st == 0, (grid, kw, gsi._lib.load().gsi_last_error_string())
    op = gsi.KernelCrossCovMatrix([gsi.CovStructure("gaussian", 1.0, 2.0)], np.zeros((1, 7)), np.ones((1, 3)))
    assert op.shape == (7, 3) and op.T.shape == (3, 7)


# ------------------------------------------------------------------ GPU: two ranks
DIST_SHAPE, DIST_NSRC, DIST_SPLIT = (70, 60), 777, 2099     # rank 1 starts at an odd target row


def dist_case():
    """(structures, targets, sources, X for C X, X' for C' X) of tests/dist_kcov_cross_check.py."""
    structures = models(2, DIST_SHAPE)["three"]
    T = oracle.grid_coords(DIST_SHAPE)
    S = np.random.default_rng(4).uniform(0, 1, (2, DIST_NSRC)) * (np.array(DIST_SHAPE, dtype=np.float64) - 1)[:, None]
    X = np.random.default_rng(1).standard_normal((DIST_NSRC, 33))
    Xt = np.random.default_rng(2).standard_normal((T.shape[1], 33))
    return structures, T, S, X, Xt


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_two_ranks(gsi):
    """Targets split unevenly and not 64-aligned: the A X blocks and the all-reduced A' X match the one-rank products
    within a rounding bound (the split reorders the sums), and randsvd on two ranks matches oracle.randsvd."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
               "127.0.0.1", "--master-port", "29543", os.path.join(ROOT, "tests", "dist_kcov_cross_check.py"), tmp]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=540, cwd=ROOT)
        assert r.returncode == 0, f"{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
        structures, T, S, X, Xt = dist_case()
        m, n = T.shape[1], S.shape[1]
        op = gsi.KernelCrossCovMatrix(structures, T, S)
        Y1, Yt1 = apply_dev(gsi, op, X), apply_dev_t(gsi, op, Xt)
        A = cross_dense(structures, T, S)
        bound = 4 * n * U * (np.abs(A) @ np.abs(X)) + 1e-300
        bound_t = 4 * m * U * (np.abs(A.T) @ np.abs(Xt)) + 1e-300
        K, p, q = 20, 10, 1
        Zref = oracle.randsvd(A, np.random.default_rng(5).standard_normal((n, K + p)), K, p, q)
        for rank in range(2):
            f = np.load(os.path.join(tmp, f"cross_rank{rank}.npz"))
            r0, Y2 = int(f["row0"]), f["Y"]
            assert r0 == (0 if rank == 0 else DIST_SPLIT) and r0 + Y2.shape[0] == (DIST_SPLIT if rank == 0 else m)
            _bound_check(Y2, Y1[r0:r0 + Y2.shape[0]], bound[r0:r0 + Y2.shape[0]], f"C X rank {rank}")
            _bound_check(f["Yt"], Yt1, bound_t, f"C' X rank {rank}")
            c = oracle.compare_Z(f["Z"], Zref, K)
            assert c["tail_zero"] and c["sv_rel"] < SV_TOL and c["sine"] < SINE_TOL, (rank, c)
