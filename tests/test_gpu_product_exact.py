"""Element-wise tests of the two FP64 tensor-core product kernels (kcov_gemm_kernel + kcov_tail_fixup_kernel,
dense_gemm_kernel + dense_splitk_fixup_kernel) at every instantiated width and every schedule branch.

* Kernel values.  With sigma2 = 1 and nugget = 0, the covariance operator applied to unit columns returns the
  device's own kernel values bit for bit (each output is one product k * 1 plus exact zeros, in the full-round
  epilogue and in the stream-K fix-up alike).  Those values are checked against a high-precision reference of
  the same argument (rebuilt exactly on the host) in ulps, for exact symmetry, for the sigma2 / nugget
  epilogue, and for independence of the width and of the k-sweep schedule.
* Covariance products.  Every width x kind x DIM template, on a product that is all stream-K tail and on one
  with a full round plus a ragged tail, against the extracted values: |Y - C X| <= 2 gamma_n (|C| |X|)
  element by element, a bound that holds for any summation order.
* Dense products.  With small integer entries every partial sum is an exact integer below 2^53, so the
  product is exact in any order and is compared bit for bit with an integer reference.

Before every checked product the same shape runs once on an X full of NaN: the pooled split-K / stream-K
scratch then holds NaN, so a scratch slot read before it is written shows up as NaN in the checked result.
Every schedule shape is derived from the device's SM count (the library's persistent grid), mirrored below.
"""
import functools
from fractions import Fraction

import numpy as np
import pytest

import oracle
from gpu_util import get_gsi, gsi  # noqa: F401

pytestmark = pytest.mark.gpu

NB_LIST = (2, 4, 6, 8, 10, 12, 14, 16, 20, 24, 27, 28, 32)      # csrc/nb_list.h
U = 2.0 ** -53
TWO_M1000 = 2.0 ** -1000


def _widths():
    """Smallest and largest column count of every instantiated width, then > 256 (256-column chunks)."""
    out, prev = [], 0
    for nb in NB_LIST:
        out += [8 * prev + 1, 8 * nb]
        prev = nb
    return out + [257, 600, 1024]


WIDTHS = _widths()


@functools.lru_cache(maxsize=None)
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------ schedule mirrors (host side of the launches)
def kcov_schedule(mloc, n, sms):
    """launch_kcov: persistent grid, full rounds of 64-row tiles, stream-K tail of the leftover tiles."""
    total_rg = _cdiv(mloc, 16)
    grid = max(1, min(sms, total_rg))
    full_rounds = total_rg // (4 * grid)
    tail_rg0 = full_rounds * 4 * grid
    tail_tiles = _cdiv(total_rg - tail_rg0, 4)
    nkt = _cdiv(n, 32)
    tail_u = _cdiv(tail_tiles * nkt, grid) if tail_tiles else 0
    tiles = [(tail_rg0 * 16 + 64 * t, min(mloc, tail_rg0 * 16 + 64 * t + 64)) for t in range(tail_tiles)]
    last_nact = total_rg - tail_rg0 - 4 * (tail_tiles - 1) if tail_tiles else 4
    busy = _cdiv(tail_tiles * nkt, tail_u) if tail_u else 0
    return dict(grid=grid, full_rounds=full_rounds, tail_tiles=tiles, tail_u=tail_u, nkt=nkt,
                last_nact=last_nact, empty_ctas=grid - busy if tail_u else 0)


def dense_schedule(out_rows, kdim, sms):
    """launch_dense: split-K for few output tiles and a long reduction, else full rounds + one tail round."""
    ntiles = _cdiv(out_rows, 64)
    nkt = _cdiv(kdim, 32)
    grid = max(1, min(sms, ntiles))
    if ntiles * 2 <= sms and nkt >= 32:
        ks = min(sms // ntiles, nkt // 8)
        if ks > 1:
            kt_per = _cdiv(nkt, ks)
            ks = _cdiv(nkt, kt_per)
            return dict(kind="splitk", ksplit=ks, kt_per=kt_per, nkt=nkt)
    total_rg = _cdiv(out_rows, 16)
    full_rounds = total_rg // (4 * grid)
    rem = total_rg - full_rounds * 4 * grid
    return dict(kind="rounds", full_rounds=full_rounds, q_tail=_cdiv(rem, grid), nkt=nkt)


# ------------------------------------------------------------------ exact / high-precision host arithmetic
def fma(a, b, c):
    """Correctly rounded a*b + c (Fraction arithmetic is exact; int / int division rounds correctly)."""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _mp():
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.prec = 160
    return mpmath


def ulp_err(dev, ref, mp):
    """|dev - ref| in units of the last place of the (real) reference."""
    if ref == 0:
        return 0.0 if dev == 0 else float("inf")
    e = max(int(mp.floor(mp.log(ref, 2))), -1022)
    return float(abs(mp.mpf(dev) - ref) / mp.ldexp(1, e - 52))


def unit_columns(n, rows):
    E = np.zeros((n, len(rows)))
    E[np.asarray(rows), np.arange(len(rows))] = 1.0
    return E


def apply_dev(gsi, op, X):
    """op * X through a TALL DeviceMatrix (up to 1024 columns: above 256 the C++ 256-column chunk path)."""
    ctx = op.ctx
    Xd = gsi.DeviceMatrix.from_host(ctx, X)
    try:
        Yd = op.apply(Xd)
        try:
            return Yd.numpy()
        finally:
            Yd.free()
    finally:
        Xd.free()


def extract(gsi, op, n, rows):
    """C_hat[:, rows] bit for bit (op built with sigma2 = 1, nugget = 0)."""
    return apply_dev(gsi, op, unit_columns(n, rows))


# ------------------------------------------------------------------ A. kernel values against a high-precision reference
# Bounds asserted here and stated beside fast_exp_neg / fast_sqrt_pos (csrc/kcov_gemm.cu) and in DESIGN.md:
#   fast_exp_neg                      2.5 ulp
#   exponential exp(-sqrt(r2))        2.5 + 4 y ulp  (y = sqrt(r2): 2 ulp of fast_sqrt_pos times the conditioning y)
#   powerlaw (library exp / log1p)    2 + 4 |z| ulp  (z = beta log1p(r2))
#   lattice table (host libm)         4 + 4 * (argument of exp) ulp (also covers the host's rounding of r2)
EXP_BOUND = 2.5


def _targets(kind, rng):
    """Arguments of exp (gaussian / exponential) or r2 (powerlaw) the points are placed at: every table slot
    k & 63 densely, y near 0, y around the 2^-1000 flush, y on both sides of 1024."""
    if kind == "powerlaw":
        return np.concatenate([10.0 ** rng.uniform(-12, 6, 1500), rng.uniform(0, 4, 500)])
    return np.concatenate([rng.uniform(0, 8, 4000), 10.0 ** rng.uniform(-12, -2, 100), rng.uniform(690, 700, 300),
                           rng.uniform(1020, 1023.99, 30), rng.uniform(1024, 1030, 30), [1024.0, 1023.9999999]])


@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", ["gaussian", "exponential", "powerlaw"])
def test_kernel_values_ulp(gsi, kind, d):
    """Arithmetic generation: every extracted value against exp / sqrt / log1p in 160-bit arithmetic of the
    device's own argument r2 (same subtraction and fma chain, in the same order, computed exactly)."""
    mp = _mp()
    rng = np.random.default_rng(100 * d + len(kind))
    beta = 0.8
    ell = np.array([1.3, 0.7, 2.1][:d])
    pre = 0.70710678118654752440 if kind == "gaussian" else 1.0
    t = _targets(kind, rng)
    rho = np.sqrt(t) if kind in ("gaussian", "powerlaw") else t              # distance in scaled coordinates
    dirs = rng.standard_normal((d, t.size))
    dirs /= np.linalg.norm(dirs, axis=0)
    origin = np.array([0.37, -1.1, 0.52][:d])
    coords = np.concatenate([origin[:, None], origin[:, None] + rho * dirs * (ell / pre)[:, None]], axis=1)
    n = coords.shape[1]
    op = gsi.KernelCovMatrix(kind, coords, ell, beta=beta)
    col = extract(gsi, op, n, [0])[:, 0]
    u = (coords / ell[:, None]) * pre                                       # the host scaling of gsi_op_kernelcov
    errs, args, bounds, nflush = [], [], [], 0
    for i in range(n):
        r2 = 1e-300 if kind == "exponential" else 0.0
        for k in range(d):
            dk = float(u[k, i] - u[k, 0])
            r2 = fma(dk, dk, r2)
        R2 = mp.mpf(r2)
        if kind == "gaussian":
            arg = R2
            bound = EXP_BOUND
        elif kind == "exponential":
            arg = mp.sqrt(R2)
            bound = EXP_BOUND + 4 * float(arg)
        else:
            arg = beta * mp.log1p(R2)
            bound = 2.0 + 4 * float(arg)
        ref = mp.exp(-arg)
        if kind != "powerlaw" and ref < TWO_M1000 and col[i] == 0.0:
            nflush += 1                                                     # flushed to zero below 2^-1000
            continue
        errs.append(ulp_err(float(col[i]), ref, mp))
        args.append(float(arg))
        bounds.append(bound)
    errs, args, bounds = np.array(errs), np.array(args), np.array(bounds)
    w = int(np.argmax(errs - bounds))
    small = args < 1.0                                                      # where the conditioning term is < 4 ulp
    msg = (f"{kind} d={d}: max error {errs.max():.3f} ulp (at argument < 1: {errs[small].max():.3f} ulp); "
           f"worst against the bound: {errs[w]:.3f} ulp at argument {args[w]!r} (bound {bounds[w]:.3f}); "
           f"{errs.size} values, {nflush} flushed")
    print(msg)
    assert np.all(errs <= bounds), msg
    if kind != "powerlaw":
        assert nflush >= 60, msg                                            # the flush region was reached


def test_fast_exp_table_points_exact(gsi):
    """At arguments y = RN(m ln2 / 64) (|y - m ln2/64| < 2^-54, m = 0..64) fast_exp_neg's polynomial is exactly 1,
    so the Gaussian kernel value is kExp2Table[-m & 63] / 2 = RN(2^(-m/64)) bit for bit: one test point per table
    slot, each of which would show a one-bit fault in its entry."""
    mp = _mp()
    c = 0.70710678118654752440
    ln2_64 = mp.log(2) / 64
    xs = [(0.0, 0.0)]
    for m in range(1, 65):
        t = float(m * ln2_64)
        assert abs(mp.mpf(t) - m * ln2_64) < mp.ldexp(1, -54) - mp.ldexp(1, -80)
        # r2 = fma(u1, u1, fl(u0^2)) with u = fl(x * c): u0^2 a few ulps below t, u1 supplies the rest exactly
        x0 = float(np.sqrt(2 * (t - 8 * np.spacing(t))))
        u0 = x0 * c
        a = u0 * u0
        x1 = float(np.sqrt(2 * float(Fraction(t) - Fraction(a))))
        for _ in range(200):
            u1 = x1 * c
            r2 = fma(u1, u1, a)
            if r2 == t:
                break
            x1 = np.nextafter(x1, np.inf if r2 < t else -np.inf)
        assert r2 == t, m
        xs.append((x0, float(x1)))
    coords = np.array(xs).T
    op = gsi.KernelCovMatrix("gaussian", coords, [1.0, 1.0])
    col = extract(gsi, op, coords.shape[1], [0])[:, 0]
    bad = []
    for m in range(65):
        want = float(mp.power(2, mp.mpf(-m) / 64))
        if col[m] != want:
            bad.append((m, (-m) & 63, float(col[m]).hex(), want.hex()))
    assert not bad, f"kernel values at table points (m, slot, got, want): {bad}"


@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", ["gaussian", "exponential", "powerlaw"])
def test_table_kernel_values_ulp(gsi, kind, d):
    """Structured grid: the looked-up values against the same high-precision reference of the host's scaled
    offsets (the table is libm on the host; the bound also covers the host's rounding of r2)."""
    mp = _mp()
    beta = 0.8
    shape, spacing = {1: ((3000,), (0.003,)), 2: ((1500, 3), (0.005, 345.5)), 3: ((500, 3, 2), (0.015, 300.0, 600.0))}[d]
    ell = np.ones(d)
    op = gsi.GridKernelCovMatrix(kind, shape, ell, spacing=spacing, beta=beta)
    n = int(np.prod(shape))
    col = extract(gsi, op, n, [0])[:, 0]
    lat = np.array(np.unravel_index(np.arange(n), shape, order="F"))
    errs, args = [], []
    for i in range(n):
        R2 = mp.mpf(0)
        for k in range(d):
            uk = (float(lat[k, i]) * spacing[k]) / ell[k]
            R2 += mp.mpf(uk) ** 2
        if kind == "gaussian":
            arg = R2 / 2
        elif kind == "exponential":
            arg = mp.sqrt(R2)
        else:
            arg = beta * mp.log1p(R2)
        errs.append(ulp_err(float(col[i]), mp.exp(-arg), mp))
        args.append(float(arg))
    errs, args = np.array(errs), np.array(args)
    bounds = 4.0 + 4 * args
    w = int(np.argmax(errs - bounds))
    msg = (f"table {kind} d={d}: max error {errs.max():.3f} ulp; worst against the bound: {errs[w]:.3f} ulp at "
           f"argument {args[w]!r} (bound {bounds[w]:.3f}); {n} values")
    print(msg)
    assert np.all(errs <= bounds), msg


# ------------------------------------------------------------------ operators at schedule-derived shapes
KINDS = ["exponential", "gaussian", "powerlaw", "table"]


def _grid_dims(d, n_min, ok):
    """Smallest structured grid (d dims, each >= 8) with ok(n) for n = prod(dims) >= n_min."""
    for n in range(n_min, n_min + 5000):
        if not ok(n):
            continue
        if d == 2:
            for a in range(int(np.sqrt(n)), 7, -1):
                if n % a == 0 and n // a >= 8:
                    return (n // a, a)
        else:
            for a in range(int(round(n ** (1 / 3))) + 2, 7, -1):
                if n % a:
                    continue
                m = n // a
                for b in range(int(np.sqrt(m)), 7, -1):
                    if m % b == 0 and m // b >= 8:
                        return (m // b, b, a)
    raise AssertionError("no grid found")


def big_ok(n, sms):
    """n just over 64 * SMs rows: one full round, then a stream-K tail of >= 3 tiles whose last tile has fewer
    than 4 active row groups, a last row group that is ragged, shares spanning two tiles and CTAs with none."""
    s = kcov_schedule(n, n, sms)
    return (n % 16 != 0 and s["full_rounds"] == 1 and len(s["tail_tiles"]) >= 3 and s["last_nact"] < 4
            and s["empty_ctas"] > 0 and s["tail_u"] % s["nkt"] != 0)


@functools.lru_cache(maxsize=None)
def grid_shape(dim, size):
    sms = num_sms()
    if size == "small":                    # all stream-K tail
        return (40, 25) if dim == 2 else (10, 10, 10)
    return _grid_dims(dim, 64 * sms + 100, lambda n: big_ok(n, sms))


def make_op(gsi, kind, dim, size, sigma2=1.0, nugget=0.0):
    shape = grid_shape(dim, size)
    ell = [s / 2.5 for s in shape]
    if kind == "table":
        return gsi.GridKernelCovMatrix("exponential", shape, ell, sigma2=sigma2, nugget=nugget)
    coords = oracle.grid_coords(shape)
    coords = coords + np.random.default_rng(7).uniform(-0.3, 0.3, coords.shape)
    return gsi.KernelCovMatrix(kind, coords, ell, sigma2=sigma2, nugget=nugget, beta=0.8)


def sample_rows(n, k=24, seed=0):
    """First and last row of every stream-K tail tile, the last row, the first rows and random rows."""
    s = kcov_schedule(n, n, num_sms())
    rows = {0, 1, 15, 16, n - 1}
    for a, b in s["tail_tiles"]:
        rows |= {a, b - 1}
    if s["full_rounds"]:
        rows |= {64 * s["grid"] - 1, 64 * s["grid"] - 17}
    rows |= set(np.random.default_rng(seed).choice(n, k, replace=False).tolist())
    return sorted(rows)


@functools.lru_cache(maxsize=None)
def extracted(kind, dim, size):
    """(operator with sigma2 = 1, nugget = 0; sampled rows S; C_hat[S, :]) -- C_hat is exactly symmetric."""
    g = get_gsi()
    op = make_op(g, kind, dim, size)
    n = op.shape[0]
    S = sample_rows(n)
    return op, S, np.ascontiguousarray(extract(g, op, n, S).T)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_kernel_values_symmetry_and_epilogue(gsi, kind, dim):
    """On rows of the full round and of the stream-K tail: C_hat[S, S] is exactly symmetric with a unit
    diagonal, and the epilogue applies sigma2 / nugget with one rounding (either fused or not)."""
    op, S, Cs = extracted(kind, dim, "big")
    n = op.shape[0]
    assert kcov_schedule(n, n, num_sms())["full_rounds"] == 1
    Css = Cs[:, S]
    assert np.array_equal(Css, Css.T)
    assert np.all(np.diag(Css) == 1.0)
    assert np.all(Cs > 0.0) and np.all(Cs <= 1.0)
    E = unit_columns(n, S)
    unit = E.T.astype(bool)                    # unit[c, j]: the nugget lands on (row S[c], column j = S[c])
    for sigma2 in (0.5, 1.7):
        Y = apply_dev(gsi, make_op(gsi, kind, dim, "big", sigma2=sigma2, nugget=0.3), E).T
        plain = sigma2 * Cs                    # off the unit entries: fl(sigma2 * c) (the nugget adds an exact 0)
        assert np.array_equal(Y[~unit], plain[~unit]), sigma2
        for c, j in zip(*np.nonzero(unit)):
            ok = (float(np.float64(sigma2 * Cs[c, j]) + 0.3), fma(sigma2, Cs[c, j], 0.3))
            assert Y[c, j] in ok, (sigma2, S[c], j, Y[c, j], ok)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_kernel_values_width_and_schedule_independent(gsi, kind, dim):
    """The same (i, j) extracted through every width and through other k-sweep schedules (lock-step, spread
    starts, sweep window) is bit-identical: the values depend on the coordinates only, not on whether a tile's
    first k-tile is generated in the prologue or in the loop, nor on full round vs stream-K tail."""
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


# ------------------------------------------------------------------ B. kcov products at every width and schedule
@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("size", ["small", "big"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_kcov_product_bound(gsi, kind, dim, size, cols):
    """Y = C X on sampled rows within 2 gamma_n (|C_hat| |X|) of C_hat X, element by element, after the same
    product on a NaN X has left NaN in the pooled stream-K scratch."""
    op, S, Cs = extracted(kind, dim, size)
    n = op.shape[0]
    sched = kcov_schedule(n, n, num_sms())
    if size == "small":
        assert sched["full_rounds"] == 0 and sched["tail_tiles"]
    else:
        assert big_ok(n, num_sms())
    apply_dev(gsi, op, np.full((n, cols), np.nan))                  # poison the pooled scratch
    X = np.random.default_rng(cols).standard_normal((n, cols))
    Y = apply_dev(gsi, op, X)[S]
    ref = Cs @ X
    gamma = n * U / (1 - n * U)
    bound = 2 * gamma * (np.abs(Cs) @ np.abs(X))
    err = np.abs(Y - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{kind} dim={dim} n={n} cols={cols}: {bad.sum()} elements out of bound, first at "
                           f"(row {S[np.nonzero(bad)[0][0]]}, col {np.nonzero(bad)[1][0]}); max err/bound "
                           f"{np.nanmax(err / bound):.3g}")


# ------------------------------------------------------------------ C. dense products, bit-exact on integers
def _ints(rng, shape, lim=8):
    return rng.integers(-lim, lim + 1, size=shape).astype(np.float64)


def int_matmul(A, B):
    """Exact product of integer-valued float64 matrices whose partial sums stay below 2^53 (then every
    summation order is exact, so BLAS returns the integer product itself)."""
    assert A.shape[1] * np.abs(A).max(initial=0) * np.abs(B).max(initial=0) < 2.0 ** 53
    return A @ B


def _apply_dense(gsi, op, X, trans):
    Xd = gsi.DeviceMatrix.from_host(op.ctx, X)
    try:
        Yd = op.apply(Xd, trans=trans)
        try:
            return Yd.numpy()
        finally:
            Yd.free()
    finally:
        Xd.free()


def _dense_check(gsi, A, trans, cols, rng):
    op = gsi.DenseMatrix(A)
    kdim = A.shape[0] if trans else A.shape[1]
    _apply_dense(gsi, op, np.full((kdim, cols), np.nan), trans)     # poison the pooled split-K scratch
    X = _ints(rng, (kdim, cols))
    Y = _apply_dense(gsi, op, X, trans)
    ref = int_matmul(A.T if trans else A, X)
    assert np.array_equal(Y, ref), (A.shape, trans, cols, int(np.sum(Y != ref)))


@pytest.mark.parametrize("cols", WIDTHS)
@pytest.mark.parametrize("shape", ["rounds", "splitk"])
@pytest.mark.parametrize("trans", [False, True])
def test_dense_integer_exact_widths(gsi, trans, shape, cols):
    """A X and A' X at every width, odd m and n (TMA's out-of-bounds zero fill), one tail round or split-K."""
    rng = np.random.default_rng(cols + 7 * trans)
    out_rows, kdim = (333, 517) if shape == "rounds" else (131, 2049)
    sched = dense_schedule(out_rows, kdim, num_sms())
    assert sched["kind"] == ("rounds" if shape == "rounds" else "splitk"), sched
    A = _ints(rng, (kdim, out_rows) if trans else (out_rows, kdim))
    _dense_check(gsi, A, trans, cols, rng)


DENSE_BRANCHES = ["splitk_ragged", "splitk_even", "single_tail_round", "full_plus_tail_q1", "full_plus_tail_q2",
                  "full_plus_tail_q3", "full_plus_tail_q4", "full_rounds_only"]


def dense_branch_shape(name, sms):
    """(out_rows, kdim) that takes launch_dense's schedule branch `name` on `sms` SMs."""
    if name.startswith("splitk"):                                   # split-K, last part ragged or not
        for kdim in range(2049, 20000, 2):
            s = dense_schedule(201, kdim, sms)
            if s["kind"] == "splitk" and (s["nkt"] % s["kt_per"] != 0) == (name == "splitk_ragged"):
                return 201, kdim
        raise AssertionError(name)
    if name == "single_tail_round":                                 # no full round, one tail round (q_tail = 4)
        return 64 * max(2, sms // 2) - 21, 77
    if name == "full_rounds_only":
        return 64 * 2 * sms, 45
    q = int(name[-1])                                               # one full round + a tail round with q_tail = q
    return 16 * (4 * sms + (q - 1) * sms + 1) - 7, 75


@pytest.mark.parametrize("cols", [5, 213])
@pytest.mark.parametrize("trans", [False, True])
@pytest.mark.parametrize("branch", DENSE_BRANCHES)
def test_dense_integer_exact_schedules(gsi, branch, trans, cols):
    """Every schedule branch of the dense kernel, bit-exact on integers after a NaN-poisoned run."""
    sms = num_sms()
    out_rows, kdim = dense_branch_shape(branch, sms)
    s = dense_schedule(out_rows, kdim, sms)
    if branch.startswith("splitk"):
        assert s["kind"] == "splitk" and s["ksplit"] > 1, s
    elif branch == "single_tail_round":
        assert s["kind"] == "rounds" and s["full_rounds"] == 0 and s["q_tail"] == 4, s
    elif branch == "full_rounds_only":
        assert s["kind"] == "rounds" and s["full_rounds"] == 2 and s["q_tail"] == 0, s
    else:
        assert s["kind"] == "rounds" and s["full_rounds"] == 1 and s["q_tail"] == int(branch[-1]), s
    rng = np.random.default_rng(DENSE_BRANCHES.index(branch) * 10 + cols + trans)
    A = _ints(rng, (kdim, out_rows) if trans else (out_rows, kdim))
    _dense_check(gsi, A, trans, cols, rng)


@pytest.mark.parametrize("cols", [1, 60, 256, 600])
@pytest.mark.parametrize("mean", ["raw", "integer_means"])
@pytest.mark.parametrize("N", [17, 65])
def test_lowrankcov_integer_exact(gsi, N, mean, cols):
    """S (S' X) / (N - 1) with integer samples and N - 1 a power of two: split-K S'X then S (S'X), exact."""
    rng = np.random.default_rng(N + cols)
    n = 3001
    D = _ints(rng, (n, N))
    if mean == "raw":
        op = gsi.LowRankCovMatrix(D, remove_mean=False)
    else:
        D[:, -1] = -D[:, :-1].sum(axis=1)                           # rows of D sum to zero
        op = gsi.LowRankCovMatrix(D + _ints(rng, (n, 1), 50), remove_mean=True)   # integer row means
    assert dense_schedule(N, n, num_sms())["kind"] == "splitk"
    apply_dev(gsi, op, np.full((n, cols), np.nan))
    X = _ints(rng, (n, cols))
    ref = int_matmul(D, int_matmul(D.T, X)) / (N - 1)
    assert np.array_equal(apply_dev(gsi, op, X), ref)


@pytest.mark.parametrize("cols", [1, 13, 256, 300])
def test_sketch_products_integer_exact(gsi, cols):
    """_Sketch.apply (S V, split-K) and _Sketch.cov (S diag(R) S' and, for a dense R, S (R S'))."""
    from gsi_b200.pcga import _Sketch
    rng = np.random.default_rng(cols)
    Nred, nobs = 37, 2501
    S = _ints(rng, (Nred, nobs))
    sk = _Sketch(S, gsi.default_context())
    assert dense_schedule(Nred, nobs, num_sms())["kind"] == "splitk"
    sk.apply(np.full((nobs, cols), np.nan))
    V = _ints(rng, (nobs, cols))
    assert np.array_equal(sk.apply(V), int_matmul(S, V))
    sk.apply(np.full((nobs, Nred), np.nan))                         # the shape of the products inside cov
    Rd = rng.integers(1, 9, nobs).astype(np.float64)
    assert np.array_equal(sk.cov(Rd), int_matmul(S * Rd, S.T))
    if cols == 1:
        S2 = _ints(rng, (Nred, 301))
        R = _ints(rng, (301, 301), 3)
        assert np.array_equal(_Sketch(S2, gsi.default_context()).cov(R), int_matmul(S2, int_matmul(R, S2.T)))
