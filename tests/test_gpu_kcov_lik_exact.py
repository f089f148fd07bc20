"""The likelihood gradient's kernel derivatives (kern_value_deriv in csrc/kcov_gemm.cu), argument by argument, against
closed-form references in 160-bit arithmetic.

The construction: n = 2P points as P pairs, pair q = (x_2q, x_2q+1), so that A is block-diagonal with 2 x 2 blocks
A_q = [a_q c_q; c_q a_q].  With one pair (n = 2), ML, p = 0 and y = 0, alpha = 0 and W = -A^-1, so
    W_01 = c / (a^2 - c^2),   W_00 = W_11 = -a / (a^2 - c^2)
and each range component of the gradient is the single term
    d l / d range_(s,a) = sill_s (-2 / range_(s,a)) W_01 k_s'(r2_s) du_(s,a)^2
(du the device's scaled coordinate difference, r2 its fma chain).  a and c are read from the device bit for bit: the
operator applied to the identity returns them (every other term of the product is k * 0 = 0).  The reference starts
from those bits and from the device's own r2, so the bound only has to cover the derivative itself, the 2 x 2
factor / inverse / sweeps that produce W_01, and the roundings of the contraction.

* Without a GPU: the closed form for many pairs (ML and REML, p in {0, 1, 3}) against host_lik / host_grad of
  tests/test_gpu_kcov_lik.py on the dense block-diagonal matrix, for every kind; and the per-argument checker rejects
  a device result perturbed by 1.5 times its bound in one argument region.
* On the GPU: every kind at d = 1, 2, 3 over s = 1e-8 .. 8 (power law: r2 = 1e-12 .. 1e6; spherical: up to 1 - 1e-12,
  at 1 and beyond), the exponential family close to the 2^-1000 flush of fast_exp_neg, and rotated three-structure
  models; every component (ranges, sills, nugget) against its bound.  Lines starting with LIKREPORT carry the worst
  ratio of error to bound per kind.
* On the GPU, many pairs per call (n = 258, 2 050, 6 000; single kinds and a rotated nested model; y != 0;
  p in {0, 1, 3}; ML and REML): value, beta and every gradient component against the closed form within the
  first-order bounds of whole_call_bounds, derived along the device's operation order (c u (n + |log det A| + q) and
  c u S_theta with c printed beside the 1e-11 S_theta of tests/test_gpu_kcov_lik.py).
* n = 65 600 (n_p = 65 664: 4.31e9 > 2^32 factor entries; past 46 341 the factor already has > 2^31): the same for an
  exponential + rotated spherical model, p = 1, REML, then KernelCovCholesky's log det, solve and simulate pair by
  pair.  It needs 40 GB of free device memory and is skipped, saying so, with less.
Every whole-call test first checks the premise: both rows of each pair in the product with the even / odd indicator
columns hold the same two values, and tiles off the pair blocks (including rows past 2^16 at n = 65 600) are exact
zeros.
"""
import math
import os
import sys

import numpy as np
import pytest

from gpu_util import gsi  # noqa: F401
from test_gpu_kcov_lik import host_grad, host_lik
from test_gpu_kcov_model import PRE, structure_coords
from test_gpu_product_exact import _mp, apply_dev, fma

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gsi_b200 as G                                   # noqa: E402

KINDS = ["exponential", "gaussian", "powerlaw", "matern32", "matern52", "spherical"]
CODE = {k: i for i, k in enumerate(KINDS)}
CS = G.CovStructure
U = 2.0 ** -53                     # unit roundoff; the bounds beside kern_eval count in units of 2^-52 = 2 U
SQRT_KINDS = (0, 3, 4, 5)          # kinds whose r2 chain starts at 1e-300 (kind_takes_sqrt)
EXP_KINDS = (0, 1, 3, 4)           # kinds flushed to zero with fast_exp_neg below 2^-1000
SECOND_ORDER = 1.0 + 2.0 ** -40    # the bounds below are first order in U; this covers the O(U^2) terms

# ------------------------------------------------------------------ error bounds and their derivations
# W_01 from the 2 x 2 factor, its inverse and the sweeps, relative, in units of U.  chol_diag_kernel computes
# L00 = RN(sqrt a), L10 = RN(c / L00), L11 = RN(sqrt(RN(a - RN(L10^2)))) (an fma only removes the inner rounding),
# X11 = RN(1 / L11), X10 = RN(-RN(L10 RN(1 / L00)) / L11); the forward sweep of the identity columns returns X bit for
# bit (one nonzero product per entry) and the backward sweep gives A^-1_01 = RN(X10 X11) (one nonzero product: every
# other term of the DMMA sums is an exact zero, the padding rows of X included); the rank update subtracts exact zeros
# (alpha = 0).  With |c| <= a / 3 (kappa(A_q) <= 2, asserted):
#   RN(1 / L00): 1 + 1 = 2;  L10 (of c / sqrt a): 1 + 1 = 2;  RN(L10 RN(1 / L00)) (of c / a): 2 + 2 + 1 = 5
#   RN(L10^2): 2 * 2 + 1 = 5;  a - L10^2: 5 (c^2 / a) / (a - c^2 / a) + 1 = 5 c^2 / (a^2 - c^2) + 1 <= 5 / 8 + 1 = 1.625
#   L11: 1.625 / 2 + 1 = 1.8125;  X11: 2.8125;  X10: 5 + 1.8125 + 1 = 7.8125;  A^-1_01: 7.8125 + 2.8125 + 1 = 11.625
E_W01 = 11.625
# W_00 = -RN(X00^2 + X10^2) (two positive terms: the larger of 2 * 2 + 1 and 2 * 7.8125 + 1, plus the sum's rounding)
# and W_11 = -RN(X11^2) (2 * 2.8125 + 1): both within 17.625 U
E_W00 = 17.625
# The range term: RN(du * du), g = RN(wt * dk) (wt = 2 wv is exact), the fma into an exact-zero accumulator, and on the
# host RN(sill / range) and its product with the sum: 5 roundings.  Every other partial sum of the contraction (the
# diagonal entries carry du = 0; padding rows are skipped) is an exact zero, so the reductions add nothing.
E_CONTR = 5.0


def deriv_bound_units(kind, s, z):
    """The bound beside kern_value_deriv, relative, in units of 2^-52 (s = sqrt(r2) exact; z = beta log1p r2)."""
    if kind == 0:
        return 5.0 + 2.0 * s
    if kind == 1:
        return 2.5
    if kind == 2:
        return 3.5 + 4.0 * abs(z)
    if kind == 3:
        return 2.5 + 2.0 * s
    if kind == 4:
        return 6.25 + 4.0 * s
    return 2.5 + 2.0 * (1.0 + s / (1.0 - s) + s / (1.0 + s))


def value_bound_units(kind, s, z):
    """The bound beside kern_eval, relative, in units of 2^-52 (the conditioning k = |s k'(s) / k(s)| of each kind)."""
    if kind == 0:
        return 2.5 + 2.0 * s
    if kind == 1:
        return 2.5
    if kind == 2:
        return 2.0 + 4.0 * abs(z)
    if kind == 3:
        return 3.0 + 2.0 * s * s / (1.0 + s)
    if kind == 4:
        return 4.25 + 2.0 * s * s * (1.0 + s) / (3.0 + 3.0 * s + s * s)
    return 2.5 + 2.0 * 3.0 * s * (1.0 + s) / ((1.0 - s) * (2.0 + s)) if s < 1.0 else 0.0


# ------------------------------------------------------------------ the device's arguments, rebuilt exactly
def pair_args(st, X):
    """(du, r2) of the pair (X[:, 1] row, X[:, 0] column) exactly as kcov_grad_kernel forms them: u scaled on the host
    as gsi_op_kernelcov does, du = RN(u_1 - u_0) per axis, r2 the fma chain from 1e-300 (kinds taking sqrt) or 0."""
    u = structure_coords(st, X, PRE[st.kind])
    du = [float(u[k, 1] - u[k, 0]) for k in range(X.shape[0])]
    r2 = 1e-300 if st.kind in SQRT_KINDS else 0.0
    for v in du:
        r2 = fma(v, v, r2)
    return du, r2


def kernel_exact(mp, kind, r2, beta):
    """(k, dk / dr2, s, z, y) at the double r2 in 160-bit arithmetic; y is the argument of exp (None: no flush)."""
    R2 = mp.mpf(r2)
    s = mp.sqrt(R2)
    z = mp.mpf(beta) * mp.log1p(R2)
    if kind == 0:
        e = mp.exp(-s)
        return e, -e / (2 * s), s, z, s
    if kind == 1:
        e = mp.exp(-R2)
        return e, -e, s, z, R2
    if kind == 2:
        return mp.exp(-z), -mp.mpf(beta) * (1 + R2) ** (-mp.mpf(beta) - 1), s, z, None
    if kind == 3:
        e = mp.exp(-s)
        return (1 + s) * e, -e / 2, s, z, s
    if kind == 4:
        e = mp.exp(-s)
        return (1 + s + R2 / 3) * e, -(1 + s) * e / 6, s, z, s
    if s < 1:
        return (1 - s) ** 2 * (2 + s) / 2, -3 * (1 - s) * (1 + s) / (4 * s), s, z, None
    return mp.mpf(0), mp.mpf(0), s, z, None


def pair_components(sts, X, nug, a, c):
    """Per gradient component (ABI order: per structure the sill and the d ranges, then the nugget): the closed-form
    value at the device's a, c and arguments, the allowed error, and a label (kind, region) for the report.  An allowed
    error of None means the device must return exactly 0 (flushed or beyond the spherical range)."""
    mp = _mp()
    d = X.shape[0]
    A, Cc = mp.mpf(a), mp.mpf(c)
    assert a > 0 and 3 * abs(c) <= a, (a, c)                         # kappa(A_q) <= 2: the premise of E_W01
    det = A * A - Cc * Cc
    W01, W00 = Cc / det, -A / det
    out = []
    for st in sts:
        du, r2 = pair_args(st, X)
        k, dk, s, z, y = kernel_exact(mp, st.kind, r2, st.beta)
        sf, zf = float(s), float(z)
        state = flush_state(mp, y, st.kind)
        flushed = state == "flush"
        ranges = np.broadcast_to(st.ranges, (d,))
        # sill: W00 + W01 k (the two diagonal terms and the off-diagonal pair, halved); the diagonal values are
        # exactly 1.  Errors: W00 (E_W00), W01 k (E_W01 + twice the value bound in U + RN(wt kv)), and the two
        # additions of the reduction tree over |W00| + |W01 k|
        kv_units = 0.0 if flushed else value_bound_units(st.kind, sf, zf)
        ref = W00 + W01 * k
        allow = (abs(W00) * E_W00 + abs(W01 * k) * (E_W01 + 2 * kv_units + 1) + 2 * (abs(W00) + abs(W01 * k))) * U
        if state != "keep":
            allow += abs(W01 * k)                                      # a flushed value drops the whole term
        out.append((ref, allow, (st.kind, "sill")))
        for ax in range(d):
            pref = abs(mp.mpf(st.sill) * 2 / mp.mpf(ranges[ax]) * W01 * mp.mpf(du[ax]) ** 2)
            ref = -mp.mpf(st.sill) * (2 / mp.mpf(ranges[ax])) * W01 * dk * mp.mpf(du[ax]) ** 2
            if flushed:
                out.append((mp.mpf(0), None, (st.kind, "flush")))
                continue
            if st.kind == 5 and s >= 1:
                # the device's s is within 2 units of 2^-52 of the exact one: below s = 1 + 2^-51 it may fall under 1,
                # where |dk| = 0.75 (1 - s)(1 + s) / s <= 3 * 2^-52; beyond, dk is exactly 0
                if s < 1 + mp.ldexp(1, -51):
                    out.append((ref, pref * 3 * 2 * U, (5, "at 1")))
                else:
                    out.append((mp.mpf(0), None, (5, "beyond")))
                continue
            units = deriv_bound_units(st.kind, sf, zf)
            allow = pref * abs(dk) * (2 * units + E_W01 + E_CONTR) * U
            if state == "either":                                      # the device may flush or keep this one
                out.append((ref, allow, (st.kind, "flush edge"), True))
                continue
            out.append((ref, allow, (st.kind, region_of(st.kind, sf, r2))))
    # nugget: W00 (halved sum of W00 and W11, one addition)
    out.append((W00, abs(W00) * (E_W00 + 1) * U, (-1, "nugget")))
    return out


def flush_state(mp, y, kind):
    """'flush', 'keep' or 'either' for an exp argument y (None: the kind has no flush).  fast_exp_neg flushes when
    k = round(-64 y / ln 2) < -64000 (e = k >> 6 < -1000) or y >= 1024.  The device's y of the kinds taking a square
    root is within 2 units of 2^-52 of the exact one, so within 1e-9 relative of the k threshold either may happen."""
    if y is None:
        return "keep"
    kk = y * 64 / mp.log(2)
    edge = mp.mpf(64000.5)
    if y >= 1024 or kk > edge * (1 + mp.mpf(1e-9)):
        return "flush"
    if kk < edge * (1 - mp.mpf(1e-9)):
        return "keep"
    return "either"


def region_of(kind, s, r2):
    if kind == 2:
        return "r2<1" if r2 < 1 else "r2>=1"
    if kind == 5 and s > 0.5:
        return "s>0.5"
    return "s<1" if s < 1 else ("s<10" if s < 10 else "s>=10")


def check_components(comps, dev):
    """[(label, ratio)] for every component (ratio = |dev - ref| / allowed; flushed components must be exact zeros:
    ratio 0 when they are, inf when not)."""
    mp = _mp()
    out = []
    for comp, v in zip(comps, dev):
        ref, allow, label = comp[:3]
        if len(comp) > 3 and v == 0.0:                                 # flush edge: zero is allowed as well
            out.append((label, 0.0))
            continue
        if allow is None:
            out.append((label, 0.0 if v == 0.0 else float("inf")))
            continue
        err = abs(mp.mpf(float(v)) - ref)
        out.append((label, float(err / (allow * SECOND_ORDER)) if allow > 0 else (0.0 if err == 0 else float("inf"))))
    return out


# ------------------------------------------------------------------ closed form for many pairs
def _obj(x):
    """float64 array -> object array of exact mpf values"""
    mp = _mp()
    x = np.asarray(x, dtype=np.float64)
    return np.array([mp.mpf(float(v)) for v in x.ravel()], dtype=object).reshape(x.shape)


def _fsum(x):
    return _mp().fsum(list(np.ravel(x)))


def pairs_closed_form(a, c, y, F, reml, diag_d, off_d):
    """Value, beta, gradient and S_theta of the pair-block-diagonal A in 160-bit arithmetic, O(P p^2).  a, c: the P
    block entries; y: n = 2P observations; F: n x p drift; diag_d[t], off_d[t][q]: dA / dtheta_t on the diagonal (the
    same for every point) and in the off-diagonal of pair q.  Also returns the per-pair pieces (A_q^-1, alpha, H H',
    M = F'A^-1 F) that whole_call_bounds needs."""
    mp = _mp()
    a, c = np.asarray(a, dtype=np.float64), np.asarray(c, dtype=np.float64)
    P, p = a.size, F.shape[1]
    n = 2 * P
    A, C = _obj(a), _obj(c)
    det = A * A - C * C
    i00, i01 = A / det, -C / det
    y0, y1 = _obj(y[0::2]), _obj(y[1::2])
    F0, F1 = _obj(F[0::2]).reshape(P, p), _obj(F[1::2]).reshape(P, p)
    h0 = i00[:, None] * F0 + i01[:, None] * F1                          # A_q^-1 F_q
    h1 = i01[:, None] * F0 + i00[:, None] * F1
    logdet = _fsum(np.frompyfunc(mp.log, 1, 1)(det))
    if p:
        M = mp.matrix([[_fsum(F0[:, j] * h0[:, k] + F1[:, j] * h1[:, k]) for k in range(p)] for j in range(p)])
        b = mp.matrix([_fsum(h0[:, j] * y0 + h1[:, j] * y1) for j in range(p)])
        beta_m = mp.lu_solve(M, b)
        beta = np.array([beta_m[j] for j in range(p)], dtype=object)
        Minv = mp.inverse(M)
        r0, r1 = y0 - (F0 * beta).sum(axis=1), y1 - (F1 * beta).sum(axis=1)
    else:
        M, Minv, beta = None, None, np.zeros(0, dtype=object)
        r0, r1 = y0, y1
    al0, al1 = i00 * r0 + i01 * r1, i01 * r0 + i00 * r1
    qv = _fsum(r0 * al0 + r1 * al1)
    W00, W11, W01 = al0 * al0 - i00, al1 * al1 - i00, al0 * al1 - i01
    hh00 = hh11 = hh01 = np.zeros(P, dtype=object)
    if reml and p:
        Mi = np.array([[Minv[j, k] for k in range(p)] for j in range(p)], dtype=object)
        v0, v1 = h0.dot(Mi), h1.dot(Mi)
        hh00, hh11, hh01 = (v0 * h0).sum(axis=1), (v1 * h1).sum(axis=1), (v0 * h1).sum(axis=1)
        W00, W11, W01 = W00 + hh00, W11 + hh11, W01 + hh01
    log2pi = mp.log(2 * mp.pi)
    ldM = mp.log(mp.det(M)) if (reml and p) else mp.mpf(0)
    if reml:
        v = -((n - p) * log2pi + logdet + ldM + qv) / 2
    else:
        v = -(n * log2pi + logdet + qv) / 2
    g, S = [], []
    for t in range(len(diag_d)):
        dd = mp.mpf(float(diag_d[t]))
        o = off_d[t] if getattr(off_d[t], "dtype", None) == object else _obj(off_d[t])
        g.append(_fsum((W00 + W11) * dd / 2 + W01 * o))
        S.append(_fsum((np.abs(W00) + np.abs(W11)) * abs(dd) / 2 + np.abs(W01) * np.abs(o)))
    parts = dict(i00=i00, i01=i01, al0=al0, al1=al1, hh=(hh00, hh11, hh01), W=(W00, W11, W01), M=M, Minv=Minv,
                 logdet=logdet, ldM=ldM, h0=h0, h1=h1)
    return v, list(beta), g, S, qv, logdet, parts


def _f(x):
    return np.asarray(x, dtype=object).astype(np.float64)


# Whole-call error bounds, first order in U, by running error analysis along the device's own operation order.  Every
# product of the pair-local stage is a single nonzero term (the factor, the inverse blocks and every sweep act on the
# 2 x 2 pair blocks; the off-block entries of L and L^-1 are exact zeros), so each pair-local quantity carries the
# relative errors derived for E_W01 above: L00 1, L10 2, L11 1.8125, X00 = 1 / L00 2, X10 7.8125, X11 2.8125 (in U).
# A forward sweep w = X v gives w0 = RN(X00 v0) (2 + 1) and w1 = X10 v0 + X11 v1 (each term its X error, its product
# and one addition: 7.8125 + 2, 2.8125 + 2); a backward sweep x = X' w gives x0 = X00 w0 + X10 w1 (2 + 2, 7.8125 + 2)
# and x1 = RN(X11 w1) (2.8125 + 1).  A fixed-order sum of N terms with reduction depth D (the longest chain of
# additions any term goes through) adds at most D U sum |terms|:
#   log det and q (chol_logdet_kernel, chol_lik_sumsq_kernel): ceil(n / 1024) per thread, then a 10-level tree;
#   F'A^-1 F, F'A^-1 y (chol_gemm_kernel over K = n_p rows): n_p, the bound of a sequential chain (the DMMA order is not
#   assumed);
#   the gradient contraction (kcov_grad_kernel + kcov_grad_reduce_kernel): 32 rows per thread, a 5-level warp tree,
#   8 warps in order, ceil(parts / 32) + 5 over the CTAs of a chunk, ceil(chunks / 32) + 5 over the chunks.
# The drift system: with Delta M, Delta b the errors of M = G'G, b = G'g, the Cholesky factor R and the two triangular
# solves of chol_lik_beta_kernel have backward error (3p + 1) U |R'||R| (Higham, Thm 10.4), so
# |Delta beta| <= |M^-1| (|Delta b| + (|Delta M| + (3p + 1) U |R'||R|) |beta|).  The value does not depend on beta to
# first order (q is minimal at beta), the gradient does, through alpha.
def whole_call_bounds(a, c, y, F, reml, diag_d, off_d, dA_err, rnd, parts, beta):
    """(value bound, beta bounds, gradient bounds, T_v) in absolute units for one loglik call on the pair matrix.
    dA_err[t][q]: error bound of the off-diagonal dA of pair q (absolute); rnd[t]: roundings of one contraction term
    of parameter t (fma, and for a range also RN(du^2), RN(wt dk) and the host's two)."""
    a, c = np.asarray(a, dtype=np.float64), np.asarray(c, dtype=np.float64)
    P, p = a.size, F.shape[1]
    n, n_p = 2 * P, -(-2 * P // 128) * 128
    L00 = np.sqrt(a)
    L11 = np.sqrt(a - c * c / a)
    X00, X10, X11 = 1.0 / L00, -(c / a) / L11, 1.0 / L11

    def fwd(v0, v1):
        """(w0, w1, mu0, mu1): w = X v and its error bound (absolute, units of U) for exact v"""
        x00, x10, x11 = (X00, X10, X11) if v0.ndim == 1 else (X00[:, None], X10[:, None], X11[:, None])
        w0, w1 = x00 * v0, x10 * v0 + x11 * v1
        return w0, w1, 3.0 * np.abs(x00 * v0), 9.8125 * np.abs(x10 * v0) + 4.8125 * np.abs(x11 * v1)

    y0, y1 = y[0::2], y[1::2]
    F0, F1 = F[0::2].reshape(P, p), F[1::2].reshape(P, p)
    g0, g1, mg0, mg1 = fwd(y0, y1)
    G0, G1, mG0, mG1 = fwd(F0, F1) if p else (np.zeros((P, 0)),) * 4
    # log det A = 2 sum log L_ii: 2 (1 + 1.8125) per pair from the factor, the log (1 ulp = 2 U of each term), the sum
    ld_terms = np.concatenate([2 * np.log(L00), 2 * np.log(L11)])
    D_ld = -(-n // 1024) + 10
    B_ld = 5.625 * P + (2 + D_ld) * np.abs(ld_terms).sum()
    betaf = np.array([float(x) for x in beta])
    if p:
        Gabs = np.vstack([np.abs(G0), np.abs(G1)])
        mG = np.vstack([mG0, mG1])
        gabs, mg = np.concatenate([np.abs(g0), np.abs(g1)]), np.concatenate([mg0, mg1])
        dM = mG.T @ Gabs + Gabs.T @ mG + n_p * (Gabs.T @ Gabs)
        db = mG.T @ gabs + Gabs.T @ mg + n_p * (Gabs.T @ gabs)
        Mf = np.array([[float(parts["M"][j, k]) for k in range(p)] for j in range(p)])
        Minvf = np.array([[float(parts["Minv"][j, k]) for k in range(p)] for j in range(p)])
        R = np.linalg.cholesky(Mf).T
        RR = np.abs(R.T) @ np.abs(R)
        dbeta = np.abs(Minvf) @ (db + (dM + (3 * p + 1) * RR) @ np.abs(betaf))
    else:
        dM, dbeta, Minvf, R, RR = np.zeros((0, 0)), np.zeros(0), np.zeros((0, 0)), np.zeros((0, 0)), np.zeros((0, 0))
    # residual e = g - G beta (chol_lik_resid_kernel, p sequential subtractions)
    e0, e1 = g0 - G0 @ betaf, g1 - G1 @ betaf
    de0 = mg0 + mG0 @ np.abs(betaf) + p * (np.abs(g0) + np.abs(G0) @ np.abs(betaf))
    de1 = mg1 + mG1 @ np.abs(betaf) + p * (np.abs(g1) + np.abs(G1) @ np.abs(betaf))
    D_q = -(-n // 1024) + 10
    B_q = 2 * (np.abs(e0) * de0 + np.abs(e1) * de1).sum() + D_q * (e0 * e0 + e1 * e1).sum()
    qf = float((e0 * e0 + e1 * e1).sum())
    logdet = float(parts["logdet"])
    B_ldM, ldM = 0.0, float(parts["ldM"])
    if reml and p:
        B_ldM = (np.abs(Minvf) * (dM + (p + 1) * RR)).sum() + (2 + p) * np.abs(2 * np.log(np.diag(R))).sum()
    host = 5 * ((n - p) * 1.8379 + abs(logdet) + abs(ldM) + qf)
    B_v = 0.5 * (B_ld + B_q + B_ldM + host) * U
    T_v = n + abs(logdet) + qf
    B_beta = dbeta * U
    # gradient: W's pair entries, then the contraction
    # beta's error moves alpha = A^-1 (y - F beta) by -A^-1 F Delta beta: its first-order effect on component t is
    # sum_k D_tk Delta beta_k with D_tk = d grad_t / d beta_k, summed exactly below (signed: it cancels over pairs);
    # every other error of alpha is local
    al0 = X00 * e0 + X10 * e1
    al1 = X11 * e1
    dal0 = np.abs(X00) * de0 + np.abs(X10) * de1 + 4 * np.abs(X00 * e0) + 9.8125 * np.abs(X10 * e1)
    dal1 = np.abs(X11) * de1 + 3.8125 * np.abs(X11 * e1)
    i00, i01 = _f(parts["i00"]), _f(parts["i01"])
    dW = [17.625 * np.abs(i00) + 2 * dal0 * np.abs(al0), 17.625 * np.abs(i00) + 2 * dal1 * np.abs(al1),
          11.625 * np.abs(i01) + dal0 * np.abs(al1) + np.abs(al0) * dal1]
    mag = [np.abs(i00) + al0 * al0, np.abs(i00) + al1 * al1, np.abs(i01) + np.abs(al0 * al1)]
    if reml and p:
        # H = L^-T G R^-1: the row solve h R = G_i (p U |h||R|) and G's own error, then the backward sweep;
        # H H' through R^-1 R^-T = M^-1 moves with Delta M: |Delta (v M^-1 v')| <= |v M^-1| |Delta M| |M^-1 v'|
        Rinv = np.linalg.inv(R)
        hr0, hr1 = G0 @ Rinv, G1 @ Rinv
        dh0 = (mG0 + p * np.abs(hr0) @ np.abs(R)) @ np.abs(Rinv)
        dh1 = (mG1 + p * np.abs(hr1) @ np.abs(R)) @ np.abs(Rinv)
        H0 = X00[:, None] * hr0 + X10[:, None] * hr1
        H1 = X11[:, None] * hr1
        dH0 = (np.abs(X00)[:, None] * dh0 + np.abs(X10)[:, None] * dh1 + 4 * np.abs(X00[:, None] * hr0)
               + 9.8125 * np.abs(X10[:, None] * hr1))
        dH1 = np.abs(X11)[:, None] * dh1 + 3.8125 * np.abs(X11[:, None] * hr1)
        V0, V1 = _f(parts["h0"]).reshape(P, p) @ np.abs(Minvf), _f(parts["h1"]).reshape(P, p) @ np.abs(Minvf)
        V0, V1 = np.abs(V0), np.abs(V1)
        dW[0] = dW[0] + 2 * (dH0 * np.abs(H0)).sum(axis=1) + ((V0 @ dM) * V0).sum(axis=1)
        dW[1] = dW[1] + 2 * (dH1 * np.abs(H1)).sum(axis=1) + ((V1 @ dM) * V1).sum(axis=1)
        dW[2] = dW[2] + (dH0 * np.abs(H1) + np.abs(H0) * dH1).sum(axis=1) + ((V0 @ dM) * V1).sum(axis=1)
        mag[0] = mag[0] + (H0 * H0).sum(axis=1)
        mag[1] = mag[1] + (H1 * H1).sum(axis=1)
        mag[2] = mag[2] + np.abs(H0 * H1).sum(axis=1)
    # the rank update Z = A^-1 - [H alpha][H alpha]' (p + 1 products and the subtraction)
    dW = [dW[k] + (p + 2) * mag[k] for k in range(3)]
    Wf = [_f(w) for w in parts["W"]]
    nchunks = -(-n // 1024)
    nparts = -(-n // 128) * 16
    D_g = 32 + 5 + 8 + (-(-nparts // 32) + 5) + (-(-nchunks // 32) + 5)
    B_g = []
    for t in range(len(diag_d)):
        dd, o, oe = abs(float(diag_d[t])), np.abs(np.asarray(off_d[t], dtype=np.float64)), np.asarray(dA_err[t])
        terms = 0.5 * (np.abs(Wf[0]) + np.abs(Wf[1])) * dd + np.abs(Wf[2]) * o
        err = 0.5 * (dW[0] + dW[1]) * dd + dW[2] * o + np.abs(Wf[2]) * oe / U + rnd[t] * terms
        dbeta_t = 0.0
        if p:
            A0, A1 = _f(parts["al0"]), _f(parts["al1"])
            hA0, hA1 = _f(parts["h0"]).reshape(P, p), _f(parts["h1"]).reshape(P, p)
            of = np.asarray([float(x) for x in np.ravel(off_d[t])])
            for kk in range(p):
                D = -(A0 * hA0[:, kk] + A1 * hA1[:, kk]) * float(diag_d[t]) - (A0 * hA1[:, kk] + hA0[:, kk] * A1) * of
                dbeta_t += abs(math.fsum(D)) * dbeta[kk]
        B_g.append((err.sum() + D_g * terms.sum() + dbeta_t) * U)
    return B_v, B_beta, np.array(B_g), T_v


def pair_points(seps, d, spacing):
    """X (d x 2P): pair q centred on the q-th node of a d-dimensional lattice of the given spacing, its two points at
    -/+ seps[:, q] / 2 from the centre."""
    P = seps.shape[1]
    side = int(np.ceil(P ** (1.0 / d) - 1e-9))
    idx = np.array(np.unravel_index(np.arange(P), (side,) * d), dtype=np.float64) * spacing
    X = np.empty((d, 2 * P))
    X[:, 0::2] = idx - seps / 2
    X[:, 1::2] = idx + seps / 2
    return X


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("reml", [False, True])
@pytest.mark.parametrize("p", [0, 1, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_closed_form_against_host(kind, p, reml):
    """The pair closed form against the dense Cholesky restatement of tests/test_gpu_kcov_lik.py, on host values of a
    and c.  Pairs sit 2000 ranges apart, so the host's cross-pair covariances are exact zeros (exp underflows, the
    spherical is 0 beyond its range); the power law is never zero, so it runs as one pair."""
    from test_gpu_kcov_lik import host_A
    if kind == "powerlaw" and p > 1:
        pytest.skip("not covered: the power law is never zero, so it runs as one pair (n = 2), which takes at most one "
                    "drift column; p = 3 is checked for every other kind")
    d = 2
    rng = np.random.default_rng(CODE[kind] + 10 * p)
    st = CS(kind, 1.3, [1.5, 0.9], beta=0.8)
    P = 1 if kind == "powerlaw" else 12
    seps = rng.uniform(-1.0, 1.0, (d, P))
    X = pair_points(seps, d, 2000.0 * 1.5)
    n = 2 * P
    nug = 0.4
    A, dA = host_A([st], X, nug)
    off_pair = np.zeros_like(A)
    for q in range(P):
        off_pair[2 * q, 2 * q + 1] = off_pair[2 * q + 1, 2 * q] = 1.0
    if kind != "powerlaw":
        assert np.all(A[(off_pair == 0) & ~np.eye(n, dtype=bool)] == 0.0)   # block-diagonal on the host
    y = rng.standard_normal(n) + 0.3
    F = np.column_stack([np.ones(n), X.T / 3000.0, rng.standard_normal(n)])[:, :p]
    if p == 0:
        F = np.zeros((n, 0))
    v, beta, W, _, _ = host_lik(A, y, F, reml)
    g, S = host_grad(W, dA)
    a = [A[2 * q, 2 * q] for q in range(P)]
    c = [A[2 * q, 2 * q + 1] for q in range(P)]
    diag_d = [D[0, 0] for D in dA]
    off_d = [[D[2 * q, 2 * q + 1] for q in range(P)] for D in dA]
    vr, br, gr, Sr, _, _, _ = pairs_closed_form(a, c, y, F, reml, diag_d, off_d)
    assert abs(float(vr) - v) <= 1e-12 * (n + abs(v))
    assert np.allclose([float(x) for x in br], beta, rtol=1e-10, atol=1e-12)
    gr, Sr = np.array([float(x) for x in gr]), np.array([float(x) for x in Sr])
    assert np.all(np.abs(gr - g) <= 1e-11 * S), (gr, g, S)
    assert np.allclose(Sr, S, rtol=1e-12)


def test_checker_rejects_perturbed_derivative():
    """Device results synthesised from the reference pass the per-argument checker at 0.5 times their bound, and the
    checker flags every range component perturbed by 1.5 times its bound in one argument region (exponential, s < 1)."""
    mp = _mp()
    d = 2
    st = CS("exponential", 0.75, [1.3, 0.7])
    rng = np.random.default_rng(3)
    seen = 0
    for s in np.concatenate([10.0 ** rng.uniform(-6, 0, 8), rng.uniform(1, 8, 8)]):
        dirv = rng.standard_normal(d)
        dirv /= np.linalg.norm(dirv)
        X = np.column_stack([np.zeros(d), s * dirv * st.ranges])
        _, r2 = pair_args(st, X)
        k = float(kernel_exact(mp, 0, r2, 1.0)[0])
        a, c = 0.75 + 1.5, 0.75 * k
        comps = pair_components([st], X, 1.5, a, c)
        for factor, in_region_fails in ((0.5, False), (1.5, True)):
            dev = []
            for ref, allow, label in comps:
                bump = factor * allow if (allow is not None and (label[1] == "s<1" or factor == 0.5)) else 0
                dev.append(float(ref + bump) if allow is not None else 0.0)
            ratios = check_components(comps, dev)
            flagged = [lab for lab, r in ratios if r > 1.0]
            if not in_region_fails:
                assert not flagged, ratios
            elif s < 1:
                assert len(flagged) == d and all(lab == (0, "s<1") for lab in flagged), ratios
                seen += 1
            else:
                assert not flagged, ratios
    assert seen == 8


# ------------------------------------------------------------------ GPU: one pair per call
ELL = np.array([1.3, 0.7, 2.1])
SILL, NUG = 0.75, 1.5                 # a = 2.25, |c| <= 0.75 = a / 3: kappa(A_q) <= 2
CARRIER_SILL, CARRIER_NUG = 0.5, 2.0  # flush sweep: a = 3, |c| <= 1


def regular_targets(kind, rng, m):
    """Scaled distances sqrt(r2) the pairs are placed at (kind-specific regions of the issue's sweep)."""
    if kind == "powerlaw":
        return np.sqrt(10.0 ** rng.uniform(-12, 6, m))
    if kind == "spherical":
        k = m // 4
        return np.concatenate([10.0 ** rng.uniform(-8, 0, k), rng.uniform(0, 1, k), 1 - 10.0 ** rng.uniform(-12, -1, k),
                               [1 - 1e-15, 1.0, 1 + 1e-15, 1 + 1e-12], rng.uniform(1, 1.5, m - 3 * k - 4)])
    return np.concatenate([10.0 ** rng.uniform(-8, 0, m // 2), rng.uniform(0, 8, m - m // 2)])


def flush_targets(kind, rng, m):
    """Scaled distances whose exp argument lies around the 2^-1000 flush (y = 693.1)."""
    y = np.concatenate([rng.uniform(680, 705, m - 2), [693.0, 693.3]])
    return np.sqrt(y) if kind == "gaussian" else y


def pair_X(sts, rho, d, rng):
    """Two points whose structure-0 scaled distance is about rho (structure 0 unrotated)."""
    st = sts[0]
    dirv = rng.standard_normal(d)
    dirv /= np.linalg.norm(dirv)
    scale = np.broadcast_to(st.ranges, (d,)) / PRE[st.kind]
    x0 = np.array([0.37, -1.1, 0.52][:d])
    return np.column_stack([x0, x0 + rho * dirv * scale])


def device_pair(gsi, sts, X, nug):
    """(a, c, gradient) of one pair: a and c from the operator applied to the identity (premise: the product is
    symmetric with equal diagonal entries), the gradient from loglik with y = 0, p = 0, ML."""
    if len(sts) == 1:
        st = sts[0]
        op = G.KernelCovMatrix(st.kind, X, st.ranges, sigma2=st.sill, nugget=nug, beta=st.beta)
    else:
        op = G.KernelCovModelMatrix(sts, X, nug)
    try:
        Y = apply_dev(gsi, op, np.eye(2))
        assert Y[0, 0] == Y[1, 1] and Y[0, 1] == Y[1, 0], Y
        _, _, g = G.loglik(op, np.zeros(2), grad=True)
    finally:
        op.free()
    return Y[0, 0], Y[1, 0], g


WORST = {}


def record(ratios):
    for (kind, region), r in ratios:
        key = "nugget" if kind == -1 else f"{KINDS[kind]}:{region}"
        WORST[key] = max(WORST.get(key, 0.0), r)


def report():
    print("LIKREPORT worst error / bound per kind and region: " +
          ", ".join(f"{k} {v:.3f}" for k, v in sorted(WORST.items())))


def run_sweep(gsi, cases):
    bad = []
    for sts, X, nug in cases:
        a, c, g = device_pair(gsi, sts, X, nug)
        comps = pair_components(sts, X, nug, a, c)
        assert len(comps) == g.size
        ratios = check_components(comps, g)
        record(ratios)
        bad += [(lab, r, X.tolist()) for lab, r in ratios if not r <= 1.0]
    report()
    assert not bad, bad[:10]


N_REGULAR, N_FLUSH = 80, 16           # pairs per kind and dimension


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3])
@pytest.mark.parametrize("kind", KINDS)
def test_derivative_per_argument(gsi, kind, d):
    """One pair per call, every component against its bound: a single kind over its argument range, and (exponential
    family) the kind beside a long-range spherical carrier that keeps c, hence W_01, away from zero while the kind's
    own value and derivative approach and cross the 2^-1000 flush."""
    rng = np.random.default_rng(1000 * d + CODE[kind])
    st = CS(kind, SILL, ELL[:d], beta=0.8)
    cases = [([st], pair_X([st], rho, d, rng), NUG) for rho in regular_targets(kind, rng, N_REGULAR)]
    if CODE[kind] in EXP_KINDS:
        model = [CS(kind, CARRIER_SILL, ELL[:d]), CS("spherical", CARRIER_SILL, np.full(d, 1e4))]
        cases += [(model, pair_X(model, rho, d, rng), CARRIER_NUG) for rho in flush_targets(kind, rng, N_FLUSH)]
    run_sweep(gsi, cases)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 3])
def test_derivative_rotated_model(gsi, d):
    """A rotated three-structure model: every structure's sill and range components of one pair per call."""
    rng = np.random.default_rng(77 + d)
    ang = (0.5,) if d == 2 else (0.5, -0.3, 0.8)
    R1, R2 = G.rotation_matrix(ang), G.rotation_matrix(tuple(-0.7 * x for x in ang))
    model = [CS("spherical", 0.4, [2.0, 1.2, 1.6][:d], R1), CS("matern32", 0.3, [0.8, 1.5, 1.1][:d], R2),
             CS("exponential", 0.3, [1.1, 0.9, 1.4][:d])]
    cases = []
    for rho in np.concatenate([10.0 ** rng.uniform(-6, 0, 20), rng.uniform(0.5, 4, 20)]):
        dirv = rng.standard_normal(d)
        dirv /= np.linalg.norm(dirv)
        x0 = np.array([0.37, -1.1, 0.52][:d])
        cases.append((model, np.column_stack([x0, x0 + rho * dirv]), 2.0))
    run_sweep(gsi, cases)


# ------------------------------------------------------------------ GPU: many pairs, whole-call bounds
def drift_of(X, p):
    """[1, xi_0, xi_last] with xi the coordinates mapped to [-1, 1] (xi_0^2 in 1-D): O(1) columns"""
    n = X.shape[1]
    lo, hi = X.min(axis=1), X.max(axis=1)
    xi = (2 * X - (lo + hi)[:, None]) / np.maximum(hi - lo, 1.0)[:, None]
    cols = np.column_stack([np.ones(n), xi[0], xi[-1] if X.shape[0] > 1 else xi[0] ** 2])
    return cols[:, :p]


def pair_case(sts, d, P, seed):
    """Pairs on a d-dimensional lattice 2000 x the largest range apart (every cross-pair covariance is an exact zero on
    the device: fast_exp_neg's argument >= 1024, the spherical's s >= 1); separations keep every structure's s <= 0.9."""
    rng = np.random.default_rng(seed)
    rmax = max(float(np.max(st.ranges)) for st in sts)
    unit = min(float(np.min(st.ranges)) / PRE[st.kind] for st in sts)   # physical length of s = 1 at worst
    dirs = rng.standard_normal((d, P))
    dirs /= np.linalg.norm(dirs, axis=0)
    return pair_points(dirs * rng.uniform(0.05, 0.9, P) * unit, d, 2000.0 * rmax)


def pair_derivatives(sts, X):
    """Per parameter (ABI order): diagonal dA, exact off-diagonal dA per pair (object), its error bound (the bounds
    beside kern_eval / kern_value_deriv at the device's r2), and the roundings of one contraction term."""
    mp = _mp()
    d, P = X.shape[0], X.shape[1] // 2
    diag_d, off_d, err, rnd = [], [], [], []
    for st in sts:
        u = structure_coords(st, X, PRE[st.kind])
        du = u[:, 1::2] - u[:, 0::2]
        ranges = np.broadcast_to(st.ranges, (d,))
        k = np.empty(P, dtype=object)
        dk = np.empty(P, dtype=object)
        kb, db = np.empty(P), np.empty(P)
        for q in range(P):
            r2 = 1e-300 if st.kind in SQRT_KINDS else 0.0
            for v in du[:, q]:
                r2 = fma(float(v), float(v), r2)
            k[q], dk[q], sq, zq, _ = kernel_exact(mp, st.kind, r2, st.beta)
            kb[q] = value_bound_units(st.kind, float(sq), float(zq))
            db[q] = deriv_bound_units(st.kind, float(sq), float(zq))
        diag_d.append(1.0)                                             # dA / dsill_s = k_s (1 on the diagonal)
        off_d.append(k)
        err.append(2 * kb * np.abs(_f(k)) * U)
        rnd.append(1.0)
        for ax in range(d):
            o = -mp.mpf(st.sill) * (2 / mp.mpf(float(ranges[ax]))) * dk * _obj(du[ax]) ** 2
            diag_d.append(0.0)
            off_d.append(o)
            err.append((2 * db + 1) * np.abs(_f(o)) * U)              # + RN(du * du)
            rnd.append(5.0)
    diag_d.append(1.0)
    off_d.append(np.zeros(P, dtype=object) + mp.mpf(0))
    err.append(np.zeros(P))
    rnd.append(1.0)
    return diag_d, off_d, err, rnd


def device_pairs(gsi, op, n):
    """(a, c) per pair from the operator applied to the even / odd indicator columns (row 2q holds a_q, c_q: every other
    term is k * 0 = 0), with the premise checked: both rows of a pair agree, and tiles off the pair blocks of
    gsi_op_kernelcov_block are exact zeros."""
    from test_gpu_kcov_chol import block
    E = np.zeros((n, 2))
    E[0::2, 0] = 1.0
    E[1::2, 1] = 1.0
    Y = apply_dev(gsi, op, E)
    a, c = Y[0::2, 0], Y[1::2, 0]
    assert np.array_equal(Y[1::2, 1], a) and np.array_equal(Y[0::2, 1], c)
    tiles = [(0, 128), (n - 128, 0), (n // 256 * 128, n // 512 * 128)]
    if n > 65536:
        tiles += [(65472, 46336), (n - 64, 65472 - 128)]
    for r0, c0 in tiles:
        rows, cols = min(128, n - r0), min(128, n - c0)
        T = block(gsi, op, r0, c0, rows, cols)
        ri, ci = np.arange(r0, r0 + rows)[:, None], np.arange(c0, c0 + cols)[None, :]
        off = (ri // 2) != (ci // 2)
        assert np.all(T[off] == 0.0), (r0, c0)
    B = block(gsi, op, 0, 0, 64, 64)                                   # inside a factor block: only the pair entries
    ri, ci = np.arange(64)[:, None], np.arange(64)[None, :]
    assert np.all(B[(ri // 2) != (ci // 2)] == 0.0)
    return a, c


def check_whole_call(gsi, sts, X, nug, p, reml, seed, single):
    n = X.shape[1]
    d = X.shape[0]
    rng = np.random.default_rng(seed)
    F = drift_of(X, p)
    y = F @ np.array([0.5, 0.3, -0.2][:p]) + rng.standard_normal(n)
    if single:
        st = sts[0]
        op = G.KernelCovMatrix(st.kind, X, st.ranges, sigma2=st.sill, nugget=nug, beta=st.beta)
    else:
        op = G.KernelCovModelMatrix(sts, X, nug)
    try:
        a, c = device_pairs(gsi, op, n)
        assert np.all(3 * np.abs(c) <= a)                               # kappa(A_q) <= 2
        vd, bd, gd = G.loglik(op, y, drift=F if p else None, reml=reml, grad=True)
    except BaseException:
        op.free()
        raise
    diag_d, off_d, err, rnd = pair_derivatives(sts, X)
    v, beta, g, S, _, _, parts = pairs_closed_form(a, c, y, F, reml, diag_d, off_d)
    B_v, B_b, B_g, T_v = whole_call_bounds(a, c, y, F, reml, diag_d, off_d, err, rnd, parts, beta)
    mp = _mp()
    rv = float(abs(mp.mpf(vd) - v) / (B_v * SECOND_ORDER))
    rb = [float(abs(mp.mpf(float(bd[j])) - beta[j]) / (B_b[j] * SECOND_ORDER)) for j in range(p)]
    rg = [float(abs(mp.mpf(float(gd[t])) - g[t]) / (B_g[t] * SECOND_ORDER)) for t in range(len(g))]
    Sf = np.array([float(x) for x in S])
    c_v, c_g = B_v / (U * T_v), float(np.max(B_g / (U * Sf)))
    print(f"LIKREPORT whole call n={n} d={d} p={p} {'REML' if reml else 'ML'}: value {rv:.3f}, beta "
          f"{max(rb, default=0):.3f}, gradient {max(rg):.3f} of their bounds; bounds c_v = {c_v:.1f} u (n + |logdet| + q), "
          f"c_g = {c_g:.1f} u S_theta (tests/test_gpu_kcov_lik.py: 1e-11 S_theta = {1e-11 / U:.0f} u S_theta)")
    assert rv <= 1.0 and max(rb, default=0) <= 1.0 and max(rg) <= 1.0, (rv, rb, rg)
    return op, a, c


ROT2 = (0.5,)
WHOLE_CASES = {
    "exponential_d2_n258_p0_ml": (lambda: [CS("exponential", 0.75, [1.3, 0.7])], 2, 129, 0, False),
    "matern52_d1_n258_p1_reml": (lambda: [CS("matern52", 0.75, [1.3])], 1, 129, 1, True),
    "spherical_d3_n2050_p3_ml": (lambda: [CS("spherical", 0.75, [1.3, 0.7, 2.1])], 3, 1025, 3, False),
    "nested_d2_n2050_p3_reml": (lambda: [CS("spherical", 0.4, [2.0, 1.2], G.rotation_matrix(0.5)),
                                         CS("matern32", 0.3, [0.8, 1.5], G.rotation_matrix(-0.35)),
                                         CS("exponential", 0.3, [1.1, 0.9])], 2, 1025, 3, True),
    "gaussian_d2_n6000_p1_ml": (lambda: [CS("gaussian", 0.75, [1.3, 0.7])], 2, 3000, 1, False),
    "matern32_d3_n6000_p3_reml": (lambda: [CS("matern32", 0.75, [1.3, 0.7, 2.1])], 3, 3000, 3, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(WHOLE_CASES))
def test_whole_call_pairs(gsi, case):
    """Value, beta and every gradient component of one loglik call on P pairs (n = 258: a ragged last 128-block;
    2 050: three 1024-column chunks of A^-1, the last ragged; 6 000) against the closed form, within the first-order
    bounds of whole_call_bounds."""
    make, d, P, p, reml = WHOLE_CASES[case]
    sts = make()
    nug = 2.0 * sum(st.sill for st in sts)                             # |c| <= total sill <= a / 3
    X = pair_case(sts, d, P, 7 + P + p)
    op, _, _ = check_whole_call(gsi, sts, X, nug, p, reml, 11 + P, single=len(sts) == 1)
    op.free()


@pytest.mark.gpu
def test_past_2_32_factor_entries(gsi):
    """n = 65 600 (n_p = 65 664: the factor has 4.31e9 > 2^32 entries), exponential + rotated spherical, p = 1, REML:
    loglik's value, beta and gradient against the closed form, then KernelCovCholesky on the same operator: log det,
    solve of three right-hand sides and simulate(Xi) (no conditioning data, k = 128), pair by pair."""
    import torch
    free = torch.cuda.mem_get_info()[0]
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory for two 34.5 GB factors in turn, {free / 1e9:.1f} GB free")
    mp = _mp()
    sts = [CS("exponential", 0.6, [1.5, 1.0]), CS("spherical", 0.4, [2.0, 1.2], G.rotation_matrix(0.5))]
    P, d = 32800, 2
    X = pair_case(sts, d, P, 65600)
    n = 2 * P
    op, a, c = check_whole_call(gsi, sts, X, 2.0, 1, True, 65601, single=False)
    try:
        chol = G.KernelCovCholesky(op)
        try:
            L00, L11 = np.sqrt(a), np.sqrt(a - c * c / a)
            X00, X10, X11 = 1.0 / L00, -(c / a) / L11, 1.0 / L11
            # log det: the factor's 2 (1 + 1.8125) per pair, the log's rounding and the fixed-order sum (see
            # whole_call_bounds)
            A_, C_ = _obj(a), _obj(c)
            det = A_ * A_ - C_ * C_
            ld_ref = _fsum(np.frompyfunc(mp.log, 1, 1)(det))
            ld_terms = np.concatenate([2 * np.log(L00), 2 * np.log(L11)])
            B_ld = (5.625 * P + (2 + -(-n // 1024) + 10) * np.abs(ld_terms).sum()) * U
            r_ld = float(abs(mp.mpf(chol.logdet) - ld_ref) / (B_ld * SECOND_ORDER))
            # solve: x = X' (X b) per pair (forward then backward sweep)
            rng = np.random.default_rng(5)
            Bm = rng.standard_normal((n, 3))
            Xs = chol.solve(Bm)
            i00, i01 = A_ / det, -C_ / det
            r_s = 0.0
            for j in range(3):
                b0, b1 = Bm[0::2, j], Bm[1::2, j]
                x0 = i00 * _obj(b0) + i01 * _obj(b1)
                x1 = i01 * _obj(b0) + i00 * _obj(b1)
                w0, w1 = X00 * b0, X10 * b0 + X11 * b1
                mw0, mw1 = 3.0 * np.abs(w0), 9.8125 * np.abs(X10 * b0) + 4.8125 * np.abs(X11 * b1)
                B0 = (np.abs(X00) * mw0 + np.abs(X10) * mw1 + 4 * np.abs(X00 * w0) + 9.8125 * np.abs(X10 * w1)) * U
                B1 = (np.abs(X11) * mw1 + 3.8125 * np.abs(X11 * w1)) * U
                e0 = _f(np.abs(_obj(Xs[0::2, j]) - x0))
                e1 = _f(np.abs(_obj(Xs[1::2, j]) - x1))
                r_s = max(r_s, float(np.max(e0 / (B0 * SECOND_ORDER))), float(np.max(e1 / (B1 * SECOND_ORDER))))
            # simulate, ns = 0: Z = L Xi, Z0 = RN(L00 xi0), Z1 = L10 xi0 + L11 xi1 (chol_trmm_kernel: one nonzero
            # product, or two and their sum); every pair in 8 columns, every column in the first and last 64 pairs
            k = 128
            Xi = rng.standard_normal((n, k))
            Z = chol.simulate(Xi)
            assert Z.shape == (n, k)
            sqrt = np.frompyfunc(mp.sqrt, 1, 1)
            L00e = sqrt(A_)
            L10e, L11e = C_ / L00e, sqrt(det / A_)
            r_z = 0.0
            sel = [(slice(None), range(8)), (slice(0, 64), range(k)), (slice(P - 64, P), range(k))]
            for rows, cols in sel:
                for j in cols:
                    xi0, xi1 = Xi[0::2, j][rows], Xi[1::2, j][rows]
                    z0 = L00e[rows] * _obj(xi0)
                    z1 = L10e[rows] * _obj(xi0) + L11e[rows] * _obj(xi1)
                    B0 = 2 * np.abs(L00[rows] * xi0) * U
                    B1 = (4 * np.abs((c / L00)[rows] * xi0) + 3.8125 * np.abs(L11[rows] * xi1)) * U
                    e0 = _f(np.abs(_obj(Z[0::2, j][rows]) - z0))
                    e1 = _f(np.abs(_obj(Z[1::2, j][rows]) - z1))
                    r_z = max(r_z, float(np.max(e0 / (B0 * SECOND_ORDER))), float(np.max(e1 / (B1 * SECOND_ORDER))))
            print(f"LIKREPORT n={n} KernelCovCholesky: logdet {r_ld:.3f}, solve {r_s:.3f}, simulate {r_z:.3f} of their "
                  f"bounds")
            assert r_ld <= 1.0 and r_s <= 1.0 and r_z <= 1.0, (r_ld, r_s, r_z)
        finally:
            chol.free()
    finally:
        op.free()
