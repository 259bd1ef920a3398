"""Host references that are exact, or far more precise than fp64, for the operators the INT8 tensor-core
kernels emulate (csrc/i8_planes.cuh): tests/test_exact_ref.py checks them against rational arithmetic, and
tests/test_gpu_i8_exact.py checks the kernels against them.

* ``exact_dot_rows``: the correctly rounded fp64 value of sum_k X[i,k] Y[j,k] for sampled (i, j);
* ``woodbury_lnlike``: log det K, r^T K^-1 r and the Gaussian log-likelihood for K = diag(d) + U U^T with a
  thin U, in 50-digit arithmetic, independent of any Cholesky factorisation;
* ``phase_fp64``, ``interp_cov_mp``, ``temporal_k_mp``: the phase of spb_phase bit for bit, and the marginal
  interpolant and the temporal kernels in mpmath, for the predict building blocks (tests/test_gpu_dmma_exact.py).
"""
import math

import numpy as np

_SPLIT = 134217729.0   # 2^27 + 1: Veltkamp's splitting constant for fp64


def _veltkamp(a):
    with np.errstate(invalid="ignore", over="ignore"):   # rows with inf / NaN are not used
        return _veltkamp_(a)


def _veltkamp_(a):
    c = _SPLIT * a
    hi = c - (c - a)
    return hi, a - hi


def exact_dot_rows(X, Y, pairs):
    """fp64 values of sum_k X[i, k] Y[j, k] for the (i, j) rows of ``pairs`` ((P, 2) integers), each
    correctly rounded from the exact sum.

    Every row is first scaled by a power of two to a maximum in [1/2, 1) (exact), every factor is split
    in two 26-bit halves (Veltkamp), so that each product is the exact sum of four doubles, and the 4K
    terms are summed exactly by ``math.fsum``; the result is scaled back with ``math.ldexp``.  Exact
    apart from two places that sit far below any tolerance built on it: a term more than 2^-900 below
    the largest product of its row pair (its halves underflow), and a result in the subnormal range
    (rounded twice, by at most one subnormal ulp).  A sum beyond the fp64 range gives +-inf; rows with a
    NaN or an infinity give NaN."""
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    out = np.empty(len(pairs), dtype=np.float64)

    def scaled(A):
        fin = np.all(np.isfinite(A), axis=1)
        mx = np.where(fin, np.max(np.abs(np.where(np.isfinite(A), A, 0.0)), axis=1), 0.0)
        ex = np.frexp(mx)[1].astype(np.int64)
        return np.ldexp(A, -ex[:, None]), ex, fin, mx > 0.0

    Xs, ex_x, fin_x, nz_x = scaled(X)
    Ys, ex_y, fin_y, nz_y = scaled(Y)
    xh, xl = _veltkamp(Xs)
    yh, yl = _veltkamp(Ys)
    for q, (i, j) in enumerate(pairs):
        if not (fin_x[i] and fin_y[j]):
            out[q] = math.nan
            continue
        if not (nz_x[i] and nz_y[j]):
            out[q] = 0.0
            continue
        terms = np.concatenate((xh[i] * yh[j], xh[i] * yl[j], xl[i] * yh[j], xl[i] * yl[j]))
        s = math.fsum(terms.tolist())
        try:
            out[q] = math.ldexp(s, int(ex_x[i] + ex_y[j]))
        except OverflowError:   # beyond the fp64 range: rounds to +-inf
            out[q] = math.copysign(math.inf, s)
    return out


def woodbury_lnlike(d, U, R, dps=50):
    """K = diag(d) + U U^T (d: (nt,) > 0, U: (nt, k), k <= 8), right-hand sides R: (M, nt).

    Returns (logdet K, quad (M,) = r^T K^-1 r, lnlike = -1/2 sum quad - M/2 logdet K - nt M/2 log 2 pi),
    as mpmath numbers (``dps`` digits); convert with ``float``.  Matrix determinant lemma and Woodbury:
        logdet K  = sum log d + logdet C,                  C = I + U^T D^-1 U   (k x k)
        r^T K^-1 r = r^T D^-1 r - w^T C^-1 w,             w = U^T D^-1 r
    every sum over the nt time stamps is taken by ``mpmath.fdot`` at ``dps`` digits, and C is solved by
    an mpmath Cholesky at the same precision."""
    import mpmath

    d = np.asarray(d, dtype=np.float64)
    U = np.asarray(U, dtype=np.float64)
    R = np.atleast_2d(np.asarray(R, dtype=np.float64))
    nt, k = U.shape
    with mpmath.workdps(dps):
        one = mpmath.mpf(1)
        dinv = [one / mpmath.mpf(float(v)) for v in d]
        cols = [[mpmath.mpf(float(v)) for v in U[:, a]] for a in range(k)]
        dcols = [[c * w for c, w in zip(col, dinv)] for col in cols]
        C = mpmath.matrix(k, k)
        for a in range(k):
            for b in range(a + 1):
                C[a, b] = C[b, a] = mpmath.fdot(dcols[a], cols[b]) + (one if a == b else 0)
        L = mpmath.cholesky(C) if k else C
        logdet = mpmath.fsum(mpmath.log(mpmath.mpf(float(v))) for v in d)
        logdet += 2 * mpmath.fsum(mpmath.log(L[a, a]) for a in range(k))
        quad = []
        for r in R:
            rm = [mpmath.mpf(float(v)) for v in r]
            rd = [x * w for x, w in zip(rm, dinv)]
            q = mpmath.fdot(rd, rm)
            if k:
                w = mpmath.matrix([mpmath.fdot(dcols[a], rm) for a in range(k)])
                z = _forward(L, w, k)   # w^T C^-1 w = |L^-1 w|^2
                q -= mpmath.fsum(z[a] ** 2 for a in range(k))
            quad.append(q)
        M = len(quad)
        ll = -mpmath.fsum(quad) / 2 - M * logdet / 2 - mpmath.mpf(nt * M) / 2 * mpmath.log(2 * mpmath.pi)
    return logdet, quad, ll


TWO_PI = 2.0 * 3.14159265358979323846   # the fp64 constant of spb_phase (pi rounded, doubled exactly)


def phase_fp64(t, period):
    """spb_phase (csrc/common.cuh) bit for bit: x = fl(t / p), w = floor(x), theta = fl(TWO_PI fl(x - w)), the
    same three IEEE roundings as on the device.  x - w is exact for x >= 0; for x just below a negative
    integer it rounds up to exactly 1 and theta to exactly TWO_PI."""
    x = np.asarray(t, dtype=np.float64) / np.float64(period)
    return TWO_PI * (x - np.floor(x))


def interp_cov_mp(cf, covpts, s):
    """The cubic interpolant of flux.py:256-276 (csrc/assemble.cu interp_cov) evaluated exactly (mpmath at the
    working precision) on a coefficient table cf (4, covpts + 1) at the scaled lag s = |dtheta| covpts / 2pi:
    bin ind = floor(s) (at most covpts), x0 = s - ind, value sum_k cf[k][ind] x0^k."""
    import mpmath

    s = mpmath.mpf(s)
    ind = min(int(mpmath.floor(s)), covpts)
    x0 = s - ind
    return mpmath.fsum(mpmath.mpf(float(cf[k][ind])) * x0 ** k for k in range(4)), ind


def temporal_k_mp(kind, dt, tau):
    """temporal.py:8-16 in mpmath at the working precision, on the fp64 inputs dt = |t1 - t2| (exact) and tau:
    kind 1 Matern-3/2 (1 + x) e^-x with x = sqrt(3) dt / tau, kind 2 exp(-dt^2 / (2 tau)).  Also returns the
    condition number x |d ln k / dx| of k in its argument: x^2 / (1 + x) for kind 1, dt^2 / (2 tau) for kind 2."""
    import mpmath

    dt, tau = mpmath.mpf(dt), mpmath.mpf(tau)
    if kind == 1:
        x = mpmath.sqrt(3) * dt / tau
        return (1 + x) * mpmath.exp(-x), x * x / (1 + x)
    a = dt * dt / (2 * tau)
    return mpmath.exp(-a), a


def _forward(L, w, k):
    """L^-1 w for a lower-triangular mpmath matrix L."""
    z = [None] * k
    for a in range(k):
        z[a] = (w[a] - sum((L[a, b] * z[b] for b in range(a)), 0)) / L[a, a]
    return z
