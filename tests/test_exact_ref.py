"""CPU: the host references of tests/exact_ref.py against rational arithmetic (fractions.Fraction) and
against a dense 60-digit evaluation, so that the GPU tests built on them (tests/test_gpu_i8_exact.py)
compare the kernels with something already trusted."""
import itertools
import math
from fractions import Fraction

import numpy as np

from exact_ref import TWO_PI, exact_dot_rows, interp_cov_mp, phase_fp64, temporal_k_mp, woodbury_lnlike


def test_phase_fp64_against_fractions():
    """theta = fl(TWO_PI fl(x - floor(x))), x = fl(t / p), each step correctly rounded; t just below a negative
    multiple of p gives exactly TWO_PI."""
    rng = np.random.default_rng(6)
    t = np.r_[rng.uniform(-50, 50, 200), 0.0, 3.0, -3.0, -3.0 * (1 + 2.0 ** -52), -1e-20]
    p = 1.5
    th = phase_fp64(t, p)
    for tv, g in zip(t, th):
        x = float(Fraction(tv) / Fraction(p))
        frac = float(Fraction(x) - math.floor(x))
        assert g == float(Fraction(TWO_PI) * Fraction(frac)), tv
    assert th[-1] == TWO_PI and th[-5] == 0.0
    assert np.all((th >= 0) & (th <= TWO_PI))


def test_interp_cov_mp_against_fractions():
    """The interpolant at rational lags, against the cubic evaluated in rational arithmetic; the bin of a lag on
    a knot is the upper one, and s = covpts takes the last bin with x0 = 0."""
    import mpmath

    rng = np.random.default_rng(7)
    covpts = 6
    cf = rng.standard_normal((4, covpts + 1))
    with mpmath.workdps(40):
        for s in (Fraction(0), Fraction(1, 3), Fraction(2), Fraction(47, 10), Fraction(covpts)):
            v, ind = interp_cov_mp(cf, covpts, mpmath.mpf(s.numerator) / s.denominator)
            i = min(math.floor(s), covpts)
            x0 = s - i
            want = sum(Fraction(float(cf[k][i])) * x0 ** k for k in range(4))
            assert ind == i
            assert abs(v - mpmath.mpf(want.numerator) / want.denominator) <= mpmath.mpf(10) ** -35 * (1 + abs(v))


def test_temporal_k_mp_closed_forms():
    """Matern-3/2 at x = 1 is 2/e, the squared exponential at dt^2 / (2 tau) = 1 is 1/e, both are 1 at dt = 0;
    the condition numbers are x^2 / (1 + x) and dt^2 / (2 tau)."""
    import mpmath

    with mpmath.workdps(40):
        k, c = temporal_k_mp(1, 2.0, 2.0 * math.sqrt(3))   # x = sqrt(3) 2 / fl(2 sqrt 3) = 1 (1 + O(u))
        x = mpmath.sqrt(3) * 2 / mpmath.mpf(2.0 * math.sqrt(3))
        assert abs(k - (1 + x) * mpmath.exp(-x)) < mpmath.mpf(10) ** -38
        assert abs(k - 2 / mpmath.e) < 1e-15 and abs(c - mpmath.mpf(1) / 2) < 1e-15
        k, c = temporal_k_mp(2, 2.0, 2.0)
        assert abs(k - 1 / mpmath.e) < mpmath.mpf(10) ** -38 and c == 1
        assert temporal_k_mp(1, 0.0, 3.0)[0] == 1 and temporal_k_mp(2, 0.0, 3.0)[0] == 1


def _adversarial_rows(rng, K):
    rows = [rng.standard_normal(K),                                   # full mantissas
            np.where(np.arange(K) % 2 == 0, 1.0, 1e-30) * rng.standard_normal(K),   # 30 decades
            np.full(K, 2.0 ** 40) * (1 - 2.0 ** -53) * np.sign(rng.standard_normal(K)),
            np.zeros(K),
            rng.standard_normal(K) * 1e-310,                          # subnormals only
            rng.standard_normal(K) * 1e150,
            rng.standard_normal(K) * 1e-160]
    return np.array(rows)


def test_exact_dot_rows_is_the_correctly_rounded_product():
    rng = np.random.default_rng(1)
    X = _adversarial_rows(rng, 5)
    Y = _adversarial_rows(rng, 5)[::-1].copy()
    pairs = np.array(list(itertools.product(range(len(X)), range(len(Y)))))
    got = exact_dot_rows(X, Y, pairs)
    for (i, j), g in zip(pairs, got):
        exact = sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(X[i], Y[j]))
        want = float(exact)   # Fraction -> float rounds to nearest
        assert g == want or (abs(want) < 2.3e-308 and abs(g - want) <= 5e-324), (i, j, g, want)
    # cancellation: the exact sum is far below the terms
    x = np.array([[1.0, 2.0 ** -60, -1.0, 3.0]])
    y = np.array([[1.0, 1.0, 1.0, 2.0 ** -70]])
    assert exact_dot_rows(x, y, [[0, 0]])[0] == 2.0 ** -60 + 3.0 * 2.0 ** -70
    # a non-finite entry makes the row NaN
    x2 = np.array([[1.0, math.nan], [1.0, math.inf]])
    assert np.all(np.isnan(exact_dot_rows(x2, y[:, :2], [[0, 0], [1, 0]])))


def test_exact_dot_rows_6x5_against_fractions():
    rng = np.random.default_rng(2)
    X = rng.standard_normal((6, 5)) * np.exp2(rng.integers(-40, 40, (6, 5)))
    Y = rng.standard_normal((6, 5))
    pairs = np.array(list(itertools.product(range(6), range(6))))
    got = exact_dot_rows(X, Y, pairs)
    for (i, j), g in zip(pairs, got):
        want = float(sum(Fraction(float(a)) * Fraction(float(b)) for a, b in zip(X[i], Y[j])))
        assert g == want


def test_woodbury_lnlike_against_dense_high_precision():
    import mpmath

    rng = np.random.default_rng(3)
    nt, k, M = 40, 3, 2
    d = rng.uniform(0.01, 2.0, nt)
    U = rng.standard_normal((nt, k))
    R = rng.standard_normal((M, nt))
    logdet, quad, ll = woodbury_lnlike(d, U, R)
    with mpmath.workdps(60):
        Km = mpmath.matrix(nt, nt)
        for i in range(nt):
            for j in range(nt):
                Km[i, j] = mpmath.fsum(mpmath.mpf(float(U[i, a])) * mpmath.mpf(float(U[j, a]))
                                       for a in range(k)) + (mpmath.mpf(float(d[i])) if i == j else 0)
        L = mpmath.cholesky(Km)
        ld = 2 * mpmath.fsum(mpmath.log(L[i, i]) for i in range(nt))
        assert abs(ld - logdet) < mpmath.mpf(10) ** -40 * abs(ld)
        for m in range(M):
            r = mpmath.matrix([mpmath.mpf(float(v)) for v in R[m]])
            y = mpmath.lu_solve(L, r)
            q = mpmath.fsum(v ** 2 for v in y)
            assert abs(q - quad[m]) < mpmath.mpf(10) ** -40 * q
        want = -mpmath.fsum(
            [mpmath.fsum(v ** 2 for v in mpmath.lu_solve(L, mpmath.matrix([mpmath.mpf(float(x)) for x in R[m]])))
             for m in range(M)]) / 2 - M * ld / 2 - nt * M * mpmath.log(2 * mpmath.pi) / 2
        assert abs(want - ll) < mpmath.mpf(10) ** -40 * abs(want)
    # rank 0 and the no-right-hand-side case reduce to the diagonal
    ld0, q0, ll0 = woodbury_lnlike(d, np.zeros((nt, 0)), R[:1])
    assert abs(float(ld0) - float(np.sum(np.log(d)))) < 1e-12 * abs(float(ld0))
    assert abs(float(q0[0]) - float(np.sum(R[0] ** 2 / d))) < 1e-12 * float(q0[0])
