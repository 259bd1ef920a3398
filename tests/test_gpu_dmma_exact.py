"""GPU (-m gpu): the FP64 tensor-core (DMMA) GEMM of csrc/gemm_nt.cuh, its callers and the small kernels of
predict and sampling against exact or high-precision host references (tests/exact_ref.py).

Every product is checked entry by entry against the correctly rounded value under the a-priori bound
    |C - C_exact| <= gamma_k sum_k |a_k b_k|,     gamma_k = k u / (1 - k u),  u = 2^-53,
with k the number of products plus the partial sums added afterwards (split-K partials, beta C, a row
vector).  Dropping a 16-wide K chunk, using a wrong edge row or reading past K breaks it by orders of
magnitude.  Entries with a subnormal result may lose one more absolute 2^-1074 per rounding (k 2^-1074).

  1. spb_gemm_nt (EPI_AXPBY): tile-edge shapes, K below / across the 3-stage ring, leading dimensions with
     NaN padding, C unaligned with sentinels, beta = 0 with NaN C, adversarial rows, non-finite operands,
     argument rejections;
  2. spb_flux_conditional(_lower) on the DMMA path: T = A Sigma, K = T A^T, the GP mean, the lower-only
     contract and the chunk loop (COND_CHUNK = 512);
  3. spb_flux_marginal: Omega(u), the 32 split-K partials of a_m = <Omega_m(u), Sigma> and the pass
     boundary of 32768 elements;
  4. spb_sample_ylm, spb_cho_cov_ylm, spb_tril, spb_temporal_scale, spb_cross_marginal.
"""
import ctypes
import math

import numpy as np
import pytest

from conftest import U_LD
from exact_ref import TWO_PI, exact_dot_rows, interp_cov_mp, phase_fp64, temporal_k_mp

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

U64 = 2.0 ** -53
TINY = 2.0 ** -1074
SENT = -3.25e77   # never a value of any output
_KEEP = []        # device copies made by dev(): alive until the end of the test that made them


@pytest.fixture(autouse=True)
def _release_device_copies():
    yield
    _KEEP.clear()


def gamma(k):
    return k * U64 / (1 - k * U64)


@pytest.fixture(scope="module")
def spb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


@pytest.fixture(scope="module")
def ctx(spb):
    return spb.get_context()


def P(t, off=0):
    return ctypes.c_void_p(t.data_ptr() + 8 * off) if t is not None else None


def dev(a):
    """A device copy kept alive until the end of the test, so that a pointer taken from it stays valid."""
    t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()
    _KEEP.append(t)
    return t


def _abs_bound(X, Y, pairs, k):
    """gamma_k sum |x y| for the pairs; the sum of the absolute products is itself correctly rounded (relative
    u), which the factor (1 + 2u) covers, plus k 2^-1074 for roundings in the subnormal range."""
    S = exact_dot_rows(np.abs(X), np.abs(Y), pairs)
    return gamma(k) * S * (1 + 2 * U64) + k * TINY


def _edges(n, rng, extra=0):
    e = {0, 1, 63, 64, 65, 127, 128, 129, n - 2, n - 1}
    e |= set(int(x) for x in rng.integers(0, n, extra))
    return sorted(i for i in e if 0 <= i < n)


def _pairs(M, N, rng, nrand=50):
    """every (tile-edge row, tile-edge column) pair plus nrand random entries"""
    p = {(i, j) for i in _edges(M, rng) for j in _edges(N, rng)}
    p |= {(int(rng.integers(M)), int(rng.integers(N))) for _ in range(nrand)}
    return np.array(sorted(p), dtype=np.int64)


# ------------------------------------------------------------------------------------------------
# 1. spb_gemm_nt
# ------------------------------------------------------------------------------------------------
def _gemm_call(ctx, batch, M, N, K, alpha, A, lda, sA, Bm, ldb, sB, beta, C, ldc, sC, offA=0, offB=0, offC=0):
    return ctx.lib.spb_gemm_nt(ctx.handle, batch, M, N, K, float(alpha), P(A, offA), lda, sA, P(Bm, offB), ldb,
                               sB, float(beta), P(C, offC), ldc, sC, None)


def _run_gemm(ctx, Ah, Bh, K, batch, alpha, beta, ldc, C0=None, gap=3):
    """Ah: (nA, M, lda), Bh: (nB, N, ldb) with nA, nB in {1, batch} (1 = stride 0).  C lives one double past a
    16-byte boundary, after a sentinel, with `gap` sentinel doubles between consecutive matrices and padding
    columns N..ldc-1 filled with the sentinel too.  Returns C (batch, M, N) and asserts every sentinel kept."""
    nA, M, lda = Ah.shape
    nB, N, ldb = Bh.shape
    sC = M * ldc + gap
    off = 3   # odd: C is 8-byte but not 16-byte aligned
    buf = np.full(off + batch * sC + 5, SENT)
    view = buf[off:off + batch * sC].reshape(batch, sC)[:, :M * ldc].reshape(batch, M, ldc)
    view[:, :, :N] = np.nan if C0 is None else C0
    Cd = dev(buf)
    st = _gemm_call(ctx, batch, M, N, K, alpha, dev(Ah), lda, 0 if nA == 1 else M * lda, dev(Bh), ldb,
                    0 if nB == 1 else N * ldb, beta, Cd, ldc, sC, offC=off)
    from starry_process_b200 import _lib

    _lib.check(st)
    out = Cd.cpu().numpy()
    res = out[off:off + batch * sC].reshape(batch, sC)[:, :M * ldc].reshape(batch, M, ldc)
    mask = np.ones(out.shape, bool)
    mview = mask[off:off + batch * sC].reshape(batch, sC)[:, :M * ldc].reshape(batch, M, ldc)
    mview[:, :, :N] = False
    assert np.all(out[mask] == SENT), "a sentinel before, between, after or beside the C matrices was written"
    return res[:, :, :N].copy()


def _operands(rng, n, rows, K, ld):
    X = np.full((n, rows, ld), np.nan)   # NaN padding columns K..ld-1: never read
    X[:, :, :K] = rng.standard_normal((n, rows, K))
    return X


def _check_gemm(A, B, C, C0, alpha, beta, K, pairs, batch):
    """C[b] = alpha A[b] B[b]^T + beta C0[b] within gamma_{K+2} (|alpha| sum |a b| + |beta C0|): the K products and
    their sums (gamma_K), alpha v (one rounding) and fma(alpha, v, beta c) with beta c rounded (two).  The host
    value alpha ex + beta c0 is itself rounded four times (ex, both products, the sum): gamma_{K+6} in all."""
    for b in range(batch):
        Ab = A[min(b, len(A) - 1)][:, :K]
        Bb = B[min(b, len(B) - 1)][:, :K]
        ex = exact_dot_rows(Ab, Bb, pairs)
        S = exact_dot_rows(np.abs(Ab), np.abs(Bb), pairs)
        c0 = C0[b][pairs[:, 0], pairs[:, 1]] if beta != 0 else 0.0
        want = alpha * ex + beta * c0
        bnd = gamma(K + 6) * (abs(alpha) * S + abs(beta * c0)) * (1 + 4 * U64) + (K + 6) * TINY
        got = C[b][pairs[:, 0], pairs[:, 1]]
        assert np.all(np.isfinite(got)), b
        err = np.abs(got - want)
        bad = np.nonzero(err > bnd)[0]
        assert len(bad) == 0, [(tuple(pairs[q]), got[q], want[q], bnd[q]) for q in bad[:5]]


MN = [1, 7, 8, 31, 63, 64, 65, 127, 128, 129, 300]
KS = [2, 4, 14, 16, 18, 30, 32, 34, 48, 256, 1000, 4096]
LAYOUTS = [(1, False, False), (3, False, False), (3, True, False), (3, False, True)]   # batch, shared A, shared B
SCALARS = [(1.0, 0.0), (-0.75, 0.0), (1.5, -2.25), (0.3, 1.0)]


@pytest.mark.parametrize("K", KS)
def test_gemm_nt_against_exact(ctx, K):
    """Every M and N of MN at this K (paired cyclically, so each value meets several partners across K), the
    batch layouts, leading dimensions lda, ldb in {K, K + 2, K + 6} with NaN padding, ldc odd or N, and the
    (alpha, beta) pairs, beta = 0 with a NaN-filled C (must not be read)."""
    rng = np.random.default_rng(K)
    shift = KS.index(K) % len(MN)
    for q, (M, N) in enumerate(zip(MN, MN[shift:] + MN[:shift])):
        batch, shA, shB = LAYOUTS[q % 4]
        alpha, beta = SCALARS[(q + shift) % 4]
        lda = K + (0, 2, 6)[q % 3]
        ldb = K + (6, 0, 2)[q % 3]
        ldc = N + (1 if N % 2 == 0 else 2) if q % 2 == 0 else N
        A = _operands(rng, 1 if shA else batch, M, K, lda)
        B = _operands(rng, 1 if shB else batch, N, K, ldb)
        C0 = rng.standard_normal((batch, M, N)) if beta != 0 else None
        C = _run_gemm(ctx, A, B, K, batch, alpha, beta, ldc, C0=C0)
        _check_gemm(A, B, C, C0, alpha, beta, K, _pairs(M, N, rng), batch)


def _adversarial(rng, rows, K):
    X = rng.standard_normal((rows, K))
    h = K // 2
    for i in range(0, rows, 6):
        case = (i // 6) % 6
        if case == 0:
            X[i] *= np.where(np.arange(K) % 2 == 0, 1.0, 1e-30)   # 30 decades in one row
        elif case == 1:
            X[i, h:2 * h] = -X[i, :h]                              # cancels against a row of equal halves
        elif case == 2:
            X[i] = 0.0
        elif case == 3:
            X[i] *= 1e-310                                         # subnormals
        elif case == 4:
            X[i] *= 1e300
    return X


@pytest.mark.parametrize("K", [34, 1000])
def test_gemm_nt_adversarial_rows(ctx, K):
    """Rows spanning 30 decades, rows whose exact dot product is 0 (the halves of A cancel against B rows with
    equal halves), zero rows, subnormal rows and rows near 1e300 (against unit rows), at M = N = 129."""
    rng = np.random.default_rng(100 + K)
    M = N = 129
    A = _adversarial(rng, M, K)[None]
    B = rng.standard_normal((N, K))
    B[1::6, K // 2:2 * (K // 2)] = B[1::6, :K // 2]   # equal halves: exact cancellation with A's case-1 rows
    B = B[None]
    C = _run_gemm(ctx, A, B, K, 1, 1.0, 0.0, N)
    zero = [(i, j) for i in range(6, M, 36) for j in range(1, N, 6)]   # case-1 rows against equal-half rows
    pairs = np.concatenate([_pairs(M, N, rng, nrand=200), [(i, j) for i in range(0, M, 6) for j in (0, 1, 64, 128)],
                            zero])
    _check_gemm(A, B, C, None, 1.0, 0.0, K, pairs, 1)
    assert np.all(exact_dot_rows(A[0], B[0], zero) == 0.0)   # the cancellation rows do cancel exactly


@pytest.mark.parametrize("where", ["A", "B"])
@pytest.mark.parametrize("val", [np.inf, np.nan])
def test_gemm_nt_nonfinite_rows(ctx, where, val):
    """An inf or NaN in row r of A[1] (column c of B[1]^T) makes exactly row r (column c) of C[1] non-finite; every
    other entry, and the other elements, bit-identical to a clean run.  M = 129, N = 65: edge tiles whose
    out-of-range rows are zero-filled and must inject nothing."""
    rng = np.random.default_rng(7)
    M, N, K, batch = 129, 65, 34, 3
    A = _operands(rng, batch, M, K, K)
    B = _operands(rng, batch, N, K, K)
    clean = _run_gemm(ctx, A, B, K, batch, 1.0, 0.0, N)
    r = 128 if where == "A" else 64
    A2, B2 = A.copy(), B.copy()
    (A2 if where == "A" else B2)[1, r, 17] = val
    C = _run_gemm(ctx, A2, B2, K, batch, 1.0, 0.0, N)
    bad = np.zeros((M, N), bool)
    if where == "A":
        bad[r, :] = True
    else:
        bad[:, r] = True
    assert np.all(~np.isfinite(C[1][bad]))
    assert np.array_equal(C[1][~bad], clean[1][~bad])
    assert np.array_equal(C[[0, 2]], clean[[0, 2]])


def test_gemm_nt_rejections(ctx):
    """Every malformed call returns non-zero with a message and launches nothing."""
    d = torch.zeros(4096, dtype=torch.float64, device="cuda")
    ok = dict(batch=1, M=4, N=4, K=8, lda=8, sA=0, ldb=8, sB=0, ldc=4, sC=0, offA=0, offB=0)
    bad = [dict(K=7, lda=8, ldb=8), dict(lda=9), dict(ldb=9), dict(offA=1), dict(offB=1), dict(sA=33, batch=2),
           dict(sB=33, batch=2), dict(batch=65536), dict(M=0), dict(N=0), dict(K=0), dict(M=-1), dict(K=-2),
           dict(lda=6), dict(ldb=6), dict(ldc=3)]
    n0 = ctx.launches()
    for kw in bad:
        a = dict(ok, **kw)
        st = _gemm_call(ctx, a["batch"], a["M"], a["N"], a["K"], 1.0, d, a["lda"], a["sA"], d, a["ldb"], a["sB"],
                        0.0, d, a["ldc"], a["sC"], offA=a["offA"], offB=a["offB"])
        assert st != 0, kw
        assert ctx.lib.spb_last_error(), kw
    assert ctx.launches() == n0
    assert _gemm_call(ctx, 1, 4, 4, 8, 1.0, d, 8, 0, d, 8, 0, 0.0, d, 4, 0) == 0


# ------------------------------------------------------------------------------------------------
# 2. spb_flux_conditional on the DMMA path
# ------------------------------------------------------------------------------------------------
def _sym(rng, B):
    X = rng.standard_normal((B, 256, 256))
    return (X + X.transpose(0, 2, 1)) / 2   # exactly symmetric: the sum commutes, the halving is exact


def _conditional(ctx, A, B, cov, mean, ldk, lower):
    nt = A.shape[-2]
    shared = A.ndim == 2
    Kd = torch.full((B, nt, ldk), SENT, dtype=torch.float64, device="cuda")
    gpm = torch.empty(B, dtype=torch.float64, device="cuda")
    nb = ctx.lib.spb_flux_conditional_workspace_bytes(ctx.handle, B, nt)
    ws = torch.zeros(nb, dtype=torch.uint8, device="cuda")
    fn = ctx.lib.spb_flux_conditional_lower if lower else ctx.lib.spb_flux_conditional
    from starry_process_b200 import _lib

    covd = cov if torch.is_tensor(cov) else dev(cov)
    _lib.check(fn(ctx.handle, B, nt, P(dev(A)), 0 if shared else nt * 256, P(dev(mean)), P(covd), P(gpm), P(Kd),
                  ldk, P(ws), nb, None))
    torch.cuda.synchronize()
    Bc = B - (B - 1) // 512 * 512
    T = ws[:Bc * nt * 256 * 8].view(torch.float64).view(Bc, nt, 256).cpu().numpy()
    return Kd.cpu().numpy(), gpm.cpu().numpy(), T


@pytest.mark.parametrize("nt", [1, 2, 63, 129, 300, 1000, 1030])
def test_flux_conditional_dmma_against_exact(ctx, nt):
    """B = 3, per-element A (B <= 512: one chunk, T of every element at the head of the workspace):
      T = A Sigma within gamma_256 sum |A Sigma|, K = T A^T within gamma_256 sum |T A| (on the kernel's own T),
      gp_mean = (A mean)[0] within gamma_256 (products and any summation order); each plus u for the
      correctly rounded reference (gamma_257);
    the lower-only call writes the lower triangle bit-identically to the mirrored one and leaves the strict upper
    triangle and the padding columns untouched; the mirrored K is bitwise symmetric.  nt = 1030 runs with
    moments_syrk_i8 off (the DMMA product at nt >= 1024)."""
    rng = np.random.default_rng(nt)
    B = 3
    A = rng.standard_normal((B, nt, 256))
    cov = _sym(rng, B)
    mean = rng.standard_normal((B, 256))
    ldk = nt + 2 if nt % 2 == 0 else nt + 1
    try:
        if nt >= 1024:
            ctx.set_option("moments_syrk_i8", 0)
        Kf, gf, T = _conditional(ctx, A, B, cov, mean, ldk, lower=False)
        Kl, gl, Tl = _conditional(ctx, A, B, cov, mean, ldk, lower=True)
    finally:
        ctx.set_option("moments_syrk_i8", 1)
    assert np.array_equal(T, Tl) and np.array_equal(gf, gl)
    low = np.tril(np.ones((nt, nt), bool))
    for b in range(B):
        pT = _pairs(nt, 256, rng)
        ex = exact_dot_rows(A[b], cov[b], pT)
        got = T[b][pT[:, 0], pT[:, 1]]
        assert np.all(np.abs(got - ex) <= _abs_bound(A[b], cov[b], pT, 257)), b
        pK = _pairs(nt, nt, rng)
        ex = exact_dot_rows(T[b], A[b], pK)
        got = Kf[b][pK[:, 0], pK[:, 1]]
        assert np.all(np.abs(got - ex) <= _abs_bound(T[b], A[b], pK, 257)), b
        exm = exact_dot_rows(A[b][:1], mean[b:b + 1], [(0, 0)])[0]
        assert abs(gf[b] - exm) <= _abs_bound(A[b][:1], mean[b:b + 1], [(0, 0)], 257)[0]
        Kb = Kf[b][:, :nt]
        assert np.array_equal(Kb, Kb.T), "mirrored K not bitwise symmetric"
        assert np.array_equal(Kl[b][:, :nt][low], Kb[low])
        assert np.all(Kl[b][:, :nt][~low] == SENT), "spb_flux_conditional_lower wrote above the diagonal"
        assert np.all(Kl[b][:, nt:] == SENT) and np.all(Kf[b][:, nt:] == SENT), "padding columns written"


@pytest.mark.parametrize("shared", [False, True])
def test_flux_conditional_chunk_loop(ctx, shared):
    """B = 1030 crosses the 512-element chunks twice.  Elements 0, 511, 512, 513, 1023, 1024 and 1029 against
    the exact A Sigma A^T: with T^ = A Sigma correctly rounded (|T - T^| <= gamma_257 |A||Sigma|),
        |K - T^ A^T| <= gamma_256 |T^||A|^T + gamma_257 |A||Sigma||A|^T   (first order; the factor (1 + 4 gamma_257)
    covers the second-order terms and the fp64 evaluation of the non-negative bound), plus u |K| for the
    correctly rounded reference (gamma_257 on the first term).  Random symmetric
    Sigma per element, so a wrong chunk offset cannot pass."""
    rng = np.random.default_rng(1030 + shared)
    nt, B = 40, 1030
    A = rng.standard_normal((nt, 256)) if shared else rng.standard_normal((B, nt, 256))
    covd = torch.empty(B, 256, 256, dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(5)
    covd.normal_(generator=g)
    covd = (covd + covd.transpose(1, 2)) / 2
    mean = rng.standard_normal((B, 256))
    K, gm, _ = _conditional(ctx, A, B, covd, mean, nt, lower=False)
    for b in (0, 511, 512, 513, 1023, 1024, 1029):
        Ab = A if shared else A[b]
        Sb = covd[b].cpu().numpy()
        rows = sorted({0, 1, 17, nt - 1} | set(int(x) for x in rng.integers(0, nt, 4)))
        That = np.zeros((nt, 256))
        for i in rows:
            That[i] = exact_dot_rows(Ab, Sb, [(i, j) for j in range(256)])
        pairs = np.array([(i, j) for i in rows for j in _edges(nt, rng, 4)])
        ex = exact_dot_rows(That, Ab, pairs)
        absT = exact_dot_rows(np.abs(That), np.abs(Ab), pairs)
        aSa = ((np.abs(Ab) @ np.abs(Sb)) @ np.abs(Ab).T)[pairs[:, 0], pairs[:, 1]]
        bnd = (gamma(257) * absT + gamma(257) * aSa) * (1 + 4 * gamma(257)) + 600 * TINY
        got = K[b][pairs[:, 0], pairs[:, 1]]
        assert np.all(np.abs(got - ex) <= bnd), b
        exm = exact_dot_rows(Ab[:1], mean[b:b + 1], [(0, 0)])[0]
        assert abs(gm[b] - exm) <= _abs_bound(Ab[:1], mean[b:b + 1], [(0, 0)], 257)[0], b


# ------------------------------------------------------------------------------------------------
# 3. spb_flux_marginal
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def omega_host(spb, ctx):
    """Omega(u) on the host: the table entry times z_{l_p} times z_{l_q}, rounded twice as in omega_scale_kernel."""
    from starry_process_b200 import _tables

    blob, off = _tables.build_tables()
    Om = blob[off["FLUX_OMEGA"]:off["FLUX_OMEGA"] + 31 * 65536].reshape(31, 256, 256)
    rT = torch.empty(1, 256, dtype=torch.float64, device="cuda")
    from starry_process_b200 import _lib

    _lib.check(ctx.lib.spb_flux_operator(ctx.handle, 1, P(dev(np.array(U_LD))), P(rT), None))
    z = rT.cpu().numpy()[0]
    l = np.floor(np.sqrt(np.arange(256)) + 1e-9).astype(int)
    zl = z[l * l + l]
    return (Om * zl[None, :, None]) * zl[None, None, :], rT


def _marginal(ctx, B, covd, mean, rT, covpts=300):
    from starry_process_b200 import _lib

    nb = ctx.lib.spb_flux_marginal_workspace_bytes(ctx.handle, B)
    ws = torch.zeros(nb, dtype=torch.uint8, device="cuda")
    gm = torch.empty(B, dtype=torch.float64, device="cuda")
    var = torch.empty(B, dtype=torch.float64, device="cuda")
    coef = torch.empty(B, 4, covpts + 1, dtype=torch.float64, device="cuda")
    _lib.check(ctx.lib.spb_flux_marginal(ctx.handle, B, P(mean), P(covd), P(rT), covpts, P(gm), P(var), P(coef),
                                         P(ws), nb, None))
    torch.cuda.synchronize()
    w = ws[:(31 * 65536 + 32 * B * 64 + B * 32) * 8].view(torch.float64)
    return w, gm, var, coef


def _check_marginal_elements(w, B, elems, cov_of, Omu):
    """a_m (the sum of the 32 partials, taken exactly by fsum) against <Omega_m(u), Sigma_b> correctly rounded:
    each partial is a 2048-term product sum (gamma_2048), and the kernel adds the 32 partials afterwards, so
    the bound of the sum is gamma_{65536 + 32} sum |Omega Sigma| (what marginal_coef_kernel may use); the fsum of
    the partials and the reference are each correctly rounded: two more u."""
    part = w[31 * 65536:31 * 65536 + 32 * B * 64].view(32, B, 64)
    Om2 = Omu.reshape(31, 65536)
    for b in elems:
        Sb = cov_of(b).reshape(1, 65536)
        pairs = [(0, m) for m in range(31)]
        ex = exact_dot_rows(Sb, Om2, pairs)
        bnd = _abs_bound(Sb, Om2, pairs, 65536 + 32 + 2)
        pb = part[:, b, :31].cpu().numpy()
        got = np.array([math.fsum(pb[:, m]) for m in range(31)])
        assert np.all(np.abs(got - ex) <= bnd), (b, np.max(np.abs(got - ex) / bnd))
        assert np.all(np.isfinite(part[:, b, :31].cpu().numpy()))


@pytest.mark.parametrize("B", [1, 63, 64, 65, 4097])
def test_flux_marginal_quadratic_forms(ctx, omega_host, B):
    """Omega(u) at the head of the workspace bitwise equal to the host's; the split-K forms of sampled elements
    (every element up to 65, the first / last / 64-boundary ones of B = 4097) against the exact forms; var
    and coef finite, and var = sum_{m<16} a_m - mean^2 through the kernel's own a_m (mu part + the 32 partials,
    summed in order: 33 roundings, then 16 + 1): within gamma_50 of the sum of absolute terms."""
    import mpmath

    Omu, rT = omega_host
    rng = np.random.default_rng(B)
    g = torch.Generator(device="cuda").manual_seed(B)
    covd = torch.empty(B, 256, 256, dtype=torch.float64, device="cuda").normal_(generator=g)
    covd = (covd + covd.transpose(1, 2)) / 2
    mean = dev(1e-2 * rng.standard_normal((B, 256)))
    w, gm, var, coef = _marginal(ctx, B, covd, mean, rT)
    assert np.array_equal(w[:31 * 65536].cpu().numpy().reshape(31, 256, 256), Omu)
    elems = sorted({0, B - 2, B - 1, 63, 64} & set(range(B))) if B < 4097 else [0, 64, 4095, 4096]
    _check_marginal_elements(w, B, elems, lambda b: covd[b].cpu().numpy(), Omu)
    assert bool(torch.isfinite(var).all()) and bool(torch.isfinite(coef).all())
    part = w[31 * 65536:31 * 65536 + 32 * B * 64].view(32, B, 64).cpu().numpy()
    amu = w[31 * 65536 + 32 * B * 64:].view(B, 32).cpu().numpy()
    g_h, v_h = gm.cpu().numpy(), var.cpu().numpy()
    with mpmath.workdps(40):
        for b in elems:
            terms = [[amu[b, m]] + list(part[:, b, m]) for m in range(16)]
            want = mpmath.fsum(mpmath.mpf(float(x)) for tm in terms for x in tm) - mpmath.mpf(float(g_h[b])) ** 2
            habs = sum(abs(float(x)) for tm in terms for x in tm) + float(g_h[b]) ** 2
            # habs: 529 fp64 additions of non-negative terms, relative error <= gamma_529
            assert abs(mpmath.mpf(float(v_h[b])) - want) <= gamma(50) * habs * (1 + gamma(529)), b


def test_flux_marginal_pass_boundary(ctx, omega_host):
    """B = 32800 (17.2 GB of cov_ylm) crosses the 32768-element pass of the split-K GEMM: elements 32766, 32767,
    32768 and 32799, built from five distinct symmetric matrices repeated (b mod 5), against the exact forms."""
    B = 32800
    free, total = torch.cuda.mem_get_info()
    need = B * 65536 * 8 + (32 * B * 64 + 31 * 65536 + B * 32) * 8 + (1 << 30)
    print("pass-boundary case: %.1f GB needed, %.1f GB free of %.1f GB" % (need / 1e9, free / 1e9, total / 1e9))
    if free < need:
        pytest.skip("%.1f GB free, %.1f GB needed" % (free / 1e9, need / 1e9))
    Omu, rT = omega_host
    rng = np.random.default_rng(32800)
    bases = _sym(rng, 5)
    covd = torch.empty(B, 256, 256, dtype=torch.float64, device="cuda")
    bd = dev(bases)
    for r in range(5):
        covd[r::5] = bd[r]
    del bd
    mean = dev(1e-2 * rng.standard_normal((B, 256)))
    w, _, var, coef = _marginal(ctx, B, covd, mean, rT)
    del covd
    _check_marginal_elements(w, B, (32766, 32767, 32768, 32799), lambda b: bases[b % 5], Omu)
    assert bool(torch.isfinite(var).all())


# ------------------------------------------------------------------------------------------------
# 4. predict and sampling building blocks
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ns", [1, 7, 128, 129, 1000])
def test_sample_ylm_against_exact(ctx, ns):
    """y[b][s] = mu[b] + L[b] u[b][s] (EPI_ADD_ROWVEC) within gamma_257 (sum |L u| + |mu|): 256 products and
    their sums, then one rounding of the add; the host's ex + mu rounds twice more (gamma_259).  B = 1 and 3,
    per-element mu."""
    from starry_process_b200 import _lib

    for B in (1, 3):
        rng = np.random.default_rng(ns * 10 + B)
        L = np.tril(rng.standard_normal((B, 256, 256)))
        u = rng.standard_normal((B, ns, 256))
        mu = rng.standard_normal((B, 256))
        y = torch.empty(B, ns, 256, dtype=torch.float64, device="cuda")
        _lib.check(ctx.lib.spb_sample_ylm(ctx.handle, B, ns, P(dev(mu)), P(dev(L)), P(dev(u)), P(y), None))
        y = y.cpu().numpy()
        for b in range(B):
            pairs = _pairs(ns, 256, rng)
            ex = exact_dot_rows(u[b], L[b], pairs)
            S = exact_dot_rows(np.abs(u[b]), np.abs(L[b]), pairs)
            m = mu[b][pairs[:, 1]]
            got = y[b][pairs[:, 0], pairs[:, 1]]
            assert np.all(np.abs(got - (ex + m)) <= gamma(259) * (S + np.abs(m)) * (1 + 2 * U64) + 259 * TINY)


def test_cho_cov_ylm_backward_error(ctx):
    """Three SPD matrices and one with a negative diagonal entry (element 2).  The strict upper triangle of L is
    exactly zero; per entry |(L L^T)_ij - Sigma_ij| <= 2 gamma_257 (|L||L|^T)_ij (Cholesky's backward error
    gamma_{n+1}, doubled for the reciprocal-times-multiply division of the panel kernel), plus u for the correctly
    rounded (L L^T)_ij; info flags element 2 alone."""
    from starry_process_b200 import _lib

    rng = np.random.default_rng(11)
    G = rng.standard_normal((4, 256, 300))
    S = G @ G.transpose(0, 2, 1) / 300 + 0.05 * np.eye(256)
    S = (S + S.transpose(0, 2, 1)) / 2
    S[2, 100, 100] = -1.0
    L = torch.empty(4, 256, 256, dtype=torch.float64, device="cuda")
    info = torch.zeros(4, dtype=torch.int32, device="cuda")
    _lib.check(ctx.lib.spb_cho_cov_ylm(ctx.handle, 4, P(dev(S)), P(L), P(info), None))
    info = info.cpu().numpy()
    L = L.cpu().numpy()
    assert info[2] != 0 and np.all(info[[0, 1, 3]] == 0), info
    for b in (0, 1, 3):
        assert np.all(np.triu(L[b], 1) == 0.0)
        pairs = np.array([(i, j) for i in _edges(256, rng, 20) for j in _edges(256, rng, 20) if j <= i])
        ex = exact_dot_rows(L[b], L[b], pairs)
        S_ij = S[b][pairs[:, 0], pairs[:, 1]]
        bnd = (2 * gamma(257) + U64) * exact_dot_rows(np.abs(L[b]), np.abs(L[b]), pairs) * (1 + 2 * U64)
        assert np.all(np.abs(ex - S_ij) <= bnd), b


@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 1000])
def test_tril(ctx, n):
    """The strict upper triangle of every matrix becomes 0; the diagonal, the lower triangle, the padding
    columns and the gaps between matrices (stride > n ld) stay bitwise unchanged."""
    from starry_process_b200 import _lib

    rng = np.random.default_rng(n)
    for ld in (n, n + 1, n + 7):
        B = 3
        stride = n * ld + 5
        buf = rng.standard_normal(B * stride + 3)
        d = dev(buf)
        _lib.check(ctx.lib.spb_tril(ctx.handle, B, n, P(d), ld, stride, None))
        out = d.cpu().numpy()
        want = buf.copy()
        for b in range(B):
            M = want[b * stride:b * stride + n * ld].reshape(n, ld)
            M[:, :n][np.triu(np.ones((n, n), bool), 1)] = 0.0
        assert np.array_equal(out, want), (n, ld)


def _temporal(ctx, B, t1, t2, kind, tau, tau_stride, off, off_stride, K, ld):
    d = dev(K)
    st = ctx.lib.spb_temporal_scale(ctx.handle, B, len(t1), len(t2), P(dev(t1)), P(dev(t2)), kind, P(dev(tau)),
                                    tau_stride, P(dev(off)) if off is not None else None, off_stride, P(d), ld,
                                    len(t1) * ld, None)
    return st, d


@pytest.mark.parametrize("kind", [1, 2])
def test_temporal_scale_against_mpmath(ctx, kind):
    """K <- K k(|t1 - t2|; tau_b) + off_b against k in 40-digit mpmath on the same fp64 inputs (dt exact).
    The device rounds dt, the scaled argument (sqrt 3, the product / square and the quotient: relative <= 4u
    of the argument) and evaluates exp within 2u, (1 + x) and the product within u each, and the fma once:
        |r - ref| <= |K k| (5 u cond + 6 u) + u |ref| + 2^-1074,   cond = x |d ln k / dx|.
    n1 != n2, tau shared and per element, offset NULL and per element; dt = 0 gives K + off exactly, lags where
    exp underflows give exactly off, padding columns ld > n2 untouched."""
    import mpmath
    from starry_process_b200 import _lib

    rng = np.random.default_rng(kind)
    n1, n2, B = 37, 53, 3
    ld = n2 + 3
    t1 = np.sort(rng.uniform(0, 10, n1))
    t2 = np.sort(rng.uniform(0, 10, n2))
    t2[5] = t1[3]            # dt = 0
    t2[-1] = 1e6             # exp underflows for every tau below
    tau = rng.uniform(0.3, 2.0, B)
    offv = rng.standard_normal(B)
    for tau_stride, off in ((0, None), (1, offv), (0, offv), (1, None)):
        K0 = np.full((B, n1, ld), SENT)
        K0[:, :, :n2] = rng.standard_normal((B, n1, n2))
        st, d = _temporal(ctx, B, t1, t2, kind, tau, tau_stride, off, 1, K0, ld)
        _lib.check(st)
        K = d.cpu().numpy()
        assert np.all(K[:, :, n2:] == SENT)
        with mpmath.workdps(40):
            for b in range(B):
                tb = tau[b * tau_stride]
                ob = off[b] if off is not None else 0.0
                assert np.array_equal(K[b, 3, 5], K0[b, 3, 5] + ob)
                assert np.all(K[b, :, n2 - 1] == ob)
                for i in list(range(0, n1, 4)) + [n1 - 1]:
                    for j in list(range(0, n2 - 1, 3)):
                        dt = abs(mpmath.mpf(float(t1[i])) - mpmath.mpf(float(t2[j])))
                        k, cond = temporal_k_mp(kind, dt, tb)
                        ref = mpmath.mpf(float(K0[b, i, j])) * k + mpmath.mpf(float(ob))
                        bnd = (abs(K0[b, i, j]) * float(k) * (5 * U64 * float(cond) + 6 * U64) + U64 * abs(float(ref))
                               + TINY)
                        assert abs(mpmath.mpf(float(K[b, i, j])) - ref) <= bnd, (b, i, j, K[b, i, j], ref, bnd)
    for kw in (dict(kind=3), dict(ld=n2 - 1), dict(B=65536)):
        a = dict(B=B, kind=kind, ld=ld)
        a.update(kw)
        st, _ = _temporal(ctx, a["B"], t1, t2, a["kind"], tau, 0, None, 0, np.zeros((B, n1, ld)), a["ld"])
        assert st != 0, kw


def _coef_table(rng, covpts):
    """A random table through the formulas of marginal_coef_kernel (so the interpolant is continuous at the
    knots up to the rounding of the coefficients)."""
    y = rng.standard_normal(covpts + 4)
    y0, y1, y2, y3 = y[:-3], y[1:-2], y[2:-1], y[3:]
    return np.stack([y1, -y0 / 3.0 - 0.5 * y1 + y2 - y3 / 6.0, 0.5 * (y0 + y2) - y1,
                     0.5 * ((y1 - y2) + (y3 - y0) / 3.0)])


@pytest.mark.parametrize("covpts", [4, 5, 300, 1000])
def test_cross_marginal_against_mpmath(ctx, covpts):
    """K_ts_t[b][i][j] = p_b(s) + off_b, s = |theta(ts_i) - theta(t_j)| covpts / 2pi, against the interpolant in
    mpmath on the kernel's own table, with the phases of spb_phase reproduced bit for bit.  The device rounds
    the difference, 1/dx = covpts / 2pi and the product: |ds| <= 3u s, and it may fuse the last product of
    theta(ts_i), which stays in a register, into the difference (an fma: theta_i unrounded, found on a B200 as
    errors up to 0.4 ulp of theta_i beyond 3u s): |ds| <= (3u s + u theta_i / dx).  Its cubic rounds within
    gamma_6 sum |c_k x0^k|; the offset adds u.  So
        |r - ref| <= D (3u s + u theta_i / dx) + gamma_10 H + J + u (|ref| + |off|)
    (gamma_10: the cubic's gamma_6 and the fp64 evaluation of J, gamma_4; the factor 1 + 8u the fp64 evaluation
    of the bound),
    D = |c1| + 2|c2| + 3|c3| of the bin (and of its neighbour, whose value the bin choice near a knot may take),
    J = the rounding-level jump of the table at the nearest knot.  Stamps on knots, dtheta = 0, negative stamps
    just below a multiple of the period (theta = 2pi exactly: the last bin ind = covpts), ts outside t, columns
    nt..ld-1 zero, offset NULL and per element, and the covpts / period rejections."""
    import mpmath
    from starry_process_b200 import _lib

    rng = np.random.default_rng(covpts)
    B, nt, nts, per = 2, 41, 23, 1.7
    cf = np.stack([_coef_table(rng, covpts) for _ in range(B)])
    t = np.sort(rng.uniform(0, 5, nt))
    t[0] = 0.0
    t[1:4] = per * np.array([1, 3, 7]) / covpts   # on knots
    ts = np.r_[rng.uniform(-8, 12, nts - 4), t[5], -per * (1 + 2.0 ** -52), -2 * per * (1 - 2.0 ** -53), -1e-17]
    ld = nt + 3
    offv = rng.standard_normal(B)
    th_t, th_s = phase_fp64(t, per), phase_fp64(ts, per)
    assert np.any(th_s == TWO_PI)
    for off in (None, offv):
        Kd = torch.full((B, nts, ld), SENT, dtype=torch.float64, device="cuda")
        _lib.check(ctx.lib.spb_cross_marginal(ctx.handle, B, nts, nt, P(dev(ts)), P(dev(t)), per, covpts,
                                              P(dev(cf)), P(dev(off)) if off is not None else None, 1, P(Kd), ld,
                                              nts * ld, None))
        K = Kd.cpu().numpy()
        assert np.all(K[:, :, nt:] == 0.0)
        with mpmath.workdps(40):
            for b in range(B):
                ob = off[b] if off is not None else 0.0
                c = cf[b]
                for i in range(nts):
                    for j in list(range(0, nt, 3)) + [1, 2, 3, 5, nt - 1]:
                        s = abs(mpmath.mpf(float(th_s[i])) - mpmath.mpf(float(th_t[j]))) * covpts / mpmath.mpf(TWO_PI)
                        v, ind = interp_cov_mp(c, covpts, s)
                        ref = v + mpmath.mpf(float(ob))
                        nb = [k for k in (ind - 1, ind, ind + 1) if 0 <= k <= covpts]
                        D = max(abs(c[1][k]) + 2 * abs(c[2][k]) + 3 * abs(c[3][k]) for k in nb)
                        H = max(sum(abs(c[q][k]) for q in range(4)) for k in nb)
                        J = max(abs(c[0][k] + c[1][k] + c[2][k] + c[3][k] - c[0][k + 1]) for k in nb if k < covpts)
                        bnd = (D * U64 * (3 * float(s) + th_s[i] * covpts / TWO_PI) + gamma(10) * H + J
                               + U64 * (abs(float(ref)) + abs(ob)) + TINY) * (1 + 8 * U64)
                        assert abs(mpmath.mpf(float(K[b, i, j])) - ref) <= bnd, (b, i, j, K[b, i, j], ref, bnd)
    dummy = torch.zeros(8 * 1024, dtype=torch.float64, device="cuda")
    for kw in (dict(covpts=3), dict(covpts=-1), dict(period=0.0), dict(period=-1.0)):
        a = dict(covpts=covpts, period=per)
        a.update(kw)
        st = ctx.lib.spb_cross_marginal(ctx.handle, 1, 2, 2, P(dummy), P(dummy), a["period"], a["covpts"], P(dummy),
                                        None, 0, P(dummy), 2, 4, None)
        assert st != 0 and ctx.lib.spb_last_error(), kw
    st = ctx.lib.spb_cross_marginal(ctx.handle, 1, 2, 2, None, P(dummy), per, covpts, P(dummy), None, 0, P(dummy),
                                    2, 4, None)
    assert st != 0
