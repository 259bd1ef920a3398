"""GPU (-m gpu): the INT8 tensor-core products (csrc/i8_planes.cuh) and both Cholesky kernels against exact or
50-digit references (tests/exact_ref.py), and the flag / non-finite contract of every log-likelihood route.

* the lower-triangle product K = (A Sigma) A^T of spb_flux_conditional_lower (gemm_i8_lower_kernel) against the
  correctly rounded product, entry by entry, under a bound derived from the digit format, on adversarial rows;
* non-finite operands of that product must come out non-finite, as on the FP64 (DMMA) GEMM;
* spb_cholesky_lnlike_affine (DMMA) and spb_cholesky_lnlike_i8 against the Woodbury evaluation of
  K = diag(d) + U U^T, power-of-two scaling, non-finite K;
* SPB_INFO_EIG_NOCONV and SPB_INFO_BOUNDS give -inf on every route of StarryProcess.log_likelihood.
"""
import ctypes
import math

import numpy as np
import pytest

from conftest import U_LD
from exact_ref import exact_dot_rows, woodbury_lnlike

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

U64 = 2.0 ** -53
NAN_SENTINEL = -7.0e77   # never a value of K


@pytest.fixture(scope="module")
def spb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


def P(t):
    return ctypes.c_void_p(t.data_ptr())


@pytest.fixture
def i8_product(spb):
    ctx = spb.get_context()
    ctx.set_option("moments_syrk_i8", 1)
    yield ctx
    ctx.set_option("moments_syrk_i8", 1)


# ------------------------------------------------------------------------------------------------
# a. the INT8 lower-triangle product against the exact product
# ------------------------------------------------------------------------------------------------
def _adversarial_rows(rng, nt):
    """Rows of 256 entries: full-mantissa random rows, plus every 7th row one of the cases the digit
    format is sensitive to.  Column 0 carries the row maximum and t_0 = 0 (see _sigma_exponents), so the
    maximum of the row of T = A diag(2^t) is the same entry: T and A both see the case."""
    A = rng.standard_normal((nt, 256))
    A[:, 1:] *= 2.0 ** -7          # |A_ik 2^t_k| <= |A_i0| / 2 for k > 0, whatever t_k <= 6
    A[:, 0] = np.abs(A[:, 0]) + 4.0
    k = int(rng.integers(-20, 20))
    specials = [
        lambda r: r * np.where(np.arange(256) % 3 == 0, 1.0, 1e-30),               # 30 decades
        lambda r: np.r_[2.0 ** k, r[1:] * 2.0 ** (k - 3)],                          # max = 2^k
        lambda r: np.r_[2.0 ** k / 1.0101 * (1 - 2.0 ** -40), r[1:] * 2.0 ** (k - 3)],   # just below 2^k/1.0101
        lambda r: np.r_[2.0 ** k / 1.0101 * (1 + 2.0 ** -40), r[1:] * 2.0 ** (k - 3)],   # just above
        lambda r: np.r_[2.0 ** k * (1 - 2.0 ** -53), r[1:] * 2.0 ** (k - 3)],       # just below 2^k
        lambda r: np.zeros(256),
        lambda r: r * 1e-310,                                                       # subnormals only
        lambda r: r * 1e299 / 8.0,
        lambda r: r * 1e-300,
        lambda r: np.r_[-2.0 ** k, np.where(np.arange(1, 256) % 2, -2.0 ** (k - 1) * (1 - 2.0 ** -53),
                                            -2.0 ** (k - 1))],                      # negative digit boundaries
    ]
    for i in range(3, nt, 7):
        A[i] = specials[(i // 7) % len(specials)](A[i])
    return A


def _sigma_exponents(rng, B):
    t = rng.integers(-6, 7, size=(B, 256))
    t[:, 0] = 0
    return t


def _scale_of(mx):
    """The row scale of slice256_kernel: 2^(e+1) with e the smallest integer with 1.0101 mx < 2^e, at least
    2^-1058; 1 for a zero row."""
    if mx == 0.0:
        return 1.0
    e = math.frexp(mx * 1.0101)[1]
    return math.ldexp(1.0, max(e + 1, -1058))


def _bound(T, A, pairs):
    """Error bound of one entry of the INT8 product (digit format of i8_planes.cuh, 7 planes of balanced 8-bit
    digits, x / E <= 1/2.02):
      each entry x is rounded to a multiple of E 2^-56: |dx| <= E 2^-57, so the first-order error is
          2^-57 (E_i sum_k |A_jk| + F_j sum_k |T_ik|)  (+ 256 2^-114 E_i F_j);
      the products of digit planes s + t >= 7 are not formed: per k at most
          2^14 sum_{d=7..12} n_d 2^(-8 (d + 2)) E_i F_j      (n_d pairs with s + t = d, |digit| <= 128);
      the Horner combine in fp64 (6 fma) and the final product with the power of two E_i F_j 2^-16 round
          relative to at most  H = sum_k (|T_ik| + E_i/250) (|A_jk| + F_j/250): 8 u H;
      a result whose scale E_i F_j 2^-16 is subnormal: an absolute 2^-1050."""
    ctr = sum(n * 2.0 ** (14 - 8 * (d + 2)) for d, n in zip(range(7, 13), (6, 5, 4, 3, 2, 1)))
    out = np.empty(len(pairs))
    for q, (i, j) in enumerate(pairs):
        ti, aj = T[i], A[j]
        E = _scale_of(float(np.max(np.abs(ti))))
        F = _scale_of(float(np.max(np.abs(aj))))
        sa, st = float(np.sum(np.abs(aj))), float(np.sum(np.abs(ti)))
        with np.errstate(over="ignore"):   # rows near 1e299 in both operands: an infinite bound, unused
            H = float(np.sum((np.abs(ti) + E / 250) * (np.abs(aj) + F / 250)))
        out[q] = (2.0 ** -57 * (E * sa + F * st) + 256 * (2.0 ** -114 + ctr) * E * F + 8 * U64 * H
                  + 2.0 ** -1050)
    return out


def _sample_pairs(rng, nt, extra=400):
    """Lower-triangle entries of every (row tile, column tile) class: the first and last 128-row tiles,
    the partial tiles, the diagonal band and both ends of tiles, plus random ones."""
    rows = {0, 1, 127, 128, 129, nt - 1, nt - 2, (nt - 1) // 128 * 128, (nt - 1) // 128 * 128 - 1}
    rows |= set(range(3, min(nt, 150), 7))   # the special rows near the top
    rows |= set(range(nt - 80 - (nt - 80) % 7 + 3, nt, 7))
    pairs = set()
    for i in rows:
        if not 0 <= i < nt:
            continue
        for j in (0, 1, 63, 64, 65, 127, i // 64 * 64, i - 1, i, (i + 1) // 2, i // 2 * 2 + 1 if i % 2 == 0 else i - 2):
            if 0 <= j <= i:
                pairs.add((i, j))
        for j in rng.integers(0, i + 1, 12):
            pairs.add((i, int(j)))
    for i in rng.integers(0, nt, extra):
        pairs.add((int(i), int(rng.integers(0, i + 1))))
    for i in range(0, nt, 7):   # the special rows against the special columns
        pairs.add((i + 3 if i + 3 < nt else nt - 1, min(i + 3, nt - 1) // 2 // 7 * 7 + 3))
    return np.array(sorted(p for p in pairs if p[1] <= p[0]))


def _run_conditional_lower(spb, A, tex, B, shared, ldk, poison=None, nan_cov=None, T_out=False):
    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    dev = torch.device("cuda")
    nt = A.shape[-2]
    Ad = torch.from_numpy(np.ascontiguousarray(A)).to(dev)
    cov = torch.zeros(B, 256, 256, dtype=torch.float64, device=dev)
    idx = torch.arange(256, device=dev)
    cov[:, idx, idx] = torch.from_numpy(np.exp2(tex.astype(np.float64))).to(dev)
    if nan_cov is not None:
        cov[nan_cov[0], nan_cov[1], nan_cov[2]] = float("nan")
    mean = torch.zeros(B, 256, dtype=torch.float64, device=dev)
    gpm = torch.empty(B, dtype=torch.float64, device=dev)
    K = torch.full((B, nt, ldk), NAN_SENTINEL, dtype=torch.float64, device=dev)
    nb = lib.spb_flux_conditional_workspace_bytes(h, B, nt)
    ws = torch.zeros(nb, dtype=torch.uint8, device=dev)
    from starry_process_b200 import _lib

    _lib.check(lib.spb_flux_conditional_lower(h, B, nt, P(Ad), 0 if shared else nt * 256, P(mean), P(cov), P(gpm),
                                              P(K), ldk, P(ws), nb, None))
    torch.cuda.synchronize()
    Tw = None
    if T_out:   # T = A Sigma of the last chunk of 512 elements, at the start of the workspace
        nlast = B - (B - 1) // 512 * 512
        Tw = ws[:nlast * nt * 256 * 8].view(torch.float64).view(nlast, nt, 256).cpu().numpy()
    return K.cpu().numpy(), Tw


@pytest.mark.parametrize("nt", [1024, 1025, 1087, 1151, 1217, 2049])
@pytest.mark.parametrize("B,shared", [(1, True), (3, True), (3, False)])
def test_int8_lower_product_against_exact_product(spb, i8_product, nt, B, shared):
    """gemm_i8_lower_kernel (nt >= 1024, moments_syrk_i8 on) against the correctly rounded product: Sigma =
    diag(2^t) makes T = A Sigma exact on the DMMA GEMM, so K_ij = sum_k T_ik A_jk is a plain exact dot product
    of the operands the INT8 kernel saw (T read back from the workspace).  Every sampled entry within the
    bound of _bound; the padding columns (ldk > nt) not written.  The bound is not vacuous: on the
    full-mantissa rows the observed error reaches more than 1/64 of it (measured on a B200: 1/50 to 1/44).
    Its largest term, the plane products that are not formed, assumes every lower digit at +-128; random
    digits reach that worst case only as a square-root sum, which is the gap.

    Entries are sampled (_sample_pairs: every row- and column-tile class, both ends of tiles, the diagonal
    band, every special row, ~1000-1400 entries a case) rather than all nt (nt + 1) / 2: the exact reference
    costs one 1024-term math.fsum per entry, so the 0.5 M entries of even the smallest case would take
    minutes of host time per case for no class of entry that the sample leaves out."""
    rng = np.random.default_rng(nt * 10 + B + shared)
    nA = 1 if shared else B
    A = np.stack([_adversarial_rows(rng, nt) for _ in range(nA)])
    tex = _sigma_exponents(rng, B)
    ldk = nt + 2 if nt % 2 == 0 else nt + 1
    K, Tw = _run_conditional_lower(spb, A[0] if shared else A, tex, B, shared, ldk, T_out=True)
    assert np.all(K[:, :, nt:] == NAN_SENTINEL), "the padding columns were written"
    pairs = _sample_pairs(rng, nt)
    worst, worst_plain = 0.0, 0.0
    plain = np.array([(i % 7 != 3) and (j % 7 != 3) for i, j in pairs])
    for b in range(B):
        Ab = A[0] if shared else A[b]
        Tb = Tw[b]
        with np.errstate(over="ignore", under="ignore"):
            Th = Ab * np.exp2(tex[b].astype(np.float64))[None, :]
        ok = np.abs(Ab).max(axis=1) > 1e-290   # rows of normal numbers: T is exactly A 2^t
        assert np.array_equal(Tb[ok], Th[ok])
        ref = exact_dot_rows(Tb, Ab, pairs)
        got = K[b][pairs[:, 0], pairs[:, 1]]
        bnd = _bound(Tb, Ab, pairs)
        fin = np.isfinite(ref)   # rows near 1e299 in both operands overflow: both sides must be inf
        assert np.array_equal(got[~fin], ref[~fin]) or np.all(np.isinf(got[~fin]) == np.isinf(ref[~fin]))
        err = np.abs(got[fin] - ref[fin])
        r = err / bnd[fin]
        bad = np.nonzero(r > 1.0)[0]
        assert len(bad) == 0, [(tuple(pairs[fin][q]), got[fin][q], ref[fin][q], bnd[fin][q]) for q in bad[:5]]
        worst = max(worst, float(r.max()))
        worst_plain = max(worst_plain, float(r[plain[fin]].max()))
    print("nt %d B %d shared %d: max err / bound %.3g (full-mantissa rows %.3g)" % (nt, B, shared, worst,
                                                                                  worst_plain))
    assert worst_plain > 1.0 / 64


def test_int8_lower_product_second_chunk(spb, i8_product):
    """B = 513 at nt = 1024 crosses COND_CHUNK = 512: the second chunk (b0 = 512, one element) takes its own
    T, design-matrix offset and K offset.  Per-element A; elements 0, 511 and 512 checked entry by entry."""
    nt, B = 1024, 513
    rng = np.random.default_rng(513)
    A = rng.standard_normal((B, nt, 256))
    tex = _sigma_exponents(rng, B)
    K, Tw = _run_conditional_lower(spb, A, tex, B, False, nt, T_out=True)
    pairs = _sample_pairs(rng, nt, extra=200)
    for b in (0, 511, 512):
        Tb = A[b] * np.exp2(tex[b].astype(np.float64))[None, :]
        if b == 512:
            assert np.array_equal(Tw[0], Tb)
        ref = exact_dot_rows(Tb, A[b], pairs)
        got = K[b][pairs[:, 0], pairs[:, 1]]
        assert np.all(np.abs(got - ref) <= _bound(Tb, A[b], pairs)), b


# ------------------------------------------------------------------------------------------------
# b. non-finite operands of the INT8 product
# ------------------------------------------------------------------------------------------------
def _nonfinite_case(spb, on, kind):
    ctx = spb.get_context()
    nt, B = 1100, 3
    rng = np.random.default_rng(11)
    A = rng.standard_normal((B, nt, 256)) * 0.1
    tex = _sigma_exponents(rng, B)
    ldk = nt
    try:
        ctx.set_option("moments_syrk_i8", on)
        clean, _ = _run_conditional_lower(spb, A, tex, B, False, ldk)
        if kind == "nan_cov":
            K, _ = _run_conditional_lower(spb, A, tex, B, False, ldk, nan_cov=(1, 17, 40))
        else:
            A2 = A.copy()
            A2[1, 300, 5] = np.inf
            K, _ = _run_conditional_lower(spb, A2, tex, B, False, ldk)
    finally:
        ctx.set_option("moments_syrk_i8", 1)
    return clean, K


@pytest.mark.parametrize("kind", ["nan_cov", "inf_A"])
def test_int8_lower_product_propagates_nonfinite_operands(spb, kind):
    """A NaN in cov_ylm[b] or an inf in a per-element design matrix: K[b] must be non-finite wherever the
    FP64 (DMMA) product is (the INT8 digits cannot represent the value and must not return a finite one),
    and the other elements bit-identical to a clean call with the same setting."""
    res = {on: _nonfinite_case(spb, on, kind) for on in (0, 1)}
    low = np.tril(np.ones((1100, 1100), dtype=bool))
    nonfin_dmma = ~np.isfinite(res[0][1][1]) & low
    assert nonfin_dmma.any()
    for on in (0, 1):
        clean, K = res[on]
        assert np.all(~np.isfinite(K[1][nonfin_dmma])), on
        for b in (0, 2):
            assert np.array_equal(K[b][low], clean[b][low]), (on, b)
    if kind == "inf_A":   # the poisoned row and column, and nothing else
        fin = np.isfinite(res[1][1][1]) | ~low
        assert not fin[300, :301].any() and not fin[300:, 300].any()
        fin[300, :] = True
        fin[:, 300] = True
        assert fin.all()


def test_nan_in_cov_ylm_scores_minus_inf_on_both_products(spb):
    """End to end: a NaN in the cached cov_ylm of one element, the conditional branch at nt = 1500 (the INT8
    product applies), both settings of moments_syrk_i8: that element -inf, the others unchanged."""
    import bench

    hp, t0, f0, _ = bench.synthetic_inputs(4, 1234)
    nt = 1500
    tt = np.linspace(0.0, 9.0, nt)
    fl = np.interp(tt, t0 * 2.25, f0)
    ctx = spb.get_context()
    try:
        for on in (0, 1):
            ctx.set_option("moments_syrk_i8", on)
            out = []
            for poison in (False, True):
                gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hp)
                gp._compute_moments()
                if poison:
                    gp._cov_ylm[2, 30, 31] = float("nan")
                out.append(gp.log_likelihood(tt, fl, 1e-6, i=60.0, p=1.3, u=U_LD).cpu().numpy())
            assert np.all(np.isfinite(out[0])), on
            assert np.isneginf(out[1][2]), (on, out[1])
            assert np.array_equal(out[1][[0, 1, 3]], out[0][[0, 1, 3]]), on
    finally:
        ctx.set_option("moments_syrk_i8", 1)


# ------------------------------------------------------------------------------------------------
# c-e. both Cholesky kernels against the Woodbury reference
# ------------------------------------------------------------------------------------------------
_REF_CACHE = {}


def _woodbury_problem(nt, seed=5, k=6):
    """K = diag(d) + U U^T with dyadic d in [1/2, 1) (8 bits) and U in (1/64) Z, |U| <= 1/2: every entry of K
    is exact in fp64, so K, the noise split over lambda_min / affine diag, and the reference agree exactly.
    Three distinct right-hand sides; the others are power-of-two multiples of them (quad scales by 4^s)."""
    key = (nt, seed, k)
    if key not in _REF_CACHE:
        rng = np.random.default_rng(seed + nt)
        d = 0.5 + rng.integers(0, 128, nt) / 256.0
        U = rng.integers(-32, 33, (nt, k)) / 64.0
        R = rng.standard_normal((3, nt))
        logdet, quad, _ = woodbury_lnlike(d, U, R)
        _REF_CACHE[key] = (d, U, R, float(logdet), [float(q) for q in quad])
    return _REF_CACHE[key]


def _rhs(R, qref, M):
    s = np.array([(m // 3) % 7 - 3 for m in range(M)])
    rows = np.stack([R[m % 3] * 2.0 ** s[m] for m in range(M)]) if M else np.zeros((0, R.shape[1]))
    q = np.array([qref[m % 3] * 4.0 ** s[m] for m in range(M)])
    return rows, q


def _chol(spb, kernel, Kh, Rh, noise, planes=78, dvec=None, lam=None, B=1, may_fall_back=()):
    """One call of spb_cholesky_lnlike_affine ("f64") or spb_cholesky_lnlike_i8 ("i8") on B copies (or the
    (B, nt, nt) stack) of K.  noise: "lambda" (noise already in K, lambda_min given to the INT8 kernel),
    "scalar" (affine diag scalar), "vector" (affine diag vector dvec).

    "i8": the INT8 kernel only reads K, while its safety net (a matrix whose digits overflowed,
    SPB_INFO_I8_RANGE, re-run on the FP64 kernel) overwrites K with L and clears the flag.  So the INT8
    kernel produced the result of matrix b exactly when K[b] is bit-identical after the call; that is
    asserted for every matrix not listed in ``may_fall_back``."""
    from starry_process_b200 import _lib

    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    dev = torch.device("cuda")
    Kh = Kh if Kh.ndim == 3 else np.broadcast_to(Kh, (B,) + Kh.shape)
    Rh = Rh if Rh.ndim == 3 else np.broadcast_to(Rh, (B,) + Rh.shape)
    B, nt = Kh.shape[0], Kh.shape[1]
    M = Rh.shape[1]
    ld = nt + (nt & 1)
    K = torch.zeros(B, nt, ld, dtype=torch.float64)
    K[:, :, :nt] = torch.from_numpy(np.ascontiguousarray(Kh))
    Mr = max(M, 1)
    r = torch.zeros(B, Mr, ld, dtype=torch.float64)
    if M:
        r[:, :M, :nt] = torch.from_numpy(np.ascontiguousarray(Rh))
    K, r = K.to(dev), r.to(dev)
    K_in = K.clone() if kernel == "i8" else None
    af = _lib.Affine()
    keep = []
    if noise == "scalar":
        t = torch.full((1,), float(lam), dtype=torch.float64, device=dev)
        af.diag, af.diag_kind, af.diag_stride = t.data_ptr(), 0, 0
        keep.append(t)
    elif noise == "vector":
        t = torch.from_numpy(np.ascontiguousarray(dvec)).to(dev)
        af.diag, af.diag_kind, af.diag_stride = t.data_ptr(), 1, 0
        keep.append(t)
    ll = torch.zeros(B, dtype=torch.float64, device=dev)
    quad = torch.zeros(B, Mr, dtype=torch.float64, device=dev)
    logdet = torch.zeros(B, dtype=torch.float64, device=dev)
    info = torch.zeros(B, dtype=torch.int32, device=dev)
    if kernel == "f64":
        _lib.check(lib.spb_cholesky_lnlike_affine(h, B, nt, P(K), ld, nt * ld, ctypes.byref(af), M, P(r), ld,
                                                  Mr * ld, P(ll), P(quad), P(logdet), P(info), None))
    else:
        nb = lib.spb_cholesky_i8_workspace_bytes(B, nt, M, planes)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.check(lib.spb_cholesky_lnlike_i8(h, B, nt, P(K), ld, nt * ld,
                                              ctypes.byref(af) if noise != "lambda" else None, M, P(r), ld,
                                              Mr * ld, P(ll), P(quad), P(logdet), P(info), planes,
                                              float(lam) if noise == "lambda" else 0.0, P(ws), nb, None))
    torch.cuda.synchronize()
    if K_in is not None:   # bitwise (NaN entries included): K untouched <=> no fall-back to the FP64 kernel
        same = (K.view(torch.int64) == K_in.view(torch.int64)).flatten(1).all(dim=1).cpu().numpy()
        fell_back = [b for b in range(B) if not same[b]]
        assert set(fell_back) <= set(may_fall_back), ("re-run on the FP64 kernel", fell_back)
    return dict(ll=ll.cpu().numpy(), quad=quad.cpu().numpy()[:, :M], logdet=logdet.cpu().numpy(),
                info=info.cpu().numpy(), y=r.cpu().numpy()[:, :M, :nt])


def _tolerance(kernel, planes, nt, kappa):
    """Relative tolerance of log det K and r^T K^-1 r.
    DMMA kernel: a backward-stable Cholesky returns the exact factor of K + dK with |dK| <= c nt u |K|, so
    both values move by at most ~ nt u kappa relative (kappa = cond(K)); c = 8.
    INT8 kernel: the panel products are exact up to the bits kept per row (55 for planes 78, 56 for 8, 49 for 7)
    instead of u: the same form with 2^-bits for u."""
    bits = {78: 55, 8: 56, 7: 49}[planes] if kernel == "i8" else 53
    return 8 * nt * kappa * 2.0 ** -bits


def _kappa(d, U):
    return (d.max() + np.linalg.norm(U, 2) ** 2) / d.min()


FULL_NT = [65, 127, 128, 129, 704, 1000, 1536, 1537, 2049]


@pytest.mark.parametrize("nt", FULL_NT)
def test_cholesky_kernels_against_woodbury(spb, nt):
    """Both kernels (DMMA; INT8 with planes 78, 8, 7) x M in {0, 1, 3, 130} (the "gap" right-hand-side layout
    M <= n64 - nt and the padded one) x the noise floor as lambda_min, affine scalar and affine vector,
    against the 50-digit Woodbury evaluation: log det K and every r^T K^-1 r within _tolerance."""
    d, U, R, ld_ref, qref = _woodbury_problem(nt)
    kappa = _kappa(d, U)
    K0 = U @ U.T   # exact: 6 products of 6-bit numbers
    lam = 0.5
    Kfull = K0 + np.diag(d)
    Kpart = K0 + np.diag(d - lam)   # + lam through the affine scalar
    for M in (0, 1, 3, 130):
        Rm, qm = _rhs(R, qref, M)
        for kernel, planes in (("f64", 0), ("i8", 78), ("i8", 8), ("i8", 7)):
            if kernel == "i8" and nt <= 64:
                continue
            tol = _tolerance(kernel, planes, nt, kappa)
            for noise in ("lambda", "scalar", "vector"):
                if kernel == "f64" and noise == "lambda":
                    Kin, kw = Kfull, {}
                elif noise == "lambda":
                    Kin, kw = Kfull, dict(lam=d.min())
                elif noise == "scalar":
                    Kin, kw = Kpart, dict(lam=lam)
                else:
                    Kin, kw = K0, dict(dvec=d)
                o = _chol(spb, kernel, Kin, Rm[None], "scalar" if (kernel == "f64" and noise == "lambda") else noise,
                          planes=planes, **(kw if kw else dict(lam=0.0)))
                tag = (nt, M, kernel, planes, noise)
                assert o["info"][0] == 0, tag
                e_ld = abs(2 * o["logdet"][0] - ld_ref) / abs(ld_ref)
                assert e_ld <= tol, (tag, e_ld, tol)
                if M:
                    e_q = np.max(np.abs(o["quad"][0] - qm) / qm)
                    assert e_q <= tol, (tag, e_q, tol)
                    want = -0.5 * qm.sum() - M * ld_ref / 2 - 0.5 * nt * M * math.log(2 * math.pi)
                    assert abs(o["ll"][0] - want) <= tol * (0.5 * qm.sum() + M * abs(ld_ref) / 2 + 1.0), tag


@pytest.mark.parametrize("nt,kernel,planes,noise,M", [(4097, "f64", 0, "scalar", 3), (4097, "i8", 7, "vector", 130),
                                                      (16384, "i8", 78, "lambda", 1)])
def test_cholesky_large_against_woodbury(spb, nt, kernel, planes, noise, M):
    """One combination per size from nt = 4097 up (one (d, U) and its reference per size)."""
    d, U, R, ld_ref, qref = _woodbury_problem(nt, k=4)
    kappa = _kappa(d, U)
    K0 = U @ U.T
    Rm, qm = _rhs(R, qref, M)
    if noise == "scalar":
        o = _chol(spb, kernel, K0 + np.diag(d - 0.5), Rm[None], "scalar", planes=planes, lam=0.5)
    elif noise == "vector":
        o = _chol(spb, kernel, K0, Rm[None], "vector", planes=planes, dvec=d)
    else:
        o = _chol(spb, kernel, K0 + np.diag(d), Rm[None], "lambda", planes=planes, lam=d.min())
    tol = _tolerance(kernel, planes, nt, kappa)
    assert o["info"][0] == 0
    assert abs(2 * o["logdet"][0] - ld_ref) / abs(ld_ref) <= tol
    assert np.max(np.abs(o["quad"][0] - qm) / qm) <= tol


def test_int8_cholesky_rejects_nt_above_16384(spb):
    """64 < nt <= 16384: nt = 16385 is refused with a non-zero status before anything is launched."""
    from starry_process_b200 import _lib

    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    dev = torch.device("cuda")
    nt, ld = 16385, 16386
    K = torch.zeros(1, 2, dtype=torch.float64, device=dev)   # never read: the call must fail first
    ll = torch.zeros(1, dtype=torch.float64, device=dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(1024, dtype=torch.uint8, device=dev)
    n0 = ctx.launches()
    for n in (nt, 64):
        st = lib.spb_cholesky_lnlike_i8(h, 1, n, P(K), ld, n * ld, None, 0, None, ld, 0, P(ll), None, None,
                                        P(info), 78, 1.0, P(ws), 1 << 40, None)
        assert st != 0, n
    assert ctx.launches() == n0


# ------------------------------------------------------------------------------------------------
# d. power-of-two scaling
# ------------------------------------------------------------------------------------------------
def test_cholesky_power_of_two_scaling(spb):
    """K' = S K S, r' = S r with S = diag(2^s), s in [-60, 60], noise scaled with K (affine diag vector
    d_i 4^s_i).  DMMA: every operation is exact under power-of-two scaling, so the solved rows y and quad are
    bitwise those of the unscaled call and log det moves by exactly 2 ln2 sum s_i (to 1e-13 of sum|log L_ii|).
    INT8 (planes 78 and 8): the same values within its tolerance, computed by the INT8 kernel itself (no
    SPB_INFO_I8_RANGE re-run on the FP64 kernel, checked by _chol): the right-hand-side row bound must be
    neither too loose (bits lost) nor too tight (digit overflow)."""
    nt, M = 1000, 3
    d, U, R, ld_ref, qref = _woodbury_problem(nt)
    rng = np.random.default_rng(9)
    s = rng.integers(-60, 61, nt).astype(np.float64)
    S = np.exp2(s)
    K0 = U @ U.T
    Ks = K0 * S[:, None] * S[None, :]
    ds = d * S * S
    Rs = R * S[None, :]
    shift = 2 * math.log(2.0) * s.sum()
    a = _chol(spb, "f64", K0, R[None], "vector", dvec=d)
    b = _chol(spb, "f64", Ks, Rs[None], "vector", dvec=ds)
    assert np.all(a["info"] == 0) and np.all(b["info"] == 0)
    assert np.array_equal(a["y"], b["y"])
    assert np.array_equal(a["quad"], b["quad"])
    assert abs((b["logdet"][0] - a["logdet"][0]) - shift / 2) <= 1e-13 * (abs(a["logdet"][0]) + abs(shift))
    tol = _tolerance("i8", 78, nt, _kappa(d, U))
    for planes in (78, 8):
        c = _chol(spb, "i8", Ks, Rs[None], "vector", planes=planes, dvec=ds)
        assert c["info"][0] == 0, c["info"]
        assert abs((c["logdet"][0] - shift / 2) - ld_ref / 2) <= tol * abs(ld_ref)
        assert np.max(np.abs(c["quad"][0] - np.array(qref)) / np.array(qref)) <= tol


def test_int8_cholesky_heteroscedastic_noise(spb):
    """Noise spanning 6 decades (affine diag vector, the marginal-branch route to the INT8 kernel).  The
    right-hand-side rows are scaled by one bound per light curve, sqrt(sum_k r_k^2 / d_k); the 1e-8 parity
    bar must hold against the Woodbury reference, on the INT8 kernel itself (no re-run, checked by _chol).
    Prints the INT8 and DMMA errors and log2 of their ratio."""
    nt, M = 2049, 3
    d, U, R, _, _ = _woodbury_problem(nt)
    rng = np.random.default_rng(4)
    dh = np.exp2(np.round(rng.uniform(-20, 0, nt)))    # 1e-6 .. 1, powers of two
    ld_ref, qref, _ = woodbury_lnlike(dh, U, R)
    ld_ref, qref = float(ld_ref), np.array([float(q) for q in qref])
    for planes in (78, 7):
        o = _chol(spb, "i8", U @ U.T, R[None], "vector", planes=planes, dvec=dh)
        f = _chol(spb, "f64", U @ U.T, R[None], "vector", dvec=dh)
        e_i8 = max(abs(2 * o["logdet"][0] - ld_ref) / abs(ld_ref), np.max(np.abs(o["quad"][0] - qref) / qref))
        e_f = max(abs(2 * f["logdet"][0] - ld_ref) / abs(ld_ref), np.max(np.abs(f["quad"][0] - qref) / qref))
        print("heteroscedastic noise, planes %d: rel err %.2e (DMMA %.2e), log2 ratio %.1f"
              % (planes, e_i8, e_f, math.log2(max(e_i8, 1e-300) / max(e_f, 2.0 ** -53))))
        assert o["info"][0] == 0
        assert e_i8 <= (1e-8 if planes == 78 else 1e-6), (planes, e_i8)


# ------------------------------------------------------------------------------------------------
# e. non-finite K
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["nan_offdiag", "inf_offdiag", "nan_diag"])
@pytest.mark.parametrize("kernel", ["f64", "i8"])
def test_cholesky_nonfinite_entry(spb, case, kernel):
    """One NaN off the diagonal (row in panel >= 2, column in panel 0), one +inf off the diagonal, a NaN on
    the diagonal: -inf and a non-zero info for that matrix; the other matrices of the batch bit-identical to
    a clean run."""
    nt, B = 1000, 4
    d, U, R, _, _ = _woodbury_problem(nt)
    K = np.broadcast_to(U @ U.T + np.diag(d), (B, nt, nt)).copy()
    Rb = np.broadcast_to(R[None, :1], (B, 1, nt)).copy()
    if case == "nan_offdiag":
        K[2, 200, 10] = K[2, 10, 200] = np.nan
    elif case == "inf_offdiag":
        K[2, 500, 70] = K[2, 70, 500] = np.inf
    else:
        K[2, 333, 333] = np.nan
    kw = dict(lam=d.min()) if kernel == "i8" else dict(lam=0.0)
    clean = _chol(spb, kernel, np.broadcast_to(U @ U.T + np.diag(d), (B, nt, nt)).copy(), Rb,
                  "lambda" if kernel == "i8" else "scalar", **kw)
    # the poisoned matrix may take the safety net (its digits cannot be cut); the others must not
    o = _chol(spb, kernel, K, Rb, "lambda" if kernel == "i8" else "scalar", may_fall_back=(2,), **kw)
    assert np.isneginf(o["ll"][2]) and o["info"][2] != 0, (o["ll"][2], o["info"][2])
    for b in (0, 1, 3):
        assert o["ll"][b] == clean["ll"][b] and o["info"][b] == 0
        assert np.array_equal(o["y"][b], clean["y"][b])


# ------------------------------------------------------------------------------------------------
# f. flags on every route
# ------------------------------------------------------------------------------------------------
ROUTES = {
    # name: (B, nt, M, StarryProcess kwargs, cholesky_i8, log_likelihood kwargs)
    "dense_batch_affine": (4, 200, 1, dict(marginalize_over_inclination=True, normalized=True), 0, {}),
    "dense_batch_plain": (4, 200, 1, dict(marginalize_over_inclination=False, normalized=True), 0, {}),
    "cluster_affine": (4, 300, 1, dict(marginalize_over_inclination=True, normalized=True), 0, {}),
    "cluster_plain": (4, 300, 1, dict(marginalize_over_inclination=False, normalized=True), 0, {}),
    "int8_affine": (4, 300, 1, dict(marginalize_over_inclination=True, normalized=True), 78, {}),
    "int8_plain": (4, 300, 1, dict(marginalize_over_inclination=False, normalized=True), 78, {}),
    "ensemble": (1, 200, 64, dict(marginalize_over_inclination=True, normalized=True), 0, {}),
    "lowrank": (4, 300, 1, dict(marginalize_over_inclination=False, normalized=False), 0, dict(method="lowrank")),
}


@pytest.mark.parametrize("bit", [8, 4])
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_info_flag_forces_minus_inf_on_every_route(spb, route, bit):
    """include/spb200.h: an element flagged SPB_INFO_EIG_NOCONV (8) -- and, as a control, SPB_INFO_BOUNDS (4)
    -- scores -inf on every route of log_likelihood (dense batch kernel, cluster kernel, INT8 Cholesky, with
    the noise deferred into the Cholesky loads or assembled, the one-factor ensemble route, the rank-31
    route); the other elements are bit-identical to an unflagged run."""
    import bench

    B, nt, M, kw, ci8, llkw = ROUTES[route]
    hp, t0, f0, _ = bench.synthetic_inputs(max(B, 2), 1234)
    hp = {k: v[:B] for k, v in hp.items()}
    tt = np.linspace(0.0, 3.0, nt)
    fl = np.interp(tt, t0, f0)
    if M > 1:
        rng = np.random.default_rng(2)
        fl = fl[None] + 1e-4 * rng.standard_normal((M, nt))
    ctx = spb.get_context()
    fb = B // 2
    out = []
    try:
        ctx.set_option("cholesky_i8", ci8)
        for flag in (False, True):
            gp = spb.StarryProcess(**kw, **hp)
            gp._compute_moments()
            if flag:
                gp.info[fb] |= bit
            out.append(gp.log_likelihood(tt, fl, 1e-6, i=60.0, p=1.0, u=U_LD, **llkw).cpu().numpy().reshape(-1))
    finally:
        ctx.set_option("cholesky_i8", -1)
    clean, flagged = out
    assert np.all(np.isfinite(clean)), clean
    assert np.isneginf(flagged[fb]), (route, bit, flagged)
    others = [b for b in range(B) if b != fb]
    assert np.array_equal(flagged[others], clean[others])
