"""GPU (-m gpu): the INT8-tensor-core Cholesky path (csrc/potrf_i8.cuh, spb_cholesky_lnlike_i8).

The digit-plane emulation of the FP64 panel updates is error-free up to the 56 (planes = 8) or 49
(planes = 7) bits kept per row, so it must reproduce the FP64 (DMMA) kernel to rounding noise and keep
the 1e-8 parity with the unmodified reference's golden values:
* C ABI: random SPD matrices, sizes that exercise the partial last panel, the "gap" and padded layouts of
  the right-hand-side planes, many right-hand sides, more matrices than SMs;
* the safety net (SPB_INFO_I8_RANGE -> FP64 kernel) on a right-hand side that cannot be scaled;
* StarryProcess.log_likelihood with ``cholesky_i8`` on against the reference golden of the bench draws.
"""
import ctypes

import numpy as np
import pytest

from conftest import U_LD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def spb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


def P(t):
    return ctypes.c_void_p(t.data_ptr())


def _both_kernels(spb, B, n, M, planes, seed, dg=1e-4, poison=None, not_pd=None):
    from starry_process_b200 import _lib

    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    dev = torch.device("cuda")
    g = torch.Generator(device="cpu").manual_seed(seed)
    ld = n + (n & 1)
    A = torch.randn(B, n, 24, dtype=torch.float64, generator=g)
    K = torch.zeros(B, n, ld, dtype=torch.float64)
    K[:, :, :n] = A @ A.transpose(1, 2) / 24.0
    if not_pd is not None:   # an indefinite element: the pivots turn negative half way through
        K[not_pd, n // 2:, n // 2:n] -= 3.0 * torch.eye(n - n // 2, dtype=torch.float64)
    Mr = max(M, 1)
    r = torch.zeros(B, Mr, ld, dtype=torch.float64)
    r[:, :, :n] = 0.01 * torch.randn(B, Mr, n, dtype=torch.float64, generator=g)
    if poison is not None:
        r[poison[0], 0, poison[1]] = poison[2]
    K, r = K.to(dev), r.to(dev)
    dgt = torch.full((1,), dg, dtype=torch.float64, device=dev)
    af = _lib.Affine()
    af.diag, af.diag_kind, af.diag_stride = dgt.data_ptr(), 0, 0
    out = {}
    for name in ("f64", "i8"):
        Kc, rc = K.clone(), r.clone()
        ll = torch.zeros(B, dtype=torch.float64, device=dev)
        quad = torch.zeros(B, Mr, dtype=torch.float64, device=dev)
        logdet = torch.zeros(B, dtype=torch.float64, device=dev)
        info = torch.zeros(B, dtype=torch.int32, device=dev)
        if name == "f64":
            _lib.check(lib.spb_cholesky_lnlike_affine(h, B, n, P(Kc), ld, n * ld, ctypes.byref(af), M, P(rc), ld,
                                                      Mr * ld, P(ll), P(quad), P(logdet), P(info), None))
        else:
            nb = lib.spb_cholesky_i8_workspace_bytes(B, n, M, planes)
            assert nb > 0
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.check(lib.spb_cholesky_lnlike_i8(h, B, n, P(Kc), ld, n * ld, ctypes.byref(af), M, P(rc), ld,
                                                  Mr * ld, P(ll), P(quad), P(logdet), P(info), planes, 0.0, P(ws), nb,
                                                  None))
            torch.cuda.synchronize()
            if poison is None and not_pd is None:
                assert torch.equal(Kc, K), "the INT8 path must leave K untouched"
            elif poison is not None:
                # only the flagged matrix goes through the FP64 safety net, which stores its factor over K
                keep = [i for i in range(B) if i != poison[0]]
                assert torch.equal(Kc[keep], K[keep]), "the safety net must re-run only the flagged matrix"
                assert not torch.equal(Kc[poison[0]], K[poison[0]]), "the flagged matrix was not re-run"
        torch.cuda.synchronize()
        out[name] = dict(ll=ll.cpu().numpy(), quad=quad.cpu().numpy(), logdet=logdet.cpu().numpy(),
                         info=info.cpu().numpy(), y=rc.cpu().numpy()[:, :M, :n])
    return out


@pytest.mark.parametrize("B,n,M", [(2, 65, 1), (2, 128, 1), (2, 200, 1), (3, 257, 2), (2, 1000, 1), (2, 1000, 3),
                                   (1, 1024, 0), (2, 1000, 24), (2, 1000, 25), (2, 1000, 130), (2, 1024, 2),
                                   (1, 2049, 1), (300, 320, 1)])
@pytest.mark.parametrize("planes", [8, 78, 7])
def test_i8_kernel_matches_fp64_kernel(spb, B, n, M, planes):
    """math.py:75-100 / sp.py:1154-1188 through both kernels: same lnlike, |y|^2, log-determinant and
    solved rows.  planes = 8: 8 x 7 bits = 56 bits per row, 78: 7 planes of 8-bit digits = 55 bits -> FP64
    rounding-noise level; planes = 7: 7 x 7 = 49 bits."""
    o = _both_kernels(spb, B, n, M, planes, seed=1000 * B + n + M)
    a, b = o["f64"], o["i8"]
    tol = 3e-9 if planes == 7 else 2e-11
    assert np.all(a["info"] == 0) and np.all(b["info"] == 0)
    assert np.max(np.abs(a["logdet"] - b["logdet"]) / np.abs(a["logdet"])) < tol
    if M:
        assert np.max(np.abs(a["ll"] - b["ll"]) / np.abs(a["ll"])) < tol
        assert np.max(np.abs(a["quad"] - b["quad"]) / np.abs(a["quad"])) < 50 * tol
        assert np.max(np.abs(a["y"] - b["y"])) < 1e3 * tol * np.max(np.abs(a["y"]))


def test_i8_safety_net_reruns_unscalable_matrices_on_the_fp64_kernel(spb):
    """A right-hand side whose scale bound overflows (an entry of 1e300) cannot be cut into digits: the
    matrix is flagged SPB_INFO_I8_RANGE inside the kernel and re-run through the FP64 kernel by the
    launcher, so both paths return the same numbers; the other matrices of the batch are unaffected."""
    o = _both_kernels(spb, 3, 500, 1, 8, seed=77, poison=(1, 10, 1e300))
    a, b = o["f64"], o["i8"]
    assert np.array_equal(np.isfinite(a["ll"]), np.isfinite(b["ll"]))
    assert np.array_equal(a["ll"][1:2], b["ll"][1:2]) or (np.isneginf(a["ll"][1]) and np.isneginf(b["ll"][1]))
    ok = [0, 2]
    assert np.max(np.abs(a["ll"][ok] - b["ll"][ok]) / np.abs(a["ll"][ok])) < 2e-11
    assert np.all(b["info"][ok] == 0)


@pytest.mark.parametrize("planes", [8, 78, 7])
def test_log_likelihood_with_i8_cholesky_against_reference_golden(spb, golden, planes):
    """The bench draws (tests/golden/bench_sweep_seed1234.npz, produced by the unmodified reference) with
    the factorisation on the INT8 tensor cores: 1e-8 relative, identical -inf pattern, and rounding-noise
    agreement with the FP64 kernel."""
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, 1234)
    sw = golden("bench_sweep_seed1234.npz")
    ns = len(sw["r"])
    ctx = spb.get_context()
    res = {}
    try:
        for pl in (0, planes):
            ctx.set_option("cholesky_i8", pl)
            gp = spb.StarryProcess(marginalize_over_inclination=True, normalized=True,
                                   **{k: hp[k][:ns] for k in hp})
            res[pl] = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
    finally:
        ctx.set_option("cholesky_i8", -1)
    ref = sw["lnlike_m1_n1"]
    ll = res[planes]
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    fin = np.isfinite(ref)
    err = np.abs(ll[fin] - ref[fin]) / np.abs(ref[fin])
    d = np.abs(ll[fin] - res[0][fin]) / np.abs(res[0][fin])
    print("i8 planes=%d: max rel err vs reference %.2e, vs FP64 kernel %.2e" % (planes, err.max(), d.max()))
    assert err.max() <= 1e-8
    assert d.max() <= (1e-9 if planes == 7 else 1e-11)


def test_i8_not_positive_definite_element(spb):
    """math.py:82-91: a matrix that is not positive definite gives -inf and SPB_INFO_NOT_PD on both kernels,
    is NOT re-run through the FP64 kernel (its digit overflow is a consequence, not a cause), and leaves the
    other matrices of the batch alone."""
    o = _both_kernels(spb, 4, 700, 1, 8, seed=5, not_pd=2)
    a, b = o["f64"], o["i8"]
    assert a["info"][2] & 1 and b["info"][2] & 1
    assert not (b["info"][2] & 16)
    assert np.isneginf(a["ll"][2]) and np.isneginf(b["ll"][2])
    ok = [0, 1, 3]
    assert np.all(b["info"][ok] == 0)
    assert np.max(np.abs(a["ll"][ok] - b["ll"][ok]) / np.abs(a["ll"][ok])) < 2e-11


def test_i8_kernel_is_deterministic_under_load(spb):
    """The producer thread reads digit planes that the compute warps of the same CTA stored a tile earlier
    (stored-tile counter + generic -> async proxy fence): 12 launches over 600 matrices (4 per SM, dynamic
    work claiming) must return bit-identical lnlike vectors -- a lost ordering would show up as a stale
    plane in some matrix of some launch."""
    from starry_process_b200 import _lib

    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    dev = torch.device("cuda")
    B, n, M = 600, 1000, 1
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn(B, n, 16, dtype=torch.float64, device=dev, generator=g)
    K = torch.bmm(A, A.transpose(1, 2)) / 16.0
    r0 = 0.01 * torch.randn(B, 1, n, dtype=torch.float64, device=dev, generator=g)
    dgt = torch.full((1,), 1e-4, dtype=torch.float64, device=dev)
    af = _lib.Affine()
    af.diag, af.diag_kind, af.diag_stride = dgt.data_ptr(), 0, 0
    nb = lib.spb_cholesky_i8_workspace_bytes(B, n, M, 78)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    first = None
    for rep in range(12):
        ws.random_(0, 255)            # stale planes from the previous launch must never be read
        ll = torch.zeros(B, dtype=torch.float64, device=dev)
        info = torch.zeros(B, dtype=torch.int32, device=dev)
        r = r0.clone()
        _lib.check(lib.spb_cholesky_lnlike_i8(h, B, n, P(K), n, n * n, ctypes.byref(af), M, P(r), n, n, P(ll),
                                              None, None, P(info), 78, 0.0, P(ws), nb, None))
        torch.cuda.synchronize()
        assert int(info.abs().sum()) == 0
        if first is None:
            first = ll.clone()
        else:
            assert torch.equal(first, ll), "launch %d differs" % rep


def test_moments_syrk_on_int8_tensor_cores_matches_fp64_syrk(spb, golden):
    """contrast.py:21-33 (+ size.py:116-125 for the dr prior): cov_ylm from the INT8-tensor-core SYRK
    (csrc/syrk_i8.cu, the default) against the FP64 (DMMA) SYRK -- elementwise to 1e-13 of the largest entry,
    exactly symmetric -- and the log-likelihood of the bench draws against the reference golden at 1e-8."""
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, 1234)
    sw = golden("bench_sweep_seed1234.npz")
    ns = len(sw["r"])
    ctx = spb.get_context()
    cov, ll, covd = {}, {}, {}
    try:
        for on in (0, 1):
            ctx.set_option("moments_syrk_i8", on)
            gp = spb.StarryProcess(marginalize_over_inclination=True, normalized=True,
                                   **{k: hp[k][:ns] for k in hp})
            cov[on] = gp.cov_ylm.cpu().numpy()
            ll[on] = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
            gd = spb.StarryProcess(r=hp["r"][:32], dr=np.full(32, 4.0), mu=hp["mu"][:32], sigma=hp["sigma"][:32],
                                   c=hp["c"][:32], n=hp["n"][:32])
            covd[on] = gd.cov_ylm.cpu().numpy()
    finally:
        ctx.set_option("moments_syrk_i8", 1)
    for a in (cov, covd):
        scale = np.abs(a[0]).max(axis=(1, 2), keepdims=True)
        assert float((np.abs(a[1] - a[0]) / scale).max()) < 1e-13
        assert np.array_equal(a[1], np.swapaxes(a[1], 1, 2))
    ref = sw["lnlike_m1_n1"]
    fin = np.isfinite(ref)
    assert np.array_equal(np.isneginf(ll[1]), np.isneginf(ref))
    assert np.max(np.abs(ll[1][fin] - ref[fin]) / np.abs(ref[fin])) <= 1e-8
    assert np.max(np.abs(ll[1][fin] - ll[0][fin]) / np.abs(ll[0][fin])) <= 1e-10


def test_uniform_time_stamps_fast_path_matches_general_assembly(spb, monkeypatch):
    """flux.py:256-276 for equally spaced time stamps: the tabulated interpolant (spb_noise_model.uniform_dt,
    rowsum_sym_kernel<UniformEntry>) against the per-entry evaluation -- several periods (0, few and many wraps per
    light curve), a shifted grid, and an irregular grid, which must not take the fast path."""
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(48, 1234)
    rng = np.random.default_rng(1)
    grids = [(1.0, t), (0.37, t), (3.3, t), (11.0, t), (1.0, np.linspace(-2.0, 7.5, 777)),
             (1.0, np.sort(rng.uniform(0, 4, 500)))]
    for period, tt in grids:
        fl = np.interp(tt, t, flux)
        out = {}
        for on in (False, True):
            if on:
                monkeypatch.delenv("SPB200_NO_UNIFORM_T", raising=False)
            else:
                monkeypatch.setenv("SPB200_NO_UNIFORM_T", "1")
            gp = spb.StarryProcess(**hp)
            out[on] = (gp.log_likelihood(tt, fl, 1e-6, p=period, u=U_LD).cpu().numpy(), gp._udt)
        uniform = bool(np.allclose(np.diff(tt), np.diff(tt)[0], rtol=1e-9, atol=0))
        assert (out[True][1] > 0) == uniform and out[False][1] == 0.0
        fin = np.isfinite(out[False][0])
        assert np.array_equal(np.isfinite(out[True][0]), fin)
        d = np.max(np.abs(out[True][0][fin] - out[False][0][fin]) / np.abs(out[False][0][fin]))
        assert d <= (2e-10 if uniform else 0.0), (period, len(tt), d)


def test_conditional_covariance_product_on_int8_tensor_cores(spb):
    """flux.py:335-343 for a long light curve: K = (A Sigma) A^T of the conditional log-likelihood (lower
    triangle, unnormalised process) evaluated on the INT8 tensor cores (gemm_i8_lower_kernel) against the
    FP64 (DMMA) GEMM: same lnlike to rounding noise, shared and per-sample inclinations, a size that is not
    a multiple of the tile."""
    import bench

    hp, t0, f0, _ = bench.synthetic_inputs(12, 1234)
    ctx = spb.get_context()
    for nt, inc in ((1500, 60.0), (1111, np.linspace(20.0, 80.0, 12))):
        tt = np.linspace(0.0, 9.0, nt)
        fl = np.interp(tt, t0 * 2.25, f0)
        out = {}
        try:
            for on in (0, 1):
                ctx.set_option("moments_syrk_i8", on)
                gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hp)
                out[on] = gp.log_likelihood(tt, fl, 1e-6, i=inc, p=1.3, u=U_LD).cpu().numpy()
        finally:
            ctx.set_option("moments_syrk_i8", 1)
        assert np.all(np.isfinite(out[0]))
        assert np.max(np.abs(out[1] - out[0]) / np.abs(out[0])) < 1e-10, nt
