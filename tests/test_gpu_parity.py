"""GPU (-m gpu): the CUDA path (libspb200 through the StarryProcess surface and the raw C ABI)
against the CPU oracle and the golden fixtures produced by the unmodified reference.

Tolerances
  * lnlike: 1e-8 relative (BASELINE.json north star), fp64 end to end.
  * For the reference's broad stability prior (joss/figures/stability.py) in the MARGINALISED branch
    the reference's own result moves by 1e-7..4e-5 relative between its two supported eigensolver
    drivers (numpy vs scipy, ops/eigh/eigh.py:11-26; measured with oracle/theano_stub) because
    noise-level (1e-15) eigen-modes of the latitude/longitude moment matrices survive its clip
    and are amplified by the 7.8e7 polynomial Wigner coefficients.  Those draws are held to the
    looser REF_NOISE_RTOL and the excess over 1e-8 is reported (DESIGN.md "numerical fragility").
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import FID, U_LD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RTOL = 1e-8
REF_NOISE_RTOL = 5e-7
# Comparisons against the oracle evaluated LIVE on the test host.  The oracle (and the reference:
# same NumPy/SciPy/BLAS calls) is not reproducible to 1e-8 across hosts: for the nt=129 marginal
# case below it returns 672.9743698036 on the development container's CPU and 672.9743602322 on
# the GPU box's CPU (1.4e-8 apart; same image, same code, OpenBLAS picks different kernels) -- the
# whole of that difference is the hyperparameter-independent longitude eigenvector table
# (VERDICT r1, weak #1).  Live comparisons therefore build the CUDA context with
# ``longitude_basis="host"`` (this host's own numpy.linalg.eigh, what the oracle uses in this
# process) and hold 1e-8 (tests/test_gpu_round2.py::test_host_basis_against_live_oracle_1e8 is the
# dedicated test); LIVE_RTOL only bounds the reported excess of a draw that sits on the reference's
# own latitude-eigensolver noise floor.
LIVE_RTOL = 1e-7


def live_tol(oracle, fn):
    """Tolerance for a live comparison that missed 1e-8: LIVE_RTOL, widened (never beyond
    REF_NOISE_RTOL) to 4x the oracle's own reproducibility floor for these inputs -- how far
    its lnlike moves between the reference's two eigensolver drivers, under a x4 change of the
    1e-15 eigenvalue clip and under one-ulp noise on the latitude moment matrix
    (oracle.reference_noise_floor).  The golden-fixture tests do not use this: they hold 1e-8."""
    floor = float(np.max(oracle.reference_noise_floor(fn)))
    return min(max(LIVE_RTOL, 4.0 * floor), REF_NOISE_RTOL), floor


@pytest.fixture(scope="module")
def spb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


def rel(a, b):
    return np.abs(a - b) / np.abs(b)


def P(t):
    return ctypes.c_void_p(t.data_ptr())


# --------------------------------------------------------------------------------------- pieces
def test_wigner_rx_bitwise(spb, oracle):
    ctx = spb.get_context(0)
    nat = oracle.get_native("port")
    th = torch.tensor([0.5 * np.pi, -np.pi / 3, 0.1, 0.0, 1.2345, -1.5707963], dtype=torch.float64,
                      device="cuda")
    R = torch.empty(th.numel(), 5456, dtype=torch.float64, device="cuda")
    assert ctx.lib.spb_Rx(ctx.handle, th.numel(), P(th), P(R), None) == 0
    for k in range(th.numel()):
        ref = nat.Rx(15, 2, th[k].item())
        assert np.abs(R[k].cpu().numpy() - ref).max() <= 2e-15


def test_tensordotRz(spb, oracle):
    ctx = spb.get_context(0)
    nat = oracle.get_native("port")
    rng = np.random.default_rng(3)
    M = rng.standard_normal((300, 256))
    th = rng.uniform(-7, 7, 300)
    f = torch.empty(300, 256, dtype=torch.float64, device="cuda")
    Mt, tt = torch.tensor(M, device="cuda"), torch.tensor(th, device="cuda")
    assert ctx.lib.spb_tensordotRz(ctx.handle, 300, P(Mt), P(tt), P(f), None) == 0
    assert np.abs(f.cpu().numpy() - nat.tensordotRz(15, 2, M, th)).max() <= 1e-13


def test_flux_operator(spb, oracle):
    ctx = spb.get_context(0)
    nat = oracle.get_native("port")
    us = np.array([[0.0, 0.0], [0.4, 0.26], [1.0, -0.3], [0.1, 0.8]])
    out = torch.empty(4, 256, dtype=torch.float64, device="cuda")
    ut = torch.tensor(us, device="cuda")
    assert ctx.lib.spb_flux_operator(ctx.handle, 4, P(ut), P(out), None) == 0
    for k in range(4):
        # the reference's sparse change of basis carries ~1e-11 cancellation noise (incl. non-zero
        # m != 0 entries); the closed form is exact to rounding
        assert np.abs(out[k].cpu().numpy() - nat.rTA1L(15, 2, us[k])).max() <= 2e-11


def test_design_matrix(spb, golden):
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **FID)
    dm = golden("design_matrix_ref.npz")
    for k, u in enumerate(([0.0, 0.0], dm["u"])):
        A = gp.design_matrix(dm["t"], i=torch.tensor(dm["incs"]), p=1.0, u=u).cpu().numpy()
        assert np.abs(A - dm["A"][k]).max() <= 2e-11
    af = golden("design_matrix_AF15.npz")  # independent `starry` matrices shipped by the reference
    A = gp.design_matrix(af["theta_deg"] / 360.0, i=torch.tensor(af["incs"]), p=1.0,
                         u=[0.0, 0.0]).cpu().numpy()
    assert np.abs(A - af["A_F"]).max() <= 5e-12
    # ragged / single-row shapes
    A1 = gp.design_matrix([0.3], i=45.0).cpu().numpy()
    A33 = gp.design_matrix(np.linspace(0, 2, 33), i=45.0).cpu().numpy()
    assert A1.shape == (1, 256) and A33.shape == (33, 256)
    assert np.abs(A1[0] - gp.design_matrix([0.3, 0.9], i=45.0).cpu().numpy()[0]).max() == 0.0


def test_cholesky_kernel_vs_lapack(spb):
    import scipy.linalg as sl

    ctx = spb.get_context(0)
    rng = np.random.default_rng(0)
    for (B, n, M) in [(2, 1, 1), (2, 7, 2), (3, 64, 0), (2, 100, 3), (2, 257, 140), (2, 1000, 1)]:
        ld = n + (n & 1)
        A = rng.standard_normal((B, n, 40))
        Kh = A @ A.transpose(0, 2, 1) / 40 + 0.5 * np.eye(n)[None]
        Kp = np.zeros((B, n, ld))
        Kp[:, :, :n] = Kh
        K = torch.tensor(Kp, device="cuda")
        Rh = rng.standard_normal((B, max(M, 1), n))
        Rp = np.zeros((B, max(M, 1), ld))
        Rp[:, :, :n] = Rh
        R = torch.tensor(Rp, device="cuda")
        ll = torch.zeros(B, dtype=torch.float64, device="cuda")
        info = torch.zeros(B, dtype=torch.int32, device="cuda")
        st = ctx.lib.spb_cholesky_lnlike(ctx.handle, B, n, P(K), ld, n * ld, M, P(R) if M else None,
                                         ld, max(M, 1) * ld, P(ll), None, None, P(info), None)
        assert st == 0
        torch.cuda.synchronize()
        for b in range(B):
            L = np.linalg.cholesky(Kh[b])
            assert np.abs(np.tril(K[b].cpu().numpy()[:, :n]) - L).max() <= 1e-12
            if M:
                y = sl.solve_triangular(L, Rh[b, :M].T, lower=True)
                ref = -0.5 * (y ** 2).sum() - M * np.log(np.diag(L)).sum() - 0.5 * n * M * np.log(
                    2 * np.pi)
                assert abs(ll[b].item() - ref) <= 1e-11 * abs(ref)
        assert int(info.abs().sum()) == 0
    # non positive-definite element -> -inf for that element only (math.py:82-91, sp.py:1186-1188)
    K = torch.eye(100, dtype=torch.float64, device="cuda").repeat(3, 1, 1).contiguous()
    K[1, 50, 50] = -1.0
    K[2, 10, 10] = float("nan")
    R = torch.ones(3, 1, 100, dtype=torch.float64, device="cuda")
    ll = torch.zeros(3, dtype=torch.float64, device="cuda")
    info = torch.zeros(3, dtype=torch.int32, device="cuda")
    assert ctx.lib.spb_cholesky_lnlike(ctx.handle, 3, 100, P(K), 100, 10000, 1, P(R), 100, 100,
                                       P(ll), None, None, P(info), None) == 0
    out = ll.cpu().numpy()
    assert np.isfinite(out[0]) and np.isneginf(out[1]) and np.isneginf(out[2])
    assert info.cpu().numpy().tolist() == [0, 1, 1]


def test_cholesky_cluster_and_batch_kernels_agree(spb):
    """The one-matrix-per-cluster kernel (small batches, cluster sizes 8 / 4 / 2) runs the same
    arithmetic per tile as the one-CTA-per-matrix kernel: identical factors and solved rows, bit
    for bit; lnlike to rounding (different summation order of |L^-1 r|^2); non-PD flagged alike."""
    ctx = spb.get_context(0)
    n, M, Bbig = 600, 3, 160   # 160 matrices: batch kernel; subsets of 3 / 20 / 60: clusters
    gen = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn(Bbig, n, 32, dtype=torch.float64, device="cuda", generator=gen)
    K0 = torch.bmm(A, A.transpose(1, 2)) / 32 + torch.eye(n, dtype=torch.float64, device="cuda")
    K0[1, 300, 300] = -5.0     # one non-PD element
    R0 = torch.randn(Bbig, M, n, dtype=torch.float64, device="cuda", generator=gen)

    def run(B):
        K, R = K0[:B].clone(), R0[:B].clone()
        ll = torch.zeros(B, dtype=torch.float64, device="cuda")
        info = torch.zeros(B, dtype=torch.int32, device="cuda")
        assert ctx.lib.spb_cholesky_lnlike(ctx.handle, B, n, P(K), n, n * n, M, P(R), n, M * n,
                                           P(ll), None, None, P(info), None) == 0
        torch.cuda.synchronize()
        return torch.tril(K), R, ll, info

    Lb, Rb, llb, ib = run(Bbig)
    for B in (3, 20, 60):
        Lc, Rc, llc, ic = run(B)
        ok = [b for b in range(B) if b != 1]
        assert torch.equal(Lc[ok], Lb[:B][ok]) and torch.equal(Rc[ok], Rb[:B][ok])
        assert float((llc[ok] - llb[:B][ok]).abs().max()) <= 1e-13 * float(llb[ok].abs().max())
        assert torch.equal(ic, ib[:B]) and int(ic[1]) == 1 and bool(torch.isneginf(llc[1]))


def test_solve_rows_many_rhs(spb):
    """y = L^-1 r for M rows against one factor, nt in {1, 2, 127, 129, 1000, 4097} (odd nt with an even, padded
    ld) x M in {1, 31, 300}.  Backward error of each solved row, the residual L y - r formed by exact dot
    products: a triangular solve returns the exact solution of (L + dL) y = r with |dL| <= gamma_nt |L|, so
    |L y - r|_i <= gamma_nt (|L||y|)_i; doubled (c = 2) for the reciprocal-times-multiply division, plus u for
    the correctly rounded residual.  quad against math.fsum(y^2) of the returned y within gamma_nt (a sum of
    nt non-negative squares, each rounded)."""
    import math

    import scipy.linalg as sl

    from exact_ref import exact_dot_rows

    ctx = spb.get_context(0)
    u = 2.0 ** -53

    def gam(k):
        return k * u / (1 - k * u)

    for n in (1, 2, 127, 129, 1000, 4097):
        rng = np.random.default_rng(n)
        ld = n + (n & 1)
        A = rng.standard_normal((n, 50))
        L = np.linalg.cholesky(A @ A.T / 50 + 0.5 * np.eye(n))
        Lp = np.zeros((n, ld))
        Lp[:, :n] = L
        Lt = torch.tensor(Lp, device="cuda")
        for M in (1, 31, 300):
            Rh = rng.standard_normal((M, n))
            Rp = np.zeros((M, ld))
            Rp[:, :n] = Rh
            R = torch.tensor(Rp, device="cuda")
            quad = torch.zeros(M, dtype=torch.float64, device="cuda")
            assert ctx.lib.spb_cholesky_solve_rows(ctx.handle, n, P(Lt), ld, M, P(R), ld, P(quad), None) == 0
            Y = R.cpu().numpy()[:, :n]
            q = quad.cpu().numpy()
            if n == 1000 and M == 300:   # the original scipy comparison
                y = sl.solve_triangular(L, Rh.T, lower=True)
                assert np.abs(Y - y.T).max() <= 1e-11
            rows = sorted({0, 1, 63, 64, 127, 128, n - 1} & set(range(n)) | set(int(x) for x in rng.integers(0, n, 8)))
            for m in sorted({0, M - 1, M // 2}):
                X = np.concatenate([L, Rh[m][:, None]], axis=1)   # (L y - r)_i = [L_i, r_i] . [y, -1]
                yv = np.concatenate([Y[m], [-1.0]])[None]
                res = exact_dot_rows(X, yv, [(i, 0) for i in rows])
                LY = exact_dot_rows(np.abs(L), np.abs(Y[m:m + 1]), [(i, 0) for i in rows])
                assert np.all(np.abs(res) <= (2 * gam(n) + u) * LY * (1 + 2 * u)), (n, M, m)
                fs = math.fsum((Y[m] ** 2).tolist())   # each square rounded once more on the host: gamma_{n+1}
                assert abs(q[m] - fs) <= gam(n + 1) * fs, (n, M, m, q[m], fs)


# --------------------------------------------------------------------------------------- moments
def test_ylm_moments(spb, golden, oracle):
    g = golden("fiducial_nt1000.npz")
    gp = spb.StarryProcess(**FID)
    mu = gp.mean_ylm.cpu().numpy()
    cov = gp.cov_ylm.cpu().numpy()
    assert np.abs(mu - g["mean_ylm"]).max() <= 1e-14 * np.abs(g["mean_ylm"]).max()
    # elementwise cov parity is bounded by the reference's own noise modes (SURVEY.md section 7)
    assert np.abs(cov - g["cov_ylm"]).max() <= 2e-7
    assert np.abs(cov - cov.T).max() == 0.0
    o = oracle.OracleProcess(**FID)
    low = slice(0, 100)  # l <= 9: far from the noise-dominated high degrees
    assert np.abs(cov[low, low] - o.cov_ylm[low, low]).max() <= 1e-8 * np.abs(o.cov_ylm).max()
    assert int(gp.info.item()) == 0
    # batched == one at a time
    sw = golden("sweep_lowc_nt1000.npz")
    gb = spb.StarryProcess(r=sw["r"][:5], mu=sw["mu"][:5], sigma=sw["sigma"][:5], c=sw["c"][:5],
                           n=sw["n"][:5])
    covb = gb.cov_ylm.cpu().numpy()
    for s in range(5):
        g1 = spb.StarryProcess(r=sw["r"][s], mu=sw["mu"][s], sigma=sw["sigma"][s], c=sw["c"][s],
                               n=sw["n"][s])
        assert np.array_equal(g1.cov_ylm.cpu().numpy(), covb[s])
    assert np.abs(gb.mean_ylm.cpu().numpy() - sw["mean_ylm"][:5]).max() <= 1e-11 * np.abs(
        sw["mean_ylm"][:5]).max()


def test_sample_ylm_given_cov(spb, golden, oracle):
    """sp.py:505-509: same u in -> same y out, for the same cov_ylm (the factor of the reference's
    own cov_ylm is fed through the C ABI; cov_ylm itself is only reproducible to the reference's
    noise floor and its Cholesky factor amplifies that by 1/sqrt(lambda_min))."""
    g = golden("fiducial_nt1000.npz")
    sy = golden("sample_ylm.npz")
    ctx = spb.get_context(0)
    cov = torch.tensor(g["cov_ylm"], device="cuda").reshape(1, 256, 256).contiguous()
    L = torch.empty_like(cov)
    info = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert ctx.lib.spb_cho_cov_ylm(ctx.handle, 1, P(cov), P(L), P(info), None) == 0
    assert np.allclose(np.diag(L[0].cpu().numpy()), g["cho_ylm_diag"], rtol=1e-9)
    assert float(torch.triu(L[0], 1).abs().max()) == 0.0
    un = torch.tensor(sy["unit_normals"].T.copy(), device="cuda").reshape(1, -1, 256).contiguous()
    mean = torch.tensor(g["mean_ylm"], device="cuda").reshape(1, 256)
    y = torch.empty(1, un.shape[1], 256, dtype=torch.float64, device="cuda")
    assert ctx.lib.spb_sample_ylm(ctx.handle, 1, un.shape[1], P(mean), P(L), P(un), P(y), None) == 0
    assert np.abs(y[0].cpu().numpy() - sy["y"]).max() <= 1e-9 * np.abs(sy["y"]).max()
    # surface-level call: shapes and first/second moments of the draws
    gp = spb.StarryProcess(**FID)
    ys = gp.sample_ylm(nsamples=4000, generator=torch.Generator(device="cuda").manual_seed(0))
    assert tuple(ys.shape) == (4000, 256)
    emp = torch.cov(ys.T).cpu().numpy()
    covg = gp.cov_ylm.cpu().numpy()
    assert np.abs(emp - covg).max() <= 0.15 * np.abs(covg).max()


# --------------------------------------------------------------------------------------- lnlike
@pytest.mark.parametrize("marg", [False, True])
@pytest.mark.parametrize("norm", [False, True])
def test_fiducial_cov_and_lnlike(spb, golden, marg, norm):
    g = golden("fiducial_nt1000.npz")
    t = g["t"]
    gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **FID)
    for uname, u in (("u0", [0.0, 0.0]), ("uld", U_LD)):
        key = "m%d_n%d_%s" % (marg, norm, uname)
        K = gp.cov(t, i=60.0, p=1.0, u=u).cpu().numpy()
        scale = np.abs(K).max()
        assert np.abs(K - K.T).max() <= 1e-15 * scale
        for row, name in ((K[0], "Krow0_"), (K[500], "Krow500_"), (np.diag(K), "Kdiag_")):
            assert np.abs(row - g[name + key]).max() <= 1e-8 * scale
        f = g["flux_norm"] if norm else g["flux"]
        fe = g["flux_ens_norm"] if norm else g["flux_ens"]
        ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=u).item()
        assert rel(ll, g["lnlike_" + key]) <= RTOL
        lle = gp.log_likelihood(t, fe, 1e-6, i=60.0, p=1.0, u=u).item()
        assert rel(lle, g["lnlike_ens_" + key]) <= RTOL
        if not norm:
            m = gp.mean(t, i=60.0, p=1.0, u=u).cpu().numpy()
            assert np.abs(m - g["gpmean_" + key]).max() <= 1e-12 * abs(g["gpmean_" + key])
    key = "m%d_n%d" % (marg, norm)
    f = g["flux_norm"] if norm else g["flux"]
    ll = gp.log_likelihood(t, f, g["data_cov_vec"], i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4,
                           baseline_var=1e-5).item()
    assert rel(ll, g["lnlike_dvec_" + key]) <= RTOL
    # full data-covariance matrix == its diagonal form
    ll2 = gp.log_likelihood(t, f, np.diag(g["data_cov_vec"]), i=60.0, p=1.0, u=U_LD,
                            baseline_mean=1e-4, baseline_var=1e-5).item()
    assert rel(ll2, ll) <= 1e-12


@pytest.mark.parametrize("name", ["sweep_lowc_nt1000.npz", "sweep_nt1000.npz"])
def test_hyperparameter_sweep_batched(spb, golden, name):
    sw = golden(name)
    g = golden("fiducial_nt1000.npz")
    t = g["t"]
    worst = {}
    for marg in (False, True):
        for norm in (False, True):
            gp = spb.StarryProcess(r=sw["r"], mu=sw["mu"], sigma=sw["sigma"], c=sw["c"], n=sw["n"],
                                   marginalize_over_inclination=marg, normalized=norm)
            f = g["flux_norm"] if norm else g["flux"]
            ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
            ref = sw["lnlike_m%d_n%d" % (marg, norm)]
            fin = np.isfinite(ref)
            # -inf pattern (normalised process outside z <= 0.023) must match exactly
            assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
            err = rel(ll[fin], ref[fin]) if fin.any() else np.zeros(1)
            worst[(marg, norm)] = err.max()
            noisy = marg and name == "sweep_nt1000.npz"
            assert err.max() <= (REF_NOISE_RTOL if noisy else RTOL), (marg, norm, err.max())
    print("max relative lnlike error per (marg, norm):", worst)


def test_bench_workload_against_reference_golden(spb, golden):
    """The first 256 hyperparameter samples of the bench.py sweep (seed 1234) against the values
    the unmodified reference produced for them (oracle/gen_golden_bench.py): 1e-8, both branches."""
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, seed=1234)
    sw = golden("bench_sweep_seed1234.npz")
    ns = len(sw["r"])
    assert ns >= 256
    for k in ("r", "mu", "sigma", "c", "n"):
        assert np.array_equal(sw[k], hp[k][:ns])
    for marg in (True, False):
        gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=True,
                               **{k: hp[k][:ns] for k in hp})
        ll = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
        ref = sw["lnlike_m%d_n1" % marg]
        assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
        fin = np.isfinite(ref)
        err = rel(ll[fin], ref[fin])
        print("bench sweep marg=%d: max rel err vs reference %.2e" % (marg, err.max()))
        assert err.max() <= RTOL


def test_calibrate_callers_against_reference(spb, golden):
    """get_log_prob (calibrate/log_prob.py:7-106), log_jac (latitude.py:281-316) and the inclination
    grid of calibrate/inclination.py:63-74, batched, against values produced by the unmodified
    reference (oracle/gen_golden_calibrate.py): 1e-8 relative."""
    from starry_process_b200 import calibrate

    g = golden("calibrate_log_prob.npz")
    t, fl = g["t"], g["flux"]
    T = lambda x: torch.tensor(np.asarray(x), dtype=torch.float64)  # noqa: E731
    gp = spb.StarryProcess(r=T(g["r"]), a=T(g["a"]), b=T(g["b"]), c=T(g["c"]), n=T(g["n"]))
    lj = gp.log_jac().cpu().numpy()
    assert rel(lj, g["log_jac"]).max() <= 1e-11
    assert spb.StarryProcess(r=10.0, mu=30.0, sigma=46.0, c=0.1, n=10.0).log_jac().item() == -np.inf
    # marginalised, three light curves scored jointly, fixed baseline, Jacobian applied
    f = calibrate.get_log_prob(t, flux=fl, ferr=1e-3, p=1.0, u=U_LD)
    lp = f(T(g["r"]), T(g["a"]), T(g["b"]), T(g["c"]), T(g["n"])).cpu().numpy()
    e1 = rel(lp, g["log_prob_marg"]).max()
    # scalar call == the reference's calling convention
    lp0 = f(float(g["r"][0]), float(g["a"][0]), float(g["b"][0]), float(g["c"][0]), float(g["n"][0]))
    assert rel(lp0.item(), g["log_prob_marg"][0]) <= RTOL
    # conditional, free flux / baseline mean / baseline log-variance / inclination, all per element
    f2 = calibrate.get_log_prob(t, flux=None, ferr=1e-3, p=1.0, marginalize_over_inclination=False,
                                baseline_mean=None, baseline_log_var=None, u=U_LD)
    lp2 = f2(fl[:1], T(g["r"]), T(g["a"]), T(g["b"]), T(g["c"]), T(g["n"]), T(g["m"]), T(g["v"]),
             T(g["inc_cond"])).cpu().numpy()
    e2 = rel(lp2, g["log_prob_cond"]).max()
    grid = calibrate.inclination_log_prob(
        t, fl[:2], np.stack([g["r"][:2], g["a"][:2], g["b"][:2], g["c"][:2], g["n"][:2]], axis=1),
        g["inc_grid"], ferr=1e-3, p=1.0).cpu().numpy()
    e3 = rel(grid, g["lp_grid"]).max()
    print("calibrate callers: max rel err marg %.2e cond %.2e grid %.2e" % (e1, e2, e3))
    # The grid uses the reference defaults baseline_log_var = 0, i.e. + 1.0 on every entry of a
    # covariance whose other eigenvalues are ~1e-6: cond(K) = 2.5e8, so two correct fp64
    # factorisations differ by ~cond * eps = 3e-8 (the pole-on column, i = 0, is rank one on top).
    assert e1 <= RTOL and e2 <= RTOL and e3 <= 1e-7


def test_long_baseline_limb_darkened(spb, golden):
    lb = golden("longbaseline_nt4096.npz")
    gp = spb.StarryProcess(r=lb["r"], mu=lb["mu"], sigma=lb["sigma"], c=lb["c"], n=lb["n"],
                           marginalize_over_inclination=False, normalized=False)
    ll = gp.log_likelihood(lb["t"], lb["flux"], 1e-6, i=60.0, p=1.0, u=lb["u"]).cpu().numpy()
    assert rel(ll, lb["lnlike"]).max() <= RTOL


def test_live_oracle_odd_sizes_and_inclinations(spb, oracle):
    """CUDA vs the oracle evaluated on the spot: ragged nt, per-element inclinations, nt == 1."""
    rng = np.random.default_rng(11)
    hp = dict(r=17.0, mu=42.0, sigma=11.0, c=0.08, n=6.0)
    for nt in (1, 2, 63, 129, 301):
        t = np.sort(rng.uniform(0, 3, nt))
        f = 1e-3 * rng.standard_normal(nt)
        for marg in (False, True):
            for norm in (False, True):
                if nt == 1 and norm:
                    continue  # mean(Sig) == Sig: the series degenerates; not a reference use case
                def fn(**kw):
                    o = oracle.OracleProcess(marginalize_over_inclination=marg, normalized=norm,
                                             **hp, **kw)
                    return o.log_likelihood(t, f, 1e-6, i=33.0, p=0.7, u=U_LD)

                gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm,
                                       longitude_basis="host", **hp)
                ref = fn()
                ll = gp.log_likelihood(t, f, 1e-6, i=33.0, p=0.7, u=U_LD).item()
                err = rel(ll, ref)
                if err > RTOL:
                    tol, floor = live_tol(oracle, fn)
                    print("live oracle nt=%d marg=%d norm=%d: err %.2e, reference floor %.2e"
                          % (nt, marg, norm, err, floor))
                    assert err <= tol, (nt, marg, norm, err, floor)
    # one inclination per batch element (calibrate/inclination.py:66-74 style grid)
    incs = np.array([5.0, 30.0, 60.0, 85.0])
    t = np.linspace(0, 2, 150)
    f = 1e-3 * rng.standard_normal(150)
    gp = spb.StarryProcess(r=np.full(4, 17.0), mu=np.full(4, 42.0), sigma=np.full(4, 11.0),
                           c=np.full(4, 0.08), n=np.full(4, 6.0), longitude_basis="host",
                           marginalize_over_inclination=False, normalized=False)
    ll = gp.log_likelihood(t, f, 1e-6, i=torch.tensor(incs), p=1.0, u=U_LD).cpu().numpy()
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **hp)
    ref = np.array([o.log_likelihood(t, f, 1e-6, i=inc, p=1.0, u=U_LD) for inc in incs])
    assert rel(ll, ref).max() <= RTOL


def test_bounds_and_flags(spb):
    with pytest.raises(ValueError):
        spb.StarryProcess(r=95.0)
    with pytest.raises(ValueError):
        spb.StarryProcess(a=1.5, b=0.2)
    with pytest.raises(ValueError):
        spb.StarryProcess(n=-1.0)
    with pytest.raises(ValueError):
        spb.StarryProcess(mu=30.0)
    gp = spb.StarryProcess(**FID)
    with pytest.raises(ValueError):
        gp.cov([0.0, 0.1], i=100.0)
    # device-resident out-of-range hyperparameters cannot raise without a sync: flagged, -inf
    r = torch.tensor([10.0, 120.0], dtype=torch.float64, device="cuda")
    gp = spb.StarryProcess(r=r, mu=30.0, sigma=5.0, c=0.1, n=10.0)
    ll = gp.log_likelihood(np.linspace(0, 1, 50), np.zeros(50), 1e-6)
    assert np.isfinite(ll[0].item()) and np.isneginf(ll[1].item())
    assert int(gp.info[1].item()) & 4


def test_full_size_properties(spb, golden):
    """BASELINE sizes, size-independent properties: a batch of identical hyperparameters gives
    identical lnlike in every slot; chunked and unchunked evaluation agree bit for bit (same
    kernel), and to rounding when the chunks take another kernel (FP64 instead of INT8 tensor cores, or
    the one-matrix-per-cluster Cholesky (different summation order of |L^-1 r|^2); joint lnlike of M curves == sum over curves
    + shared log-determinant bookkeeping."""
    g = golden("fiducial_nt1000.npz")
    t = g["t"]
    B = 296
    gp = spb.StarryProcess(r=np.full(B, 10.0), mu=np.full(B, 30.0), sigma=np.full(B, 5.0),
                           c=np.full(B, 0.1), n=np.full(B, 10.0))
    ll = gp.log_likelihood(t, g["flux_norm"], 1e-6, u=U_LD)
    assert float((ll - ll[0]).abs().max()) == 0.0
    assert rel(ll[0].item(), g["lnlike_m1_n1_uld"]) <= RTOL
    gp2 = spb.StarryProcess(r=np.full(B, 10.0), mu=np.full(B, 30.0), sigma=np.full(B, 5.0),
                            c=np.full(B, 0.1), n=np.full(B, 10.0), max_chunk_bytes=1 << 30)
    ll2 = gp2.log_likelihood(t, g["flux_norm"], 1e-6, u=U_LD)     # chunks of ~60 matrices
    # the 296-matrix batch factorises on the INT8 tensor cores, the small chunks on the FP64 kernel:
    # same numbers to rounding noise (csrc/potrf_i8.cuh)
    assert float((ll2 - ll).abs().max()) <= 1e-11 * float(ll.abs().max())
    ctx = spb.get_context()
    try:                                                          # same kernel: bit for bit
        ctx.set_option("cholesky_i8", 0)
        gp2 = spb.StarryProcess(r=np.full(B, 10.0), mu=np.full(B, 30.0), sigma=np.full(B, 5.0),
                                c=np.full(B, 0.1), n=np.full(B, 10.0), max_chunk_bytes=2 << 30)
        lla = gp.log_likelihood(t, g["flux_norm"], 1e-6, u=U_LD)
        llb = gp2.log_likelihood(t, g["flux_norm"], 1e-6, u=U_LD)
        assert torch.equal(lla, llb)
    finally:
        ctx.set_option("cholesky_i8", -1)
    gp3 = spb.StarryProcess(r=np.full(B, 10.0), mu=np.full(B, 30.0), sigma=np.full(B, 5.0),
                            c=np.full(B, 0.1), n=np.full(B, 10.0), max_chunk_bytes=100 << 20)
    ll3 = gp3.log_likelihood(t, g["flux_norm"], 1e-6, u=U_LD)     # chunks of ~12: cluster kernel
    assert float((ll3 - ll3[0]).abs().max()) == 0.0               # deterministic
    assert float((ll3 - ll).abs().max()) <= 1e-13 * float(ll.abs().max())
    g1 = spb.StarryProcess(**FID)
    fe = g["flux_ens_norm"]
    joint = g1.log_likelihood(t, fe, 1e-6, u=U_LD).item()
    singles = [g1.log_likelihood(t, fe[m], 1e-6, u=U_LD).item() for m in range(fe.shape[0])]
    assert abs(joint - sum(singles)) <= 1e-10 * abs(joint)
