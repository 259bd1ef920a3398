"""GPU (-m gpu), round 2: the branches and claims round 1 left untested.

* parity on THIS host: a context built with ``longitude_basis="host"`` against the same-process live
  oracle at 1e-8 (the pinned table reproduces the build container's values instead);
* the ``M >= 64`` ensemble branch of ``log_likelihood`` (configs[1]) against the reference golden;
* 16 nt = 4096 draws incl. a non positive-definite element and a z > zmax element (configs[3]);
* the z-range flag is re-evaluated per call (not sticky);
* TMA-fed vs cp.async-fed Cholesky operand ring: bit-identical factors and lnlike under load;
* run-to-run determinism of the full 4096-matrix step.
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import FID, U_LD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RTOL = 1e-8


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


# ------------------------------------------------------------------------- parity on this host
def test_host_basis_against_live_oracle_1e8(spb, oracle, golden):
    """VERDICT r1 weak #1: with the longitude eigenvector table taken from THIS host's
    numpy.linalg.eigh (``longitude_basis="host"``: exactly what the reference / oracle computes in
    this process) the CUDA path meets the 1e-8 north-star tolerance against the live oracle --
    64 draws of the bench workload in both branches and the four fiducial modes at nt = 1000."""
    import bench
    from starry_process_b200 import _tables

    # the product's host table is the oracle's own U_lon, bit for bit (same NumPy call, same process)
    U_or = oracle.longitude_tensors(15)[0]
    assert np.array_equal(_tables.longitude_U("host"), U_or)
    hp, t, flux, _ = bench.synthetic_inputs(4096, seed=1234)
    ns = 64
    worst = {}
    for marg in (True, False):
        gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=True,
                               longitude_basis="host", **{k: hp[k][:ns] for k in hp})
        assert gp._ctx.longitude_basis == "host"
        ll = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
        ref = np.array([oracle.OracleProcess(marginalize_over_inclination=marg, normalized=True,
                                             **{k: hp[k][s] for k in hp}).log_likelihood(
            t, flux, 1e-6, i=60.0, p=1.0, u=U_LD) for s in range(ns)])
        assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
        fin = np.isfinite(ref)
        worst["bench marg=%d" % marg] = float(rel(ll[fin], ref[fin]).max())
    g = golden("fiducial_nt1000.npz")
    for marg in (False, True):
        for norm in (False, True):
            gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm,
                                   longitude_basis="host", **FID)
            f = g["flux_norm"] if norm else g["flux"]
            ll = gp.log_likelihood(g["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD).item()
            ref = oracle.OracleProcess(marginalize_over_inclination=marg, normalized=norm,
                                       **FID).log_likelihood(g["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD)
            worst["fiducial m%d n%d" % (marg, norm)] = float(rel(ll, ref))
    print("host basis vs live oracle (max rel lnlike err):", worst)
    assert max(worst.values()) <= RTOL, worst


def test_pinned_and_host_contexts_coexist(spb):
    a = spb.get_context(0)
    b = spb.get_context(0, "host")
    assert a is not b and a.longitude_basis == "pinned" and b.longitude_basis == "host"
    assert spb.get_context(0, "host") is b
    with pytest.raises(ValueError):
        spb.get_context(0, "nonsense")


# ------------------------------------------------------------------------- configs[1]: M >= 64
def test_ensemble_branch_against_reference_golden(spb, golden):
    """sp.py:1157-1173 with flux (1024, 1000): one factorisation + spb_cholesky_solve_rows over the
    whole GPU + the host-side reduction (StarryProcess.log_likelihood, ``Bc == 1 and M >= 64``), in
    all four modes, with a scalar and a per-point data covariance, against the unmodified
    reference (oracle/gen_golden_r2.py)."""
    import bench

    g = golden("ensemble_nt1000.npz")
    M = int(g["M"])
    for norm in (False, True):
        t, f = bench.ensemble_flux(M, normalized=norm)
        chk = float(np.sum(f * np.cos(np.arange(f.size)).reshape(f.shape)))
        assert abs(chk - float(g["flux_checksum_n%d" % norm])) <= 1e-9 * abs(chk)  # same inputs
        for marg in (False, True):
            key = "m%d_n%d" % (marg, norm)
            gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **FID)
            ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=U_LD).item()
            assert rel(ll, float(g["lnlike_" + key])) <= RTOL, (key, ll)
            lld = gp.log_likelihood(t, f, g["data_cov_vec"], i=60.0, p=1.0, u=U_LD,
                                    baseline_mean=1e-4, baseline_var=1e-5).item()
            assert rel(lld, float(g["lnlike_dvec_" + key])) <= RTOL, (key, lld)
            l64 = gp.log_likelihood(t, f[:64], 1e-6, i=60.0, p=1.0, u=U_LD).item()
            assert rel(l64, float(g["lnlike_64_" + key])) <= RTOL, (key, l64)
            # the branch boundary: 63 curves take the augmented-rows kernel, 64 the split solve;
            # joint lnlike is additive over curves up to the shared log-determinant bookkeeping
            l63 = gp.log_likelihood(t, f[:63], 1e-6, i=60.0, p=1.0, u=U_LD).item()
            l1 = gp.log_likelihood(t, f[63], 1e-6, i=60.0, p=1.0, u=U_LD).item()
            assert abs((l63 + l1) - l64) <= 1e-10 * abs(l64)
    # a non positive-definite K on this branch -> -inf, as math.py:82-91 / sp.py:1186-1188
    gp = spb.StarryProcess(marginalize_over_inclination=True, normalized=False, **FID)
    t, f = bench.ensemble_flux(128, normalized=False)
    assert gp.log_likelihood(t, f, -1e-2, u=U_LD).item() == -np.inf


# ------------------------------------------------------------------------- configs[3]: nt = 4096
def test_long_baseline_16_draws(spb, golden):
    lb = golden("longbaseline_nt4096.npz")
    r2 = golden("longbaseline_nt4096_r2.npz")
    t, f = lb["t"], lb["flux"]
    fn = (1 + f) / np.mean(1 + f) - 1
    hp = {k: r2[k] for k in ("r", "mu", "sigma", "c", "n")}
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hp)
    ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=r2["u"],
                           baseline_var=torch.tensor(r2["baseline_var"])).cpu().numpy()
    ref = r2["lnlike_n0"]
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref)) and np.isneginf(ll[5])
    assert int(gp.info[5].item()) & 1 and int((gp.info.cpu().numpy() != 0).sum()) == 1
    fin = np.isfinite(ref)
    e0 = rel(ll[fin], ref[fin]).max()
    gpn = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **hp)
    lln = gpn.log_likelihood(t, fn, 1e-6, i=60.0, p=1.0, u=r2["u"]).cpu().numpy()
    refn = r2["lnlike_n1"]
    assert np.array_equal(np.isneginf(lln), np.isneginf(refn)) and np.isneginf(lln[11])
    assert int(gpn.info[11].item()) & 2
    z = gpn._z.cpu().numpy()
    assert rel(z, r2["z_n1"]).max() <= 1e-8 and z[11] > 0.023
    finn = np.isfinite(refn)
    e1 = rel(lln[finn], refn[finn]).max()
    print("nt=4096, 16 draws: max rel err unnormalised %.2e, normalised %.2e" % (e0, e1))
    assert e0 <= RTOL and e1 <= RTOL


def test_full_prior_bench_line_against_reference_golden(spb, golden):
    """bench.py's second line item (the reference's full stability prior): -inf pattern identical,
    finite values to the noise bound the round-1 broad-prior sweep documents."""
    import bench

    g = golden("bench_fullprior_seed4321.npz")
    ns = len(g["r"])
    hp, t, flux, _ = bench.synthetic_inputs(4096, seed=4321, prior="full")
    for k in ("r", "mu", "sigma", "c", "n"):
        assert np.array_equal(g[k], hp[k][:ns])
    gp = spb.StarryProcess(**{k: hp[k][:ns] for k in hp})
    ll = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
    ref = g["lnlike_m1_n1"]
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    fin = np.isfinite(ref)
    if fin.any():
        err = rel(ll[fin], ref[fin])
        print("full prior: %d finite of %d, max rel err %.2e" % (fin.sum(), ns, err.max()))
        assert err.max() <= 5e-7   # REF_NOISE_RTOL of tests/test_gpu_parity.py (broad prior, marg.)


# ------------------------------------------------------------------------- flags
def test_z_range_flag_is_reevaluated_per_call(spb):
    """ADVICE r1: SPB_INFO_Z_RANGE depends on (t, i, p, u); it must not stick to the process object.
    The reference re-evaluates z > zmax on every call (sp.py:1178-1183)."""
    rng = np.random.default_rng(5)
    t = np.linspace(0, 2, 120)
    f = 1e-3 * rng.standard_normal(120)
    gp = spb.StarryProcess(r=20.0, mu=30.0, sigma=5.0, c=0.4, n=10.0,
                           marginalize_over_inclination=False, normalized=True)
    incs = np.linspace(1.0, 89.0, 45)
    zs = []
    for inc in incs:
        gp.cov(t, i=float(inc))
        zs.append(float(gp._z.item()))
    zs = np.array(zs)
    assert zs.max() > 0.023 > zs.min(), "test setup: z must cross zmax over inclination"
    hi, lo = float(incs[zs.argmax()]), float(incs[zs.argmin()])
    assert gp.log_likelihood(t, f, 1e-6, i=hi).item() == -np.inf
    assert int(gp.info.item()) & 2
    ll = gp.log_likelihood(t, f, 1e-6, i=lo).item()      # same object, in-range inclination
    assert np.isfinite(ll) and not (int(gp.info.item()) & 2)
    fresh = spb.StarryProcess(r=20.0, mu=30.0, sigma=5.0, c=0.4, n=10.0,
                              marginalize_over_inclination=False, normalized=True)
    assert fresh.log_likelihood(t, f, 1e-6, i=lo).item() == ll
    # cov() / sample() of an out-of-range configuration leave no trace either
    gp.cov(t, i=hi)
    assert gp.log_likelihood(t, f, 1e-6, i=lo).item() == ll


# ------------------------------------------------------------------------- Cholesky stress
def _spd_batch(B, n, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(B, n, 24, dtype=torch.float64, device="cuda", generator=gen)
    K = torch.bmm(A, A.transpose(1, 2)) / 24
    K += torch.eye(n, dtype=torch.float64, device="cuda") * 0.7
    R = torch.randn(B, 1, n, dtype=torch.float64, device="cuda", generator=gen)
    return K, R


@pytest.mark.parametrize("B,n", [(3000, 192), (1200, 320), (700, 1000)])
def test_cholesky_tma_and_cp_async_rings_bitwise(spb, B, n):
    """ADVICE r1 (high): the factor is written with st.global (generic proxy) and re-read through
    TMA (async proxy) in the next panel; a missing fence.proxy.async shows up as stale operands at
    small nt (64-column panels follow their producer immediately) and large B (every SM busy).  The
    TMA-fed ring must reproduce the cp.async-fed ring bit for bit, launch after launch."""
    ctx = spb.get_context(0)
    K0, R0 = _spd_batch(B, n, seed=n)

    def run(tma):
        ctx.set_option("cholesky_tma", tma)
        K, R = K0.clone(), R0.clone()
        ll = torch.zeros(B, dtype=torch.float64, device="cuda")
        info = torch.zeros(B, dtype=torch.int32, device="cuda")
        assert ctx.lib.spb_cholesky_lnlike(ctx.handle, B, n, P(K), n, n * n, 1, P(R), n, n,
                                           P(ll), None, None, P(info), None) == 0
        torch.cuda.synchronize()
        assert int(info.abs().sum()) == 0
        return torch.tril(K), R, ll

    try:
        Lc, Rc, llc = run(0)
        for rep in range(3):
            Lt, Rt, llt = run(1)
            assert torch.equal(llt, llc), "lnlike differs between the TMA and cp.async rings"
            assert torch.equal(Lt, Lc) and torch.equal(Rt, Rc)
    finally:
        ctx.set_option("cholesky_tma", 1)
    # and against LAPACK on a few elements
    for b in (0, B // 2, B - 1):
        L = np.linalg.cholesky(K0[b].cpu().numpy())
        assert np.abs(Lc[b].cpu().numpy() - L).max() <= 1e-12


def test_full_step_is_deterministic_run_to_run(spb, golden):
    """VERDICT r1 weak #8: the same 4096-draw step 20 times -> bit-identical log-likelihoods (the
    mbarrier hand-offs of the operand ring that racecheck cannot follow would show up here as
    run-to-run differences under full load)."""
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, seed=1234)
    hd = {k: torch.tensor(v, device="cuda") for k, v in hp.items()}
    td, fd = torch.tensor(t, device="cuda"), torch.tensor(flux, device="cuda")
    first = None
    for rep in range(20):
        ll = spb.StarryProcess(**hd).log_likelihood(td, fd, 1e-6, p=1.0, u=U_LD)
        if first is None:
            first = ll.clone()
            sw = golden("bench_sweep_seed1234.npz")
            ref = sw["lnlike_m1_n1"]
            got = first[: len(ref)].cpu().numpy()
            fin = np.isfinite(ref)
            assert rel(got[fin], ref[fin]).max() <= RTOL
        else:
            assert torch.equal(ll, first), "run %d differs from run 0" % rep


@pytest.mark.parametrize("B, n, M", [(5, 1, 1), (3, 70, 2), (4, 257, 140), (300, 333, 1), (40, 1000, 3)])
def test_cholesky_rings_bitwise_ragged_shapes(spb, B, n, M):
    """The batch kernel with its operand ring fed by TMA and by cp.async: identical factors, solved rows
    and info, bit for bit, and the same lnlike, on ragged sizes (partial last panel), many right-hand-side
    rows and a non positive-definite element (flagged, lnlike = -inf, the other matrices unaffected)."""
    ctx = spb.get_context(0)
    ld = n + (n & 1)
    gen = torch.Generator(device="cuda").manual_seed(n)
    A = torch.randn(B, n, 24, dtype=torch.float64, device="cuda", generator=gen)
    K0 = torch.zeros(B, n, ld, dtype=torch.float64, device="cuda")
    K0[:, :, :n] = torch.bmm(A, A.transpose(1, 2)) / 24 + 0.7 * torch.eye(n, dtype=torch.float64, device="cuda")
    if n > 50:
        K0[1, 40, 40] = -3.0
    R0 = torch.zeros(B, M, ld, dtype=torch.float64, device="cuda")
    R0[:, :, :n] = torch.randn(B, M, n, dtype=torch.float64, device="cuda", generator=gen)
    outs = {}
    try:
        ctx.set_option("cholesky_cluster", 0)
        for tma in (1, 0):
            ctx.set_option("cholesky_tma", tma)
            K, R = K0.clone(), R0.clone()
            ll = torch.zeros(B, dtype=torch.float64, device="cuda")
            info = torch.zeros(B, dtype=torch.int32, device="cuda")
            assert ctx.lib.spb_cholesky_lnlike(ctx.handle, B, n, P(K), ld, n * ld, M, P(R), ld, M * ld, P(ll),
                                               None, None, P(info), None) == 0
            torch.cuda.synchronize()
            outs[tma] = (torch.tril(K[:, :, :n]), R, ll, info)
    finally:
        ctx.set_option("cholesky_tma", 1)
        ctx.set_option("cholesky_cluster", 1)
    ref, o = outs[1], outs[0]
    ok = [b for b in range(B) if not (n > 50 and b == 1)]
    assert torch.equal(o[3], ref[3])
    assert torch.equal(o[0][ok], ref[0][ok]) and torch.equal(o[1][ok], ref[1][ok])
    assert float((o[2][ok] - ref[2][ok]).abs().max()) <= 1e-13 * float(ref[2][ok].abs().max())
    assert int(ref[3][ok].abs().sum()) == 0 and bool(torch.isfinite(ref[2][ok]).all())
    if n > 50:
        assert int(ref[3][1]) == 1 and bool(torch.isneginf(ref[2][1]))


# ------------------------------------------------------------------------- uniform spot-size prior
def test_uniform_spot_size_prior_against_reference_golden(spb, golden):
    """SURVEY.md section 8(f) rank 4, first half (size.py:55-89, 116-125): StarryProcess(r, dr, ...).
    The reference's own test point (tests/test_size.py: r = 15, dr = 5) and a 24-draw sweep, batched:
    mean_ylm, cov_ylm and lnlike in all four modes against the unmodified reference at 1e-8."""
    g = golden("size_dr.npz")
    hp = {k: g[k] for k in ("r", "dr", "mu", "sigma", "c", "n")}
    gp = spb.StarryProcess(**hp)
    mean = gp.mean_ylm.cpu().numpy()
    cov = gp.cov_ylm.cpu().numpy()
    # (the profile average goes through exp / log, whose last bit differs between CUDA and glibc; the
    # ill-conditioned Legendre fit Bp amplifies that to ~1e-11 of the mean)
    assert np.abs(mean - g["mean_ylm"]).max() <= 1e-10 * np.abs(g["mean_ylm"]).max()
    # elementwise cov_ylm parity is bounded by the reference's own noise modes at high degree, as for
    # the delta prior (tests/test_gpu_parity.py::test_ylm_moments: 2e-7 absolute); the degrees l <= 9
    # that carry the flux signal hold 1e-7 of the largest entry over the 24 draws
    dg = np.diagonal(cov, axis1=1, axis2=2)
    cmax = np.abs(g["cov_ylm_diag"]).max(axis=1)[:, None]
    assert np.abs(dg - g["cov_ylm_diag"]).max() <= 5e-7
    assert (np.abs(dg[:, :100] - g["cov_ylm_diag"][:, :100]) / cmax).max() <= 1e-7
    assert (np.abs(cov[:, 6, :100] - g["cov_ylm_row6"][:, :100]) / cmax).max() <= 1e-7
    assert np.abs(cov - cov.transpose(0, 2, 1)).max() == 0.0
    assert int(gp.info.abs().sum().item()) == 0
    worst = {}
    for marg in (False, True):
        for norm in (False, True):
            gpm = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **hp)
            f = g["flux_norm"] if norm else g["flux"]
            ll = gpm.log_likelihood(g["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
            ref = g["lnlike_m%d_n%d" % (marg, norm)]
            assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
            fin = np.isfinite(ref)
            worst[(marg, norm)] = float(rel(ll[fin], ref[fin]).max())
    print("uniform-dr prior: max rel lnlike err per (marg, norm):", worst)
    assert max(worst.values()) <= RTOL, worst
    # scalar call == the reference's own calling convention, and batched == one at a time
    g0 = spb.StarryProcess(r=15.0, dr=5.0, mu=30.0, sigma=5.0, c=0.1, n=10.0)
    assert np.array_equal(g0.cov_ylm.cpu().numpy(), cov[0])
    ll0 = g0.log_likelihood(g["t"], g["flux_norm"], 1e-6, i=60.0, p=1.0, u=U_LD).item()
    assert rel(ll0, g["lnlike_m1_n1"][0]) <= RTOL
    # dr -> 0 tends to the delta prior; bounds as CheckBoundsOp (size.py:120)
    gd = spb.StarryProcess(r=15.0, mu=30.0, sigma=5.0, c=0.1, n=10.0)
    gs = spb.StarryProcess(r=15.0, dr=0.01, mu=30.0, sigma=5.0, c=0.1, n=10.0)
    scale = float(gd.cov_ylm.abs().max())
    assert float((gd.cov_ylm - gs.cov_ylm).abs().max()) <= 1e-4 * scale
    with pytest.raises(ValueError):
        spb.StarryProcess(r=15.0, dr=95.0)
    bad = spb.StarryProcess(r=15.0, dr=torch.tensor([5.0, 120.0], dtype=torch.float64, device="cuda"),
                            mu=30.0, sigma=5.0, c=0.1, n=10.0)
    ll = bad.log_likelihood(g["t"][:50], np.zeros(50), 1e-6)
    assert np.isfinite(ll[0].item()) and np.isneginf(ll[1].item()) and int(bad.info[1].item()) & 4


# ------------------------------------------------------------------------- gradient (8(f) rank 4)
# The reference accepts its own gradient at 1e-4 (theano.gradient.verify_grad defaults for float64,
# tests/test_lnlike.py:105-136).  Two statements are tested here:
#   (1) the CUDA gradient IS the derivative of the CUDA forward function: <= 1e-4 relative against
#       plain central differences of log_likelihood in the hyperparameters (measured 5e-6..4e-5: that
#       is the noise floor of the DIFFERENCES -- eigenvalue-clip modes enter and leave between the
#       two displaced evaluations -- which the tangent-wise scheme of the product avoids);
#   (2) it agrees with the analytic, clip-free gradient oracle to <= 3e-4: the two forward
#       functions agree to ~1e-9 |lnlike| (the reference's eigenvalue-clip floor, different modes
#       are dropped in the 256- and the 31-dimensional eigen-problems), which pins slopes only to
#       1e-9 |lnlike| / (|g| x correlation length) ~ 1e-4.
GRAD_RTOL_SELF = 1e-4
GRAD_RTOL_ORACLE = 3e-4


@pytest.mark.parametrize("marg", [False, True])
@pytest.mark.parametrize("norm", [False, True])
def test_lnlike_gradient_against_analytic_oracle(spb, oracle, marg, norm):
    """``log_likelihood(..., return_grad=True)``: d lnlike / d (r, a, b, c, n) per batch element against
    the analytic gradient oracle (oracle/sp_oracle_grad.py, itself pinned to finite differences of
    the unmodified reference at the reference's own verify_grad tolerance, tests/test_oracle_grad.py)
    and against central differences of the CUDA forward."""
    from oracle import sp_oracle_grad as sg

    rng = np.random.default_rng(42)
    t = np.linspace(0, 3, 100)
    flux = 1e-3 * rng.standard_normal(100)
    hps = [dict(r=20.0, a=0.40, b=0.27, c=0.1, n=10.0),
           dict(r=12.0, a=0.55, b=0.12, c=0.05, n=4.0),
           dict(r=27.0, a=0.25, b=0.45, c=0.12, n=2.0)]
    batch = {k: np.array([h[k] for h in hps]) for k in hps[0]}
    gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **batch)
    ll, g = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, return_grad=True)
    ll0 = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD)
    assert torch.equal(ll, ll0)            # the base variant is the plain evaluation, bit for bit
    # (1) derivative of the CUDA forward: plain central differences, relative step 1e-3
    worst_self = 0.0
    for p_ in sg.PARAMS:
        d = 1e-3 * batch[p_]
        up, dn = dict(batch), dict(batch)
        up[p_] = batch[p_] + d
        dn[p_] = batch[p_] - d
        lu = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **up).log_likelihood(
            t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
        ld = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **dn).log_likelihood(
            t, flux, 1e-6, i=60.0, p=1.0, u=U_LD).cpu().numpy()
        fd = (lu - ld) / (2 * d)
        gg = g[p_].cpu().numpy()
        scale = np.maximum(np.abs(fd), 1e-3 * np.max([np.abs(g[q].cpu().numpy()) for q in sg.PARAMS], axis=0))
        err = np.abs(gg - fd) / scale
        worst_self = max(worst_self, err.max())
        assert err.max() <= GRAD_RTOL_SELF, (p_, gg, fd)
    # (2) the analytic oracle
    worst = 0.0
    for k, hp in enumerate(hps):
        llo, go = sg.lnlike_and_grad(hp, t, flux, 1e-6, i=60.0, p=1.0, u=U_LD,
                                     marginalize_over_inclination=marg, normalized=norm)
        assert rel(ll[k].item(), llo) <= 1e-8
        errs = {}
        for p_ in sg.PARAMS:
            errs[p_] = abs(g[p_][k].item() - go[p_]) / max(
                abs(go[p_]), 1e-3 * max(abs(v) for v in go.values()))
            worst = max(worst, errs[p_])
        assert max(errs.values()) <= GRAD_RTOL_ORACLE, (k, errs, {a: g[a][k].item() for a in g}, go)
    print("gradient marg=%d norm=%d: max rel err %.1e vs central differences of the CUDA forward, "
          "%.1e vs the analytic oracle" % (marg, norm, worst_self, worst))


def test_lnlike_gradient_mu_sigma_and_flags(spb, oracle):
    """Chain rule through gauss2beta (latitude.py:14-77) when the process is built from (mu, sigma);
    scalar processes return scalars; -inf elements return a zero gradient; the uniform-dr prior and
    time-variable processes raise."""
    rng = np.random.default_rng(1)
    t = np.linspace(0, 2, 80)
    flux = 1e-3 * rng.standard_normal(80)
    gp = spb.StarryProcess(r=15.0, mu=35.0, sigma=8.0, c=0.08, n=5.0)
    ll, g = gp.log_likelihood(t, flux, 1e-6, u=U_LD, return_grad=True)
    assert ll.ndim == 0 and set(g) == {"r", "mu", "sigma", "c", "n"}
    for key, h in (("mu", 1e-3), ("sigma", 1e-3), ("r", 1e-3), ("c", 1e-6), ("n", 1e-4)):
        hp = dict(r=15.0, mu=35.0, sigma=8.0, c=0.08, n=5.0)
        up, dn = dict(hp), dict(hp)
        up[key] += h
        dn[key] -= h
        fd = (oracle.OracleProcess(**up).log_likelihood(t, flux, 1e-6, u=U_LD)
              - oracle.OracleProcess(**dn).log_likelihood(t, flux, 1e-6, u=U_LD)) / (2 * h)
        assert abs(g[key].item() - fd) <= 1e-4 * max(abs(fd), 1.0), (key, g[key].item(), fd)
    # an element outside the validity range of the normalised process: lnlike = -inf, gradient 0
    gb = spb.StarryProcess(r=np.array([15.0, 10.107390922311073]), mu=np.array([35.0, 51.978254148197465]), sigma=np.array([8.0, 11.733947364331115]),
                           c=np.array([0.08, 0.5845712920357633]), n=np.array([5.0, 41.4605890605386]))
    ll, g = gb.log_likelihood(t, flux, 1e-6, u=U_LD, return_grad=True)
    assert np.isfinite(ll[0].item()) and np.isneginf(ll[1].item())
    assert all(float(v[1]) == 0.0 and np.isfinite(float(v[0])) for v in g.values())
    with pytest.raises(NotImplementedError):
        spb.StarryProcess(r=15.0, dr=5.0).log_likelihood(t, flux, 1e-6, return_grad=True)
    with pytest.raises(NotImplementedError):
        spb.StarryProcess(r=15.0, tau=1.0).log_likelihood(t, flux, 1e-6, return_grad=True)


# ------------------------------------------------------------------------- ydeg < 15, keyword options
@pytest.mark.parametrize("case", ["y5", "y10", "y15opt"])
def test_lower_degree_and_keyword_options_against_reference_golden(spb, golden, case):
    """VERDICT r1 missing #5: spherical-harmonic degrees below 15 (the reference bakes ydeg in at JIT
    time, ops/base_op.py:85-86, and its quadrature tests run ydeg = 3 / 5) and the keyword options
    epsy, epsy15, abmin, log_alpha_max, log_beta_max (sp.py:241-262), against the unmodified
    reference (oracle/gen_golden_lowdeg.py).  Lower degrees are embedded in the degree-15 kernels with
    the spot operator of that degree; the leading (ydeg+1)^2 block is compared."""
    g = golden("lowdeg_options.npz")
    kw = {"y5": dict(ydeg=5), "y10": dict(ydeg=10),
          "y15opt": dict(ydeg=15, epsy=1e-10, epsy15=1e-8, abmin=1e-3, log_alpha_max=8.0,
                         log_beta_max=9.0)}[case]
    ny = (kw["ydeg"] + 1) ** 2
    hp = {k: g[k] for k in ("r", "a", "b", "c", "n")}
    gp = spb.StarryProcess(**hp, **kw)
    mean, cov = gp.mean_ylm.cpu().numpy(), gp.cov_ylm.cpu().numpy()
    assert mean.shape == (4, ny) and cov.shape == (4, ny, ny) and gp.ydeg == kw["ydeg"]
    assert np.abs(mean - g[case + "_mean"]).max() <= 1e-12 * np.abs(g[case + "_mean"]).max()
    if case == "y15opt":
        dg = np.diagonal(cov, axis1=1, axis2=2)
        assert np.abs(dg - g["y15opt_cov_diag"])[:, :100].max() <= 1e-7 * np.abs(g["y15opt_cov_diag"]).max()
    else:
        low = min(ny, 100)
        assert np.abs(cov - g[case + "_cov"])[:, :low, :low].max() <= 1e-7 * np.abs(g[case + "_cov"]).max()
    A = gp.design_matrix(g["t"][:7], i=55.0, p=0.8, u=U_LD).cpu().numpy()
    assert A.shape == (7, ny) and np.abs(A - g[case + "_A"]).max() <= 2e-11
    worst = {}
    for marg in (False, True):
        for norm in (False, True):
            gpm = spb.StarryProcess(marginalize_over_inclination=marg, normalized=norm, **hp, **kw)
            f = g["flux_norm"] if norm else g["flux"]
            ll = gpm.log_likelihood(g["t"], f, 1e-6, i=55.0, p=0.8, u=U_LD).cpu().numpy()
            worst[(marg, norm)] = float(rel(ll, g["%s_lnlike_m%d_n%d" % (case, marg, norm)]).max())
    print("%s: max rel lnlike err per (marg, norm): %s" % (case, worst))
    assert max(worst.values()) <= RTOL, worst
    # prior draws live in the (ydeg+1)^2 space
    ys = gp.sample_ylm(nsamples=3, generator=torch.Generator(device="cuda").manual_seed(0))
    assert tuple(ys.shape) == (4, 3, ny)
    assert tuple(gp.cho_cov_ylm.shape) == (4, ny, ny)
    F = spb.StarryProcess(r=15.0, a=0.4, b=0.3, c=0.1, n=5.0, normalized=False, **kw)
    fl = F.flux(F.sample_ylm(nsamples=2), g["t"][:9], i=55.0, p=0.8, u=U_LD)
    assert tuple(fl.shape) == (2, 9)
    with pytest.raises(AssertionError):
        spb.StarryProcess(ydeg=4)
    with pytest.raises(NotImplementedError):
        spb.StarryProcess(ydeg=16)
