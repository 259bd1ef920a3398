"""GPU (-m gpu): ``log_likelihood(method="lowrank")`` -- the rank-31 conditional branch (DESIGN.md
section 4.6) -- against the values the unmodified reference produced (1e-8 relative, identical -inf
pattern and SPB_INFO_Z_RANGE), against the dense CUDA path on the same moments, against the oracle's
rank-31 restatement at nt = 1e5, and for determinism, batch invariance, gradients and errors."""
import numpy as np
import pytest

from conftest import FID, U_LD

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RTOL = 1e-8
DENSE_RTOL = 1e-10
SWEEP_DENSE_FLOOR = 3e-10
SEC = dict(r=20.0, mu=60.0, sigma=10.0, c=0.05, n=5.0)


@pytest.fixture(scope="module")
def spb():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)) / np.abs(np.asarray(b))


def both(gp, *args, **kw):
    """(lowrank lnlike, its info) and (dense lnlike, its info) on the same process object."""
    lr = gp.log_likelihood(*args, method="lowrank", **kw)
    ilr = gp.info.clone()
    de = gp.log_likelihood(*args, **kw)
    return (np.atleast_1d(lr.cpu().numpy()), np.atleast_1d(ilr.cpu().numpy()),
            np.atleast_1d(de.cpu().numpy()), np.atleast_1d(gp.info.cpu().numpy()))


def check(ll, ref, tol, info=None, info_ref=None):
    ll, ref = np.atleast_1d(ll), np.atleast_1d(ref)
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    fin = np.isfinite(ref)
    err = rel(ll[fin], ref[fin]).max() if fin.any() else 0.0
    assert err <= tol, err
    if info is not None:
        assert np.array_equal(info & 2, info_ref & 2)   # SPB_INFO_Z_RANGE
    return err


# ------------------------------------------------------------------ reference goldens
@pytest.mark.parametrize("norm", [False, True])
def test_fiducial_conditional_keys(spb, golden, norm):
    g = golden("fiducial_nt1000.npz")
    t = g["t"]
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm, **FID)
    f = g["flux_norm"] if norm else g["flux"]
    fe = g["flux_ens_norm"] if norm else g["flux_ens"]
    for uname, u in (("u0", [0.0, 0.0]), ("uld", U_LD)):
        key = "m0_n%d_%s" % (norm, uname)
        ll, il, de, idn = both(gp, t, f, 1e-6, i=60.0, p=1.0, u=u)
        check(ll, g["lnlike_" + key], RTOL, il, idn)
        check(ll, de, DENSE_RTOL)
        if norm:
            gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=u, method="lowrank")
            assert rel(gp._z.item(), g["z_" + key]) <= RTOL
        lle = gp.log_likelihood(t, fe, 1e-6, i=60.0, p=1.0, u=u, method="lowrank").item()
        check(lle, g["lnlike_ens_" + key], RTOL)
    ll, il, de, idn = both(gp, t, f, g["data_cov_vec"], i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4,
                           baseline_var=1e-5)
    check(ll, g["lnlike_dvec_m0_n%d" % norm], RTOL)
    check(ll, de, DENSE_RTOL)


@pytest.mark.parametrize("name", ["sweep_nt1000.npz", "sweep_lowc_nt1000.npz"])
@pytest.mark.parametrize("norm", [False, True])
def test_sweeps(spb, golden, name, norm):
    g = golden(name)
    fid = golden("fiducial_nt1000.npz")
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm,
                           **{k: g[k] for k in ("r", "mu", "sigma", "c", "n")})
    f = fid["flux_norm"] if norm else fid["flux"]
    ll, il, de, idn = both(gp, fid["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD)
    e = check(ll, g["lnlike_m0_n%d" % norm], RTOL, il, idn)
    # Some of these draws are ill-conditioned: there the dense fp64 Cholesky of K rounds at up to 3e-10
    # (the reference's LAPACK evaluation and the oracle's dense restatement of the same K differ by that
    # much, tests/test_oracle_golden.py::test_sweep), and both paths sit 2e-9 from the reference's value
    # (its eigen-solver noise in the moments).  The rank-31 path never forms K, so it cannot be held to the
    # dense one more tightly than two dense evaluations agree with each other.
    d = check(ll, de, SWEEP_DENSE_FLOOR)
    print("%s n%d: max rel err vs reference %.1e, vs the dense path %.1e" % (name, norm, e, d))


def test_bench_sweep(spb, golden):
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, 1234)
    sw = golden("bench_sweep_seed1234.npz")
    ns = len(sw["r"])
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **{k: hp[k][:ns] for k in hp})
    ll, il, de, idn = both(gp, t, flux, 1e-6, i=60.0, p=1.0, u=U_LD)
    e = check(ll, sw["lnlike_m0_n1"], RTOL, il, idn)
    check(ll, de, DENSE_RTOL)
    print("bench sweep m0_n1: max rel err vs reference %.1e" % e)


def test_ensemble(spb, golden):
    import bench

    g = golden("ensemble_nt1000.npz")
    M = int(g["M"])
    for norm in (False, True):
        t, f = bench.ensemble_flux(M, normalized=norm)
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm, **FID)
        ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank").item()
        check(ll, float(g["lnlike_m0_n%d" % norm]), RTOL)
        lld = gp.log_likelihood(t, f, g["data_cov_vec"], i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4,
                                baseline_var=1e-5, method="lowrank").item()
        check(lld, float(g["lnlike_dvec_m0_n%d" % norm]), RTOL)


def test_long_baseline(spb, golden):
    lb = golden("longbaseline_nt4096.npz")
    r2 = golden("longbaseline_nt4096_r2.npz")
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False,
                           **{k: lb[k] for k in ("r", "mu", "sigma", "c", "n")})
    ll, il, de, idn = both(gp, lb["t"], lb["flux"], 1e-6, i=60.0, p=1.0, u=lb["u"])
    check(ll, lb["lnlike"], RTOL)
    check(ll, de, DENSE_RTOL)
    t, f = lb["t"], lb["flux"]
    fn = (1 + f) / np.mean(1 + f) - 1
    hp = {k: r2[k] for k in ("r", "mu", "sigma", "c", "n")}
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hp)
    ll, il, de, idn = both(gp, t, f, 1e-6, i=60.0, p=1.0, u=U_LD, baseline_var=r2["baseline_var"])
    check(ll, r2["lnlike_n0"], RTOL)
    check(ll, de, DENSE_RTOL)
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **hp)
    ll, il, de, idn = both(gp, t, fn, 1e-6, i=60.0, p=1.0, u=U_LD)
    check(ll, r2["lnlike_n1"], RTOL, il, idn)
    check(ll, de, DENSE_RTOL)
    gp.log_likelihood(t, fn, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank")
    assert rel(gp._z.cpu().numpy(), r2["z_n1"]).max() <= RTOL


def test_calibrate_callers(spb, golden):
    from starry_process_b200 import calibrate

    g = golden("calibrate_log_prob.npz")
    t, fl = g["t"], g["flux"]
    T = lambda x: torch.tensor(np.asarray(x), dtype=torch.float64)  # noqa: E731
    lp = {}
    for method in ("lowrank", "dense"):
        f2 = calibrate.get_log_prob(t, flux=None, ferr=1e-3, p=1.0, marginalize_over_inclination=False,
                                    baseline_mean=None, baseline_log_var=None, u=U_LD, method=method)
        cond = f2(fl[:1], T(g["r"]), T(g["a"]), T(g["b"]), T(g["c"]), T(g["n"]), T(g["m"]), T(g["v"]),
                  T(g["inc_cond"])).cpu().numpy()
        grid = calibrate.inclination_log_prob(
            t, fl[:2], np.stack([g["r"][:2], g["a"][:2], g["b"][:2], g["c"][:2], g["n"][:2]], axis=1),
            g["inc_grid"], ferr=1e-3, p=1.0, method=method).cpu().numpy()
        lp[method] = (cond, grid)
    e1 = check(lp["lowrank"][0], g["log_prob_cond"], RTOL)
    check(lp["lowrank"][0], lp["dense"][0], DENSE_RTOL)
    # The grid keeps the reference default baseline_log_var = 0: + 1.0 on a covariance whose other
    # eigenvalues are ~1e-6, cond(K) = 2.5e8.  The GPU moments differ from the reference's in the last bits
    # and that condition number turns it into ~3e-8 of lnlike for either method, which is why the dense
    # path's own test allows 1e-7 here (tests/test_gpu_parity.py::test_calibrate_callers).  Both methods
    # start from the same moments, so they agree to 1e-8.
    e2 = check(lp["lowrank"][1].ravel(), g["lp_grid"].ravel(), 1e-7)
    check(lp["lowrank"][1].ravel(), lp["dense"][1].ravel(), 1e-8)
    print("calibrate lowrank: cond %.1e grid %.1e vs reference" % (e1, e2))


def test_size_dr_lowdeg_and_sum(spb, golden):
    g = golden("size_dr.npz")
    hp = {k: g[k] for k in ("r", "dr", "mu", "sigma", "c", "n")}
    for norm in (False, True):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm, **hp)
        f = g["flux_norm"] if norm else g["flux"]
        ll, il, de, idn = both(gp, g["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD)
        check(ll, g["lnlike_m0_n%d" % norm], RTOL, il, idn)
        check(ll, de, DENSE_RTOL)
    g = golden("lowdeg_options.npz")
    for case, kw in (("y5", dict(ydeg=5)), ("y10", dict(ydeg=10))):
        for norm in (False, True):
            gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm,
                                   **{k: g[k] for k in ("r", "a", "b", "c", "n")}, **kw)
            f = g["flux_norm"] if norm else g["flux"]
            ll, il, de, idn = both(gp, g["t"], f, 1e-6, i=55.0, p=0.8, u=U_LD)
            check(ll, g["%s_lnlike_m0_n%d" % (case, norm)], RTOL, il, idn)
            check(ll, de, DENSE_RTOL)
    g = golden("sum_flux_nt300.npz")
    for norm in (False, True):
        kw = dict(marginalize_over_inclination=False, normalized=norm)
        gp = spb.StarryProcess(**kw, **FID) + spb.StarryProcess(**kw, **SEC)
        f = g["flux_norm"] if norm else g["flux"]
        ll, il, de, idn = both(gp, g["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD)
        check(ll, float(g["lnlike_m0_n%d" % norm]), RTOL)
        check(ll, de, DENSE_RTOL)


# ------------------------------------------------------------------ the dense CUDA path
@pytest.mark.parametrize("nt", [31, 32, 100, 1000, 4096])
@pytest.mark.parametrize("M", [1, 3])
def test_against_dense_path(spb, nt, M):
    """Per-element flux, inclinations, baseline mean and baseline variance; per-point noise."""
    import bench

    rng = np.random.default_rng(nt + M)
    hp, _, _, _ = bench.synthetic_inputs(4096, seed=99)
    B = 12
    t = np.sort(rng.uniform(0, 3.7, nt))
    dc = 1e-6 * (1 + rng.uniform(size=nt))
    for norm in (False, True):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm,
                               **{k: hp[k][:B] for k in hp})
        f = 1e-3 * rng.standard_normal((B, M, nt))
        inc = rng.uniform(5, 90, B)
        bm = 1e-4 * rng.standard_normal(B)
        bv = 10.0 ** rng.uniform(-6, -4, B)
        ll, il, de, idn = both(gp, t, f, dc, i=inc, p=1.3, u=U_LD, baseline_mean=bm, baseline_var=bv)
        e = check(ll, de, DENSE_RTOL, il, idn)
        print("nt=%d M=%d norm=%d: max rel err vs dense %.1e" % (nt, M, norm, e))


# ------------------------------------------------------------------ long light curves
def test_nt1e5_against_oracle_and_memory(spb, oracle):
    import bench
    from test_lowrank_oracle import log_likelihood_lowrank

    nt, B = 100_000, 64
    rng = np.random.default_rng(5)
    t = np.linspace(0, 90.0, nt)
    hp, _, _, _ = bench.synthetic_inputs(4096, seed=7)
    f = 1e-3 * rng.standard_normal(nt)
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **{k: hp[k][:B] for k in hp})
    gp.mean_ylm
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    ll = gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank").cpu().numpy()
    peak = torch.cuda.max_memory_allocated() - base
    print("nt=1e5, B=64: peak additional memory %.2f GB (one dense K: %.0f GB)" % (peak / 1e9, nt * nt * 8 / 1e9))
    assert peak < 2e9
    ref = []
    for s in range(0, B, 9):
        o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=True,
                                 **{k: float(hp[k][s]) for k in hp})
        ref.append(log_likelihood_lowrank(o, t, f, 1e-6, i=60.0, p=1.0, u=U_LD))
    check(ll[::9], np.array(ref), 1e-10)


# ------------------------------------------------------------------ determinism / batch invariance
def test_bitwise_deterministic_and_batch_invariant(spb):
    import bench

    hp, t, flux, _ = bench.synthetic_inputs(4096, seed=1234)
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **hp)
    a = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank")
    b = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank")
    assert torch.equal(a, b)
    one = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **{k: hp[k][5:6] for k in hp})
    c = one.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank")
    assert torch.equal(c[0], a[5])


# ------------------------------------------------------------------ gradient
@pytest.mark.parametrize("norm", [False, True])
def test_gradient_against_analytic_oracle(spb, norm):
    from oracle import sp_oracle_grad as sg

    rng = np.random.default_rng(42)
    t = np.linspace(0, 3, 100)
    flux = 1e-3 * rng.standard_normal(100)
    hps = [dict(r=20.0, a=0.40, b=0.27, c=0.1, n=10.0),
           dict(r=12.0, a=0.55, b=0.12, c=0.05, n=4.0),
           dict(r=27.0, a=0.25, b=0.45, c=0.12, n=2.0)]
    batch = {k: np.array([h[k] for h in hps]) for k in hps[0]}
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=norm, **batch)
    ll, g = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, return_grad=True, method="lowrank")
    ll0 = gp.log_likelihood(t, flux, 1e-6, i=60.0, p=1.0, u=U_LD, method="lowrank")
    assert torch.equal(ll, ll0)
    for k, hp in enumerate(hps):
        llo, go = sg.lnlike_and_grad(hp, t, flux, 1e-6, i=60.0, p=1.0, u=U_LD,
                                     marginalize_over_inclination=False, normalized=norm)
        assert rel(ll[k].item(), llo) <= 1e-8
        for p_ in sg.PARAMS:
            err = abs(g[p_][k].item() - go[p_]) / max(abs(go[p_]), 1e-3 * max(abs(v) for v in go.values()))
            assert err <= 3e-4, (k, p_, err)


# ------------------------------------------------------------------ errors
def test_rejected_inputs(spb):
    t = np.linspace(0, 2, 64)
    f = np.zeros(64)
    cond = spb.StarryProcess(marginalize_over_inclination=False, **FID)
    kw = dict(method="lowrank")
    with pytest.raises(ValueError, match="marginalize"):
        spb.StarryProcess(**FID).log_likelihood(t, f, 1e-6, **kw)
    with pytest.raises(ValueError, match="tau"):
        spb.StarryProcess(marginalize_over_inclination=False, tau=0.5, normalized=False,
                          **FID).log_likelihood(t, f, 1e-6, **kw)
    with pytest.raises(ValueError, match="full matrix"):
        cond.log_likelihood(t, f, 1e-6 * np.eye(64), **kw)
    with pytest.raises(ValueError, match="full matrix"):
        cond.log_likelihood(t, f, 1e-6, baseline_var=np.eye(64), **kw)
    with pytest.raises(ValueError, match="positive"):
        cond.log_likelihood(t, f, 0.0, **kw)
    with pytest.raises(ValueError, match="positive"):
        cond.log_likelihood(t, f, np.r_[1e-6 * np.ones(63), -1.0], **kw)
    with pytest.raises(ValueError, match="nt >= 31"):
        cond.log_likelihood(t[:30], f[:30], 1e-6, **kw)
    with pytest.raises(ValueError, match="unknown method"):
        cond.log_likelihood(t, f, 1e-6, method="woodbury")
