"""CPU: a NumPy restatement of the rank-31 conditional log-likelihood (DESIGN.md section 4.6), built on
the oracle's OracleProcess, against the values the unmodified reference produced and against the
oracle's own dense evaluation.  tests/test_gpu_lowrank.py uses the same restatement at nt = 1e5."""
import numpy as np
import pytest

from conftest import FID, U_LD


def phase_basis(theta):
    """Phi (nt, 31) = [1, cos(m theta) (m = 1..15), sin(m theta) (m = 1..15)]: every row of the design
    matrix is Phi(theta) B_inc (the z-rotation is band-limited to |m| <= 15)."""
    m = np.arange(1, 16)
    return np.hstack([np.ones((theta.size, 1)), np.cos(np.outer(theta, m)), np.sin(np.outer(theta, m))])


def inclination_basis(o, i=60.0, u=(0.0, 0.0)):
    """B_inc (31, N) from the oracle's own design matrix at 31 equally spaced phases (a DFT solve),
    independent of how the library builds it."""
    tj = np.arange(31) / 31.0
    return np.linalg.solve(phase_basis(2 * np.pi * tj), o.design_matrix(tj, i, 1.0, u))


def log_likelihood_lowrank(o, t, flux, data_cov, i=60.0, p=1.0, u=(0.0, 0.0), baseline_mean=0.0,
                           baseline_var=0.0):
    """The conditional log-likelihood of ``o.log_likelihood`` through K = Phi C~ Phi^T + D: thin QR of the
    whitened phase basis D^-1/2 Phi = Q R, N = I + R C~ R^T, logdet K = sum log D + logdet N,
    r^T K^-1 r = |y - Q w|^2 + w^T N^-1 w with y = D^-1/2 r, w = Q^T y.  Sets ``o.z`` as the dense path
    does."""
    from oracle.sp_oracle import alpha_beta_series, check_bounds

    if o.marg or o.tau is not None:
        raise ValueError("the rank-31 form covers the static conditional branch only")
    t = np.asarray(t, dtype=float).reshape(-1)
    nt = t.size
    p = float(check_bounds("p", p, 0, np.inf))
    Bm = inclination_basis(o, i, u)
    Phi = phase_basis(2 * np.pi * np.mod(t / p, 1.0))
    C = Bm @ o.cov_ylm @ Bm.T
    gp_mean = float(Phi[0] @ (Bm @ o.mean_ylm))          # (A mean_ylm)[0]
    if o.normalized:
        s = Phi.sum(axis=0)
        m = s @ C @ s / nt ** 2                         # mean(A Sigma A^T)
        mu = 1.0 + gp_mean
        o.z = m / mu ** 2
        alpha, beta = alpha_beta_series(o.z, o.normN)
        qh = C @ s / (nt * m)                           # q = Phi qh
        ph = -qh
        ph[0] += 1.0                                    # 1 - q = Phi (e0 - qh)
        C = (alpha / mu ** 2) * C + o.z * ((alpha + beta) * np.outer(ph, ph) - alpha * np.outer(qh, qh))
        gp_mean = 0.0
    bv = np.asarray(baseline_var, dtype=float)
    if bv.ndim != 0:
        raise ValueError("baseline_var must be a scalar in the rank-31 form")
    C[0, 0] += float(bv)                                # 1 1^T = Phi e0 e0^T Phi^T
    D = np.asarray(data_cov, dtype=float)
    if D.ndim > 1:
        raise ValueError("data_cov must be a scalar or a vector in the rank-31 form")
    D = np.broadcast_to(D, (nt,)).astype(float)
    sd = np.sqrt(D)
    Q, R = np.linalg.qr(Phi / sd[:, None])
    Nm = np.eye(31) + R @ C @ R.T
    try:
        L = np.linalg.cholesky(0.5 * (Nm + Nm.T))
    except np.linalg.LinAlgError:
        return -np.inf
    r = np.reshape(np.transpose(np.asarray(flux, dtype=float)), (nt, -1)) - (gp_mean + baseline_mean)
    M = r.shape[1]
    y = r / sd[:, None]
    w = Q.T @ y
    v = np.linalg.solve(L, w)
    quad = np.sum((y - Q @ w) ** 2) + np.sum(v ** 2)
    logdet = np.sum(np.log(D)) + 2.0 * np.sum(np.log(np.diag(L)))
    lnlike = -0.5 * quad - 0.5 * M * logdet - 0.5 * nt * M * np.log(2 * np.pi)
    if (o.normalized and o.z > o.normzmax) or np.isnan(lnlike):
        return -np.inf
    return float(lnlike)


def rel(a, b):
    return abs(a - b) / abs(b)


def check_draws(ll, ref, tol):
    ll, ref = np.asarray(ll), np.asarray(ref)
    assert np.array_equal(np.isneginf(ll), np.isneginf(ref))
    fin = np.isfinite(ref)
    assert np.all(np.abs(ll[fin] - ref[fin]) <= tol * np.abs(ref[fin]))


@pytest.mark.parametrize("u", [[0.0, 0.0], U_LD])
def test_phase_basis_times_inclination_basis_is_the_design_matrix(oracle, u):
    o = oracle.OracleProcess(marginalize_over_inclination=False, **FID)
    t = np.random.default_rng(3).uniform(-2.0, 7.0, 200)
    for inc in (0.0, 22.5, 60.0, 90.0):
        A = o.design_matrix(t, inc, 1.3, u)
        Bm = inclination_basis(o, inc, u)
        A2 = phase_basis(2 * np.pi * np.mod(t / 1.3, 1.0)) @ Bm
        assert np.abs(A2 - A).max() <= 1e-14 * np.abs(A).max()


@pytest.mark.parametrize("norm", [False, True])
def test_fiducial_conditional(oracle, golden, norm):
    g = golden("fiducial_nt1000.npz")
    t = g["t"]
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=norm, **FID)
    f = g["flux_norm"] if norm else g["flux"]
    fe = g["flux_ens_norm"] if norm else g["flux_ens"]
    for uname, u in (("u0", [0.0, 0.0]), ("uld", U_LD)):
        key = "m0_n%d_%s" % (norm, uname)
        ll = log_likelihood_lowrank(o, t, f, 1e-6, i=60.0, p=1.0, u=u)
        assert rel(ll, g["lnlike_" + key]) <= 1e-12
        if norm:
            assert rel(o.z, g["z_" + key]) <= 1e-12
        lle = log_likelihood_lowrank(o, t, fe, 1e-6, i=60.0, p=1.0, u=u)
        assert rel(lle, g["lnlike_ens_" + key]) <= 1e-12
    ll = log_likelihood_lowrank(o, t, f, g["data_cov_vec"], i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4,
                                  baseline_var=1e-5)
    assert rel(ll, g["lnlike_dvec_m0_n%d" % norm]) <= 1e-12


@pytest.mark.parametrize("name", ["sweep_nt1000.npz", "sweep_lowc_nt1000.npz"])
@pytest.mark.parametrize("norm", [False, True])
def test_sweeps(oracle, golden, name, norm):
    g = golden(name)
    fid = golden("fiducial_nt1000.npz")
    f = fid["flux_norm"] if norm else fid["flux"]
    ll = []
    for s in range(len(g["r"])):
        o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=norm, r=g["r"][s],
                                 mu=g["mu"][s], sigma=g["sigma"][s], c=g["c"][s], n=g["n"][s])
        ll.append(log_likelihood_lowrank(o, fid["t"], f, 1e-6, i=60.0, p=1.0, u=U_LD))
    check_draws(ll, g["lnlike_m0_n%d" % norm], 1e-9)


def test_long_baseline(oracle, golden):
    lb = golden("longbaseline_nt4096.npz")
    ll = []
    for s in range(len(lb["r"])):
        o = oracle.OracleProcess(r=lb["r"][s], mu=lb["mu"][s], sigma=lb["sigma"][s], c=lb["c"][s],
                                 n=lb["n"][s], marginalize_over_inclination=False, normalized=False)
        ll.append(log_likelihood_lowrank(o, lb["t"], lb["flux"], 1e-6, i=60.0, p=1.0, u=lb["u"]))
    check_draws(ll, lb["lnlike"], 1e-9)


def test_long_baseline_r2(oracle, golden):
    """Per-draw baseline variance, both normalisations, the non-PD and the z > zmax draws."""
    lb = golden("longbaseline_nt4096.npz")
    r2 = golden("longbaseline_nt4096_r2.npz")
    t, f = lb["t"], lb["flux"]
    fn = (1 + f) / np.mean(1 + f) - 1
    ll0, ll1, z1 = [], [], []
    for s in range(len(r2["r"])):
        hp = {k: float(r2[k][s]) for k in ("r", "mu", "sigma", "c", "n")}
        o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **hp)
        ll0.append(log_likelihood_lowrank(o, t, f, 1e-6, i=60.0, p=1.0, u=U_LD,
                                            baseline_var=float(r2["baseline_var"][s])))
        o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=True, **hp)
        ll1.append(log_likelihood_lowrank(o, t, fn, 1e-6, i=60.0, p=1.0, u=U_LD))
        z1.append(o.z)
    check_draws(ll0, r2["lnlike_n0"], 1e-9)
    check_draws(ll1, r2["lnlike_n1"], 1e-9)
    assert np.all(np.abs(np.array(z1) - r2["z_n1"]) <= 1e-9 * np.abs(r2["z_n1"]))


def test_calibrate_conditional(oracle, golden):
    """calibrate/log_prob.py conditional: free baseline mean / variance / inclination, and the
    inclination grid with baseline_var = 1 (cond(K) = 2.5e8)."""
    g = golden("calibrate_log_prob.npz")
    t, fl = g["t"], g["flux"]

    def lp(s, flux, inc, m, v, u):
        o = oracle.OracleProcess(r=g["r"][s], a=g["a"][s], b=g["b"][s], c=g["c"][s], n=g["n"][s],
                                 marginalize_over_inclination=False, normalized=True,
                                 normalization_zmax=np.inf, covpts=len(t) - 1)
        return log_likelihood_lowrank(o, t, flux, 1e-6, i=inc, p=1.0, u=u, baseline_mean=m,
                                        baseline_var=10.0 ** v) + o.log_jac()

    for s in range(len(g["r"])):
        assert rel(lp(s, fl[:1], g["inc_cond"][s], g["m"][s], g["v"][s], U_LD), g["log_prob_cond"][s]) <= 1e-8
    for l in range(2):
        for s in range(2):
            for k, inc in enumerate(g["inc_grid"]):
                assert rel(lp(s, fl[l:l + 1], inc, 0.0, 0.0, [0.0, 0.0]), g["lp_grid"][l, s, k]) <= 1e-8


@pytest.mark.parametrize("norm", [False, True])
def test_against_dense_oracle_degenerate_time_stamps(oracle, norm):
    """Light curves covering a tenth of a period (Phi nearly rank-deficient), integer time stamps (one
    phase: Phi of rank one) and random time stamps, with per-point noise and a baseline variance."""
    rng = np.random.default_rng(7)
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=norm,
                             r=18.0, mu=40.0, sigma=9.0, c=0.05, n=4.0)
    for t in (np.linspace(0.0, 0.1, 300), np.arange(120.0), np.sort(rng.uniform(0, 5, 257))):
        f = 1e-3 * rng.standard_normal((2, t.size))
        dc = 1e-6 * (1 + rng.uniform(size=t.size))
        for bv in (0.0, 1e-5):
            ll = log_likelihood_lowrank(o, t, f, dc, i=35.0, p=1.0, u=U_LD, baseline_mean=2e-4,
                                          baseline_var=bv)
            ref = o.log_likelihood(t, f, dc, i=35.0, p=1.0, u=U_LD, baseline_mean=2e-4, baseline_var=bv)
            assert rel(ll, ref) <= 1e-12


def test_rejects_what_it_does_not_cover(oracle):
    t = np.linspace(0, 1, 50)
    with pytest.raises(ValueError):
        log_likelihood_lowrank(oracle.OracleProcess(marginalize_over_inclination=True, **FID), t, t, 1e-6)
    o = oracle.OracleProcess(marginalize_over_inclination=False, **FID)
    with pytest.raises(ValueError):
        log_likelihood_lowrank(o, t, t, 1e-6 * np.eye(50))
    with pytest.raises(ValueError):
        log_likelihood_lowrank(o, t, t, 1e-6, baseline_var=np.eye(50))
