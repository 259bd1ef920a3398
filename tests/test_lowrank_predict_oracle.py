"""CPU: a NumPy restatement of the rank-31 predictive distribution (``predict`` / ``sample_conditional`` with
``method="lowrank"``, DESIGN.md section 4.6), built on the oracle's OracleProcess and the phase / inclination
bases of tests/test_lowrank_oracle.py, against the values the unmodified reference produced and against the
oracle's own dense evaluation.  tests/test_gpu_lowrank_predict.py uses the same restatement at nt = 1e5."""
import numpy as np
import pytest

from conftest import FID, U_LD
from test_lowrank_oracle import inclination_basis, phase_basis

KW = dict(i=60.0, p=1.0, u=U_LD)
KWB = dict(i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4, baseline_var=1e-5)


def posterior_lowrank(o, t, flux, data_cov, i=60.0, p=1.0, u=(0.0, 0.0), baseline_mean=0.0, baseline_var=0.0):
    """(a, P, gp_mean) of the predictive distribution in the phase basis: with D^-1/2 Phi = Q R,
    N = I + R C~ R^T, w = Q^T D^-1/2 (flux - baseline_mean - gp_mean):  a = C~ R^T N^-1 w,  P = C~ - V^T V,
    V = L_N^-1 R C~.  Then mean(ts) = gp_mean + Phi(ts) a and cov(ts, ts) = Phi(ts) P Phi(ts)^T."""
    from oracle.sp_oracle import check_bounds

    if o.normalized:
        raise NotImplementedError("Method not implemented when the flux is normalized.")
    if o.marg or o.tau is not None:
        raise ValueError("the rank-31 form covers the static conditional branch only")
    t = np.asarray(t, dtype=float).reshape(-1)
    nt = t.size
    p = float(check_bounds("p", p, 0, np.inf))
    Bm = inclination_basis(o, i, u)
    Phi = phase_basis(2 * np.pi * np.mod(t / p, 1.0))
    C = Bm @ o.cov_ylm @ Bm.T
    gp_mean = float(phase_basis(np.zeros(1))[0] @ (Bm @ o.mean_ylm))   # the mean at t = 0, as the oracle
    bv = np.asarray(baseline_var, dtype=float)
    if bv.ndim != 0:
        raise ValueError("baseline_var must be a scalar in the rank-31 form")
    C[0, 0] += float(bv)                                # 1 1^T = Phi e0 e0^T Phi^T
    D = np.asarray(data_cov, dtype=float)
    if D.ndim > 1:
        raise ValueError("data_cov must be a scalar or a vector in the rank-31 form")
    sd = np.sqrt(np.broadcast_to(D, (nt,)).astype(float))
    Q, R = np.linalg.qr(Phi / sd[:, None])
    L = np.linalg.cholesky(np.eye(31) + R @ C @ R.T)
    w = Q.T @ ((np.asarray(flux, dtype=float).reshape(-1) - baseline_mean - gp_mean) / sd)
    a = C @ R.T @ np.linalg.solve(L.T, np.linalg.solve(L, w))
    V = np.linalg.solve(L, R @ C)
    return a, C - V.T @ V, gp_mean


def predict_lowrank(o, t, flux, data_cov, t_sample=None, p=1.0, return_cov="full", **kw):
    """``o.predict`` through the rank-31 posterior: mean (nts,) and covariance (nts, nts) or variance (nts,)."""
    a, P, gp_mean = posterior_lowrank(o, t, flux, data_cov, p=p, **kw)
    ts = np.asarray(t if t_sample is None else t_sample, dtype=float).reshape(-1)
    Phis = phase_basis(2 * np.pi * np.mod(ts / p, 1.0))
    mu = gp_mean + Phis @ a
    if return_cov == "diag":
        return mu, np.einsum("ij,jk,ik->i", Phis, P, Phis)
    return mu, Phis @ P @ Phis.T


def sqrt_factor(P):
    """G with G G^T = P: eigenvectors scaled by the square roots of the eigenvalues clipped at zero."""
    lam, U = np.linalg.eigh(0.5 * (P + P.T))
    return U * np.sqrt(np.clip(lam, 0.0, None))


def sample_conditional_lowrank(o, t, flux, data_cov, unit_normals, t_sample=None, eps=1e-8, p=1.0, G=None, **kw):
    """Draws (nsamples, nts) = mean + Phi(ts) G z1 + sqrt(eps) z2, ``unit_normals`` (32 + nts, nsamples): 32 rows
    z1 for the basis coefficients (the 32nd multiplies the zero padding of the basis), then nts rows z2."""
    a, P, gp_mean = posterior_lowrank(o, t, flux, data_cov, p=p, **kw)
    G = sqrt_factor(P) if G is None else np.asarray(G)[:31, :31]
    ts = np.asarray(t if t_sample is None else t_sample, dtype=float).reshape(-1)
    Phis = phase_basis(2 * np.pi * np.mod(ts / p, 1.0))
    z = np.asarray(unit_normals, dtype=float)
    out = (gp_mean + Phis @ a)[:, None] + Phis @ (G @ z[:31]) + np.sqrt(eps) * z[32:]
    return out.T


def relmax(a, b):
    return float(np.abs(np.asarray(a) - b).max() / np.abs(b).max())


def test_reference_golden(oracle, golden):
    g = golden("predict_nt200.npz")
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **FID)
    prior_scale = float(np.abs(g["sample_m0"]).max()) ** 2
    mu, K = predict_lowrank(o, g["t"], g["flux"], 1e-6, **KW)
    assert relmax(mu, g["pred_mu_m0"]) <= 1e-10
    assert np.abs(K - g["pred_K_m0"]).max() <= 1e-10 * prior_scale
    mu, K = predict_lowrank(o, g["t"], g["flux"], g["data_cov_vec"], t_sample=g["t_sample"], **KWB)
    assert relmax(mu, g["pred_ts_mu_m0"]) <= 1e-10
    assert np.abs(K - g["pred_ts_K_m0"]).max() <= 1e-10 * prior_scale
    mu2, var = predict_lowrank(o, g["t"], g["flux"], g["data_cov_vec"], t_sample=g["t_sample"],
                               return_cov="diag", **KWB)
    assert np.array_equal(mu2, mu)
    assert relmax(var, np.diag(K)) <= 1e-13


def test_against_dense_oracle_degenerate_time_stamps(oracle):
    """A tenth of a period (Phi nearly rank-deficient), integer time stamps (one phase: Phi of rank one) and
    random time stamps, with per-point noise and a baseline variance; output points inside the data and
    extrapolated."""
    rng = np.random.default_rng(11)
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False,
                             r=18.0, mu=40.0, sigma=9.0, c=0.05, n=4.0)
    ts = np.concatenate([np.linspace(0.0, 0.1, 20), rng.uniform(-3.0, 9.0, 40)])
    scale = float(np.abs(o.cov(ts, i=35.0, p=1.0, u=U_LD)).max())
    for t in (np.linspace(0.0, 0.1, 300), np.arange(120.0), np.sort(rng.uniform(0, 5, 257))):
        f = 1e-3 * rng.standard_normal(t.size)
        dc = 1e-6 * (1 + rng.uniform(size=t.size))
        for bv in (0.0, 1e-5):
            kw = dict(i=35.0, p=1.0, u=U_LD, baseline_mean=2e-4, baseline_var=bv)
            mu, K = predict_lowrank(o, t, f, dc, t_sample=ts, **kw)
            mo, Ko = o.predict(t, f, dc, t_sample=ts, **kw)
            assert relmax(mu, mo) <= 1e-10
            assert np.abs(K - Ko).max() <= 1e-10 * scale


def test_draws_have_the_predictive_distribution(oracle, golden):
    """G G^T = P, and 20 000 draws at nts = 24 have the predictive mean and covariance (+ eps) within Monte
    Carlo error."""
    g = golden("predict_nt200.npz")
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **FID)
    ts = np.linspace(-0.3, 1.4, 24)
    a, P, _ = posterior_lowrank(o, g["t"], g["flux"], g["data_cov_vec"], **KWB)
    G = sqrt_factor(P)
    assert np.abs(G @ G.T - P).max() <= 1e-12 * np.abs(P).max()
    mu, K = predict_lowrank(o, g["t"], g["flux"], g["data_cov_vec"], t_sample=ts, **KWB)
    n, eps = 20000, 1e-8
    z = np.random.default_rng(4).standard_normal((32 + ts.size, n))
    x = sample_conditional_lowrank(o, g["t"], g["flux"], g["data_cov_vec"], z, t_sample=ts, eps=eps, **KWB)
    assert x.shape == (n, ts.size)
    Kx = K + eps * np.eye(ts.size)
    sd = np.sqrt(np.diag(Kx))
    assert np.all(np.abs(x.mean(axis=0) - mu) <= 5 * sd / np.sqrt(n))
    # sample covariance: entry (i, j) has standard error sqrt((K_ii K_jj + K_ij^2) / n)
    se = np.sqrt((np.outer(np.diag(Kx), np.diag(Kx)) + Kx ** 2) / n)
    assert np.all(np.abs(np.cov(x, rowvar=False) - Kx) <= 6 * se)


def test_rejects_what_it_does_not_cover(oracle):
    t = np.linspace(0, 1, 50)
    with pytest.raises(ValueError):
        predict_lowrank(oracle.OracleProcess(marginalize_over_inclination=True, normalized=False, **FID), t, t, 1e-6)
    with pytest.raises(NotImplementedError):
        predict_lowrank(oracle.OracleProcess(marginalize_over_inclination=False, normalized=True, **FID), t, t, 1e-6)
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **FID)
    with pytest.raises(ValueError):
        predict_lowrank(o, t, t, 1e-6 * np.eye(50))
    with pytest.raises(ValueError):
        predict_lowrank(o, t, t, 1e-6, baseline_var=np.eye(50))
