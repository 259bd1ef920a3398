"""SURVEY.md section 8(f) rank 2 -- ``sample``, ``predict``, ``sample_conditional``,
``sample_ylm_conditional`` (reference sp.py:518-641, 729-765, 767-1002).

CPU: the oracle restatement against the fixtures produced by the unmodified reference
(oracle/gen_golden_predict.py).  GPU (-m gpu): the CUDA path against the same fixtures, plus the
reference's own ``tests/test_sample.py::test_sample_conditional`` criterion (chi^2 per point < 1).

Tolerances (relative to the largest magnitude of the compared array, fp64 end to end):
  * predicted mean, prior / conditional draws: 1e-8 (the lnlike tolerance of BASELINE.json);
  * predictive covariance: its entries are the O(1e-7) remainder of a cancellation between O(1e-4)
    terms (K(ts,ts) - V V^T), so 1e-8 of the PRIOR scale, which is what the subtraction resolves;
  * sample_ylm_conditional: the reference inverts cov_ylm (cond 1.2e8, lambda_min = 1e-12)
    explicitly (sp.py:267-271).  The pipeline is held to 1e-7 with the reference's own Ylm moments
    as input; end to end (CUDA moments, which differ from the reference's in its noise modes) the
    draws are compared through the flux they imply (A y, 1e-5).
"""
import numpy as np
import pytest

from conftest import FID, U_LD

KW = dict(i=60.0, p=1.0, u=U_LD)
KWB = dict(i=60.0, p=1.0, u=U_LD, baseline_mean=1e-4, baseline_var=1e-5)


def relmax(a, b):
    return float(np.abs(np.asarray(a) - b).max() / np.abs(b).max())


# ------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("marg", [False, True])
def test_oracle_predict_sample_vs_reference(oracle, golden, marg):
    g = golden("predict_nt200.npz")
    tag = "m%d" % marg
    o = oracle.OracleProcess(marginalize_over_inclination=marg, normalized=False, **FID)
    s = o.sample(g["t"], g["sample_U_" + tag], eps=1e-8, **KW)
    assert relmax(s, g["sample_" + tag]) <= 1e-10
    mu, K = o.predict(g["t"], g["flux"], 1e-6, **KW)
    assert relmax(mu, g["pred_mu_" + tag]) <= 1e-12
    assert relmax(K, g["pred_K_" + tag]) <= 1e-10
    mu, K = o.predict(g["t"], g["flux"], g["data_cov_vec"], t_sample=g["t_sample"], **KWB)
    assert relmax(mu, g["pred_ts_mu_" + tag]) <= 1e-12
    assert relmax(K, g["pred_ts_K_" + tag]) <= 1e-10
    sc = o.sample_conditional(g["t"], g["flux"], g["data_cov_vec"], g["cond_U_" + tag],
                              t_sample=g["t_sample"], **KWB)
    assert relmax(sc, g["cond_sample_" + tag]) <= 1e-10


def test_oracle_sample_ylm_conditional_vs_reference(oracle, golden):
    g = golden("predict_nt200.npz")
    o = oracle.OracleProcess(marginalize_over_inclination=False, normalized=False, **FID)
    y = o.sample_ylm_conditional(g["t"], g["flux"], 1e-6, g["ylmc_U"], **KWB)
    assert relmax(y, g["ylmc_y"]) <= 1e-8


def test_oracle_normalized_raises(oracle, golden):
    g = golden("predict_nt200.npz")
    o = oracle.OracleProcess(normalized=True, **FID)
    with pytest.raises(NotImplementedError):
        o.predict(g["t"], g["flux"], 1e-6)


# ------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def spb():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as m

    return m


@pytest.mark.gpu
@pytest.mark.parametrize("marg", [False, True])
def test_gpu_sample_predict_vs_reference_golden(spb, golden, marg):
    g = golden("predict_nt200.npz")
    tag = "m%d" % marg
    gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=False, **FID)
    s = gp.sample(g["t"], nsamples=3, eps=1e-8, unit_normals=g["sample_U_" + tag], **KW)
    assert tuple(s.shape) == (3, 200)
    assert relmax(s.cpu().numpy(), g["sample_" + tag]) <= 1e-8
    mu, K = gp.predict(g["t"], g["flux"], 1e-6, **KW)
    prior_scale = float(np.abs(g["sample_" + tag]).max()) ** 2
    assert relmax(mu.cpu().numpy(), g["pred_mu_" + tag]) <= 1e-8
    assert np.abs(K.cpu().numpy() - g["pred_K_" + tag]).max() <= 1e-8 * prior_scale
    mu, K = gp.predict(g["t"], g["flux"], g["data_cov_vec"], t_sample=g["t_sample"], **KWB)
    assert tuple(mu.shape) == (120,) and tuple(K.shape) == (120, 120)
    assert relmax(mu.cpu().numpy(), g["pred_ts_mu_" + tag]) <= 1e-8
    assert np.abs(K.cpu().numpy() - g["pred_ts_K_" + tag]).max() <= 1e-8 * prior_scale
    sc = gp.sample_conditional(g["t"], g["flux"], g["data_cov_vec"], t_sample=g["t_sample"],
                               nsamples=3, eps=1e-8, unit_normals=g["cond_U_" + tag], **KWB)
    assert tuple(sc.shape) == (3, 120)
    # the draws add L u with |L u| ~ sqrt(K + eps): compare on the scale of the mean
    assert relmax(sc.cpu().numpy(), g["cond_sample_" + tag]) <= 1e-6


@pytest.mark.gpu
def test_gpu_sample_ylm_conditional_vs_reference_golden(spb, golden):
    """(1) The conditional-sampling pipeline itself, fed the REFERENCE's Ylm moments (as
    test_gpu_parity.py::test_sample_ylm_given_cov does for the prior draws): this method inverts
    ``cov_ylm`` explicitly (sp.py:267-271) and ``cov_ylm`` is only reproducible to the reference's
    own noise modes (2e-7 absolute, DESIGN.md "numerical fragility"), which 1/lambda_min = 1e12
    amplifies.  (2) End to end with the CUDA moments: compared through the flux the draws imply."""
    import torch

    g = golden("predict_nt200.npz")
    fid = golden("fiducial_nt1000.npz")
    gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **FID)
    gp._compute_moments()
    A = gp.design_matrix(g["t"], **KW).cpu().numpy()
    y_own = gp.sample_ylm_conditional(g["t"], g["flux"], 1e-6, nsamples=3,
                                      unit_normals=g["ylmc_U"], **KWB).cpu().numpy()
    # (1) reference moments injected
    gp._mean_ylm = torch.tensor(fid["mean_ylm"], device="cuda").reshape(1, 256).contiguous()
    gp._cov_ylm = torch.tensor(fid["cov_ylm"], device="cuda").reshape(1, 256, 256).contiguous()
    gp._cho_cov_ylm = None
    y = gp.sample_ylm_conditional(g["t"], g["flux"], 1e-6, nsamples=3, unit_normals=g["ylmc_U"],
                                  **KWB)
    assert tuple(y.shape) == (3, 256)
    y = y.cpu().numpy()
    err_y, err_flux = relmax(y, g["ylmc_y"]), relmax(y @ A.T, g["ylmc_flux"])
    # (2) own moments
    own_y, own_flux = relmax(y_own, g["ylmc_y"]), relmax(y_own @ A.T, g["ylmc_flux"])
    print("sample_ylm_conditional: reference moments -> y %.2e flux %.2e; CUDA moments -> y %.2e "
          "flux %.2e" % (err_y, err_flux, own_y, own_flux))
    assert err_y <= 1e-7 and err_flux <= 1e-8
    assert own_flux <= 1e-5 and own_y <= 2e-2


@pytest.mark.gpu
def test_gpu_reference_test_sample_conditional(spb):
    """tests/test_sample.py:8-26 of the reference, with the design matrix in place of starry."""
    import torch

    gp = spb.StarryProcess(normalized=False, marginalize_over_inclination=False)
    t = np.linspace(0, 2, 300)
    gen = torch.Generator(device="cuda").manual_seed(3)
    flux = gp.sample(t, p=1.0, i=60.0, generator=gen).reshape(-1)
    data_cov = 1e-6
    y = gp.sample_ylm_conditional(t, flux, data_cov, p=1.0, i=60.0, generator=gen)
    A = gp.design_matrix(t, i=60.0, p=1.0)
    flux_pred = (A @ y.reshape(-1))
    chisq = float(((flux - flux_pred) ** 2 / data_cov).sum())
    assert chisq / len(t) < 1


@pytest.mark.gpu
def test_gpu_predict_batched_and_errors(spb, golden):
    """(B,) hyperparameters give a leading batch axis; element 0 equals the scalar call."""
    g = golden("predict_nt200.npz")
    hp = dict(r=[10.0, 15.0], mu=[30.0, 40.0], sigma=[5.0, 8.0], c=[0.1, 0.08], n=[10.0, 5.0])
    gp = spb.StarryProcess(normalized=False, **hp)
    mu, K = gp.predict(g["t"], g["flux"], 1e-6, t_sample=g["t_sample"], **KW)
    assert tuple(mu.shape) == (2, 120) and tuple(K.shape) == (2, 120, 120)
    gp0 = spb.StarryProcess(normalized=False, **FID)
    mu0, K0 = gp0.predict(g["t"], g["flux"], 1e-6, t_sample=g["t_sample"], **KW)
    assert float((mu[0] - mu0).abs().max()) <= 1e-12 * float(mu0.abs().max())
    assert float((K[0] - K0).abs().max()) <= 1e-16
    with pytest.raises(NotImplementedError):
        spb.StarryProcess(normalized=True, **FID).predict(g["t"], g["flux"], 1e-6)
    with pytest.raises(NotImplementedError):
        spb.StarryProcess(normalized=True, **FID).sample_ylm_conditional(g["t"], g["flux"], 1e-6)


HP3 = dict(r=[10.0, 15.0, 20.0], mu=[30.0, 40.0, 50.0], sigma=[5.0, 8.0, 10.0], c=[0.1, 0.08, 0.05],
           n=[10.0, 5.0, 3.0])


@pytest.mark.gpu
@pytest.mark.parametrize("marg", [False, True])
def test_gpu_predict_per_element_baseline_mean(spb, golden, marg):
    """A (B,) baseline_mean gives every batch element its own: element b of the batched predict and
    sample_conditional equals, bit for bit, the same call with the scalar baseline_mean[b]."""
    import torch

    g = golden("predict_nt200.npz")
    gp = spb.StarryProcess(normalized=False, marginalize_over_inclination=marg, **HP3)
    bm = np.array([-2e-4, 0.0, 3e-4])
    un = np.random.default_rng(0).standard_normal((120, 2))
    kw = dict(t_sample=g["t_sample"], i=60.0, p=1.0, u=U_LD, baseline_var=1e-5)
    args = (g["t"], g["flux"], g["data_cov_vec"])
    mu, K = gp.predict(*args, baseline_mean=bm, **kw)
    s = gp.sample_conditional(*args, baseline_mean=bm, unit_normals=un, **kw)
    assert tuple(mu.shape) == (3, 120) and tuple(s.shape) == (3, 2, 120)
    for b in range(3):
        mu_b, K_b = gp.predict(*args, baseline_mean=float(bm[b]), **kw)
        s_b = gp.sample_conditional(*args, baseline_mean=float(bm[b]), unit_normals=un, **kw)
        assert torch.equal(mu[b], mu_b[b]) and torch.equal(K[b], K_b[b]) and torch.equal(s[b], s_b[b])


@pytest.mark.gpu
def test_gpu_sample_ylm_conditional_rejects_per_element_baseline(spb, golden):
    """sample_ylm_conditional factorises one noise covariance and one residual for the whole batch:
    a (B,) baseline_mean or baseline_var raises ValueError before any kernel launch."""
    g = golden("predict_nt200.npz")
    gp = spb.StarryProcess(normalized=False, marginalize_over_inclination=False, **HP3)
    gp.design_matrix(g["t"], **KW)          # moments and flux operator computed ahead
    gp.mean_ylm
    n0 = gp._ctx.launches()
    for bad in (dict(baseline_mean=np.array([0.0, 1e-4, 2e-4])), dict(baseline_var=np.full(3, 1e-5))):
        with pytest.raises(ValueError, match="whole batch"):
            gp.sample_ylm_conditional(g["t"], g["flux"], 1e-6, **KW, **bad)
    assert gp._ctx.launches() == n0


@pytest.mark.gpu
@pytest.mark.parametrize("marg", [False, True])
def test_gpu_predict_odd_sizes_vs_live_oracle(spb, oracle, golden, marg):
    """Odd nt / nts (padded leading dimensions), vector data_cov, default t_sample, against the
    oracle evaluated LIVE on this host.  The marginalised branch of the reference algorithm is
    only reproducible to ~3e-6 between CPUs (LAPACK kernel selection moves its noise-level
    eigenmodes; DESIGN.md "numerical fragility" -- the pinned 1e-8 check is the golden-fixture
    test above), hence the looser bound there."""
    g = golden("predict_nt200.npz")
    nt, nts = 151, 77
    t, f = g["t"][:nt], g["flux"][:nt]
    ts = np.linspace(0.05, 0.7, nts)
    dv = g["data_cov_vec"][:nt]
    gp = spb.StarryProcess(marginalize_over_inclination=marg, normalized=False, **FID)
    o = oracle.OracleProcess(marginalize_over_inclination=marg, normalized=False, **FID)
    mu, K = gp.predict(t, f, dv, t_sample=ts, baseline_var=2e-6, **KW)
    mo, Ko = o.predict(t, f, dv, t_sample=ts, baseline_var=2e-6, **KW)
    scale = float(np.abs(o.cov(t, **KW)).max())
    tol = 5e-6 if marg else 1e-7
    assert tuple(mu.shape) == (nts,) and tuple(K.shape) == (nts, nts)
    assert np.abs(mu.cpu().numpy() - mo).max() <= tol * np.abs(mo).max()
    assert np.abs(K.cpu().numpy() - Ko).max() <= tol * scale
    mu2, K2 = gp.predict(t, f, dv, **KW)          # t_sample = t
    mo2, Ko2 = o.predict(t, f, dv, **KW)
    assert np.abs(mu2.cpu().numpy() - mo2).max() <= tol * np.abs(mo2).max()
    assert np.abs(K2.cpu().numpy() - Ko2).max() <= tol * scale
    # draws: finite, right shape, reproducible for a fixed generator
    import torch

    s1 = gp.sample_conditional(t, f, dv, t_sample=ts, nsamples=4,
                               generator=torch.Generator(device="cuda").manual_seed(1), **KW)
    s2 = gp.sample_conditional(t, f, dv, t_sample=ts, nsamples=4,
                               generator=torch.Generator(device="cuda").manual_seed(1), **KW)
    assert tuple(s1.shape) == (4, nts) and bool(torch.isfinite(s1).all()) and torch.equal(s1, s2)
    s3 = gp.sample(t, nsamples=2, generator=torch.Generator(device="cuda").manual_seed(2), **KW)
    assert tuple(s3.shape) == (2, nt) and bool(torch.isfinite(s3).all())


@pytest.mark.gpu
def test_gpu_sample_predict_chunked_equals_unchunked():
    """ADVICE r1: sample / predict / sample_conditional / sample_ylm_conditional split a large batch
    into chunks (max_chunk_bytes, and at most 65535 elements per launch) like log_likelihood does;
    chunked and unchunked evaluation agree bit for bit (same kernels per element)."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import starry_process_b200 as spb

    rng = np.random.default_rng(2)
    B, nt = 9, 60
    hp = dict(r=rng.uniform(10, 30, B), mu=rng.uniform(0, 80, B), sigma=rng.uniform(5, 30, B),
              c=rng.uniform(0.02, 0.12, B), n=rng.uniform(1, 10, B))
    t = np.linspace(0, 2, nt)
    ts = np.linspace(0.1, 2.3, 37)
    f = 1e-3 * rng.standard_normal(nt)
    un = rng.standard_normal((nt, 3))
    un_s = rng.standard_normal((37, 2))
    un_y = rng.standard_normal((256, 2))
    inc = torch.tensor(rng.uniform(20, 80, B))
    for marg in (True, False):
        kw = dict(normalized=False, marginalize_over_inclination=marg, **hp)
        big = spb.StarryProcess(**kw)
        small = spb.StarryProcess(max_chunk_bytes=3 << 20, **kw)     # ~ 2 elements per chunk
        ii = 60.0 if marg else inc
        a = big.sample(t, i=ii, unit_normals=un)
        b = small.sample(t, i=ii, unit_normals=un)
        assert a.shape == (B, 3, nt) and torch.equal(a, b)
        (m1, K1), (m2, K2) = big.predict(t, f, 1e-6, t_sample=ts, i=ii), small.predict(t, f, 1e-6, t_sample=ts, i=ii)
        assert torch.equal(m1, m2) and torch.equal(K1, K2)
        c1 = big.sample_conditional(t, f, 1e-6, t_sample=ts, i=ii, unit_normals=un_s)
        c2 = small.sample_conditional(t, f, 1e-6, t_sample=ts, i=ii, unit_normals=un_s)
        assert torch.equal(c1, c2)
    y1 = big.sample_ylm_conditional(t, f, 1e-6, i=60.0, unit_normals=un_y)
    y2 = small.sample_ylm_conditional(t, f, 1e-6, i=60.0, unit_normals=un_y)
    assert y1.shape == (B, 2, 256) and torch.equal(y1, y2)
