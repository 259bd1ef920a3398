"""Small end-to-end workload for compute-sanitizer (memcheck / racecheck): every kernel family once."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import starry_process_b200 as spb
t = np.linspace(0, 2, 301)
rng = np.random.default_rng(0)
f = 1e-3 * rng.standard_normal(301)
for marg in (True, False):
    gp = spb.StarryProcess(r=[12.0, 20.0, 15.0], mu=[30.0, 50.0, 10.0], sigma=[5.0, 10.0, 20.0], c=[0.1, 0.05, 0.2],
                           n=[10.0, 3.0, 5.0], marginalize_over_inclination=marg)
    print("lnlike", gp.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=[0.4, 0.26]).cpu().numpy())
gp = spb.StarryProcess(r=12.0, mu=30.0, sigma=5.0, c=0.1, n=10.0, normalized=False, tau=0.5)
mu, K = gp.predict(t, f, 1e-6, t_sample=t[:77], i=60.0)
print("predict", float(mu.sum()), float(K.trace()))
print("sample", float(gp.sample(t[:100], nsamples=2).sum()))
gp2 = spb.StarryProcess(r=12.0, mu=30.0, sigma=5.0, c=0.1, n=10.0, normalized=False,
                        marginalize_over_inclination=False)
print("ylm cond", float(gp2.sample_ylm_conditional(t, f, 1e-6, i=60.0).sum()))
print("design", float(gp2.design_matrix(t, i=[10.0, 80.0]).sum()))
print("sample_ylm", float(gp2.sample_ylm(nsamples=3).sum()))
torch.cuda.synchronize()
print("done")
# round 2: uniform spot-size prior, gradient (tangent kernels)
gd = spb.StarryProcess(r=[15.0, 20.0], dr=[5.0, 3.0], mu=30.0, sigma=5.0, c=0.1, n=10.0)
print("dr lnlike", gd.log_likelihood(t, f, 1e-6, u=[0.4, 0.26]).cpu().numpy())
gg = spb.StarryProcess(r=[12.0, 20.0], a=[0.4, 0.5], b=[0.27, 0.2], c=0.1, n=10.0)
ll, g = gg.log_likelihood(t[:120], f[:120], 1e-6, u=[0.4, 0.26], return_grad=True)
print("grad", {k: v.cpu().numpy() for k, v in g.items()})
ctx = spb.get_context(0)
ctx.set_option("cholesky_cluster", 0)   # few matrices: the one-CTA-per-matrix kernel instead of clusters
print("batch kernel", gg.log_likelihood(t, f, 1e-6, u=[0.4, 0.26]).cpu().numpy())
ctx.set_option("cholesky_cluster", 1)
torch.cuda.synchronize()
print("done round 2")
# round 2: Cholesky on the INT8 tensor cores (tcgen05 / TMEM / 4-D TMA), all three digit formats, both branches,
# sizes with a partial last panel, the "gap" and the padded layouts of the right-hand-side planes
for code in (78, 87, 77):
    ctx.set_option("cholesky_i8", code)
    for marg in (True, False):
        gi = spb.StarryProcess(r=[12.0, 20.0, 15.0], mu=[30.0, 50.0, 10.0], sigma=[5.0, 10.0, 20.0],
                               c=[0.1, 0.05, 0.2], n=[10.0, 3.0, 5.0], marginalize_over_inclination=marg)
        print("i8", code, marg, gi.log_likelihood(t, f, 1e-6, i=60.0, p=1.0, u=[0.4, 0.26]).cpu().numpy())
    fm = np.stack([f + 1e-4 * k for k in range(30)])       # 30 light curves: more rows than the gap holds
    print("i8 M=30", code, gi.log_likelihood(t, fm, 1e-6, i=60.0, p=1.0, u=[0.4, 0.26]).cpu().numpy())
ctx.set_option("cholesky_i8", -1)
torch.cuda.synchronize()
print("done int8")
# round 2: conditional flux covariance (A Sigma) A^T on the INT8 tensor cores (nt >= 1024, lower triangle) and
# the tabulated marginal assembly of equally spaced time stamps (already taken by the linspace grids above)
tl = np.linspace(0, 5, 1100)
fl = 1e-3 * rng.standard_normal(1100)
gc = spb.StarryProcess(r=[12.0, 20.0, 15.0], mu=[30.0, 50.0, 10.0], sigma=[5.0, 10.0, 20.0], c=[0.1, 0.05, 0.2],
                       n=[10.0, 3.0, 5.0], marginalize_over_inclination=False, normalized=False)
print("conditional nt=1100", gc.log_likelihood(tl, fl, 1e-6, i=[40.0, 60.0, 80.0], p=1.7, u=[0.4, 0.26]).cpu().numpy())
print("conditional nt=1100, one inclination", gc.log_likelihood(tl, fl, 1e-6, i=60.0, p=1.7, u=[0.4, 0.26]).cpu().numpy())
ti = np.sort(rng.uniform(0, 2, 301))
print("irregular stamps", gp2.log_likelihood(ti, f, 1e-6, i=60.0).cpu().numpy())
torch.cuda.synchronize()
print("done conditional int8")
