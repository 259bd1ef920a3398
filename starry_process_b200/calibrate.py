"""Batched callers of the likelihood path (SURVEY.md section 8(f), rank 1): the B200-native
counterparts of ``starry_process/calibrate/log_prob.py:7-106`` (``get_log_prob``) and of the
evaluation loop of ``starry_process/calibrate/inclination.py:44-74`` (``compute_inclination_pdf``).

The reference compiles a Theano function of scalar hyperparameters and calls it once per posterior
sample (and, for the inclination posterior, once per light curve x sample x inclination).  Here the
returned callable takes scalars *or* ``(B,)`` tensors and evaluates the whole batch in one pass of
the CUDA path; everything else (argument order, defaults, the always-added ``10 ** baseline_log_var``
term, ``covpts = len(t) - 1``, no normalisation-range cut, NaN -> -inf, the latitude Jacobian) follows
the reference.
"""
import numpy as np
import torch

from .sp import StarryProcess, defaults

__all__ = ["get_log_prob", "inclination_log_prob"]


def get_log_prob(t, flux=None, ferr=1.0e-3, p=1.0, ydeg=15, baseline_log_var=0.0, baseline_mean=0.0,
                 apply_jac=True, normalized=True, marginalize_over_inclination=True, u=(0.0, 0.0),
                 device=None, method="dense"):
    """calibrate/log_prob.py:7-106.  Returns ``log_prob(*args)`` with the reference's argument order
    ``[flux,] r, a, b, c, n [, m] [, v] [, i]`` (``flux`` only if it was not fixed here, ``m`` only if
    ``baseline_mean is None``, ``v`` only if ``baseline_log_var is None``, ``i`` only if
    ``marginalize_over_inclination`` is false).  ``method``: as in ``StarryProcess.log_likelihood``
    (``"lowrank"`` needs ``marginalize_over_inclination=False``)."""
    t = np.asarray(t, dtype=np.float64).reshape(-1)
    K = t.size
    free_flux = flux is None
    fixed_flux = None if free_flux else flux

    def log_prob(*args):
        args = list(args)
        fl = args.pop(0) if free_flux else fixed_flux
        r, a, b, c, n = args[:5]
        rest = args[5:]
        m = rest.pop(0) if baseline_mean is None else baseline_mean
        v = rest.pop(0) if baseline_log_var is None else baseline_log_var
        inc = defaults["i"] if marginalize_over_inclination else rest.pop(0)
        if rest:
            raise TypeError("too many arguments for log_prob")
        gp = StarryProcess(
            ydeg=ydeg, r=r, a=a, b=b, c=c, n=n, normalized=normalized,
            marginalize_over_inclination=marginalize_over_inclination, covpts=K - 1,
            normalization_zmax=float("inf"),      # log_prob.py uses sp.cov() directly: no z cut
            device=device)
        if isinstance(v, torch.Tensor):
            bvar = 10.0 ** v.to(torch.float64)
        elif isinstance(v, np.ndarray):
            bvar = 10.0 ** v.astype(np.float64)
        else:
            bvar = torch.tensor(10.0 ** float(v), dtype=torch.float64)   # 10 ** 0 = 1 by default
        ll = gp.log_likelihood(t, fl, float(ferr) ** 2, i=inc, p=p, u=list(u), baseline_mean=m,
                               baseline_var=bvar, method=method)
        if apply_jac:
            ll = ll + gp.log_jac()
        return ll

    return log_prob


def inclination_log_prob(t, flux, samples, inc, ferr=1.0e-3, p=1.0, ydeg=15, baseline_log_var=0.0,
                         baseline_mean=0.0, apply_jac=True, normalized=True, u=(0.0, 0.0),
                         device=None, method="dense"):
    """The (light curve x posterior sample x inclination) grid of conditional log-probabilities that
    calibrate/inclination.py:63-74 fills with ``nlc * ninc_samples * ninc_pts`` separate calls.

    ``flux``: ``(nlc, nt)``; ``samples``: ``(ns, 5)`` rows ``r, a, b, c, n`` (the posterior draws the
    caller selected); ``inc``: ``(ninc,)`` degrees.  Returns ``lp`` of shape ``(nlc, ns, ninc)``.
    ``method="lowrank"`` evaluates every element through the rank-31 form (DESIGN.md section 4.6)."""
    flux = torch.as_tensor(np.asarray(flux), dtype=torch.float64)
    samples = torch.as_tensor(np.asarray(samples), dtype=torch.float64)
    inc = torch.as_tensor(np.asarray(inc), dtype=torch.float64).reshape(-1)
    nlc, nt = flux.shape
    ns, ninc = samples.shape[0], inc.numel()
    # element (l, s, k): light curve l, sample s, inclination k
    hp = samples[None, :, None, :].expand(nlc, ns, ninc, 5).reshape(-1, 5)
    ii = inc[None, None, :].expand(nlc, ns, ninc).reshape(-1)
    fl = flux[:, None, None, :].expand(nlc, ns, ninc, nt).reshape(-1, 1, nt)
    fn = get_log_prob(t, flux=None, ferr=ferr, p=p, ydeg=ydeg, baseline_log_var=baseline_log_var,
                      baseline_mean=baseline_mean, apply_jac=apply_jac, normalized=normalized,
                      marginalize_over_inclination=False, u=u, device=device, method=method)
    lp = fn(fl, hp[:, 0].contiguous(), hp[:, 1].contiguous(), hp[:, 2].contiguous(),
            hp[:, 3].contiguous(), hp[:, 4].contiguous(), ii.contiguous())
    return lp.reshape(nlc, ns, ninc)
