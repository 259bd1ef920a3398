"""
``StarryProcess`` -- B200-native drop-in for the batched likelihood path of
``starry_process.StarryProcess`` (reference: starry_process/sp.py:38-284, 420-441, 489-509,
643-727, 1052-1188).

Same constructor keywords, property names and method signatures as the reference for the hot
path; inputs/outputs are ``torch.float64`` CUDA tensors and evaluation is eager.  Extension: any of
``r, mu, sigma, a, b, c, n`` may be a ``(B,)`` tensor (one hyperparameter sample per element), and
``i`` may be ``(B,)`` in the conditional branch; outputs then carry a leading batch axis and
``log_likelihood`` returns ``(B,)``.  All numerics run in ``libspb200.so`` (hand-written sm_100a CUDA
behind ``include/spb200.h``) -- there is no CPU or PyTorch fallback: without the library (or without
a CUDA device) construction raises.

SURVEY.md section 8(f) ranks 2 and 3 are covered as well: ``sample``, ``predict``,
``sample_conditional`` and ``sample_ylm_conditional`` (sp.py:518-641, 729-765, 767-1002), composed
from the same Cholesky / GEMM / assembly kernels, and time-variable surfaces (``tau``,
``temporal_kernel``: temporal.py:8-16, sp.py:697-698, 893-894, 510-516).

The uniform spot-size prior (``dr``, size.py:55-89, 116-125; SURVEY.md section 8(f) rank 4) is
supported.  Out of scope in this drop-in: pixel-space moments and visualisation.
"""
import ctypes
import math
import os

import numpy as np
import torch

from . import _lib, _tables, temporal as _temporal

__all__ = ["StarryProcess", "StarryProcessSum", "gauss2beta", "beta2gauss", "defaults"]

# starry_process/defaults.py:4-35
defaults = dict(
    ydeg=15, udeg=2, r=20.0, dr=None, a=0.40, b=0.27, c=0.1, n=10.0, p=1.0, i=60.0,
    u=[0.0, 0.0], tau=None, normalized=True, normalization_order=20, normalization_zmax=0.023,
    marginalize_over_inclination=True, baseline_mean=0.0, baseline_var=0.0, covpts=300,
    log_alpha_max=10, log_beta_max=10, abmin=1e-12, sigma_max=45.0, epsy=1e-12, epsy15=1e-9,
    eps=1e-8,
)

_CTX = {}
# module-wide default of the `longitude_basis` keyword (environment: SPB200_LONGITUDE_BASIS)
DEFAULT_LONGITUDE_BASIS = os.environ.get("SPB200_LONGITUDE_BASIS", "pinned")


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class _Context(object):
    """One libspb200 context (constant tables resident in HBM) per CUDA device."""

    def __init__(self, device, longitude_basis="pinned"):
        if not torch.cuda.is_available():
            raise RuntimeError("starry_process_b200 needs a CUDA device (sm_100a); no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device("cuda", device)
        self.longitude_basis = longitude_basis
        blob, _ = _tables.build_tables(longitude_basis)
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            torch.cuda.current_stream().synchronize()
            _lib.check(self.lib.spb_create(device, blob.ctypes.data_as(ctypes.c_void_p), blob.size,
                                           ctypes.byref(h)))
        self.handle = h
        # INT8-tensor-core Cholesky (spb_cholesky_lnlike_i8): 0 = always the FP64 (DMMA) kernel; 78 = seven
        # planes of 8-bit digits (55 bits per row: FP64 rounding-noise level), 8 / 87 = eight planes of 7-bit
        # digits (56 bits), 7 / 77 = seven planes of 7-bit digits (49 bits) whenever the path applies;
        # -1 (default) = automatic: 78 where that kernel is the faster one on B200 -- nt >= 704 and more
        # matrices than the cluster kernel takes (measured Cholesky stage, INT8 vs DMMA: nt = 512 +14 %,
        # 768 -10 %, 1000 -13 % (-25 % conditional), 1536 -45 %, 4096 -55 %)
        self.cholesky_i8 = int(os.environ.get("SPB200_CHOLESKY_I8", "-1"))
        self.num_sms = torch.cuda.get_device_properties(self.device).multi_processor_count

    def i8_planes(self, nt, batch):
        """Digit planes the batched ``log_likelihood`` uses for ``batch`` matrices of size ``nt`` (0: the
        FP64 kernel)."""
        if self.cholesky_i8 >= 0:
            return self.cholesky_i8
        return 78 if (nt >= 704 and 2 * batch > self.num_sms) else 0

    def set_option(self, name, value):
        """Run-time switches of the library (include/spb200.h: spb_set_option), plus
        ``"cholesky_i8"`` (-1 | 0 | 7 | 8): batched ``log_likelihood`` factorises on the INT8 tensor cores
        with that many 7-bit digit planes (``spb_cholesky_lnlike_i8``); -1 = automatic, 0 = never."""
        if name == "cholesky_i8":
            if int(value) not in (-1, 0, 7, 8, 77, 78, 87):
                raise ValueError("cholesky_i8 must be -1, 0, 7 (= 77), 8 (= 87) or 78")
            self.cholesky_i8 = int(value)
            return
        _lib.check(self.lib.spb_set_option(self.handle, name.encode(), int(value)))

    def launches(self):
        n = ctypes.c_longlong()
        _lib.check(self.lib.spb_launch_count(self.handle, ctypes.byref(n)))
        return n.value


def get_context(device=None, longitude_basis=None):
    """The libspb200 context of ``device`` (created on first use).  ``longitude_basis``:
    ``"pinned"`` (default; the shipped longitude eigenvector table, identical on every host) or
    ``"host"`` (this host's own ``numpy.linalg.eigh``, what a reference run in this process uses) --
    see ``_tables.build_tables``.  The two bases are separate contexts."""
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    basis = DEFAULT_LONGITUDE_BASIS if longitude_basis is None else longitude_basis
    key = (int(device), basis)
    if key not in _CTX:
        _CTX[key] = _Context(int(device), basis)
    return _CTX[key]


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _is_batched(x):
    return (isinstance(x, torch.Tensor) and x.ndim > 0) or (isinstance(x, np.ndarray) and x.ndim > 0) \
        or isinstance(x, (list, tuple))


def _nt(t):
    """Number of time stamps of host or device ``t``."""
    return t.numel() if isinstance(t, torch.Tensor) else int(np.size(t))


def _four_arrays(n1, n2):
    """Device bytes per element of ``sample``, ``predict`` and the conditional samplers: about four
    (n1 x n2) arrays, and the moments."""
    return 4 * n1 * (n2 + (n2 & 1)) * 8 + 4 * 256 * 256 * 8


# arguments of a chunk body (StarryProcess._batch) that carry a leading batch axis of B entries when
# they have this many dimensions
_BATCH_NDIM = dict(inc=1, f=3, bm=1, bvar=1, unit_normals=3)


def gauss2beta(mu, sigma, log_alpha_max=10, log_beta_max=10):
    """latitude.py:14-77 (host utility; accepts floats, arrays or tensors, angles in degrees)."""
    tens = isinstance(mu, torch.Tensor) or isinstance(sigma, torch.Tensor)
    m = torch.as_tensor(mu, dtype=torch.float64) * math.pi / 180
    v = (torch.as_tensor(sigma, dtype=torch.float64) * math.pi / 180) ** 2
    c1, c2, c3 = torch.cos(m), torch.cos(2 * m), torch.cos(3 * m)
    term = 1.0 / (16 * v * torch.cos(0.5 * m) ** 4)
    alpha = (2 + 4 * v + (3 + 8 * v) * c1 + 2 * c2 + c3) * term
    beta = (c1 + 2 * v * (3 + c2) - c3) * term
    a = torch.log(alpha) / log_alpha_max
    b = torch.clamp((torch.log(beta) - math.log(0.5)) / (log_beta_max - math.log(0.5)), min=0.0)
    if tens:
        return a, b
    if a.ndim == 0:
        return float(a), float(b)
    return a.numpy(), b.numpy()


def beta2gauss(a, b, log_alpha_max=10, log_beta_max=10):
    """latitude.py:80-168 (host utility)."""
    tens = isinstance(a, torch.Tensor) or isinstance(b, torch.Tensor)
    a_ = torch.as_tensor(a, dtype=torch.float64)
    b_ = torch.as_tensor(b, dtype=torch.float64)
    alpha = torch.exp(a_ * log_alpha_max)
    beta = torch.exp(math.log(0.5) + b_ * (log_beta_max - math.log(0.5)))
    term = 4 * alpha ** 2 - 8 * alpha - 6 * beta + 4 * alpha * beta + beta ** 2 + 5
    mu = 2 * torch.atan(torch.sqrt(2 * alpha + beta - 2 - torch.sqrt(term)))
    term = 1 - alpha + beta + (beta - 1) * torch.cos(mu) + (alpha - 1) / torch.cos(mu) ** 2
    sigma = torch.sin(mu) / torch.sqrt(term)
    invalid = (alpha <= 1) | (beta <= 0.5)
    nan = torch.full_like(mu, float("nan"))
    mu = torch.where(invalid, nan, mu) * 180 / math.pi
    sigma = torch.where(invalid, nan, sigma) * 180 / math.pi
    if tens:
        return mu, sigma
    if mu.ndim == 0:
        return float(mu), float(sigma)
    return mu.numpy(), sigma.numpy()


def _check_bounds(name, x, lower=-np.inf, upper=np.inf, tol=1e-6):
    """ops/exceptions.py:30-48 for host-resident values."""
    xv = np.atleast_1d(np.asarray(x, dtype=np.float64))
    low = xv < lower - tol
    high = xv > upper + tol
    if low.any():
        raise ValueError("%s out of bounds: %f %s %f" % (name, xv[low][0], "<=", lower))
    if high.any():
        raise ValueError("%s out of bounds: %f %s %f" % (name, xv[high][0], ">=", upper))


class StarryProcess(object):
    def __init__(self, r=defaults["r"], dr=defaults["dr"], c=defaults["c"], n=defaults["n"],
                 tau=defaults["tau"], temporal_kernel=None,
                 marginalize_over_inclination=defaults["marginalize_over_inclination"],
                 normalized=defaults["normalized"], covpts=defaults["covpts"], device=None,
                 **kwargs):
        # sp.py:204-222
        mu = kwargs.pop("mu", None)
        sigma = kwargs.pop("sigma", None)
        if mu is None and sigma is None:
            a = kwargs.pop("a", defaults["a"])
            b = kwargs.pop("b", defaults["b"])
        elif (kwargs.get("a", None) is None and kwargs.get("b", None) is None) and (
                mu is not None and sigma is not None):
            a = b = None
        else:
            raise ValueError("Must provide either `a` and `b` *or* `mu` and `sigma`.")
        # sp.py:225-232; the reference accepts any callable f(t1, t2, tau): the CUDA assembly
        # implements the two kernels the reference ships (temporal.py)
        self._time_variable = tau is not None
        self._tkind = 0
        if self._time_variable:
            tk = _temporal.Matern32Kernel if temporal_kernel is None else temporal_kernel
            if isinstance(tk, str):
                tk = {"matern32": _temporal.Matern32Kernel,
                      "expsquared": _temporal.ExpSquaredKernel}.get(tk.lower())
            kind = getattr(tk, "spb_kind", None)
            if kind is None:
                kind = {"Matern32Kernel": 1, "ExpSquaredKernel": 2}.get(
                    getattr(tk, "__name__", ""), None)
            if kind is None:
                raise NotImplementedError("temporal_kernel must be Matern32Kernel or "
                                          "ExpSquaredKernel (starry_process_b200.temporal)")
            self._tkind = int(kind)
            self._temporal_kernel = tk
        self._ydeg = int(kwargs.pop("ydeg", defaults["ydeg"]))
        self._udeg = int(kwargs.pop("udeg", defaults["udeg"]))
        assert self._ydeg >= 5, "Degree of map must be >= 5."           # sp.py:236
        if self._ydeg > 15:
            raise NotImplementedError("libspb200 evaluates spherical-harmonic degrees up to 15 (the "
                                      "reference is numerically unstable above: joss/paper.md:174-191)")
        if self._udeg not in (0, 2):
            raise NotImplementedError("udeg must be 0 or 2")
        # keyword options the reference threads through its integrals (sp.py:241-262):
        # contrast.py:26-32 (epsy, epsy15), latitude.py:171-200 (abmin, log_alpha_max, log_beta_max)
        self._opt_kw = dict(epsy=float(kwargs.pop("epsy", defaults["epsy"])),
                            epsy15=float(kwargs.pop("epsy15", defaults["epsy15"])),
                            abmin=float(kwargs.pop("abmin", defaults["abmin"])),
                            log_alpha_max=float(kwargs.pop("log_alpha_max", defaults["log_alpha_max"])),
                            log_beta_max=float(kwargs.pop("log_beta_max", defaults["log_beta_max"])))
        self._normN = int(kwargs.pop("normalization_order", defaults["normalization_order"]))
        self._normzmax = float(kwargs.pop("normalization_zmax", defaults["normalization_zmax"]))
        self._max_chunk_bytes = int(kwargs.pop("max_chunk_bytes", 96 << 30))
        self._sigma_max = float(kwargs.pop("sigma_max", defaults["sigma_max"]))
        kwargs.pop("seed", None)
        self._nylm = (self._ydeg + 1) ** 2
        self._covpts = int(covpts)
        self._normalized = bool(normalized)
        self._marginalize_over_inclination = bool(marginalize_over_inclination)

        self._ctx = get_context(device, kwargs.pop("longitude_basis", None))
        self.device = self._ctx.device
        self._lib = self._ctx.lib
        self._opt, self._opt_keep = self._moments_options()

        params = dict(r=r, c=c, n=n)
        if dr is not None:     # uniform prior on the spot radius over [r - dr, r + dr], size.py:116-125
            params["dr"] = dr
        if self._time_variable:
            params["tau"] = tau
        if a is None:
            params.update(mu=mu, sigma=sigma)
        else:
            params.update(a=a, b=b)
        self._batched = any(_is_batched(v) for v in params.values())
        # host-side bounds checks, as the reference raises (device-resident tensors are flagged
        # per element through info[] instead of forcing a device->host sync)
        hostvals = {k: v for k, v in params.items()
                    if not (isinstance(v, torch.Tensor) and v.is_cuda)}
        if "r" in hostvals:
            _check_bounds("r", np.asarray(hostvals["r"], dtype=np.float64) * np.pi / 180, 0,
                          0.5 * np.pi)
        if "dr" in hostvals:
            _check_bounds("dr", np.asarray(hostvals["dr"], dtype=np.float64) * np.pi / 180, 0,
                          0.5 * np.pi)
        if "a" in hostvals:
            _check_bounds("a", hostvals["a"], 0, 1)
        if "b" in hostvals:
            _check_bounds("b", hostvals["b"], 0, 1)
        if "n" in hostvals:
            _check_bounds("n", hostvals["n"], 0, np.inf)
        if "tau" in hostvals:
            _check_bounds("tau", hostvals["tau"], 0, np.inf)
        tens = {k: torch.as_tensor(v, dtype=torch.float64).to(self.device).reshape(-1)
                for k, v in params.items()}
        B = max(t.numel() for t in tens.values())
        for k, t in tens.items():
            if t.numel() not in (1, B):
                raise ValueError("hyperparameter `%s` has %d elements, expected 1 or %d" %
                                 (k, t.numel(), B))
            tens[k] = t.expand(B).contiguous()
        self._B = B
        self._r, self._c, self._n = tens["r"], tens["c"], tens["n"]
        self._tau = tens.get("tau", None)
        self._dr = tens.get("dr", None)
        self._mu_sigma = None
        if a is None:
            self._mu_sigma = (tens["mu"], tens["sigma"])
            self._a = torch.empty(B, dtype=torch.float64, device=self.device)
            self._b = torch.empty(B, dtype=torch.float64, device=self.device)
            with torch.cuda.device(self.device):
                _lib.check(self._lib.spb_gauss2beta(self._ctx.handle, B, _ptr(tens["mu"]),
                                                    _ptr(tens["sigma"]), _ptr(self._a),
                                                    _ptr(self._b), _stream()))
            if "mu" in hostvals:
                ah, bh = gauss2beta(torch.as_tensor(hostvals["mu"], dtype=torch.float64),
                                    torch.as_tensor(hostvals["sigma"], dtype=torch.float64))
                _check_bounds("a", ah.numpy(), 0, 1)
                _check_bounds("b", bh.numpy(), 0, 1)
        else:
            self._a, self._b = tens["a"], tens["b"]
        self._mean_ylm = None
        self._cov_ylm = None
        self._cho_cov_ylm = None
        self._info = torch.zeros(B, dtype=torch.int32, device=self.device)
        self._z = None
        self._rTA1_cache = {}

    def _moments_options(self):
        """spb_moments_options for non-default keywords / a degree below 15 (None: all defaults).
        A lower degree is EMBEDDED in the degree-15 machinery: the spot operator ``Bp`` of that degree
        (size.py:10-43, rows l > ydeg zero) and a jitter vector that vanishes for l > ydeg make every
        Ylm moment with l > ydeg exactly zero, the rotations are block-diagonal in l, and the
        leading ``(ydeg+1)^2`` block is the reference's degree-``ydeg`` result."""
        kw, ydeg = self._opt_kw, self._ydeg
        default = (ydeg == 15 and kw["epsy"] == defaults["epsy"] and kw["epsy15"] == defaults["epsy15"]
                   and kw["abmin"] == defaults["abmin"]
                   and kw["log_alpha_max"] == defaults["log_alpha_max"]
                   and kw["log_beta_max"] == defaults["log_beta_max"])
        if default:
            return None, ()
        opt = _lib.MomentsOptions()
        keep = []
        if ydeg < 15:
            Bp = np.zeros((16, 1000))
            Bp[: ydeg + 1] = _tables.spot_operator(ydeg)
            bp_d = torch.tensor(Bp, dtype=torch.float64, device=self.device).contiguous()
            keep.append(bp_d)
            opt.Bp = bp_d.data_ptr()
        lam = np.zeros(256)
        lam[: self._nylm] = kw["epsy"]
        lam[15 ** 2: self._nylm] = kw["epsy15"]        # contrast.py:28-31 (only l = 15 exists there)
        lam_d = torch.tensor(lam, dtype=torch.float64, device=self.device)
        keep.append(lam_d)
        opt.lambda_ = lam_d.data_ptr()
        opt.abmin, opt.log_alpha_max, opt.log_beta_max = kw["abmin"], kw["log_alpha_max"], kw["log_beta_max"]
        return opt, tuple(keep)

    def _optp(self):
        return ctypes.byref(self._opt) if self._opt is not None else None

    @property
    def ydeg(self):
        """sp.py:347-350."""
        return self._ydeg

    def _cut(self, x, dims):
        """Leading (ydeg+1)^2 block along the given Ylm axes (no-op at degree 15)."""
        if self._nylm == 256:
            return x
        for d in dims:
            x = x.narrow(d, 0, self._nylm)
        return x.contiguous()

    def _pad_ylm(self, x, dim):
        """Zero-pad a Ylm axis of length (ydeg+1)^2 to 256."""
        if x.shape[dim] == 256:
            return x
        if x.shape[dim] != self._nylm:
            raise ValueError("expected a spherical-harmonic axis of length %d" % self._nylm)
        shape = list(x.shape)
        shape[dim] = 256
        out = torch.zeros(shape, dtype=x.dtype, device=x.device)
        out.narrow(dim, 0, self._nylm).copy_(x)
        return out

    # ------------------------------------------------------------------ hyperparameters
    @property
    def a(self):
        return self._out(self._a)

    @property
    def b(self):
        return self._out(self._b)

    @property
    def batch_size(self):
        return self._B

    @property
    def info(self):
        """Per-element status bits (include/spb200.h: SPB_INFO_*)."""
        return self._info

    def _out(self, t):
        return t if self._batched else t[0]

    # optional per-stage CUDA-event timing (bench.py sets ``_stage_ms`` to a dict)
    _stage_ms = None

    def _mark(self, name):
        """Opens an NVTX range for one phase of the path (SURVEY.md section 5: moments, flux_marginal /
        design, assemble, cholesky; visible in nsys / ncu --nvtx) and, when ``_stage_ms`` is set,
        brackets it with CUDA events on the launching stream."""
        torch.cuda.nvtx.range_push("spb200:" + name)
        if self._stage_ms is None:
            return False
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        self._stage_ms.setdefault(name, []).append((e0, e1))
        return e1

    @staticmethod
    def _mark_end(ev):
        if ev is not False:
            ev.record()
        torch.cuda.nvtx.range_pop()

    def log_jac(self):
        """sp.py:1004-1050 -> LatitudeIntegral._log_jac (latitude.py:281-316): log-Jacobian of the
        ``(a, b) -> (mu, sigma)`` transform, ``-inf`` where ``sigma > sigma_max``."""
        out = torch.empty(self._B, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.spb_log_jac_opt(self._ctx.handle, self._B, _ptr(self._a),
                                                 _ptr(self._b), self._sigma_max, self._optp(),
                                                 _ptr(out), _stream()))
        return self._out(out)

    # ------------------------------------------------------------------ Ylm moments
    def _compute_moments(self):
        if self._mean_ylm is not None:
            return
        B = self._B
        with torch.cuda.device(self.device):
            mean = torch.empty(B, 256, dtype=torch.float64, device=self.device)
            cov = torch.empty(B, 256, 256, dtype=torch.float64, device=self.device)
            nbytes = self._lib.spb_ylm_moments_workspace_bytes(self._ctx.handle, B)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            ev = self._mark("moments")
            _lib.check(self._lib.spb_ylm_moments_dr(
                self._ctx.handle, B, _ptr(self._r), _ptr(self._dr), _ptr(self._a), _ptr(self._b),
                _ptr(self._c), _ptr(self._n), self._optp(), _ptr(mean), _ptr(cov), _ptr(self._info),
                _ptr(ws), nbytes, _stream()))
            self._mark_end(ev)
            del ws
        self._mean_ylm, self._cov_ylm = mean, cov

    @property
    def mean_ylm(self):
        """sp.py:420-426."""
        self._compute_moments()
        return self._out(self._cut(self._mean_ylm, (1,)))

    @property
    def cov_ylm(self):
        """sp.py:428-434."""
        self._compute_moments()
        return self._out(self._cut(self._cov_ylm, (1, 2)))

    @property
    def cho_cov_ylm(self):
        """sp.py:436-441 (lower Cholesky factor of ``cov_ylm``)."""
        self._compute_moments()
        if self._cho_cov_ylm is None:
            with torch.cuda.device(self.device):
                cov = self._cov_ylm
                if self._nylm < 256:     # embedded lower degree: unit diagonal on the padded block
                    cov = cov.clone()
                    cov[:, self._nylm:, self._nylm:] += torch.eye(256 - self._nylm, dtype=torch.float64,
                                                                  device=self.device)
                L = torch.empty_like(cov)
                info = torch.zeros(self._B, dtype=torch.int32, device=self.device)
                _lib.check(self._lib.spb_cho_cov_ylm(self._ctx.handle, self._B, _ptr(cov),
                                                     _ptr(L), _ptr(info), _stream()))
                bad = (info & 1) != 0
                L = torch.where(bad[:, None, None], torch.full_like(L, float("nan")), L)
            self._cho_cov_ylm = L
        return self._out(self._cut(self._cho_cov_ylm, (1, 2)))

    def sample_ylm(self, t=None, nsamples=1, u=None, generator=None):
        """sp.py:489-509 (``t`` must be None: static surfaces).  ``u`` optionally supplies the
        standard-normal draws, shape ``(nylm, nsamples)`` as in the reference's
        ``random_normal(self.random, (nylm, nsamples))`` or ``(B, nylm, nsamples)``."""
        if t is not None:
            return self._sample_ylm_temporal(t, nsamples, u, generator)
        self.cho_cov_ylm
        L = self._cho_cov_ylm          # (B, 256, 256), padded at degrees below 15
        B, ny = self._B, self._nylm
        with torch.cuda.device(self.device):
            if u is None:
                un = torch.zeros(B, nsamples, 256, dtype=torch.float64, device=self.device)
                un[:, :, :ny] = torch.randn(B, nsamples, ny, dtype=torch.float64, device=self.device,
                                            generator=generator)
            else:
                un = torch.as_tensor(u, dtype=torch.float64).to(self.device)
                nsamples = un.shape[-1]
                if un.ndim == 2:
                    un = un[None].expand(B, un.shape[0], nsamples)
                un = self._pad_ylm(un.transpose(1, 2).contiguous(), 2)
            y = torch.empty(B, nsamples, 256, dtype=torch.float64, device=self.device)
            _lib.check(self._lib.spb_sample_ylm(self._ctx.handle, B, nsamples, _ptr(self._mean_ylm),
                                                _ptr(L.contiguous()), _ptr(un.contiguous()), _ptr(y),
                                                _stream()))
        return self._out(self._cut(y, (2,)))

    # ------------------------------------------------------------------ flux operator / design
    def _u(self, u):
        u = torch.as_tensor(defaults["u"] if u is None else u, dtype=torch.float64).reshape(-1)
        if self._udeg == 0:
            return torch.zeros(2, dtype=torch.float64, device=self.device)
        if u.numel() < self._udeg:
            raise ValueError("Vector `u` has the wrong size. Expected %d, got %d." %
                             (self._udeg, u.numel()))
        return u[: self._udeg].to(self.device).contiguous()

    def _rTA1(self, u):
        """Flux operator row vector for limb darkening ``u`` (a13), cached per process object for
        host-resident ``u`` (it only depends on ``u``; keyed by value, so no device sync)."""
        key = None
        if not (isinstance(u, torch.Tensor) and u.is_cuda):
            uh = np.asarray(defaults["u"] if u is None else
                            (u.detach().cpu().numpy() if isinstance(u, torch.Tensor) else u),
                            dtype=np.float64).reshape(-1)
            key = tuple(uh.tolist())
            if key in self._rTA1_cache:
                return self._rTA1_cache[key]
        ud = self._u(u)
        out = torch.empty(256, dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.spb_flux_operator(self._ctx.handle, 1, _ptr(ud), _ptr(out),
                                                   _stream()))
        if key is not None:
            self._rTA1_cache[key] = out
        return out

    def _t(self, t):
        return torch.as_tensor(t, dtype=torch.float64).to(self.device).reshape(-1).contiguous()

    _udt_cache = None

    def _uniform_dt(self, t):
        """Spacing of equally spaced time stamps (``t_k = t_0 + k dt`` to 4e-12 of a step, e.g. any
        ``linspace`` / fixed-cadence grid), else 0: the marginal assembly then tabulates the covariance
        interpolant instead of evaluating it per entry (``spb_noise_model.uniform_dt``).  Host arrays are
        checked with NumPy; device tensors once per (storage, length, version) with one reduction."""
        if isinstance(t, torch.Tensor) and t.is_cuda:
            key = (t.data_ptr(), t.numel(), t._version)
            if self._udt_cache is not None and self._udt_cache[0] == key:
                return self._udt_cache[1]
            tt = t.detach().reshape(-1).to(torch.float64)
            n = tt.numel()
            if n < 3:
                return 0.0
            dt = (tt[-1] - tt[0]) / (n - 1)
            dev_ = (tt - (tt[0] + dt * torch.arange(n, dtype=torch.float64, device=tt.device))).abs().max()
            dt, dev_ = float(dt), float(dev_)
            out = dt if (dt > 0.0 and dev_ <= 4e-12 * dt) else 0.0
            self._udt_cache = (key, out)
            return out
        ta = np.asarray(t, dtype=np.float64).reshape(-1)
        n = ta.size
        if n < 3:
            return 0.0
        dt = (ta[-1] - ta[0]) / (n - 1)
        if not dt > 0.0:
            return 0.0
        return float(dt) if np.max(np.abs(ta - (ta[0] + dt * np.arange(n)))) <= 4e-12 * dt else 0.0

    def _inc(self, i):
        if not (isinstance(i, torch.Tensor) and i.is_cuda):
            _check_bounds("i", np.asarray(i, dtype=np.float64) * np.pi / 180, 0, 0.5 * np.pi)
        it = torch.as_tensor(i, dtype=torch.float64).to(self.device).reshape(-1) * (math.pi / 180)
        return it.contiguous()

    def design_matrix(self, t, i=defaults["i"], p=defaults["p"], u=None):
        """flux.py:345-350: ``A (nt, nylm)``, or ``(I, nt, nylm)`` for a vector of inclinations."""
        A = self._cut(self._design_full(t, i, p, u), (2,))
        return A if _is_batched(i) else A[0]

    def _design_full(self, t, i, p, u):
        """The degree-15 design matrix ``(I, nt, 256)`` (a lower degree is its leading block)."""
        t = self._t(t)
        inc = self._inc(i)
        _check_bounds("p", p, 0, np.inf)
        return self._design(t, inc, p, self._rTA1(u))

    def _design(self, t, inc, p, rta1):
        """``A (I, nt, 256)`` of the device time stamps ``t`` at the inclinations ``inc`` [rad]."""
        lib, h, dev = self._lib, self._ctx.handle, self.device
        I, nt = inc.numel(), t.numel()
        with torch.cuda.device(dev):
            per = torch.full((I,), float(p), dtype=torch.float64, device=dev)
            A = torch.empty(I, nt, 256, dtype=torch.float64, device=dev)
            nbytes = lib.spb_design_matrix_workspace_bytes(h, I, nt)
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            _lib.check(lib.spb_design_matrix(h, I, nt, _ptr(t), _ptr(inc), _ptr(per), _ptr(rta1), 0,
                                             _ptr(A), _ptr(ws), nbytes, _stream()))
        return A

    # ------------------------------------------------------------------ flux mean / covariance
    def _curves(self, flux, baseline_mean, baseline_var, nt, M=None):
        """The light-curve inputs of one call, on the device: ``(f, per_element, M, bm, bvar)`` with
        ``f`` of shape ``(B, M, nt)`` when ``per_element``, else ``(1, M, nt)``; ``bm`` a scalar or
        ``(B,)``; ``bvar`` a scalar, ``(B,)`` or ``(nt, nt)``, or None for zero.  ``M=1``: the
        single light curve ``(nt,)`` of ``predict`` and the conditional samplers."""
        dev, B = self.device, self._B
        f = torch.as_tensor(flux, dtype=torch.float64).to(dev)
        if M == 1:
            if f.numel() != nt:
                raise ValueError("flux must have shape (nt,)")
            f = f.reshape(1, nt)
        elif f.ndim == 1:
            f = f[None]
        per_element = f.ndim == 3
        if per_element and f.shape[0] != B:
            raise ValueError("per-element flux must have shape (B, M, nt)")
        if f.shape[-1] != nt:
            raise ValueError("flux must have shape (nt,), (M, nt) or (B, M, nt)")
        f = (f if per_element else f[None]).contiguous()
        bm = torch.as_tensor(baseline_mean, dtype=torch.float64).to(dev).contiguous()
        if bm.ndim == 1 and bm.numel() != B:
            raise ValueError("a 1-D baseline_mean must have one entry per batch element")
        bvar = None
        if isinstance(baseline_var, (torch.Tensor, np.ndarray)) or baseline_var != 0.0:
            bvar = torch.as_tensor(baseline_var, dtype=torch.float64).to(dev).contiguous()
            # extension: one baseline variance per batch element (the free `v` of
            # calibrate/log_prob.py:70-74)
            if bvar.ndim == 1 and bvar.numel() != B:
                raise ValueError("a 1-D baseline_var must have one entry per batch element")
            if bvar.ndim > 1 and tuple(bvar.shape) != (nt, nt):
                raise ValueError("baseline_var must be a scalar or an (nt, nt) matrix")
        return f, per_element, f.shape[1], bm, bvar

    def _noise_model(self, nt, data_cov, baseline_var, keep, lower_only=False, uniform_dt=0.0):
        """spb_noise_model of one assembly of ``nt`` time stamps; ``uniform_dt`` is their spacing
        (``_spacing``; 0 takes the general kernel), ``baseline_var`` as ``_curves`` returns it.
        ``keep`` collects the device buffers it points to."""
        nm = _lib.NoiseModel()
        nm.lower_only = 1 if lower_only else 0
        nm.defer = 0
        nm.normalized = 1 if self._normalized else 0
        nm.normalization_order = self._normN
        nm.normalization_zmax = self._normzmax
        nm.data_cov = None
        nm.baseline_var = None
        nm.data_stride = 0
        nm.base_stride = 0
        nm.temporal_kind = self._tkind
        nm.uniform_dt = float(uniform_dt)
        nm.tau = self._tau.data_ptr() if self._tkind else None
        nm.tau_stride = 1 if self._tkind else 0
        if data_cov is not None:
            d = torch.as_tensor(data_cov, dtype=torch.float64).to(self.device).contiguous()
            if d.ndim == 0:
                nm.data_kind, d = 0, d.reshape(1)
            elif d.ndim == 1:
                if d.numel() != nt:
                    raise ValueError("data_cov vector has the wrong length")
                nm.data_kind = 1
            else:
                if tuple(d.shape) != (nt, nt):
                    raise ValueError("data_cov matrix has the wrong shape")
                nm.data_kind = 2
            keep.append(d)
            nm.data_cov = d.data_ptr()
        if baseline_var is not None:
            bv = torch.as_tensor(baseline_var, dtype=torch.float64).to(self.device).contiguous()
            if bv.ndim == 0:
                nm.base_kind, bv = 0, bv.reshape(1)
            elif bv.ndim == 1:
                nm.base_kind, nm.base_stride = 0, 1
            else:
                nm.base_kind = 2
            keep.append(bv)
            nm.baseline_var = bv.data_ptr()
        return nm

    def _flux_cov(self, t, inc, p, rta1, marg, udt, data_cov, baseline_var, ldk, lower_only=False,
                  defer=False):
        """GP mean (scalar per element) and the (noise-augmented) covariance of every batch element.
        Returns ``(gp_mean, K, z, coef, affine)``: ``coef`` is the marginal kernel table ``(B, 4,
        covpts + 1)`` (None in the conditional branch).  With ``defer`` (marginal branch, scalar /
        per-point noise terms) the covariance is left raw and ``affine`` is the ``spb_cholesky_lnlike_affine``
        argument that applies the normalisation + noise inside the Cholesky kernel; else it is None."""
        lib, h = self._lib, self._ctx.handle
        B, nt = self._B, t.numel()
        dev = self.device
        keep = []
        nm = self._noise_model(nt, data_cov, baseline_var, keep, lower_only and marg, udt)
        defer_req = bool(defer)
        defer = bool(defer and marg and lower_only and nm.data_kind != 2 and nm.base_kind != 2)
        nm.defer = 1 if defer else 0
        gp_mean = torch.empty(B, dtype=torch.float64, device=dev)
        K = torch.empty(B, nt, ldk, dtype=torch.float64, device=dev)
        z = torch.zeros(B, dtype=torch.float64, device=dev)
        nb_as = lib.spb_assemble_workspace_bytes(h, B, nt)
        ws_as = torch.empty(nb_as, dtype=torch.uint8, device=dev)
        coef = None
        if marg:
            nc = self._covpts + 1
            var = torch.empty(B, dtype=torch.float64, device=dev)
            coef = torch.empty(B, 4, nc, dtype=torch.float64, device=dev)
            nb = lib.spb_flux_marginal_workspace_bytes(h, B)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            ev = self._mark("flux_marginal")
            _lib.check(lib.spb_flux_marginal(h, B, _ptr(self._mean_ylm), _ptr(self._cov_ylm), _ptr(rta1),
                                             self._covpts, _ptr(gp_mean), _ptr(var), _ptr(coef),
                                             _ptr(ws), nb, _stream()))
            self._mark_end(ev)
            ev = self._mark("assemble")
            _lib.check(lib.spb_assemble_marginal(h, B, nt, _ptr(t), float(p), self._covpts,
                                                 _ptr(coef), _ptr(var), _ptr(gp_mean),
                                                 ctypes.byref(nm), _ptr(K), ldk, _ptr(z),
                                                 _ptr(self._info), _ptr(ws_as), nb_as, _stream()))
            self._mark_end(ev)
        else:
            A = self._design(t, inc, p, rta1)
            nb = lib.spb_flux_conditional_workspace_bytes(h, B, nt)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            # log-likelihood path of an unnormalised, static process: only the lower triangle is needed and
            # the noise terms are added inside the Cholesky kernel's loads (no read-modify-write pass)
            defer_c = bool(defer_req and lower_only and not self._normalized and not self._tkind
                           and nm.data_kind != 2 and nm.base_kind != 2)
            fc = lib.spb_flux_conditional_lower if defer_c else lib.spb_flux_conditional
            _lib.check(fc(h, B, nt, _ptr(A), 0 if A.shape[0] == 1 else nt * 256, _ptr(self._mean_ylm),
                          _ptr(self._cov_ylm), _ptr(gp_mean), _ptr(K), ldk, _ptr(ws), nb, _stream()))
            if defer_c:
                defer = True
            elif self._tkind:   # sp.py:697-698
                _lib.check(lib.spb_temporal_scale(h, B, nt, nt, _ptr(t), _ptr(t), self._tkind,
                                                  _ptr(self._tau), 1, None, 0, _ptr(K), ldk, nt * ldk,
                                                  _stream()))
            if not defer_c:
                _lib.check(lib.spb_assemble_conditional(h, B, nt, _ptr(gp_mean), ctypes.byref(nm),
                                                        _ptr(K), ldk, _ptr(z), _ptr(self._info),
                                                        _ptr(ws_as), nb_as, _stream()))
        affine = None
        if defer:
            affine = _lib.Affine()
            if self._normalized:
                qp, sp_ = ctypes.c_void_p(), ctypes.c_void_p()
                lib.spb_assemble_workspace_layout(B, nt, _ptr(ws_as), ctypes.byref(qp),
                                                  ctypes.byref(sp_))
                affine.q, affine.scal = qp, sp_
            affine.diag = nm.data_cov
            affine.diag_kind = nm.data_kind
            affine.diag_stride = 0
            affine.offset = nm.baseline_var
            affine.offset_stride = nm.base_stride
            affine.keep = (keep, ws_as)   # the device buffers it points into
        return gp_mean, K, z, coef, affine

    # ---- batch chunking: every batched method runs its body on views of batch chunks
    def _cov_bytes(self, nt, ldk):
        """Device bytes per element of ``log_likelihood`` / ``mean`` / ``cov``: K, the moments and
        the digit planes of the INT8 path, which live next to K."""
        per = nt * ldk * 8 + 4 * 256 * 256 * 8
        code = self._ctx.i8_planes(nt, self._B)   # 7 | 8 | 77 | 78 | 87: the first digit is the plane count
        if code:
            per += (code // 10 if code > 10 else code) * (nt + 64) * (nt + 64)
        return per

    def _chunks(self, per):
        """Batch chunks ``(b0, b1)`` at ``per`` device bytes per element: as few as the memory bound
        allows (96 GB by default: the B200 has 180 GB), and at most 65535 elements each (the assembly
        and GEMM kernels carry the batch in grid.y), of equal size: the Cholesky kernel claims
        matrices dynamically, so one long launch has a shorter tail than several short ones."""
        step = max(1, min(self._B, self._max_chunk_bytes // per, 65535))
        nchunks = -(-self._B // step)
        step = -(-self._B // nchunks)
        return [(b0, min(self._B, b0 + step)) for b0 in range(0, self._B, step)]

    def _sub(self, b0, b1):
        """A view of batch elements b0:b1 as a process of its own (moments already computed)."""
        sub = object.__new__(type(self))
        sub.__dict__.update(self.__dict__)
        sub._B, sub._batched = b1 - b0, True
        for k in ("_r", "_a", "_b", "_c", "_n", "_tau", "_dr", "_mean_ylm", "_cov_ylm", "_info"):
            v = getattr(self, k, None)
            setattr(sub, k, None if v is None else v[b0:b1])
        sub._cho_cov_ylm = None if self._cho_cov_ylm is None else self._cho_cov_ylm[b0:b1]
        if getattr(self, "_mu_sigma", None) is not None:
            sub._mu_sigma = (self._mu_sigma[0][b0:b1], self._mu_sigma[1][b0:b1])
        return sub

    def _batch(self, per, run, **elem):
        """``run(gp, **elem)`` over the chunks of the batch (``_chunks(per)``), ``gp`` the view of a
        chunk (the process itself when one chunk holds the batch).  ``elem`` are the per-element
        arguments, sliced to the chunk when they carry a batch axis.  Returns the outputs of the
        chunks concatenated along the batch axis."""
        bounds = self._chunks(per)
        if len(bounds) == 1:
            return run(self, **elem)
        outs = []
        for b0, b1 in bounds:
            kw = {k: v[b0:b1] if getattr(v, "ndim", None) == _BATCH_NDIM[k] and v.shape[0] == self._B
                  else v for k, v in elem.items()}
            outs.append(run(self._sub(b0, b1), **kw))
        if isinstance(outs[0], tuple):
            return tuple(torch.cat(o) for o in zip(*outs))
        return torch.cat(outs)

    def _spacing(self, t):
        """``spb_noise_model.uniform_dt`` of the time stamps ``t`` (0 with ``SPB200_NO_UNIFORM_T`` set),
        also left in ``_udt`` as a record of the last call, as ``_z`` is."""
        udt = 0.0 if os.environ.get("SPB200_NO_UNIFORM_T") is not None else self._uniform_dt(t)
        self._udt = udt
        return udt

    def _prep(self, t, i, p, u, marginalize_over_inclination):
        marg = self._marginalize_over_inclination if marginalize_over_inclination is None \
            else bool(marginalize_over_inclination)
        self._compute_moments()
        t = self._t(t)
        inc = self._inc(i)
        if inc.numel() not in (1, self._B):
            raise ValueError("`i` must be a scalar or have one entry per batch element")
        _check_bounds("p", p, 0, np.inf)
        rta1 = self._rTA1(u)
        return marg, t, inc, rta1

    def mean(self, t, i=defaults["i"], p=defaults["p"], u=None, marginalize_over_inclination=None):
        """sp.py:643-672."""
        udt = self._spacing(t)
        marg, t, inc, rta1 = self._prep(t, i, p, u, marginalize_over_inclination)
        nt = t.numel()
        if self._normalized:
            out = torch.zeros(self._B, nt, dtype=torch.float64, device=self.device)
            return self._out(out)
        ldk = nt + (nt & 1)
        with torch.cuda.device(self.device):
            g = self._batch(self._cov_bytes(nt, ldk),
                            lambda gp, inc: gp._flux_cov(t, inc, p, rta1, marg, udt, None, None, ldk)[0],
                            inc=inc)
        return self._out(g[:, None].expand(self._B, nt).contiguous())

    def cov(self, t, i=defaults["i"], p=defaults["p"], u=None, marginalize_over_inclination=None):
        """sp.py:674-703: the (normalised, if requested) GP flux covariance, ``(nt, nt)`` or
        ``(B, nt, nt)``."""
        udt = self._spacing(t)
        marg, t, inc, rta1 = self._prep(t, i, p, u, marginalize_over_inclination)
        nt = t.numel()
        ldk = nt + (nt & 1)

        def run(gp, inc):
            _, K, z, _, _ = gp._flux_cov(t, inc, p, rta1, marg, udt, None, None, ldk)
            return K[:, :, :nt], z

        with torch.cuda.device(self.device):
            K, self._z = self._batch(self._cov_bytes(nt, ldk), run, inc=inc)
        return self._out(K)

    # ------------------------------------------------------------------ log likelihood
    def log_likelihood(self, t, flux, data_cov, i=defaults["i"], p=defaults["p"], u=None,
                       baseline_mean=defaults["baseline_mean"],
                       baseline_var=defaults["baseline_var"], marginalize_over_inclination=None,
                       return_grad=False, method="dense"):
        """sp.py:1052-1188.  ``flux`` is ``(nt,)`` or ``(M, nt)`` (M light curves sharing period,
        limb darkening, inclination and noise, scored jointly); returns a scalar, or ``(B,)`` for a
        batch of hyperparameter samples.  Extension: ``flux`` of shape ``(B, M, nt)`` gives every
        batch element its own light curve(s) (the light-curve x sample x inclination batches of
        calibrate/inclination.py:63-74).

        ``method``: ``"dense"`` (default) factorises the ``(nt, nt)`` covariance of every element, as
        the reference does.  ``"lowrank"`` evaluates the same conditional-branch likelihood through its
        rank-31 form (DESIGN.md section 4.6): time and memory linear in ``nt``, so light curves of
        1e5-1e6 points fit.  It covers the static process conditional on inclination with a scalar or
        ``(nt,)`` positive ``data_cov`` and a scalar or ``(B,)`` ``baseline_var``, and raises
        ``ValueError`` otherwise."""
        lowrank = self._lowrank_checks(method, t, data_cov, baseline_var, marginalize_over_inclination)
        if return_grad:
            return self.log_likelihood_and_grad(
                t, flux, data_cov, i=i, p=p, u=u, baseline_mean=baseline_mean,
                baseline_var=baseline_var, marginalize_over_inclination=marginalize_over_inclination,
                method=method)
        if lowrank:
            return self._log_likelihood_lowrank(t, flux, data_cov, i, p, u, baseline_mean, baseline_var)
        udt = self._spacing(t)
        marg, t, inc, rta1 = self._prep(t, i, p, u, marginalize_over_inclination)
        nt = t.numel()
        ldk = nt + (nt & 1)
        f, _, _, bm, bvar = self._curves(flux, baseline_mean, baseline_var, nt)
        # white-noise floor of K (a lower bound of its smallest eigenvalue): scales the right-hand-side
        # digit planes of the INT8 path when the noise was already added by the assembly kernels
        lam_min, noise_free = 0.0, False
        if isinstance(data_cov, (int, float)) or (
                isinstance(data_cov, (torch.Tensor, np.ndarray)) and data_cov.ndim == 0):
            lam_min = float(data_cov)
            noise_free = not (lam_min > 0.0)   # no white-noise floor: nothing bounds the solved rows
        with torch.cuda.device(self.device):
            lnlike, self._z = self._batch(
                self._cov_bytes(nt, ldk),
                lambda gp, inc, f, bm, bvar: gp._log_likelihood_dense(
                    t, inc, p, rta1, marg, udt, f, bm, data_cov, bvar, lam_min, noise_free),
                inc=inc, f=f, bm=bm, bvar=bvar)
        return self._out(lnlike)

    def _log_likelihood_dense(self, t, inc, p, rta1, marg, udt, f, bm, data_cov, bvar, lam_min,
                              noise_free):
        """``(lnlike, z)`` of every batch element: assembly, then one of the Cholesky kernels."""
        dev, Bc = self.device, self._B
        nt, M = t.numel(), f.shape[1]
        ldk = nt + (nt & 1)
        lib, h = self._lib, self._ctx.handle
        gp_mean, K, z, _, affine = self._flux_cov(t, inc, p, rta1, marg, udt, data_cov, bvar, ldk,
                                                  lower_only=True, defer=True)
        lnlike = torch.empty(Bc, dtype=torch.float64, device=dev)
        # r = flux - (gp_mean + baseline_mean)  (sp.py:1157-1161); normalised: mean == 0
        resid = torch.zeros(Bc, M, ldk, dtype=torch.float64, device=dev)
        bmc = bm[:, None, None] if bm.ndim == 1 else bm   # (B,) baseline means
        if self._normalized:
            resid[:, :, :nt] = f - bmc
        else:
            resid[:, :, :nt] = f - (gp_mean[:, None, None] + bmc)
        ev = self._mark("cholesky")
        if Bc == 1 and M >= 64:
            # one factorisation + many right-hand sides (ensemble of light curves sharing
            # K): factor on one CTA, then spread the RHS rows over the whole GPU
            logdet = torch.empty(1, dtype=torch.float64, device=dev)
            quad = torch.empty(M, dtype=torch.float64, device=dev)
            if affine is not None:
                _lib.check(lib.spb_cholesky_lnlike_affine(
                    h, 1, nt, _ptr(K), ldk, nt * ldk, ctypes.byref(affine), 0, None, ldk, 0,
                    None, None, _ptr(logdet), _ptr(self._info), _stream()))
            else:
                _lib.check(lib.spb_cholesky_lnlike(
                    h, 1, nt, _ptr(K), ldk, nt * ldk, 0, None, ldk, 0, None, None,
                    _ptr(logdet), _ptr(self._info), _stream()))
            _lib.check(lib.spb_cholesky_solve_rows(h, nt, _ptr(K), ldk, M, _ptr(resid), ldk,
                                                   _ptr(quad), _stream()))
            ll = -0.5 * quad.sum() - M * logdet[0] - 0.5 * nt * M * math.log(2 * math.pi)
            flagged = (self._info != 0) | torch.isnan(ll)
            lnlike[:] = torch.where(flagged, torch.full_like(ll, -float("inf")), ll)
        elif self._ctx.i8_planes(nt, Bc) and nt > 64 and not noise_free and (
                (affine is not None and affine.diag) or lam_min > 0.0):
            # factorisation on the INT8 tensor cores (K is only read; potrf_i8.cuh)
            planes = self._ctx.i8_planes(nt, Bc)
            nb_i8 = lib.spb_cholesky_i8_workspace_bytes(Bc, nt, M, planes)
            ws_i8 = torch.empty(nb_i8, dtype=torch.uint8, device=dev)
            _lib.check(lib.spb_cholesky_lnlike_i8(
                h, Bc, nt, _ptr(K), ldk, nt * ldk,
                ctypes.byref(affine) if affine is not None else None, M, _ptr(resid), ldk,
                M * ldk, _ptr(lnlike), None, None, _ptr(self._info), planes,
                0.0 if affine is not None and affine.diag else lam_min, _ptr(ws_i8), nb_i8,
                _stream()))
            del ws_i8
        elif affine is not None:
            _lib.check(lib.spb_cholesky_lnlike_affine(
                h, Bc, nt, _ptr(K), ldk, nt * ldk, ctypes.byref(affine), M, _ptr(resid), ldk,
                M * ldk, _ptr(lnlike), None, None, _ptr(self._info), _stream()))
        else:
            _lib.check(lib.spb_cholesky_lnlike(
                h, Bc, nt, _ptr(K), ldk, nt * ldk, M, _ptr(resid), ldk, M * ldk,
                _ptr(lnlike), None, None, _ptr(self._info), _stream()))
        self._mark_end(ev)
        return lnlike, z

    def _log_likelihood_lowrank(self, t, flux, data_cov, i, p, u, baseline_mean, baseline_var):
        """``log_likelihood(method="lowrank")``: include/spb200.h spb_lowrank_*."""
        udt = self._spacing(t)
        _, t, inc, rta1 = self._prep(t, i, p, u, False)
        nt = t.numel()
        dev, B = self.device, self._B
        f, per_element, M, bm, bvar = self._curves(flux, baseline_mean, baseline_var, nt)
        keep = []
        nm = self._noise_model(nt, data_cov, bvar, keep, uniform_dt=udt)
        lib, h = self._lib, self._ctx.handle
        I = inc.numel()
        lnlike = torch.empty(B, dtype=torch.float64, device=dev)
        z = torch.zeros(B, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            Binc, Q, R, aux = self._lowrank_basis(t, inc, rta1, p, nm)
            ev = self._mark("lowrank_lnlike")
            nb = lib.spb_lowrank_lnlike_workspace_bytes(h, B, M, nt)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            _lib.check(lib.spb_lowrank_lnlike(
                h, B, nt, _ptr(Binc), 0 if I == 1 else 32 * 256, _ptr(self._mean_ylm), _ptr(self._cov_ylm),
                _ptr(Q), _ptr(R), _ptr(aux), ctypes.byref(nm), M, _ptr(f), nt, M * nt if per_element else 0,
                _ptr(bm), 1 if bm.ndim == 1 else 0, _ptr(lnlike), None, None, _ptr(z), _ptr(self._info),
                _ptr(ws), nb, _stream()))
            self._mark_end(ev)
            del ws, keep
        self._z = z
        return self._out(lnlike)

    def _lowrank_checks(self, method, t, data_cov, baseline_var, marginalize_over_inclination):
        """``method`` of ``log_likelihood`` / ``predict`` / ``sample_conditional``: False for ``"dense"``, True
        for ``"lowrank"`` once the inputs are found to be covered by the rank-31 form (ValueError otherwise)."""
        if method not in ("dense", "lowrank"):
            raise ValueError("unknown method %r: expected 'dense' or 'lowrank'" % (method,))
        if method == "dense":
            return False
        marg = self._marginalize_over_inclination if marginalize_over_inclination is None \
            else bool(marginalize_over_inclination)
        if marg:
            raise ValueError("method='lowrank' needs marginalize_over_inclination=False: the marginalised "
                             "covariance is the cubic interpolant of flux.py:256-276, which is not low-rank")
        if self._tkind:
            raise ValueError("method='lowrank' does not cover time-variable surfaces (tau): the temporal "
                             "kernel makes the covariance full-rank")
        dc = data_cov if isinstance(data_cov, torch.Tensor) else np.asarray(data_cov, dtype=np.float64)
        if dc.ndim > 1:
            raise ValueError("method='lowrank' needs a scalar or (nt,) data_cov, not a full matrix")
        if not (isinstance(dc, torch.Tensor) and dc.is_cuda):
            if not np.all(np.asarray(dc.cpu() if isinstance(dc, torch.Tensor) else dc) > 0.0):
                raise ValueError("method='lowrank' needs a positive data_cov (it whitens with D^-1/2)")
        if isinstance(baseline_var, (torch.Tensor, np.ndarray)) and baseline_var.ndim > 1:
            raise ValueError("method='lowrank' needs a scalar or (B,) baseline_var, not a full matrix")
        if _nt(t) < 31:
            raise ValueError("method='lowrank' needs nt >= 31 time stamps (the rank of the phase basis)")
        return True

    def _lowrank_basis(self, t, inc, rta1, p, nm):
        """B_inc (I, 32, 256) and the thin QR of the whitened phase basis, Q (nt, 32), R (32, 32), aux (65)."""
        lib, h, dev = self._lib, self._ctx.handle, self.device
        I, nt = inc.numel(), t.numel()
        ev = self._mark("lowrank_inclination")
        Binc = torch.empty(I, 32, 256, dtype=torch.float64, device=dev)
        nb = lib.spb_lowrank_inclination_workspace_bytes(h, I)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.check(lib.spb_lowrank_inclination(h, I, _ptr(inc), _ptr(rta1), 0, _ptr(Binc), _ptr(ws), nb,
                                               _stream()))
        self._mark_end(ev)
        ev = self._mark("lowrank_basis")
        Q = torch.empty(nt, 32, dtype=torch.float64, device=dev)
        R = torch.empty(32, 32, dtype=torch.float64, device=dev)
        aux = torch.empty(65, dtype=torch.float64, device=dev)
        nb = lib.spb_lowrank_basis_workspace_bytes(h, nt)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.check(lib.spb_lowrank_basis(h, nt, _ptr(t), float(p), nm.data_kind, ctypes.c_void_p(nm.data_cov),
                                         _ptr(Q), _ptr(R), _ptr(aux), _ptr(ws), nb, _stream()))
        self._mark_end(ev)
        return Binc, Q, R, aux

    # ------------------------------------------------------------------ SURVEY 8(f) rank 4: gradient
    def log_likelihood_and_grad(self, t, flux, data_cov, i=defaults["i"], p=defaults["p"], u=None,
                                baseline_mean=defaults["baseline_mean"],
                                baseline_var=defaults["baseline_var"],
                                marginalize_over_inclination=None, rel_step=1e-4, method="dense"):
        """``log_likelihood`` and its gradient with respect to the hyperparameters the process was
        built from -- ``r`` [deg], ``a`` and ``b`` (or ``mu`` and ``sigma`` [deg]), ``c``, ``n`` -- as
        ``(lnlike, {"r": ..., "a" | "mu": ..., "b" | "sigma": ..., "c": ..., "n": ...})``, one value
        per batch element.  What the reference obtains by Theano reverse mode (``tt.grad`` of
        sp.py:1052-1188 through ops/include/latitude.h:22-173, eigh.h:19-65, wigner.h:345-404,
        465-531, math.py:40-72; checked there with ``verify_grad`` at 1e-4, tests/test_lnlike.py:105-136).

        Here: the Ylm moments move along their ANALYTIC tangents (``spb_ylm_moments_grad``: derivative
        lanes of the Beta moments, profile derivative, monomial scalings in c and n; exact because
        the rest of the moment pipeline is linear / quadratic), and the log-likelihood of the ten
        displaced moment sets is evaluated by the same kernels in ONE batch of 11 B elements; the
        central difference along each tangent has a relative truncation error of ``rel_step**2``
        (the flux-side likelihood is smooth in the moments) and no eigen-solver noise, because the
        displaced sets share the base eigen-problem up to the smooth perturbation.  Measured against
        the analytic oracle (oracle/sp_oracle_grad.py): <= 1e-6 relative.  ``method`` selects the
        likelihood evaluation of the 11 B elements, as in ``log_likelihood``."""
        if self._dr is not None or self._time_variable or not hasattr(self, "_r") or self._r is None:
            raise NotImplementedError("gradients: delta spot-size prior, static surfaces, a single "
                                      "process (not a sum)")
        dev, B = self.device, self._B
        lib, h = self._lib, self._ctx.handle
        with torch.cuda.device(dev):
            mean = torch.empty(11 * B, 256, dtype=torch.float64, device=dev)
            cov = torch.empty(11 * B, 256, 256, dtype=torch.float64, device=dev)
            eps = torch.empty(5, B, dtype=torch.float64, device=dev)
            info = torch.zeros(B, dtype=torch.int32, device=dev)
            nb = lib.spb_ylm_moments_grad_workspace_bytes(h, B)
            ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            ev = self._mark("moments_grad")
            _lib.check(lib.spb_ylm_moments_grad(h, B, _ptr(self._r), _ptr(self._a), _ptr(self._b),
                                                _ptr(self._c), _ptr(self._n), self._optp(),
                                                float(rel_step),
                                                _ptr(mean), _ptr(cov), _ptr(eps), _ptr(info), _ptr(ws),
                                                nb, _stream()))
            self._mark_end(ev)
            del ws
            # an 11 B-wide process over the displaced moments; everything else is shared
            big = self._sub(0, B)
            big._B = 11 * B
            big._mean_ylm, big._cov_ylm, big._cho_cov_ylm = mean, cov, None
            big._info = info.repeat(11).contiguous()

            def tile(x, per_dim):
                """Per-element arguments (leading dimension B) are repeated for the 11 variants."""
                if isinstance(x, (torch.Tensor, np.ndarray)):
                    xt = torch.as_tensor(x, dtype=torch.float64).to(dev)
                    if xt.ndim == per_dim and xt.shape[0] == B and B > 1:
                        return xt.repeat((11,) + (1,) * (xt.ndim - 1))
                    return xt
                return x

            ll_all = big.log_likelihood(
                t, tile(flux, 3), data_cov, i=tile(i, 1), p=p, u=u, baseline_mean=tile(baseline_mean, 1),
                baseline_var=tile(baseline_var, 1),
                marginalize_over_inclination=marginalize_over_inclination, method=method).reshape(11, B)
            self._z = None if big._z is None else big._z[:B]
            self._info = big._info[:B].clone()
            ll = ll_all[0]
            g = (ll_all[1::2] - ll_all[2::2]) / (2.0 * eps)          # (5, B): r, a, b, c, n
            ok = torch.isfinite(ll)[None, :] & torch.isfinite(ll_all[1:]).reshape(5, 2, B).all(dim=1)
            g = torch.where(torch.isfinite(ll)[None, :].expand(5, B), g, torch.zeros_like(g))
            g = torch.where(ok | ~torch.isfinite(ll)[None, :], g, torch.full_like(g, float("nan")))
            grad = {"r": self._out(g[0]), "c": self._out(g[3]), "n": self._out(g[4])}
            if getattr(self, "_mu_sigma", None) is None:
                grad["a"], grad["b"] = self._out(g[1]), self._out(g[2])
            else:
                # (a, b) = gauss2beta(mu, sigma), latitude.py:14-77: elementwise 2 x 2 Jacobian
                mu = self._mu_sigma[0].detach().clone().requires_grad_(True)
                sg = self._mu_sigma[1].detach().clone().requires_grad_(True)
                a_, b_ = gauss2beta(mu, sg)
                da = torch.autograd.grad(a_.sum(), (mu, sg), retain_graph=True)
                db = torch.autograd.grad(b_.sum(), (mu, sg))
                grad["mu"] = self._out(g[1] * da[0] + g[2] * db[0])
                grad["sigma"] = self._out(g[1] * da[1] + g[2] * db[1])
        return self._out(ll), grad

    # ------------------------------------------------------------------ SURVEY 8(f) rank 2
    def _factor_rows(self, K, n, ldk, rows=None, diag_add=None):
        """In-place batched Cholesky of ``K (Bq, n, ldk)`` (lower triangle read, ``L`` written over
        it; ``diag_add`` is added to the diagonal inside the kernel's loads); ``rows (Bq, M, ldr)``
        are replaced by ``L^-1 row`` (math.py:20-38 forward substitution).  Returns ``info``."""
        lib, h = self._lib, self._ctx.handle
        Bq = K.shape[0]
        info = torch.zeros(Bq, dtype=torch.int32, device=self.device)
        if rows is None:
            M, rp, ldr, rstride = 0, None, ldk, 0
        else:
            M, ldr = rows.shape[1], rows.shape[2]
            rp, rstride = _ptr(rows), M * ldr
        if diag_add is None:
            _lib.check(lib.spb_cholesky_lnlike(h, Bq, n, _ptr(K), ldk, n * ldk, M, rp, ldr, rstride,
                                               None, None, None, _ptr(info), _stream()))
        else:
            af = _lib.Affine()
            dg = torch.full((1,), float(diag_add), dtype=torch.float64, device=self.device)
            af.diag, af.diag_kind, af.diag_stride = dg.data_ptr(), 0, 0
            _lib.check(lib.spb_cholesky_lnlike_affine(h, Bq, n, _ptr(K), ldk, n * ldk,
                                                      ctypes.byref(af), M, rp, ldr, rstride, None,
                                                      None, None, _ptr(info), _stream()))
        return info

    def _gemm(self, batch, M, N, K, A, lda, sA, Bm, ldb, sB, C, ldc, sC, alpha=1.0, beta=0.0):
        """``C = alpha A Bm^T + beta C`` (spb_gemm_nt); tensors or raw device addresses."""
        ad = lambda x: ctypes.c_void_p(x) if isinstance(x, int) else _ptr(x)   # noqa: E731
        _lib.check(self._lib.spb_gemm_nt(self._ctx.handle, batch, M, N, K, float(alpha), ad(A), lda,
                                         sA, ad(Bm), ldb, sB, float(beta), ad(C), ldc, sC,
                                         _stream()))

    def _draw(self, mu, L, n, ld, nsamples, unit_normals, generator):
        """``mu[:, None] + L u`` for ``u ~ N(0, 1)`` of shape ``(n, nsamples)`` (or ``(B, n,
        nsamples)``), returned as ``(B, nsamples, n)``.  ``L (B, n, ld)`` must be clean lower."""
        B, dev = L.shape[0], self.device
        if unit_normals is None:
            un = torch.zeros(B, nsamples, ld, dtype=torch.float64, device=dev)
            un[:, :, :n] = torch.randn(B, nsamples, n, dtype=torch.float64, device=dev,
                                       generator=generator)
        else:
            u_ = torch.as_tensor(unit_normals, dtype=torch.float64).to(dev)
            if u_.ndim == 2:
                u_ = u_[None].expand(B, u_.shape[0], u_.shape[1])
            if u_.shape[1] != n:
                raise ValueError("unit normals must have shape (%d, nsamples)" % n)
            nsamples = u_.shape[2]
            un = torch.zeros(B, nsamples, ld, dtype=torch.float64, device=dev)
            un[:, :, :n] = u_.transpose(1, 2)
        out = mu[:, None, :].expand(B, nsamples, n).contiguous()
        self._gemm(B, nsamples, n, ld, un, ld, nsamples * ld, L, ld, n * ld, out, n, nsamples * n,
                   alpha=1.0, beta=1.0)
        return out

    def sample(self, t, i=defaults["i"], p=defaults["p"], u=None, nsamples=1, eps=defaults["eps"],
               unit_normals=None, generator=None, marginalize_over_inclination=None):
        """sp.py:729-765: draws from the prior over light curves, ``(nsamples, nt)`` (or
        ``(B, nsamples, nt)``).  ``unit_normals`` optionally supplies the reference's
        ``random_normal(self.random, (nt, nsamples))``."""
        udt = self._spacing(t)
        marg, t, inc, rta1 = self._prep(t, i, p, u, marginalize_over_inclination)
        nt = t.numel()
        ldk = nt + (nt & 1)

        def run(gp, inc, unit_normals):
            # eps I is the scalar "data covariance" of the assembly (added after the normalisation,
            # as sp.py:762 adds it to the output of cov())
            gp_mean, K, _, _, _ = gp._flux_cov(t, inc, p, rta1, marg, udt, float(eps), None, ldk)
            info = gp._factor_rows(K, nt, ldk)
            _lib.check(gp._lib.spb_tril(gp._ctx.handle, gp._B, nt, _ptr(K), ldk, nt * ldk, _stream()))
            if nt & 1:
                K[:, :, nt:] = 0.0
            mu = torch.zeros(gp._B, nt, dtype=torch.float64, device=gp.device)
            if not gp._normalized:
                mu += gp_mean[:, None]
            out = gp._draw(mu, K, nt, ldk, nsamples, unit_normals, generator)
            return torch.where(((info & 1) != 0)[:, None, None], torch.full_like(out, float("nan")), out)

        with torch.cuda.device(self.device):
            out = self._batch(_four_arrays(nt, nt), run, inc=inc, unit_normals=unit_normals)
        return self._out(out)

    def predict(self, t, flux, data_cov, t_sample=None, i=defaults["i"], p=defaults["p"], u=None,
                baseline_mean=defaults["baseline_mean"], baseline_var=defaults["baseline_var"],
                marginalize_over_inclination=None, method="dense", return_cov="full"):
        """sp.py:767-922: mean ``(nts,)`` and covariance ``(nts, nts)`` of the light-curve
        distribution conditioned on ``flux`` (leading ``B`` axis for batched hyperparameters).
        ``return_cov="diag"`` returns the predictive variance ``(nts,)`` (or ``(B, nts)``) in place of
        the matrix.  Extension: a ``(B,)`` ``baseline_mean`` gives every batch element its own.

        One augmented factorisation does the work: the rows ``[K(ts, t); y - mean]`` are appended
        to ``K(t, t)``, the Cholesky kernel returns ``V = (L^-1 K(t, ts))^T`` and ``w = L^-1 (y -
        mean)``, and ``mu = mean + V w``, ``K = K(ts, ts) - V V^T`` are two tensor-core GEMMs.

        ``method="lowrank"`` evaluates the same distribution through the rank-31 form of the conditional
        branch (DESIGN.md section 4.6): time and memory linear in ``nt`` and, with ``return_cov="diag"``,
        in ``nts``.  It covers what ``log_likelihood(method="lowrank")`` covers and raises ``ValueError``
        otherwise."""
        if self._normalized:
            raise NotImplementedError("Method not implemented when the flux is normalized.")
        if return_cov not in ("full", "diag"):
            raise ValueError("unknown return_cov %r: expected 'full' or 'diag'" % (return_cov,))
        lowrank = self._lowrank_checks(method, t, data_cov, baseline_var, marginalize_over_inclination)
        marg, t, inc, rta1, udt, ts, udt_s, f, bm, bvar = self._conditional_inputs(
            t, flux, t_sample, i, p, u, baseline_mean, baseline_var,
            False if lowrank else marginalize_over_inclination)
        nt, nts = t.numel(), ts.numel()
        with torch.cuda.device(self.device):
            if lowrank:
                def run(gp, inc, bm, bvar):
                    return gp._predictive_lowrank(t, ts, inc, p, rta1, udt, f, bm, bvar, data_cov,
                                                  return_cov)[:2]

                if return_cov == "diag":   # linear in nts as well: one launch sequence for the batch
                    mu, cov = run(self, inc, bm, bvar)
                else:
                    mu, cov = self._batch(_four_arrays(nts, nts), run, inc=inc, bm=bm, bvar=bvar)
            else:
                def run(gp, inc, bm, bvar):
                    mu, K = gp._predict_dense(t, ts, inc, p, rta1, marg, udt, udt_s, f, bm, bvar, data_cov)
                    return mu, (K.diagonal(dim1=1, dim2=2).contiguous() if return_cov == "diag" else K)

                n = max(nt, nts)
                mu, cov = self._batch(_four_arrays(n, n), run, inc=inc, bm=bm, bvar=bvar)
        return self._out(mu), self._out(cov)

    def _conditional_inputs(self, t, flux, t_sample, i, p, u, baseline_mean, baseline_var,
                            marginalize_over_inclination):
        """``_prep`` plus the prediction grid ``ts`` and its spacing, and the one light curve
        ``f (nt,)`` with its baseline terms (``_curves``) of ``predict`` / ``sample_conditional``."""
        udt_s = None if t_sample is None else self._spacing(t_sample)
        udt = self._spacing(t)           # second, so that _udt records the spacing of t
        marg, t, inc, rta1 = self._prep(t, i, p, u, marginalize_over_inclination)
        ts, udt_s = (t, udt) if t_sample is None else (self._t(t_sample), udt_s)
        f, _, _, bm, bvar = self._curves(flux, baseline_mean, baseline_var, t.numel(), M=1)
        return marg, t, inc, rta1, udt, ts, udt_s, f.reshape(-1), bm, bvar

    def _predict_dense(self, t, ts, inc, p, rta1, marg, udt, udt_s, f, bm, bvar, data_cov):
        """Predictive mean ``(B, nts)`` and covariance ``(B, nts, nts)`` of every batch element (NaN
        where ``K(t, t)`` is not positive definite)."""
        dev, B = self.device, self._B
        nt, nts = t.numel(), ts.numel()
        ldk, lds = nt + (nt & 1), nts + (nts & 1)
        # scalar (or one value per batch element) vs. a full (nt, nt) matrix of extra covariance
        scalar_bvar = bvar is None or bvar.ndim <= 1
        lib, h = self._lib, self._ctx.handle
        # K(ts, ts) + baseline_var first (the marginal kernel table is shared by both calls)
        _, Kss, _, _, _ = self._flux_cov(ts, inc, p, rta1, marg, udt_s, None,
                                         bvar if (scalar_bvar or nts == nt) else None, lds)
        gp_mean, Ktt, _, coef, _ = self._flux_cov(t, inc, p, rta1, marg, udt, data_cov, bvar, ldk)
        # right-hand sides: rows 0..nts-1 = K(ts, t) + baseline_var, row nts = y - mean
        R = torch.zeros(B, nts + 1, ldk, dtype=torch.float64, device=dev)
        rstride = (nts + 1) * ldk
        off = None
        if bvar is not None and scalar_bvar:
            off = bvar.reshape(-1).contiguous()
        off_s = 0 if off is None or off.numel() == 1 else 1
        late_off = off if self._tkind else None   # K(ts,t) *= k_temporal BEFORE + baseline_var
        if self._tkind:
            off = None
        if marg:
            _lib.check(lib.spb_cross_marginal(
                h, B, nts, nt, _ptr(ts), _ptr(t), float(p), self._covpts,
                _ptr(coef), _ptr(off), off_s, _ptr(R), ldk, rstride, _stream()))
        else:
            I = inc.numel()
            A_ts, A_t = self._design(ts, inc, p, rta1), self._design(t, inc, p, rta1)
            T = torch.empty(B, nts, 256, dtype=torch.float64, device=dev)
            # T = A_ts Sigma (Sigma symmetric), K(ts, t) = T A_t^T   (sp.py:903-906)
            self._gemm(B, nts, 256, 256, A_ts, 256, 0 if I == 1 else nts * 256, self._cov_ylm,
                       256, 65536, T, 256, nts * 256)
            if off is not None:
                R[:, :nts, :nt] = off.reshape(-1, 1, 1)
            self._gemm(B, nts, nt, 256, T, 256, nts * 256, A_t, 256, 0 if I == 1 else nt * 256,
                       R, ldk, rstride, alpha=1.0, beta=1.0)
        if self._tkind:   # sp.py:893-895
            _lib.check(lib.spb_temporal_scale(h, B, nts, nt, _ptr(ts), _ptr(t), self._tkind,
                                              _ptr(self._tau), 1, _ptr(late_off), off_s,
                                              _ptr(R), ldk, rstride, _stream()))
        if bvar is not None and not scalar_bvar:
            R[:, :nts, :nt] += bvar
        R[:, nts, :nt] = (f[None, :] - (bm[:, None] if bm.ndim == 1 else bm)) - gp_mean[:, None]
        info = self._factor_rows(Ktt, nt, ldk, rows=R)
        # mu = mean + V w ; K = K(ts, ts) - V V^T
        mu = gp_mean[:, None].expand(B, nts).contiguous()
        wrow = R.data_ptr() + nts * ldk * 8
        self._gemm(B, nts, 1, ldk, R, ldk, rstride, wrow, ldk, rstride, mu, 1, nts,
                   alpha=1.0, beta=1.0)
        self._gemm(B, nts, nts, ldk, R, ldk, rstride, R, ldk, rstride, Kss, lds, nts * lds,
                   alpha=-1.0, beta=1.0)
        bad = ((info & 1) != 0)
        mu = torch.where(bad[:, None], torch.full_like(mu, float("nan")), mu)
        Kc = Kss[:, :, :nts]
        return mu, torch.where(bad[:, None, None], torch.full_like(Kc, float("nan")), Kc)

    def sample_conditional(self, t, flux, data_cov, t_sample=None, i=defaults["i"],
                           p=defaults["p"], u=None, baseline_mean=defaults["baseline_mean"],
                           baseline_var=defaults["baseline_var"], nsamples=1, eps=defaults["eps"],
                           unit_normals=None, generator=None, marginalize_over_inclination=None,
                           method="dense"):
        """sp.py:924-1002: draws ``(nsamples, nts)`` from the conditional light-curve distribution.
        (The reference body reads an undefined name ``ts``; the intended ``ts = t_sample or t`` is
        what is implemented.)  ``unit_normals``: ``(nts, nsamples)`` (or ``(B, nts, nsamples)``).

        ``method="lowrank"`` draws ``mean + Phi(ts) G z1 + sqrt(eps) z2`` with ``G G^T`` the predictive
        covariance in the 32-dimensional phase basis (DESIGN.md section 4.6), in time and memory linear in
        ``nt`` and ``nts``.  Its ``unit_normals`` have shape ``(32 + nts, nsamples)`` (or ``(B, 32 + nts,
        nsamples)``): 32 rows ``z1`` for the basis coefficients, then ``nts`` rows ``z2`` for the white
        ``eps`` term.  The draws have the dense route's distribution but not its values for the same
        normals: the square root of the covariance is a different one."""
        if self._normalized and method == "lowrank":   # as predict: checked before the inputs
            raise NotImplementedError("Method not implemented when the flux is normalized.")
        lowrank = self._lowrank_checks(method, t, data_cov, baseline_var, marginalize_over_inclination)
        if self._normalized:
            raise NotImplementedError("Method not implemented when the flux is normalized.")
        marg, t, inc, rta1, udt, ts, udt_s, f, bm, bvar = self._conditional_inputs(
            t, flux, t_sample, i, p, u, baseline_mean, baseline_var,
            False if lowrank else marginalize_over_inclination)
        nt, nts = t.numel(), ts.numel()
        lds = nts + (nts & 1)
        with torch.cuda.device(self.device):
            if lowrank:
                _, _, out = self._predictive_lowrank(t, ts, inc, p, rta1, udt, f, bm, bvar, data_cov, None,
                                                     nsamples, eps, unit_normals, generator)
                return self._out(out)

            def run(gp, inc, bm, bvar, unit_normals):
                mu, K = gp._predict_dense(t, ts, inc, p, rta1, marg, udt, udt_s, f, bm, bvar, data_cov)
                Kp = torch.zeros(gp._B, nts, lds, dtype=torch.float64, device=gp.device)
                Kp[:, :, :nts] = K
                info = gp._factor_rows(Kp, nts, lds, diag_add=eps)
                _lib.check(gp._lib.spb_tril(gp._ctx.handle, gp._B, nts, _ptr(Kp), lds, nts * lds, _stream()))
                out = gp._draw(mu, Kp, nts, lds, nsamples, unit_normals, generator)
                return torch.where(((info & 1) != 0)[:, None, None], torch.full_like(out, float("nan")),
                                   out)

            n = max(nt, nts)
            out = self._batch(_four_arrays(n, n), run, inc=inc, bm=bm, bvar=bvar,
                              unit_normals=unit_normals)
        return self._out(out)

    def _predictive_lowrank(self, t, ts, inc, p, rta1, udt, f, bm, bvar, data_cov, return_cov, nsamples=0,
                            eps=0.0, unit_normals=None, generator=None):
        """``predict`` / ``sample_conditional`` with ``method="lowrank"``: spb_lowrank_posterior, then
        spb_lowrank_predict_eval.  Returns ``(mean, var | cov | None, draws | None)``, each with a leading
        batch axis.  Elements whose ``K(t, t)`` is not PD are NaN throughout; elements whose predictive
        covariance is not PSD beyond rounding have NaN draws only (include/spb200.h)."""
        dev, B, nt, nts = self.device, self._B, t.numel(), ts.numel()
        keep = []
        nm = self._noise_model(nt, data_cov, bvar, keep, uniform_dt=udt)
        lib, h = self._lib, self._ctx.handle
        I = inc.numel()
        f64 = dict(dtype=torch.float64, device=dev)
        a = torch.empty(B, 32, **f64)
        P = torch.empty(B, 32, 32, **f64)
        G = torch.empty(B, 32, 32, **f64)
        gp_mean = torch.empty(B, **f64)
        info = torch.zeros(B, dtype=torch.int32, device=dev)
        z = None
        if unit_normals is not None:
            z = torch.as_tensor(unit_normals, dtype=torch.float64).to(dev)
            if z.ndim not in (2, 3) or z.shape[-2] != 32 + nts or (z.ndim == 3 and z.shape[0] != B):
                raise ValueError("unit normals must have shape (%d, nsamples) or (B, %d, nsamples) for "
                                 "method='lowrank': 32 basis coefficients, then nts white-noise terms"
                                 % (32 + nts, 32 + nts))
            nsamples = z.shape[-1]
            z = z.transpose(-1, -2).contiguous()            # (S, 32 + nts) per draw
        elif nsamples:
            z = torch.randn(B, nsamples, 32 + nts, generator=generator, **f64)
        Binc, Q, R, aux = self._lowrank_basis(t, inc, rta1, p, nm)
        ev = self._mark("lowrank_posterior")
        nb = lib.spb_lowrank_posterior_workspace_bytes(h, B, nt)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.check(lib.spb_lowrank_posterior(
            h, B, nt, _ptr(Binc), 0 if I == 1 else 32 * 256, _ptr(self._mean_ylm), _ptr(self._cov_ylm),
            _ptr(Q), _ptr(R), _ptr(aux), ctypes.byref(nm), _ptr(f), _ptr(bm), 1 if bm.ndim == 1 else 0,
            _ptr(a), _ptr(P), _ptr(G), _ptr(gp_mean), _ptr(info), _ptr(ws), nb, _stream()))
        self._mark_end(ev)
        del ws, Q
        ev = self._mark("lowrank_eval")
        mean = torch.empty(B, nts, **f64)
        var = torch.empty(B, nts, **f64) if return_cov == "diag" else None
        cov = torch.empty(B, nts, nts, **f64) if return_cov == "full" else None
        draws = torch.empty(B, nsamples, nts, **f64) if nsamples else None
        nb = lib.spb_lowrank_predict_eval_workspace_bytes(h, B, nts, nsamples, cov is not None)
        ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        _lib.check(lib.spb_lowrank_predict_eval(
            h, B, nts, _ptr(ts), float(p), _ptr(a), _ptr(P), _ptr(G), _ptr(gp_mean), int(nsamples), _ptr(z),
            0 if z is None or z.ndim == 2 else nsamples * (32 + nts), float(eps), _ptr(mean), _ptr(var),
            _ptr(cov), nts, _ptr(draws), _ptr(ws), nb, _stream()))
        self._mark_end(ev)
        del ws, keep
        return mean, (var if cov is None else cov), draws

    def sample_ylm_conditional(self, t, flux, data_cov, i=defaults["i"], p=defaults["p"], u=None,
                               baseline_mean=defaults["baseline_mean"],
                               baseline_var=defaults["baseline_var"], nsamples=1,
                               unit_normals=None, generator=None):
        """sp.py:518-641: draws ``(nsamples, 256)`` of the Ylm coefficients conditioned on the
        observed flux (the inclination is always used).  ``baseline_mean`` and ``baseline_var`` are
        shared by the batch (``baseline_var`` may be an ``(nt, nt)`` matrix).

        With ``C = data_cov + baseline_var = L_C L_C^T``, ``G = (L_C^-1 A)^T`` and ``Y = L_y^-T``
        (``cov_ylm = L_y L_y^T``):  ``W = G G^T + Y Y^T``,  ``rhs = G L_C^-1 (f - b) + Y L_y^-1 mu``,
        ``ymu = W^-1 rhs``, ``ycov = W^-1 = Y_W Y_W^T`` -- every product a tensor-core GEMM, every
        inverse a forward substitution on appended rows of the Cholesky kernel."""
        if self._normalized:
            raise NotImplementedError("Method not implemented when the flux is normalized.")
        if self._time_variable:
            raise NotImplementedError("Method not implemented for time-variable maps.")
        if self._nylm != 256:
            raise NotImplementedError("sample_ylm_conditional is implemented at ydeg = 15")
        _, t, inc, rta1 = self._prep(t, i, p, u, None)
        nt = t.numel()
        ldk = nt + (nt & 1)
        f, _, _, bm, bvar = self._curves(flux, baseline_mean, baseline_var, nt, M=1)
        if bm.ndim == 1 or (bvar is not None and bvar.ndim == 1):
            raise ValueError("sample_ylm_conditional factorises one noise covariance and one residual for "
                             "the whole batch: baseline_mean and baseline_var cannot be per element")
        f = f.reshape(-1)

        def run(gp, inc, unit_normals):
            dev, B = gp.device, gp._B
            lib, h = gp._lib, gp._ctx.handle
            A = gp._design(t, inc, p, rta1)
            I = A.shape[0]
            # C = data_cov (+ baseline_var on every entry): input assembly, sp.py:594-607
            d = torch.as_tensor(data_cov, dtype=torch.float64).to(dev)
            C = torch.zeros(1, nt, ldk, dtype=torch.float64, device=dev)
            if d.ndim == 0:
                C[0, :, :nt].diagonal().fill_(float(d))
            elif d.ndim == 1:
                C[0, :, :nt].diagonal().copy_(d)
            else:
                C[0, :, :nt] = d
            if bvar is not None:
                C[0, :, :nt] += bvar
            infoC = gp._factor_rows(C, nt, ldk)
            # rows: A^T (256 per inclination) and the residual, all against the one factor of C
            R = torch.zeros(I * 256 + 1, ldk, dtype=torch.float64, device=dev)
            R[: I * 256, :nt] = A.transpose(1, 2).reshape(I * 256, nt)
            R[I * 256, :nt] = f - bm
            quad = torch.empty(I * 256 + 1, dtype=torch.float64, device=dev)
            _lib.check(lib.spb_cholesky_solve_rows(h, nt, _ptr(C), ldk, I * 256 + 1, _ptr(R), ldk,
                                                   _ptr(quad), _stream()))
            grow = R.data_ptr() + I * 256 * ldk * 8
            # cov_ylm = L_y L_y^T with rows [I; mu] appended: Y = L_y^-T (as rows), wmu = L_y^-1 mu
            Ly = gp._cov_ylm.clone()
            Ry = torch.zeros(B, 257, 256, dtype=torch.float64, device=dev)
            Ry[:, :256, :] = torch.eye(256, dtype=torch.float64, device=dev)
            Ry[:, 256, :] = gp._mean_ylm
            infoY = gp._factor_rows(Ly, 256, 256, rows=Ry)
            sY = 257 * 256
            W = torch.empty(B, 256, 256, dtype=torch.float64, device=dev)
            sG = 0 if I == 1 else 256 * ldk
            gp._gemm(B, 256, 256, ldk, R, ldk, sG, R, ldk, sG, W, 256, 65536)
            gp._gemm(B, 256, 256, 256, Ry, 256, sY, Ry, 256, sY, W, 256, 65536, beta=1.0)
            # rhs = Y wmu + G g, appended (with the identity) to the factorisation of W
            Rw = torch.zeros(B, 257, 256, dtype=torch.float64, device=dev)
            Rw[:, :256, :] = torch.eye(256, dtype=torch.float64, device=dev)
            rhs = Rw.data_ptr() + 256 * 256 * 8
            gp._gemm(B, 256, 1, 256, Ry, 256, sY, Ry.data_ptr() + 256 * 256 * 8, 256, sY, rhs, 1, sY)
            gp._gemm(B, 256, 1, ldk, R, ldk, sG, grow, ldk, 0, rhs, 1, sY, beta=1.0)
            infoW = gp._factor_rows(W, 256, 256, rows=Rw)
            # ycov = Y_W Y_W^T, ymu = Y_W (L_W^-1 rhs)
            ycov = torch.empty(B, 256, 256, dtype=torch.float64, device=dev)
            gp._gemm(B, 256, 256, 256, Rw, 256, sY, Rw, 256, sY, ycov, 256, 65536)
            ymu = torch.empty(B, 256, dtype=torch.float64, device=dev)
            gp._gemm(B, 256, 1, 256, Rw, 256, sY, rhs, 256, sY, ymu, 1, 256)
            infoS = gp._factor_rows(ycov, 256, 256)
            _lib.check(lib.spb_tril(h, B, 256, _ptr(ycov), 256, 65536, _stream()))
            out = gp._draw(ymu, ycov, 256, 256, nsamples, unit_normals, generator)
            bad = (((infoY | infoW | infoS) & 1) != 0) | ((infoC & 1) != 0)
            return torch.where(bad[:, None, None], torch.full_like(out, float("nan")), out)

        with torch.cuda.device(self.device):
            out = self._batch(_four_arrays(nt, 256), run, inc=inc, unit_normals=unit_normals)
        return self._out(out)

    # ------------------------------------------------------------------ SURVEY 8(f) rank 3
    @property
    def tau(self):
        """sp.py:337-340."""
        return None if self._tau is None else self._out(self._tau)

    @property
    def temporal_kernel(self):
        """sp.py:342-345."""
        return getattr(self, "_temporal_kernel", None)

    def _sample_ylm_temporal(self, t, nsamples, u, generator):
        """sp.py:510-516 + ops/sample.py:24-33 (a triple Python loop in the reference):
        ``y_i = L_t U_i L_y^T`` with ``L_t = cho_factor(temporal_kernel(t, t, tau))`` -- two
        tensor-core GEMMs per batch element.  As in the reference, ``mean_ylm`` is NOT added on
        this branch.  ``u`` optionally supplies ``U`` of shape ``(nsamples, nt, nylm)``."""
        if not self._time_variable:
            raise ValueError("sample_ylm(t=...) needs a time-variable process (tau)")
        if self._nylm != 256:
            raise NotImplementedError("time-variable sample_ylm is implemented at ydeg = 15")
        t = self._t(t)
        nt = t.numel()
        ldt = nt + (nt & 1)
        dev, B = self.device, self._B
        Ly = self.cho_cov_ylm
        Ly = (Ly if self._batched else Ly[None]).contiguous()
        lib, h = self._lib, self._ctx.handle
        with torch.cuda.device(dev):
            Kt = torch.zeros(B, nt, ldt, dtype=torch.float64, device=dev)
            Kt[:, :, :nt] = 1.0
            _lib.check(lib.spb_temporal_scale(h, B, nt, nt, _ptr(t), _ptr(t), self._tkind,
                                              _ptr(self._tau), 1, None, 0, _ptr(Kt), ldt, nt * ldt,
                                              _stream()))
            info = self._factor_rows(Kt, nt, ldt)
            _lib.check(lib.spb_tril(h, B, nt, _ptr(Kt), ldt, nt * ldt, _stream()))
            if u is None:
                U = torch.randn(nsamples, nt, 256, dtype=torch.float64, device=dev,
                                generator=generator)
            else:
                U = torch.as_tensor(u, dtype=torch.float64).to(dev)
                if U.ndim != 3 or U.shape[1] != nt or U.shape[2] != 256:
                    raise ValueError("u must have shape (nsamples, nt, 256)")
                nsamples = U.shape[0]
            # Two batched tensor-core GEMMs for the whole (B x nsamples) set, no Python loop:
            #   V[b] (nt, ns*256) = L_t[b] (nt, nt) . [U_0 | U_1 | ...]   (NT form: Bm = the stacked
            #   U_s^T, (ns*256, ldt), shared by every b; k = time, zero-padded to an even length)
            #   W[b] (nt*ns, 256) = V[b] viewed as (nt*ns, 256) . L_y[b]^T
            # and one permutation (t, s) -> (s, t) of the result.
            Ut = torch.zeros(nsamples * 256, ldt, dtype=torch.float64, device=dev)
            Ut[:, :nt] = U.transpose(1, 2).reshape(nsamples * 256, nt)
            V = torch.empty(B, nt, nsamples * 256, dtype=torch.float64, device=dev)
            self._gemm(B, nt, nsamples * 256, ldt, Kt, ldt, nt * ldt, Ut, ldt, 0, V, nsamples * 256,
                       nt * nsamples * 256)
            W = torch.empty(B, nt * nsamples, 256, dtype=torch.float64, device=dev)
            self._gemm(B, nt * nsamples, 256, 256, V, 256, nt * nsamples * 256, Ly, 256, 65536, W,
                       256, nt * nsamples * 256)
            out = W.view(B, nt, nsamples, 256).transpose(1, 2).contiguous()
            out = torch.where(((info & 1) != 0)[:, None, None, None],
                              torch.full_like(out, float("nan")), out)
        return self._out(out)

    # ------------------------------------------------------------------ flux of given surfaces, sums
    def flux(self, y, t, i=defaults["i"], p=defaults["p"], u=None):
        """sp.py:1237-1283: light curves ``(nsamples, nt)`` of spherical-harmonic vectors ``y``
        (``(nsamples, nylm)``, or ``(nsamples, nt, nylm)`` for time-variable surfaces, e.g. the
        output of ``sample_ylm``); mean-normalised when the process is ``normalized``."""
        dev = self.device
        yt = torch.as_tensor(y, dtype=torch.float64).to(dev)
        squeeze = yt.ndim == 1
        if squeeze:
            yt = yt[None]
        if _is_batched(i):
            raise ValueError("flux() takes a scalar inclination")
        A = self._design_full(t, i, p, u)[0]
        yt = self._pad_ylm(yt, yt.ndim - 1)
        nt = A.shape[0]
        with torch.cuda.device(dev):
            if self._time_variable:
                if yt.ndim != 3 or yt.shape[1] != nt or yt.shape[2] != 256:
                    raise ValueError("time-variable surfaces: y must have shape (nsamples, nt, 256)")
                ns = yt.shape[0]
                yt = yt.contiguous()
                out = torch.empty(nt, ns, dtype=torch.float64, device=dev)
                # F[k][s] = A[k] . y[s][k]  -- one (ns x 256)(256 x 1) product per time
                self._gemm(nt, ns, 1, 256, yt, nt * 256, 256, A, 256, 256, out, 1, ns)
                F = out.transpose(0, 1).contiguous()
            else:
                if yt.ndim != 2 or yt.shape[1] != 256:
                    raise ValueError("y must have shape (nsamples, 256)")
                ns = yt.shape[0]
                F = torch.empty(ns, nt, dtype=torch.float64, device=dev)
                self._gemm(1, ns, nt, 256, yt.contiguous(), 256, 0, A, 256, 0, F, nt, 0)
            if self._normalized:   # sp.py:1279-1282
                F = (1.0 + F) / (1.0 + F).mean(dim=-1, keepdim=True) - 1.0
        return F[0] if squeeze else F

    def __add__(self, other):
        """sp.py:1190-1191."""
        return StarryProcessSum(self, other)

    def __radd__(self, other):
        """sp.py:1193-1197 (so that ``sum([...])`` works)."""
        if isinstance(other, (int, float)) and other == 0:
            return self
        return self.__add__(other)


class StarryProcessSum(StarryProcess):
    """sp.py:1335-1400: the sum of independent processes -- Ylm means and covariances add; every
    flux-space method then runs on the summed moments through the same kernels."""

    def __init__(self, first, second):
        assert isinstance(second, StarryProcess), \
            "Can only add instances of `StarryProcess` to each other."
        assert first._ydeg == second._ydeg, "Mismatch in `ydeg`."
        assert first._udeg == second._udeg, "Mismatch in `udeg`."
        assert first._normalized == second._normalized, "Mismatch in `normalized`."
        assert first._marginalize_over_inclination == second._marginalize_over_inclination, \
            "Mismatch in `marginalize_over_inclination`."
        assert first._covpts == second._covpts, "Mismatch in `covpts`."
        assert first._time_variable is False and second._time_variable is False, \
            "Sums of `StarryProcess` instances not implemented for time-variable surfaces."
        assert first.device == second.device, "Mismatch in device."
        for k in ("_ydeg", "_udeg", "_nylm", "_normalized", "_marginalize_over_inclination",
                  "_covpts", "_normN", "_normzmax", "_max_chunk_bytes", "_sigma_max", "_ctx",
                  "device", "_lib", "_opt", "_opt_keep", "_opt_kw"):
            setattr(self, k, getattr(first, k))
        self._time_variable, self._tkind, self._tau = False, 0, None
        self._children = []
        for child in (first, second):
            self._children += getattr(child, "_children", [child])
        if first._B != second._B and 1 not in (first._B, second._B):
            raise ValueError("batched summands must have the same batch size")
        self._B = max(first._B, second._B)
        self._batched = first._batched or second._batched
        first._compute_moments()
        second._compute_moments()
        B = self._B
        # Sum the random variables (sp.py:1383-1385)
        self._mean_ylm = (first._mean_ylm + second._mean_ylm).expand(B, 256).contiguous()
        self._cov_ylm = (first._cov_ylm + second._cov_ylm).expand(B, 256, 256).contiguous()
        self._info = (first._info | second._info).expand(B).contiguous()
        self._cho_cov_ylm = None
        self._z = None
        self._rTA1_cache = {}
        self._a = self._b = self._r = self._c = self._n = self._dr = None

    def _compute_moments(self):
        return

    def log_jac(self):
        raise NotImplementedError("log_jac is defined for a single process (sp.py:1004-1050)")

    @property
    def a(self):
        raise AttributeError("a sum of processes has no single latitude distribution")

    b = a
