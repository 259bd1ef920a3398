"""ctypes binding of libspb200.so (include/spb200.h).  There is NO fallback: if the CUDA library
is missing or fails to load, importing a compute entry point raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libspb200.so")

_c = ctypes
_P = _c.c_void_p
_I = _c.c_int
_LL = _c.c_longlong
_D = _c.c_double
_SZ = _c.c_size_t


class NoiseModel(_c.Structure):
    """spb_noise_model (include/spb200.h)."""

    _fields_ = [
        ("normalized", _I), ("normalization_order", _I), ("normalization_zmax", _D),
        ("data_kind", _I), ("data_cov", _P), ("data_stride", _LL),
        ("base_kind", _I), ("baseline_var", _P), ("base_stride", _LL),
        ("lower_only", _I), ("defer", _I),
        ("temporal_kind", _I), ("tau", _P), ("tau_stride", _LL),
        ("uniform_dt", _D),
    ]


class MomentsOptions(_c.Structure):
    """spb_moments_options (include/spb200.h)."""
    _fields_ = [("Bp", _P), ("lambda_", _P), ("abmin", _D), ("log_alpha_max", _D),
                ("log_beta_max", _D)]


class Affine(_c.Structure):
    """spb_affine (include/spb200.h)."""
    _fields_ = [
        ("scal", _P), ("q", _P), ("diag", _P), ("diag_kind", _I), ("diag_stride", _LL),
        ("offset", _P), ("offset_stride", _LL),
    ]


# name -> (restype, argtypes); mirrors include/spb200.h one to one
PROTOTYPES = {
    "spb_last_error": (_c.c_char_p, []),
    "spb_version": (_I, []),
    "spb_create": (_I, [_I, _P, _SZ, _c.POINTER(_P)]),
    "spb_destroy": (None, [_P]),
    "spb_device": (_I, [_P]),
    "spb_gauss2beta": (_I, [_P, _I, _P, _P, _P, _P, _P]),
    "spb_log_jac": (_I, [_P, _I, _P, _P, _D, _P, _P]),
    "spb_ylm_moments_workspace_bytes": (_SZ, [_P, _I]),
    "spb_ylm_moments": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "spb_ylm_moments_dr": (_I, [_P, _I, _P, _P, _P, _P, _P, _P, _c.POINTER(MomentsOptions), _P, _P,
                                _P, _P, _SZ, _P]),
    "spb_gauss2beta_opt": (_I, [_P, _I, _P, _P, _c.POINTER(MomentsOptions), _P, _P, _P]),
    "spb_log_jac_opt": (_I, [_P, _I, _P, _P, _D, _c.POINTER(MomentsOptions), _P, _P]),
    "spb_ylm_moments_grad_workspace_bytes": (_SZ, [_P, _I]),
    "spb_ylm_moments_grad": (_I, [_P, _I, _P, _P, _P, _P, _P, _c.POINTER(MomentsOptions), _D, _P, _P,
                                  _P, _P, _P, _SZ, _P]),
    "spb_cho_cov_ylm": (_I, [_P, _I, _P, _P, _P, _P]),
    "spb_sample_ylm": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "spb_flux_operator": (_I, [_P, _I, _P, _P, _P]),
    "spb_Rx": (_I, [_P, _I, _P, _P, _P]),
    "spb_tensordotRz": (_I, [_P, _I, _P, _P, _P, _P]),
    "spb_design_matrix_workspace_bytes": (_SZ, [_P, _I, _I]),
    "spb_design_matrix": (_I, [_P, _I, _I, _P, _P, _P, _P, _I, _P, _P, _SZ, _P]),
    "spb_flux_marginal_workspace_bytes": (_SZ, [_P, _I]),
    "spb_flux_marginal": (_I, [_P, _I, _P, _P, _P, _I, _P, _P, _P, _P, _SZ, _P]),
    "spb_flux_conditional_workspace_bytes": (_SZ, [_P, _I, _I]),
    "spb_flux_conditional": (_I, [_P, _I, _I, _P, _LL, _P, _P, _P, _P, _I, _P, _SZ, _P]),
    "spb_flux_conditional_lower": (_I, [_P, _I, _I, _P, _LL, _P, _P, _P, _P, _I, _P, _SZ, _P]),
    "spb_assemble_workspace_bytes": (_SZ, [_P, _I, _I]),
    "spb_assemble_marginal": (_I, [_P, _I, _I, _P, _D, _I, _P, _P, _P, _c.POINTER(NoiseModel),
                                   _P, _I, _P, _P, _P, _SZ, _P]),
    "spb_assemble_conditional": (_I, [_P, _I, _I, _P, _c.POINTER(NoiseModel), _P, _I, _P, _P,
                                      _P, _SZ, _P]),
    "spb_cholesky_lnlike": (_I, [_P, _I, _I, _P, _I, _LL, _I, _P, _I, _LL, _P, _P, _P, _P, _P]),
    "spb_cholesky_lnlike_affine": (_I, [_P, _I, _I, _P, _I, _LL, _c.POINTER(Affine), _I, _P, _I, _LL,
                                        _P, _P, _P, _P, _P]),
    "spb_assemble_workspace_layout": (None, [_I, _I, _P, _c.POINTER(_P), _c.POINTER(_P)]),
    "spb_cholesky_i8_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "spb_cholesky_lnlike_i8": (_I, [_P, _I, _I, _P, _I, _LL, _c.POINTER(Affine), _I, _P, _I, _LL,
                                    _P, _P, _P, _P, _I, _D, _P, _SZ, _P]),
    "spb_cholesky_solve_rows": (_I, [_P, _I, _P, _I, _I, _P, _I, _P, _P]),
    "spb_lowrank_inclination_workspace_bytes": (_SZ, [_P, _I]),
    "spb_lowrank_inclination": (_I, [_P, _I, _P, _P, _I, _P, _P, _SZ, _P]),
    "spb_lowrank_basis_workspace_bytes": (_SZ, [_P, _I]),
    "spb_lowrank_basis": (_I, [_P, _I, _P, _D, _I, _P, _P, _P, _P, _P, _SZ, _P]),
    "spb_lowrank_lnlike_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "spb_lowrank_lnlike": (_I, [_P, _I, _I, _P, _LL, _P, _P, _P, _P, _P, _c.POINTER(NoiseModel), _I, _P,
                                _I, _LL, _P, _LL, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "spb_lowrank_posterior_workspace_bytes": (_SZ, [_P, _I, _I]),
    "spb_lowrank_posterior": (_I, [_P, _I, _I, _P, _LL, _P, _P, _P, _P, _P, _c.POINTER(NoiseModel), _P, _P,
                                   _LL, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "spb_lowrank_predict_eval_workspace_bytes": (_SZ, [_P, _I, _I, _I, _I]),
    "spb_lowrank_predict_eval": (_I, [_P, _I, _I, _P, _D, _P, _P, _P, _P, _I, _P, _LL, _D, _P, _P, _P, _I, _P,
                                      _P, _SZ, _P]),
    "spb_temporal_scale":(_I, [_P, _I, _I, _I, _P, _P, _I, _P, _LL, _P, _LL, _P, _I, _LL, _P]),
    "spb_gemm_nt": (_I, [_P, _I, _I, _I, _I, _D, _P, _I, _LL, _P, _I, _LL, _D, _P, _I, _LL, _P]),
    "spb_tril": (_I, [_P, _I, _I, _P, _I, _LL, _P]),
    "spb_cross_marginal": (_I, [_P, _I, _I, _I, _P, _P, _D, _I, _P, _P, _LL, _P, _I, _LL, _P]),
    "spb_dmma_peak": (_I, [_P, _I, _c.POINTER(_D), _c.POINTER(_D)]),
    "spb_launch_count": (_I, [_P, _c.POINTER(_LL)]),
    "spb_set_option": (_I, [_P, _c.c_char_p, _I]),
}

_lib = None


def load(allow_missing_symbols=False):
    """Load libspb200.so and attach prototypes.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "starry_process_b200: %s not found -- build it with `python -m starry_process_b200.build`"
            " (there is no CPU fallback)" % LIB_PATH)
    lib = _c.CDLL(LIB_PATH)
    missing = []
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    if missing and not allow_missing_symbols:
        raise RuntimeError("libspb200.so lacks symbols: %s" % ", ".join(missing))
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().spb_last_error()
        raise RuntimeError("libspb200 error %d: %s" % (status, msg.decode() if msg else "?"))
