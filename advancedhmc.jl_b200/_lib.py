"""_lib.py -- ctypes binding of libahmc_b200.so (include/ahmc_b200.h).  Plain pointers and sizes only.

There is NO CPU fallback: if the shared library is missing or no CUDA device is usable the import of
the product path fails loudly (RuntimeError)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AHMC_B200_LIB", os.path.join(HERE, "libahmc_b200.so"))  # override: A/B builds

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM, ERR_CALLBACK = 0, -1, -2, -3, -4, -5
METRIC_UNIT, METRIC_DIAG, METRIC_DENSE = 0, 1, 2
MODEL_STD_NORMAL, MODEL_DIAG_GAUSS, MODEL_DENSE_GAUSS, MODEL_FUNNEL, MODEL_CALLBACK, MODEL_USER = 0, 1, 2, 3, 4, 5
FLAG_HOST_BUFFERS, FLAG_COMPAT_BREAK_ALL, FLAG_ASYNC, FLAG_EXACT_CHECKS, FLAG_NO_REFRESH = 1, 2, 4, 8, 16
FLAG_NUTS_SLICE_TS, FLAG_NUTS_CLASSIC, FLAG_NUTS_STRICT = 32, 64, 128
STATUS_NONFINITE = 1

_dp = C.POINTER(C.c_double)
_vp = C.c_void_p


class Metric(C.Structure):
    _fields_ = [("kind", C.c_int32), ("Minv", _vp), ("chain_stride", C.c_int64), ("cholU", _vp)]


class PhasePoint(C.Structure):
    _fields_ = [("theta", _vp), ("r", _vp), ("lp_value", _vp), ("lp_gradient", _vp), ("lk_value", _vp),
                ("lk_gradient", _vp), ("ld", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [("n_steps", _vp), ("is_accept", _vp), ("acceptance_rate", _vp), ("log_density", _vp),
                ("hamiltonian_energy", _vp), ("hamiltonian_energy_error", _vp),
                ("max_hamiltonian_energy_error", _vp), ("tree_depth", _vp), ("numerical_error", _vp)]


class Rng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("offset", C.c_uint64), ("normal_tape", _vp), ("exp_tape", _vp),
                ("exp_stride", C.c_int64), ("dir_tape", _vp), ("dir_stride", C.c_int64),
                ("partial_refresh_alpha", C.c_double), ("temper_alpha", C.c_double)]


class AdaptCfg(C.Structure):
    _fields_ = [("n_adapts", C.c_int32), ("init_buffer", C.c_int32), ("term_buffer", C.c_int32), ("window_size", C.c_int32),
                ("delta", C.c_double), ("gamma", C.c_double), ("t0", C.c_double), ("kappa", C.c_double),
                ("adapt_metric", C.c_int32), ("n_min", C.c_int32), ("eps_chain", _vp), ("Minv_chain", _vp),
                ("eps_trace", _vp)]


class PooledCfg(C.Structure):
    _fields_ = [("n_adapts", C.c_int32), ("init_buffer", C.c_int32), ("term_buffer", C.c_int32), ("window_size", C.c_int32),
                ("delta", C.c_double), ("gamma", C.c_double), ("t0", C.c_double), ("kappa", C.c_double), ("eps0", C.c_double),
                ("adapt_metric", C.c_int32), ("n_min", C.c_int32)]


LOGP_GRAD_FN = C.CFUNCTYPE(C.c_int, _vp, _vp, _vp, _vp, C.c_int32, C.c_int64, C.c_int64, _vp)

# name -> (restype, argtypes): exactly the entry points include/ahmc_b200.h declares
PROTOTYPES = {
    "ahmc_version": (C.c_char_p, []),
    "ahmc_create": (C.c_int, [C.POINTER(_vp), C.c_int32, _vp]),
    "ahmc_destroy": (C.c_int, [_vp]),
    "ahmc_last_error": (C.c_char_p, [_vp]),
    "ahmc_synchronize": (C.c_int, [_vp]),
    "ahmc_stream": (_vp, [_vp]),
    "ahmc_launch_count": (C.c_int64, [_vp]),
    "ahmc_last_transport": (C.c_char_p, [_vp]),
    "ahmc_model_create": (C.c_int, [_vp, C.c_int32, C.c_int32, _dp, _dp, C.c_double, C.POINTER(_vp)]),
    "ahmc_model_create_callback": (C.c_int, [_vp, C.c_int32, LOGP_GRAD_FN, _vp, C.POINTER(_vp)]),
    "ahmc_model_create_user": (C.c_int, [_vp, C.c_int32, C.c_char_p, _dp, C.c_int32, C.c_double, C.POINTER(_vp)]),
    "ahmc_user_source_check": (C.c_int, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_int64]),
    "ahmc_model_destroy": (C.c_int, [_vp, _vp]),
    "ahmc_phasepoint_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.POINTER(PhasePoint),
                                      C.c_uint32]),
    "ahmc_leapfrog_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp, C.c_int32,
                                    C.c_double, C.POINTER(PhasePoint), C.POINTER(PhasePoint), _vp, _vp, C.c_uint32]),
    "ahmc_leapfrog_trajectory_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp,
                                               C.c_int32, C.c_double, C.POINTER(PhasePoint), C.POINTER(PhasePoint),
                                               C.c_int64, _vp, C.c_uint32]),
    "ahmc_hmc_multinomial_transition_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp,
                                                      C.c_int32, C.c_int32, C.POINTER(Rng), C.POINTER(PhasePoint),
                                                      C.POINTER(PhasePoint), C.POINTER(Stats), C.c_uint32]),
    "ahmc_rand_momentum_f64": (C.c_int, [_vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.POINTER(Rng), _vp,
                                         C.c_int64, C.c_uint32]),
    "ahmc_hmc_transition_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp,
                                          C.c_int32, C.POINTER(Rng), C.POINTER(PhasePoint), C.POINTER(PhasePoint),
                                          C.POINTER(Stats), C.c_uint32]),
    "ahmc_nuts_transition_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp,
                                           C.c_int32, C.c_double, C.POINTER(Rng), C.POINTER(PhasePoint),
                                           C.POINTER(PhasePoint), C.POINTER(Stats), C.c_uint32]),
    "ahmc_hmc_sample_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp, C.c_int32,
                                      C.c_int32, C.POINTER(Rng), C.POINTER(PhasePoint), C.POINTER(PhasePoint), _vp,
                                      C.POINTER(Stats), C.c_uint32]),
    "ahmc_nuts_sample_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_double, _vp, C.c_int32,
                                       C.c_double, C.c_int32, C.POINTER(Rng), C.POINTER(PhasePoint),
                                       C.POINTER(PhasePoint), _vp, C.POINTER(Stats), C.c_uint32]),
    "ahmc_nuts_adapt_sample_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.c_int32, C.c_double,
                                             C.c_int32, C.POINTER(AdaptCfg), C.POINTER(Rng), C.POINTER(PhasePoint),
                                             C.POINTER(PhasePoint), _vp, C.POINTER(Stats), C.c_uint32]),
    "ahmc_adapt_summary_f64": (C.c_int, [_vp, C.c_int32, C.c_int64, _vp, C.c_int64, _vp, _vp, C.c_uint32]),
    "ahmc_adapt_cov_f64": (C.c_int, [_vp, C.c_int32, C.c_int64, _vp, C.c_int64, _vp, _vp, C.c_uint32]),
    "ahmc_find_good_stepsize_f64": (C.c_int, [_vp, _vp, C.POINTER(Metric), C.c_int32, C.c_int64, C.POINTER(PhasePoint),
                                                C.POINTER(Rng), C.c_double, C.c_int32, _vp, _vp, C.c_uint32]),
    "ahmc_comm_unique_id": (C.c_int, [_vp, _vp]),
    "ahmc_comm_create": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "ahmc_comm_from_nccl": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    "ahmc_comm_destroy": (C.c_int, [_vp, _vp]),
    "ahmc_adapt_allgather_f64": (C.c_int, [_vp, _vp, _vp, C.c_int64, _vp, C.c_uint32]),
    "ahmc_pooled_create": (C.c_int, [_vp, C.c_int32, C.c_int64, C.POINTER(PooledCfg), _dp, C.POINTER(_vp)]),
    "ahmc_pooled_destroy": (C.c_int, [_vp, _vp]),
    "ahmc_pooled_eps": (_vp, [_vp]),
    "ahmc_pooled_minv": (_vp, [_vp]),
    "ahmc_adapt_exchange_f64": (C.c_int, [_vp, _vp, _vp, C.c_int32, C.c_int64, _vp, C.c_int64, _vp, _vp, C.c_uint32]),
    "ahmc_pooled_state": (C.c_int, [_vp, _vp, _dp, _dp, C.POINTER(C.c_int32), _dp]),
    "ahmc_pooled_create_dense": (C.c_int, [_vp, C.c_int32, C.c_int64, C.POINTER(PooledCfg), _dp, C.POINTER(_vp)]),
    "ahmc_pooled_cholu": (_vp, [_vp]),
    "ahmc_pooled_state_dense": (C.c_int, [_vp, _vp, _dp, _dp, _dp, C.POINTER(C.c_int32), _dp, C.POINTER(C.c_int32)]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen libahmc_b200.so and bind every prototype.  Raises if the library is absent (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python advancedhmc.jl_b200/build.py` "
            "(or __graft_entry__.build()). There is no CPU fallback for the product path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class AhmcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ahmc error {code}: {msg}")
        self.code = code


class InvalidArgument(AhmcError, ValueError):
    """AHMC_ERR_INVALID -- the ArgumentError / @argcheck analogue of the reference."""
