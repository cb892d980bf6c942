"""ctypes binding of libnpbnn_b200.so (C ABI in include/npbnn_b200.h).

The library is the product path: there is no CPU fallback.  If it is missing this module tries
to build it with nvcc (npbnn_b200/build.py) and raises otherwise.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# NPBNN_B200_LIB loads another build of the library instead (e.g. to compare two builds on the same inputs)
LIB_PATH = os.environ.get("NPBNN_B200_LIB") or os.path.join(HERE, "libnpbnn_b200.so")

MAX_LAYERS = 8
MAX_OUT = 32

ACT = {"ReLU": 0, "genReLU": 1, "swish": 2, "tanh": 3}
LIK_CATEGORICAL, LIK_GAUSSIAN, LIK_GAUSSIAN_HEAD = 0, 1, 2
LIK_POISSON, LIK_NEGBIN, LIK_NEGBIN10 = 3, 4, 5          # count likelihoods (estimation_mode="custom")
LIK_COUNT = (LIK_POISSON, LIK_NEGBIN, LIK_NEGBIN10)
PRIOR_UNIFORM, PRIOR_NORMAL, PRIOR_CAUCHY, PRIOR_LAPLACE = 0, 1, 2, 3
SIGMA_FIXED, SIGMA_EMPIRICAL = 0, 1

# state slots (enum in include/npbnn_b200.h)
F_LOGLIK, F_LOGPRIOR, F_LOGPOST, F_TEMPERATURE, F_ACC_RATE, F_LOGLIK_PROP, F_LOGPRIOR_PROP, F_LOG_U, F_ADD_PROB = range(9)
F_ALPHA_PROP = 176
F_UPDATE_F, F_UPDATE_WS, F_FREQ_LAYER, F_ALPHA, F_SIGMA, F_SUM_R, F_SUM_R2, F_SUM_R2_TEST, F_STRIDE = \
    16, 24, 32, 40, 48, 80, 112, 144, 192
I_ITERATION, I_LAST_ACCEPTED, I_N_ACCEPTED, I_RING_LEN, I_RING_HEAD, I_RING_SUM = range(6)
I_UPDATE_N, I_MAX_N, I_PROPOSED, I_N_CORRECT, I_N_CORRECT_TEST, I_CLASS_CORRECT, I_PRED_HIST, I_RING, I_STRIDE = \
    8, 16, 24, 32, 33, 34, 66, 98, 200


class NetSpec(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("n_features", C.c_int32), ("out_dim", C.c_int32 * MAX_LAYERS),
                ("has_bias", C.c_int32 * MAX_LAYERS), ("act", C.c_int32), ("lik", C.c_int32)]


class SamplerConfig(C.Structure):
    _fields_ = [("prior", C.c_int32), ("sigma_mode", C.c_int32), ("sample_from_prior", C.c_int32),
                ("adapt_freq", C.c_int32), ("adapt_stop", C.c_int32), ("use_mask", C.c_int32),
                ("adapt_f", C.c_double), ("adapt_fM", C.c_double), ("lik_temp", C.c_double),
                ("w_bound", C.c_double), ("prior_scale", C.c_double * MAX_LAYERS), ("seed", C.c_uint64),
                ("n_act_prm", C.c_int32), ("chain_offset", C.c_int32), ("init_additional_prob", C.c_double),
                ("prior_ind1", C.c_double), ("use_indicators", C.c_int32), ("use_feature_indicators", C.c_int32),
                ("freq_indicator", C.c_double)]


class Injection(C.Structure):
    _fields_ = [("n_steps", C.c_int32), ("cap", C.c_int32), ("proposed", C.c_void_p), ("count", C.c_void_p),
                ("ix", C.c_void_p), ("iy", C.c_void_p), ("dz", C.c_void_p), ("log_u", C.c_void_p),
                ("alpha_ix", C.c_void_p), ("alpha_dz", C.c_void_p), ("add_prob", C.c_void_p),
                ("ind_move", C.c_void_p), ("ind_flip", C.c_void_p), ("fi_move", C.c_void_p), ("fi_flip", C.c_void_p)]


class NpbnnError(RuntimeError):
    pass


_lib = None

_SIGNATURES = {
    "bnn_last_error": (C.c_char_p, []),
    "bnn_abi_version": (C.c_int, []),
    "bnn_ctx_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "bnn_ctx_destroy": (C.c_int, [C.c_void_p]),
    "bnn_set_net": (C.c_int, [C.c_void_p, C.POINTER(NetSpec)]),
    "bnn_n_params": (C.c_int64, [C.c_void_p]),
    "bnn_set_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p]),
    "bnn_forward_lik": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_double,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_forward_lik_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_log_prior": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_log_prior_entries": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_snapshot": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "bnn_snapshot_ready": (C.c_int, [C.c_void_p, C.c_int32]),
    "bnn_snapshot_read": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_snapshot_read_indicators": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "bnn_set_feature_means": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_read_indicators": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_write_indicators": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_write": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_set_prior_scales": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_set_additional_prob": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_init": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(SamplerConfig), C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_mh_steps": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(Injection), C.c_void_p]),
    "bnn_chains_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_chains_state_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "bnn_chains_gather": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "bnn_forward_time": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "bnn_measure_fp64_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "bnn_chains_set_temperature": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_predict_sample_philox": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_uint64,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_predict_sample_philox_at": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.c_uint64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p]),
    "bnn_predict_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_launch_count": (C.c_int64, [C.c_void_p]),
    "bnn_last_kernel": (C.c_char_p, [C.c_void_p]),
    "bnn_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "bnn_rowshard_config": (C.c_int, [C.c_void_p, C.c_int64]),
    "bnn_rowshard_n_values": (C.c_int, [C.c_void_p]),
    "bnn_rowshard_local": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_rowshard_commit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "bnn_rowshard_update": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(Injection), C.c_void_p]),
    "bnn_debug_read_part": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))


def load(build_if_missing=True):
    """Load the shared library (building it with nvcc if it is absent).  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise NpbnnError("libnpbnn_b200.so is missing: run `python -m npbnn_b200.build`")
        from . import build as _build
        _build.build()
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.bnn_abi_version() != 2:
        raise NpbnnError("libnpbnn_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise NpbnnError(load().bnn_last_error().decode())
