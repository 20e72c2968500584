"""ctypes binding of libss_b200.so (include/ss_b200.h).  Fails loudly: there is no
CPU fallback behind this module."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libss_b200.so")

SS_OK, SS_EINVAL, SS_ECUDA, SS_ESINGULAR, SS_ESTATE, SS_EUNSUPPORTED = 0, -1, -2, -3, -4, -5
PENALTY_REFERENCE, PENALTY_PER_SAMPLE = 0, 1
PRECISION_FP32, PRECISION_BF16_TC, PRECISION_AUTO, PRECISION_FP64 = 0, 1, 2, 3

_c_double_p = C.POINTER(C.c_double)
_c_float_p = C.POINTER(C.c_float)
_c_int64_p = C.POINTER(C.c_int64)
_c_int_p = C.POINTER(C.c_int)

# name -> (restype, argtypes); kept in one table so tests can check it against the header
class ValueNetStruct(C.Structure):
    """ss_value_net of include/ss_b200.h."""
    _fields_ = ([(n, C.c_int) for n in ("d", "da", "h1a", "h2a", "h1c", "h2c", "layer_norm", "last_layer_tanh")] +
                [(n, C.c_void_p) for n in ("aW1", "ab1", "ag1", "abe1", "aW2", "ab2", "ag2", "abe2", "aW3", "ab3",
                                           "cW1", "cb1", "cg1", "cbe1", "cW2", "cb2", "cg2", "cbe2", "cW3", "cb3",
                                           "obs_mean", "obs_std")] +
                [("obs_clip_lo", C.c_double), ("obs_clip_hi", C.c_double), ("has_ret_norm", C.c_int),
                 ("ret_mean", C.c_double), ("ret_std", C.c_double), ("ret_clip_lo", C.c_double),
                 ("ret_clip_hi", C.c_double)])


SIGNATURES = {
    "ss_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "ss_destroy": (C.c_int, [C.c_void_p]),
    "ss_last_error": (C.c_char_p, [C.c_void_p]),
    "ss_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ss_device_info": (C.c_int, [C.c_void_p, _c_int_p, _c_int_p, _c_int_p, _c_int_p]),
    "ss_last_timings": (C.c_int, [C.c_void_p, _c_float_p, C.POINTER(C.c_char_p), C.c_int]),
    "ss_launch_count": (C.c_int64, [C.c_void_p]),
    "ss_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "ss_host_alloc": (C.c_void_p, [C.c_int64]),
    "ss_host_free": (None, [C.c_void_p]),
    "ss_device_alloc": (C.c_void_p, [C.c_int64]),
    "ss_device_free": (None, [C.c_void_p]),
    "ss_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "ss_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "ss_kde_ucb_argmax": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                    C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                    C.c_void_p, C.c_void_p, _c_int64_p, _c_double_p]),
    "ss_kde_ucb_argmax_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                        C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                        C.c_void_p, C.c_void_p, _c_int64_p, _c_double_p]),
    "ss_kde_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "ss_mpc_set_model": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)] + [C.c_void_p] * 6),
    "ss_mpc_set_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "ss_mpc_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                              C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                              C.c_int, C.c_int, _c_int64_p, _c_double_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    "ss_mpc_rollout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                 C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                 C.c_int, C.c_int]),
    "ss_mpc_projection_sums": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), _c_int_p]),
    "ss_mpc_finish": (C.c_int, [C.c_void_p, _c_int64_p, _c_double_p, C.c_void_p]),
    "ss_mpc_finish_package": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), _c_int_p]),
    "ss_mpc_read_package": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "ss_mpc_get_states": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ss_mpc_forward_sim": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                     C.c_void_p]),
    "ss_mpc_replay": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "ss_mpc_sample_actions": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_uint64,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "ss_mpc_tc_supported": (C.c_int, [C.c_void_p]),
    "ss_mpc_last_kernel": (C.c_int, [C.c_void_p]),
    "ss_mt19937_uniform": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                     C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ss_mt19937_state": (C.c_int, [C.c_void_p, C.c_void_p, _c_int_p]),
    "ss_mpc_plan_mt19937": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                      C.c_int, C.c_int, _c_int64_p, _c_double_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ss_mt19937_jump_poly": (C.c_int, [C.c_uint64, C.c_void_p]),
    "ss_mt19937_phi_exponents": (C.c_int, [_c_int_p, C.c_int]),
    "ss_py_random_sample": (C.c_int, [C.c_void_p, _c_int_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "ss_peer_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "ss_peer_open": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "ss_peer_close": (C.c_int, [C.c_void_p]),
    "ss_peer_ready": (C.c_int, [C.c_void_p]),
    "ss_peer_argmax_merge": (C.c_int, [C.c_void_p, C.c_double, C.c_int64, _c_double_p, _c_int64_p]),
    "ss_dyn_set_data": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]),
    "ss_dyn_train_batches": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double,
                                       C.c_void_p]),
    "ss_dyn_eval_loss": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_double_p, _c_int_p]),
    "ss_dyn_commit": (C.c_int, [C.c_void_p]),
    "ss_dyn_get_params": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "ss_dyn_reset_optimizer": (C.c_int, [C.c_void_p]),
    "ss_dyn_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "ss_value_net_set": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ss_value_net_eval": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "ss_mirror_write": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_void_p]),
    "ss_mirror_reset": (C.c_int, [C.c_void_p]),
    "ss_kde_ucb_argmax_mirror": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                           C.c_int64, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p,
                                           _c_int64_p, _c_double_p]),
    "ss_path_shortcut": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p,
                                   _c_int_p]),
    "ss_path_close_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p,
                                      C.c_int64, _c_int64_p]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load():
    """dlopen libss_b200.so and declare every entry point.  Raises LibraryMissing when the
    shared object has not been built (python -m smartstartcontinuous_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            "libss_b200.so is not built: run `python -m smartstartcontinuous_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError = symbol missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
