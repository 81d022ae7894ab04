"""ctypes binding of libmjrl_b200.so (the C ABI declared in include/mjrl_b200.h).

The library is the product: if it is missing or cannot be loaded this module raises -- there is no
Python/CPU fallback for any of the entry points.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmjrl_b200.so")


class MjbError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("n_hidden", C.c_int32),
                ("hidden", C.c_int32 * 2), ("vf_hidden", C.c_int32 * 2), ("min_log_std", C.c_float),
                ("max_samples", C.c_int64), ("max_paths", C.c_int32), ("world_size", C.c_int32),
                ("rank", C.c_int32)]


class StepStats(C.Structure):
    _fields_ = [("alpha", C.c_double), ("delta", C.c_double), ("kl_dist", C.c_double),
                ("surr_before", C.c_double), ("surr_after", C.c_double), ("vpg_dot_npg", C.c_double),
                ("backtracks", C.c_int32), ("cg_iters_run", C.c_int32), ("time_vpg_ms", C.c_float),
                ("time_npg_ms", C.c_float), ("time_eval_ms", C.c_float), ("fvp_kernel_ms_sum", C.c_float),
                ("fvp_launches", C.c_int32)]


class BatchStats(C.Structure):
    _fields_ = [("mean_return", C.c_double), ("std_return", C.c_double), ("min_return", C.c_double),
                ("max_return", C.c_double), ("adv_mean", C.c_double), ("adv_std", C.c_double),
                ("n_samples_global", C.c_int64)]


class TransferStats(C.Structure):
    _fields_ = [("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("uploads", C.c_int64)]


# name -> (restype, argtypes); every symbol of include/mjrl_b200.h is listed (tests check the header against this)
_P = C.c_void_p
_SIGNATURES = {
    "mjb_version": (C.c_int, []),
    "mjb_last_error": (C.c_char_p, [_P]),
    "mjb_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "mjb_destroy": (None, [_P]),
    "mjb_synchronize": (C.c_int, [_P]),
    "mjb_comm_unique_id": (C.c_int, [_P]),
    "mjb_comm_init": (C.c_int, [_P, _P]),
    "mjb_ridge_features": (C.c_int, [_P, C.c_int]),
    "mjb_ridge_gram": (C.c_int, [_P, C.c_int, _P]),
    "mjb_ridge_predict": (C.c_int, [_P, C.c_int, _P, _P]),
    "mjb_p2p_export": (C.c_int, [_P, _P]),
    "mjb_p2p_import": (C.c_int, [_P, _P]),
    "mjb_p2p_enable": (C.c_int, [_P, C.c_int]),
    "mjb_p2p_calls": (C.c_longlong, [_P]),
    "mjb_batch_upload": (C.c_int, [_P, C.c_int, C.c_int32, _P, _P, _P, _P, _P]),
    "mjb_batch_upload_flat": (C.c_int, [_P, C.c_int, C.c_int32, _P, _P, _P, _P, _P]),
    "mjb_batch_upload_rollouts": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int, _P, _P]),
    "mjb_batch_set_advantages": (C.c_int, [_P, _P]),
    "mjb_batch_set_baseline": (C.c_int, [_P, _P]),
    "mjb_batch_set_returns": (C.c_int, [_P, _P]),
    "mjb_batch_set_adv_white": (C.c_int, [_P, _P]),
    "mjb_batch_size": (C.c_int64, [_P, C.c_int]),
    "mjb_compute_returns": (C.c_int, [_P, C.c_double]),
    "mjb_vf_predict": (C.c_int, [_P]),
    "mjb_vf_predict_prefit": (C.c_int, [_P]),
    "mjb_compute_advantages": (C.c_int, [_P, C.c_double, C.c_double, C.c_int]),
    "mjb_get_returns": (C.c_int, [_P, _P]),
    "mjb_get_baseline": (C.c_int, [_P, _P]),
    "mjb_get_advantages": (C.c_int, [_P, _P]),
    "mjb_get_adv_white": (C.c_int, [_P, _P]),
    "mjb_process_paths": (C.c_int, [_P, C.POINTER(BatchStats)]),
    "mjb_policy_dim": (C.c_int, [_P]),
    "mjb_policy_set_params": (C.c_int, [_P, _P, C.c_int, C.c_int]),
    "mjb_policy_get_params": (C.c_int, [_P, _P, C.c_int]),
    "mjb_policy_set_transforms": (C.c_int, [_P, _P, _P, _P, _P, C.c_int]),
    "mjb_policy_eval": (C.c_int, [_P, C.POINTER(C.c_double * 2)]),
    "mjb_policy_vpg": (C.c_int, [_P, C.c_int, C.c_double, _P]),
    "mjb_policy_fvp": (C.c_int, [_P, _P, C.c_float, _P, C.c_int64, _P]),
    "mjb_policy_cg": (C.c_int, [_P, _P, C.c_int, C.c_float, C.c_float, _P, C.c_int64, _P]),
    "mjb_policy_step": (C.c_int, [_P, C.c_int, C.c_double, C.c_double, C.c_int, C.c_float, C.c_double, _P,
                                  C.c_int64, C.POINTER(StepStats)]),
    "mjb_policy_set_tensor_cores": (C.c_int, [_P, C.c_int]),
    "mjb_policy_last_vectors": (C.c_int, [_P, _P, _P]),
    "mjb_policy_set_hvp_lengths": (C.c_int, [_P, _P, C.c_int]),
    "mjb_policy_sgd": (C.c_int, [_P, C.c_int, _P, C.c_int64, C.c_int, C.c_float, C.c_float, _P, _P]),
    "mjb_policy_adam_set": (C.c_int, [_P, _P, _P, C.c_int64]),
    "mjb_policy_adam_get": (C.c_int, [_P, _P, _P, C.POINTER(C.c_int64)]),
    "mjb_policy_bc_loss": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double)]),
    "mjb_policy_sgd_timing": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "mjb_vf_dim": (C.c_int, [_P]),
    "mjb_vf_set_state": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "mjb_vf_get_state": (C.c_int, [_P, _P, _P, _P, C.POINTER(C.c_int64)]),
    "mjb_vf_fit": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_float, C.c_float, C.POINTER(C.c_double * 2)]),
    "mjb_vf_fit_begin": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_float, C.c_float, C.POINTER(C.c_double)]),
    "mjb_vf_fit_end": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "mjb_vf_set_tensor_cores": (C.c_int, [_P, C.c_int]),
    "mjb_event_record": (C.c_int, [_P, C.c_int]),
    "mjb_event_elapsed_ms": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "mjb_kernel_launches": (C.c_int64, [_P]),
    "mjb_host_permutation": (C.c_int, [_P, C.POINTER(C.c_int32), C.c_int64, _P]),
    "mjb_fvp_timing": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "mjb_vf_fit_timing": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "mjb_transfer_stats": (C.c_int, [_P, C.POINTER(TransferStats)]),
    "mjb_dev_vf_profile": (C.c_int, [_P, _P, C.c_int]),
    "mjb_dev_lin_profile": (C.c_int, [_P, _P, C.c_int]),
}

_lib = None


def load():
    """dlopen the in-tree library and attach prototypes.  Fails loudly when it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MjbError("%s not built: run `python -m mjrl_b200.build` (or __graft_entry__.build()); "
                       "mjrl_b200 has no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.mjb_version() != 1:
        raise MjbError("libmjrl_b200.so version mismatch")
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)
