"""ctypes binding of libyagre_b200.so (include/yagre_b200.h).

There is NO CPU fallback: if the library is missing or cannot be loaded the
import of the backend fails loudly (`BackendUnavailable`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# YAGRE_B200_LIB: development override (an alternative build of the same library, e.g. tools/_build/...)
LIB_PATH = os.environ.get("YAGRE_B200_LIB") or os.path.join(_HERE, "libyagre_b200.so")

YG_ABI_VERSION = 5
YG_MAX_LEVELS = 3
KEEP_DIAGNOSTICS, KEEP_ADAPTATION = 1, 2
YG_MAX_DIM = 8
YG_MAX_DATA_DIM = 8
YG_BIG_MAX_DIM = 64
YG_BIG_MAX_DATA_DIM = 256

YG_OK, YG_ERR_INVALID, YG_ERR_CUDA, YG_ERR_UNSUPPORTED, YG_ERR_ABI, YG_ERR_STATE = 0, -1, -2, -3, -4, -5
MODEL_GAUSS, MODEL_LINEAR, MODEL_LV = 0, 1, 2
EQ_EXACT, EQ_ISCLOSE = 0, 1
NOISE_PHILOX, NOISE_INJECT, NOISE_RECORD = 0, 1, 2
PROPOSAL_MRW, PROPOSAL_PCN = 0, 1

_dp = C.POINTER(C.c_double)


class BackendUnavailable(RuntimeError):
    pass


class YgLevel(C.Structure):
    _fields_ = [("g_mean", _dp), ("g_prec", _dp), ("g_logconst", C.c_double),
                ("n_data", C.c_int32), ("data_dim", C.c_int32),
                ("data", _dp), ("noise_prec", _dp), ("prior_mean", _dp), ("prior_prec", _dp),
                ("G", _dp), ("b", _dp), ("design", _dp),
                ("alpha", C.c_double), ("gamma", C.c_double), ("T", C.c_double),
                ("rk4_steps", C.c_int32), ("tempered", C.c_int32), ("tempering", C.c_double)]


class YgProblem(C.Structure):
    _fields_ = [("prop_L", _dp), ("level", YgLevel * YG_MAX_LEVELS),
                ("proposal", C.c_int32), ("_pad", C.c_int32), ("pcn_step", C.c_double), ("pcn_mean", _dp)]


class YgConfig(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("device", C.c_int32),
                ("n_chains", C.c_int64), ("chain_offset", C.c_int64), ("seed", C.c_uint64),
                ("model", C.c_int32), ("dim", C.c_int32), ("n_levels", C.c_int32),
                ("sub_chain_length", C.c_int32), ("eq_mode", C.c_int32), ("adaptive", C.c_int32),
                ("am_idle_steps", C.c_int64), ("am_collection_steps", C.c_int64),
                ("am_refresh", C.c_int32), ("_pad0", C.c_int32),
                ("am_eps", C.c_double), ("am_scale", C.c_double),
                ("blocks_per_sm", C.c_int32), ("threads_per_block", C.c_int32),
                ("rk4_segment", C.c_int32), ("aem", C.c_int32), ("aem_min_data", C.c_int32),
                ("aem_heuristic", C.c_int32), ("acceptance_only", C.c_int32), ("early_reject_off", C.c_int32)]


class YgNoise(C.Structure):
    _fields_ = [("mode", C.c_int32), ("_pad", C.c_int32),
                ("z_dev", C.c_void_p), ("u_c_dev", C.c_void_p), ("u_f_dev", C.c_void_p)]


class YgOutputs(C.Structure):
    _fields_ = [("samples_dev", C.c_void_p), ("accepted_dev", C.c_void_p), ("logpost_dev", C.c_void_p)]


class YgState(C.Structure):
    _fields_ = [("theta_dev", C.c_void_p), ("logpost_dev", C.c_void_p), ("n_accept_dev", C.c_void_p),
                ("w_mean_dev", C.c_void_p), ("w_m2_dev", C.c_void_p), ("prop_L_dev", C.c_void_p),
                ("am_mean_dev", C.c_void_p), ("am_m2_dev", C.c_void_p),
                ("aem_n_dev", C.c_void_p), ("aem_mean_dev", C.c_void_p), ("aem_m2_dev", C.c_void_p),
                ("aem_cache_dev", C.c_void_p)]


# every symbol include/yagre_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "yg_last_error": (C.c_char_p, []),
    "yg_abi_version": (C.c_uint32, []),
    "yg_create": (C.c_int, [C.POINTER(YgConfig), C.POINTER(C.c_void_p)]),
    "yg_destroy": (C.c_int, [C.c_void_p]),
    "yg_set_problem": (C.c_int, [C.c_void_p, C.POINTER(YgProblem)]),
    "yg_set_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "yg_seek": (C.c_int, [C.c_void_p, C.c_int64]),
    "yg_set_proposal_factor": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "yg_run": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.POINTER(YgOutputs), C.POINTER(YgNoise), C.c_void_p]),
    "yg_get_state": (C.c_int, [C.c_void_p, C.POINTER(YgState), C.c_void_p]),
    "yg_load_state": (C.c_int, [C.c_void_p, C.POINTER(YgState), C.c_int64, C.c_int64, C.c_int64, C.c_void_p]),
    "yg_get_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "yg_logpost": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "yg_iat_ess": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_double,
                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "yg_pooled_len": (C.c_int64, [C.c_int32]),
    "yg_pooled_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "yg_split_moments": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "yg_pooled_samples_workspace_len": (C.c_int64, [C.c_int32, C.c_int64]),
    "yg_pooled_samples": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_void_p]),
    "yg_fp64_peak": (C.c_int, [C.c_int32, C.c_double, C.POINTER(C.c_double)]),
    "yg_rk4_loop_rate": (C.c_int, [C.c_int32, C.c_double, C.POINTER(C.c_double)]),
    "yg_fp64_tensor_peak": (C.c_int, [C.c_int32, C.c_double, C.POINTER(C.c_double)]),
    "yg_last_launch": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int64)]),
}

_lib = None


def load():
    """Loads the shared library and types every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BackendUnavailable(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C yagre_mcmc_b200/csrc). There is no CPU fallback.")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:
        raise BackendUnavailable(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.yg_abi_version() != YG_ABI_VERSION:
        raise BackendUnavailable(f"ABI mismatch: library {lib.yg_abi_version()} vs binding {YG_ABI_VERSION}")
    _lib = lib
    return lib


def last_error():
    return load().yg_last_error().decode("utf-8", "replace")


def check(rc):
    """Maps yg_status to the exception types the reference raises for the same faults:
    ValueError for bad builder configuration (chain/builder.py:42-50, mrw.py:88-91),
    NotImplementedError where the reference says so (chain/adaptive.py:41-43),
    RuntimeError otherwise."""
    if rc == YG_OK:
        return
    msg = last_error()
    if rc == YG_ERR_INVALID:
        raise ValueError(msg)
    if rc == YG_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"libyagre_b200 error {rc}: {msg}")
