"""
ctypes binding of libevcplm.so (C ABI declared in include/evcplm.h).

There is NO fallback: if the CUDA library is missing or cannot be loaded the
import of the engine fails loudly (EngineUnavailableError).  Build it in-tree
with ``python -c "import __graft_entry__ as g; g.build()"`` or
``evcouplings_b200/csrc/build.sh``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libevcplm.so")
ABI_VERSION = 2
EVC_NOT_SPD = 2      # evc_spd_inverse_f64: the matrix is not positive definite


class EngineUnavailableError(RuntimeError):
    """libevcplm.so (the sm_100a CUDA engine) is missing / unloadable / has no device."""


class EngineError(RuntimeError):
    """A libevcplm call returned non-zero."""


c_void_p = ctypes.c_void_p
c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_f32 = ctypes.c_float
c_f64 = ctypes.c_double


class FitParams(ctypes.Structure):
    """evc_fit_params_t (include/evcplm.h)."""
    _fields_ = [("max_iterations", c_i32), ("m", c_i32), ("epsilon", c_f32), ("lambda_h", c_f32),
                ("lambda_J", c_f32), ("max_linesearch", c_i32), ("min_step", c_f64), ("max_step", c_f64),
                ("ftol", c_f64), ("gtol", c_f64), ("xtol", c_f64), ("precision_schedule", c_i32),
                ("switch_factor", c_f32)]


class FitResult(ctypes.Structure):
    """evc_fit_result_t (include/evcplm.h)."""
    _fields_ = [("status", c_i32), ("iterations", c_i32), ("evaluations", c_i32), ("switched_at", c_i32),
                ("fx", c_f64), ("negloglk", c_f64), ("seconds", c_f64)]


ALLREDUCE_CB = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, c_i64, ctypes.c_void_p)
PROGRESS_CB = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, c_i32, c_f64, c_f64, c_f64, c_f64, c_i32, c_f64,
                               c_f64, c_f64)

# status codes of evc_plm_fit -> libLBFGS names (what plmc prints after "Gradient optimization:")
LBFGS_STATUS = {
    0: "LBFGS_SUCCESS", 2: "LBFGS_ALREADY_MINIMIZED", -1021: "LBFGSERR_CANCELED",
    -1000: "LBFGSERR_INVALIDPARAMETERS", -1001: "LBFGSERR_MINIMUMSTEP", -1002: "LBFGSERR_MAXIMUMSTEP",
    -1003: "LBFGSERR_MAXIMUMLINESEARCH", -1004: "LBFGSERR_MAXIMUMITERATION", -1005: "LBFGSERR_WIDTHTOOSMALL",
    -1006: "LBFGSERR_ROUNDING_ERROR", -1007: "LBFGSERR_INCREASEGRADIENT",
}

# name -> (restype, argtypes); mirrors include/evcplm.h one to one
PROTOTYPES = {
    "evc_abi_version": (ctypes.c_int, []),
    "evc_last_error": (ctypes.c_char_p, []),
    "evc_device_count": (ctypes.c_int, []),
    "evc_device_info": (ctypes.c_int, [c_i32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "evc_hamming_counts": (ctypes.c_int, [c_void_p, c_i64, c_i32, c_i32, c_i32, c_void_p]),
    "evc_hamming_plane_words": (c_i64, [c_i64, c_i32]),
    "evc_hamming_num_tiles": (c_i64, [c_i64]),
    "evc_hamming_pack": (ctypes.c_int, [c_void_p, c_i64, c_i32, c_void_p, c_void_p]),
    "evc_hamming_count_tiles": (ctypes.c_int, [c_void_p, c_i64, c_i32, c_i32, c_i64, c_i64, c_void_p, c_void_p]),
    "evc_a2m_scan": (ctypes.c_int, [ctypes.c_char_p, c_void_p, c_void_p, c_void_p]),
    "evc_a2m_read": (ctypes.c_int, [ctypes.c_char_p, c_i64, c_i64, c_void_p, c_void_p, c_i64]),
    "evc_msa_encode": (ctypes.c_int, [c_void_p, c_i64, c_i64, c_void_p, c_void_p, c_i64, c_void_p, c_void_p, c_void_p]),
    "evc_identities_to_seq": (ctypes.c_int, [c_void_p, c_void_p, c_i64, c_i32, c_void_p, c_void_p]),
    "evc_plm_create": (ctypes.c_int, [c_void_p, c_void_p, c_i64, c_i32, c_i32, c_i32, c_void_p, c_i32]),
    "evc_plm_destroy": (None, [c_void_p]),
    "evc_plm_num_params": (c_i64, [c_void_p]),
    "evc_plm_eval_data": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "evc_plm_set_backward": (ctypes.c_int, [c_void_p, c_i32]),
    "evc_plm_set_forward": (ctypes.c_int, [c_void_p, c_i32]),
    "evc_plm_set_precision": (ctypes.c_int, [c_void_p, c_i32]),
    "evc_fit_default_params": (None, [c_void_p]),
    "evc_plm_fit": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "evc_plm_pack_fx": (ctypes.c_int, [c_void_p, c_void_p, c_void_p]),
    "evc_plm_unpack_fx": (ctypes.c_int, [c_void_p, c_void_p, c_void_p]),
    "evc_plm_set_profiling": (ctypes.c_int, [c_void_p, c_i32]),
    "evc_plm_last_stage_ms": (ctypes.c_int, [c_void_p, c_void_p]),
    "evc_plm_add_regulariser": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_f32, c_void_p]),
    "evc_plm_eval_host": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_f32]),
    "evc_plm_weighted_counts": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "evc_vec_dot": (ctypes.c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p]),
    "evc_vec_axpby": (ctypes.c_int, [c_void_p, c_void_p, c_f32, c_f32, c_i64, c_void_p]),
    "evc_vec_copy": (ctypes.c_int, [c_void_p, c_void_p, c_i64, c_void_p]),
    "evc_vec_sub": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_i64, c_void_p]),
    "evc_lbfgs_direction": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_i64, c_i32, c_i32, c_i32, c_void_p]),
    "evc_lbfgs_update_pair": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_i64, c_void_p]),
    "evc_ec_scores": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "evc_plm_energies": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "evc_fn_scores": (ctypes.c_int, [c_void_p, c_i32, c_i32, c_void_p, c_void_p]),
    "evc_mf_weighted_counts_f64": (ctypes.c_int, [c_void_p, c_void_p, c_i64, c_i32, c_i32, c_f64, c_void_p, c_void_p]),
    "evc_mf_covariance": (ctypes.c_int, [c_void_p, c_i32, c_i32, c_f64, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p]),
    "evc_spd_inverse_f64": (ctypes.c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_void_p]),
    "evc_mf_couplings_fields": (ctypes.c_int, [c_void_p, c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_void_p]),
    "evc_mf_di_scores": (ctypes.c_int, [c_void_p, c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_void_p]),
    "evc_ec_scores_f64": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_i32, c_i32, c_void_p, c_void_p, c_void_p,
                                         c_void_p]),
}

_lib = None


def load():
    """Load libevcplm.so and bind every symbol of the C ABI (no device needed)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineUnavailableError(
            "CUDA engine library not built: %s is missing. There is no CPU fallback; "
            "build it with evcouplings_b200/csrc/build.sh (nvcc, sm_100a)." % LIB_PATH)
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:
        raise EngineUnavailableError("cannot load %s: %s" % (LIB_PATH, e))
    for name, (restype, argtypes) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise EngineUnavailableError("%s does not export %s" % (LIB_PATH, name))
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.evc_abi_version() != ABI_VERSION:
        raise EngineUnavailableError("libevcplm ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().evc_last_error()
        raise EngineError("%s failed: %s" % (what or "libevcplm call", msg.decode() if msg else "unknown error"))


def require_device():
    """Raise unless at least one CUDA device is usable through the library."""
    lib = load()
    n = lib.evc_device_count()
    if n <= 0:
        raise EngineUnavailableError(
            "libevcplm found no CUDA device; the PLM engine has no CPU fallback")
    return n
