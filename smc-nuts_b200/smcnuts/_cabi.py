"""ctypes binding of include/smcnuts_b200.h (the drop-in C-ABI)."""
import ctypes
import re
from pathlib import Path

_PKG = Path(__file__).resolve().parent
import os
# SMCB_LIB_PATH: load another build of the same library (A/B experiments of kernel variants on the GPU box)
LIB_PATH = Path(os.environ.get("SMCB_LIB_PATH") or (_PKG / "_lib" / "libsmcnuts_b200.so"))
HEADER = _PKG.parents[1] / "include" / "smcnuts_b200.h"

MODEL_KINDS = {"arma": 0, "PRMwCD": 1, "gauss": 2}
STREAM_NUTS, STREAM_MOMENTUM, STREAM_ACCREJ, STREAM_RESAMPLE, STREAM_INIT, STREAM_ESTIMATE = range(6)
CONSTRAIN_NONE, CONSTRAIN_EXP_LAST = 0, 1
CONSTRAIN_MODEL = 2   # host side only: constrain through the model (smcb_model_constrain) first, then unconstrained moments

_vp, _ll, _i, _d = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_double
_u64, _u32 = ctypes.c_uint64, ctypes.c_uint32

# name -> argtypes (restype is int unless listed in _RESTYPES); pointers are passed as integers (void*)
_SIGS = {
    "smcb_model_create": [_i, _vp, _ll, _i, ctypes.POINTER(_vp)],
    "smcb_model_create_plugin": [ctypes.c_char_p, _vp, _ll, ctypes.POINTER(_vp)],
    "smcb_model_set_scale": [_vp, _vp],
    "smcb_model_destroy": [_vp],
    "smcb_model_dim": [_vp],
    "smcb_model_constrained_dim": [_vp],
    "smcb_model_constrain": [_vp, _vp, _ll, _vp, _vp],
    "smcb_debug_pack_prm": [_vp, _i, _i, _vp, _ll],
    "smcb_logp_grad": [_vp, _vp, _ll, _d, _vp, _vp, _vp, _vp],
    "smcb_combine_logp": [_vp, _vp, _d, _ll, _vp, _vp],
    "smcb_nuts_workspace_bytes": [_vp, _ll, _i, ctypes.POINTER(_ll)],
    "smcb_nuts_set_blocks_per_sm": [_i],
    "smcb_nuts_transition": [_vp, _vp, _vp, _ll, _d, _d, _i, _i, _u64, _u32, _u64] + [_vp] * 16 + [_vp, _ll, _vp],
    "smcb_normals": [_u64, _u32, _u32, _u64, _ll, _i, _vp, _vp],
    "smcb_uniforms": [_u64, _u32, _u32, _u64, _ll, _u32, _vp, _vp],
    "smcb_row_half_sqnorm": [_vp, _ll, _i, _vp, _vp],
    "smcb_init_logw": [_vp, _vp, _ll, _i, _vp, _vp],
    "smcb_std_normal_logpdf": [_vp, _ll, _i, _vp, _vp],
    "smcb_uniform_logw": [_vp, _ll, _ll, _vp, _vp],
    "smcb_affine": [_vp, _ll, _d, _d, _vp, _vp],
    "smcb_reweight_forward": [_vp, _vp, _vp, _vp, _vp, _ll, _i, _vp, _vp],
    "smcb_reweight_forward_ke": [_vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp],
    "smcb_reweight_forward_split": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _ll, _vp, _vp],
    "smcb_reweight_general": [_vp, _vp, _vp, _vp, _vp, _ll, _vp, _vp],
    "smcb_reweight_asymptotic": [_vp, _vp, _vp, _d, _d, _ll, _vp, _vp],
    "smcb_lse_partial": [_vp, _ll, _vp, _vp, _vp],
    "smcb_lse_finalize": [_vp, _i, _vp, _vp],
    "smcb_normalise": [_vp, _ll, _vp, _vp, _vp],
    "smcb_tempering_arrays": [_vp, _vp, _d, _ll, _vp, _vp, _vp, _vp],
    "smcb_ess_multi_phi": [_vp, _vp, _vp, _ll, _vp, _i, _vp, _vp, _vp],
    "smcb_bisect_state_bytes": [],
    "smcb_bisect_max_candidates": [],
    "smcb_bisect_passes": [],
    "smcb_bisect_init": [_vp, _d, _d, _d, _vp],
    "smcb_bisect_eval": [_vp, _vp, _d, _ll, _vp, _vp, _vp, _vp],
    "smcb_bisect_step": [_vp, _i, _vp, _vp],
    "smcb_bisect_read": [_vp, _vp, _vp],
    "smcb_cdf": [_vp, _ll, _vp, _vp, _vp, _vp, _vp, _vp],
    "smcb_normalise_tilesums": [_vp, _ll, _vp, _vp, _vp, _vp, _vp],
    "smcb_cdf_from_tilesums": [_vp, _ll, _vp, _vp, _vp, _vp],
    "smcb_ancestors_multinomial": [_vp, _ll, _vp, _ll, _vp, _vp],
    "smcb_ancestors_systematic": [_vp, _ll, _d, _ll, _ll, _ll, _vp, _vp],
    "smcb_resample_systematic": [_vp, _ll, _d, _vp, _ll, _ll, _ll, _vp, _i, _vp, _vp, _vp, _vp],
    "smcb_resample_workspace_bytes": [_ll, _i],
    "smcb_resample_systematic_push": [_vp, _ll, _d, _ll, _ll, _ll, _vp, _i, _vp, _ll, _vp, _vp, _vp],
    "smcb_resample_multinomial_push": [_vp, _ll, _vp, _i, _i, _u64, _u32, _u32, _ll, _ll, _vp, _i, _vp, _vp, _ll, _vp],
    "smcb_rank_offsets": [_vp, _i, _i, _vp, _vp],
    "smcb_peer_alloc": [_ll, ctypes.POINTER(_vp), _vp],
    "smcb_peer_open": [_vp, ctypes.POINTER(_vp)],
    "smcb_peer_close": [_vp],
    "smcb_peer_free": [_vp],
    "smcb_gather_rows": [_vp, _vp, _ll, _i, _vp, _vp],
    "smcb_weighted_moment": [_vp, _vp, _ll, _i, _i, _vp, _i, _vp, _vp, _vp],
    "smcb_weighted_moments12": [_vp, _vp, _ll, _i, _i, _vp, _vp, _vp, _vp],
    "smcb_moments12_finalize": [_vp, _vp, _i, _vp, _vp, _vp],
    "smcb_count_moved": [_vp, _vp, _ll, _i, _vp, _vp, _vp],
    "smcb_gaussL_sums": [_vp, _vp, _ll, _i, _vp, _vp],
    "smcb_gaussL_gram": [_vp, _vp, _ll, _i, _vp, _vp, _vp],
    "smcb_gaussL_factor": [_vp, _ll, _i, _d, _vp, _vp, _vp, _vp],
    "smcb_gaussL_logpdf": [_vp, _vp, _ll, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "smcb_gaussL_logpdf_scratch_bytes": [_i],
    "smcb_sum_int32": [_vp, _ll, _vp, _vp, _vp],
    "smcb_sum_f64": [_vp, _ll, _vp, _vp, _vp],
    "smcb_scale_rows": [_vp, _ll, _i, _vp, _i, _vp, _vp],
    "smcb_fast_exp": [_vp, _ll, _vp, _vp],
    "smcb_fast_log": [_vp, _ll, _vp, _vp],
    "smcb_probe_fp64": [_i, _i, _i, _vp, _vp],
    "smcb_probe_dmma": [_i, _i, _i, _vp, _vp],
    "smcb_debug_dmma": [_vp, _vp, _vp, _vp, _i, _vp],
    "smcb_build_flavour": [],
    "smcb_version": [],
    "smcb_last_error": [],
    "smcb_launch_count": [],
    "smcb_reduce_workspace_bytes": [],
    "smcb_scan_workspace_bytes": [_ll],
}
_RESTYPES = {"smcb_last_error": ctypes.c_char_p, "smcb_launch_count": _ll, "smcb_reduce_workspace_bytes": _ll,
             "smcb_scan_workspace_bytes": _ll, "smcb_bisect_state_bytes": _ll, "smcb_resample_workspace_bytes": _ll,
             "smcb_gaussL_logpdf_scratch_bytes": _ll}

_LIB = None


class SmcbError(RuntimeError):
    pass


def declared_symbols():
    """Every function name declared in include/smcnuts_b200.h."""
    text = HEADER.read_text()
    return sorted(set(re.findall(r"\b(smcb_[a-zA-Z0-9_]+)\s*\(", text)))


def lib():
    """Load the CUDA library; fail loudly when it has not been built (no CPU fallback exists)."""
    global _LIB
    if _LIB is None:
        if not LIB_PATH.exists():
            raise SmcbError(f"{LIB_PATH} is missing: build it with `python smc-nuts_b200/build_ext.py` "
                            "(the smcnuts device path has no CPU fallback)")
        L = ctypes.CDLL(str(LIB_PATH))
        for name, args in _SIGS.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, ctypes.c_int)
        _LIB = L
    return _LIB


PARITY_LIB_PATH = _PKG / "_lib" / "libsmcnuts_b200_parity.so"


class use_library:
    """Context manager for the parity tests: route the C-ABI calls of this process to another build of the library
    (normally libsmcnuts_b200_parity.so).  Model handles are per library: create, use and drop models inside the block."""

    def __init__(self, path):
        self.path = Path(path)

    def __enter__(self):
        global _LIB, LIB_PATH
        self._saved = (_LIB, LIB_PATH, dict(_FN))
        _LIB, LIB_PATH = None, self.path
        _FN.clear()
        return lib()

    def __exit__(self, *exc):
        global _LIB, LIB_PATH
        _LIB, LIB_PATH = self._saved[:2]
        _FN.clear()
        _FN.update(self._saved[2])
        return False


_FN = {}


def call(name, *args):
    """Invoke a status-returning entry point and raise SmcbError on failure."""
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(lib(), name)
    rc = fn(*args)
    if rc != 0:
        raise SmcbError(f"{name} failed ({rc}): {lib().smcb_last_error().decode()}")
    return rc
