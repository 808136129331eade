"""ctypes binding of libpdeip.so (include/pdeip.h).  No torch types cross this boundary:
device pointers are passed as integers, the stream as a void*.

The product path has no CPU fallback: if the library is missing or a call returns a negative
status, a PdeipError is raised with the library's own message.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List

_HERE = os.path.dirname(os.path.abspath(__file__))
# PDEIP_LIB: an instrumented build of the same library (tools/tensor_phase_trace.py); the product path has no other source
LIB_PATH = os.environ.get("PDEIP_LIB") or os.path.join(_HERE, "libpdeip.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "pdeip.h")


class PdeipError(RuntimeError):
    pass


# constants of include/pdeip.h
OK = 0
LAYOUT_AOS, LAYOUT_SOA, LAYOUT_BLOCK128 = 0, 2, 3
TRAJ_PARTICLE_MAJOR, TRAJ_TIME_MAJOR, TRAJ_TIME_SOA, TRAJ_BLOCK128 = 0, 1, 2, 3
DRIFT_NONE, DRIFT_LINEAR, DRIFT_GMM, DRIFT_MEANFIELD, DRIFT_IN_POINTS, DRIFT_MEANFIELD_TABLE = 0, 1, 2, 3, 4, 5
SCHEDULE_REFERENCE, SCHEDULE_UNIFORM = 0, 1
MODEL_MLP, MODEL_GMM, MODEL_QUADRATIC = 0, 1, 2
SET_KFP_0T, SET_KFP_BOUNDARY, SET_FP_0T, SET_FP_BOUNDARY, SET_KMV_PAIRS = 0, 1, 2, 3, 4
PATH_FP32, PATH_TENSOR = 0, 1
SUM_G2, SUM_D2, SUM_D1, SUM_GTRUE2, SUM_GT, SUM_BOUNDARY, SUM_LOSS, SUM_GRADNORM = range(8)
NUM_SUMS = 8

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_f = C.c_float
_u64 = C.c_uint64
_u32 = C.c_uint32
_sz = C.c_size_t

# name -> (restype, argtypes); must list every function declared in include/pdeip.h
SIGNATURES: Dict[str, tuple] = {
    "pdeip_abi_version": (_i, []),
    "pdeip_last_error": (C.c_char_p, []),
    "pdeip_sm_count": (_i, []),
    "pdeip_kl_integrate": (_i, [_p, _p, _p, _p, _l, _i, _i, _f, _f, _i, _p, _i, _f, _p, _p, _u64, _u64, _u32,
                                _i, _i, _i, _i, _i, _i, _p]),
    "pdeip_kl_integrate_path": (_i, [_p, _p, _p, _p, _l, _i, _i, _f, _f, _i, _p, _i, _f, _p, _p, _u64, _u64, _u32,
                                     _i, _i, _i, _i, _i, _i, _i, _p]),
    "pdeip_kl_integrate_model": (_i, [_p, _p, _p, _p, _l, _i, _i, _f, _f, _i, _p, _i, _i, _i, _p, _p, _u64, _u64, _u32,
                                      _i, _i, _i, _i, _i, _i, _i, _p]),
    "pdeip_overdamped_integrate": (_i, [_p, _p, _p, _l, _i, _i, _f, _i, _p, _i, _f, _p, _u64, _u64, _u32, _i, _i, _i,
                                        _i, _i, _i, _p]),
    "pdeip_overdamped_integrate_model": (_i, [_p, _p, _p, _l, _i, _i, _f, _i, _p, _i, _i, _i, _p, _u64, _u64, _u32,
                                              _i, _i, _i, _i, _i, _i, _p]),
    "pdeip_philox_normals": (_i, [_p, _l, _i, _i, _u64, _u64, _u32, _p]),
    "pdeip_philox_uniforms": (_i, [_p, _l, _u64, _u64, _p]),
    "pdeip_philox_raw": (_i, [_p, _p, _p, _l, _p]),
    "pdeip_gaussian_sample": (_i, [_p, _l, _i, _p, _p, _u64, _u64, _i, _p]),
    "pdeip_gaussian_sample_grouped": (_i, [_p, _l, _i, _i, _p, _p, _u64, _u64, _p]),
    "pdeip_ou_exact_sample": (_i, [_p, _p, _l, _i, _p, _p, _p, _p, _p, _f, _f, _u64, _u64, _p]),
    "pdeip_gmm_value_grad": (_i, [_p, _p, _i, _f, _p, _p, _l, _i, _p]),
    "pdeip_linear_grad": (_i, [_p, _p, _p, _l, _i, _p]),
    "pdeip_model_eval": (_i, [_i, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _l, _p]),
    "pdeip_model_num_params": (_l, [_i, _i, _i, _i, _i]),
    "pdeip_residual_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "pdeip_residual_begin": (_i, [_p, _sz, _i, _i, _i, _i, _i, _p]),
    "pdeip_residual_accumulate": (_i, [_p, _sz, _i, _i, _p, _i, _i, _i, _i, _p, _l, _i, _f, _f, _i, _p, _i, _f,
                                       _i, _p]),
    "pdeip_kmv_workspace_bytes": (_sz, [_l, _i, _i]),
    "pdeip_kmv_mean_grad": (_i, [_i, _p, _i, _i, _i, _p, _l, _i, _p, _p, _p, _p, _sz, _p]),
    "pdeip_residual_accumulate_kmv": (_i, [_p, _sz, _i, _p, _i, _i, _i, _p, _l, _i, _p, _p, _p, _f, _p]),
    "pdeip_residual_finalize": (_i, [_p, _sz, _i, _i, _i, _i, _i, _p, _p, _p]),
    "pdeip_adam_l2_step": (_i, [_p, _p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _l, _f, _i, _f, _p, _p]),
    "pdeip_moments_workspace_bytes": (_sz, [_i]),
    "pdeip_ensemble_moments": (_i, [_p, _l, _i, _i, _p, _p, _sz, _p]),
    "pdeip_tensor_path_status": (_i, [_p, _p]),
    "pdeip_debug_umma": (_i, [_i, _p, _p, _p, _i, _i, _p, _p]),
    "pdeip_gather_0T": (_i, [_p, _l, _i, _i, _p, _l, _i, _i, _i, _p, _p]),
    "pdeip_meanfield_noise_sums": (_i, [_p, _l, _i, _i, _u64, _u64, _u32, _p, _p]),
    "pdeip_meanfield_xbar_table": (_i, [_p, _l, _i, _i, _f, _f, _p, _p, _p, _p]),
    "pdeip_kmv_workspace_bytes_ref": (_sz, [_l, _i, _i, _l]),
    "pdeip_kmv_mean_grad_ref": (_i, [_i, _p, _i, _i, _i, _p, _l, _i, _p, _l, _p, _p, _p, _p, _sz, _p]),
    "pdeip_residual_accumulate_kmv_ref": (_i, [_p, _sz, _i, _p, _i, _i, _i, _p, _l, _i, _p, _l, _p, _p, _p, _f, _p]),
    "pdeip_kmv_closure_correction": (_i, [_p, _sz, _p, _i, _l, _i, _p, _p, _f, _p]),
    "pdeip_kmv_density_terms": (_i, [_p, _l, _i, _i, _p, _f, _p, _p, _p, _p]),
}

_lib = None


def header_functions() -> List[str]:
    """Names of every function declared in include/pdeip.h."""
    with open(HEADER_PATH) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pdeip_[a-z0-9_A-Z]+)\s*\(", text)))


def load() -> C.CDLL:
    """Load libpdeip.so and bind every declared symbol.  Raises PdeipError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PdeipError(
            f"{LIB_PATH} not found: the CUDA extension has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C pde_inverse_problem_b200/csrc`). "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:  # pragma: no cover
            raise PdeipError(f"libpdeip.so does not export {name}") from exc
        fn.restype = res
        fn.argtypes = args
    if lib.pdeip_abi_version() != 1:
        raise PdeipError(f"libpdeip.so ABI version {lib.pdeip_abi_version()} != 1")
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != OK:
        msg = load().pdeip_last_error().decode("utf-8", "replace")
        raise PdeipError(f"{what} failed with status {status}: {msg}")
