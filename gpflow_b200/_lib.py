"""ctypes binding of libgpk.so (include/gpk.h).  There is NO CPU fallback: if the CUDA library
cannot be loaded the product path raises, and every numeric call needs a CUDA device."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_void_p
from typing import Optional

GPK_F32, GPK_F64 = 0, 1
GPK_FULL, GPK_LOWER = 0, 1
GPK_GEMM_LOWER_ONLY, GPK_GEMM_A_LOWER, GPK_GEMM_COLSUMSQ = 1, 2, 4
GPK_MAX_CHILDREN = 8

(K_RBF, K_MATERN12, K_MATERN32, K_MATERN52, K_RQ, K_EXPONENTIAL, K_LINEAR, K_WHITE, K_CONSTANT, K_SUM,
 K_PRODUCT, K_POLYNOMIAL) = range(12)


class KNode(ctypes.Structure):
    """Mirror of `gpk_knode` (include/gpk.h)."""

    _fields_ = [
        ("op", c_int32),
        ("n_children", c_int32),
        ("child", c_int32 * GPK_MAX_CHILDREN),
        ("variance", c_double),
        ("lengthscale", c_double),
        ("alpha", c_double),
        ("n_dims", c_int32),
        ("dims_off", c_int32),
        ("n_ard", c_int32),
        ("ard_off", c_int32),
    ]


KAUX_COSINE, KAUX_PERIODIC, KAUX_ARCCOS, KAUX_COREGION = range(4)
GPK_KAUX_MAXD = 32


class KAux(ctypes.Structure):
    """Mirror of `gpk_kaux` (include/gpk.h): kernels that are not functions of a Gram term."""

    _fields_ = [
        ("op", c_int32), ("base", c_int32), ("order", c_int32), ("n_dims", c_int32), ("table_dim", c_int32),
        ("pad_", c_int32), ("variance", c_double), ("alpha", c_double), ("bias", c_double), ("table", c_void_p),
        ("dims", c_int32 * GPK_KAUX_MAXD), ("scale", c_double * GPK_KAUX_MAXD), ("period", c_double * GPK_KAUX_MAXD),
    ]


_KN = POINTER(KNode)
_I32 = POINTER(c_int32)
_F64 = POINTER(c_double)

# name -> (restype, argtypes); every symbol include/gpk.h declares
SIGNATURES = {
    "gpk_version": (c_int, []),
    "gpk_last_error": (c_char_p, []),
    "gpk_kbuild": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64,
                           c_void_p, c_int64, c_int, c_int, c_double, c_void_p, c_void_p]),
    "gpk_kdiag": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    "gpk_potrf_ws": (c_size_t, [c_int64, c_int64, c_int]),
    "gpk_potrf": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "gpk_potrf_batched_ws": (c_size_t, [c_int64, c_int, c_int]),
    "gpk_potrf_batched": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gpk_trsm_ws": (c_size_t, [c_int64, c_int]),
    "gpk_trsm": (c_int, [c_int, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p,
                         c_void_p]),
    "gpk_gemm": (c_int, [c_int, c_int, c_int64, c_int64, c_int64, c_double, c_void_p, c_int64, c_void_p, c_int64,
                         c_double, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "gpk_colsumsq": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_double, c_int, c_void_p, c_int, c_void_p]),
    "gpk_reduce": (c_int, [c_int, c_void_p, c_int64, c_int64, c_double, c_int, c_void_p, c_int, c_void_p]),
    "gpk_tril_sumsq": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_double, c_int, c_void_p, c_int,
                               c_void_p]),
    "gpk_axpby": (c_int, [c_int64, c_int64, c_double, c_void_p, c_int64, c_double, c_void_p, c_int64, c_int,
                          c_void_p]),
    "gpk_scale_cols": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p]),
    "gpk_scale_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p]),
    "gpk_add_diag": (c_int, [c_void_p, c_int64, c_int64, c_double, c_void_p, c_int, c_void_p]),
    "gpk_fill": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_double, c_int, c_void_p]),
    "gpk_tril": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "gpk_transpose": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "gpk_gaussian_varexp_sum": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_double, c_int,
                                        c_void_p, c_int, c_void_p]),
    "gpk_gaussian_log_density": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_double, c_void_p, c_int,
                                         c_void_p]),
    "gpk_kaux": (c_int, [POINTER(KAux), c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int,
                         c_void_p]),
    "gpk_kaux_diag": (c_int, [POINTER(KAux), c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p]),
    "gpk_changepoint_weights": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_double, c_double, c_int, c_double,
                                        c_double, c_void_p, c_int, c_void_p]),
    "gpk_clamp_min": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_double, c_int, c_int, c_void_p]),
    "gpk_hadamard": (c_int, [c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "gpk_launch_count": (c_int64, []),
    "gpk_launch_count_reset": (None, []),
    "gpk_debug_leaf": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "gpk_debug_trace": (c_int, [c_void_p, c_void_p, ctypes.c_uint]),
    "gpk_prof_enable": (c_int, [c_int]),
    "gpk_prof_read": (c_int, [_F64, POINTER(c_int64), c_int]),
    "gpk_prof_read2": (c_int, [_F64, POINTER(c_int64), _F64, c_int]),
    "gpk_peak_probe": (c_int, [_F64, c_void_p]),
    "gpk_potrf_last_slices": (c_int, []),
    "gpk_warm": (c_int, [c_size_t, c_void_p]),
    "gpk_gpr_lml_ws": (c_size_t, [c_int64, c_int64, c_int]),
    "gpk_gpr_lml": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_double,
                            c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "gpk_gpr_lml_grad_ws": (c_size_t, [c_int64, c_int64, c_int]),
    "gpk_gpr_lml_grad": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_double,
                                 c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "gpk_sgpr_elbo_ws": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "gpk_sgpr_elbo": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                              c_void_p, c_int64, c_int64, c_double, c_double, c_int, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p]),
    "gpk_sgpr_elbo_grad_ws": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "gpk_sgpr_elbo_grad": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                   c_void_p, c_int64, c_int64, c_double, c_double, c_int, c_void_p, c_int, c_void_p,
                                   c_int64, c_void_p, c_void_p]),
    "gpk_svgp_elbo_ws": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "gpk_svgp_elbo": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                              c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_double, c_double,
                              c_double, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "gpk_svgp_elbo_A": (c_size_t, [c_int64, c_int64, c_int64, c_int, POINTER(c_int64)]),
    "gpk_svgp_elbo_staged": (c_int, [_KN, c_int, _I32, _F64, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                     c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int, c_int, c_double, c_double,
                                     c_double, c_int, c_int, c_int, c_int64, c_int64, c_int, c_void_p, c_void_p,
                                     c_void_p]),
}

# GPFLOW_B200_LIB selects another build of the same ABI (kernel experiments); default = the in-tree library
LIB_PATH = os.environ.get("GPFLOW_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libgpk.so")
_lib: Optional[ctypes.CDLL] = None


class GpkError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Loads libgpk.so (building it in-tree with nvcc if it is absent and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build

        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise GpkError(
                f"libgpk.so is missing and could not be built ({e}); gpflow_b200 has no CPU fallback"
            ) from e
    elif "GPFLOW_B200_LIB" not in os.environ:
        # a library older than its sources is a silent trap while developing kernels: rebuild when asked to, else warn
        try:
            from . import build as _build

            if _build.needs_build():
                if os.environ.get("GPFLOW_B200_AUTOBUILD") == "1":
                    _build.build()
                else:
                    import sys
                    sys.stderr.write("gpflow_b200: libgpk.so is older than csrc/ or include/gpk.h "
                                     "(python -m gpflow_b200.build, or GPFLOW_B200_AUTOBUILD=1)\n")
        except Exception:  # noqa: BLE001  (no nvcc on a deployment box: the shipped library is what runs)
            pass
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.gpk_version() != 1:
        raise GpkError(f"libgpk.so ABI version {lib.gpk_version()} != 1")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().gpk_last_error().decode("utf-8", "replace")
        if status == -1:
            raise ValueError(f"{what}: {msg}")
        raise GpkError(f"{what}: {msg} (status {status})")
