"""ctypes binding of ``libtbk.so`` (C ABI declared in ``include/tbk.h``).

The library is loaded from the package directory (built in-tree by ``tbmodels_b200.build``).  There is
no fallback of any kind: if the shared object is missing the import of this module raises, and every
compute entry point fails when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtbk.so")

#: every symbol ``include/tbk.h`` declares (tests check that the shared object exports all of them)
SYMBOLS = (
    "tbk_version",
    "tbk_last_error",
    "tbk_model_create",
    "tbk_kdotp_create",
    "tbk_supercell_create",
    "tbk_model_vectors",
    "tbk_model_destroy",
    "tbk_model_info",
    "tbk_hamilton",
    "tbk_eigenval",
    "tbk_eigenval_push",
    "tbk_eigenval_mesh",
    "tbk_eigenval_mesh_host",
    "tbk_mesh_factorised",
    "tbk_eigh",
    "tbk_eigh_host",
    "tbk_band_velocity",
    "tbk_band_velocity_host",
    "tbk_berry_curvature",
    "tbk_berry_curvature_host",
    "tbk_kdotp_coefficients",
    "tbk_kdotp_coefficients_host",
    "tbk_hamilton_host",
    "tbk_eigenval_host",
    "tbk_model_check",
    "tbk_launch_count",
    "tbk_workspace_bytes",
    "tbk_profile",
    "tbk_profile_read",
    "tbk_host_alloc",
    "tbk_host_free",
    "tbk_measure_fp64_peak",
    "tbk_measure_int8_peak",
    "tbk_host_tridiag_ql",
    "tbk_host_tridiag_bisect",
    "tbk_host_sincospi",
    "tbk_host_hetrd",
    "tbk_host_pack_weights",
)

TBK_OK, TBK_E_INVALID, TBK_E_CUDA, TBK_E_UNSUPPORTED, TBK_E_NOCONV = 0, 1, 2, 3, 4


class TbkError(RuntimeError):
    """A libtbk call returned a non-zero status."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libtbk error {code}: {message}")
        self.code = code
        self.message = message


_lib = None


def load() -> C.CDLL:
    """Load libtbk.so (once) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m tbmodels_b200.build` "
            "(tbmodels_b200 has no CPU fallback)"
        )
    lib = C.CDLL(LIB_PATH)
    dp = C.POINTER(C.c_double)
    vp = C.c_void_p
    lib.tbk_version.restype = C.c_int
    lib.tbk_last_error.restype = C.c_char_p
    lib.tbk_model_create.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.POINTER(vp)]
    lib.tbk_model_create.restype = C.c_int
    lib.tbk_kdotp_create.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, C.POINTER(vp)]
    lib.tbk_kdotp_create.restype = C.c_int
    lib.tbk_supercell_create.argtypes = [C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int, C.POINTER(vp)]
    lib.tbk_supercell_create.restype = C.c_int
    lib.tbk_model_vectors.argtypes = [vp, vp]
    lib.tbk_model_vectors.restype = C.c_int
    lib.tbk_model_destroy.argtypes = [vp]
    lib.tbk_model_destroy.restype = C.c_int
    lib.tbk_model_info.argtypes = [vp] + [C.POINTER(C.c_int)] * 4
    lib.tbk_model_info.restype = C.c_int
    lib.tbk_hamilton.argtypes = [vp, vp, C.c_int64, C.c_int, vp, vp]
    lib.tbk_hamilton.restype = C.c_int
    lib.tbk_eigenval.argtypes = [vp, vp, C.c_int64, vp, vp]
    lib.tbk_eigenval.restype = C.c_int
    lib.tbk_eigenval_push.argtypes = [vp, vp, C.c_int64, vp, C.POINTER(vp), C.c_int, C.c_int64, vp]
    lib.tbk_eigenval_push.restype = C.c_int
    lib.tbk_eigenval_mesh.argtypes = [vp, C.POINTER(C.c_int64), dp, C.c_int64, C.c_int64, vp, vp]
    lib.tbk_eigenval_mesh.restype = C.c_int
    lib.tbk_eigenval_mesh_host.argtypes = [vp, C.POINTER(C.c_int64), dp, C.c_int64, C.c_int64, vp]
    lib.tbk_eigenval_mesh_host.restype = C.c_int
    lib.tbk_mesh_factorised.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.tbk_mesh_factorised.restype = C.c_int
    lib.tbk_eigh.argtypes = [vp, vp, C.c_int64, vp, vp, vp]
    lib.tbk_eigh.restype = C.c_int
    lib.tbk_eigh_host.argtypes = [vp, vp, C.c_int64, vp, vp]
    lib.tbk_eigh_host.restype = C.c_int
    lib.tbk_band_velocity.argtypes = [vp, vp, C.c_int64, C.c_double, vp, vp, vp]
    lib.tbk_band_velocity.restype = C.c_int
    lib.tbk_band_velocity_host.argtypes = [vp, vp, C.c_int64, C.c_double, vp, vp]
    lib.tbk_band_velocity_host.restype = C.c_int
    lib.tbk_berry_curvature.argtypes = [vp, vp, C.c_int64, C.c_int, C.c_double, vp, vp, vp]
    lib.tbk_berry_curvature.restype = C.c_int
    lib.tbk_berry_curvature_host.argtypes = [vp, vp, C.c_int64, C.c_int, C.c_double, vp, vp]
    lib.tbk_berry_curvature_host.restype = C.c_int
    lib.tbk_kdotp_coefficients.argtypes = [vp, vp, C.c_int64, vp, C.c_int, vp, vp]
    lib.tbk_kdotp_coefficients.restype = C.c_int
    lib.tbk_kdotp_coefficients_host.argtypes = [vp, vp, C.c_int64, vp, C.c_int, vp]
    lib.tbk_kdotp_coefficients_host.restype = C.c_int
    lib.tbk_hamilton_host.argtypes = [vp, vp, C.c_int64, C.c_int, vp]
    lib.tbk_hamilton_host.restype = C.c_int
    lib.tbk_eigenval_host.argtypes = [vp, vp, C.c_int64, vp]
    lib.tbk_eigenval_host.restype = C.c_int
    lib.tbk_model_check.argtypes = [vp]
    lib.tbk_model_check.restype = C.c_int
    lib.tbk_launch_count.argtypes = [vp]
    lib.tbk_launch_count.restype = C.c_int64
    lib.tbk_workspace_bytes.argtypes = [vp]
    lib.tbk_workspace_bytes.restype = C.c_int64
    lib.tbk_profile.argtypes = [vp, C.c_int]
    lib.tbk_profile.restype = C.c_int
    lib.tbk_profile_read.argtypes = [vp, dp, C.POINTER(C.c_int64)]
    lib.tbk_profile_read.restype = C.c_int
    lib.tbk_host_alloc.argtypes = [C.POINTER(vp), C.c_size_t]
    lib.tbk_host_alloc.restype = C.c_int
    lib.tbk_host_free.argtypes = [vp]
    lib.tbk_host_free.restype = C.c_int
    lib.tbk_measure_fp64_peak.argtypes = [C.c_int, C.c_int]
    lib.tbk_measure_fp64_peak.restype = C.c_double
    lib.tbk_measure_int8_peak.argtypes = [C.c_int64]
    lib.tbk_measure_int8_peak.restype = C.c_double
    lib.tbk_host_tridiag_ql.argtypes = [C.c_int, dp, dp]
    lib.tbk_host_tridiag_ql.restype = C.c_int
    lib.tbk_host_tridiag_bisect.argtypes = [C.c_int, dp, dp]
    lib.tbk_host_tridiag_bisect.restype = C.c_int
    lib.tbk_host_sincospi.argtypes = [C.c_double, dp, dp]
    lib.tbk_host_sincospi.restype = C.c_int
    lib.tbk_host_hetrd.argtypes = [C.c_int, dp, dp, dp]
    lib.tbk_host_hetrd.restype = C.c_int
    lib.tbk_host_pack_weights.argtypes = [C.c_int, C.c_int, dp, dp]
    lib.tbk_host_pack_weights.restype = C.c_int
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != TBK_OK:
        msg = load().tbk_last_error()
        raise TbkError(status, msg.decode("utf-8", "replace") if msg else "")
