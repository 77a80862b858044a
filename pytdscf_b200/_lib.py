"""ctypes binding of libtdvp_b200.so (the C ABI declared in include/tdvp_b200.h).

PyTorch is used only as the device-buffer holder: tensors are complex128 CUDA tensors whose
``data_ptr()`` is handed to the library.  There is NO CPU fallback: if the shared library or a CUDA
device is missing every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtdvp_b200.so")

KIND_IDENTITY, KIND_DIAG, KIND_FULL = 0, 3, 4
KRYLOV_LANCZOS_REF, KRYLOV_ARNOLDI = 0, 1
GAUGE_A, GAUGE_B = 0, 1


class TdvpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libtdvp_b200 error {code}: {msg}")
        self.code = code


class NotConverged(TdvpError, ValueError):
    """Mirrors the ValueError of the reference's Krylov solvers (pytdscf/_integrator.py:430, :653)."""


class c128(C.Structure):
    _fields_ = [("re", C.c_double), ("im", C.c_double)]


class HeffTerm(C.Structure):
    _fields_ = [
        ("L", C.c_void_p), ("W", C.c_void_p), ("Wp", C.c_void_p), ("R", C.c_void_p),
        ("wl", C.c_int32), ("wr", C.c_int32), ("w_kind", C.c_int32), ("id_channels", C.c_int32),
        ("coef_re", C.c_double), ("coef_im", C.c_double),
    ]


class KeffTerm(C.Structure):
    _fields_ = [
        ("L", C.c_void_p), ("R", C.c_void_p), ("w", C.c_int32), ("id_channels", C.c_int32),
        ("coef_re", C.c_double), ("coef_im", C.c_double),
    ]


class Heff2Term(C.Structure):
    _fields_ = [
        ("L", C.c_void_p), ("W1", C.c_void_p), ("W1p", C.c_void_p), ("W2", C.c_void_p), ("W2p", C.c_void_p),
        ("R", C.c_void_p), ("wl", C.c_int32), ("wm", C.c_int32), ("wr", C.c_int32), ("w1_kind", C.c_int32),
        ("w2_kind", C.c_int32), ("id_channels", C.c_int32), ("coef_re", C.c_double), ("coef_im", C.c_double),
    ]


ERR_NO_MEMORY = -6

# name -> (restype, argtypes); must list every symbol include/tdvp_b200.h declares
SIGNATURES = {
    "tdvp_abi_version": (C.c_int, []),
    "tdvp_launch_count": (C.c_ulonglong, []),
    "tdvp_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "tdvp_destroy": (C.c_int, [C.c_void_p]),
    "tdvp_last_error": (C.c_char_p, [C.c_void_p]),
    "tdvp_get_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), C.POINTER(C.c_double)]),
    "tdvp_reset_stats": (C.c_int, [C.c_void_p]),
    "tdvp_gemm_profile": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "tdvp_profile_json": (C.c_size_t, [C.c_char_p, C.c_size_t]),
    "tdvp_set_gemm_config": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "tdvp_heff_apply": (C.c_int, [C.c_void_p, C.POINTER(HeffTerm), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tdvp_keff_apply": (C.c_int, [C.c_void_p, C.POINTER(KeffTerm), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tdvp_env_update": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "tdvp_set_krylov_size": (C.c_int, [C.c_void_p, C.c_longlong]),
    "tdvp_krylov_expm": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                   C.POINTER(HeffTerm), C.POINTER(KeffTerm), C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.POINTER(C.c_int)]),
    "tdvp_lanczos_eigvec": (C.c_int, [C.c_void_p, C.POINTER(HeffTerm), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                      C.c_int, C.c_double, C.POINTER(C.c_int)]),
    "tdvp_qr_shift": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tdvp_absorb": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tdvp_svd_truncate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "tdvp_svd": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "tdvp_pinv": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p]),
    "tdvp_inner": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(c128)]),
    "tdvp_overlap_site": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_int, C.c_void_p]),
    "tdvp_zgemm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                             C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_int]),
}

# the two-site entry points of include/tdvp_b200_two_site.h
SIGNATURES_TWO_SITE = {
    "tdvp_heff2_apply": (C.c_int, [C.c_void_p, C.POINTER(Heff2Term), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p]),
    "tdvp_krylov_expm2": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                    C.POINTER(Heff2Term), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.POINTER(C.c_int)]),
    "tdvp_split2": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_int,
                              C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
}

_lib = None


def load_library():
    """Load the shared library and attach the prototypes.  Raises if the .so was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(
            f"{LIB_PATH} is missing: build it with `python pytdscf_b200/csrc/build.py` "
            "(or __graft_entry__.build()).  There is no CPU fallback for backend='cuda'."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in {**SIGNATURES, **SIGNATURES_TWO_SITE}.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(handle, rc: int):
    if rc == 0:
        return
    msg = load_library().tdvp_last_error(handle)
    text = msg.decode() if msg else ""
    if rc == -3:
        raise NotConverged(rc, text)
    raise TdvpError(rc, text)
