"""ctypes binding of libcsb200.so (C ABI: include/cs_b200.h).

There is NO CPU fallback: importing works anywhere (so host logic can be tested),
but the first call that needs the device raises `B200Unavailable` if the shared
library is missing or no CUDA device is visible.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcsb200.so")

OK, ERR_ARG, ERR_CUDA, ERR_RESIDUAL, ERR_MAXITER, ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
F32, F64 = 0, 1
PRECOND_JACOBI, PRECOND_AMG = 0, 1


class B200Unavailable(RuntimeError):
    pass


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


class Opts(C.Structure):
    _fields_ = [("precond", C.c_int32), ("panel_width", C.c_int32), ("check_every", C.c_int32),
                ("use_graph", C.c_int32), ("atol", C.c_double), ("resid_gate", C.c_double),
                ("log_transform", C.c_int32), ("window", C.c_int32), ("mixed", C.c_int32), ("setup", C.c_int32),
                ("stencil", C.c_int32), ("reserved", C.c_int32 * 3)]


class Stats(C.Structure):
    _fields_ = [("setup_ms", C.c_double), ("solve_ms", C.c_double), ("kernel_ms", C.c_double),
                ("iterations", C.c_int64), ("spmm_launches", C.c_int64),
                ("kernel_launches", C.c_int64), ("h2d_bytes", C.c_double), ("d2h_bytes", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every exported symbol of include/cs_b200.h: name -> (restype, argtypes)
_H = C.c_void_p
_PROTOS = {
    "cs_b200_version": (C.c_int, []),
    "cs_b200_last_error": (C.c_char_p, [_H]),
    "cs_b200_create": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.POINTER(Opts), C.POINTER(_H)]),
    "cs_b200_create_from_device": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_int, C.POINTER(Opts), C.POINTER(_H)]),
    "cs_b200_create_from_raster": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(Opts), C.POINTER(_H), C.POINTER(C.c_int64),
                                             C.POINTER(C.c_int64)]),
    "cs_b200_get_csr": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cs_b200_set_grounds": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "cs_b200_level_info": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "cs_b200_level_csr": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cs_b200_create_from_raster_poly": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                  C.c_int, C.POINTER(Opts), C.POINTER(_H), C.POINTER(C.c_int64),
                                                  C.POINTER(C.c_int64), C.c_void_p]),
    "cs_b200_components": (C.c_int, [_H, C.c_void_p, C.POINTER(C.c_int64)]),
    "cs_b200_get_dims": (C.c_int, [_H, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cs_b200_destroy": (None, [_H]),
    "cs_b200_spmv": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_double)]),
    "cs_b200_spmm": (C.c_int, [_H, C.c_int, C.c_void_p, C.c_void_p]),
    "cs_b200_bench_spmm": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "cs_b200_bench_cg_iter": (C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "cs_b200_solve_rhs": (C.c_int, [_H, C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_int64,
                                    C.c_void_p, C.c_void_p]),
    "cs_b200_solve_pairs": (C.c_int, [_H, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                      C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_void_p, C.c_void_p]),
    "cs_b200_solve_pairs_superposed": (C.c_int, [_H, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_double, C.c_int64, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cs_b200_solve_sources": (C.c_int, [_H, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_void_p]),
    "cs_b200_read_currents": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "cs_b200_reset_currents": (C.c_int, [_H]),
    "cs_b200_currents_device_ptrs": (C.c_int, [_H, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "cs_b200_get_stats": (C.c_int, [_H, C.POINTER(Stats)]),
    "cs_b200_stream": (C.c_int, [_H, C.POINTER(C.c_void_p)]),
    "cs_b200_profile_spmm": (C.c_int, [_H, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "cs_b200_profile_classes": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cs_b200_profile_bytes": (C.c_int, [_H, C.POINTER(C.c_double)]),
    "cs_b200_comm_unique_id": (C.c_int, [C.c_void_p]),
    "cs_b200_comm_init": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(_H)]),
    "cs_b200_comm_destroy": (None, [_H]),
    "cs_b200_comm_last_error": (C.c_char_p, [_H]),
    "cs_b200_create_bcast": (C.c_int, [_H, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_int, C.c_int, C.POINTER(Opts), C.POINTER(_H)]),
    "cs_b200_comm_reduce_currents": (C.c_int, [_H, _H]),
    "cs_b200_comm_gather_pairs": (C.c_int, [_H, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cs_b200_comm_max_double": (C.c_int, [_H, C.c_void_p, C.c_int]),
    "cs_b200_comm_barrier": (C.c_int, [_H]),
}
EXPORTED_SYMBOLS = tuple(_PROTOS)

_lib = None


def load():
    """dlopen libcsb200.so and bind every prototype (no device call)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise B200Unavailable(
            f"{LIB_PATH} not built -- run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(the CUDA path has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def np_dtype(dtype_code):
    return np.float64 if dtype_code == F64 else np.float32


def dtype_code(dt):
    dt = np.dtype(dt)
    if dt == np.float64:
        return F64
    if dt == np.float32:
        return F32
    raise TypeError(f"unsupported dtype {dt}")


def check(lib, h, rc, allow=()):
    if rc == OK or rc in allow:
        return rc
    msg = lib.cs_b200_last_error(h)
    msg = msg.decode() if msg else f"libcsb200 error {rc}"
    if rc == ERR_CUDA and "no CUDA device" in msg:
        raise B200Unavailable(msg)
    raise B200Error(rc, msg)
