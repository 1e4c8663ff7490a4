"""ctypes binding of ``lib/libtfem.so`` (C ABI declared in ``include/tfem.h``).

This is the only way the Python host code reaches the solver: there is no CPU or PyTorch fallback.  If
the library has not been built (``python -m mop_truss_marl_b200.build``) importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFEM_LIB", os.path.join(_HERE, "lib", "libtfem.so"))

MAX_NX = 16
NSEC = 5
MAX_FAMILIES = 16

STATUS_OK, STATUS_NOT_SPD, STATUS_NONFINITE, STATUS_BAD_FAMILY = 0, 1, 2, 4


class FamilyDesc(C.Structure):
    _fields_ = [
        ("num_x", C.c_int32), ("truss_type", C.c_int32), ("support_case", C.c_int32), ("symmetry", C.c_int32),
        ("span_x", C.c_double * (MAX_NX - 1)), ("span_y", C.c_double), ("tar_y", C.c_double * MAX_NX),
        ("d_min", C.c_double), ("load_y", C.c_double),
        ("section_area_cm2", C.c_double * NSEC), ("section_inertia_cm4", C.c_double * NSEC),
        ("young", C.c_double), ("allow_stress", C.c_double),
    ]


class Dims(C.Structure):
    _fields_ = [("N", C.c_int32), ("E", C.c_int32), ("ndof", C.c_int32), ("nres", C.c_int32),
                ("num_x", C.c_int32), ("n_internal", C.c_int32), ("band", C.c_int32), ("device", C.c_int32)]


class StepIn(C.Structure):
    _fields_ = [("set_node", C.c_void_p), ("set_element", C.c_void_p), ("a_geo", C.c_void_p),
                ("a_topo", C.c_void_p), ("coin", C.c_void_p), ("move_range", C.c_void_p),
                ("set_node_y", C.c_void_p), ("set_element_section", C.c_void_p)]


class StepOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "x_n", "A_s", "A_n_ts", "A_n_cs", "nN_x_n", "nN_x_e", "point", "point64", "d", "axial", "ratio", "U",
        "reactions", "status", "y", "y_weak", "node_y", "element_section")]


# table ids (enum in tfem.h) -> (dtype, shape builder)
TABLES = {
    "conn": (0, np.int32, lambda d: (d.E, 2)),
    "tnsc": (1, np.int32, lambda d: (d.N, 2)),
    "res": (2, np.int32, lambda d: (d.N, 2)),
    "top": (3, np.int32, lambda d: (d.N,)),
    "pair": (4, np.int32, lambda d: (d.N,)),
    "loaded": (5, np.int32, lambda d: (d.N,)),
    "loadvec": (6, np.float64, lambda d: (d.ndof,)),
    "x": (7, np.float64, lambda d: (d.N,)),
    "y0": (8, np.float64, lambda d: (d.N,)),
    "target": (9, np.float64, lambda d: (d.N,)),
    "A_n": (10, np.float32, lambda d: (d.N, d.N)),
    "mask": (11, np.float32, lambda d: (d.N, d.N)),
    "nC_e": (12, np.float32, lambda d: (d.E, d.N)),
    "sym_src": (13, np.int32, lambda d: (2, d.N)),
    "sym_elem": (14, np.int32, lambda d: (d.E,)),
    "int_obj": (15, np.float32, lambda d: (2,)),
    "scalars": (16, np.float64, lambda d: (8,)),
}

class GenesOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("point", "point64", "y", "section", "d", "axial", "ratio", "U", "reactions", "status")]


EXPORTS = ("tfem_version", "tfem_last_error", "tfem_create", "tfem_destroy", "tfem_get_dims", "tfem_get_table",
           "tfem_reset", "tfem_step", "tfem_solve_only", "tfem_read_genes", "tfem_solve_dense_dmma", "tfem_step_host", "tfem_launch_count", "tfem_book_launches",
           "tfem_create_mixed", "tfem_reset_mixed", "tfem_step_mixed")


class TfemError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libtfem.so is not built (%s). Run `python -m mop_truss_marl_b200.build`; there is no CPU fallback."
            % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.tfem_version.restype = C.c_char_p
    lib.tfem_last_error.restype = C.c_char_p
    lib.tfem_create.argtypes = [C.POINTER(FamilyDesc), C.c_int, C.POINTER(C.c_void_p)]
    lib.tfem_destroy.argtypes = [C.c_void_p]
    lib.tfem_get_dims.argtypes = [C.c_void_p, C.POINTER(Dims)]
    lib.tfem_get_table.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
    lib.tfem_reset.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(StepOut), C.c_void_p]
    lib.tfem_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(StepIn), C.POINTER(StepOut), C.c_void_p]
    lib.tfem_solve_only.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_void_p]
    lib.tfem_read_genes.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_float, C.c_float,
                                    C.POINTER(GenesOut), C.c_void_p]
    lib.tfem_solve_dense_dmma.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5
    lib.tfem_step_host.argtypes = [C.c_void_p, C.c_int, C.POINTER(StepIn), C.POINTER(StepOut), C.c_void_p]
    lib.tfem_create_mixed.argtypes = [C.POINTER(FamilyDesc), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.tfem_reset_mixed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(StepOut), C.c_void_p]
    lib.tfem_step_mixed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(StepIn), C.POINTER(StepOut), C.c_void_p]
    lib.tfem_launch_count.argtypes = [C.c_void_p]
    lib.tfem_launch_count.restype = C.c_int64
    for name in EXPORTS:
        getattr(lib, name)
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != 0:
        raise TfemError("libtfem error %d: %s" % (rc, lib.tfem_last_error().decode()))


class Handle:
    """One (device, family) handle: ``tfem_create`` ... ``tfem_destroy``."""

    def __init__(self, desc: FamilyDesc, device: int = 0):
        self._h = C.c_void_p()
        check(lib.tfem_create(C.byref(desc), int(device), C.byref(self._h)))
        self.device = int(device)
        self.dims = Dims()
        check(lib.tfem_get_dims(self._h, C.byref(self.dims)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib.tfem_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def ptr(self):
        return self._h

    def table(self, name: str) -> np.ndarray:
        tid, dtype, shape = TABLES[name]
        arr = np.empty(shape(self.dims), dtype=dtype)
        check(lib.tfem_get_table(self._h, tid, arr.ctypes.data_as(C.c_void_p), arr.nbytes))
        return arr

    def launch_count(self) -> int:
        return int(lib.tfem_launch_count(self._h))


class MixedHandle(Handle):
    """One handle over several families of one topology: ``tfem_create_mixed``.  With more than one family only the
    topology tables can be read (``table``)."""

    def __init__(self, descs, device: int = 0):
        self._h = C.c_void_p()
        arr = (FamilyDesc * len(descs))(*descs)
        check(lib.tfem_create_mixed(arr, len(descs), int(device), C.byref(self._h)))
        self.n_families = len(descs)
        self.device = int(device)
        self.dims = Dims()
        check(lib.tfem_get_dims(self._h, C.byref(self.dims)))
