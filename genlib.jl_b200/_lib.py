"""ctypes binding of libgenlib_cuda.so (include/genlib_cuda.h).

The library is the product: if it is missing, or no CUDA device is usable,
the calls below raise -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GENLIB_CUDA_LIB") or os.path.join(_HERE, "libgenlib_cuda.so")

OK, EINVAL, EKEY, EORDER, ECUDA, ENOMEM, ECOMM, ERESTART, EOVERFLOW = range(9)
SCHEDULES = {"phi": 0, "sparse_phi": 1, "sparse_phi_symmetric": 2}
NUMERICS = {"reference": 0, "fp64": 1, 0: 0, 1: 1}
DTYPES = {np.dtype(np.float32): 0, np.dtype(np.float64): 1}


class GenlibError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libgenlib_cuda status {status}: {message}")
        self.status = status


class PlanBoundsExceeded(GenlibError):
    """genlib_engine_run on an engine of a plan that was still being made (Plan(..., stream=True)): a size
    bound did not hold (GENLIB_ERESTART).  Close the engine, create it again -- the plan is finished by
    then -- and run."""


class GenlibOverflowError(GenlibError, OverflowError):
    """gen.occ: a descent-path count or a row sum does not fit an Int64 (GENLIB_EOVERFLOW).
    `ancestor_index` / `proband_index`: the 0-based list positions of the pair the library names."""

    def __init__(self, status: int, message: str):
        super().__init__(status, message)
        m = re.search(r"ancestor position (-?\d+).*proband position (-?\d+)", message)
        self.ancestor_index, self.proband_index = (int(m.group(1)), int(m.group(2))) if m else (None, None)


class LayerInfo(C.Structure):
    _fields_ = [("n_new", C.c_int32), ("n_fam", C.c_int32), ("live_before", C.c_int32),
                ("carried", C.c_int32), ("ref_founders", C.c_int32), ("ref_probands", C.c_int32),
                ("ref_both", C.c_int32), ("strip_width", C.c_int32), ("alg_elems", C.c_double),
                ("ms_layer", C.c_double), ("ms_wait", C.c_double), ("dram_read_bytes", C.c_double),
                ("dram_write_bytes", C.c_double), ("l2_bytes", C.c_double), ("nvlink_bytes", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class Stats(C.Structure):
    _fields_ = [("n_unique", C.c_int32), ("n_layers", C.c_int32), ("row_updates", C.c_int64),
                ("capacity", C.c_int64), ("device_bytes", C.c_int64), ("alg_bytes", C.c_double),
                ("ms_plan", C.c_double), ("ms_upload", C.c_double), ("ms_kernels", C.c_double),
                ("ms_fetch", C.c_double), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("kernel_launches", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class GcStats(C.Structure):
    _fields_ = [("n_pro", C.c_int32), ("n_anc", C.c_int32), ("n_layers", C.c_int32), ("direction", C.c_int32),
                ("rows", C.c_int64), ("inputs", C.c_int64), ("width", C.c_int64), ("capacity", C.c_int64),
                ("device_bytes", C.c_int64), ("alg_bytes", C.c_double), ("ms_plan", C.c_double),
                ("ms_kernels", C.c_double), ("ms_fetch", C.c_double), ("d2h_bytes", C.c_int64),
                ("kernel_launches", C.c_int32), ("n_dev", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


GC_DIRECTIONS = {0: "descend", 1: "ascend"}

# every symbol include/genlib_cuda.h declares: (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "genlib_version": (C.c_int, []),
    "genlib_last_error": (C.c_char_p, []),
    "genlib_device_count": (C.c_int, []),
    "genlib_release_cache": (C.c_int, []),
    "genlib_pinned_alloc": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "genlib_pinned_free": (C.c_int, [_P]),
    "genlib_genealogy_csv": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_P)]),
    "genlib_genealogy_arrays": (C.c_int, [C.c_int64, _P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    "genlib_pedigree_destroy": (None, [_P]),
    "genlib_pedigree_n": (C.c_int64, [_P]),
    "genlib_pedigree_depth": (C.c_int32, [_P]),
    "genlib_pedigree_arrays": (C.c_int, [_P, _P, _P, _P, _P]),
    "genlib_pedigree_pro": (C.c_int64, [_P, _P]),
    "genlib_pedigree_ranks": (C.c_int, [_P, C.c_int64, _P, _P]),
    "genlib_plan_create": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, C.POINTER(_P)]),
    "genlib_plan_create_scheduled": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, C.c_int, C.POINTER(_P)]),
    "genlib_plan_create_ex": (C.c_int, [C.c_int32, _P, _P, _P, C.c_int32, _P, C.c_int32, C.c_int, C.POINTER(_P)]),
    "genlib_plan_layer_ranks": (C.c_int, [_P, C.c_int32, _P]),
    "genlib_plan_schedule": (C.c_int32, [_P]),
    "genlib_plan_destroy": (None, [_P]),
    "genlib_plan_n_unique": (C.c_int32, [_P]),
    "genlib_plan_n_layers": (C.c_int32, [_P]),
    "genlib_plan_capacity": (C.c_int64, [_P]),
    "genlib_plan_row_updates": (C.c_int64, [_P]),
    "genlib_plan_layer_info": (C.c_int, [_P, C.c_int32, C.POINTER(LayerInfo)]),
    "genlib_plan_device_bytes": (C.c_int64, [_P, C.c_int, C.c_int32]),
    "genlib_plan_layer_arrays": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "genlib_plan_layer_shard": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "genlib_plan_layer_live_rows": (C.c_int, [_P, C.c_int32, _P, _P]),
    "genlib_plan_rank_rows": (C.c_int64, [_P, C.c_int32]),
    "genlib_plan_world": (C.c_int32, [_P]),
    "genlib_plan_proband_rows": (C.c_int, [_P, _P, _P]),
    "genlib_plan_layer_flags": (C.c_int, [_P, C.c_int32, _P]),
    "genlib_plan_proband_slots": (C.c_int, [_P, _P]),
    "genlib_plan_digest": (C.c_uint64, [_P, C.c_int]),
    "genlib_phi": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, _P, C.c_int, C.c_int, C.c_int,
                             C.POINTER(Stats)]),
    "genlib_phi_multi": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, _P, C.c_int, C.c_int, C.c_int32, _P,
                                   C.POINTER(Stats)]),
    "genlib_plan_create_async": (C.c_int, [C.c_int32, _P, _P, _P, C.c_int32, _P, C.c_int32, C.c_int, C.POINTER(_P)]),
    "genlib_plan_stream_selftest": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, C.c_double, _P, _P]),
    "genlib_engine_create": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P)]),
    "genlib_engine_destroy": (None, [_P]),
    "genlib_engine_run": (C.c_int, [_P, C.c_int]),
    "genlib_engine_layer_info": (C.c_int, [_P, C.c_int32, C.POINTER(LayerInfo)]),
    "genlib_engine_stats": (C.c_int, [_P, C.POINTER(Stats)]),
    "genlib_engine_fetch": (C.c_int, [_P, _P, C.c_int]),
    "genlib_engine_own_probands": (C.c_int32, [_P, _P]),
    "genlib_engine_create_dist": (C.c_int, [_P, C.c_int, C.c_int, C.c_int32, C.POINTER(_P)]),
    "genlib_engine_ipc_export": (C.c_int, [_P, _P]),
    "genlib_engine_ipc_attach": (C.c_int, [_P, _P, C.c_size_t]),
    "genlib_engine_phi_mean": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "genlib_engine_row_sums": (C.c_int, [_P, _P]),
    "genlib_engine_set_layer_limit": (C.c_int, [_P, C.c_int32]),
    "genlib_engine_read_block": (C.c_int, [_P, C.c_int32, _P, _P]),
    "genlib_gc": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.c_int, C.c_int, C.c_int32, _P,
                            C.POINTER(GcStats)]),
    "genlib_gc_plan_create": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, _P, C.POINTER(_P)]),
    "genlib_gc_plan_destroy": (None, [_P]),
    "genlib_gc_plan_info": (C.c_int, [_P, C.POINTER(GcStats)]),
    "genlib_gc_plan_layer": (C.c_int, [_P, C.c_int32, _P, _P]),
    "genlib_gc_plan_layer_arrays": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "genlib_occ": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.c_int, C.c_int, C.c_int32, _P,
                             C.POINTER(GcStats)]),
    "genlib_rec": (C.c_int, [C.c_int32, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.c_int32, _P,
                             C.POINTER(GcStats)]),
}

_lib = None


def lib():
    """Load libgenlib_cuda.so; raise if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C genlib.jl_b200/csrc`. There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status: int):
    if status != OK:
        msg = lib().genlib_last_error().decode(errors="replace")
        if status == EKEY:
            raise KeyError(msg)          # the reference raises KeyError (src/create.jl:70)
        if status == EINVAL and ("duplicate" in msg or "malformed" in msg or "same length" in msg):
            raise ValueError(msg)
        if status == EINVAL and msg.startswith("cannot open"):
            raise FileNotFoundError(msg)
        if status == ENOMEM:
            raise MemoryError(msg)
        if status == ERESTART:
            raise PlanBoundsExceeded(status, msg)
        if status == EOVERFLOW:
            raise GenlibOverflowError(status, msg)
        raise GenlibError(status, msg)


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
