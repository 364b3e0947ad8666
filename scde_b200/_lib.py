"""ctypes binding of libscde_b200.so (the C ABI in include/scde_b200.h).

This is the only way the Python host layer reaches the device code -- the same entry points an R/Rcpp shim would
bind (INTEGRATION.md).  There is no CPU fallback: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCDE_B200_LIB") or os.path.join(_HERE, "libscde_b200.so")

T_DEDUP, T_LPTABLE, T_CONTRACT, T_RATIO, T_OTHER, T_SOFTMAX, T_BOUND, T_TOTAL, T_COUNT = range(9)
STAGE_NAMES = ["dedup", "lp_table", "contract", "ratio", "other", "softmax", "bound", "total"]

i32p = C.POINTER(C.c_int32)
f64p = C.POINTER(C.c_double)


class ScdeB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libscde_b200 error {code}: {msg}")
        self.code = code


class DiffArgs(C.Structure):
    _fields_ = [
        ("n_genes", C.c_int32), ("n_cells", C.c_int32), ("n_grid", C.c_int32),
        ("counts", i32p), ("models", f64p), ("prior_x", f64p), ("prior_y", f64p),
        ("group", i32p), ("batch", i32p), ("n_batch_levels", C.c_int32),
        ("n_boot", C.c_int32), ("seed", C.c_int32),
        ("boot_idx", i32p * 4),
        ("zero_index", i32p), ("n_zero", C.c_int32), ("zero_index_adjusted", i32p),
        ("local_theta", C.c_int32), ("square_logit_conc", C.c_int32),
        ("gene_begin", C.c_int32), ("gene_end", C.c_int32),
        ("batch_models", f64p), ("batch_local_theta", C.c_int32), ("batch_square_logit_conc", C.c_int32),
        ("draw_chunks", C.c_int32),
    ]


class DiffOut(C.Structure):
    _fields_ = [
        ("idx", i32p), ("z", f64p), ("batch_idx", i32p), ("batch_z", f64p),
        ("adjusted_idx", i32p), ("adjusted_z", f64p),
        ("difference_posterior", f64p), ("batch_difference_posterior", f64p),
        ("adjusted_difference_posterior", f64p),
        ("joint_posteriors", f64p * 2), ("batch_joint_posteriors", f64p * 2),
        ("cz", f64p), ("batch_cz", f64p), ("adjusted_cz", f64p),
    ]


class DatasetArgs(C.Structure):
    """scde_b200_dataset_args (include/scde_b200.h)."""
    _fields_ = [
        ("n_genes", C.c_int32), ("n_cells", C.c_int32), ("n_grid", C.c_int32),
        ("counts", i32p), ("models", f64p), ("prior_x", f64p), ("prior_y", f64p),
        ("local_theta", C.c_int32), ("square_logit_conc", C.c_int32),
    ]


class ContrastArgs(C.Structure):
    """scde_b200_contrast_args (include/scde_b200.h)."""
    _fields_ = [
        ("n_groups", C.c_int32), ("group_offsets", i32p), ("group_cells", i32p),
        ("n_contrasts", C.c_int32), ("pairs", i32p),
        ("n_boot", C.c_int32), ("seed", C.c_int32),
        ("zero_index", i32p), ("n_zero", C.c_int32), ("zero_index_adjusted", i32p),
        ("batch", i32p), ("n_batch_levels", C.c_int32),
        ("batch_models", f64p), ("batch_local_theta", C.c_int32), ("batch_square_logit_conc", C.c_int32),
        ("draw_chunks", C.c_int32),
    ]


class ContrastOut(C.Structure):
    """scde_b200_contrast_out (include/scde_b200.h)."""
    _fields_ = [
        ("idx", i32p), ("z", f64p), ("cz", f64p),
        ("batch_idx", i32p), ("batch_z", f64p), ("batch_cz", f64p),
        ("adjusted_idx", i32p), ("adjusted_z", f64p), ("adjusted_cz", f64p),
        ("difference_posterior", f64p), ("adjusted_difference_posterior", f64p), ("joint_posteriors", f64p),
    ]


class Stats(C.Structure):
    _fields_ = [("ms", C.c_float * T_COUNT), ("launches", C.c_int32 * T_COUNT),
                ("table_rows", C.c_int64), ("contract_cells", C.c_int64),
                ("prune_items", C.c_int64), ("prune_live", C.c_int64),
                ("prune_work", C.c_int64), ("prune_live_work", C.c_int64)]

    def as_dict(self):
        return {"ms": {STAGE_NAMES[i]: float(self.ms[i]) for i in range(T_COUNT - 1)},
                "launches": {STAGE_NAMES[i]: int(self.launches[i]) for i in range(T_COUNT - 1)},
                "table_rows": int(self.table_rows), "contract_cells": int(self.contract_cells),
                "prune_items": int(self.prune_items), "prune_live": int(self.prune_live),
                "prune_work": int(self.prune_work), "prune_live_work": int(self.prune_live_work)}


class Options(C.Structure):
    """scde_b200_options (include/scde_b200.h)."""
    _fields_ = [(n, C.c_int32) for n in (
        "contract_kernel", "zero_base", "fused_fixed_point", "lp_rows_kernel", "count_chunks", "split_front",
        "uniform_chunks", "pipeline_front", "item_order", "hot_rank", "cold_evict_first", "trace", "epilogue_timing",
        "debug_contract", "ring_stages", "twin_batch_joints", "prune_pieces")] + [("reserved", C.c_int32 * 4)]


# every symbol include/scde_b200.h declares
EXPORTED = [
    "scde_b200_create_multi", "scde_b200_n_devices", "scde_b200_get_options", "scde_b200_set_options",
    "scde_b200_version", "scde_b200_last_error", "scde_b200_device_count", "scde_b200_create", "scde_b200_destroy",
    "scde_b200_stream", "scde_b200_synchronize", "scde_b200_boot_indices", "scde_b200_batch_boot_indices",
    "scde_b200_log_boot_posterior", "scde_b200_log_boot_batch_posterior", "scde_b200_jpmat_log_boot",
    "scde_b200_jpmat_log_batch_boot", "scde_b200_mat_slide_mult", "scde_b200_ratio_posterior_summary",
    "scde_b200_bh_cz", "scde_b200_expression_difference", "scde_b200_diff_upload", "scde_b200_diff_run",
    "scde_b200_diff_download", "scde_b200_diff_free", "scde_b200_expression_magnitude", "scde_b200_cell_table",
    "scde_b200_measure_fp64_peak", "scde_b200_set_contract_kernel", "scde_b200_probe_contract_i8", "scde_b200_probe_table",
    "scde_b200_probe_table_bounds", "scde_b200_probe_prune_i8",
    "scde_b200_failure_probability", "scde_b200_expression_prior", "scde_b200_dataset_create",
    "scde_b200_dataset_contrasts", "scde_b200_dataset_free",
]

_lib = None


def lib():
    """Load libscde_b200.so; fails loudly when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m scde_b200.build` (nvcc, sm_100a). "
                              "scde_b200 has no CPU or PyTorch fallback.")
        L = C.CDLL(LIB_PATH)
        L.scde_b200_last_error.restype = C.c_char_p
        L.scde_b200_stream.restype = C.c_void_p
        L.scde_b200_stream.argtypes = [C.c_void_p]
        L.scde_b200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.scde_b200_destroy.argtypes = [C.c_void_p]
        L.scde_b200_destroy.restype = None
        L.scde_b200_synchronize.argtypes = [C.c_void_p]
        L.scde_b200_diff_upload.argtypes = [C.c_void_p, C.POINTER(DiffArgs), C.c_int32, C.POINTER(C.c_void_p)]
        L.scde_b200_diff_run.argtypes = [C.c_void_p, C.c_void_p]
        L.scde_b200_diff_download.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(DiffOut), C.POINTER(Stats)]
        L.scde_b200_diff_free.argtypes = [C.c_void_p, C.c_void_p]
        L.scde_b200_diff_free.restype = None
        L.scde_b200_expression_difference.argtypes = [C.c_void_p, C.POINTER(DiffArgs), C.POINTER(DiffOut),
                                                      C.POINTER(Stats)]
        L.scde_b200_measure_fp64_peak.argtypes = [C.c_void_p, f64p]
        L.scde_b200_set_contract_kernel.argtypes = [C.c_void_p, C.c_int32]
        L.scde_b200_failure_probability.argtypes = [C.c_void_p, f64p, C.c_int32, i32p, f64p, C.c_int32, C.c_int32, f64p]
        L.scde_b200_expression_prior.argtypes = [C.c_void_p, f64p, C.c_int32, i32p, C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_double, C.c_double, C.c_double, C.c_double, f64p, f64p, f64p, f64p]
        L.scde_b200_dataset_create.argtypes = [C.c_void_p, C.POINTER(DatasetArgs), C.POINTER(C.c_void_p), C.POINTER(Stats)]
        L.scde_b200_dataset_contrasts.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(ContrastArgs), C.POINTER(ContrastOut),
                                                  C.POINTER(Stats)]
        L.scde_b200_dataset_free.argtypes = [C.c_void_p, C.c_void_p]
        L.scde_b200_dataset_free.restype = None
        L.scde_b200_create_multi.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
        L.scde_b200_n_devices.argtypes = [C.c_void_p]
        L.scde_b200_probe_table.argtypes = [C.c_void_p, f64p, C.c_int32, i32p, i32p, f64p, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_int32, C.c_void_p, C.c_void_p, i32p, i32p, f64p]
        L.scde_b200_probe_table_bounds.argtypes = L.scde_b200_probe_table.argtypes + [C.c_void_p]
        L.scde_b200_probe_prune_i8.argtypes = [C.c_void_p] + [C.c_void_p] + [C.c_int32] * 2 + [C.c_void_p] * 4 + [C.c_int32] + \
            [C.c_void_p] * 3 + [C.c_int32] * 2 + [C.c_void_p] * 6
        L.scde_b200_get_options.argtypes = [C.c_void_p, C.POINTER(Options)]
        L.scde_b200_set_options.argtypes = [C.c_void_p, C.POINTER(Options)]
        _lib = L
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise ScdeB200Error(code, lib().scde_b200_last_error().decode("utf-8", "replace"))


def p_i32(a):
    return a.ctypes.data_as(i32p) if a is not None else None


def p_f64(a):
    return a.ctypes.data_as(f64p) if a is not None else None


def f64(a, order="F"):
    return np.require(np.asarray(a, dtype=np.float64), requirements=["F" if order == "F" else "C", "A"])


def i32(a, order="F"):
    return np.require(np.asarray(a, dtype=np.int32), requirements=["F" if order == "F" else "C", "A"])


class Context:
    """One CUDA device + stream (scde_b200_ctx), or -- `devices` a list -- a multi-device context
    (scde_b200_create_multi): scde_b200_expression_difference then shards the genes over the devices."""

    def __init__(self, device: int = 0, devices=None):
        self._h = C.c_void_p()
        if devices is not None:
            devs = (C.c_int * len(devices))(*[int(d) for d in devices])
            check(lib().scde_b200_create_multi(len(devices), devs, C.byref(self._h)))
            self.device = int(devices[0])
            self.devices = [int(d) for d in devices]
        else:
            check(lib().scde_b200_create(int(device), C.byref(self._h)))
            self.device = int(device)
            self.devices = [self.device]

    def options(self) -> "Options":
        o = Options()
        check(lib().scde_b200_get_options(self._h, C.byref(o)))
        return o

    def set_options(self, **kw) -> "Options":
        """Change the named scde_b200_options fields; returns the previous options (for restoring)."""
        old = self.options()
        new = self.options()
        for k, v in kw.items():
            if not hasattr(new, k):
                raise AttributeError(f"scde_b200_options has no field {k}")
            setattr(new, k, int(v))
        check(lib().scde_b200_set_options(self._h, C.byref(new)))
        return old

    def restore_options(self, old: "Options"):
        check(lib().scde_b200_set_options(self._h, C.byref(old)))

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return int(lib().scde_b200_stream(self._h) or 0)

    def synchronize(self):
        check(lib().scde_b200_synchronize(self._h))

    def set_contract_kernel(self, which: int):
        check(lib().scde_b200_set_contract_kernel(self._h, int(which)))

    def measure_fp64_peak(self) -> float:
        v = C.c_double()
        check(lib().scde_b200_measure_fp64_peak(self._h, C.byref(v)))
        return float(v.value)

    def close(self):
        if self._h:
            lib().scde_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
