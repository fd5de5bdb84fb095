"""ctypes binding of lib/libbnbp.so (the C ABI in include/bnbp.h).

Fails loudly when the library is missing or cannot be loaded: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

_lib = None


class BnbpError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libbnbp error {code}: {msg}")
        self.code = code


class FlatNetworkC(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("card", C.c_void_p), ("parent_off", C.c_void_p),
                ("parents", C.c_void_p), ("cpt_off", C.c_void_p), ("cpt", C.c_void_p)]


class OptionsC(C.Structure):
    _fields_ = [("precision", C.c_int32), ("device", C.c_int32), ("max_resident_cases", C.c_int64),
                ("specialize", C.c_int32), ("dense_min_cpt", C.c_int32), ("dense_tensor", C.c_int32),
                ("onchip", C.c_int32), ("reserved", C.c_int32 * 4)]


class EvidenceC(C.Structure):
    _fields_ = [("n_cases", C.c_int64), ("ev_off", C.c_void_p), ("ev_node", C.c_void_p),
                ("ev_state", C.c_void_p), ("ev_val_off", C.c_void_p), ("ev_values", C.c_void_p)]


class RunParamsC(C.Structure):
    _fields_ = [("epsilon", C.c_double), ("max_sweeps", C.c_int32), ("damping", C.c_double),
                ("check_interval", C.c_int32), ("out_precision", C.c_int32), ("gather", C.c_int32),
                ("n_query", C.c_int32), ("query_nodes", C.c_void_p), ("semiring", C.c_int32), ("reserved", C.c_int32 * 3)]


class SummaryC(C.Structure):
    _fields_ = [("n_cases", C.c_int64), ("case_sweeps", C.c_int64), ("not_converged", C.c_int64),
                ("max_sweeps", C.c_int64)]


COMM_ID_BYTES = 128


class StatsC(C.Structure):
    _fields_ = [("state_values_per_case", C.c_int64), ("msg_values_per_case", C.c_int64),
                ("belief_values_per_case", C.c_int64), ("cpt_values", C.c_int64),
                ("bytes_per_value", C.c_int64), ("last_case_sweeps", C.c_int64),
                ("last_sweep_launches", C.c_int64), ("last_kernel_launches", C.c_int64),
                ("last_sweep_ms", C.c_double), ("last_total_ms", C.c_double),
                ("resident_cases", C.c_int64), ("last_specialised", C.c_int64), ("cases_per_tile", C.c_int64),
                ("spec_compile_ms", C.c_double), ("dense_nodes", C.c_int64), ("dense_values_per_case", C.c_int64),
                ("dense_flops_per_case_sweep", C.c_double), ("last_dense_launches", C.c_int64),
                ("last_dense_ms", C.c_double), ("dense_tensor_jobs", C.c_int64),
                ("dense_tensor_flops_per_case_sweep", C.c_double), ("last_dense_tensor_launches", C.c_int64),
                ("last_fused", C.c_int64), ("last_compactions", C.c_int64),
                ("last_host_ms", C.c_double), ("last_host_wait_ms", C.c_double),
                ("last_onchip", C.c_int64), ("onchip_roles", C.c_int64), ("onchip_smem_bytes", C.c_int64),
                ("onchip_blocks_per_sm", C.c_int64), ("onchip_role_imbalance", C.c_double),
                ("spec_class_count", C.c_int64)]


EXPORTS = ["bnbp_device_count", "bnbp_last_error", "bnbp_create", "bnbp_destroy", "bnbp_run_batch",
           "bnbp_run_batch_device", "bnbp_check_errors", "bnbp_lw_run_batch", "bnbp_estimate_cpt", "bnbp_get_stats", "bnbp_refresh_cpt", "bnbp_precompile", "bnbp_spec_source",
           "bnbp_host_alloc", "bnbp_host_free", "bnbp_create_multi", "bnbp_get_summary", "bnbp_comm_unique_id",
           "bnbp_comm_init", "bnbp_comm_summary", "bnbp_run_batch_log_evidence", "bnbp_run_batch_device_log_evidence",
           "bnbp_run_batch_expected_counts", "bnbp_run_batch_device_expected_counts",
           "bnbp_netfile_parse", "bnbp_netfile_load", "bnbp_netfile_network", "bnbp_netfile_name",
           "bnbp_netfile_node_name", "bnbp_netfile_state_name", "bnbp_netfile_free"]


def lib_path() -> str:
    # BNBP_LIB: kernel-tuning knob (an alternative build of the same library), not a fallback
    return os.environ.get("BNBP_LIB") or _build.LIB


def load():
    """Load libbnbp.so (building it first if the sources are newer and nvcc is available)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise BnbpError(-1, f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(needs nvcc). There is no CPU fallback.")
    lib = C.CDLL(path)
    lib.bnbp_last_error.restype = C.c_char_p
    lib.bnbp_device_count.restype = C.c_int
    lib.bnbp_create.restype = C.c_int
    lib.bnbp_create.argtypes = [C.POINTER(FlatNetworkC), C.POINTER(OptionsC), C.POINTER(C.c_void_p)]
    lib.bnbp_destroy.restype = None
    lib.bnbp_destroy.argtypes = [C.c_void_p]
    lib.bnbp_run_batch.restype = C.c_int
    lib.bnbp_run_batch.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC),
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bnbp_run_batch_device.restype = C.c_int
    lib.bnbp_run_batch_device.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC),
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bnbp_run_batch_log_evidence.restype = C.c_int
    lib.bnbp_run_batch_log_evidence.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC),
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bnbp_run_batch_device_log_evidence.restype = C.c_int
    lib.bnbp_run_batch_device_log_evidence.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC),
                                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bnbp_run_batch_expected_counts.restype = C.c_int
    lib.bnbp_run_batch_expected_counts.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC), C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.bnbp_run_batch_device_expected_counts.restype = C.c_int
    lib.bnbp_run_batch_device_expected_counts.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.POINTER(RunParamsC),
                                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                          C.c_void_p, C.c_void_p]
    lib.bnbp_host_alloc.restype = C.c_void_p
    lib.bnbp_host_alloc.argtypes = [C.c_size_t]
    lib.bnbp_host_free.restype = None
    lib.bnbp_host_free.argtypes = [C.c_void_p]
    lib.bnbp_create_multi.restype = C.c_int
    lib.bnbp_create_multi.argtypes = [C.POINTER(FlatNetworkC), C.POINTER(OptionsC), C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]
    lib.bnbp_get_summary.restype = C.c_int
    lib.bnbp_get_summary.argtypes = [C.c_void_p, C.POINTER(SummaryC)]
    lib.bnbp_comm_unique_id.restype = C.c_int
    lib.bnbp_comm_unique_id.argtypes = [C.c_void_p]
    lib.bnbp_comm_init.restype = C.c_int
    lib.bnbp_comm_init.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    lib.bnbp_comm_summary.restype = C.c_int
    lib.bnbp_comm_summary.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(SummaryC), C.c_void_p]
    lib.bnbp_check_errors.restype = C.c_int
    lib.bnbp_check_errors.argtypes = [C.c_void_p, C.c_void_p]
    lib.bnbp_lw_run_batch.restype = C.c_int
    lib.bnbp_lw_run_batch.argtypes = [C.c_void_p, C.POINTER(EvidenceC), C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p]
    lib.bnbp_estimate_cpt.restype = C.c_int
    lib.bnbp_estimate_cpt.argtypes = [C.POINTER(FlatNetworkC), C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    lib.bnbp_get_stats.restype = C.c_int
    lib.bnbp_get_stats.argtypes = [C.c_void_p, C.POINTER(StatsC)]
    lib.bnbp_refresh_cpt.restype = C.c_int
    lib.bnbp_refresh_cpt.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.bnbp_precompile.restype = C.c_int
    lib.bnbp_precompile.argtypes = [C.POINTER(FlatNetworkC), C.POINTER(OptionsC), C.c_int32]
    lib.bnbp_spec_source.restype = C.c_int
    lib.bnbp_spec_source.argtypes = [C.POINTER(FlatNetworkC), C.POINTER(OptionsC), C.c_int32, C.c_char_p, C.c_int64,
                                     C.POINTER(C.c_int64)]
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise BnbpError(rc, load().bnbp_last_error().decode("utf-8", "replace"))
