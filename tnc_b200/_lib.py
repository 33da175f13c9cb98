"""ctypes binding of libtncb200 (include/tncb.h).  There is no fallback: if the shared
library is missing or lacks a symbol this module raises, and every compute entry point needs
a CUDA device (tncb_ctx_create fails with TNCB_ERR_CUDA otherwise)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtncb200.so")

u64p = C.POINTER(C.c_uint64)
f64p = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int)
vpp = C.POINTER(C.c_void_p)


class TncbTn(C.Structure):
    pass


TncbTn._fields_ = [
    ("n_children", C.c_size_t),
    ("children", C.POINTER(TncbTn)),
    ("rank", C.c_int),
    ("legs", u64p),
    ("dims", u64p),
    ("kind", C.c_int),
    ("host_re_im", f64p),
    ("gate_name", C.c_char_p),
    ("gate_angles", f64p),
    ("n_gate_angles", C.c_int),
    ("gate_adjoint", C.c_int),
    ("device", C.c_void_p),
    ("file_path", C.c_char_p),
    ("file_adjoint", C.c_int),
]


class TncbPath(C.Structure):
    pass


TncbPath._fields_ = [
    ("n_pairs", C.c_size_t),
    ("pairs", u64p),
    ("n_nested", C.c_size_t),
    ("nested_index", u64p),
    ("nested", C.POINTER(TncbPath)),
]

# every symbol include/tncb.h declares: (restype, argtypes)
SIGNATURES = {
    "tncb_strerror": (C.c_char_p, [C.c_int]),
    "tncb_last_error": (C.c_char_p, []),
    "tncb_version": (C.c_char_p, []),
    "tncb_ctx_create": (C.c_int, [C.c_int, C.c_size_t, vpp]),
    "tncb_ctx_destroy": (None, [C.c_void_p]),
    "tncb_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "tncb_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "tncb_ctx_stats": (C.c_int, [C.c_void_p, u64p, u64p, u64p]),
    "tncb_ctx_reset_stats": (C.c_int, [C.c_void_p]),
    "tncb_ctx_set_tcgen05_slices": (C.c_int, [C.c_void_p, C.c_int]),
    "tncb_ctx_set_tcgen05_engine": (C.c_int, [C.c_void_p, C.c_int]),
    "tncb_ctx_set_tolerance": (C.c_int, [C.c_void_p, C.c_double]),
    "tncb_ctx_set_tcgen05_moduli": (C.c_int, [C.c_void_p, C.c_int]),
    "tncb_tcgen05_bound": (C.c_int, [C.c_uint64, C.c_double, C.c_int, i32p, i32p, i32p, f64p]),
    "tncb_tcgen05_tables": (C.c_int, [C.c_int, i32p, f64p, f64p, f64p]),
    "tncb_ctx_set_tcgen05_workspace": (C.c_int, [C.c_void_p, C.c_size_t]),
    "tncb_ctx_engine_counts": (C.c_int, [C.c_void_p, u64p]),
    "tncb_ctx_last_tcgen05_info": (C.c_int, [C.c_void_p, f64p, i32p]),
    "tncb_ctx_last_tcgen05_products": (C.c_int, [C.c_void_p, i32p]),
    "tncb_ctx_trim": (C.c_int, [C.c_void_p, u64p, u64p]),
    "tncb_path_reconfigure": (C.c_int, [C.c_int, C.c_int, u64p, f64p, i32p, C.c_int, C.c_int, C.c_double, f64p, C.c_uint64, f64p, f64p, f64p]),
    "tncb_path_leg_scores": (C.c_int, [C.c_int, C.c_int, u64p, f64p, i32p, C.c_double, f64p, f64p, f64p, f64p, f64p]),
    "tncb_ctx_set_tcgen05_products": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong]),
    "tncb_ctx_set_tcgen05_threshold": (C.c_int, [C.c_void_p, C.c_longlong, C.c_longlong]),
    "tncb_ctx_time_gemm": (C.c_int, [C.c_void_p, C.c_int]),
    "tncb_ctx_gemm_totals": (C.c_int, [C.c_void_p, f64p, f64p, u64p]),
    "tncb_ctx_last_gemm_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "tncb_tensor_upload": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_void_p, vpp]),
    "tncb_tensor_alloc": (C.c_int, [C.c_void_p, C.c_int, u64p, vpp]),
    "tncb_tensor_upload_dt": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_int, C.c_void_p, vpp]),
    "tncb_tensor_alloc_dt": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_int, vpp]),
    "tncb_tensor_dtype": (C.c_int, [C.c_void_p]),
    "tncb_tensor_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tncb_tensor_write": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tncb_tensor_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tncb_tensor_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tncb_tensor_rank": (C.c_int, [C.c_void_p]),
    "tncb_tensor_dims": (C.c_int, [C.c_void_p, u64p]),
    "tncb_tensor_elements": (C.c_uint64, [C.c_void_p]),
    "tncb_tensor_device_ptr": (C.c_void_p, [C.c_void_p]),
    "tncb_contract_pair": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_int, u64p, C.c_void_p, C.c_int, u64p, C.c_void_p, vpp]),
    "tncb_contract_pair_keep": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_void_p, C.c_int, u64p, C.c_void_p, vpp]),
    "tncb_contract_pair_into": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_void_p, C.c_int, u64p, C.c_void_p, C.c_void_p]),
    "tncb_contract_pair_host": (C.c_int, [C.c_void_p, C.c_int, u64p, u64p, C.c_void_p, C.c_int, u64p, u64p, C.c_void_p, C.c_void_p]),
    "tncb_pair_out_legs": (C.c_int, [C.c_int, u64p, u64p, C.c_int, u64p, u64p, i32p, u64p, u64p, u64p, u64p, u64p]),
    "tncb_pair_kernel_class": (C.c_int, [C.c_int, u64p, u64p, C.c_int, u64p, u64p]),
    "tncb_permute": (C.c_int, [C.c_void_p, C.c_void_p, i32p, vpp]),
    "tncb_conjugate": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tncb_tensor_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tncb_gate_matrix": (C.c_int, [C.c_char_p, f64p, C.c_int, C.c_int, f64p, i32p]),
    "tncb_contract_tensor_network": (C.c_int, [C.c_void_p, C.POINTER(TncbTn), C.POINTER(TncbPath), vpp, i32p, u64p]),
    "tncb_contract_tensor_network_dt": (C.c_int, [C.c_void_p, C.POINTER(TncbTn), C.POINTER(TncbPath), C.c_int, vpp, i32p, u64p]),
    "tncb_network_out_legs": (C.c_int, [C.POINTER(TncbTn), C.POINTER(TncbPath), i32p, u64p, u64p]),
    "tncb_plan_create": (C.c_int, [C.c_void_p, C.POINTER(TncbTn), C.POINTER(TncbPath), vpp]),
    "tncb_plan_create_dt": (C.c_int, [C.c_void_p, C.POINTER(TncbTn), C.POINTER(TncbPath), C.c_int, vpp]),
    "tncb_plan_execute": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(TncbTn), vpp, i32p, u64p]),
    "tncb_plan_stage": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(TncbTn)]),
    "tncb_plan_run": (C.c_int, [C.c_void_p, C.c_void_p, vpp, i32p, u64p]),
    "tncb_plan_stage_slices": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.POINTER(TncbTn))]),
    "tncb_plan_run_slices": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, vpp, i32p, u64p]),
    "tncb_plan_info": (C.c_int, [C.c_void_p, u64p, f64p, f64p, u64p, u64p]),
    "tncb_plan_destroy": (None, [C.c_void_p]),
    "tncb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "tncb_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tncb_comm_send": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "tncb_comm_recv": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_int, vpp]),
    "tncb_comm_allreduce_sum": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tncb_comm_destroy": (C.c_int, [C.c_void_p]),
    "tncb_fanin_mapping": (C.c_int, [C.c_size_t, u64p, C.c_size_t, u64p, C.c_int, i32p]),
    "tncb_hdf5_open": (C.c_int, [C.c_char_p, C.c_char_p, vpp]),
    "tncb_hdf5_close": (None, [C.c_void_p]),
    "tncb_hdf5_count": (C.c_size_t, [C.c_void_p]),
    "tncb_hdf5_name": (C.c_char_p, [C.c_void_p, C.c_size_t]),
    "tncb_hdf5_shape": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), u64p, u64p]),
    "tncb_hdf5_attr": (C.c_int, [C.c_void_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_int64), C.POINTER(C.c_size_t)]),
    "tncb_hdf5_read": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "tncb_hdf5_load_leaf": (C.c_int, [C.c_char_p, C.c_int, C.c_int, u64p, C.c_void_p]),
    "tncb_hdf5_store_data": (C.c_int, [C.c_char_p, C.c_int, u64p, C.c_void_p]),
    "tncb_hdf5_store": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(u64p),
                                  C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(u64p)]),
}

# tncb_dtype values
TNCB_C128 = 0
TNCB_C64 = 1

_lib = None


class TncbError(RuntimeError):
    """Raised for any non-zero tncb_status (the reference panics in the same places)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[tncb status {status}] {message}")
        self.status = status


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                "(tnc_b200 has no CPU or PyTorch fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int) -> None:
    if status != 0:
        l = lib()
        msg = l.tncb_last_error().decode("utf-8", "replace") or l.tncb_strerror(status).decode()
        raise TncbError(status, msg)


def u64_array(values):
    values = list(values)
    return (C.c_uint64 * max(len(values), 1))(*values)
