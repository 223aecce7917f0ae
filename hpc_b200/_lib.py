"""ctypes binding of libspmm_b200.so (the C ABI declared in include/spmm_b200.h).

There is no fallback: if the CUDA library has not been built the import fails loudly
(build it with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C hpc_b200/csrc`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SPMM_B200_LIB points at another build of the same library (tuning experiments); there is still no fallback.
LIB_PATH = os.environ.get("SPMM_B200_LIB") or os.path.join(_HERE, "libspmm_b200.so")


class PlanInfo(C.Structure):
    """spmm_b200_plan_info_t"""

    _fields_ = [
        ("num_v", C.c_int), ("num_e", C.c_int), ("feat_in", C.c_int),
        ("seg_len", C.c_int), ("kslice", C.c_int), ("n_slices", C.c_int), ("block", C.c_int),
        ("n_light", C.c_int), ("n_heavy", C.c_int), ("n_seg", C.c_int),
        ("panel_len", C.c_longlong), ("lanes", C.c_int), ("vec", C.c_int),
        ("n_ltask", C.c_int), ("n_utask", C.c_int), ("lpanel_len", C.c_longlong), ("light_steps", C.c_int), ("reorder", C.c_int), ("resident_warps", C.c_int),
        ("n_col_blocks", C.c_int), ("col_begin", C.c_int), ("col_end", C.c_int),
        ("persistent", C.c_int), ("n_row_groups", C.c_int), ("n_tickets", C.c_int),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/spmm_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I = C.c_int
_LL = C.c_longlong
_U64 = C.c_uint64
SIGNATURES = {
    "spmm_b200_create": (_I, [_P, _P, _P, _I, _I, _I, C.POINTER(_P)]),
    "spmm_b200_set_feat": (_I, [_P, _I]),
    "spmm_b200_set_option": (_I, [_P, C.c_char_p, _LL]),
    "spmm_b200_set_gather": (_I, [_P, _I, C.POINTER(_P), _P, _LL]),
    "spmm_b200_preprocess": (_I, [_P, _P, _P, _P]),
    "spmm_b200_refresh_values": (_I, [_P, _P]),
    "spmm_b200_run": (_I, [_P, _P, _P, _P]),
    "spmm_b200_run_values": (_I, [_P, _P, _P, _P, _P]),
    "spmm_b200_run_profiled": (_I, [_P, _P, _P, _P, C.POINTER(C.c_float)]),
    "spmm_b200_create_transposed": (_I, [_P, _I, _P, C.POINTER(_P)]),
    "spmm_b200_sddmm": (_I, [_P, _P, _P, _P, _P]),
    "spmm_b200_edge_softmax": (_I, [_P, _P, _P, _P]),
    "spmm_b200_edge_softmax_backward": (_I, [_P, _P, _P, _P, _P]),
    "spmm_b200_reduce": (_I, [_P, _I, _P, _P, _P, _P]),
    "spmm_b200_reduce_backward": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "spmm_b200_create_column_sorted": (_I, [_P, _I, _P, C.POINTER(_P)]),
    "spmm_b200_destroy": (_I, [_P]),
    "spmm_b200_trim_memory": (_I, []),
    "spmm_b200_run_host": (_I, [_P, _P, _P, _P]),
    "spmm_b200_last_error": (C.c_char_p, []),
    "spmm_b200_launches_per_run": (_I, [_P]),
    "spmm_b200_plan_select": (_I, [_P, _I]),
    "spmm_b200_plan_info": (_I, [_P, C.POINTER(PlanInfo)]),
    "spmm_b200_plan_copy": (_I, [_P, _I, _P, C.c_size_t]),
    "spmm_b200_plan_host": (_I, [_P, _I, _I, _LL, _I, _P, C.POINTER(_I), _P, C.POINTER(_I), _P, _P, C.POINTER(_I),
                                 C.POINTER(_LL)]),
    "spmm_b200_pack_light_host": (_I, [_P, _I, _I, _I, _P, _P, C.POINTER(_I), C.POINTER(_LL)]),
    "spmm_b200_fill_normal": (_I, [_P, _LL, _U64, _U64, C.c_float, C.c_float, _P]),
    "spmm_b200_valid": (_I, [_P, _P, _LL, C.POINTER(_LL), _P]),
    "spmm_b200_gen_graph": (_I, [_I, _LL, _I, _I, _I, _I, _I, _U64, _P, _P]),
    "spmm_b200_gen_degrees": (_I, [_I, _LL, _I, _I, _I, _U64, _P]),
    "spmm_b200_set_host_threads": (_I, [_I]),
    "spmm_b200_load_graph": (_I, [C.c_char_p, C.c_char_p, C.POINTER(_I), C.POINTER(_I), _P, _P]),
    "spmm_b200_write_graph": (_I, [C.c_char_p, C.c_char_p, _I, _I, _P, _P, _I]),
    "spmm_b200_partition_rows": (_I, [_P, _I, _I, _P]),
    "spmm_b200_partition_rows_weighted": (_I, [_P, _I, _I, _I, _P]),
    "spmm_b200_plan_row_cost": (_I, [_I, _LL, _I, _I]),
    "spmm_b200_rebase_ptr": (_I, [_P, _I, _I, _P]),
    "spmm_b200_set_replicate": (_I, [_P, _I, _I, C.POINTER(_P), _P, C.POINTER(_P)]),
    "spmm_b200_run_host_sharded": (_I, [_P, _P, _P, _P]),
    "spmm_b200_replicate_h2d_bytes": (_LL, [_P]),
    "spmm_b200_mg_create": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, C.POINTER(_P)]),
    "spmm_b200_mg_set_option": (_I, [_P, C.c_char_p, _LL]),
    "spmm_b200_mg_preprocess": (_I, [_P]),
    "spmm_b200_mg_info": (_I, [_P, C.POINTER(_I), _P, C.POINTER(_I)]),
    "spmm_b200_mg_device_buffers": (_I, [_P, _I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(_P)]),
    "spmm_b200_mg_run_host": (_I, [_P, _P, _P]),
    "spmm_b200_mg_run": (_I, [_P]),
    "spmm_b200_mg_sync": (_I, [_P]),
    "spmm_b200_mg_set_fused": (_I, [_P, _I]),
    "spmm_b200_mg_allgather": (_I, [_P]),
    "spmm_b200_mg_swap": (_I, [_P]),
    "spmm_b200_mg_destroy": (_I, [_P]),
}


class SpmmB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"spmm_b200 status {code}: {message}")
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no "
            "CPU fallback. Run `make -C hpc_b200/csrc` (or __graft_entry__.build())."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library diverge
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(status: int) -> None:
    if status != 0:
        raise SpmmB200Error(status, lib.spmm_b200_last_error().decode("utf-8", "replace"))
