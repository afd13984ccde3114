"""ctypes binding of the C ABI in include/circom_b200.h (libcircom_b200.so).

The library is the product: if it is missing it is built with nvcc; if it cannot be
loaded the import fails loudly (there is no Python / CPU fallback for the hot path).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p

from . import build as _build

CW_OK, CW_EINVAL, CW_EIO, CW_EFORMAT, CW_ECUDA, CW_ENOTFOUND, CW_ESTATE, CW_ENODEV = 0, -1, -2, -3, -4, -5, -6, -7
CW_FLAG_NO_ASSERTS, CW_FLAG_HOST_ONLY, CW_FLAG_O0, CW_FLAG_NO_PEEPHOLE, CW_FLAG_BITPLANE, CW_FLAG_REUSE = 1, 2, 4, 8, 16, 32
CW_FLAG_COMPACT = CW_FLAG_BITPLANE | CW_FLAG_REUSE
CW_FLAG_FUSE = 64
CW_FLAG_NO_TYPED = 128


class CwError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("circom_b200 error %d: %s" % (code, msg))
        self.code = code


class CwStats(ctypes.Structure):
    _fields_ = [(n, c_uint64) for n in (
        "n_signals", "n_witness", "n_inputs", "n_outputs", "n_components", "n_constants", "n_ir_ops",
        "n_tape_ops", "n_slots", "n_levels", "n_constraints", "n_nnz", "n_mul_ops", "n_conv_ops",
        "max_level_width", "n_slot_operands", "n_bitwords", "n_resident_slots", "n_items", "n_stored", "n_values")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def _load() -> ctypes.CDLL:
    path = os.environ.get("CW_LIB_PATH") or _build.LIB   # (CW_LIB_PATH: an experimental build of the same ABI)
    if not os.path.exists(path):
        _build.build()
    lib = ctypes.CDLL(path)
    P = c_void_p
    sig = {
        "cw_version": (c_int, []),
        "cw_last_error": (c_char_p, []),
        "cw_device_count": (c_int, []),
        "cw_circuit_load": (c_int, [c_char_p, c_uint32, POINTER(P)]),
        "cw_circuit_load_mem": (c_int, [c_void_p, c_size_t, c_uint32, POINTER(P)]),
        "cw_circuit_destroy": (None, [P]),
        "cw_circuit_stats": (c_int, [P, POINTER(CwStats)]),
        "cw_circuit_prime": (c_int, [P, POINTER(c_int), POINTER(c_uint64)]),
        "cw_get_main_input_signal_start": (c_uint32, [P]),
        "cw_get_main_input_signal_no": (c_uint32, [P]),
        "cw_get_total_signal_no": (c_uint32, [P]),
        "cw_get_number_of_components": (c_uint32, [P]),
        "cw_get_size_of_input_hashmap": (c_uint32, [P]),
        "cw_get_size_of_witness": (c_uint32, [P]),
        "cw_get_size_of_constants": (c_uint32, [P]),
        "cw_fnv1a": (c_uint64, [c_char_p]),
        "cw_get_input_signal_size": (c_int, [P, c_uint64, POINTER(c_uint64)]),
        "cw_get_input_signal_id": (c_int, [P, c_uint64, POINTER(c_uint64)]),
        "cw_circuit_tape": (c_int, [P, c_void_p, c_void_p, c_void_p]),
        "cw_circuit_tape_items": (c_int, [P, c_void_p]),
        "cw_circuit_slot_census": (c_int, [P, POINTER(c_uint64)]),
        "cw_circuit_witness2signal": (c_int, [P, c_void_p]),
        "cw_circuit_write_dat": (c_int, [P, c_char_p]),
        "cw_circuit_write_sym": (c_int, [P, c_char_p]),
        "cw_circuit_functions": (c_int, [P, POINTER(c_uint32), POINTER(c_uint32)]),
        "cw_batch_create": (c_int, [P, c_uint32, c_int, POINTER(P)]),
        "cw_batch_destroy": (None, [P]),
        "cw_batch_set_input": (c_int, [P, c_uint32, c_uint64, c_uint32, POINTER(c_uint64)]),
        "cw_batch_remaining_inputs": (c_int, [P, c_uint32, POINTER(c_uint32)]),
        "cw_batch_set_inputs": (c_int, [P, c_void_p, c_int]),
        "cw_batch_run": (c_int, [P]),
        "cw_batch_sync": (c_int, [P]),
        "cw_batch_status": (c_int, [P, c_void_p]),
        "cw_batch_get_witness": (c_int, [P, c_void_p]),
        "cw_batch_last_d2h_bytes": (c_uint64, [P]),
        "cw_batch_layout": (c_int, [P, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint64)]),
        "cw_batch_get_witness_async": (c_int, [P, c_void_p]),
        "cw_batch_get_witness_wait": (c_int, [P]),
        "cw_batch_get_witness_packed": (c_int, [P, c_void_p]),
        "cw_circuit_pack_info": (c_int, [P, POINTER(c_uint64), c_void_p]),
        "cw_batch_expand_witness": (c_int, [P, c_uint32, c_uint32, c_void_p]),
        "cw_r1cs_check_batch": (c_int, [P, P, c_void_p, POINTER(c_float)]),
        "cw_r1cs_eval_batch": (c_int, [P, P, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p]),
        "cw_comm_unique_id": (c_int, [c_void_p]),
        "cw_comm_init": (c_int, [c_void_p, c_int, c_int, c_int, POINTER(P)]),
        "cw_comm_from_nccl": (c_int, [c_void_p, c_int, c_int, c_int, POINTER(P)]),
        "cw_comm_destroy": (None, [P]),
        "cw_comm_stats": (c_int, [P, POINTER(c_uint64), POINTER(c_uint64)]),
        "cw_circuit_serialize": (c_int, [P, c_void_p, c_size_t, POINTER(c_size_t)]),
        "cw_circuit_deserialize": (c_int, [c_void_p, c_size_t, POINTER(P)]),
        "cw_circuit_broadcast": (c_int, [P, POINTER(P), c_int]),
        "cw_batch_pack_device": (c_int, [P, c_uint32, c_uint32, c_void_p]),
        "cw_batch_gather_witness_packed": (c_int, [P, P, c_uint32, c_uint32, c_int, c_void_p, c_void_p, POINTER(c_float)]),
        "cw_status_allreduce": (c_int, [P, P, POINTER(c_uint64)]),
        "cw_circuit_expand_record": (c_int, [P, c_void_p, c_void_p, c_int]),
        "cw_host_expand_isa": (c_char_p, []),
        "cw_host_pool_info": (c_char_p, []),
        "cw_host_expand_bench": (c_int, [P, c_uint32, c_uint32, c_int, c_void_p]),
        "cw_wtns_read": (c_int, [c_char_p, POINTER(c_int), POINTER(c_uint64), c_void_p, c_size_t]),
        "cw_r1cs_check_files": (c_int, [c_char_p, c_char_p, c_int, POINTER(c_int64)]),
        "cw_batch_witness_device": (c_int, [P, POINTER(c_void_p)]),
        "cw_batch_witness_strided": (c_int, [P, POINTER(c_void_p), POINTER(c_uint64)]),
        "cw_batch_stream": (c_void_p, [P]),
        "cw_batch_last_ms": (c_int, [P, POINTER(c_float), POINTER(c_float)]),
        "cw_batch_write_wtns": (c_int, [P, c_uint32, c_char_p]),
        "cw_batch_wtns_bytes": (c_int, [P, c_uint32, c_void_p, c_size_t, POINTER(c_size_t)]),
        "cw_r1cs_from_circuit": (c_int, [P, POINTER(P)]),
        "cw_r1cs_load": (c_int, [c_char_p, POINTER(P)]),
        "cw_r1cs_write": (c_int, [P, c_char_p, c_uint32, c_uint32, c_uint32]),
        "cw_r1cs_info": (c_int, [P, POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint64), POINTER(c_int)]),
        "cw_r1cs_compiled_info": (c_int, [P, P, c_int, POINTER(c_uint64)]),
        "cw_circuit_assert_info": (c_int, [P, c_uint32, c_char_p, c_size_t, POINTER(c_size_t)]),
        "cw_circuit_format_log": (c_int, [P, c_void_p, c_char_p, c_size_t, POINTER(c_size_t)]),
        "cw_batch_log": (c_int, [P, c_uint32, c_char_p, c_size_t, POINTER(c_size_t)]),
        "cw_r1cs_destroy": (None, [P]),
        "cw_r1cs_check": (c_int, [P, c_void_p, c_int, c_uint32, c_int, c_void_p, POINTER(c_float)]),
        "cw_r1cs_check_strided": (c_int, [P, c_void_p, c_uint64, c_int, c_uint32, c_int, c_void_p, POINTER(c_float)]),
        "cw_fr_batch_op": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int]),
        "cw_fr_mul_bench": (c_int, [c_int, c_size_t, c_int, c_int, POINTER(c_float)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    lib._cw_symbols = sorted(sig)
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != CW_OK:
        raise CwError(rc, (lib.cw_last_error() or b"").decode())
