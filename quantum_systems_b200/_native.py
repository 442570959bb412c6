"""ctypes binding of libqsb200.so -- the C ABI declared in include/qsb200.h.

This is the only place where Python touches the native library.  Device pointers come from
``torch.Tensor.data_ptr()`` and the stream from ``torch.cuda.current_stream()``; torch is plumbing
(allocator, streams, NCCL), never arithmetic on the hot path.  There is no CPU fallback: if the
library is missing, or a call fails, a ``RuntimeError`` is raised.
"""

import ctypes
import os

QS_F64 = 0
QS_C128 = 1

_LIB = None
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libqsb200.so")

_i64 = ctypes.c_int64
_int = ctypes.c_int
_ptr = ctypes.c_void_p
_dbl = ctypes.c_double

# name -> argtypes; every function returns int status except the two noted below
SIGNATURES = {
    "qs_version": [],
    "qs_last_error": [],
    "qs_transform_two_body_workspace_bytes": [_i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_transform_two_body": [_ptr, _int, _ptr, _ptr, _int, _i64, _i64, _ptr, _ptr, _i64, _ptr],
    "qs_two_body_symmetry": [_ptr, _int, _i64, _int, ctypes.POINTER(_int), _ptr, _ptr],
    "qs_transform_two_body_symmetric": [_ptr, _int, _ptr, _ptr, _int, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr],
    "qs_transform_two_body_mixed": [_ptr, _int, _ptr, _ptr, _ptr, _ptr, _int, _i64, _i64, _ptr, _ptr, _i64, _ptr],
    "qs_coeff_image_bytes": [_i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_build_coeff_image": [_ptr, _int, _i64, _i64, _int, _i64, _i64, _int, _ptr, _ptr],
    "qs_quarter_transform": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _ptr],
    "qs_scatter_deal": [_i64, ctypes.POINTER(_i64)],
    "qs_build_coeff_image_dealt": [_ptr, _int, _i64, _i64, _int, _i64, _i64, _int, _i64, _ptr, _ptr],
    "qs_quarter_transform_scatter": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, ctypes.POINTER(_ptr), _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _int, _ptr],
    "qs_quarter_transform_scatter_pairs": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, ctypes.POINTER(_ptr), _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _int, _ptr, _i64, _ptr],
    "qs_quarter_transform_scatter_columns": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, ctypes.POINTER(_ptr), _i64, _ptr, _ptr, _int, _i64, _i64, _i64, _i64, _i64, _i64, _ptr],
    "qs_transform_two_body_diagonal_workspace_bytes": [_i64, _i64, _int, _int, _int, ctypes.POINTER(_i64)],
    "qs_transform_two_body_diagonal": [_ptr, _int, _ptr, _ptr, _int, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr],
    "qs_is_antisymmetric_last_pair": [_ptr, _int, _i64, _i64, ctypes.POINTER(_int), _ptr, _ptr],
    "qs_cyclic_antisymmetric_fill": [_ptr, _int, _i64, _i64, _ptr],
    "qs_cyclic_pair_wanted": [_i64, _i64, _i64],
    "qs_quarter_plan_tiles": [_i64, _i64, _i64, _int, _int, _i64, _int, _int, _i64, _i64, _i64, _i64, _ptr, _ptr, _i64, ctypes.POINTER(_i64)],
    "qs_quarter_tile_list_bytes": [_i64, _i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_quarter_transform_rows": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, _ptr, _i64, _i64, _ptr, _ptr, _i64, _i64, _i64, _ptr, _i64, _ptr],
    "qs_quarter_transform_scatter_rows": [_ptr, _int, _i64, _i64, _i64, _ptr, _int, _i64, ctypes.POINTER(_ptr), _i64, _i64, _i64, _ptr, _i64, _i64, _i64, _int, _ptr],
    "qs_pad_rows": [_ptr, _ptr, _i64, _i64, _i64, _int, _ptr],
    "qs_ipc_handle_bytes": [],
    "qs_ipc_alloc": [_i64, ctypes.POINTER(_ptr), _ptr],
    "qs_ipc_open": [_ptr, ctypes.POINTER(_ptr)],
    "qs_ipc_close": [_ptr],
    "qs_ipc_free": [_ptr],
    "qs_transform_one_body_workspace_bytes": [_i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_transform_one_body": [_ptr, _int, _ptr, _ptr, _int, _i64, _i64, _ptr, _ptr, _ptr],
    "qs_add_spin_two_body": [_ptr, _int, _i64, _ptr, _int, _int, _i64, _i64, _ptr],
    "qs_anti_symmetrize": [_ptr, _int, _i64, _ptr, _i64, _i64, _ptr],
    "qs_add_spin_one_body": [_ptr, _int, _i64, _ptr, _int, _ptr],
    "qs_spin_orbital_two_body": [_ptr, _ptr, _ptr, _ptr, _int, _i64, _ptr, _ptr, _ptr, _int, _i64, _i64, _ptr],
    "qs_spin_squared_two_body": [_ptr, _ptr, _ptr, _i64, _int, _ptr, _i64, _i64, _ptr],
    "qs_fock_gathered": [_ptr, _int, _ptr, _ptr, _int, _i64, _i64, _dbl, _dbl, _ptr, _ptr],
    "qs_fock_general": [_ptr, _int, _ptr, _int, _i64, _i64, _ptr, _i64, _i64, _ptr],
    "qs_fock_general_cols": [_ptr, _int, _ptr, _int, _i64, _i64, _ptr, _i64, _i64, _ptr],
    "qs_fock_spatial": [_ptr, _int, _ptr, _int, _i64, _i64, _ptr, _i64, _i64, _ptr],
    "qs_fock_density_workspace_bytes": [_i64, _i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_fock_density": [_ptr, _int, _ptr, _int, _ptr, _int, _i64, _dbl, _dbl, _ptr, _int, _i64, _i64, _ptr, _i64, _ptr],
    "qs_fock_density_unrestricted_workspace_bytes": [_i64, _i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_fock_density_unrestricted": [_ptr, _int, _ptr, _int, _ptr, _ptr, _int, _i64, _ptr, _ptr, _int, _i64, _i64, _ptr, _i64, _ptr],
    "qs_coulomb_exchange_batch_workspace_bytes": [_i64, _i64, _i64, _i64, _int, _int, ctypes.POINTER(_i64)],
    "qs_coulomb_exchange_batch": [_ptr, _int, _ptr, _int, _i64, _i64, _ptr, _ptr, _i64, _i64, _ptr, _i64, _ptr],
    "qs_odqd_coulomb_workspace_bytes": [_i64, _i64, ctypes.POINTER(_i64)],
    "qs_odqd_coulomb": [_ptr, _ptr, _dbl, _dbl, _i64, _i64, _ptr, _ptr, _i64, _ptr],
    "qs_odqd_coulomb_planes": [_ptr, _ptr, _dbl, _dbl, _i64, _i64, _ptr, _i64, _i64, _ptr, _i64, _ptr],
    "qs_tdho_coulomb_workspace_bytes": [ctypes.POINTER(_i64), ctypes.POINTER(_i64), _i64, ctypes.POINTER(_i64)],
    "qs_tdho_coulomb": [ctypes.POINTER(_i64), ctypes.POINTER(_i64), _i64, _dbl, _ptr, _i64, _i64, _ptr, _i64, _ptr],
    "qs_extract_block": [_ptr, _int, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _ptr, _ptr],
    "qs_scale_add": [_ptr, _ptr, _int, _i64, _dbl, _dbl, _dbl, _dbl, _ptr, _ptr],
    "qs_occupied_traces": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _ptr],
    "qs_set_bulk_epilogue_mode": [_int],
    "qs_launch_count": [],
    "qs_kernel_timing_enable": [_int],
    "qs_kernel_timing_read": [_int, ctypes.POINTER(_dbl), ctypes.POINTER(_dbl), ctypes.POINTER(_i64)],
    "qs_probe_dmma_tflops": [ctypes.POINTER(_dbl), _ptr],
    "qs_probe_copy_gbs": [ctypes.POINTER(_dbl), _ptr, _i64, _ptr],
}


def library_path():
    return _LIB_PATH


def load():
    """dlopen libqsb200.so (once) and declare every prototype.  Raises if the library is absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} not found: build it with `python -m quantum_systems_b200.build` "
            "(quantum_systems_b200 has no CPU fallback)"
        )
    lib = ctypes.CDLL(_LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.argtypes = argtypes
        fn.restype = {"qs_last_error": ctypes.c_char_p, "qs_launch_count": ctypes.c_int64}.get(name, ctypes.c_int)
    _LIB = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().qs_last_error()
        raise RuntimeError(f"{what} failed (status {status}): {msg.decode() if msg else 'no message'}")


def call(name, *args):
    """Call a status-returning entry point and raise on failure."""
    check(getattr(load(), name)(*args), name)
