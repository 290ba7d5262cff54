"""ctypes binding of the C-ABI in include/queasars_b200.h.  There is no CPU fallback: if the shared
library is missing this raises, and every compute call needs a CUDA device."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_uint64, c_void_p

import numpy as np

from . import schedule
from ._build import LIB_PATH

QB_OK = 0
QB_C128, QB_C64 = 0, 1
QB_ERR_INVALID, QB_ERR_CUDA, QB_ERR_MEMORY, QB_ERR_NOT_FOUND = -1, -2, -3, -4


class NativeLibraryError(RuntimeError):
    pass


class QbError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"queasars_b200 native error {code}: {message}")
        self.code = code


_lib = None


def _declare(lib):
    P = POINTER
    sigs = {
        "qb_context_create": [c_int, c_void_p, P(c_void_p)],
        "qb_device_count": [P(c_int)],
        "qb_context_destroy": [c_void_p],
        "qb_context_stream": [c_void_p],
        "qb_context_launch_count": [c_void_p],
        "qb_context_set_workspace_limit": [c_void_p, c_uint64],
        "qb_context_synchronize": [c_void_p],
        "qb_context_set_index_width": [c_void_p, c_int],
        "qb_plan_create": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, P(c_int64)],
        "qb_plan_destroy": [c_void_p, c_int64],
        "qb_plan_set_prefix": [c_void_p, c_int64, c_int64],
        "qb_hamiltonian_create": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, P(c_int64)],
        "qb_hamiltonian_destroy": [c_void_p, c_int64],
        "qb_hamiltonian_diag_energies": [c_void_p, c_int64, c_int64, c_void_p, c_void_p],
        "qb_evaluate_expectation": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
        "qb_evaluate_expectation_multi": [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
        "qb_evaluate_expectation_submit": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64],
        "qb_evaluate_expectation_collect": [c_void_p, c_int, c_void_p],
        "qb_context_sm_count": [c_void_p],
        "qb_sample": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p],
        "qb_evaluate_cvar": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_double, c_void_p],
        "qb_observables_create": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, P(c_int64)],
        "qb_observables_destroy": [c_void_p, c_int64],
        "qb_evaluate_observables": [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
        "qb_statevector": [c_void_p, c_int64, c_void_p, c_int, c_void_p],
        "qb_batch_create": [c_void_p, c_int, c_void_p, c_int64, P(c_int64)],
        "qb_batch_set_params": [c_void_p, c_int64, c_void_p, c_void_p],
        "qb_batch_run": [c_void_p, c_int64],
        "qb_batch_read": [c_void_p, c_int64, c_void_p],
        "qb_batch_run_timed": [c_void_p, c_int64, c_int, c_void_p, c_void_p, P(c_int)],
        "qb_batch_destroy": [c_void_p, c_int64],
        "qb_batch_stats": [c_void_p, c_int64, P(c_int64), P(c_int64), P(c_int64), P(c_int64)],
        "qb_apply_plan_device": [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_int, c_uint64],
        "qb_expectation_device": [c_void_p, c_int64, c_int, c_int, c_void_p, c_uint64, P(c_double)],
        "qb_sample_device": [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p],
        "qb_cvar_select_device": [c_void_p, c_int64, c_int, c_int, c_void_p, c_uint64, c_void_p, c_int, c_uint64, c_int, c_int, c_int, c_void_p,
                                  c_uint64, c_uint64, c_void_p, c_void_p],
        "qb_swap_global_p2p": [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
        "qb_device_alloc": [c_void_p, c_uint64, P(c_void_p)],
        "qb_device_free": [c_void_p, c_void_p],
        "qb_device_read": [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p],
        "qb_enable_peer_access": [c_void_p, c_int],
        "qb_ipc_export": [c_void_p, c_void_p, c_void_p],
        "qb_ipc_open": [c_void_p, c_void_p, P(c_void_p)],
        "qb_ipc_close": [c_void_p, c_void_p],
    }
    for name, argtypes in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = c_int
    lib.qb_context_stream.restype = c_void_p
    lib.qb_context_launch_count.restype = c_int64
    lib.qb_context_workspace.argtypes = [c_void_p]
    lib.qb_context_workspace.restype = c_uint64
    lib.qb_last_error.argtypes = []
    lib.qb_last_error.restype = c_char_p
    lib.qb_record_sizes.argtypes = [P(c_int32)]
    lib.qb_record_sizes.restype = None
    return sigs


EXPORTED_SYMBOLS = (
    "qb_device_count qb_context_create qb_context_destroy qb_last_error qb_context_stream qb_context_launch_count "
    "qb_context_set_workspace_limit qb_context_workspace qb_context_synchronize qb_context_set_index_width qb_plan_create qb_plan_destroy qb_plan_set_prefix qb_hamiltonian_create "
    "qb_hamiltonian_destroy qb_hamiltonian_diag_energies qb_evaluate_expectation qb_sample qb_evaluate_cvar qb_statevector "
    "qb_observables_create qb_observables_destroy qb_evaluate_observables "
    "qb_evaluate_expectation_multi qb_evaluate_expectation_submit qb_evaluate_expectation_collect qb_context_sm_count "
    "qb_batch_create qb_batch_set_params qb_batch_run qb_batch_run_timed qb_batch_read qb_batch_destroy qb_batch_stats "
    "qb_apply_plan_device qb_expectation_device qb_sample_device qb_cvar_select_device qb_swap_global_p2p qb_record_sizes "
    "qb_device_alloc qb_device_free qb_device_read qb_enable_peer_access qb_ipc_export qb_ipc_open qb_ipc_close"
).split()


def load():
    """Load (once) and return the native library; raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("QB_NATIVE_LIB", LIB_PATH)  # development aid: A/B a differently built library
    if not os.path.exists(path):
        raise NativeLibraryError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  queasars_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(path)
    _declare(lib)
    sizes = (c_int32 * 4)()
    lib.qb_record_sizes(sizes)
    expect = [schedule.SWEEP_DTYPE.itemsize, schedule.PASS_DTYPE.itemsize, schedule.PASSOP_DTYPE.itemsize, schedule.ANGLE_DTYPE.itemsize]
    if list(sizes) != expect:
        raise NativeLibraryError(f"record layout mismatch between schedule.py {expect} and the native library {list(sizes)}")
    _lib = lib
    return lib


def check(code: int):
    if code != QB_OK:
        raise QbError(code, load().qb_last_error().decode("utf-8", "replace"))


def ptr(arr: np.ndarray):
    """Address of the array's buffer (the c_void_p argtypes take a plain int: half the cost of ``ctypes.data_as``, which matters
    on the single-circuit call path).  The caller keeps the array alive across the native call."""
    return arr.ctypes.data


def device_count() -> int:
    out = c_int()
    check(load().qb_device_count(ctypes.byref(out)))
    return int(out.value)


_pyhelper = None


def pyhelper():
    """ctypes.PyDLL handle of the list -> float64 marshalling helper (csrc/qb_pyhelper.c), or False when it is not built /
    not loadable (callers then convert with NumPy: this is host-side data marshalling, not a compute fallback)."""
    global _pyhelper
    if _pyhelper is None:
        from ._build import PYHELPER_PATH

        try:
            lib = ctypes.PyDLL(PYHELPER_PATH)
            lib.qb_pack_rows.argtypes = [ctypes.py_object, c_void_p, c_void_p, ctypes.c_longlong]
            lib.qb_pack_rows.restype = ctypes.c_longlong
            lib.qb_single_expectation.argtypes = [c_void_p, c_void_p, ctypes.c_longlong, ctypes.c_longlong, ctypes.py_object, ctypes.c_longlong]
            lib.qb_single_expectation.restype = ctypes.py_object
            _pyhelper = lib
        except (OSError, AttributeError):
            _pyhelper = False
    return _pyhelper
