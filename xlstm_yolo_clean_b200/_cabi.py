"""ctypes binding of include/mlstm_b200.h (the C-ABI shared library).

The library is the ONLY compute path: if it is missing or cannot be loaded, every call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmlstm_b200.so")

F32, BF16, F16 = 0, 1, 2
IMPL_AUTO, IMPL_EXACT, IMPL_TENSOR = 0, 1, 2
ABI_VERSION = 4

EXPORTS = (
    "mlstm_b200_abi_version",
    "mlstm_b200_last_error",
    "mlstm_b200_workspace_bytes",
    "mlstm_b200_states_bytes",
    "mlstm_b200_tensor_path_supported",
    "mlstm_b200_chunkwise_fw",
    "mlstm_b200_chunkwise_bw",
    "mlstm_b200_last_launch_count",
    "mlstm_b200_debug_set_clock_buffer",
    "mlstm_b200_debug_fw_epilogue_clusters",
    "mlstm_b200_recurrent_sequence",
    "mlstm_b200_cellout_workspace_bytes",
    "mlstm_b200_cellout_fw",
    "mlstm_b200_cellout_bw",
    "mlstm_b200_rmsnorm_workspace_bytes",
    "mlstm_b200_rmsnorm_fw",
    "mlstm_b200_rmsnorm_bw",
    "mlstm_b200_convert16",
)


class Tensor(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride", C.c_int64 * 4)]


class Shape(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("NH", C.c_int32), ("S", C.c_int32), ("DHQK", C.c_int32), ("DHHV", C.c_int32),
        ("chunk_size", C.c_int32), ("dtype", C.c_int32), ("impl", C.c_int32), ("reverse", C.c_int32), ("siging", C.c_int32),
        ("eps", C.c_float), ("qk_scale", C.c_float), ("gate_soft_cap", C.c_float), ("grad_dtype", C.c_int32),
    ]


class FwEpilogue(C.Structure):
    _fields_ = [
        ("y", Tensor), ("x", Tensor),
        ("weight", C.c_void_p), ("bias", C.c_void_p), ("skip", C.c_void_p),
        ("eps", C.c_float), ("xy_dtype", C.c_int32),
    ]


class FwArgs(C.Structure):
    _fields_ = [
        ("shape", Shape),
        ("q", Tensor), ("k", Tensor), ("v", Tensor), ("i", Tensor), ("f", Tensor),
        ("c_initial", C.c_void_p), ("n_initial", C.c_void_p), ("m_initial", C.c_void_p),
        ("h", Tensor),
        ("n_out", C.c_void_p), ("m_out", C.c_void_p),
        ("c_last", C.c_void_p), ("n_last", C.c_void_p), ("m_last", C.c_void_p),
        ("c_states", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("epilogue", C.POINTER(FwEpilogue)),
    ]


class BwArgs(C.Structure):
    _fields_ = [
        ("shape", Shape),
        ("q", Tensor), ("k", Tensor), ("v", Tensor), ("i", Tensor), ("f", Tensor),
        ("c_initial", C.c_void_p), ("n_initial", C.c_void_p), ("m_initial", C.c_void_p),
        ("n_out", C.c_void_p), ("m_out", C.c_void_p),
        ("c_states", C.c_void_p),
        ("dh", Tensor),
        ("dc_last", C.c_void_p),
        ("dq", Tensor), ("dk", Tensor), ("dv", Tensor), ("di", Tensor), ("df", Tensor),
        ("dc_initial", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class RecurrentArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("NH", C.c_int32), ("S", C.c_int32), ("DHQK", C.c_int32), ("DHHV", C.c_int32),
        ("dtype", C.c_int32), ("siging", C.c_int32), ("eps", C.c_float),
        ("q", Tensor), ("k", Tensor), ("v", Tensor), ("i", Tensor), ("f", Tensor),
        ("c_initial", C.c_void_p), ("n_initial", C.c_void_p), ("m_initial", C.c_void_p),
        ("h", Tensor),
        ("c_last", C.c_void_p), ("n_last", C.c_void_p), ("m_last", C.c_void_p),
    ]


class CellOutArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("NH", C.c_int32), ("S", C.c_int32), ("D", C.c_int32),
        ("h_dtype", C.c_int32), ("x_dtype", C.c_int32), ("y_dtype", C.c_int32),
        ("eps", C.c_float),
        ("h", Tensor), ("x", Tensor), ("y", Tensor),
        ("weight", C.c_void_p), ("bias", C.c_void_p), ("skip", C.c_void_p),
    ]


class CellOutBwArgs(C.Structure):
    _fields_ = [
        ("fw", CellOutArgs),
        ("dy", Tensor), ("dh", Tensor), ("dx", Tensor),
        ("dweight", C.c_void_p), ("dbias", C.c_void_p), ("dskip", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class RmsNormArgs(C.Structure):
    _fields_ = [
        ("rows", C.c_int64), ("C", C.c_int32), ("x_dtype", C.c_int32), ("y_dtype", C.c_int32), ("eps", C.c_float),
        ("x", C.c_void_p), ("y", C.c_void_p), ("weight", C.c_void_p), ("rstd", C.c_void_p),
    ]


class RmsNormBwArgs(C.Structure):
    _fields_ = [
        ("fw", RmsNormArgs),
        ("dy", C.c_void_p), ("dx", C.c_void_p), ("dweight", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


_lib = None


class LibraryMissing(RuntimeError):
    pass


def load_library(path: str | None = None):
    """dlopen the C-ABI library and declare prototypes.  Raises LibraryMissing if absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("MLSTM_B200_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise LibraryMissing(
            f"{path} not found: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for this backend.")
    lib = C.CDLL(path)
    lib.mlstm_b200_abi_version.restype = C.c_int
    lib.mlstm_b200_last_error.restype = C.c_char_p
    lib.mlstm_b200_workspace_bytes.restype = C.c_size_t
    lib.mlstm_b200_workspace_bytes.argtypes = [C.POINTER(Shape), C.c_int]
    lib.mlstm_b200_states_bytes.restype = C.c_size_t
    lib.mlstm_b200_states_bytes.argtypes = [C.POINTER(Shape)]
    lib.mlstm_b200_tensor_path_supported.restype = C.c_int
    lib.mlstm_b200_tensor_path_supported.argtypes = [C.POINTER(Shape)]
    lib.mlstm_b200_chunkwise_fw.restype = C.c_int
    lib.mlstm_b200_chunkwise_fw.argtypes = [C.POINTER(FwArgs), C.c_void_p]
    lib.mlstm_b200_chunkwise_bw.restype = C.c_int
    lib.mlstm_b200_chunkwise_bw.argtypes = [C.POINTER(BwArgs), C.c_void_p]
    lib.mlstm_b200_last_launch_count.restype = C.c_int
    lib.mlstm_b200_debug_set_clock_buffer.restype = None
    lib.mlstm_b200_debug_set_clock_buffer.argtypes = [C.c_void_p]
    lib.mlstm_b200_debug_fw_epilogue_clusters.restype = C.c_int
    lib.mlstm_b200_debug_fw_epilogue_clusters.argtypes = [C.POINTER(Shape)]
    lib.mlstm_b200_recurrent_sequence.restype = C.c_int
    lib.mlstm_b200_recurrent_sequence.argtypes = [C.POINTER(RecurrentArgs), C.c_void_p]
    lib.mlstm_b200_cellout_workspace_bytes.restype = C.c_size_t
    lib.mlstm_b200_cellout_workspace_bytes.argtypes = [C.POINTER(CellOutArgs)]
    lib.mlstm_b200_cellout_fw.restype = C.c_int
    lib.mlstm_b200_cellout_fw.argtypes = [C.POINTER(CellOutArgs), C.c_void_p]
    lib.mlstm_b200_cellout_bw.restype = C.c_int
    lib.mlstm_b200_cellout_bw.argtypes = [C.POINTER(CellOutBwArgs), C.c_void_p]
    lib.mlstm_b200_rmsnorm_workspace_bytes.restype = C.c_size_t
    lib.mlstm_b200_rmsnorm_workspace_bytes.argtypes = [C.POINTER(RmsNormArgs)]
    lib.mlstm_b200_rmsnorm_fw.restype = C.c_int
    lib.mlstm_b200_rmsnorm_fw.argtypes = [C.POINTER(RmsNormArgs), C.c_void_p]
    lib.mlstm_b200_rmsnorm_bw.restype = C.c_int
    lib.mlstm_b200_rmsnorm_bw.argtypes = [C.POINTER(RmsNormBwArgs), C.c_void_p]
    lib.mlstm_b200_convert16.restype = C.c_int
    lib.mlstm_b200_convert16.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    v = lib.mlstm_b200_abi_version()
    if v != ABI_VERSION:
        raise RuntimeError(f"ABI mismatch: library {v}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(status: int, what: str):
    if status != 0:
        msg = load_library().mlstm_b200_last_error().decode()
        kind = "invalid argument" if status < 0 else f"CUDA error {status}"
        if status == -1 and "not divisible" in msg:
            raise AssertionError(msg)  # same error class as the reference (native/fw.py:252-254)
        raise RuntimeError(f"{what}: {kind}: {msg}")
