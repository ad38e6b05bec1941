"""CPU oracle (test infrastructure only - see ``oracle/sage_oracle.py`` for the contract)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build_c_oracle() -> str:
    """Compile ``csr_oracle.c`` into ``oracle/_build/liboracle.so`` (gcc, ~1 s)."""
    so = os.path.join(_HERE, "_build", "liboracle.so")
    src = os.path.join(_HERE, "csr_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return so


def c_oracle():
    global _LIB
    if _LIB is None:
        lib = ctypes.CDLL(build_c_oracle())
        lib.oracle_csr_build.restype = ctypes.c_int
        lib.oracle_csr_build.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int] + [ctypes.c_void_p] * 4
        lib.oracle_csr_aggregate_f32.restype = None
        lib.oracle_csr_aggregate_f32.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int64, ctypes.c_int64]
        lib.oracle_csr_aggregate_ex_f32.restype = None
        lib.oracle_csr_aggregate_ex_f32.argtypes = [ctypes.c_void_p] * 7 + [ctypes.c_int64, ctypes.c_int64]
        _LIB = lib
    return _LIB


def csr_oracle_c(edge_index: np.ndarray, num_nodes: int, by: str = "dst"):
    """Same contract as ``sage_oracle.csr_oracle`` but through the C restatement."""
    ei = np.ascontiguousarray(edge_index, dtype=np.int64)
    E = ei.shape[1]
    rowptr = np.empty(num_nodes + 1, np.int32)
    col = np.empty(E, np.int32)
    perm = np.empty(E, np.int32)
    inv = np.empty(num_nodes, np.float32)
    rc = c_oracle().oracle_csr_build(ei.ctypes.data, E, num_nodes, int(by == "src"),
                                     rowptr.ctypes.data, col.ctypes.data, perm.ctypes.data, inv.ctypes.data)
    if rc == 1:
        raise IndexError("edge_index out of range")
    if rc:
        raise MemoryError
    return rowptr, col, perm, inv


def csr_aggregate_c(rowptr, col, inv_deg, x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty_like(x)
    c_oracle().oracle_csr_aggregate_f32(rowptr.ctypes.data, col.ctypes.data,
                                        inv_deg.ctypes.data if inv_deg is not None else None,
                                        x.ctypes.data, out.ctypes.data, x.shape[0], x.shape[1])
    return out


def csr_aggregate_ex(rowptr, col, x: np.ndarray, row_scale=None, src_scale=None, addend=None, n_rows=None) -> np.ndarray:
    """The gather kernel's arithmetic in every form (``oracle_csr_aggregate_ex_f32``): per row, in CSR order,
    ``acc = fmaf(x, src_scale[col], acc)`` or ``acc += x``, then ``fmaf(acc, row_scale, addend)`` or ``acc * row_scale``.
    fp32 in, fp32 out; ``x`` may have more rows than the ``n_rows`` destination rows (default: as many)."""
    def f32(a, shape):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float32)
        assert a.shape == shape, (a.shape, shape)
        return a

    x = np.ascontiguousarray(x, dtype=np.float32)
    n = x.shape[0] if n_rows is None else int(n_rows)
    H = x.shape[1]
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
    col = np.ascontiguousarray(col, dtype=np.int32)
    assert rowptr.shape == (n + 1,) and int(rowptr[-1]) == col.size
    assert col.size == 0 or (int(col.min()) >= 0 and int(col.max()) < x.shape[0])
    row_scale, src_scale, addend = f32(row_scale, (n,)), f32(src_scale, (x.shape[0],)), f32(addend, (n, H))
    out = np.empty((n, H), np.float32)
    p = lambda a: None if a is None else a.ctypes.data
    c_oracle().oracle_csr_aggregate_ex_f32(rowptr.ctypes.data, col.ctypes.data, p(row_scale), p(src_scale), x.ctypes.data,
                                           p(addend), out.ctypes.data, n, H)
    return out
