"""TEST INFRASTRUCTURE ONLY — ctypes binding of the CPU checkers of core and truss numbers (tests/cpp/truss_oracle.cpp).

The library is compiled on first use into a temporary directory keyed by the source's hash, so a read-only tree works.
Both functions take a symmetric CSR as the oracle's Graph.csr() or gms_b200's Graph.export_csr() return it."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cpp", "truss_oracle.cpp")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_lib = None


def lib():
    global _lib
    if _lib is None:
        digest = hashlib.sha256(open(SRC, "rb").read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"gmsb_truss_oracle_{os.getuid()}_{digest}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-shared", "-fPIC", SRC, "-o", tmp])
            os.replace(tmp, path)
        dll = C.CDLL(path)
        dll.tor_core_numbers.restype = None
        dll.tor_core_numbers.argtypes = [C.c_int64, _i64p, _i32p, _i32p]
        dll.tor_truss_numbers.restype = C.c_int64
        dll.tor_truss_numbers.argtypes = [C.c_int64, _i64p, _i32p, C.c_void_p]
        _lib = dll
    return _lib


def _csr(off, nbr):
    off = np.ascontiguousarray(off, np.int64)
    nbr = np.ascontiguousarray(nbr, np.int32)
    return off, (nbr if len(nbr) else np.zeros(1, np.int32))


def core_numbers(off, nbr):
    """Core number of every vertex (Batagelj-Zaversnik bucket peel)."""
    off, nbr = _csr(off, nbr)
    out = np.zeros(max(len(off) - 1, 1), np.int32)
    lib().tor_core_numbers(len(off) - 1, off, nbr, out)
    return out[:len(off) - 1]


def truss_numbers(off, nbr):
    """Truss number of every undirected edge u<v in CSR order (sequential bucket peel of triangle support)."""
    off, nbr = _csr(off, nbr)
    m = lib().tor_truss_numbers(len(off) - 1, off, nbr, None)
    out = np.zeros(max(m, 1), np.int32)
    lib().tor_truss_numbers(len(off) - 1, off, nbr, out.ctypes.data)
    return out[:m]
