"""TEST INFRASTRUCTURE: the min-cost walk over a match table (tests/c/mincost_walk.c), the checker of the GPU's
min-cost parse.  It takes the table from the oracle (oracle.Oracle.match_table) and walks it with the min-cost
rule instead of the oracle's greedy one.  The C file is compiled on first use into a temporary directory, which
is removed when the process exits; nothing is written into the tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "mincost_walk.c")
SEGMENT = 16384
_lib = None


def _load():
    global _lib
    if _lib is None:
        where = tempfile.mkdtemp(prefix="sqz_mincost_walk_")
        atexit.register(shutil.rmtree, where, True)
        so = os.path.join(where, "libmincostwalk.so")
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Werror", "-shared", "-fPIC", SRC, "-o", so])
        L = C.CDLL(so)
        u64 = C.c_uint64
        L.mincost_tokens_from_table.argtypes = [C.POINTER(C.c_uint8), u64, C.POINTER(C.c_uint16),
                                                C.POINTER(C.c_uint16), C.c_uint32, u64, C.POINTER(C.c_uint32), u64,
                                                C.POINTER(u64)]
        L.mincost_tokens_from_table.restype = u64
        _lib = L
    return _lib


def mincost_tokens_from_table(data, ln, ds, min_len: int = 3, start: int = 0):
    """(tokens, end position) of the min-cost walk from `start`, the arguments of Oracle.tokens_from_table."""
    d = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data,
                             dtype=np.uint8)
    ln = np.ascontiguousarray(ln, dtype=np.uint16)
    ds = np.ascontiguousarray(ds, dtype=np.uint16)
    t = np.zeros(max(d.size, 1), dtype=np.uint32)
    end = C.c_uint64()
    n = _load().mincost_tokens_from_table(d.ctypes.data_as(C.POINTER(C.c_uint8)), d.size,
                                          ln.ctypes.data_as(C.POINTER(C.c_uint16)),
                                          ds.ctypes.data_as(C.POINTER(C.c_uint16)),
                                          min_len, start, t.ctypes.data_as(C.POINTER(C.c_uint32)), t.size,
                                          C.byref(end))
    if n == 2 ** 64 - 1:
        raise MemoryError("mincost_tokens_from_table")
    return t[:n].copy(), int(end.value)
