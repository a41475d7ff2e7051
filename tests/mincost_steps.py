"""TEST INFRASTRUCTURE: the table words the min-cost rewrite leaves (tests/c/mincost_steps.c), the checker of
sqz_gpu_mincost_steps_device and of the premise that min-cost shards chain like greedy ones.  The C file is
compiled on first use into a temporary directory, which is removed when the process exits; nothing is written
into the tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "c", "mincost_steps.c")
_lib = None


def _load():
    global _lib
    if _lib is None:
        where = tempfile.mkdtemp(prefix="sqz_mincost_steps_")
        atexit.register(shutil.rmtree, where, True)
        so = os.path.join(where, "libmincoststeps.so")
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Werror", "-shared", "-fPIC",
                               "-I" + os.path.join(HERE, "c"), SRC, "-o", so])
        L = C.CDLL(so)
        u16p = C.POINTER(C.c_uint16)
        L.mincost_steps_from_table.argtypes = [u16p, u16p, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint32)]
        L.mincost_steps_from_table.restype = C.c_int
        _lib = L
    return _lib


def mincost_steps_from_table(ln, ds, min_len: int = 3) -> np.ndarray:
    """The rewritten table, word for word: (k << 16) | dist for the chosen match of k, 0 for a literal, with
    segments of 16384 positions from the start of `ln` / `ds`."""
    ln = np.ascontiguousarray(ln, dtype=np.uint16)
    ds = np.ascontiguousarray(ds, dtype=np.uint16)
    words = np.zeros(max(ln.size, 1), dtype=np.uint32)
    rc = _load().mincost_steps_from_table(ln.ctypes.data_as(C.POINTER(C.c_uint16)),
                                          ds.ctypes.data_as(C.POINTER(C.c_uint16)), ln.size, min_len,
                                          words.ctypes.data_as(C.POINTER(C.c_uint32)))
    if rc != 0:
        raise MemoryError("mincost_steps_from_table")
    return words[: ln.size].copy()


def walk_steps(data, words, start: int = 0):
    """(tokens, end position) of the greedy walk over rewritten words from `start`: what the device parse of a
    rewritten table emits."""
    d = np.asarray(data, dtype=np.uint8)
    w = np.asarray(words, dtype=np.uint32)
    out, i = [], start
    while i < w.size:
        k = int(w[i]) >> 16
        out.append(int(w[i]) if k else int(d[i]))
        i += k if k else 1
    return np.array(out, dtype=np.uint32), i
