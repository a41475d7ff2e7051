"""TEST INFRASTRUCTURE: the reference decoder's copy loop (tests/c/lz_execute.c), the checker of the GPU
copy phase (sqz_gpu_expand_tokens and its device form), and the seeded token-stream generators the
tests share.  The C file is compiled on first use into a temporary directory, which is removed when
the process exits; nothing is written into the tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "lz_execute.c")
SHORT = (1 << 64) - 1          # lz_execute: every token is good, but they describe too few bytes
_lib = None


def _load():
    global _lib
    if _lib is None:
        where = tempfile.mkdtemp(prefix="sqz_lz_execute_")
        atexit.register(shutil.rmtree, where, True)
        so = os.path.join(where, "liblzexecute.so")
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Werror", "-shared", "-fPIC", SRC, "-o", so])
        L = C.CDLL(so)
        L.lz_execute.argtypes = [C.POINTER(C.c_uint32), C.c_uint64, C.POINTER(C.c_uint8), C.c_uint64]
        L.lz_execute.restype = C.c_uint64
        _lib = L
    return _lib


def execute(tokens, nbytes: int, out=None):
    """(code, out): lz_execute's code (0, 1 + index of the first bad token, or SHORT) and the buffer it
    wrote, `out` (a uint8 array of at least nbytes) or a new zeroed one."""
    t = np.ascontiguousarray(tokens, dtype=np.uint32)
    if out is None:
        out = np.zeros(max(nbytes, 1), dtype=np.uint8)
    assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size >= nbytes
    code = _load().lz_execute(t.ctypes.data_as(C.POINTER(C.c_uint32)), t.size,
                              out.ctypes.data_as(C.POINTER(C.c_uint8)), nbytes)
    return int(code), out


def expand(tokens, nbytes: int) -> np.ndarray:
    """The nbytes bytes a valid token stream describes."""
    code, out = execute(tokens, nbytes)
    assert code == 0, ("lz_execute refused the stream", code)
    return out[:nbytes]


# ---- seeded token streams -------------------------------------------------------------------------

def _lengths(rng, n: int, lit: float, long: float, min_len: int, max_len: int) -> np.ndarray:
    """n token lengths, 0 for a literal (probability `lit`).  A match is min_len..min(32, max_len) long
    or, with probability `long`, a log-uniform draw from min_len..max_len (the heavy tail)."""
    ln = rng.integers(min_len, min(32, max_len) + 1, n, dtype=np.int64)
    u = rng.random(n)
    tail = u < long
    span = np.log(max_len - min_len + 1)
    ln[tail] = min_len + np.minimum(np.exp(rng.random(int(tail.sum())) * span).astype(np.int64) - 1,
                                    max_len - min_len)
    ln[u >= 1 - lit] = 0
    if n > 0:
        ln[0] = 0                                          # nothing to copy from before byte 0
    return ln


def _tokens(rng, ln: np.ndarray, overlap: float, max_dist: int):
    """(tokens, bytes) for the lengths ln: literal bytes at random; a match at output position p gets a
    distance in 1..min(max_dist, p), and with probability `overlap` one below its length (a copy that
    reads its own output)."""
    assert ln.size == 0 or ln[0] == 0
    size = np.maximum(ln, 1)
    pos = np.cumsum(size) - size
    hi = np.minimum(max_dist, pos)
    ov = (rng.random(ln.size) < overlap) & (ln >= 2)
    hi = np.maximum(np.where(ov, np.minimum(hi, ln - 1), hi), 1)
    dist = rng.integers(1, hi + 1) if ln.size else hi
    lits = rng.integers(0, 256, ln.size)
    toks = np.where(ln == 0, lits, (ln << 16) | dist).astype(np.uint32)
    return toks, int(size.sum())


def stream_of_lengths(seed: int, lengths, overlap: float = 0.3, max_dist: int = 65535):
    """(tokens, bytes): a random valid stream with the given token lengths (0 = literal, the first one
    must be), for shapes made by hand."""
    return _tokens(np.random.default_rng(seed), np.asarray(lengths, dtype=np.int64), overlap, max_dist)


def stream_of_count(seed: int, n_tokens: int, lit: float = 0.4, long: float = 1e-4, overlap: float = 0.3,
                    min_len: int = 1, max_len: int = 65535, max_dist: int = 65535):
    """(tokens, bytes): a random valid stream of exactly n_tokens tokens."""
    rng = np.random.default_rng(seed)
    return _tokens(rng, _lengths(rng, n_tokens, lit, long, min_len, max_len), overlap, max_dist)


def stream_of_bytes(seed: int, nbytes: int, lit: float = 0.4, long: float = 1e-4, overlap: float = 0.3,
                    min_len: int = 1, max_len: int = 65535, max_dist: int = 65535) -> np.ndarray:
    """A random valid stream that describes exactly nbytes bytes (its last match may be cut short,
    to no less than min(min_len, what is left))."""
    rng = np.random.default_rng(seed)
    parts, total = [], 0
    while total < nbytes:
        ln = _lengths(rng, nbytes // 8 + 64, lit, long, min_len, max_len)
        if parts:
            ln[0] = rng.integers(min_len, min(32, max_len) + 1)    # only the stream's first token must be a literal
        parts.append(ln)
        total += int(np.maximum(ln, 1).sum())
    ln = np.concatenate(parts) if parts else np.zeros(0, np.int64)
    end = np.cumsum(np.maximum(ln, 1))
    k = int(np.searchsorted(end, nbytes))                  # the token that reaches nbytes
    ln = ln[: k + 1] if nbytes > 0 else ln[:0]
    if nbytes > 0 and end[k] > nbytes:
        ln[k] = nbytes - (end[k - 1] if k > 0 else 0)      # >= 1: token k starts before nbytes
        if ln[k] < min_len:                                # too short for the rules: literals instead
            ln = np.r_[ln[:k], np.zeros(int(ln[k]), np.int64)]
    toks, size = _tokens(rng, ln, overlap, max_dist)
    assert size == nbytes
    return toks
