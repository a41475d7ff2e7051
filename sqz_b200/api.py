"""Host-side mirror of the reference codec interface, over the C-ABI.

The reference exposes one vtable, ``squeeze_interface squeeze``
(/root/reference/attic/map_experiment/squeeze.h:109-125): write_header,
compress, read_header, decompress.  ``compress`` / ``decompress`` below are the
same operations on whole buffers (memory-mode bitstream, header included);
``match_table`` / ``tokens`` expose the GPU half on its own
(include/sqz_gpu.h).  Everything goes through libsqz_b200.so; nothing here
computes a match on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import Bitstream, State, u8p, u16p, u32p

G1_MIN_LEN, G1_MAX_LEN = 3, 257      # squeeze.h:13-15


class SqzError(OSError):
    pass


def _check(rc: int, what: str) -> None:
    if rc != 0:
        msg = _lib.load().sqz_gpu_last_error() or b""
        raise SqzError(rc, f"{what}: {os.strerror(rc)} ({msg.decode(errors='replace')})")


def _u8(a) -> np.ndarray:
    if isinstance(a, (bytes, bytearray, memoryview)):
        a = np.frombuffer(a, dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def _rules(window: int, min_len: int, max_len: int, max_dist):
    return window, min_len, max_len, (window - 1 if max_dist is None else max_dist)


def device_count() -> int:
    return int(_lib.load().sqz_gpu_device_count())


def select_kernel(which: int) -> None:
    """0 = automatic, 1 = thread-per-position kernel, 2 = bit-sliced kernel (A/B tests)."""
    _check(_lib.load().sqz_gpu_select_kernel(int(which)), "sqz_gpu_select_kernel")


def launch_count() -> int:
    return int(_lib.load().sqz_gpu_launch_count())


# ---- GPU half, host buffers (sqz_gpu_match_table / sqz_gpu_tokens) ----------

def match_table(data, window: int = 1 << 15, min_len: int = G1_MIN_LEN, max_len: int = G1_MAX_LEN,
                max_dist: int | None = None, out=None):
    """(len[u16], dist[u16]) for every position: squeeze.h:340-358 at every i."""
    L = _lib.load()
    d = _u8(data)
    w, lo, hi, md = _rules(window, min_len, max_len, max_dist)
    if out is None:
        ln = np.empty(d.size, dtype=np.uint16)
        ds = np.empty(d.size, dtype=np.uint16)
    else:
        ln, ds = out
        for name, a in (("len", ln), ("dist", ds)):     # the library writes d.size uint16 values into each
            if not (isinstance(a, np.ndarray) and a.dtype == np.uint16 and a.flags.c_contiguous
                    and a.flags.writeable and a.size >= d.size):
                raise ValueError(f"out[{name}] must be a writeable C-contiguous uint16 array of at least {d.size} elements")
    rc = L.sqz_gpu_match_table(d.ctypes.data_as(u8p), d.size, w, lo, hi, md,
                               ln.ctypes.data_as(u16p), ds.ctypes.data_as(u16p))
    _check(rc, "sqz_gpu_match_table")
    return ln, ds


def _parse_flags(lazy: bool, mincost: bool) -> int:
    if lazy and mincost:
        raise ValueError("lazy and mincost are two different parses: choose one")
    return (_lib.STREAM_LAZY if lazy else 0) | (_lib.STREAM_MINCOST if mincost else 0)


def tokens(data, window: int = 1 << 15, min_len: int = G1_MIN_LEN, max_len: int = G1_MAX_LEN,
           max_dist: int | None = None, lazy: bool = False, mincost: bool = False) -> np.ndarray:
    """Token stream, greedy (squeeze.h:337,377-394; the default), lazy or min-cost: literal byte or
    (len << 16) | dist.  lazy=True parses with lazy matching (sqz_gpu_tokens_ex with SQZ_GPU_STREAM_LAZY):
    the tokens sq.compress(data, lazy=True) codes.  mincost=True parses by cost (SQZ_GPU_STREAM_MINCOST,
    within the bitstream's limits only): the tokens sq.compress(data, mincost=True) codes."""
    L = _lib.load()
    d = _u8(data)
    w, lo, hi, md = _rules(window, min_len, max_len, max_dist)
    out = np.empty(max(d.size, 1), dtype=np.uint32)
    n = C.c_size_t()
    rc = L.sqz_gpu_tokens_ex(d.ctypes.data_as(u8p), d.size, w, lo, hi, md, _parse_flags(lazy, mincost),
                             out.ctypes.data_as(u32p), out.size, C.byref(n))
    _check(rc, "sqz_gpu_tokens_ex")
    return out[: n.value].copy()


def tokens_multi(data, devices, window: int = 1 << 15, min_len: int = G1_MIN_LEN, max_len: int = G1_MAX_LEN,
                 max_dist: int | None = None, return_shard_counts: bool = False, lazy: bool = False,
                 mincost: bool = False, cuts=None):
    """The same token stream computed on several GPUs of this process: contiguous shards with halos, seams
    chained on the host, token arrays concatenated in shard order by copies sized by their counts.
    Identical to tokens(lazy=lazy, mincost=mincost) for every device list.  The default cut gives shards
    whose sizes differ by at most one byte (sqz_gpu_tokens_multi_ex); mincost=True cuts at multiples of
    16384 instead (shard.plan(..., align=shard.SEGMENT)), and `cuts` (len(devices) - 1 global offsets) sets
    the shard boundaries -- both go through sqz_gpu_tokens_multi_cuts."""
    flags = _parse_flags(lazy, mincost)
    L = _lib.load()
    d = _u8(data)
    w, lo, hi, md = _rules(window, min_len, max_len, max_dist)
    devs = (C.c_int * len(devices))(*[int(x) for x in devices])
    out = np.empty(max(d.size, 1), dtype=np.uint32)
    n = C.c_size_t()
    per = (C.c_size_t * len(devices))()
    if mincost or cuts is not None:
        if cuts is not None and len(cuts) != len(devices) - 1:
            raise ValueError("cuts: len(devices) - 1 offsets")
        at = None if cuts is None else (C.c_size_t * max(len(cuts), 1))(*[int(c) for c in cuts])
        rc = L.sqz_gpu_tokens_multi_cuts(devs, len(devices), at, d.ctypes.data_as(u8p), d.size, w, lo, hi, md, flags,
                                         out.ctypes.data, out.size, C.byref(n), per)
        _check(rc, "sqz_gpu_tokens_multi_cuts")
    else:
        rc = L.sqz_gpu_tokens_multi_ex(devs, len(devices), d.ctypes.data_as(u8p), d.size, w, lo, hi, md, flags,
                                       out.ctypes.data, out.size, C.byref(n), per)
        _check(rc, "sqz_gpu_tokens_multi_ex")
    t = out[: n.value].copy()
    return (t, [int(x) for x in per]) if return_shard_counts else t


def release() -> None:
    """Free the device and pinned staging buffers the library keeps between calls (sqz_gpu_release)."""
    _lib.load().sqz_gpu_release()


# ---- codec (sqz.h) ----------------------------------------------------------

def _capacity(nbytes: int) -> int:
    # worst case: every byte an escaped literal (NYT code + 9 raw bits), header, padding
    return nbytes * 10 + 4096


def compress(data, win_bits: int = 15, file_mode: bool = False, stats: dict | None = None,
             threads: int = 0, into=None, lazy: bool = False, mincost: bool = False):
    """squeeze.write_header + squeeze.compress: GPU search, host entropy stage.  Returns the bitstream as
    bytes -- or, with `into` (a C-contiguous writable uint8 array of at least capacity(len(data)) bytes, the
    caller's buffer as in the C API), a view of the part of it that was written, without a copy.
    lazy=True parses with lazy matching (struct sqz's `lazy`): a smaller stream on text and code, in the
    same format; the default greedy parse gives the reference's exact bytes.  mincost=True (struct sqz's
    `mincost`) parses by cost: smaller still on text and code, also in the same format.  Not both."""
    _parse_flags(lazy, mincost)
    L = _lib.load()
    d = _u8(data)
    if into is not None:
        if not (isinstance(into, np.ndarray) and into.dtype == np.uint8 and into.flags.c_contiguous and
                into.flags.writeable and into.size >= _capacity(d.size)):
            raise ValueError("into: a writable C-contiguous uint8 array of at least capacity(len(data)) bytes")
        out = into
    else:
        out = np.empty(_capacity(d.size), dtype=np.uint8)
    bs = Bitstream()
    sink = {"at": 0}
    if file_mode:
        # callback mode: 8 bytes at &b64 in host byte order, like fwrite(&bs->b64, 8, 1, f)
        def _out(pbs):
            word = int(pbs.contents.b64)
            out[sink["at"]: sink["at"] + 8] = np.frombuffer(word.to_bytes(8, "little"), dtype=np.uint8)
            sink["at"] += 8
            return 0
        cb = _lib.OUTPUT_FN(_out)
        bs.output = cb
    else:
        bs.data = out.ctypes.data_as(u8p)
        bs.capacity = out.size
    L.sqz_write_header(C.byref(bs), d.size, win_bits)
    _check(bs.error, "sqz_write_header")
    s = State()
    L.sqz_init(C.byref(s))
    s.coder_threads = threads
    s.lazy = 1 if lazy else 0
    s.mincost = 1 if mincost else 0
    L.sqz_compress(C.byref(s), C.byref(bs), d.ctypes.data_as(u8p), d.size, 1 << win_bits)
    _check(s.error, "sqz_compress")
    if stats is not None:
        stats.update(tokens=int(s.tokens), matches=int(s.matches),
                     search_seconds=float(s.search_seconds), entropy_seconds=float(s.entropy_seconds))
    return out[: bs.bytes].tobytes() if into is None else out[: bs.bytes]


def capacity(nbytes: int) -> int:
    """Bytes a bitstream of `nbytes` input bytes can need at most (what `compress(into=...)` asks for)."""
    return _capacity(nbytes)


def _encode(entry: str, arr, nbytes: int, win_bits: int, file_mode: bool, lib=None, threads: int = 0) -> bytes:
    L = lib or _lib.load()
    t = np.ascontiguousarray(arr, dtype=np.uint32)
    out = np.empty(_capacity(nbytes) + 64, dtype=np.uint8)
    bs = Bitstream()
    sink = {"at": 0}
    if file_mode:
        def _out(pbs):
            word = int(pbs.contents.b64)
            out[sink["at"]: sink["at"] + 8] = np.frombuffer(word.to_bytes(8, "little"), dtype=np.uint8)
            sink["at"] += 8
            return 0
        cb = _lib.OUTPUT_FN(_out)
        bs.output = cb
    else:
        bs.data = out.ctypes.data_as(u8p)
        bs.capacity = out.size
    L.sqz_write_header(C.byref(bs), nbytes, win_bits)
    _check(bs.error, "sqz_write_header")
    s = State()
    L.sqz_init(C.byref(s))
    s.coder_threads = threads
    getattr(L, entry)(C.byref(s), C.byref(bs), t.ctypes.data_as(u32p), t.size)
    _check(s.error, entry)
    return out[: bs.bytes].tobytes()


def encode_tokens(toks, nbytes: int, win_bits: int = 15, file_mode: bool = False, lib=None) -> bytes:
    """Host entropy stage alone (squeeze.h:278-315 + huffman.h + bitstream.h) on a token list."""
    return _encode("sqz_encode_tokens", toks, nbytes, win_bits, file_mode, lib)


def encode_symbols(words, nbytes: int, win_bits: int = 15, file_mode: bool = False, lib=None,
                   threads: int = 0) -> bytes:
    """The same on symbol words (include/sqz_gpu.h), the form the GPU parse emits for the coder.
    threads: 0 = automatic, 1 = one thread, 2 = model and bit packing on two threads (same bytes)."""
    return _encode("sqz_encode_symbols", words, nbytes, win_bits, file_mode, lib, threads)


def symbols_of_tokens(toks) -> np.ndarray:
    """Host statement of token -> symbol word (squeeze.h:290-315 bucket arithmetic)."""
    t = np.ascontiguousarray(toks, dtype=np.uint32)
    w = np.empty_like(t)
    _lib.load().sqz_symbols_of_tokens(t.ctypes.data_as(u32p), t.size, w.ctypes.data_as(u32p))
    return w


def read_header(comp) -> tuple[int, int]:
    L = _lib.load()
    c = _u8(comp)
    bs = Bitstream()
    bs.data = c.ctypes.data_as(u8p)
    bs.capacity = c.size
    bs.bytes = c.size
    n, wb = C.c_uint64(), C.c_uint8()
    L.sqz_read_header(C.byref(bs), C.byref(n), C.byref(wb))
    _check(bs.error, "sqz_read_header")
    return int(n.value), int(wb.value)


def decode_tokens(comp) -> np.ndarray:
    """The serial half of the decoder: the token stream of a compressed buffer, not executed."""
    L = _lib.load()
    c = _u8(comp)
    n, _ = read_header(c)
    bs = Bitstream()
    bs.data = c.ctypes.data_as(u8p)
    bs.capacity = c.size
    bs.bytes = c.size
    hdr_n, hdr_w = C.c_uint64(), C.c_uint8()
    L.sqz_read_header(C.byref(bs), C.byref(hdr_n), C.byref(hdr_w))
    toks = np.empty(max(n, 1), dtype=np.uint32)
    cnt = C.c_uint64()
    s = State()
    L.sqz_init(C.byref(s))
    L.sqz_decode_tokens(C.byref(s), C.byref(bs), n, toks.ctypes.data_as(u32p), toks.size, C.byref(cnt))
    _check(s.error, "sqz_decode_tokens")
    return toks[: cnt.value].copy()


def expand_tokens(toks, nbytes: int) -> bytes:
    """The copy phase of the decoder on the GPU (squeeze.h:533-539 for all tokens at once)."""
    L = _lib.load()
    t = np.ascontiguousarray(toks, dtype=np.uint32)
    out = np.empty(max(nbytes, 1), dtype=np.uint8)
    rc = L.sqz_gpu_expand_tokens(t.ctypes.data_as(u32p), t.size, out.ctypes.data_as(u8p), nbytes)
    _check(rc, "sqz_gpu_expand_tokens")
    return out[:nbytes].tobytes()


def decompress_gpu(comp, stats: dict | None = None) -> bytes:
    """squeeze.read_header + squeeze.decompress with the copy phase on the GPU (sqz_decompress_gpu)."""
    L = _lib.load()
    c = _u8(comp)
    bs = Bitstream()
    bs.data = c.ctypes.data_as(u8p)
    bs.capacity = c.size
    bs.bytes = c.size
    n, wb = C.c_uint64(), C.c_uint8()
    L.sqz_read_header(C.byref(bs), C.byref(n), C.byref(wb))
    _check(bs.error, "sqz_read_header")
    out = np.empty(max(n.value, 1), dtype=np.uint8)
    s = State()
    L.sqz_init(C.byref(s))
    L.sqz_decompress_gpu(C.byref(s), C.byref(bs), out.ctypes.data_as(u8p), n.value)
    _check(s.error, "sqz_decompress_gpu")
    if stats is not None:
        stats.update(tokens=int(s.tokens), entropy_seconds=float(s.entropy_seconds),
                     expand_seconds=float(s.search_seconds))
    return out[: n.value].tobytes()


def decompress(comp, into=None):
    """squeeze.read_header + squeeze.decompress (host only, never touches the GPU).  Returns bytes -- or,
    with `into` (a C-contiguous writable uint8 array of at least the stream's size, the caller's buffer as
    in the C API), a view of the part of it that was written, without a copy."""
    L = _lib.load()
    c = _u8(comp)
    n, _ = read_header(c)
    if into is not None:
        if not (isinstance(into, np.ndarray) and into.dtype == np.uint8 and into.flags.c_contiguous and
                into.flags.writeable and into.size >= max(n, 1)):
            raise ValueError("into: a writable C-contiguous uint8 array of at least read_header(comp)[0] bytes")
        out = into
    else:
        out = np.empty(max(n, 1), dtype=np.uint8)
    got = C.c_uint64()
    rc = L.sqz_decompress_buffer(c.ctypes.data_as(u8p), c.size, out.ctypes.data_as(u8p), out.size, C.byref(got))
    _check(rc, "sqz_decompress")
    return out[: got.value].tobytes() if into is None else out[: got.value]
