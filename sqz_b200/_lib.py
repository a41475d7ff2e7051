"""ctypes loader for the in-tree libsqz_b200.so (include/sqz.h + include/sqz_gpu.h).

Fails loudly: a missing library is an ImportError-grade problem, never a reason
to fall back to a CPU path (there is none in this package).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SQZ_B200_LIB points experiments at another build of the same ABI (tools/variants)
LIB_PATH = os.environ.get("SQZ_B200_LIB") or os.path.join(HERE, "lib", "libsqz_b200.so")

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
size_t = C.c_size_t


class Bitstream(C.Structure):
    """struct sqz_bitstream (include/sqz.h)."""


OUTPUT_FN = C.CFUNCTYPE(C.c_int, C.POINTER(Bitstream))
Bitstream._fields_ = [
    ("stream", C.c_void_p), ("data", u8p), ("capacity", C.c_uint64), ("bytes", C.c_uint64),
    ("read", C.c_uint64), ("b64", C.c_uint64), ("bits", C.c_int32), ("error", C.c_int32),
    ("output", OUTPUT_FN), ("input", OUTPUT_FN),
]


class Tree(C.Structure):
    _fields_ = [("freq", u64p), ("path", u64p), ("code", u64p),
                ("up", C.POINTER(C.c_int16)), ("lo", C.POINTER(C.c_int16)), ("hi", C.POINTER(C.c_int16)),
                ("plan", u16p), ("steps", u8p), ("bits", u8p), ("watcher", C.c_void_p), ("lut", u16p), ("lut_bits", C.c_int32),
                ("n", C.c_int32), ("next", C.c_int32), ("depth", C.c_int32), ("complete", C.c_int32),
                ("lazy", C.c_int32), ("lazy_start", C.c_int32), ("eager", C.c_int32)]


def _store(n: int):
    class Store(C.Structure):
        _fields_ = [("plan", C.c_uint16 * 32 * n),
                    ("freq", C.c_uint64 * (2 * n + 9)), ("path", C.c_uint64 * (2 * n - 1)), ("code", C.c_uint64 * n),
                    ("up", C.c_int16 * (2 * n - 1)), ("lo", C.c_int16 * (2 * n - 1)), ("hi", C.c_int16 * (2 * n - 1)),
                    ("steps", C.c_uint8 * n), ("bits", C.c_uint8 * (2 * n - 1))]
    return Store


class State(C.Structure):
    """struct sqz (include/sqz.h)."""
    _fields_ = [
        ("error", C.c_int32), ("device", C.c_int32), ("bs", C.POINTER(Bitstream)),
        ("tokens", C.c_uint64), ("matches", C.c_uint64),
        ("search_seconds", C.c_double), ("entropy_seconds", C.c_double),
        ("coder_threads", C.c_int32), ("lazy", C.c_int32),
        ("lit", Tree), ("len_index", C.c_uint8 * 259), ("mincost", C.c_int32), ("apart", C.c_uint8 * 60), ("pos", Tree),
        ("lit_store", _store(512)), ("pos_store", _store(32)),
        ("lit_lut", C.c_uint16 * 1024), ("pos_lut", C.c_uint16 * 64),
    ]


# every symbol the two public headers declare; tests/test_abi.py checks the
# list against the headers and against the loaded library
SYMBOLS = {
    # include/sqz.h
    "sqz_write_header": (None, [C.POINTER(Bitstream), C.c_uint64, C.c_uint8]),
    "sqz_read_header": (None, [C.POINTER(Bitstream), u64p, u8p]),
    "sqz_init": (None, [C.POINTER(State)]),
    "sqz_compress": (None, [C.POINTER(State), C.POINTER(Bitstream), u8p, C.c_uint64, C.c_uint32]),
    "sqz_encode_tokens": (None, [C.POINTER(State), C.POINTER(Bitstream), u32p, C.c_uint64]),
    "sqz_encode_symbols": (None, [C.POINTER(State), C.POINTER(Bitstream), u32p, C.c_uint64]),
    "sqz_encode_symbols_chunked": (None, [C.POINTER(State), C.POINTER(Bitstream), u32p, C.c_uint64, C.c_uint64]),
    "sqz_symbols_of_tokens": (None, [u32p, C.c_uint64, u32p]),
    "sqz_decode_tokens": (None, [C.POINTER(State), C.POINTER(Bitstream), C.c_uint64, u32p, C.c_uint64, u64p]),
    "sqz_decompress_gpu": (None, [C.POINTER(State), C.POINTER(Bitstream), u8p, C.c_uint64]),
    "sqz_decompress": (None, [C.POINTER(State), C.POINTER(Bitstream), u8p, C.c_uint64]),
    "sqz_compress_buffer": (C.c_int, [u8p, C.c_uint64, C.c_uint8, u8p, C.c_uint64, u64p]),
    "sqz_decompress_buffer": (C.c_int, [u8p, C.c_uint64, u8p, C.c_uint64, u64p]),
    # include/sqz_gpu.h
    "sqz_gpu_match_table": (C.c_int, [u8p, size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u16p, u16p]),
    "sqz_gpu_tokens": (C.c_int, [u8p, size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u32p, size_t,
                                 C.POINTER(size_t)]),
    "sqz_gpu_tokens_ex": (C.c_int, [u8p, size_t, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, u32p,
                                    size_t, C.POINTER(size_t)]),
    "sqz_gpu_tokens_multi": (C.c_int, [C.POINTER(C.c_int), C.c_int, u8p, size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                       C.c_uint32, C.c_void_p, size_t, C.POINTER(size_t), C.POINTER(size_t)]),
    "sqz_gpu_tokens_multi_ex": (C.c_int, [C.POINTER(C.c_int), C.c_int, u8p, size_t, C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, size_t, C.POINTER(size_t),
                                          C.POINTER(size_t)]),
    "sqz_gpu_tokens_multi_cuts": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(size_t), u8p, size_t, C.c_uint32,
                                            C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, size_t,
                                            C.POINTER(size_t), C.POINTER(size_t)]),
    "sqz_gpu_stream_open": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, u8p, size_t, C.c_uint32, C.c_uint32,
                                      C.c_uint32, C.c_uint32, size_t, C.c_uint32]),
    "sqz_gpu_stream_next": (C.c_int, [C.c_void_p, C.POINTER(u32p), C.POINTER(size_t)]),
    "sqz_gpu_stream_close": (None, [C.c_void_p]),
    "sqz_gpu_match_workspace": (size_t, [size_t]),
    "sqz_gpu_match_table_device_ws": (C.c_int, [C.c_void_p, size_t, size_t, size_t, C.c_uint32, C.c_uint32,
                                                C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_match_table_device": (C.c_int, [C.c_void_p, size_t, size_t, size_t, C.c_uint32, C.c_uint32,
                                             C.c_uint32, C.c_void_p, C.c_void_p]),
    "sqz_gpu_match_seam_device": (C.c_int, [C.c_void_p, size_t, size_t, size_t, C.c_uint32, C.c_uint32,
                                            C.c_uint32, C.c_void_p, C.c_void_p]),
    "sqz_gpu_unpack_table_device": (C.c_int, [C.c_void_p, size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_parse_workspace": (size_t, [size_t]),
    "sqz_gpu_parse_device": (C.c_int, [C.c_void_p, C.c_void_p, size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                       C.c_void_p, size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_parse_symbols_device": (C.c_int, [C.c_void_p, C.c_void_p, size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                               C.c_void_p, size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_parse_exit_map_device": (C.c_int, [C.c_void_p, size_t, C.c_uint32, C.c_uint32, C.c_void_p,
                                                C.c_void_p, C.c_void_p]),
    "sqz_gpu_parse_device_ex": (C.c_int, [C.c_void_p, C.c_void_p, size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_void_p, size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_parse_exit_map_device_ex": (C.c_int, [C.c_void_p, size_t, C.c_uint32, C.c_uint32, C.c_uint32,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "sqz_gpu_mincost_steps_device": (C.c_int, [C.c_void_p, size_t, size_t, size_t, C.c_uint32, C.c_uint32,
                                               C.c_uint32, C.c_void_p]),
    "sqz_gpu_device_alloc": (C.c_int, [C.POINTER(C.c_void_p), size_t]),
    "sqz_gpu_device_free": (None, [C.c_void_p]),
    "sqz_gpu_ipc_export": (C.c_int, [C.c_void_p, C.c_char_p]),
    "sqz_gpu_ipc_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "sqz_gpu_ipc_close": (C.c_int, [C.c_void_p]),
    "sqz_gpu_put_tokens": (C.c_int, [C.c_void_p, size_t, C.c_void_p, size_t, C.c_void_p]),
    "sqz_gpu_expand_tokens": (C.c_int, [u32p, size_t, u8p, size_t]),
    "sqz_gpu_expand_workspace": (size_t, [size_t, size_t]),
    "sqz_gpu_expand_tokens_device": (C.c_int, [C.c_void_p, size_t, C.c_void_p, size_t, C.c_void_p, C.c_void_p]),
    "sqz_gpu_abi_version": (C.c_int, []),
    "sqz_gpu_device_count": (C.c_int, []),
    "sqz_gpu_last_error": (C.c_char_p, []),
    "sqz_gpu_host_alloc": (C.c_void_p, [size_t]),
    "sqz_gpu_host_free": (None, [C.c_void_p]),
    "sqz_gpu_release": (None, []),
    "sqz_gpu_select_kernel": (C.c_int, [C.c_int]),
    "sqz_gpu_debug_tile_cycles": (None, [C.c_void_p]),
    "sqz_gpu_launch_count": (C.c_uint64, []),
    "sqz_gpu_set_timing": (None, [C.c_int]),
    "sqz_gpu_match_kernel_seconds": (C.c_double, [C.c_int, u64p]),
    "sqz_gpu_mincost_kernel_seconds": (C.c_double, [C.c_int, u64p]),
}

# flag bits of include/sqz_gpu.h (SQZ_GPU_STREAM_*)
STREAM_SYMBOLS = 1
STREAM_LAZY = 8
STREAM_MINCOST = 32

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m sqz_b200.build` "
                "(or __graft_entry__.build()). sqz_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError here = ABI drift, by design
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
