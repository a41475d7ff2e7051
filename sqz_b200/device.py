"""Device-buffer entry points (include/sqz_gpu.h) on torch CUDA tensors.

torch is plumbing here: it owns the device memory and the stream; every kernel launched is
this library's own (libsqz_b200.so).  A "shard" is a view into a uint8 CUDA tensor that also
holds its halos: positions [first, first+n) of `buf`, with `back` readable bytes before and
`ahead` after.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .api import G1_MAX_LEN, G1_MIN_LEN, _check


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need(t: torch.Tensor, what: str, dtype, numel: int, device) -> None:
    """The library writes through raw pointers: a wrong dtype, size or device corrupts memory."""
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.device == device and t.dtype == dtype
            and t.is_contiguous() and t.numel() >= numel):
        raise ValueError(f"{what} must be a contiguous {dtype} CUDA tensor on {device} with at least {numel} elements")


def match_table(buf: torch.Tensor, first: int, n: int, back: int, ahead: int, min_len: int = G1_MIN_LEN,
                max_len: int = G1_MAX_LEN, max_dist: int = (1 << 15) - 1, out: torch.Tensor | None = None,
                seam: bool = False) -> torch.Tensor:
    """Packed table words (len << 16 | dist) for buf[first : first+n]  (squeeze.h:340-358 at every i).
    seam=True: n + 1 words, the last one the seam word a lazy parse of the shard reads (the best match at
    first + n from the same halos, 0 at the end of the input; sqz_gpu_match_seam_device)."""
    _need(buf, "buf", torch.uint8, first + n + ahead, buf.device if isinstance(buf, torch.Tensor) else None)
    if first - back < 0 or n < 0:
        raise ValueError("the look-back halo reaches before the buffer")
    words = n + 1 if seam else n
    if out is None:
        out = torch.empty(max(words, 1), dtype=torch.int32, device=buf.device)
    else:
        _need(out, "out", torch.int32, words, buf.device)
    L = _lib.load()
    rc = L.sqz_gpu_match_table_device(buf.data_ptr() + first, back, n, ahead, min_len, max_len, max_dist,
                                      out.data_ptr(), _stream())
    _check(rc, "sqz_gpu_match_table_device")
    if seam:
        rc = L.sqz_gpu_match_seam_device(buf.data_ptr() + first, back, n, ahead, min_len, max_len, max_dist,
                                         out.data_ptr(), _stream())
        _check(rc, "sqz_gpu_match_seam_device")
    return out[:words]


def exit_map(table: torch.Tensor, n: int, min_len: int = G1_MIN_LEN, max_len: int = G1_MAX_LEN,
             lazy: bool = False) -> torch.Tensor:
    """exit_map[e] = overshoot of the shard when entered at offset e (512 x int16 on the device).
    lazy=True: of the lazy parse, whose table holds n + 1 words (match_table(..., seam=True))."""
    L = _lib.load()
    _need(table, "table", torch.int32, n + 1 if lazy else n, table.device if isinstance(table, torch.Tensor) else None)
    work = torch.empty(L.sqz_gpu_parse_workspace(n), dtype=torch.uint8, device=table.device)
    out = torch.zeros(512, dtype=torch.int16, device=table.device)
    rc = L.sqz_gpu_parse_exit_map_device_ex(table.data_ptr(), n, min_len, max_len, _lib.STREAM_LAZY if lazy else 0,
                                            work.data_ptr(), out.data_ptr(), _stream())
    _check(rc, "sqz_gpu_parse_exit_map_device_ex")
    torch.cuda.current_stream().synchronize()      # `work` must outlive the kernels
    return out


def mincost_steps(table: torch.Tensor, first: int, n: int, total: int, min_len: int = G1_MIN_LEN,
                  max_len: int = G1_MAX_LEN, max_dist: int = (1 << 15) - 1) -> torch.Tensor:
    """Rewrites a shard's n table words (match_table with the same rules) in place into min-cost steps and
    returns the table; exit_map and parse (greedy, the default) of it then give the min-cost parse.  `first`
    is the shard's global offset, `total` the whole input's size: the shard starts at a multiple of 16384
    and holds whole segments or ends at `total` (shard.plan(..., align=shard.SEGMENT)).  Once per table
    (sqz_gpu_mincost_steps_device)."""
    L = _lib.load()
    _need(table, "table", torch.int32, n, table.device if isinstance(table, torch.Tensor) else None)
    rc = L.sqz_gpu_mincost_steps_device(table.data_ptr(), first, n, total, min_len, max_len, max_dist, _stream())
    _check(rc, "sqz_gpu_mincost_steps_device")
    return table


def parse(buf: torch.Tensor, first: int, table: torch.Tensor, n: int, entry: int = 0, min_len: int = G1_MIN_LEN,
          max_len: int = G1_MAX_LEN, symbols: bool = False, lazy: bool = False):
    """Greedy (squeeze.h:337,377-394; the default) or lazy parse of one shard: (tokens int32[count], overshoot).
    symbols=True: symbol words (include/sqz_gpu.h) instead of plain tokens.  lazy=True: the lazy parse,
    whose table holds n + 1 words (match_table(..., seam=True))."""
    L = _lib.load()
    dev = buf.device if isinstance(buf, torch.Tensor) else None
    _need(buf, "buf", torch.uint8, first + n, dev)
    _need(table, "table", torch.int32, n + 1 if lazy else n, dev)
    work = torch.empty(L.sqz_gpu_parse_workspace(n), dtype=torch.uint8, device=dev)
    tokens = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    result = torch.zeros(2, dtype=torch.int64, device=dev)
    flags = (_lib.STREAM_SYMBOLS if symbols else 0) | (_lib.STREAM_LAZY if lazy else 0)
    rc = L.sqz_gpu_parse_device_ex(buf.data_ptr() + first, table.data_ptr(), n, entry, min_len, max_len, flags,
                                   tokens.data_ptr(), n, work.data_ptr(), result.data_ptr(), _stream())
    _check(rc, "sqz_gpu_parse_device_ex")
    count, overshoot = (int(x) for x in result.cpu())
    return tokens[:count], overshoot
