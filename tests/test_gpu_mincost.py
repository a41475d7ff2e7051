"""The min-cost parse on the GPU: the token stream and the one-shot call with SQZ_GPU_STREAM_MINCOST against the
min-cost walk (tests/mincost_oracle.py) over the oracle's match table, across chunk sizes, chunk seams, segment
ends, rule sets and sizes; sq.compress(mincost=True), whose streams every decoder reads; and the entry points
that refuse the flag."""
import ctypes as C
import errno

import numpy as np
import pytest
import torch

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

from lazy_oracle import lazy_tokens_from_table
from mincost_oracle import SEGMENT, mincost_tokens_from_table
from test_gpu_lazy import mixed, stream
from test_mincost import MINCOST_SIZES

pytestmark = pytest.mark.gpu

SYMBOLS, SHORT_START, LAZY, MINCOST = 1, 2, 8, 32
G1 = (1 << 15, 3, 257, 32767)


def walk(oracle, d, rules=G1):
    window, mn, mx, md = rules
    ln, ds = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    toks, end = mincost_tokens_from_table(d, ln, ds, mn)
    assert end == d.size
    return toks


def one_shot(d, rules=G1, flags=MINCOST):
    L = _lib.load()
    d = np.ascontiguousarray(d, dtype=np.uint8)
    out = np.zeros(max(d.size, 1), np.uint32)
    n = C.c_size_t()
    rc = L.sqz_gpu_tokens_ex(d.ctypes.data_as(_lib.u8p), d.size, *rules, flags, out.ctypes.data_as(_lib.u32p),
                             out.size, C.byref(n))
    return rc, out[: n.value].copy()


def same(got, want):
    return got.size == want.size and bool((got == want).all())


@pytest.mark.parametrize("flags", [MINCOST, MINCOST | SYMBOLS], ids=["tokens", "symbols"])
@pytest.mark.parametrize("chunk", [0, 4096, 16384, 50001, 65536, 1 << 20])
def test_stream_chunk_sizes(chunk, flags, inputs, oracle):
    """Chunk sizes that are not multiples of the segment (4096, 50001) are rounded up to them."""
    d = mixed(inputs)
    want = walk(oracle, d)
    if flags & SYMBOLS:
        want = sq.symbols_of_tokens(want)
    got, chunks = stream(d, chunk, flags)
    assert same(got, want)
    if chunk:
        seg_chunk = -(-chunk // SEGMENT) * SEGMENT
        assert chunks == -(-d.size // seg_chunk)


def test_short_start_and_default_ramp(oracle):
    """An explicit chunk with its short start (quarter and half rounded up to whole segments), and the
    default ramp of 2, 4 MiB ..., on 7 MiB."""
    d = corpus.synthetic(7 << 20, 5 << 20)
    want = walk(oracle, d)
    for chunk, flags, chunks in (((4 << 20) + 5, MINCOST | SHORT_START, 3), (0, MINCOST, 3),
                                 ((1 << 20) + 12345, MINCOST | SYMBOLS, 7)):
        got, n = stream(d, chunk, flags)
        assert n == chunks and same(got, sq.symbols_of_tokens(want) if flags & SYMBOLS else want), (chunk, flags)
    rc, got = one_shot(d)
    assert rc == 0 and same(got, want)


def test_one_shot_small_inputs(inputs, oracle):
    for d in [np.frombuffer(bytes(range(k)), np.uint8) for k in range(10)] + [inputs["x64.elf"], mixed(inputs)]:
        rc, got = one_shot(d)
        assert rc == 0 and same(got, walk(oracle, d)), d.size
        assert same(sq.tokens(d, mincost=True), got)


def seam_input(segments, seed):
    """Random bytes (nothing to match) with a long match across every segment end: 300 bytes that repeat a
    block from 2 KiB earlier, starting 150 bytes before the end.  With 64 KiB chunks every fourth segment end is
    a chunk seam as well."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, segments * SEGMENT + 999, dtype=np.uint8)
    for k in range(1, segments + 1):
        e = k * SEGMENT
        block = rng.integers(0, 256, 300, dtype=np.uint8)
        d[e - 2150: e - 1850] = block
        d[e - 150: e + 150] = block
    return d


@pytest.mark.parametrize("flags", [MINCOST, MINCOST | SYMBOLS], ids=["tokens", "symbols"])
def test_seams_and_segment_ends(flags, oracle):
    segments = 12
    d = seam_input(segments, 7)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    want, _ = mincost_tokens_from_table(d, ln, ds, 3)
    greedy, _ = oracle.tokens_from_table(d, ln, ds, 3)
    # the case is really there: the parse takes a match that runs over every segment end
    lens = np.where(want > 0xFFFF, want >> 16, 1).astype(np.int64)
    starts = np.cumsum(lens) - lens
    for k in range(1, segments + 1):
        e = k * SEGMENT
        assert ln[e - 150] >= 257 - 1 and ((starts < e) & (starts + lens > e) & (lens > 1)).any(), k
    assert not same(greedy, want)
    if flags & SYMBOLS:
        want = sq.symbols_of_tokens(want)
    for chunk in (SEGMENT, 4 * SEGMENT, 1 << 20):
        got, chunks = stream(d, chunk, flags)
        assert chunks == -(-d.size // chunk) and same(got, want), chunk


@pytest.mark.parametrize("kernel", [1, 2], ids=["per_position", "bit_sliced"])
@pytest.mark.parametrize("rules", [G1, (1 << 15, 4, 16, 32767), (1 << 15, 3, 64, 32767), (1 << 15, 3, 257, 1024),
                                   (1 << 10, 3, 31, 5), (1 << 15, 5, 200, 20000)])
def test_rule_sets(rules, kernel, inputs, oracle):
    d = mixed(inputs)[:400000]
    want = walk(oracle, d, rules)
    sq.select_kernel(kernel)
    try:
        for chunk in (50001, 1 << 20):
            got, _ = stream(d, chunk, MINCOST, rules)
            assert same(got, want), (rules, chunk)
        rc, got = one_shot(d, rules)
        assert rc == 0 and same(got, want), rules
    finally:
        sq.select_kernel(0)


def test_flags_and_limits():
    """MINCOST combines with SYMBOLS and SHORT_START, not with LAZY; only within the bitstream's limits; the
    multi-device call and the device-buffer parse entry points refuse it."""
    L = _lib.load()
    d = corpus.synthetic(1 << 20, 777)
    p8 = d.ctypes.data_as(_lib.u8p)
    st = C.c_void_p()
    for flags, rules in ((MINCOST | LAZY, G1), (MINCOST, (1 << 15, 2, 257, 32767)), (MINCOST, (1 << 15, 3, 258, 32767)),
                         (MINCOST, (1 << 16, 3, 257, 32768)), (MINCOST | SYMBOLS | LAZY, G1)):
        assert L.sqz_gpu_stream_open(C.byref(st), 0, p8, d.size, *rules, 0, flags) == errno.EINVAL, (flags, rules)
        assert one_shot(d, rules, flags & ~SYMBOLS)[0] == errno.EINVAL, (flags, rules)
    out = np.zeros(d.size, np.uint32)
    n = C.c_size_t()
    devs = (C.c_int * 2)(0, 0)
    assert L.sqz_gpu_tokens_multi_ex(devs, 2, p8, d.size, *G1, MINCOST, out.ctypes.data, out.size, C.byref(n),
                                     None) == errno.EINVAL
    buf = torch.from_numpy(d).cuda()
    t = torch.zeros(d.size + 1, dtype=torch.int32, device="cuda")
    work = torch.empty(L.sqz_gpu_parse_workspace(d.size), dtype=torch.uint8, device="cuda")
    o = torch.zeros(d.size, dtype=torch.int32, device="cuda")
    r = torch.zeros(2, dtype=torch.int64, device="cuda")
    m = torch.zeros(512, dtype=torch.int16, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    for flags in (MINCOST, MINCOST | SYMBOLS):
        assert L.sqz_gpu_parse_device_ex(buf.data_ptr(), t.data_ptr(), d.size, 0, 3, 257, flags, o.data_ptr(), d.size,
                                         work.data_ptr(), r.data_ptr(), s) == errno.EINVAL
    assert L.sqz_gpu_parse_exit_map_device_ex(t.data_ptr(), d.size, 3, 257, MINCOST, work.data_ptr(), m.data_ptr(),
                                              s) == errno.EINVAL
    torch.cuda.synchronize()


def test_greedy_and_lazy_unchanged(inputs, oracle):
    """Greedy and lazy streams of the same input, before and after min-cost calls, are what their walks give."""
    d = mixed(inputs)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    greedy = oracle.tokens_from_table(d, ln, ds)[0]
    lazy = lazy_tokens_from_table(d, ln, ds)[0]
    mincost = mincost_tokens_from_table(d, ln, ds)[0]
    for _ in range(2):
        assert same(stream(d, 65536, 0)[0], greedy) and same(sq.tokens(d), greedy)
        assert same(stream(d, 65536, LAZY)[0], lazy) and same(sq.tokens(d, lazy=True), lazy)
        assert same(stream(d, 65536, MINCOST)[0], mincost) and same(sq.tokens(d, mincost=True), mincost)


def test_kernel_timing():
    """The timing aid counts one launch of the min-cost kernel per chunk, and none for a greedy stream."""
    L = _lib.load()
    d = corpus.synthetic(3 << 20, 0)
    L.sqz_gpu_set_timing(1)
    try:
        L.sqz_gpu_mincost_kernel_seconds(1, None)
        stream(d, 1 << 20, 0)
        launches = C.c_uint64()
        L.sqz_gpu_mincost_kernel_seconds(0, C.byref(launches))
        assert launches.value == 0
        stream(d, 1 << 20, MINCOST)
        seconds = L.sqz_gpu_mincost_kernel_seconds(1, C.byref(launches))
        assert launches.value == 3 and seconds > 0
    finally:
        L.sqz_gpu_set_timing(0)
        L.sqz_gpu_match_kernel_seconds(1, None)


@pytest.mark.parametrize("name", sorted(MINCOST_SIZES))
def test_compress(name, inputs, oracle):
    d = inputs[name]
    comp = sq.compress(d, mincost=True)
    assert comp == sq.encode_tokens(walk(oracle, d), d.size, 15)
    assert len(comp) == MINCOST_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()
    assert sq.decompress_gpu(comp) == d.tobytes()


def test_larger_input_every_coder_crew(oracle):
    """64 MiB of the synthetic corpus: the stream in its default ramp and in 3 MiB + 1 chunks, the one-shot call,
    and sq.compress with 1, 2 and 4 coder threads -- all equal to the walk, the same bytes, a round trip."""
    d = corpus.synthetic(64 << 20, 100 << 20)
    want = walk(oracle, d)
    got, chunks = stream(d, 0, MINCOST)
    assert chunks > 4 and same(got, want)
    got, _ = stream(d, (3 << 20) + 1, MINCOST | SYMBOLS)
    assert same(got, sq.symbols_of_tokens(want))
    del got
    rc, got = one_shot(d)
    assert rc == 0 and same(got, want)
    del got
    outs = [sq.compress(d, mincost=True, threads=t) for t in (1, 2, 4)]
    assert outs[0] == outs[1] == outs[2]
    assert outs[0] == sq.encode_tokens(want, d.size, 15)
    assert sq.decompress(outs[0]) == d.tobytes()
    assert len(outs[0]) < len(sq.compress(d, lazy=True)) < len(sq.compress(d))
