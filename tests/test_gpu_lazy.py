"""Lazy matching on the GPU: the streaming parse with SQZ_GPU_STREAM_LAZY against the lazy walk
(tests/lazy_oracle.py) over the oracle's match table, across chunk seams, rule sets and sizes; and
sq.compress(lazy=True), whose streams every decoder reads."""
import ctypes as C
import errno

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

from lazy_oracle import lazy_tokens_from_table
from test_lazy import LAZY_SIZES

pytestmark = pytest.mark.gpu

LAZY = 8
SYMBOLS = 1
G1 = (1 << 15, 3, 257, 32767)


def stream(d, chunk, flags, rules=G1):
    """Everything sqz_gpu_stream_next delivers, concatenated, and the number of chunks."""
    L = _lib.load()
    d = np.ascontiguousarray(d, dtype=np.uint8)
    st = C.c_void_p()
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, *rules, chunk, flags)
    assert rc == 0, L.sqz_gpu_last_error()
    got = []
    try:
        while True:
            p, n = _lib.u32p(), C.c_size_t()
            rc = L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n))
            assert rc == 0, L.sqz_gpu_last_error()
            if n.value == 0:
                break
            got.append(np.ctypeslib.as_array(p, shape=(n.value,)).copy())
    finally:
        L.sqz_gpu_stream_close(st)
    return (np.concatenate(got) if got else np.zeros(0, np.uint32)), len(got)


def oracle_tokens(oracle, d, rules=G1):
    window, mn, mx, md = rules
    ln, ds = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    toks, end = lazy_tokens_from_table(d, ln, ds, mn)
    assert end == d.size
    return toks


def mixed(inputs):
    return np.concatenate([inputs["confucius.txt"], inputs["x64.elf"][:200000], inputs["mandrill.bmp"][:50000]])


@pytest.mark.parametrize("flags", [LAZY, LAZY | SYMBOLS], ids=["tokens", "symbols"])
@pytest.mark.parametrize("chunk", [4096, 50001, 65536, 1 << 20])
def test_stream_chunk_sizes(chunk, flags, inputs, oracle):
    d = mixed(inputs)
    want = oracle_tokens(oracle, d)
    if flags & SYMBOLS:
        want = sq.symbols_of_tokens(want)
    got, _ = stream(d, chunk, flags)
    assert got.size == want.size and (got == want).all()


def seam_input(chunk, seams, seed):
    """Random bytes (no matches to speak of), and at the last position n - 1 of each of the first `seams`
    chunks a match of 11 whose next position starts a match of 40: lazy and greedy decide differently
    right at the seam, where the lazy step reads the next chunk's first table word."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, chunk * (seams + 1) + 777, dtype=np.uint8)
    for k in range(1, seams + 1):
        n = k * chunk
        unit = rng.integers(0, 256, 40, dtype=np.uint8)
        x = rng.integers(0, 256, 1, dtype=np.uint8)
        d[n - 3000: n - 2960] = unit                      # the 40 for position n
        d[n - 2000: n - 1989] = np.concatenate([x, unit[:10]])   # the 11 for position n - 1
        d[n - 1: n + 40] = np.concatenate([x, unit])
        d[n + 40] = unit[10] ^ 0xFF                       # neither match runs on
    return d


@pytest.mark.parametrize("flags", [LAZY, LAZY | SYMBOLS], ids=["tokens", "symbols"])
@pytest.mark.parametrize("chunk", [4096, 65536])
def test_seam_words(chunk, flags, oracle):
    seams = 5
    d = seam_input(chunk, seams, chunk)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    lazy, _ = lazy_tokens_from_table(d, ln, ds, 3)
    greedy, _ = oracle.tokens_from_table(d, ln, ds, 3)
    # the case is really there: the lazy parse stands on n - 1, with len(n - 1) >= 3 < len(n)
    lens = np.where(lazy > 0xFFFF, lazy >> 16, 1).astype(np.int64)
    visited = set((np.cumsum(lens) - lens).tolist())
    for k in range(1, seams + 1):
        n = k * chunk
        assert ln[n - 1] >= 3 and ln[n] > ln[n - 1] and n - 1 in visited, (k, ln[n - 1], ln[n])
    assert greedy.size != lazy.size or (greedy != lazy).any()
    want = sq.symbols_of_tokens(lazy) if flags & SYMBOLS else lazy
    got, chunks = stream(d, chunk, flags)
    assert chunks == seams + 2
    assert got.size == want.size and (got == want).all()
    got_greedy, _ = stream(d, chunk, flags & SYMBOLS)
    want_greedy = sq.symbols_of_tokens(greedy) if flags & SYMBOLS else greedy
    assert got_greedy.size == want_greedy.size and (got_greedy == want_greedy).all()


def test_large_parse_blocks(oracle):
    """One 12 MiB chunk: shards above 8 Mi positions use the 4096-position parse blocks."""
    d = corpus.synthetic(12 << 20, 3 << 20)
    want = oracle_tokens(oracle, d)
    got, chunks = stream(d, 12 << 20, LAZY)
    assert chunks == 1 and got.size == want.size and (got == want).all()
    got, chunks = stream(d, 5 << 20, LAZY | SYMBOLS)
    assert chunks == 3 and (got == sq.symbols_of_tokens(want)).all()


@pytest.mark.parametrize("kernel", [0, 1], ids=["auto", "per_position"])
@pytest.mark.parametrize("rules", [(1 << 15, 2, 254, 32767), (1 << 15, 4, 16, 32767), (1 << 15, 3, 64, 32767),
                                   (1 << 15, 3, 257, 1024), (1 << 10, 2, 31, 5)])
def test_rule_sets(rules, kernel, inputs, oracle):
    d = mixed(inputs)[:400000]
    want = oracle_tokens(oracle, d, rules)
    sq.select_kernel(kernel)
    try:
        for chunk in (50001, 1 << 20):
            got, _ = stream(d, chunk, LAZY, rules)
            assert got.size == want.size and (got == want).all(), (rules, chunk)
    finally:
        sq.select_kernel(0)


def test_flags():
    """The lazy flag combines with the others; flags nobody defined are refused."""
    L = _lib.load()
    d = corpus.synthetic(3 << 20, 0)
    want = sq.symbols_of_tokens(stream(d, 0, LAZY)[0])
    got, chunks = stream(d, 4 << 20, LAZY | SYMBOLS | 2)
    assert chunks == 2 and (got == want).all()                # 1 + 2 MiB
    st = C.c_void_p()
    for bad in (4, 16, LAZY | 4):
        assert L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, *G1, 0, bad) == errno.EINVAL


@pytest.mark.parametrize("name", sorted(LAZY_SIZES))
def test_compress(name, inputs, oracle):
    d = inputs[name]
    comp = sq.compress(d, lazy=True)
    assert comp == sq.encode_tokens(oracle_tokens(oracle, d), d.size, 15)
    assert len(comp) == LAZY_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()
    assert sq.decompress_gpu(comp) == d.tobytes()


@pytest.mark.parametrize("name", sorted(LAZY_SIZES))
def test_reference_decoder_reads_lazy_streams(name, inputs):
    from oracle import Reference
    if not Reference.available():
        pytest.skip("the reference codec is not built here (oracle/_ref)")
    d = inputs[name]
    assert Reference.get().decompress(sq.compress(d, lazy=True)) == d.tobytes()


def test_larger_input_every_coder_crew():
    """64 MiB: several chunks, the crew of coder threads; the same bytes for 1, 2 and 4 threads."""
    d = corpus.synthetic(64 << 20, 100 << 20)
    outs = [sq.compress(d, lazy=True, threads=t) for t in (1, 2, 4)]
    assert outs[0] == outs[1] == outs[2]
    assert sq.decompress(outs[0]) == d.tobytes()
    assert len(outs[0]) < len(sq.compress(d))
