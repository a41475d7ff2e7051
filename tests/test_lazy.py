"""Lazy matching, CPU side: the lazy walk over the oracle's match table (tests/lazy_oracle.py) against a
direct statement of the rule, and the encoded sizes of its token streams (the decoders read them like any other stream)."""
import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import corpus

from lazy_oracle import lazy_tokens_from_table

# compressed bytes (header included) of the lazy token stream, window 2^15, G1 rules
LAZY_SIZES = {"laozi.txt": 9160, "confucius.txt": 26424, "csrc.cat": 33552, "x64.elf": 453400,
              "arm64.elf": 417464, "mandrill.bmp": 777704, "mandrill.png": 637928}


def lazy_rule(data, ln, ds, min_len):
    """The rule as stated: at i, len(i) >= min_len and len(i+1) > len(i) (len(bytes) = 0) emits the literal
    data[i] and moves on by 1; otherwise the greedy step."""
    ln, ds = ln.tolist(), ds.tolist()
    n = len(ln)
    out, i = [], 0
    while i < n:
        here = ln[i]
        after = ln[i + 1] if i + 1 < n else 0
        if here >= min_len and after <= here:
            out.append(here << 16 | ds[i])
            i += here
        else:
            out.append(int(data[i]))
            i += 1
    return np.array(out, dtype=np.uint32)


def check(oracle, data, ln, ds, min_len):
    want = lazy_rule(data, ln, ds, min_len)
    got, end = lazy_tokens_from_table(data, ln, ds, min_len)
    assert end == len(data)
    assert got.size == want.size and (got == want).all()
    return got


@pytest.mark.parametrize("name", sorted(LAZY_SIZES))
def test_fixture_sizes_and_round_trip(name, inputs, oracle):
    d = inputs[name]
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    toks = check(oracle, d, ln, ds, 3)
    greedy = oracle.tokens_from_table(d, ln, ds)[0]
    comp = sq.encode_tokens(toks, d.size, 15)
    assert len(comp) == LAZY_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()
    assert toks.size != greedy.size or (toks != greedy).any()


@pytest.mark.parametrize("name", ["zeros4096", "pat1234x1024", "hello", "abc40", "lorem3", "empty", "one", "two",
                                  "aaa", "aaaa"])
def test_small_fixtures(name, inputs, oracle):
    d = inputs[name]
    for min_len in (2, 3, 4):
        ln, ds = oracle.match_table(d, 1 << 15, min_len=min_len, max_len=257)
        toks = check(oracle, d, ln, ds, min_len)
        if min_len == 3:
            assert sq.decompress(sq.encode_tokens(toks, d.size, 15)) == d.tobytes()


def test_hand_made_tables(oracle):
    """Made-up tables (the walk only reads them): a longer match at the very last position, chains of
    growing lengths, a match longer than min_len followed by a shorter one."""
    data = np.arange(12, dtype=np.uint8)
    cases = [
        ([0, 0, 0, 0, 0, 0, 0, 0, 2, 3, 0, 0], 2),              # literal at 8, then the 3 at 9 ends the input
        ([0, 3, 4, 5, 6, 0, 0, 0, 0, 0, 0, 0], 3),              # a chain of literals, then the 6
        ([0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 2, 2], 2),              # the last position: len(bytes) = 0
        ([0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1], 1),              # a match at the last position
        ([0, 5, 4, 3, 0, 0, 0, 0, 0, 0, 0, 0], 3),              # shrinking: greedy
        ([0, 4, 4, 4, 4, 0, 0, 0, 0, 0, 0, 0], 4),              # equal: greedy
        ([0, 2, 3, 2, 4, 0, 0, 0, 0, 0, 0, 0], 2),
        ([0, 2, 3, 2, 4, 0, 0, 0, 0, 0, 0, 0], 3),
        ([0, 2, 3, 2, 4, 0, 0, 0, 0, 0, 0, 0], 4),
    ]
    for lens, min_len in cases:
        ln = np.array(lens, dtype=np.uint16)
        ds = np.where(ln > 0, 1, 0).astype(np.uint16)
        check(oracle, data, ln, ds, min_len)
    # the lazy decision changes the stream: literal 1, 2, 3, then the 6 at 4
    ln = np.array(cases[1][0], dtype=np.uint16)
    got = check(oracle, data, ln, np.where(ln > 0, 1, 0).astype(np.uint16), 3)
    assert got.tolist()[:6] == [0, 1, 2, 3, 6 << 16 | 1, 10]


@pytest.mark.parametrize("min_len,max_len", [(2, 254), (3, 257), (4, 16)])
def test_adversarial_inputs(min_len, max_len, oracle):
    """Runs whose matches grow by one per position, a longer match right at the end, random data with
    short repeats."""
    rng = np.random.default_rng(min_len)
    unit = rng.integers(0, 256, 40, dtype=np.uint8)
    growing = np.concatenate([np.concatenate([unit[:k], rng.integers(0, 256, 1, dtype=np.uint8)]) for k in range(2, 40)])
    tail = np.concatenate([unit, rng.integers(0, 256, 30, dtype=np.uint8), unit[1:8], unit[:9]])
    noisy = rng.integers(0, 4, 3000, dtype=np.uint8)
    for d in (growing, tail, noisy, np.concatenate([growing, tail])):
        ln, ds = oracle.match_table(d, 1 << 15, min_len=min_len, max_len=max_len)
        check(oracle, d, ln, ds, min_len)


@pytest.mark.parametrize("lazy", [2, -1])
def test_compress_refuses_other_lazy_values(lazy):
    """struct sqz's `lazy` is 0 or 1; anything else is EINVAL before the GPU is asked for anything."""
    import ctypes as C
    import errno
    from sqz_b200 import _lib
    L = _lib.load()
    d = np.frombuffer(b"abcabcabcabc", dtype=np.uint8)
    out = np.zeros(4096, dtype=np.uint8)
    bs = _lib.Bitstream()
    bs.data = out.ctypes.data_as(_lib.u8p)
    bs.capacity = out.size
    s = _lib.State()
    L.sqz_init(C.byref(s))
    assert s.lazy == 0
    s.lazy = lazy
    L.sqz_compress(C.byref(s), C.byref(bs), d.ctypes.data_as(_lib.u8p), d.size, 1 << 15)
    assert s.error == errno.EINVAL


def test_synthetic_sizes(oracle):
    """The two 8 MiB samples of the synthetic corpus: lazy smaller than greedy, round trip."""
    for offset, greedy_size, lazy_size in ((0, 5899320, 5872024), (512 << 20, 6242192, 6152528)):
        d = corpus.synthetic(8 << 20, offset)
        ln, ds = oracle.match_table(d, 1 << 15, fast=True)
        greedy = sq.encode_tokens(oracle.tokens_from_table(d, ln, ds)[0], d.size, 15)
        lazy = sq.encode_tokens(lazy_tokens_from_table(d, ln, ds)[0], d.size, 15)
        assert (len(greedy), len(lazy)) == (greedy_size, lazy_size)
        assert sq.decompress(lazy) == d.tobytes()
