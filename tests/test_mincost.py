"""Min-cost parse, CPU side: the min-cost walk over the oracle's match table (tests/mincost_oracle.py) against a
direct statement of the rule, the encoded sizes of its token streams (the decoders read them like any other
stream), and the checks sqz_compress makes before it touches the GPU."""
import ctypes as C
import errno
import os
import subprocess

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

from conftest import ROOT
from mincost_oracle import SEGMENT, mincost_tokens_from_table

# compressed bytes (header included) of the min-cost token stream, window 2^15, G1 rules
MINCOST_SIZES = {"laozi.txt": 9032, "confucius.txt": 26040, "csrc.cat": 32512, "x64.elf": 447288,
                 "arm64.elf": 410816, "mandrill.bmp": 776288, "mandrill.png": 637928}
# the same for the two 8 MiB samples of the synthetic corpus: offset -> (greedy, min-cost)
SYNTHETIC_SIZES = {0: (5899320, 5796320), 512 << 20: (6242192, 6127968)}

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
            227, 258]
LEN_EXTRA = [0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0]
POS_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
            4097, 6145, 8193, 12289, 16385, 24577]
POS_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]


def extra(base, bits, v):
    return bits[max(b for b in range(len(base)) if base[b] <= v)]


LEN_COST = np.array([0] * 3 + [6 + extra(LEN_BASE, LEN_EXTRA, k) for k in range(3, 258)], dtype=np.int64)


def mincost_rule(data, ln, ds, min_len):
    """The rule as stated: segments of SEGMENT positions at multiples of SEGMENT; in each, backwards with
    c(j) = 0 for j at or past its end, c(i) = min(8 + c(i + 1), 6 + len_extra + 5 + pos_extra + c(i + k) for
    min_len <= k <= len(i)), ties to the longest step; then the walk from 0 along the chosen steps."""
    ln, ds = np.asarray(ln, dtype=np.int64), np.asarray(ds, dtype=np.int64)
    n = ln.size
    step = np.ones(n, dtype=np.int64)
    for s in range(0, n, SEGMENT):
        e = min(s + SEGMENT, n)
        c = np.zeros(e - s + 258, dtype=np.int64)          # c[j - s]; zeros at and past e
        for i in range(e - 1, s - 1, -1):
            best, k_best = 8 + c[i + 1 - s], 1
            if ln[i] >= min_len:
                ks = np.arange(min_len, ln[i] + 1)
                v = LEN_COST[ks] + 5 + extra(POS_BASE, POS_EXTRA, int(ds[i])) + c[i + ks - s]
                if v.min() <= best:
                    best, k_best = v.min(), int(ks[v == v.min()].max())
            c[i - s], step[i] = best, k_best
    out, i = [], 0
    while i < n:
        out.append(int(step[i]) << 16 | int(ds[i]) if step[i] > 1 else int(data[i]))
        i += int(step[i])
    return np.array(out, dtype=np.uint32)


def check(data, ln, ds, min_len):
    want = mincost_rule(data, ln, ds, min_len)
    got, end = mincost_tokens_from_table(data, ln, ds, min_len)
    assert end == len(data)
    assert got.size == want.size and (got == want).all()
    return got


@pytest.mark.parametrize("name", sorted(MINCOST_SIZES))
def test_fixture_sizes_and_round_trip(name, inputs, oracle):
    d = inputs[name]
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    toks, end = mincost_tokens_from_table(d, ln, ds)
    assert end == d.size
    comp = sq.encode_tokens(toks, d.size, 15)
    assert len(comp) == MINCOST_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()


def test_the_walk_is_the_rule_on_text(inputs, oracle):
    """The direct statement on a whole fixture of several segments (confucius.txt: 67,735 positions)."""
    d = inputs["confucius.txt"]
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    check(d, ln, ds, 3)


def test_synthetic_sizes(oracle):
    """The two 8 MiB samples of the synthetic corpus: min-cost smaller than greedy, round trip."""
    for offset, (greedy_size, mincost_size) in SYNTHETIC_SIZES.items():
        d = corpus.synthetic(8 << 20, offset)
        ln, ds = oracle.match_table(d, 1 << 15, fast=True)
        greedy = sq.encode_tokens(oracle.tokens_from_table(d, ln, ds)[0], d.size, 15)
        mincost = sq.encode_tokens(mincost_tokens_from_table(d, ln, ds)[0], d.size, 15)
        assert (len(greedy), len(mincost)) == (greedy_size, mincost_size)
        assert sq.decompress(mincost) == d.tobytes()


@pytest.mark.parametrize("name", ["zeros4096", "pat1234x1024", "hello", "abc40", "lorem3", "empty", "one", "two",
                                  "aaa", "aaaa"])
def test_small_fixtures(name, inputs, oracle):
    d = inputs[name]
    for min_len in (3, 4):
        ln, ds = oracle.match_table(d, 1 << 15, min_len=min_len, max_len=257)
        toks = check(d, ln, ds, min_len)
        if min_len == 3:
            assert sq.decompress(sq.encode_tokens(toks, d.size, 15)) == d.tobytes()


def table(n, matches):
    """A made-up table of n positions (the walk only reads it): {position: (len, dist)}."""
    ln = np.zeros(n, dtype=np.uint16)
    ds = np.zeros(n, dtype=np.uint16)
    for i, (k, d) in matches.items():
        ln[i], ds[i] = k, d
    return ln, ds


def test_hand_made_tables():
    n = 2 * SEGMENT + 100
    data = (np.arange(n) % 251).astype(np.uint8)
    e = SEGMENT
    cases = {
        # a literal and a match of equal cost: 8 + c(1) = 8 + 11 + c(4) against 11 + c(3) = 11 + 8 + c(4)
        "literal tie": ({0: (3, 1), 1: (3, 1)}, [3 << 16 | 1, 3]),
        # three literals (24) against a match at the farthest distance bucket (6 + 5 + 13): the match
        "far tie": ({0: (3, 30000)}, [3 << 16 | 30000, 3]),
        # two lengths of equal cost: at e - 3, k = 3 and k = 4 both cost 11 + 0 (c is 0 past the segment's
        # end); the longer step wins and crosses the end
        "length tie across the end": ({e - 3: (4, 2)}, None),
        # a long match across the end, and a match at the input's last position
        "across the end": ({e - 100: (257, 7), n - 1: (3, 1), n - 5: (5, 9)}, None),
        # a length with extra bits: 11 costs one more bit than 10
        "extra bits": ({40: (11, 3), 41: (10, 3)}, None),
    }
    for name, (matches, head) in cases.items():
        ln, ds = table(n, matches)
        got = check(data, ln, ds, 3)
        if head is not None:
            assert got.tolist()[:len(head)] == head, name
    # the tie at the segment's end, spelled out: literals up to e - 3, then (4, 2) over the end
    ln, ds = table(n, {e - 3: (4, 2)})
    got = check(data, ln, ds, 3).tolist()
    assert got[e - 3] == 4 << 16 | 2 and got[e - 2] == data[e + 1]
    # inputs shorter than a segment, and a last segment of one position
    for size in (1, 2, 3, 17, SEGMENT - 1, SEGMENT, SEGMENT + 1):
        ln, ds = table(size, {i: (3, 1) for i in range(1, size - 2, 5)})
        check(data[:size], ln, ds, 3)
        check(data[:size], ln, ds, 4)


@pytest.mark.parametrize("min_len,max_len", [(3, 257), (4, 16), (3, 64)])
def test_adversarial_inputs(min_len, max_len, oracle):
    """Long zero runs across the 16 KiB segment ends, matches that grow by one per position, random data with
    short repeats."""
    rng = np.random.default_rng(min_len * 1000 + max_len)
    zeros = np.concatenate([rng.integers(0, 256, SEGMENT - 300, dtype=np.uint8), np.zeros(SEGMENT + 700, np.uint8),
                            rng.integers(0, 256, 500, dtype=np.uint8), np.zeros(1000, np.uint8),
                            rng.integers(0, 256, 200, dtype=np.uint8)])
    unit = rng.integers(0, 256, 40, dtype=np.uint8)
    growing = np.concatenate([np.concatenate([unit[:k], rng.integers(0, 256, 1, dtype=np.uint8)]) for k in range(2, 40)])
    noisy = rng.integers(0, 4, 3000, dtype=np.uint8)
    for d in (zeros, growing, noisy, np.concatenate([growing, zeros[:SEGMENT + 50], noisy])):
        ln, ds = oracle.match_table(d, 1 << 15, min_len=min_len, max_len=max_len)
        toks = check(d, ln, ds, min_len)
        if max_len <= 257:
            assert sq.decompress(sq.encode_tokens(toks, d.size, 15)) == d.tobytes()


def compress_status(**fields):
    """struct sqz's error after sqz_compress with the given fields set (on an input whose search would
    need the GPU)."""
    L = _lib.load()
    d = np.frombuffer(b"abcabcabcabc", dtype=np.uint8)
    out = np.zeros(4096, dtype=np.uint8)
    bs = _lib.Bitstream()
    bs.data = out.ctypes.data_as(_lib.u8p)
    bs.capacity = out.size
    s = _lib.State()
    L.sqz_init(C.byref(s))
    assert s.mincost == 0 and s.lazy == 0
    for k, v in fields.items():
        setattr(s, k, v)
    L.sqz_compress(C.byref(s), C.byref(bs), d.ctypes.data_as(_lib.u8p), d.size, 1 << 15)
    return s.error


@pytest.mark.parametrize("fields", [{"mincost": 2}, {"mincost": -1}, {"mincost": 1, "lazy": 1}],
                         ids=["two", "minus_one", "with_lazy"])
def test_compress_refuses_other_mincost_values(fields):
    """struct sqz's `mincost` is 0 or 1, and not 1 together with `lazy`: anything else is EINVAL before the GPU
    is asked for anything (without a device the answer would otherwise be ENODEV)."""
    assert compress_status(**fields) == errno.EINVAL


def test_python_refuses_both_parses():
    d = b"abcabcabcabc"
    with pytest.raises(ValueError):
        sq.compress(d, lazy=True, mincost=True)
    with pytest.raises(ValueError):
        sq.tokens(d, lazy=True, mincost=True)


def test_mincost_field_has_the_c_offset(tmp_path):
    """`mincost` sits where the C compiler puts it, and the fields around it did not move."""
    src = tmp_path / "o.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqz.h"\nint main(void){printf("%zu %zu %zu %zu\\n", '
                   'offsetof(struct sqz, mincost), offsetof(struct sqz, apart), offsetof(struct sqz, pos), '
                   'sizeof(struct sqz));return 0;}\n')
    exe = tmp_path / "o"
    subprocess.check_call(["gcc", "-std=c99", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = tuple(map(int, subprocess.check_output([str(exe)]).split()))
    S = _lib.State
    assert got == (S.mincost.offset, S.apart.offset, S.pos.offset, C.sizeof(S))
    assert S.pos.offset == S.len_index.offset + 259 + 69      # as with apart[64]: 5 bytes of padding before pos
