"""The token stream (sqz_gpu_stream_*) where its chunk hand-offs are hardest: chunks shorter than a match, every
overshoot a seam can pass to the next chunk, rule sets off G1 (the thread-per-position kernel, distances past
32 KiB), the default ramp and the short start at their boundaries, explicit chunks at and far past the input, and
the stream's lifecycle; and the output contract of the one-shot call sqz_gpu_tokens_ex.

References: the oracle's match table walked by the greedy, lazy or min-cost rule; for inputs above 8 MiB the
one-shot call, which the full-size tests pin to the oracle.  Every stream is drained by `drain`, which records the
count of every sqz_gpu_stream_next call, and checked by `check` against the chunk schedule of include/sqz_gpu.h
(`schedule`): a count of 0 only at the end, the end repeated, and every delivery exactly the tokens that start in
the chunks read since the previous one."""
import ctypes as C
import errno
import threading

import numpy as np
import pytest
import torch

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

from lazy_oracle import lazy_tokens_from_table
from mincost_oracle import SEGMENT, mincost_tokens_from_table

pytestmark = pytest.mark.gpu

SYMBOLS, SHORT_START, LAZY, MINCOST = 1, 2, 8, 32
MiB = 1 << 20
SIZE_MAX = 2 ** 64 - 1
G1 = (1 << 15, 3, 257, 32767)
LONG = (1 << 15, 3, 512, 32767)          # matches longer than symbol words can carry: plain tokens only


def walk(oracle, d, rules=G1, flags=0):
    """The reference tokens of the parse `flags` selects: the oracle's table walked by that rule."""
    window, mn, mx, md = rules
    ln, ds = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    rule = lazy_tokens_from_table if flags & LAZY else mincost_tokens_from_table if flags & MINCOST else \
        oracle.tokens_from_table
    toks, end = rule(d, ln, ds, mn)
    assert end == d.size
    return toks


def lengths(toks):
    return np.where(toks > 0xFFFF, toks >> 16, 1).astype(np.int64)


def schedule(nbytes, chunk, flags):
    """The ends of the chunks a stream of `nbytes` is cut into (include/sqz_gpu.h): chunk_bytes = 0 gives 2, 4,
    8, 16, then 32 MiB (one chunk when the input is at most 2 MiB); SHORT_START with chunk_bytes >= 4 MiB starts
    with a quarter and a half of it; MINCOST rounds an explicit size and its quarter up to whole segments."""
    def whole(b):
        return -(-b // SEGMENT) * SEGMENT if flags & MINCOST and b <= SIZE_MAX - SEGMENT else b
    chunk = whole(chunk)
    size = chunk or max(min(nbytes, 32 * MiB), 1)
    ramp = 2 * MiB if chunk == 0 and size > 2 * MiB else 0
    if flags & SHORT_START and chunk >= 4 * MiB:
        ramp = whole(chunk // 4)
    ends, at = [], 0
    while at < nbytes:
        n = min(size, nbytes - at)
        if ramp:
            n = min(n, ramp)
            ramp = 0 if 2 * ramp >= size else 2 * ramp
        at += n
        ends.append(at)
    return ends


def open_stream(d, chunk, flags, rules=G1, device=0):
    L = _lib.load()
    st = C.c_void_p()
    rc = L.sqz_gpu_stream_open(C.byref(st), device, d.ctypes.data_as(_lib.u8p), d.size, *rules, chunk, flags)
    assert rc == 0, L.sqz_gpu_last_error()
    return st


def next_words(st):
    """One sqz_gpu_stream_next call: its words, copied."""
    L = _lib.load()
    p, n = _lib.u32p(), C.c_size_t()
    rc = L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n))
    assert rc == 0, L.sqz_gpu_last_error()
    return np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, np.uint32)


def drain_open(st):
    """Calls sqz_gpu_stream_next until it returns a count of 0, as every consumer does, then twice more (the end
    repeats: rc 0, count 0), and closes the stream.  The words and the count of every call up to the first 0."""
    pieces, counts = [], []
    try:
        while True:
            w = next_words(st)
            counts.append(w.size)
            if w.size == 0:
                break
            pieces.append(w)
        after = [next_words(st).size for _ in range(2)]
    finally:
        _lib.load().sqz_gpu_stream_close(st)
    assert after == [0, 0], f"the stream went on after a count of 0: {after}"
    return (np.concatenate(pieces) if pieces else np.zeros(0, np.uint32)), counts


def drain(d, chunk, flags, rules=G1, device=0):
    return drain_open(open_stream(d, chunk, flags, rules, device))


def check(d, chunk, flags, want, rules=G1, device=0, got=None):
    """Drains the stream (or takes `got`, a drain's result) and compares it with the plain tokens `want`.  Returns
    the number of tokens that start in every chunk of the schedule (0: the chunk lies inside one token)."""
    got, counts = drain(d, chunk, flags, rules, device) if got is None else got
    lens = lengths(want)
    ends = schedule(d.size, chunk, flags)
    assert sum(counts) == want.size, \
        f"the stream ended after {sum(counts)} of {want.size} tokens, {int(lens[:sum(counts)].sum())} of {d.size} bytes"
    words = sq.symbols_of_tokens(want) if flags & SYMBOLS else want
    assert (got == words).all(), int(np.argmax(got != words))
    # every delivery ends at a chunk end b of the schedule, its tokens running past b by less than max_len ...
    done = np.cumsum(lens)[np.cumsum(counts[:-1], dtype=np.int64) - 1]
    if len(ends):
        b = np.asarray(ends, np.int64)[np.searchsorted(ends, done, side="right") - 1]
        assert (done >= b).all() and (done - b < rules[2]).all()
    # ... and holds exactly the tokens that start in the chunks since the previous delivery
    starts = np.cumsum(lens) - lens
    per_chunk = np.diff(np.searchsorted(starts, [0] + ends))
    assert counts[:-1] == [int(c) for c in per_chunk if c]
    return per_chunk


# ---- 1. chunks shorter than a match --------------------------------------------------------------------------

def swallowing_input(nbytes, seed):
    """Random stretches between byte runs and short-period repeats of 200-3000 bytes: max_len matches at dist 1-4,
    long enough to swallow whole chunks shorter than max_len.  A chunk of max_len - 1 fits inside a token only when
    the token starts one byte before the chunk: runs planted at 1018, 2046 and 3064 start such matches at
    4 x 255 - 1, 8 x 256 - 1 and 6 x 511 - 1."""
    rng = np.random.default_rng(seed)
    parts, size = [], 0
    while size < nbytes:
        parts.append(rng.integers(0, 256, int(rng.integers(1, 600)), dtype=np.uint8))
        unit = rng.integers(0, 256, int(rng.integers(1, 5)), dtype=np.uint8)
        parts.append(np.tile(unit, int(rng.integers(200, 3000)) // unit.size + 1))
        size += parts[-2].size + parts[-1].size
    d = np.concatenate(parts)[:nbytes]
    d[:4000] = rng.integers(0, 256, 4000, dtype=np.uint8)
    for run in (1018, 2046, 3064):
        d[run: run + 600] = d[run - 1] ^ 0xFF
    return d


@pytest.fixture(scope="module")
def swallowing(oracle):
    """(input, {(rules, parse flags): reference tokens}) for the one-byte-per-chunk sizes and for the rest."""
    cases = {}
    for small, nbytes in ((True, 20000), (False, 200000)):
        d = swallowing_input(nbytes, nbytes)
        cases[small] = d, {(r, f): walk(oracle, d, r, f) for r in (G1, LONG) for f in (0, LAZY)}
    return cases


@pytest.mark.parametrize("parse", [0, LAZY, SYMBOLS, LAZY | SYMBOLS, (LONG, 0), (LONG, LAZY)],
                         ids=["greedy", "lazy", "greedy-symbols", "lazy-symbols", "greedy-512", "lazy-512"])
@pytest.mark.parametrize("chunk", [1, 2, 3, 7, 64, 255, 256, 257, 258, 511, 512, 513])
def test_chunks_shorter_than_a_match(chunk, parse, swallowing):
    rules, flags = parse if isinstance(parse, tuple) else (G1, parse)
    d, refs = swallowing[chunk <= 7]
    per_chunk = check(d, chunk, flags, refs[(rules, flags & LAZY)], rules)
    # the case is really there: some chunk holds no token start, exactly when it is shorter than max_len
    assert (per_chunk == 0).any() == (chunk < rules[2]), (chunk, rules)


# ---- 2. every seam overshoot ---------------------------------------------------------------------------------

def overshoot_input(chunk, max_len, seed):
    """Random bytes with a block of max_len bytes repeated so that the match starting at seam k - max_len +
    (k mod max_len) ends k mod max_len bytes into the next chunk, for the seams k = 1 .. max_len."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, (max_len + 1) * chunk + 777, dtype=np.uint8)
    for k in range(1, max_len + 1):
        b = k * chunk
        at = b + k % max_len - max_len
        src = b - 1500 - max_len
        d[src: src + max_len] = d[at: at + max_len]
        d[src - 1] = d[at - 1] ^ 0xFF           # the match starts where it is planted, not a byte before
    return d


def seam_overshoots(toks, ends):
    """For every chunk end b: how far the token that covers position b - 1 runs past b."""
    stops = np.cumsum(lengths(toks))
    return stops[np.searchsorted(stops, ends, side="left")] - np.asarray(ends)


@pytest.mark.parametrize("rules, flags, chunk",
                         [(G1, f, 4096) for f in (0, LAZY, SYMBOLS, LAZY | SYMBOLS)] +
                         [(G1, f, SEGMENT) for f in (MINCOST, MINCOST | SYMBOLS)] +
                         [(LONG, f, 4096) for f in (0, LAZY)],
                         ids=["greedy", "lazy", "greedy-symbols", "lazy-symbols", "mincost", "mincost-symbols",
                              "greedy-512", "lazy-512"])
def test_every_seam_overshoot(rules, flags, chunk, oracle):
    """The entry of every chunk is the previous chunk's overshoot, read from device memory.  Greedy and lazy see
    every overshoot 0 .. max_len - 1.  A min-cost step crosses a segment end only on a cost tie with the step that
    ends there, and at G1 the longest lengths cost the same from 131 on: its seams see every overshoot up to
    257 - 131 = 126."""
    mx = rules[2]
    d = overshoot_input(chunk, mx, mx + chunk)
    want = walk(oracle, d, rules, flags)
    seen = set(seam_overshoots(want, schedule(d.size, chunk, flags)[:-1]).tolist())
    assert seen >= set(range(mx if not flags & MINCOST else 127)), sorted(set(range(mx)) - seen)[:20]
    check(d, chunk, flags, want, rules)


# ---- 3. rule sets off G1 -------------------------------------------------------------------------------------

FAR = (1 << 16, 2, 254, 65535)
OFF_G1 = [(1 << 15, 4, 16, 32767), (1 << 15, 3, 20, 32767), FAR, (1 << 15, 1, 8, 300)]


@pytest.fixture(scope="module")
def off_g1_input(inputs):
    """Text, code and an image, then 16 KiB of random bytes and the text again: matches 45-50 KiB back."""
    text = inputs["confucius.txt"][:30000]
    noise = np.random.default_rng(5).integers(0, 256, 16384, dtype=np.uint8)
    return np.concatenate([text, inputs["x64.elf"][:60000], inputs["mandrill.bmp"][:20000], noise, text])


@pytest.mark.parametrize("rules", OFF_G1, ids=["4-16", "3-20", "2-254-64K", "1-8-300"])
def test_rules_off_g1(rules, off_g1_input, oracle):
    """(4, 16) and (3, 20) run on the thread-per-position kernel; (2, 254, 65535) reaches past 32 KiB.  Every
    parse and word form the rules allow, at chunks of 257, 4097 and 64 KiB; the others are refused."""
    L = _lib.load()
    d = off_g1_input
    _, mn, mx, md = rules
    bitstream = mn >= 3 and mx <= 257 and md <= 32767
    refs = {f: walk(oracle, d, rules, f) for f in ((0, LAZY, MINCOST) if bitstream else (0, LAZY))}
    if rules == FAR:
        assert (refs[0] & 0xFFFF)[refs[0] > 0xFFFF].max() > 32767
    for parse in (0, LAZY, MINCOST):
        for flags in (parse, parse | SYMBOLS):
            if not bitstream and flags & (SYMBOLS | MINCOST):
                st = C.c_void_p()
                assert L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, *rules, 4097,
                                             flags) == errno.EINVAL, flags
                continue
            for chunk in (257, 4097, 65536):
                check(d, chunk, flags, refs[parse], rules)


# ---- 4. the schedule ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("nbytes, chunks", [(2 * MiB - 1, 1), (2 * MiB, 1), (2 * MiB + 1, 2), (6 * MiB + 1, 3),
                                            (30 * MiB + 1, 5), (62 * MiB + 1, 6)])
def test_default_ramp(nbytes, chunks, oracle):
    """chunk_bytes = 0: one chunk up to 2 MiB, then 2, 4, 8, 16 MiB and 32 MiB chunks.  The larger inputs take the
    one-shot call as reference, and the lazy parse's symbol words."""
    d = corpus.synthetic(nbytes, nbytes)
    assert len(schedule(nbytes, 0, 0)) == chunks
    if nbytes <= 8 * MiB:
        per_chunk = check(d, 0, 0, walk(oracle, d))
    else:
        per_chunk = check(d, 0, LAZY | SYMBOLS, sq.tokens(d, lazy=True))
    assert len(per_chunk) == chunks


def test_short_start(oracle):
    """SQZ_GPU_STREAM_SHORT_START starts with a quarter and a half of an explicit chunk of at least 4 MiB, 4 MiB - 1
    has no short start, and MINCOST rounds 4 MiB - 1 up to 4 MiB first.  MINCOST rounds explicit sizes up to
    whole segments."""
    d = corpus.synthetic(7 * MiB + 3, 11)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    greedy = oracle.tokens_from_table(d, ln, ds)[0]
    mincost = mincost_tokens_from_table(d, ln, ds)[0]
    for chunk, flags, chunks in ((4 * MiB - 1, SHORT_START, 2), (4 * MiB, SHORT_START, 4),
                                 (4 * MiB - 1, SHORT_START | MINCOST, 4), (4 * MiB, SHORT_START | MINCOST | SYMBOLS, 4)):
        ends = schedule(d.size, chunk, flags)
        assert len(ends) == chunks and (chunks == 2 or ends[:2] == [MiB, 3 * MiB]), (chunk, flags)
        assert len(check(d, chunk, flags, mincost if flags & MINCOST else greedy)) == chunks
    small = d[:300000]
    want = walk(oracle, small, G1, MINCOST)
    for chunk, rounded in ((1, SEGMENT), (16383, SEGMENT), (16385, 2 * SEGMENT), (40000, 3 * SEGMENT)):
        assert schedule(small.size, chunk, MINCOST)[:2] == [rounded, 2 * rounded]
        assert len(check(small, chunk, MINCOST, want)) == -(-small.size // rounded)


# ---- 5. explicit sizes at and past the input, and the stream's lifecycle ------------------------------------

@pytest.fixture(scope="module")
def beyond(oracle):
    return {n: (d, walk(oracle, d), walk(oracle, d, G1, MINCOST))
            for n, d in ((1000, corpus.synthetic(1000, 3)), (3 * MiB, corpus.synthetic(3 * MiB, 3)))}


@pytest.mark.parametrize("flags", [0, MINCOST], ids=["greedy", "mincost"])
@pytest.mark.parametrize("nbytes", [1000, 3 * MiB])
@pytest.mark.parametrize("chunk", ["bytes", "bytes+1", "1GiB", "2^42", "SIZE_MAX-1", "SIZE_MAX"])
def test_chunk_past_the_input(chunk, nbytes, flags, beyond):
    """One chunk however far the size is past the input, and staging sized by the input: it is set aside when the
    stream opens, so the device memory it takes is measured around the open."""
    d, greedy, mincost = beyond[nbytes]
    size = {"bytes": nbytes, "bytes+1": nbytes + 1, "1GiB": 1 << 30, "2^42": 1 << 42, "SIZE_MAX-1": SIZE_MAX - 1,
            "SIZE_MAX": SIZE_MAX}[chunk]
    sq.release()
    torch.cuda.init()
    free = torch.cuda.mem_get_info(0)[0]
    st = open_stream(d, size, flags)
    taken = free - torch.cuda.mem_get_info(0)[0]
    per_chunk = check(d, size, flags, mincost if flags & MINCOST else greedy, got=drain_open(st))
    assert len(per_chunk) == 1
    assert taken < (1 << 30), f"{taken / 2 ** 30:.1f} GiB of device memory for {nbytes} bytes"


def test_empty_input():
    for flags in (0, LAZY | SYMBOLS, MINCOST, SHORT_START):
        got, counts = drain(np.zeros(0, np.uint8), 4096, flags)
        assert got.size == 0 and counts == [0]
        got, counts = drain(np.zeros(0, np.uint8), 0, flags)
        assert got.size == 0 and counts == [0]


@pytest.fixture(scope="module")
def lifecycle_input(inputs, oracle):
    d = np.concatenate([inputs["confucius.txt"], inputs["x64.elf"][:100000]])
    return d, walk(oracle, d), walk(oracle, d, G1, LAZY)


def test_devices(lifecycle_input):
    """device = -1 is the calling thread's current device; an explicit device leaves the current one as it was."""
    d, greedy, lazy = lifecycle_input
    check(d, 4096, LAZY, lazy, device=-1)
    if sq.device_count() < 2:
        return
    torch.cuda.set_device(0)
    check(d, 4096, SYMBOLS, greedy, device=1)
    assert torch.cuda.current_device() == 0
    torch.cuda.set_device(1)
    try:
        check(d, 65536, 0, greedy, device=-1)
        assert torch.cuda.current_device() == 1
    finally:
        torch.cuda.set_device(0)


def test_close_early(lifecycle_input):
    """A stream closed right after it opened, and one closed after its first delivery, leave nothing behind that
    changes the next stream of the same shape."""
    d, greedy, lazy = lifecycle_input
    for chunk, flags, want in ((4096, 0, greedy), (257, LAZY | SYMBOLS, lazy), (0, 0, greedy)):
        _lib.load().sqz_gpu_stream_close(open_stream(d, chunk, flags))
        check(d, chunk, flags, want)
        st = open_stream(d, chunk, flags)
        assert next_words(st).size > 0
        _lib.load().sqz_gpu_stream_close(st)
        check(d, chunk, flags, want)


def test_two_streams(lifecycle_input, oracle):
    """Two streams with different rules and flags drained alternately on one thread, and two drained at once from
    two threads (ctypes lets go of the GIL during the calls): each is its own reference."""
    d, greedy, lazy = lifecycle_input
    rules = (1 << 15, 4, 16, 32767)
    other = walk(oracle, d, rules, MINCOST)
    a, b = open_stream(d, 4096, LAZY | SYMBOLS), open_stream(d, 1000, MINCOST, rules)
    got = {a.value: [], b.value: []}
    live = [a, b]
    while live:
        for st in list(live):
            w = next_words(st)
            got[st.value].append(w)
            if w.size == 0:
                _lib.load().sqz_gpu_stream_close(st)
                live.remove(st)
    assert (np.concatenate(got[a.value]) == sq.symbols_of_tokens(lazy)).all()
    assert np.concatenate(got[b.value]).size == other.size and (np.concatenate(got[b.value]) == other).all()
    jobs = [(4096, LAZY, G1, lazy), (777, MINCOST | SYMBOLS, rules, other)]
    results = [None, None]

    def run(k):
        chunk, flags, r, _ = jobs[k]
        results[k] = drain(d, chunk, flags, r)

    threads = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for (chunk, flags, r, want), res in zip(jobs, results):
        assert res is not None, "a drain thread failed"
        check(d, chunk, flags, want, r, got=res)


# ---- 6. the one-shot call's output contract -----------------------------------------------------------------

def test_one_shot_capacity():
    """sqz_gpu_tokens_ex on a little more than two of its 128 MiB chunks: with any tokens_cap below the count E2BIG,
    the exact count, the first tokens_cap tokens and nothing written past them; with tokens_out = NULL and cap 0
    a count query."""
    L = _lib.load()
    d = corpus.synthetic(256 * MiB + 12345, 1 << 30)
    p8 = d.ctypes.data_as(_lib.u8p)
    full = np.zeros(d.size, np.uint32)
    n = C.c_size_t()
    assert L.sqz_gpu_tokens_ex(p8, d.size, *G1, 0, full.ctypes.data_as(_lib.u32p), full.size, C.byref(n)) == 0
    count = n.value
    full = full[:count]
    lens = lengths(full)
    first, second = np.searchsorted(np.cumsum(lens) - lens, [128 * MiB, 256 * MiB]).tolist()
    del lens
    assert 0 < first < second < count
    canary = np.uint32(0xA5C3E1F7)
    for cap in (0, 1, first, (first + second) // 2, count - 1, count):
        out = np.full(cap + 64, canary, np.uint32)
        n.value = 12345
        rc = L.sqz_gpu_tokens_ex(p8, d.size, *G1, 0, out.ctypes.data_as(_lib.u32p), cap, C.byref(n))
        assert rc == (0 if cap == count else errno.E2BIG) and n.value == count, (cap, rc, n.value)
        assert (out[:cap] == full[:cap]).all(), cap
        assert (out[cap:] == canary).all(), cap
    n.value = 0
    assert L.sqz_gpu_tokens_ex(p8, d.size, *G1, 0, None, 0, C.byref(n)) == errno.E2BIG and n.value == count
