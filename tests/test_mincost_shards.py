"""The min-cost parse across shard seams, stated without the GPU.  A min-cost step depends only on the table
words of its own 16384-position segment, and segments sit at global offsets that are multiples of 16384.  So
a shard that starts at a multiple of 16384 and holds whole segments (all but the last) can rewrite its own
part of the table (tests/mincost_steps.py, the rule of tests/c/mincost_walk.c) and get exactly the words of
the whole input's rewrite.  Every step is 1 or min_len <= k <= len <= max_len, so the greedy walk over those
words enters and leaves a shard below max_len, exactly as the greedy parse does: per-shard exit maps, chained
over shard.plan(..., align=SEGMENT), must give the positions the whole min-cost walk visits at every seam, and
the shards' own walks must concatenate to it.  The cut of shard.plan(...) (align 1) does not have the
property: shard-local segments give a different stream."""
import numpy as np
import pytest

from sqz_b200 import corpus, shard

from mincost_oracle import SEGMENT, mincost_tokens_from_table
from mincost_steps import mincost_steps_from_table, walk_steps
from test_lazy_seams import exit_maps, positions

G1 = (1 << 15, 3, 257, 32767)
RULES = [G1, (1 << 15, 4, 16, 32767), (1 << 15, 3, 64, 32767), (1 << 10, 3, 31, 5)]
TOTALS = [0, 1, 5, 16383, 16384, 16385, 10 ** 6 + 7]


def table(oracle, d, rules):
    window, mn, mx, md = rules
    return oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)


def steps_of(words):
    return np.where(words >> 16 != 0, words >> 16, 1).astype(np.int64)


def long_matches_across_segment_ends(segments, seed):
    """Random bytes with a 300-byte repeat of a block from 2 KiB earlier across every segment end."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, segments * SEGMENT + 999, dtype=np.uint8)
    for k in range(1, segments + 1):
        e = k * SEGMENT
        block = rng.integers(0, 256, 300, dtype=np.uint8)
        d[e - 2150: e - 1850] = block
        d[e - 150: e + 150] = block
    return d


def shard_words(ln, ds, plan, min_len):
    """Every shard rewrites its own part of the table, with segments counted from its first position."""
    return [mincost_steps_from_table(ln[s.first:s.first + s.n], ds[s.first:s.first + s.n], min_len) for s in plan]


def check_seams(d, ln, ds, rules, world):
    """Shard-local rewrites over plan(align=SEGMENT) against the whole min-cost walk; returns the entries."""
    window, mn, mx, md = rules
    whole, end = mincost_tokens_from_table(d, ln, ds, mn)
    assert end == d.size
    visited = np.append(positions(whole), end)
    plan = shard.plan(d.size, world, md, mx, align=SEGMENT)
    parts = shard_words(ln, ds, plan, mn)
    words = np.concatenate(parts) if d.size else np.zeros(0, np.uint32)
    assert (words == mincost_steps_from_table(ln, ds, mn)).all()
    maps = exit_maps(steps_of(words), plan, mx)
    entries = shard.chain_entries(maps)
    assert entries[-1] == 0
    cat = []
    for s, w, e, m in zip(plan, parts, entries, maps):
        assert e < mx
        if s.n == 0:
            continue
        k = np.searchsorted(visited, s.first)
        assert visited[k] == s.first + e, (s, e, visited[k])          # the whole walk enters here
        toks, stop = walk_steps(d[s.first:s.first + s.n], w, e)
        assert stop - s.n == m[e] == entries[s.rank + 1]
        cat.append(toks)
    cat = np.concatenate(cat) if cat else np.zeros(0, np.uint32)
    assert cat.size == whole.size and (cat == whole).all()
    return entries


@pytest.mark.parametrize("name", ["laozi.txt", "confucius.txt", "csrc.cat", "x64.elf", "mandrill.bmp", "hello",
                                  "zeros4096", "empty"])
def test_walk_over_the_rewritten_table(name, inputs, oracle):
    """The greedy walk over the rewritten words is the min-cost walk; every word is a literal (0) or a prefix
    (k, dist) of the best match."""
    d = inputs[name]
    ln, ds = table(oracle, d, G1)
    words = mincost_steps_from_table(ln, ds, 3)
    k = (words >> 16).astype(np.int64)
    assert ((k == 0) | ((k >= 3) & (k <= ln))).all()
    assert ((k == 0) | ((words & 0xFFFF) == ds)).all()
    want, _ = mincost_tokens_from_table(d, ln, ds, 3)
    got, end = walk_steps(d, words)
    assert end == d.size and got.size == want.size and (got == want).all()


def test_walk_over_the_rewritten_table_long_matches_and_corpus(oracle):
    for d in (long_matches_across_segment_ends(5, 3), corpus.synthetic((3 << 20) + 7, 3276897 - (1 << 20))):
        ln, ds = table(oracle, d, G1)
        want, _ = mincost_tokens_from_table(d, ln, ds, 3)
        got, end = walk_steps(d, mincost_steps_from_table(ln, ds, 3))
        assert end == d.size and got.size == want.size and (got == want).all()


@pytest.mark.parametrize("total", TOTALS)
def test_plan_align(total):
    for world in range(1, 14):
        assert shard.plan(total, world, 32767, 257, align=1) == shard.plan(total, world, 32767, 257)
        plan = shard.plan(total, world, 32767, 257, align=SEGMENT)
        assert len(plan) == world and plan[0].first == 0 and sum(s.n for s in plan) == total
        segments = []
        for s, t in zip(plan, plan[1:]):
            assert t.first == s.first + s.n
        for s in plan:
            assert s.first % SEGMENT == 0 or s.first == total
            end = s.first + s.n
            assert end % SEGMENT == 0 or end == total
            segments.append(-(-s.n // SEGMENT))
            assert s.back == min(s.first, 32767) and s.ahead == min(total - end, 257)
        assert max(segments) - min(segments) <= 1 and sum(segments) == -(-total // SEGMENT)
        assert segments == sorted(segments, reverse=True)                # the longer shards come first


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8, 13])
@pytest.mark.parametrize("name", ["laozi.txt", "csrc.cat", "x64.elf", "mandrill.bmp"])
def test_fixtures(name, world, inputs, oracle):
    d = inputs[name]
    ln, ds = table(oracle, d, G1)
    check_seams(d, ln, ds, G1, world)


@pytest.mark.parametrize("rules", RULES)
def test_rule_sets_odd_sizes(rules, inputs, oracle):
    d = np.ascontiguousarray(inputs["x64.elf"][300001:500000])          # an odd size, 12+ segments
    ln, ds = table(oracle, d, rules)
    for world in range(1, 14):
        check_seams(d, ln, ds, rules, world)


@pytest.mark.parametrize("world", [2, 3, 4, 8, 13])
def test_synthetic_corpus_and_long_matches(world, oracle):
    for d in (corpus.synthetic((3 << 20) + 4097, 1 << 20), long_matches_across_segment_ends(12, world)):
        ln, ds = table(oracle, d, G1)
        check_seams(d, ln, ds, G1, world)


@pytest.mark.parametrize("size", [0, 1, 7, 16383, 16384, 16385, 40000])
def test_small_inputs_and_empty_shards(size, oracle):
    """Fewer segments than shards: the shards past the segment count are empty."""
    d = np.ascontiguousarray(np.resize(corpus.synthetic(50000, 77), size))
    ln, ds = table(oracle, d, G1)
    for world in (1, 2, 3, 8, 13):
        check_seams(d, ln, ds, G1, world)
        plan = shard.plan(size, world, 32767, 257, align=SEGMENT)
        assert all(s.n == 0 for s in plan[-(-size // SEGMENT):])


def test_the_cut_must_be_aligned(oracle):
    """At the cut of plan(align=1), shard 0's last segment ends at the cut instead of at a multiple of 16384.
    A match of 20 starts 5 bytes before the cut: the whole walk takes all 20 (13 bits plus the distance's,
    against 11 for a 10 and another match for the rest), while shard 0, which prices everything past its end at
    0, takes the 10 with no extra bits.  The same input at plan(align=SEGMENT) gives the whole walk."""
    d = long_matches_across_segment_ends(4, 11)
    cut = -(-d.size // 2)
    block = np.random.default_rng(5).integers(0, 256, 20, dtype=np.uint8)
    d[cut - 2000: cut - 1980] = block
    d[cut - 5: cut + 15] = block
    ln, ds = table(oracle, d, G1)
    assert ln[cut - 5] == 20 and ln[cut - 6] == 0
    whole, _ = mincost_tokens_from_table(d, ln, ds, 3)
    plan = shard.plan(d.size, 2, 32767, 257)
    assert plan[1].first == cut and cut % SEGMENT != 0
    got, end = walk_steps(d, np.concatenate(shard_words(ln, ds, plan, 3)))
    at_whole = dict(zip(positions(whole).tolist(), whole.tolist()))
    at_got = dict(zip(positions(got).tolist(), got.tolist()))
    assert at_whole[cut - 5] == 20 << 16 | 1995 and at_got[cut - 5] == 10 << 16 | 1995
    assert end == d.size and not (got.size == whole.size and (got == whole).all())
    check_seams(d, ln, ds, G1, 2)


def test_refusals_come_before_any_device():
    """sqz_gpu_tokens_multi_cuts and sqz_gpu_mincost_steps_device check every argument before they touch a
    device: EINVAL with *n_tokens 0 on any host, with or without a GPU."""
    import ctypes as C
    import errno
    from sqz_b200 import _lib
    L = _lib.load()
    d = np.zeros(100000, np.uint8)
    out = np.zeros(d.size, np.uint32)
    devs = (C.c_int * 4)(0, 0, 0, 0)

    def multi(cuts, flags, rules=G1):
        n = C.c_size_t(7)
        at = None if cuts is None else (C.c_size_t * 3)(*cuts)
        rc = L.sqz_gpu_tokens_multi_cuts(devs, 4, at, d.ctypes.data_as(_lib.u8p), d.size, *rules, flags,
                                         out.ctypes.data, out.size, C.byref(n), None)
        return rc, n.value

    for cuts, flags in (([SEGMENT + 1, 2 * SEGMENT, 3 * SEGMENT], 32), ([SEGMENT, 2 * SEGMENT, 99999], 32),
                        ([3, 2, 1], 0), ([1, 2, d.size + 1], 8), (None, 8 | 32), (None, 1), (None, 2), (None, 4),
                        (None, 16)):
        assert multi(cuts, flags) == (errno.EINVAL, 0), (cuts, flags)
    for rules in ((1 << 15, 2, 257, 32767), (1 << 15, 3, 258, 32767), (1 << 16, 3, 257, 32768)):
        assert multi(None, 32, rules) == (errno.EINVAL, 0), rules
    for first, n, total, rules in ((1, SEGMENT, 10 ** 5, G1[1:]), (0, SEGMENT + 1, 10 ** 5, G1[1:]),
                                   (0, 10 ** 5 + 1, 10 ** 5, G1[1:]), (0, SEGMENT, 10 ** 5, (2, 257, 32767)),
                                   (0, SEGMENT, 10 ** 5, (3, 258, 32767)), (0, SEGMENT, 10 ** 5, (3, 257, 32768))):
        assert L.sqz_gpu_mincost_steps_device(None, first, n, total, *rules, None) == errno.EINVAL, (first, n, rules)
    assert L.sqz_gpu_mincost_steps_device(None, SEGMENT, 0, 10 ** 5, *G1[1:], None) == 0
