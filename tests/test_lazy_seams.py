"""The lazy parse across shard seams, stated without the GPU.  The lazy step is 1 or len <= max_len, so a
shard is entered at an offset < max_len and leaves with an overshoot < max_len, exactly as under the greedy
rule; its only input beyond the shard is the table word at the next shard's first position.  So per-shard
exit maps of the lazy walk, chained over shard.plan, must give exactly the positions the whole-input lazy
walk (tests/lazy_oracle.py over the oracle's table) visits at each seam, and the shards' own walks from
those entries must concatenate to the whole walk."""
import numpy as np
import pytest

from sqz_b200 import corpus, shard

from lazy_oracle import lazy_tokens_from_table

G1 = (1 << 15, 3, 257, 32767)
RULES = [G1, (1 << 15, 2, 254, 32767), (1 << 15, 4, 16, 32767), (1 << 10, 2, 31, 5)]


def lazy_steps(ln, min_len):
    """Step of the lazy walk at every position: len(i) when len(i) >= min_len and len(i+1) <= len(i)
    (len(bytes) = 0), else 1."""
    here = ln.astype(np.int64)
    after = np.append(here[1:], 0)
    return np.where((here >= min_len) & (after <= here), here, 1)


def exit_maps(steps, plan, max_len):
    """For every shard and every entry e < max_len: where the lazy walk from first + e first lands at or
    past first + n, as an offset from first + n (e - n for an entry beyond the shard).  Pointer doubling over
    the steps, every shard at once."""
    total = steps.size
    end = np.zeros(total, np.int64)
    for s in plan:
        end[s.first:s.first + s.n] = s.first + s.n
    jump = np.arange(total, dtype=np.int64) + steps
    inside = jump < end
    while inside.any():
        jump = np.where(inside, jump[np.minimum(jump, total - 1)], jump)
        inside = jump < end
    maps = []
    for s in plan:
        e = np.arange(max_len, dtype=np.int64)
        at = np.minimum(s.first + e, max(total - 1, 0))
        land = jump[at] if total else e
        maps.append(np.where(e < s.n, land - (s.first + s.n), e - s.n).astype(np.uint16))
    return maps


def positions(toks, start=0):
    lens = np.where(toks > 0xFFFF, toks >> 16, 1).astype(np.int64)
    return start + np.cumsum(lens) - lens


def table(oracle, d, rules):
    window, mn, mx, md = rules
    return oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)


def check_seams(d, ln, ds, rules, world):
    """Chained per-shard maps against the whole lazy walk; returns (plan, maps, entries)."""
    window, mn, mx, md = rules
    whole, end = lazy_tokens_from_table(d, ln, ds, mn)
    assert end == d.size
    visited = np.append(positions(whole), end)                   # the end, where a walk past a last shard lands
    plan = shard.plan(d.size, world, md, mx)
    maps = exit_maps(lazy_steps(ln, mn), plan, mx)
    entries = shard.chain_entries(maps)
    assert entries[-1] == 0
    parts = []
    for s, e in zip(plan, entries):
        assert e < mx
        if s.n == 0:
            continue
        k = np.searchsorted(visited, s.first)
        assert visited[k] == s.first + e, (s, e, visited[k])          # the whole walk enters here
        toks, _ = lazy_tokens_from_table(d, ln, ds, mn, start=s.first + e)
        parts.append(toks[positions(toks, s.first + e) < s.first + s.n])
    cat = np.concatenate(parts) if parts else np.zeros(0, np.uint32)
    assert cat.size == whole.size and (cat == whole).all()
    return plan, maps, entries


@pytest.mark.parametrize("world", [2, 3, 5, 8])
@pytest.mark.parametrize("name", ["laozi.txt", "confucius.txt", "csrc.cat", "x64.elf", "mandrill.bmp"])
def test_fixtures(name, world, inputs, oracle):
    d = inputs[name]
    ln, ds = table(oracle, d, G1)
    check_seams(d, ln, ds, G1, world)


@pytest.mark.parametrize("rules", RULES[1:])
@pytest.mark.parametrize("world", [2, 3, 7, 8])
def test_other_rules(rules, world, inputs, oracle):
    d = np.ascontiguousarray(inputs["x64.elf"][300001:500000])          # an odd size
    ln, ds = table(oracle, d, rules)
    check_seams(d, ln, ds, rules, world)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_synthetic_corpus(world, oracle):
    d = corpus.synthetic((3 << 20) + 4097, 1 << 20)
    ln, ds = table(oracle, d, G1)
    check_seams(d, ln, ds, G1, world)


@pytest.mark.parametrize("name", ["empty", "one", "two", "aaa", "aaaa", "hello", "abc40", "zeros4096"])
def test_tiny_inputs_and_empty_shards(name, inputs, oracle):
    """Fewer bytes than shards: the first bytes % world shards hold one byte, the rest none."""
    d = inputs[name]
    ln, ds = table(oracle, d, G1)
    for world in (1, 2, 3, 8, 13):
        check_seams(d, ln, ds, G1, world)


@pytest.mark.parametrize("rules", RULES)
def test_maps_are_the_walks_from_every_entry(rules, inputs, oracle):
    """The doubling above against the plain statement: for every entry e < max_len, the lazy walk over the
    oracle's table from first + e, stopped at the first position at or past first + n."""
    d = np.ascontiguousarray(inputs["laozi.txt"][:9001])
    window, mn, mx, md = rules
    ln, ds = table(oracle, d, rules)
    plan = shard.plan(d.size, 3, md, mx)
    for s, m in zip(plan, exit_maps(lazy_steps(ln, mn), plan, mx)):
        for e in range(mx):
            toks, stop = lazy_tokens_from_table(d, ln, ds, mn, start=s.first + e)
            at = positions(toks, s.first + e)
            after = at[at >= s.first + s.n]
            land = int(after[0]) if after.size else stop
            assert m[e] == land - (s.first + s.n), (s, e)


def test_a_seam_decided_lazily(oracle):
    """The case the seam word exists for: at a cut, position n-1 holds a match of 11 and position n one of
    40.  The greedy walk takes the 11 and enters the next shard at 10; the lazy walk emits a literal and
    enters at 0, where the 40 starts."""
    rng = np.random.default_rng(4)
    d = rng.integers(0, 256, 20000, dtype=np.uint8)
    n = 10000
    unit, x = rng.integers(0, 256, 40, dtype=np.uint8), rng.integers(0, 256, 1, dtype=np.uint8)
    d[n - 3000: n - 2960] = unit
    d[n - 2000: n - 1989] = np.concatenate([x, unit[:10]])
    d[n - 1: n + 40] = np.concatenate([x, unit])
    d[n + 40] = unit[10] ^ 0xFF
    ln, ds = table(oracle, d, G1)
    assert ln[n - 1] == 11 and ln[n] == 40
    plan, maps, entries = check_seams(d, ln, ds, G1, 2)
    assert entries[1] == 0
    greedy = np.where(ln >= 3, ln, 1).astype(np.int64)
    assert exit_maps(greedy, plan, 257)[0][0] == 10
