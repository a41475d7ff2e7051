"""The bit-sliced match search in its throughput shape off the default rules, and every plan of its latency
shape, against oracle B word for word.

How a shard is searched (sqz_gpu.cu: slice_plan, launch_tiles; match_bitsliced.cuh):
- More than one wave of throughput tiles -- 444 CTAs (kWaveQ4 = 148 x 3) of 16,256 positions (tile_pos(4)),
  i.e. more than 7,217,664 positions -- runs the throughput shape (kQ = 4), unsliced.
- Below that, the latency shape (kQ = 1, 3,968 positions per CTA, tile_pos(1)) with the distance range cut
  into as many slices as give about two waves of 740 CTAs (kWaveQ1 = 148 x 5): a power of two of at most 32,
  each slice a whole number of 1024-distance units.  From 1,480 tiles (5,868,673 positions) on, unsliced.
- Only the throughput shape has the quiet body, which compares six hashed bit planes and leaves the bytes to
  the scalar path.  The hash-twin inputs (tests/match_inputs.py) are equal to earlier bytes in those planes
  and not in the bytes, over whole blocks.
"""
import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import corpus
from lazy_oracle import lazy_tokens_from_table
from match_inputs import far_repeat_input, hash_twins, quiet_far_repeats
from mincost_oracle import mincost_tokens_from_table

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from sqz_b200 import device  # noqa: E402  (needs torch)

TILE_Q1, TILE_Q4 = 3968, 16256                  # v2::tile_pos(1), v2::tile_pos(4)
ONE_WAVE_Q4 = 148 * 3 * TILE_Q4                 # 7,217,664: the largest shard of the latency shape
N = int(7.5 * (1 << 20))                        # 484 throughput tiles, the last one partial

G1 = (1 << 15, 3, 257, 32767)                   # (window, min_len, max_len, max_dist)
WIDE2 = (1 << 16, 2, 254, 65535)
WIDE3 = (1 << 16, 3, 512, 65535)
SHORT33 = (1 << 15, 3, 33, 32767)               # phase 2's capped-inheritance slack is max_len - 32
NEAR64 = (1 << 15, 2, 64, 1000)
WINDOW = (1 << 15, 3, 257, 32768)               # max_dist equal to the window
WIN10 = (1 << 10, 3, 257, 1023)                 # sqz_compress at win_bits 10
DIST5 = (1 << 15, 3, 257, 5)                    # below one word of distances
DIST33 = (1 << 15, 3, 257, 33)


def unpack(t):
    w = t.cpu().numpy().view(np.uint32)
    return (w >> 16).astype(np.uint16), (w & 0xFFFF).astype(np.uint16)


def assert_table(ln, ds, oln, ods, what):
    bad = np.nonzero((ln != oln) | (ds != ods))[0]
    assert bad.size == 0, (what, bad.size, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])


def assert_same(got, want, what):
    assert got.size == want.size and (got == want).all(), (what, got.size, want.size)


def device_buffer(d):
    return torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])


def sampled_positions(rng, blocks, stretches):
    """Around the twin blocks' edges and the true stretches' ends, and inside the blocks."""
    pos = []
    for k in rng.choice(len(blocks), 30, replace=False).tolist():
        at, size, _ = blocks[k]
        pos += [at - 1, at, at + 1, at + size - 1, at + size, int(rng.integers(at, at + size))]
    for k in rng.choice(len(stretches), 50, replace=False).tolist():
        at, r, _ = stretches[k]
        pos += [at - 1, at, at + 1, at + r - 1, at + r]
    return sorted(p for p in set(pos) if p < N)


# (generator, rules, also as an interior shard with full halos through device.match_table)
MATRIX = [
    ("twins", G1, True), ("twins", WIDE2, True), ("twins", SHORT33, False), ("twins", WIDE3, False),
    ("far", SHORT33, False), ("far", NEAR64, True), ("far", WIDE3, True),
    ("text_far", SHORT33, False),
    ("synthetic", WINDOW, False), ("synthetic", WIN10, True), ("synthetic", DIST5, False), ("synthetic", DIST33, False),
]


@pytest.mark.parametrize("gen,rules,as_shard", MATRIX,
                         ids=["%s-%d-%d-%d-%d" % (g, r[0].bit_length() - 1, *r[1:]) for g, r, _ in MATRIX])
def test_throughput_shape(gen, rules, as_shard, oracle):
    """7.5 MiB through sq.match_table and sq.tokens: leading edge, interior and trailing edge tiles of the
    throughput shape (match_table<min_len, *, 4>), table == oracle B, tokens == its greedy parse."""
    window, mn, mx, md = rules
    rng = np.random.default_rng(MATRIX.index((gen, rules, as_shard)))
    if gen == "twins":
        d, blocks, stretches = hash_twins(rng, N, mn, mx, md)
    elif gen == "far":
        d = quiet_far_repeats(rng, N, md)[0]
    elif gen == "text_far":
        d = far_repeat_input(rng, N)
    else:
        d = corpus.synthetic(N, 3276897 * (md % 7))
    oln, ods = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    ln, ds = sq.match_table(d, window, mn, mx, md)
    assert_table(ln, ds, oln, ods, (gen, rules))
    t = sq.tokens(d, window, mn, mx, md)
    ot, end = oracle.tokens_from_table(d, oln, ods, mn)
    assert end == N
    assert_same(t, ot, (gen, rules))
    if as_shard:                                       # no edge tiles but the partial last one
        first, cnt = md, N - md - mx
        tb = unpack(device.match_table(device_buffer(d), first, cnt, md, mx, mn, mx, md))
        assert_table(*tb, oln[first:first + cnt], ods[first:first + cnt], (gen, rules, "shard"))
    if gen == "twins":
        # the stretches are found where the generator put them ...
        long_enough = [(at, r) for at, r, _ in stretches if r >= mn]
        assert all(oln[at] >= min(r, mx) for at, r in long_enough)
        # ... and oracle B agrees with the restated reference loop (oracle A) at the edges
        for i in sampled_positions(rng, blocks, stretches):
            assert oracle.best(d, i, window, min_len=mn, max_len=mx, max_dist=md) == (int(ln[i]), int(ds[i])), i
    if gen in ("far", "text_far") and mx <= 64:        # capped matches: phase 2's capped inheritance
        assert (oln == mx).sum() > N // 100


# Plan sweep: (n, distance slices) at max_dist 65535 and at max_dist 5000, from the constants above.  The
# sizes are whole tiles of the latency shape below one wave of the throughput shape, so that the tile size
# shows in the launch count; 7,217,665 is the first throughput shard and 7,233,920 is 445 whole tiles of it.
SWEEP_65535 = [(297_600, 32), (499_968, 16), (999_936, 8), (1_999_872, 4), (3_999_744, 2), (6_499_584, 1),
               (ONE_WAVE_Q4, 1), (ONE_WAVE_Q4 + 1, 1), (ONE_WAVE_Q4 + TILE_Q4, 1)]
SWEEP_5000 = [(297_600, 5), (499_968, 5), (999_936, 5), (1_999_872, 3), (3_999_744, 2), (6_499_584, 1),
              (ONE_WAVE_Q4, 1), (ONE_WAVE_Q4 + 1, 1), (ONE_WAVE_Q4 + TILE_Q4, 1)]
SWEEP = ([((1 << 16, 2, 254, 65535), n, s) for n, s in SWEEP_65535] +
         [((1 << 16, 3, 257, 65535), n, s) for n, s in SWEEP_65535] +
         [((1 << 15, 3, 257, 5000), n, s) for n, s in SWEEP_5000])


def expected_launches(n, slices):
    """launch_tiles with full halos: the interior tiles are one range, a partial last tile is a second one
    (the trailing edge).  A range costs 1 launch unsliced and 2 sliced (the nearest slice, then the seeded
    ones); combine_slices adds 1 to a sliced plan, finish_marked 1 to every plan."""
    tile = TILE_Q4 if n > ONE_WAVE_Q4 else TILE_Q1
    ranges = 1 if n % tile == 0 else 2
    return ranges * (2 if slices > 1 else 1) + (1 if slices > 1 else 0) + 1


@pytest.mark.parametrize("rules,n,slices", SWEEP, ids=["%d-%d-%d-%d" % (r[1], r[3], n, s) for r, n, s in SWEEP])
def test_slice_plans(rules, n, slices, oracle):
    """Every slice plan of the latency shape, its unsliced band and both sides of one throughput wave, as an
    interior shard with full halos: table == oracle B, and the launch count is the plan's.  The count tells
    sliced from unsliced and, at these sizes, the tile size; the number of slices follows from the constants."""
    window, mn, mx, md = rules
    d = corpus.synthetic(md + n + mx, (n * 7919 + md) % (64 << 20))
    oln, ods = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    buf = device_buffer(d)
    before = sq.launch_count()
    t = device.match_table(buf, md, n, md, mx, mn, mx, md)
    launches = sq.launch_count() - before
    assert launches == expected_launches(n, slices), (n, slices, launches)
    assert_table(*unpack(t), oln[md:md + n], ods[md:md + n], (rules, n))


@pytest.mark.parametrize("win_bits", [10, 12])
def test_compress_off_the_default_window(win_bits, oracle):
    """sq.compress on 40 MiB: chunks of 8, 16 and 10 MiB in the default ramp and of 11 MiB under a crew of
    coders (all above one throughput wave), at max_dist 1023 or 4095.  The bytes are the coder's on the oracle's
    greedy tokens, and at win_bits 12 likewise for the lazy and the min-cost parse; all decode to the input."""
    d = corpus.synthetic(40 << 20, 9 << 20)
    oln, ods = oracle.match_table(d, 1 << win_bits, fast=True)
    walks = {"greedy": oracle.tokens_from_table(d, oln, ods)[0]}
    if win_bits == 12:
        walks["lazy"] = lazy_tokens_from_table(d, oln, ods)[0]
        walks["mincost"] = mincost_tokens_from_table(d, oln, ods)[0]
    for mode, want in walks.items():
        want = sq.encode_tokens(want, d.size, win_bits)
        for threads in (1, 4):
            comp = sq.compress(d, win_bits, threads=threads, lazy=mode == "lazy", mincost=mode == "mincost")
            assert comp == want, (mode, threads, len(comp), len(want))
        assert sq.decompress(comp) == d.tobytes(), mode


@pytest.mark.parametrize("gen,rules", [("twins", WIDE2), ("synthetic", WIDE3)])
def test_tokens_multi_throughput_shards(gen, rules, oracle):
    """sq.tokens_multi with 2 and 3 shards of 7.5 MiB or more: throughput-shape shards with 65535-byte halos
    at their seams, tokens == the oracle's parse of the whole input."""
    window, mn, mx, md = rules
    n = 3 * N
    if gen == "twins":
        d = hash_twins(np.random.default_rng(77), n, mn, mx, md)[0]
    else:
        d = corpus.synthetic(n, 17 << 20)
    want = oracle.tokens_from_table(d, *oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx,
                                                           max_dist=md), mn)[0]
    n_dev = torch.cuda.device_count()
    for world in (2, 3):
        got = sq.tokens_multi(d, [g % n_dev for g in range(world)], window, mn, mx, md)
        assert_same(got, want, (gen, rules, world))
