"""The premises of the generators in tests/match_inputs.py, without a GPU.

hash_twins is only worth something while its blocks are equal to their source in the bit-sliced kernel's
hashed planes and different in the bytes.  plane_hash restates fold_byte (match_bitsliced.cuh:97-101); if
kQuietPlanes or kFold change there, the restatement, TWIN_XOR and this test have to change with them."""
import numpy as np
import pytest

from match_inputs import TWIN_XOR, hash_twins, plane_hash, quiet_far_repeats, stretch_lengths


def test_twin_patterns_keep_the_hash_of_every_byte():
    b = np.arange(256, dtype=np.uint8)
    h = plane_hash(b)
    for x in TWIN_XOR:
        assert (plane_hash(b ^ x) == h).all() and ((b ^ x) >> 6 != b >> 6).all()
    # and the hash with the two high bits determines the byte: all eight planes tell every pair apart
    assert np.unique(h.astype(np.uint16) | (b.astype(np.uint16) >> 6 << 8)).size == 256


@pytest.mark.parametrize("min_len,max_len,max_dist", [(3, 257, 32767), (2, 254, 65535), (3, 33, 32767),
                                                      (3, 512, 65535)])
def test_hash_twins_keep_their_premise(min_len, max_len, max_dist):
    n = 8 << 20
    d, blocks, stretches = hash_twins(np.random.default_rng(max_len + max_dist), n, min_len, max_len, max_dist)
    assert d.size == n and len(blocks) > 300
    covered = sum(size for _, size, _ in blocks)
    assert covered > n // 3
    dists = np.array([dd for _, _, dd in blocks])
    assert dists.min() > 512 and dists.max() <= max_dist
    if max_dist > 32767:
        assert (dists > 32767).sum() > len(blocks) // 4
    h = plane_hash(d)
    differ = 0
    for at, size, dd in blocks:
        assert at - dd >= 0
        assert (h[at:at + size] == h[at - dd:at - dd + size]).all(), (at, size, dd)
        differ += int((d[at:at + size] != d[at - dd:at - dd + size]).sum())
    # most of a block is equal only in the hash; the rest are the true stretches
    assert differ > 0.85 * covered
    got = set()
    for at, r, dd in stretches:
        assert (d[at:at + r] == d[at - dd:at - dd + r]).all(), (at, r, dd)
        assert d[at - 1] != d[at - 1 - dd] and d[at + r] != d[at + r - dd], (at, r, dd)
        got.add(r)
    assert got == set(stretch_lengths(min_len, max_len))
    # the fillers between blocks: random, and long enough to keep the blocks' warps quiet first
    for (a0, s0, _), (a1, _, _) in zip(blocks, blocks[1:]):
        assert a1 - (a0 + s0) >= 4608


@pytest.mark.parametrize("max_dist", [1000, 65535])
def test_quiet_far_repeats_are_true_copies(max_dist):
    n = 4 << 20
    d, copies = quiet_far_repeats(np.random.default_rng(5), n, max_dist)
    assert d.size == n and len(copies) > n // 2000
    sizes = np.array([size for _, size, _ in copies])
    dists = np.array([dd for _, _, dd in copies])
    assert sizes.min() == 2 and sizes.max() == 600 and dists.min() >= 600 and dists.max() <= max_dist
    for at, size, dd in copies:
        assert (d[at:at + size] == d[at - dd:at - dd + size]).all(), (at, size, dd)
