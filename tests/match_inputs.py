"""TEST INFRASTRUCTURE: seeded generators of match-search inputs that the GPU tests share.

far_repeat_input  -- text-like blocks repeated at distances of 30,000-32,767 (phase 2's capped inheritance).
hash_twins        -- blocks equal to earlier bytes in the bit-sliced kernel's hashed planes, not in the bytes
                     (the quiet body of the throughput shape, match_bitsliced.cuh).
quiet_far_repeats -- random bytes with true copies at distances from 600 up (the quiet body finding real
                     matches).
"""
import numpy as np

# The hashed bit planes of match_bitsliced.cuh:97-101 (kQuietPlanes = 6, kFold): planes 0-5 hold
# fold_byte(b) & 63, where fold_byte XORs the low six bits with a constant chosen by the two high bits.
# A byte b and b ^ x for every x in TWIN_XOR have the same hash and differ in both high bits' planes and
# the byte.  A change of kQuietPlanes or kFold must be followed here and in tests/test_match_inputs.py.
FOLD = 0x2B << 8 | 0x16 << 16 | (0x2B ^ 0x16) << 24
QUIET_PLANES = 6
TWIN_XOR = np.array([0x6B, 0x96, 0xFD], np.uint8)


def plane_hash(b: np.ndarray) -> np.ndarray:
    """The bits of fold_byte(b) that the quiet body compares (match_bitsliced.cuh:101)."""
    b = np.asarray(b, dtype=np.uint32)
    return ((b ^ ((FOLD >> (8 * (b >> QUIET_PLANES))) & 0xFF)) & ((1 << QUIET_PLANES) - 1)).astype(np.uint8)


def far_repeat_input(rng, n):
    """Blocks of 4-12 KiB repeated at distances of 30,000-32,767 with a few defects, runs of 32
    spaces and of one byte value in between: the far max_len early-out (squeeze.h:353) next to
    thousands of near candidates that tie on their first bytes."""
    out = []
    size = 0
    words = [b"    " * 8, b"\t\t", b"static ", b"const ", b"uint32_t ", b"return ", b";\n", b"if (", b") {\n", b"}\n"]
    def filler(k):
        parts, got = [], 0
        while got < k:
            w = words[int(rng.integers(0, len(words)))] if rng.random() < 0.7 else bytes(rng.integers(97, 123, int(rng.integers(1, 9)), dtype=np.uint8))
            parts.append(w); got += len(w)
        return np.frombuffer(b"".join(parts)[:k], np.uint8)
    while size < n:
        block = filler(int(rng.integers(4096, 12288)))
        gap = int(rng.integers(30000, 32768)) - block.size
        mid = filler(max(gap, 1)).copy()
        if rng.random() < 0.5:
            at = int(rng.integers(0, max(mid.size - 600, 1)))
            mid[at:at + int(rng.integers(33, 600))] = 32 if rng.random() < 0.5 else 0
        again = block.copy()
        for at in rng.integers(0, block.size, int(rng.integers(0, 4))).tolist():
            again[at] ^= 1
        out += [block, mid, again]
        size += 2 * block.size + mid.size
    return np.concatenate(out)[:n].copy()


def stretch_lengths(min_len, max_len):
    """The true-stretch lengths hash_twins plants: around min_len, around the scalar path's 32-bit window
    and around max_len."""
    return sorted({min_len - 1, min_len, min_len + 1, 31, 32, 33, max_len - 1, max_len, max_len + 1} - {0})


def hash_twins(rng, n, min_len, max_len, max_dist):
    """Random filler of 4.5-12 KiB (more than one warp's positions and the 512 distances after which a quiet
    warp drops its need masks) before every block of 2-16 KiB.  A block copies the bytes one distance d back,
    512 < d <= max_dist, each XORed with one of TWIN_XOR: equal to them in the hashed planes only, and the only
    distance of its group at which the block's positions meet candidates.  Inside a block, true stretches (XOR 0)
    of r bytes, r one of stretch_lengths(min_len, max_len), each followed by 2r + 300-1500 twin bytes.
    Returns (data, blocks [(start, length, d)], stretches [(start, length, d)])."""
    lens = stretch_lengths(min_len, max_len)
    out = rng.integers(0, 256, n, dtype=np.uint8)
    blocks, stretches = [], []
    at = int(rng.integers(4608, 12288))
    while True:
        size = int(rng.integers(2048, 16385))
        if at + size > n:
            break
        d = int(rng.integers(513, min(max_dist, at) + 1))
        mask = TWIN_XOR[rng.integers(0, 3, size)]
        k = int(rng.integers(16, 300))
        while True:
            r = lens[int(rng.integers(0, len(lens)))]
            if k + r + 1 > size:
                break
            mask[k:k + r] = 0
            stretches.append((at + k, r, d))
            k += 3 * r + int(rng.integers(300, 1500))
        for c in range(0, size, d):               # d < size: the source overlaps the block, copy d at a time
            m = min(d, size - c)
            out[at + c:at + c + m] = out[at + c - d:at + c - d + m] ^ mask[c:c + m]
        blocks.append((at, size, d))
        at += size + int(rng.integers(4608, 12288))
    return out, blocks, stretches


def quiet_far_repeats(rng, n, max_dist):
    """Random bytes with true copies of 2-600 bytes from 600..max_dist back, one every 300-3000 bytes.
    Returns (data, copies [(start, length, d)])."""
    out = rng.integers(0, 256, n, dtype=np.uint8)
    copies = []
    at = max_dist + 1
    while True:
        size = int(rng.integers(2, 601))
        if at + size > n:
            break
        d = int(rng.integers(600, max_dist + 1))
        for c in range(0, size, d):
            m = min(d, size - c)
            out[at + c:at + c + m] = out[at + c - d:at + c - d + m]
        copies.append((at, size, d))
        at += size + int(rng.integers(300, 3001))
    return out, copies
