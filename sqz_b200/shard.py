"""Multi-GPU sharding of the match search (host logic only, no compute).

The path shards by contiguous byte ranges (SURVEY.md section 8e): the match table of
shard g depends only on its own bytes plus a look-back halo of max_dist bytes and a
look-ahead halo of max_len bytes, so no data-path collective exists.  The greedy parse
has one scalar dependency per seam: the first parse position of shard g+1 is the
overshoot of shard g's last token.  Every shard publishes exit_map[e] = "overshoot I
produce when entered at offset e" (sqz_gpu_parse_exit_map_device); chaining those maps
gives every shard its true entry after one tiny all-gather.

The lazy parse steps 1 or len <= max_len as well, so entries and overshoots keep their bounds;
its one extra input at a seam, the best match at the next shard's first position, every shard
searches itself from its own look-ahead halo (device.match_table(..., seam=True)), and its maps
(device.exit_map(..., lazy=True)) chain here unchanged.

The min-cost parse is the one rule the cut matters to: its steps depend on the table words of
their own 16384-position segment, at global offsets that are multiples of 16384, so every shard
has to start at a segment and hold whole ones (all but the last): plan(..., align=SEGMENT).  Each
shard then rewrites its own table (device.mincost_steps) and the greedy exit maps and parse of the
rewritten table chain here unchanged, with no extra input at the seams.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np

SEGMENT = 16384     # positions of a min-cost segment (include/sqz_gpu.h, SQZ_GPU_STREAM_MINCOST)


@dataclass(frozen=True)
class Shard:
    rank: int
    first: int      # global offset of the first owned position
    n: int          # owned positions
    back: int       # look-back halo bytes available before `first`
    ahead: int      # look-ahead halo bytes available after first + n

    @property
    def lo(self) -> int:
        """Global offset of the first byte the shard needs."""
        return self.first - self.back

    @property
    def hi(self) -> int:
        """One past the last byte the shard needs."""
        return self.first + self.n + self.ahead


def plan(total: int, world: int, max_dist: int, max_len: int, *, align: int = 1) -> list[Shard]:
    """Cut [0, total) into `world` contiguous shards of whole `align`-byte units: ceil(total / align) units
    shared out as evenly as they go (the first ones one unit more), every cut clamped to `total`.  align=1:
    sizes differ by at most one byte (the cut of sqz_gpu_tokens_multi_ex); align=SEGMENT: the cut of the
    min-cost parse, the partial last segment in the last non-empty shard, shards past the segments empty."""
    if world < 1:
        raise ValueError("world must be >= 1")
    if align < 1:
        raise ValueError("align must be >= 1")
    base, extra = divmod(-(-total // align), world)
    out, first = [], 0
    for r in range(world):
        n = min(total, first + (base + (1 if r < extra else 0)) * align) - first
        out.append(Shard(r, first, n, min(first, max_dist), min(total - (first + n), max_len)))
        first += n
    return out


def chain_entries(exit_maps: Sequence[np.ndarray], first_entry: int = 0) -> list[int]:
    """entry[0] = first_entry, entry[g+1] = exit_maps[g][entry[g]]; returns world+1 values
    (the last one is the overshoot past the end of the data, 0 for a complete parse)."""
    entries = [int(first_entry)]
    for m in exit_maps:
        entries.append(int(np.asarray(m).astype(np.int64)[entries[-1]] & 0xFFFF))
    return entries


def offsets(counts: Sequence[int]) -> list[int]:
    """Where every shard's tokens start in the concatenated stream (exclusive prefix sum)."""
    out, at = [], 0
    for c in counts:
        out.append(at)
        at += int(c)
    return out


class Mailbox:
    """The seam exchange of a one-process-per-GPU job, without a collective library.

    A file in shared memory (/dev/shm) holds one slot per rank: the rank's exit map (<= 512 x u16),
    its token count and a sequence number for each.  A rank publishes by writing the payload and
    then the sequence number; readers poll the sequence number (x86 keeps the two stores in order).
    Per step every rank publishes its exit map, reads the maps of the ranks before it and chains
    them into its parse entry (`entry`); after its parse it publishes its token count and reads the
    earlier ones, whose sum is its offset in the concatenated stream (`offset`).  1 KiB + 8 bytes per
    rank and step cross the host; nothing else does.  `blob` carries set-up data (the CUDA IPC handle
    of the gather buffer).  Rank 0 creates the file and is the one to unlink it.
    """

    SLOT = 160          # u64 words per rank: [0] seq_map, [1] seq_count, [2] count, [3] seq_flag, [16..144) map
    HEAD = 32           # u64 words: [0] magic, [1] world, [2] blob seq, [8..24) blob

    def __init__(self, path: str, rank: int, world: int, create: bool, timeout: float = 120.0):
        import os
        import time
        self.path, self.rank, self.world, self.timeout = path, rank, world, timeout
        nbytes = 8 * (self.HEAD + self.SLOT * world)
        if create:
            with open(path + ".tmp", "wb") as f:
                f.write(bytes(nbytes))
            os.replace(path + ".tmp", path)           # appears complete or not at all
        else:
            t0 = time.time()
            while not (os.path.exists(path) and os.path.getsize(path) == nbytes):
                if time.time() - t0 > timeout:
                    raise TimeoutError("mailbox %s never appeared" % path)
                time.sleep(0.01)
        self.mm = np.memmap(path, dtype=np.uint64, mode="r+", shape=(self.HEAD + self.SLOT * world,))

    def _slot(self, r: int) -> int:
        return self.HEAD + self.SLOT * r

    def _wait(self, index: int, seq: int) -> None:
        import time
        spins, t0 = 0, None
        while int(self.mm[index]) < seq:
            spins += 1
            if spins > 2000:
                if t0 is None:
                    t0 = time.time()
                elif time.time() - t0 > self.timeout:
                    raise TimeoutError("mailbox: rank %d waited %.0f s for word %d to reach %d"
                                       % (self.rank, self.timeout, index, seq))
                time.sleep(20e-6)

    # -- set-up blob (rank 0 -> all) --
    def put_blob(self, data: bytes) -> None:
        assert len(data) <= 128
        buf = np.zeros(128, np.uint8)
        buf[: len(data)] = np.frombuffer(data, np.uint8)
        self.mm[8:24] = buf.view(np.uint64)
        self.mm[2] = self.mm[2] + np.uint64(1)

    def get_blob(self, seq: int = 1) -> bytes:
        self._wait(2, seq)
        return self.mm[8:24].tobytes()

    # -- per step --
    def entry(self, seq: int, exit_map: np.ndarray) -> tuple[int, list[int]]:
        """Publish this rank's exit map for step `seq` (1, 2, ...), chain the earlier ranks' maps.
        Returns (entry offset of this rank's parse, entries of ranks 0..rank)."""
        s = self._slot(self.rank)
        m = np.zeros(512, np.uint16)
        m[: exit_map.size] = exit_map
        self.mm[s + 16: s + 144] = m.view(np.uint64)
        self.mm[s + 0] = np.uint64(seq)
        entries = [0]
        for r in range(self.rank):
            b = self._slot(r)
            self._wait(b + 0, seq)
            other = np.array(self.mm[b + 16: b + 144]).view(np.uint16)
            entries.append(int(other[entries[-1]]))
        return entries[-1], entries

    def offset(self, seq: int, count: int) -> int:
        """Publish this rank's token count for step `seq`; the earlier ranks' counts sum to the
        offset of its tokens in the concatenated stream."""
        s = self._slot(self.rank)
        self.mm[s + 2] = np.uint64(count)
        self.mm[s + 1] = np.uint64(seq)
        at = 0
        for r in range(self.rank):
            b = self._slot(r)
            self._wait(b + 1, seq)
            at += int(self.mm[b + 2])
        return at

    def counts(self, seq: int) -> list[int]:
        """Every rank's token count of step `seq` (waits for all of them)."""
        out = []
        for r in range(self.world):
            b = self._slot(r)
            self._wait(b + 1, seq)
            out.append(int(self.mm[b + 2]))
        return out

    def barrier(self, seq: int) -> None:
        """Host-side barrier (no device work): everyone has reached flag value `seq`."""
        self.mm[self._slot(self.rank) + 3] = np.uint64(seq)
        for r in range(self.world):
            self._wait(self._slot(r) + 3, seq)

    def close(self, unlink: bool = False) -> None:
        import os
        self.mm.flush()
        del self.mm
        if unlink:
            try:
                os.unlink(self.path)
            except OSError:
                pass
