"""The min-cost parse on several devices (sqz_gpu_tokens_multi_cuts, sq.tokens_multi(mincost=True)) and on the
device buffers of a one-process-per-device job (sqz_gpu_mincost_steps_device, device.mincost_steps, then the
flag-0 exit map and parse).  Everything is checked against the min-cost walk over the oracle's table
(tests/mincost_oracle.py), the rewritten words against tests/mincost_steps.py, the maps against the CPU maps
of tests/test_mincost_shards.py.  With fewer devices than shards, the shards share device 0."""
import ctypes as C
import errno

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus, shard

from mincost_oracle import SEGMENT, mincost_tokens_from_table
from mincost_steps import mincost_steps_from_table
from test_gpu_mincost import seam_input, walk
from test_lazy_seams import exit_maps, positions
from test_mincost import MINCOST_SIZES
from test_mincost_shards import steps_of

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SYMBOLS, SHORT_START, LAZY, MINCOST = 1, 2, 8, 32
G1 = (1 << 15, 3, 257, 32767)


def devices_for(world):
    n_dev = torch.cuda.device_count()
    return [g % n_dev for g in range(world)]


def same(got, want):
    return got.size == want.size and bool((got == want).all())


def multi_cuts(d, devices, cuts, flags, rules=G1, out=None):
    """sqz_gpu_tokens_multi_cuts: (rc, tokens, per-shard counts, *n_tokens); `out` a device tensor to gather
    into."""
    L = _lib.load()
    d = np.ascontiguousarray(d, dtype=np.uint8)
    devs = (C.c_int * len(devices))(*devices)
    at = None if cuts is None else (C.c_size_t * max(len(cuts), 1))(*cuts)
    buf = np.empty(max(d.size, 1), np.uint32) if out is None else out
    ptr = buf.ctypes.data if out is None else out.data_ptr()
    n, per = C.c_size_t(), (C.c_size_t * len(devices))()
    rc = L.sqz_gpu_tokens_multi_cuts(devs, len(devices), at, d.ctypes.data_as(_lib.u8p), d.size, *rules, flags,
                                     ptr, max(d.size, 1), C.byref(n), per)
    got = buf[: n.value] if out is None else out[: n.value].cpu().numpy().view(np.uint32)
    return rc, np.array(got, dtype=np.uint32), [int(x) for x in per], n.value


def per_shard(toks, plan):
    """How many of the walk's tokens start in each shard."""
    at = positions(toks)
    return [int(((at >= s.first) & (at < s.first + s.n)).sum()) for s in plan]


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_multi_equals_walk(world, inputs, oracle):
    devices = devices_for(world)
    for d in [inputs[k] for k in ("hello", "laozi.txt", "csrc.cat", "x64.elf")] + [corpus.synthetic((3 << 20) + 7, 0)]:
        want = walk(oracle, d)
        got, per = sq.tokens_multi(d, devices, mincost=True, return_shard_counts=True)
        assert same(got, want), (d.size, world)
        assert same(sq.tokens(d, mincost=True), want)
        assert per == per_shard(want, shard.plan(d.size, world, 32767, 257, align=SEGMENT)), (d.size, world)


def test_multi_small_inputs_and_empty_shards(oracle):
    rng = np.random.default_rng(9)
    for size in list(range(10)) + [16383, 16384, 16385, 40000]:
        d = rng.integers(0, 4, size, dtype=np.uint8)
        want = walk(oracle, d) if size else np.zeros(0, np.uint32)
        for world in (1, 3, 8):
            got, per = sq.tokens_multi(d, devices_for(world), mincost=True, return_shard_counts=True)
            assert same(got, want), (size, world)
            segments = -(-size // SEGMENT)
            assert sum(per) == want.size and all(c == 0 for c in per[segments:]), (size, world, per)
            if size == 40000 and world == 8:
                assert segments == 3 and all(c > 0 for c in per[:3])


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_multi_cuts_inside_long_matches(world, oracle):
    """seam_input puts a long match across every segment end; at the cuts of plan(align=SEGMENT), which are
    segment ends, the walk's token runs across every cut."""
    d = seam_input(12, 30 + world)
    want = walk(oracle, d)
    got, per = sq.tokens_multi(d, devices_for(world), mincost=True, return_shard_counts=True)
    assert same(got, want)
    lens = np.where(want > 0xFFFF, want >> 16, 1).astype(np.int64)
    starts = positions(want)
    plan = shard.plan(d.size, world, 32767, 257, align=SEGMENT)
    for s in plan[1:]:
        assert ((starts < s.first) & (starts + lens > s.first) & (lens > 1)).any(), s
    assert per == per_shard(want, plan)


def test_explicit_cuts(oracle):
    L = _lib.load()
    d = seam_input(12, 5)
    total = d.size
    want = walk(oracle, d)
    devices = devices_for(4)
    for cuts in ([SEGMENT, 2 * SEGMENT, 10 * SEGMENT], [0, 7 * SEGMENT, 7 * SEGMENT], [3 * SEGMENT, 12 * SEGMENT, total],
                 [total, total, total], [0, 0, 0]):
        rc, got, per, _ = multi_cuts(d, devices, cuts, MINCOST)
        assert rc == 0, L.sqz_gpu_last_error()
        assert same(got, want), cuts
        plan = [shard.Shard(g, a, b - a, 0, 0) for g, (a, b) in enumerate(zip([0] + cuts, cuts + [total]))]
        assert per == per_shard(want, plan), cuts
        assert same(sq.tokens_multi(d, devices, mincost=True, cuts=cuts), want)
    misaligned = [SEGMENT + 1, 5 * SEGMENT, 9 * SEGMENT - 7]
    rc, _, _, n = multi_cuts(d, devices, misaligned, MINCOST)
    assert rc == errno.EINVAL and n == 0
    for flags, lazy in ((0, False), (LAZY, True)):
        rc, got, _, _ = multi_cuts(d, devices, misaligned, flags)
        assert rc == 0 and same(got, sq.tokens(d, lazy=lazy)), flags
        assert same(sq.tokens_multi(d, devices, lazy=lazy, cuts=misaligned), got)
    for cuts, flags in (([2 * SEGMENT, SEGMENT, 3 * SEGMENT], MINCOST), ([2 * SEGMENT, SEGMENT, 3 * SEGMENT], 0),
                        ([SEGMENT, 2 * SEGMENT, total + 1], 0), ([SEGMENT, 2 * SEGMENT, 14 * SEGMENT], MINCOST),
                        (None, LAZY | MINCOST), (None, SYMBOLS), (None, MINCOST | SYMBOLS), (None, SHORT_START),
                        (None, 4), (None, 16), (None, 1 << 31)):
        rc, _, _, n = multi_cuts(d, devices, cuts, flags)
        assert rc == errno.EINVAL and n == 0, (cuts, flags)
    for rules in ((1 << 15, 2, 257, 32767), (1 << 15, 3, 258, 32767), (1 << 16, 3, 257, 32768)):
        rc, _, _, n = multi_cuts(d, devices, None, MINCOST, rules)
        assert rc == errno.EINVAL and n == 0, rules
    with pytest.raises(ValueError):
        sq.tokens_multi(d, devices, cuts=[SEGMENT])
    with pytest.raises(ValueError):
        sq.tokens_multi(d, devices, lazy=True, mincost=True)


def test_multi_gathers_on_a_device(oracle):
    d = corpus.synthetic(2 << 20, 12345)
    want = walk(oracle, d)
    for world in (2, 4):
        out = torch.zeros(d.size, dtype=torch.int32, device="cuda:0")
        rc, got, per, _ = multi_cuts(d, devices_for(world), None, MINCOST, out=out)
        assert rc == 0, _lib.load().sqz_gpu_last_error()
        assert same(got, want) and sum(per) == want.size


@pytest.mark.parametrize("kernel", [1, 2], ids=["per_position", "bit_sliced"])
@pytest.mark.parametrize("rules", [G1, (1 << 15, 4, 16, 32767), (1 << 15, 3, 64, 32767), (1 << 15, 3, 257, 1024),
                                   (1 << 10, 3, 31, 5)])
def test_rule_sets(rules, kernel, inputs, oracle):
    d = np.concatenate([inputs["confucius.txt"], inputs["x64.elf"][:200000], inputs["mandrill.bmp"][:50000]])
    want = walk(oracle, d, rules)
    w, mn, mx, md = rules
    sq.select_kernel(kernel)
    try:
        for world in (2, 5):
            got = sq.tokens_multi(d, devices_for(world), w, mn, mx, md, mincost=True)
            assert same(got, want), (rules, world)
    finally:
        sq.select_kernel(0)


@pytest.mark.parametrize("name", sorted(MINCOST_SIZES))
def test_codec(name, inputs):
    d = inputs[name]
    comp = sq.encode_tokens(sq.tokens_multi(d, devices_for(4), mincost=True), d.size, 15)
    assert comp == sq.compress(d, mincost=True) and len(comp) == MINCOST_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_device_buffer_hand_off(world, oracle):
    """The one-process-per-device path at plan(align=SEGMENT): match_table, mincost_steps (== the CPU words),
    exit maps == the CPU maps, chained; every shard parsed from its entry overshoots into the next entry;
    tokens and symbol words concatenated == the min-cost walk and its symbol words."""
    from sqz_b200 import device
    L = _lib.load()
    d = seam_input(16, 40 + world)                                    # 17 segments
    total = d.size
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    whole, _ = mincost_tokens_from_table(d, ln, ds, 3)
    words_cpu = mincost_steps_from_table(ln, ds, 3)
    buf = torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    plan = shard.plan(total, world, 32767, 257, align=SEGMENT)
    cpu_maps = exit_maps(steps_of(words_cpu), plan, 257)
    tables, maps = [], []
    for s, want_map in zip(plan, cpu_maps):
        t = device.match_table(buf, s.first, s.n, s.back, s.ahead)
        assert device.mincost_steps(t, s.first, s.n, total) is t
        w = t.cpu().numpy().view(np.uint32)
        assert (w == words_cpu[s.first:s.first + s.n]).all(), s
        m = device.exit_map(t, s.n).cpu().numpy().view(np.uint16)[:257]
        assert (m == want_map).all(), (s, np.nonzero(m != want_map)[0][:5])
        tables.append(t)
        maps.append(m)
    entries = shard.chain_entries(maps)
    assert entries[-1] == 0
    parts, syms = [], []
    for s, t, e in zip(plan, tables, entries):
        tok, over = device.parse(buf, s.first, t, s.n, e)
        assert over == entries[s.rank + 1]
        parts.append(tok.cpu().numpy().view(np.uint32))
        sym, over = device.parse(buf, s.first, t, s.n, e, symbols=True)
        assert over == entries[s.rank + 1]
        syms.append(sym.cpu().numpy().view(np.uint32))
    assert same(np.concatenate(parts), whole)
    assert same(np.concatenate(syms), sq.symbols_of_tokens(whole))
    # the refusals, and n = 0
    t = tables[0].clone()
    st = torch.cuda.current_stream().cuda_stream
    for first, n, size, rules in ((1, SEGMENT, total, (3, 257, 32767)), (SEGMENT, SEGMENT + 1, total, (3, 257, 32767)),
                                  (0, total + 1, total, (3, 257, 32767)), (total, 1, total, (3, 257, 32767)),
                                  (16 * SEGMENT, total - 16 * SEGMENT - 1, total, (3, 257, 32767)),
                                  (0, SEGMENT, total, (2, 257, 32767)), (0, SEGMENT, total, (3, 258, 32767)),
                                  (0, SEGMENT, total, (3, 257, 32768)), (0, SEGMENT, total, (3, 2, 32767))):
        assert L.sqz_gpu_mincost_steps_device(t.data_ptr(), first, n, size, *rules, st) == errno.EINVAL, (first, n)
    with pytest.raises(ValueError):
        device.mincost_steps(t[:10], 0, SEGMENT, total)
    k = sq.launch_count()
    assert L.sqz_gpu_mincost_steps_device(t.data_ptr(), SEGMENT, 0, total, 3, 257, 32767, st) == 0
    assert L.sqz_gpu_mincost_steps_device(t.data_ptr(), 16 * SEGMENT, total - 16 * SEGMENT, total, 3, 257, 32767,
                                          st) == 0                         # a last shard of a partial segment
    assert L.sqz_gpu_mincost_steps_device(t.data_ptr(), 0, 0, 0, 3, 257, 32767, st) == 0
    torch.cuda.synchronize()
    assert sq.launch_count() - k == 1
    assert (t[total - 16 * SEGMENT:] == tables[0][total - 16 * SEGMENT:]).all()


def test_256_mib_in_4_and_8_shards(oracle):
    """256 MiB of the bench corpus: the one-shot call (two chunks) and 4 and 8 shards, the walk over oracle B."""
    d = corpus.synthetic(256 << 20, 0)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    want, end = mincost_tokens_from_table(d, ln, ds, 3)
    del ln, ds
    assert end == d.size
    one = sq.tokens(d, mincost=True)
    assert same(one, want)
    del one
    for world in (4, 8):
        got, per = sq.tokens_multi(d, devices_for(world), mincost=True, return_shard_counts=True)
        assert same(got, want) and sum(per) == want.size, world
        del got


def test_kernel_timing():
    """One launch of the min-cost kernel per non-empty shard, none for the greedy and lazy multi calls."""
    L = _lib.load()
    d = corpus.synthetic(3 << 20, 0)
    small = d[:40000]
    L.sqz_gpu_set_timing(1)
    try:
        L.sqz_gpu_mincost_kernel_seconds(1, None)
        launches = C.c_uint64()
        for lazy in (False, True):
            sq.tokens_multi(d, devices_for(4), lazy=lazy)
            sq.tokens_multi(d, devices_for(4), lazy=lazy, cuts=[SEGMENT, 2 * SEGMENT, 3 * SEGMENT])
        L.sqz_gpu_mincost_kernel_seconds(0, C.byref(launches))
        assert launches.value == 0
        sq.tokens_multi(d, devices_for(4), mincost=True)
        sq.tokens_multi(small, devices_for(8), mincost=True)              # 3 non-empty shards
        seconds = L.sqz_gpu_mincost_kernel_seconds(1, C.byref(launches))
        assert launches.value == 4 + 3 and seconds > 0
    finally:
        L.sqz_gpu_set_timing(0)
        L.sqz_gpu_match_kernel_seconds(1, None)


def test_the_old_calls_are_unchanged():
    """sqz_gpu_tokens_multi_cuts(NULL, 0 | LAZY) == sqz_gpu_tokens_multi_ex, bit for bit and with as many
    kernel launches; _ex still refuses MINCOST."""
    L = _lib.load()
    d = corpus.synthetic((1 << 20) + 3, 777)
    p8 = d.ctypes.data_as(_lib.u8p)
    out = np.zeros(d.size, np.uint32)
    n = C.c_size_t()
    for world in (2, 3):
        devs = (C.c_int * world)(*devices_for(world))
        for flags in (0, LAZY):
            per = (C.c_size_t * world)()
            k0 = sq.launch_count()
            assert L.sqz_gpu_tokens_multi_ex(devs, world, p8, d.size, *G1, flags, out.ctypes.data, out.size,
                                             C.byref(n), per) == 0
            old, old_per, k1 = out[: n.value].copy(), list(per), sq.launch_count()
            rc, got, new_per, _ = multi_cuts(d, devices_for(world), None, flags)
            assert rc == 0 and same(got, old) and new_per == old_per
            assert sq.launch_count() - k1 == k1 - k0, (world, flags)
        assert L.sqz_gpu_tokens_multi_ex(devs, world, p8, d.size, *G1, MINCOST, out.ctypes.data, out.size,
                                         C.byref(n), None) == errno.EINVAL
