"""The lazy parse on every GPU token entry point: the one-shot call (sqz_gpu_tokens_ex), several devices
(sqz_gpu_tokens_multi_ex) and the device-buffer entry points a one-process-per-device job chains itself
(sqz_gpu_match_seam_device, sqz_gpu_parse_exit_map_device_ex, sqz_gpu_parse_device_ex).  Everything is
checked against the lazy walk over the oracle's table (tests/lazy_oracle.py) and the per-shard maps of
tests/test_lazy_seams.py.  With fewer devices than shards, the shards share device 0."""
import ctypes as C
import errno

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus, shard

from lazy_oracle import lazy_tokens_from_table
from test_gpu_lazy import mixed, oracle_tokens, stream
from test_lazy import LAZY_SIZES
from test_lazy_seams import exit_maps, lazy_steps, positions

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

LAZY, SYMBOLS, SHORT_START = 8, 1, 2
G1 = (1 << 15, 3, 257, 32767)
RULE_SETS = [(1 << 15, 2, 254, 32767), (1 << 15, 4, 16, 32767), (1 << 15, 3, 64, 32767),
             (1 << 15, 3, 257, 1024), (1 << 10, 2, 31, 5)]


def devices_for(world):
    n_dev = torch.cuda.device_count()
    return [g % n_dev for g in range(world)]


def multi(d, devices, flags, rules=G1, out=None):
    """sqz_gpu_tokens_multi_ex: (rc, tokens, per-shard counts); `out` a device tensor to gather into."""
    L = _lib.load()
    d = np.ascontiguousarray(d, dtype=np.uint8)
    devs = (C.c_int * len(devices))(*devices)
    buf = np.empty(max(d.size, 1), np.uint32) if out is None else out
    ptr = buf.ctypes.data if out is None else out.data_ptr()
    n, per = C.c_size_t(), (C.c_size_t * len(devices))()
    rc = L.sqz_gpu_tokens_multi_ex(devs, len(devices), d.ctypes.data_as(_lib.u8p), d.size, *rules, flags, ptr,
                                   max(d.size, 1), C.byref(n), per)
    got = buf[: n.value] if out is None else out[: n.value].cpu().numpy().view(np.uint32)
    return rc, np.array(got, dtype=np.uint32), [int(x) for x in per]


@pytest.mark.parametrize("kernel", [0, 1], ids=["auto", "per_position"])
@pytest.mark.parametrize("rules", RULE_SETS)
def test_one_shot_rule_sets(rules, kernel, inputs, oracle):
    """sq.tokens(lazy=True) == the lazy walk == the concatenated SQZ_GPU_STREAM_LAZY stream."""
    sq.select_kernel(kernel)
    try:
        for d in (inputs["laozi.txt"], inputs["csrc.cat"], mixed(inputs)[:400000]):
            want = oracle_tokens(oracle, d, rules)
            w, mn, mx, md = rules
            got = sq.tokens(d, w, mn, mx, md, lazy=True)
            assert got.size == want.size and (got == want).all(), rules
            streamed, _ = stream(d, 50001, LAZY, rules)
            assert (streamed == got).all()
    finally:
        sq.select_kernel(0)


@pytest.mark.parametrize("name", sorted(LAZY_SIZES))
def test_one_shot_fixtures_and_codec(name, inputs, oracle):
    """On the fixtures: one-shot == stream == walk; the tokens of several devices, coded on the host, are
    sq.compress(lazy=True)'s bytes and decode to the input."""
    d = inputs[name]
    want = oracle_tokens(oracle, d)
    got = sq.tokens(d, lazy=True)
    assert got.size == want.size and (got == want).all()
    assert (stream(d, 0, LAZY)[0] == want).all()
    toks = sq.tokens_multi(d, devices_for(4), lazy=True)
    comp = sq.encode_tokens(toks, d.size, 15)
    assert comp == sq.compress(d, lazy=True) and len(comp) == LAZY_SIZES[name]
    assert sq.decompress(comp) == d.tobytes()


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_multi_equals_one_shot(world, inputs, oracle):
    devices = devices_for(world)
    for name in ["hello", "laozi.txt", "csrc.cat", "x64.elf"]:
        d = inputs[name]
        want = sq.tokens(d, lazy=True)
        got, per = sq.tokens_multi(d, devices, lazy=True, return_shard_counts=True)
        assert got.size == want.size and (got == want).all(), (name, world)
        assert sum(per) == want.size and len(per) == world
    d = corpus.synthetic((3 << 20) + 7, 3276897 - (1 << 20))
    got = sq.tokens_multi(d, devices, lazy=True)
    want = oracle_tokens(oracle, d)
    assert got.size == want.size and (got == want).all()


def test_multi_tiny_inputs_and_empty_shards(oracle):
    """0 and 1 bytes, and fewer bytes than shards: the shards past the first `bytes` ones are empty, the last
    non-empty one reads seam word 0."""
    rng = np.random.default_rng(9)
    for size in (0, 1, 2, 3, 5, 7, 9):
        d = np.tile(np.frombuffer(b"ab", np.uint8), 8)[:size].copy() if size % 2 else rng.integers(0, 2, size, dtype=np.uint8)
        want = oracle_tokens(oracle, d) if size else np.zeros(0, np.uint32)
        for world in (1, 3, 8):
            got, per = sq.tokens_multi(d, devices_for(world), lazy=True, return_shard_counts=True)
            assert got.size == want.size and (got == want).all(), (size, world)
            assert sum(per) == want.size and all(c == 0 for c in per[size:])
        assert (sq.tokens(d, lazy=True) == want).all()


def test_multi_gathers_on_a_device():
    """tokens_out in device memory: the lazy shards' tokens concatenated there by peer copies."""
    d = corpus.synthetic(2 << 20, 12345)
    want = sq.tokens(d, lazy=True)
    for world in (2, 4):
        out = torch.zeros(d.size, dtype=torch.int32, device="cuda:0")
        rc, got, per = multi(d, devices_for(world), LAZY, out=out)
        assert rc == 0, _lib.load().sqz_gpu_last_error()
        assert got.size == want.size and (got == want).all() and sum(per) == want.size


def multi_seam_input(total, world, seed, control):
    """Random bytes, and at every cut sqz_gpu_tokens_multi makes (shards of total // world bytes, the first
    total % world one byte longer) a match of 11 at n - 1 whose next position starts a match of 40: lazy and
    greedy decide differently right at the seam, where the lazy step reads the next shard's first word.  At
    the cut `control` position n starts a match of only 10: both take the 11."""
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 256, total, dtype=np.uint8)
    base, extra = divmod(total, world)
    cuts = np.cumsum([base + (1 if g < extra else 0) for g in range(world)])[:-1].tolist()
    for k, n in enumerate(cuts):
        unit = rng.integers(0, 256, 40, dtype=np.uint8)
        x = rng.integers(0, 256, 1, dtype=np.uint8)
        d[n - 2000: n - 1989] = np.concatenate([x, unit[:10]])           # the 11 for position n - 1
        if k == control:
            d[n - 1: n + 10] = np.concatenate([x, unit[:10]])
            d[n + 10] = unit[10] ^ 0xFF
        else:
            d[n - 3000: n - 2960] = unit                                  # the 40 for position n
            d[n - 1: n + 40] = np.concatenate([x, unit])
            d[n + 40] = unit[10] ^ 0xFF                                   # neither match runs on
    return d, cuts


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_multi_seams_that_hold_a_lazy_decision(world, oracle):
    total = world * 20011 + world - 1
    control = world // 2 - 1 if world > 2 else -1
    d, cuts = multi_seam_input(total, world, 100 + world, control)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    lazy_want, _ = lazy_tokens_from_table(d, ln, ds, 3)
    greedy_want, _ = oracle.tokens_from_table(d, ln, ds, 3)
    visited = set(positions(lazy_want).tolist())
    for k, n in enumerate(cuts):
        assert ln[n - 1] == 11 and n - 1 in visited, (k, n)
        assert ln[n] == (10 if k == control else 40), (k, ln[n])
    devices = devices_for(world)
    lazy = sq.tokens_multi(d, devices, lazy=True)
    greedy = sq.tokens_multi(d, devices)
    assert lazy.size == lazy_want.size and (lazy == lazy_want).all()
    assert greedy.size == greedy_want.size and (greedy == greedy_want).all()
    at_lazy = dict(zip(positions(lazy).tolist(), lazy.tolist()))
    at_greedy = dict(zip(positions(greedy).tolist(), greedy.tolist()))
    for k, n in enumerate(cuts):
        assert at_greedy[n - 1] >> 16 == 11
        if k == control:
            assert at_lazy[n - 1] >> 16 == 11 and n not in at_lazy
        else:
            assert at_lazy[n - 1] == d[n - 1] and at_lazy[n] >> 16 == 40 and n not in at_greedy


@pytest.mark.parametrize("world", [2, 3, 8])
def test_device_buffer_hand_off(world, oracle):
    """The one-process-per-device path: match_table(seam=True), lazy exit maps == the CPU maps for every
    entry, chained; every shard parsed from its entry overshoots into the next entry; tokens and symbol words
    concatenated == the lazy walk and its symbol words."""
    from sqz_b200 import device
    total = 200000
    d, _ = multi_seam_input(total, world, 7, -1)           # the cuts of shard.plan are those of tokens_multi
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    whole, _ = lazy_tokens_from_table(d, ln, ds, 3)
    buf = torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    plan = shard.plan(total, world, 32767, 257)
    cpu_maps = exit_maps(lazy_steps(ln, 3), plan, 257)
    tables, maps = [], []
    for s, want_map in zip(plan, cpu_maps):
        t = device.match_table(buf, s.first, s.n, s.back, s.ahead, seam=True)
        assert t.numel() == s.n + 1
        w = t.cpu().numpy().view(np.uint32)
        q = s.first + s.n
        assert w[s.n] == (0 if q == total else int(ln[q]) << 16 | int(ds[q]))
        m = device.exit_map(t, s.n, lazy=True).cpu().numpy().view(np.uint16)[:257]
        assert (m == want_map).all(), (s, np.nonzero(m != want_map)[0][:5])
        tables.append(t)
        maps.append(m)
    entries = shard.chain_entries(maps)
    assert entries[-1] == 0
    parts, words = [], []
    for s, t, e in zip(plan, tables, entries):
        tok, over = device.parse(buf, s.first, t, s.n, e, lazy=True)
        assert over == entries[s.rank + 1]
        parts.append(tok.cpu().numpy().view(np.uint32))
        sym, over = device.parse(buf, s.first, t, s.n, e, symbols=True, lazy=True)
        assert over == entries[s.rank + 1]
        words.append(sym.cpu().numpy().view(np.uint32))
    cat = np.concatenate(parts)
    assert cat.size == whole.size and (cat == whole).all()
    assert (np.concatenate(words) == sq.symbols_of_tokens(whole)).all()
    with pytest.raises(ValueError):
        device.parse(buf, plan[0].first, tables[0][: plan[0].n], plan[0].n, 0, lazy=True)


def seam_test_input():
    """Random bytes with runs of period 3 and 4, the last 700 bytes of period 4: near the end every match
    runs to the end of the input, which is the last byte of the look-ahead halo."""
    rng = np.random.default_rng(21)
    parts = [rng.integers(0, 256, 6000, dtype=np.uint8), np.tile(rng.integers(0, 256, 3, dtype=np.uint8), 700),
             rng.integers(0, 256, 999, dtype=np.uint8), np.tile(rng.integers(0, 256, 37, dtype=np.uint8), 40),
             rng.integers(0, 256, 301, dtype=np.uint8), np.tile(rng.integers(0, 256, 4, dtype=np.uint8), 175)]
    return np.concatenate(parts)


@pytest.mark.parametrize("rules", [G1, (1 << 15, 2, 254, 32767), (1 << 10, 2, 31, 5), (1 << 10, 3, 257, 1023)])
def test_match_seam_device(rules, oracle):
    """sqz_gpu_match_seam_device alone: the word at n == oracle A at the seam position, for a shard given
    nothing but its own bytes and halos; seam matches that run to the last halo byte; 0 at the end."""
    L = _lib.load()
    d = seam_test_input()
    total = d.size
    window, mn, mx, md = rules
    seams = [1, 2, 100, 6001, 8050, total - 700, total - mx - 1, total - mx, total - 100, total - 2, total - 1, total]
    reached = 0
    for q in seams:
        n = min(q, 3000)
        first = q - n
        back, ahead = min(first, md), min(total - q, mx)
        lo, hi = first - back, q + ahead
        buf = torch.zeros(hi - lo + 3 + 64, dtype=torch.uint8, device="cuda")
        buf[3:3 + hi - lo] = torch.from_numpy(d[lo:hi].copy()).cuda()
        out = torch.full((n + 1,), -1, dtype=torch.int32, device="cuda")
        rc = L.sqz_gpu_match_seam_device(buf.data_ptr() + 3 + back, back, n, ahead, mn, mx, md, out.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream)
        assert rc == 0, L.sqz_gpu_last_error()
        w = out.cpu().numpy().view(np.uint32)
        assert (w[:n] == 0xFFFFFFFF).all()                      # nothing but word n is written
        if q == total:
            assert w[n] == 0
            continue
        oln, ods = oracle.match_table(d, window, first=q, count=1, min_len=mn, max_len=mx, max_dist=md)
        assert w[n] == ((int(oln[0]) << 16) | int(ods[0])), (rules, q, w[n] >> 16, w[n] & 0xFFFF, oln[0], ods[0])
        reached += int(oln[0]) == ahead and ahead > 0
    assert reached >= 3                                         # matches up to the last halo byte


def test_256_mib_in_4_and_8_shards(oracle):
    """256 MiB of the bench corpus: two chunks of the one-shot call, 4 and 8 shards, the lazy walk over
    oracle B."""
    d = corpus.synthetic(256 << 20, 0)
    ln, ds = oracle.match_table(d, 1 << 15, fast=True)
    want, end = lazy_tokens_from_table(d, ln, ds, 3)
    del ln, ds
    assert end == d.size
    one = sq.tokens(d, lazy=True)
    assert one.size == want.size and (one == want).all()
    del one
    for world in (4, 8):
        got, per = sq.tokens_multi(d, devices_for(world), lazy=True, return_shard_counts=True)
        assert got.size == want.size and (got == want).all() and sum(per) == want.size, world
        del got


def test_flags_and_the_old_entry_points():
    """Bits an entry point does not take are EINVAL; flags = 0 (and SYMBOLS for the parse) of every _ex entry
    point gives what the old one gives, bit for bit and with as many kernel launches."""
    from sqz_b200 import device
    L = _lib.load()
    d = corpus.synthetic(1 << 20, 777)
    p8 = d.ctypes.data_as(_lib.u8p)
    out = np.zeros(d.size, np.uint32)
    n = C.c_size_t()
    devs = (C.c_int * 2)(0, 0)
    for bad in (SYMBOLS, SHORT_START, 4, 16, LAZY | SYMBOLS, 1 << 31):
        assert L.sqz_gpu_tokens_ex(p8, d.size, *G1, bad, out.ctypes.data_as(_lib.u32p), out.size, C.byref(n)) == errno.EINVAL
        assert L.sqz_gpu_tokens_multi_ex(devs, 2, p8, d.size, *G1, bad, out.ctypes.data, out.size, C.byref(n),
                                         None) == errno.EINVAL
    # host calls
    k0 = sq.launch_count()
    assert L.sqz_gpu_tokens(p8, d.size, *G1, out.ctypes.data_as(_lib.u32p), out.size, C.byref(n)) == 0
    old, k1 = out[: n.value].copy(), sq.launch_count()
    assert L.sqz_gpu_tokens_ex(p8, d.size, *G1, 0, out.ctypes.data_as(_lib.u32p), out.size, C.byref(n)) == 0
    assert (out[: n.value] == old).all() and sq.launch_count() - k1 == k1 - k0
    assert L.sqz_gpu_tokens_multi(devs, 2, p8, d.size, *G1, out.ctypes.data, out.size, C.byref(n), None) == 0
    assert (out[: n.value] == old).all()
    rc, got, _ = multi(d, [0, 0], 0)
    assert rc == 0 and (got == old).all()
    # device calls, on one shard of the whole input
    buf = torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    t = device.match_table(buf, 0, d.size, 0, 0, seam=True)
    work = torch.empty(L.sqz_gpu_parse_workspace(d.size), dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream

    def parse(fn, *flags, min_len=3):
        o = torch.zeros(d.size, dtype=torch.int32, device="cuda")
        r = torch.zeros(2, dtype=torch.int64, device="cuda")
        k = sq.launch_count()
        rc = fn(buf.data_ptr(), t.data_ptr(), d.size, 0, min_len, 257, *flags, o.data_ptr(), d.size, work.data_ptr(),
                r.data_ptr(), s)
        torch.cuda.synchronize()
        return rc, o.cpu().numpy(), r.cpu().numpy(), sq.launch_count() - k

    def exit_map(fn, *flags):
        o = torch.zeros(512, dtype=torch.int16, device="cuda")
        k = sq.launch_count()
        rc = fn(t.data_ptr(), d.size, 3, 257, *flags, work.data_ptr(), o.data_ptr(), s)
        torch.cuda.synchronize()
        return rc, o.cpu().numpy(), sq.launch_count() - k

    for a, b in ((parse(L.sqz_gpu_parse_device), parse(L.sqz_gpu_parse_device_ex, 0)),
                 (parse(L.sqz_gpu_parse_symbols_device), parse(L.sqz_gpu_parse_device_ex, SYMBOLS)),
                 (exit_map(L.sqz_gpu_parse_exit_map_device), exit_map(L.sqz_gpu_parse_exit_map_device_ex, 0))):
        assert a[0] == 0 and b[0] == 0
        assert all((x == y).all() for x, y in zip(a[1:-1], b[1:-1])) and a[-1] == b[-1]
    assert (parse(L.sqz_gpu_parse_device)[1][: int(parse(L.sqz_gpu_parse_device)[2][0])].view(np.uint32) == old).all()
    for bad in (SHORT_START, 4, 16, 1 << 31):
        assert parse(L.sqz_gpu_parse_device_ex, bad)[0] == errno.EINVAL
    for bad in (SYMBOLS, SHORT_START, 4, 16, LAZY | SYMBOLS):
        assert exit_map(L.sqz_gpu_parse_exit_map_device_ex, bad)[0] == errno.EINVAL
    # SYMBOLS keeps the limits of symbol words, with or without LAZY
    for flags in (SYMBOLS, SYMBOLS | LAZY):
        assert parse(L.sqz_gpu_parse_device_ex, flags, min_len=2)[0] == errno.EINVAL
    assert L.sqz_gpu_match_seam_device(buf.data_ptr(), 0, 10, 5, 3, 600, 100, t.data_ptr(), s) == errno.EINVAL
