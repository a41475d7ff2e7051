"""GPU parity beyond whole files: rule sets, shards with halos through the device ABI, the
chunked streaming pipeline, seam hand-off, and size-independent properties at larger sizes."""
import errno
import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import corpus, shard
from match_inputs import far_repeat_input

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(params=[2, 1], ids=["bitsliced", "per_position"])
def kernel(request):
    sq.select_kernel(request.param)
    yield request.param
    sq.select_kernel(0)


def unpack(t):
    w = t.cpu().numpy().view(np.uint32)
    return (w >> 16).astype(np.uint16), (w & 0xFFFF).astype(np.uint16)


RULES = [(3, 257, None), (2, 254, None), (2, 254, "window"), (3, 20, None), (3, 40, 100), (2, 31, 5),
         (4, 16, None), (1, 8, 300), (3, 512, None)]


@pytest.mark.parametrize("rules", RULES)
@pytest.mark.parametrize("name,lo,hi", [("laozi.txt", 0, 20760), ("x64.elf", 902000, 926536), ("arm64.elf", 100000, 140000)])
def test_rule_sets(rules, name, lo, hi, inputs, oracle, kernel):
    """min_len / max_len / max_dist are runtime parameters (SURVEY 8a: three rule sets in the reference)."""
    d = np.ascontiguousarray(inputs[name][lo:hi])
    mn, mx, md = rules
    for window in (1 << 10, 1 << 15):
        dist = window if md == "window" else (window - 1 if md is None else md)
        ln, ds = sq.match_table(d, window, mn, mx, dist)
        oln, ods = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=dist)
        bad = np.nonzero((ln != oln) | (ds != ods))[0]
        assert bad.size == 0, (rules, window, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])
        t = sq.tokens(d, window, mn, mx, dist)
        ot, end = oracle.tokens_from_table(d, oln, ods, mn)
        assert end == d.size and t.size == ot.size and (t == ot).all()


def test_rule_set_iii_against_bst_c(inputs, reference):
    d = np.ascontiguousarray(inputs["x64.elf"][904000:909000])
    rl, rd = reference.bst_table(d, 1024)
    ln, ds = sq.match_table(d, 1 << 16, 2, 254, 1024)
    assert (rl == ln).all() and (rd == ds).all()


def test_bad_rules_are_einval():
    import errno
    for args in [(1 << 15, 3, 2, 100), (1 << 15, 0, 10, 100), (1 << 15, 3, 513, 100), (1 << 15, 3, 257, 0),
                 (1 << 16, 3, 257, 65536), (1000, 3, 257, 999), (1 << 10, 3, 257, 2000)]:
        with pytest.raises(sq.SqzError) as e:
            sq.match_table(b"abcabcabcabc", *args)
        assert e.value.errno == errno.EINVAL


@pytest.mark.parametrize("first,n", [(0, 1), (0, 31), (0, 15872), (5, 15873), (40000, 70001), (32767, 4000),
                                     (100001, 15872 * 3), (250000, 33), (299000, 1000)])
def test_shard_with_halos_device_abi(first, n, oracle, kernel):
    """A shard sees only its bytes + halos and must reproduce the whole-buffer table."""
    from sqz_b200 import device
    total = 300000
    data = corpus.synthetic(total, 3276897 - 150000)
    oln, ods = oracle.match_table(data, 1 << 15, fast=True)
    back, ahead = min(first, 32767), min(total - first - n, 257)
    lo, hi = first - back, first + n + ahead
    # hand the kernel nothing but the shard + halos, at an odd address
    buf = torch.zeros(hi - lo + 3 + 64, dtype=torch.uint8, device="cuda")
    buf[3:3 + hi - lo] = torch.from_numpy(data[lo:hi]).cuda()
    t = device.match_table(buf, 3 + back, n, back, ahead)
    ln, ds = unpack(t)
    bad = np.nonzero((ln != oln[first:first + n]) | (ds != ods[first:first + n]))[0]
    assert bad.size == 0, (first, n, bad[:5], ln[bad[:5]], oln[first:first + n][bad[:5]])


@pytest.mark.parametrize("world", [2, 3, 8])
def test_seam_hand_off_between_shards(world, oracle):
    """Shards parsed independently + exit-map chain == one parse of the whole input."""
    from sqz_b200 import device
    total = 200000
    data = corpus.synthetic(total, 1000)
    whole = oracle.tokens_from_table(data, *oracle.match_table(data, 1 << 15, fast=True))[0]
    dev = torch.from_numpy(data).cuda()
    dev = torch.cat([dev, torch.zeros(64, dtype=torch.uint8, device="cuda")])
    plan = shard.plan(total, world, 32767, 257)
    tables = [device.match_table(dev, s.first, s.n, s.back, s.ahead) for s in plan]
    maps = [device.exit_map(t, s.n).cpu().numpy().view(np.uint16) for t, s in zip(tables, plan)]
    entries = shard.chain_entries(maps)
    assert entries[-1] == 0
    parts, words = [], []
    for s, t, e in zip(plan, tables, entries):
        tok, over = device.parse(dev, s.first, t, s.n, e)
        assert over == entries[s.rank + 1]
        parts.append(tok.cpu().numpy().view(np.uint32))
        sym, over = device.parse(dev, s.first, t, s.n, e, symbols=True)
        assert over == entries[s.rank + 1]
        words.append(sym.cpu().numpy().view(np.uint32))
    cat = np.concatenate(parts)
    assert cat.size == whole.size and (cat == whole).all()
    # symbol words from the GPU, entropy-coded, == the bytes the reference's own encoder
    # (squeeze_encode_len/pos/literal, squeeze.h:278-315) makes of the same token stream
    from oracle import Reference
    if Reference.available():
        assert sq.encode_symbols(np.concatenate(words), total, 15) == Reference.get().encode_tokens(whole, total, 15)
    assert (np.concatenate(words) == sq.symbols_of_tokens(whole)).all()


def test_symbol_words_cover_every_bucket():
    """Every length 3..257 and distances over every bucket edge, through the GPU emit kernel."""
    from sqz_b200 import device
    rng = np.random.default_rng(11)
    pieces = []
    for ln in list(range(3, 40)) + [41, 42, 43, 50, 51, 58, 59, 66, 67, 82, 83, 98, 99, 114, 115, 130, 131, 162,
                                    163, 194, 195, 226, 227, 256, 257]:
        for gap in (0, 1, 2, 3, 4, 5, 7, 12, 23, 40, 100, 500, 3000, 9000, 30000):
            unit = rng.integers(0, 256, ln, dtype=np.uint8)
            pieces += [unit, rng.integers(0, 256, gap + 1, dtype=np.uint8), unit, rng.integers(0, 256, 3, dtype=np.uint8)]
    data = np.concatenate(pieces)[: 6 << 20]
    whole = oracle_tokens_fast(data)
    dev = torch.cat([torch.from_numpy(data).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    t = device.match_table(dev, 0, data.size, 0, 0)
    sym, over = device.parse(dev, 0, t, data.size, 0, symbols=True)
    assert over == 0
    got = sym.cpu().numpy().view(np.uint32)
    # pinned to the reference: the GPU's words through the coder == the reference's encoder on the tokens
    from oracle import Reference
    if Reference.available():
        assert sq.encode_symbols(got, data.size, 15) == Reference.get().encode_tokens(whole, data.size, 15)
    want = sq.symbols_of_tokens(whole)
    assert got.size == want.size and (got == want).all()
    lens = set((whole[whole > 0xFFFF] >> 16).tolist())
    assert {3, 10, 11, 18, 19, 34, 35, 66, 67, 130, 131, 226, 227, 257} <= lens


def oracle_tokens_fast(data):
    from oracle import Oracle
    o = Oracle.get()
    return o.tokens_from_table(data, *o.match_table(data, 1 << 15, fast=True))[0]


@pytest.mark.parametrize("flags", [0, 1], ids=["tokens", "symbols"])
@pytest.mark.parametrize("chunk", [4096, 50001, 65536, 1 << 20])
def test_streaming_pipeline_chunk_sizes(chunk, flags, inputs, oracle):
    """sqz_gpu_stream_*: any chunking of the input gives the same token stream; in symbols mode
    (SQZ_GPU_STREAM_SYMBOLS) the words equal the host statement of squeeze.h:290-315."""
    import ctypes as C
    from sqz_b200 import _lib
    L = _lib.load()
    d = np.concatenate([inputs["confucius.txt"], inputs["x64.elf"][:200000], inputs["mandrill.bmp"][:50000]])
    want = oracle.tokens_from_table(d, *oracle.match_table(d, 1 << 15, fast=True))[0]
    st = C.c_void_p()
    if flags:
        want = sq.symbols_of_tokens(want)
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767, chunk,
                               flags)
    assert rc == 0, L.sqz_gpu_last_error()
    got = []
    while True:
        p, n = _lib.u32p(), C.c_size_t()
        rc = L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n))
        assert rc == 0, L.sqz_gpu_last_error()
        if n.value == 0:
            break
        got.append(np.ctypeslib.as_array(p, shape=(n.value,)).copy())
    L.sqz_gpu_stream_close(st)
    got = np.concatenate(got)
    assert got.size == want.size and (got == want).all()


def test_streaming_pipeline_short_start_and_flags(oracle):
    """SQZ_GPU_STREAM_SHORT_START: explicit chunks of 4 MiB, the first two 1 and 2 MiB (what sqz_compress
    asks for when it codes with a crew) -- the same symbol words, chunk sizes as described; a flag nobody
    defined is refused."""
    import ctypes as C
    from sqz_b200 import _lib, corpus
    L = _lib.load()
    d = corpus.synthetic(11 << 20, 7 << 20)
    want = sq.symbols_of_tokens(sq.tokens(d))
    st = C.c_void_p()
    assert L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767, 4 << 20, 4) == errno.EINVAL
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767, 4 << 20, 1 | 2)
    assert rc == 0, L.sqz_gpu_last_error()
    got = []
    while True:
        p, n = _lib.u32p(), C.c_size_t()
        rc = L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n))
        assert rc == 0, L.sqz_gpu_last_error()
        if n.value == 0:
            break
        got.append(np.ctypeslib.as_array(p, shape=(n.value,)).copy())
    L.sqz_gpu_stream_close(st)
    assert len(got) == 4                                   # 1 + 2 + 4 + 4 MiB
    assert got[0].size < got[1].size < got[2].size
    got = np.concatenate(got)
    assert got.size == want.size and (got == want).all()


def lz77_decode(tokens, n):
    """Independent check of a token stream: plain LZ77 expansion."""
    out = np.zeros(n, np.uint8)
    i = 0
    for t in tokens.tolist():
        ln, ds = t >> 16, t & 0xFFFF
        if ln == 0:
            out[i] = t
            i += 1
        else:
            for k in range(ln):
                out[i + k] = out[i + k - ds]
            i += ln
    assert i == n
    return out


def test_tokens_expand_to_the_input(inputs):
    d = np.concatenate([inputs["laozi.txt"], inputs["arm64.elf"][820000:]])
    assert (lz77_decode(sq.tokens(d), d.size) == d).all()


def test_large_synthetic_full_table_and_round_trip(oracle, reference):
    """48 MiB of the bench corpus (two pipeline chunks): full table == oracle B, the compressed
    stream round-trips through OUR decoder and through the REFERENCE decoder, and its size is
    the size the reference's own encoder produces for the oracle's tokens."""
    n = 48 << 20
    d = corpus.synthetic(n, 0)
    ln, ds = sq.match_table(d)
    oln, ods = oracle.match_table(d, 1 << 15, fast=True)
    assert (ln == oln).all() and (ds == ods).all()
    t = sq.tokens(d)
    ot, end = oracle.tokens_from_table(d, oln, ods)
    assert end == n and t.size == ot.size and (t == ot).all()
    part = np.ascontiguousarray(d[: 6 << 20])
    stats = {}
    comp = sq.compress(part, 15, stats=stats)
    assert stats["tokens"] > 0 and sq.decompress(comp) == part.tobytes()
    assert reference.decompress(comp) == part.tobytes()
    pt = sq.tokens(part)
    assert reference.encode_tokens(pt, part.size, 15) == comp


def test_sampled_positions_against_the_brute_force_oracle(oracle):
    """Oracle A (the restated reference loop) on seeded-random positions and around seams."""
    n = 8 << 20
    d = corpus.synthetic(n, 5 * 3276897 - (4 << 20))
    ln, ds = sq.match_table(d)
    rng = np.random.default_rng(3)
    pos = np.unique(np.concatenate([rng.integers(0, n, 1500), np.arange(0, 300), np.arange(n - 300, n),
                                    np.arange((4 << 20) - 150, (4 << 20) + 150)]))
    for i in pos.tolist():
        assert oracle.best(d, i, 1 << 15) == (int(ln[i]), int(ds[i])), i


def _random_input(rng, n):
    kind = rng.integers(0, 6)
    if kind == 0:
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == 1:
        return rng.integers(0, rng.integers(2, 6), n, dtype=np.uint8)
    if kind == 2:                                          # byte runs of random length
        vals = rng.integers(0, 4, n, dtype=np.uint8)
        return np.repeat(vals, rng.integers(1, 600, n))[:n].copy()
    if kind == 3:                                          # periodic with a few defects
        d = np.tile(rng.integers(0, 256, int(rng.integers(1, 300)), dtype=np.uint8), n)[:n].copy()
        d[rng.integers(0, n, max(n // 500, 1))] ^= 1
        return d
    if kind == 4:                                          # zero-rich records
        d = np.zeros(n, np.uint8)
        idx = rng.integers(0, n, n // 12 + 1)
        d[idx] = rng.integers(1, 256, idx.size, dtype=np.uint8)
        return d
    base = corpus.base()
    at = int(rng.integers(0, base.size - n))
    return base[at:at + n].copy()


@pytest.mark.parametrize("seed", range(24))
def test_randomised_inputs_and_rules(seed, oracle, kernel):
    """Seeded fuzz: random structure, random (min_len, max_len, max_dist, window), table + tokens."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.choice([1, 2, 3, 31, 32, 33, 257, 1000, 4064, 16256, 16257, 40000, 70000]))
    d = _random_input(rng, n)
    window = 1 << int(rng.integers(10, 16))
    mn = int(rng.integers(2, 4))
    mx = int(rng.choice([33, 64, 254, 257, 258, 300, 512]))
    md = int(rng.choice([1, 7, 31, 32, 33, 1000, window - 1, window]))
    md = min(md, window, 65535)
    ln, ds = sq.match_table(d, window, mn, mx, md)
    oln, ods = oracle.match_table(d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
    bad = np.nonzero((ln != oln) | (ds != ods))[0]
    assert bad.size == 0, (seed, n, window, mn, mx, md, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])
    if n <= 20000:                                          # and oracle B against the restated reference loop
        aln, ads = oracle.match_table(d, window, min_len=mn, max_len=mx, max_dist=md)
        assert (aln == oln).all() and (ads == ods).all()
    t = sq.tokens(d, window, mn, mx, md)
    ot, end = oracle.tokens_from_table(d, oln, ods, mn)
    assert end == n and t.size == ot.size and (t == ot).all()


@pytest.mark.parametrize("seed", range(6))
def test_far_repeats_fuzz(seed, oracle, kernel):
    """Full table == oracle B on far-repeat inputs, == the brute-force loop on sampled positions."""
    rng = np.random.default_rng(7000 + seed)
    n = int(rng.choice([90000, 200000, 400000]))
    d = far_repeat_input(rng, n)
    ln, ds = sq.match_table(d, 1 << 15)
    oln, ods = oracle.match_table(d, 1 << 15, fast=True)
    bad = np.nonzero((ln != oln) | (ds != ods))[0]
    assert bad.size == 0, (seed, n, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])
    assert ((ln == 257) & (ds >= 30000)).sum() > n // 20
    for i in rng.integers(0, n, 300).tolist():
        assert oracle.best(d, i, 1 << 15) == (int(ln[i]), int(ds[i])), i
    t = sq.tokens(d)
    ot, end = oracle.tokens_from_table(d, oln, ods)
    assert end == n and t.size == ot.size and (t == ot).all()


@pytest.mark.parametrize("mx,md", [(257, 32767), (64, 32767), (40, 5000), (300, 40000), (512, 65535)])
def test_capped_inheritance_other_caps(mx, md, oracle):
    """The far-repeat shortcut of phase 2 depends on max_len (its slack shrinks to max_len - 32)."""
    rng = np.random.default_rng(mx * 7 + md)
    d = far_repeat_input(rng, 150000)
    window = 1 << 16 if md > 32767 else 1 << 15
    ln, ds = sq.match_table(d, window, 3, mx, md)
    oln, ods = oracle.match_table(d, window, fast=True, min_len=3, max_len=mx, max_dist=md)
    bad = np.nonzero((ln != oln) | (ds != ods))[0]
    assert bad.size == 0, (mx, md, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])


def test_symbol_mode_rejects_length_258():
    """max_len 258 has a bucket but no decoder accepts it (squeeze.h:529-545): EINVAL at open time."""
    import ctypes as C, errno
    from sqz_b200 import _lib
    L = _lib.load()
    d = np.zeros(1000, np.uint8)
    st = C.c_void_p()
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 258, 32767, 0, 1)
    assert rc == errno.EINVAL
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767, 0, 1)
    assert rc == 0
    L.sqz_gpu_stream_close(st)


def test_calls_keep_the_current_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    torch.cuda.set_device(0)
    sq.tokens_multi(corpus.fixtures()["laozi.txt"], [1])
    assert torch.cuda.current_device() == 0


@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_tokens_multi_equals_single_device(world, inputs, oracle):
    """sqz_gpu_tokens_multi: the input cut into `world` shards, every shard on a device (all on
    device 0 when the box has fewer), seams chained, tokens concatenated == one parse of the whole."""
    n_dev = torch.cuda.device_count()
    devices = [g % n_dev for g in range(world)]           # fewer devices than shards: they share
    for name in ["hello", "laozi.txt", "csrc.cat", "x64.elf"]:
        d = inputs[name]
        want = sq.tokens(d)
        got, per = sq.tokens_multi(d, devices, return_shard_counts=True)
        assert got.size == want.size and (got == want).all(), (name, world)
        assert sum(per) == want.size and len(per) == world
    d = corpus.synthetic(3 << 20, 3276897 - (1 << 20))
    want = oracle.tokens_from_table(d, *oracle.match_table(d, 1 << 15, fast=True))[0]
    got = sq.tokens_multi(d, devices)
    assert got.size == want.size and (got == want).all()


def test_tokens_multi_gathers_on_a_device():
    """tokens_out in device memory: the shards' tokens are concatenated there by peer copies."""
    import ctypes as C
    from sqz_b200 import _lib
    L = _lib.load()
    n_dev = torch.cuda.device_count()
    devices = list(range(min(n_dev, 4)))
    d = corpus.synthetic(2 << 20, 12345)
    want = sq.tokens(d)
    out = torch.zeros(d.size, dtype=torch.int32, device="cuda:0")
    n = C.c_size_t()
    devs = (C.c_int * len(devices))(*devices)
    rc = L.sqz_gpu_tokens_multi(devs, len(devices), d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767,
                                out.data_ptr(), out.numel(), C.byref(n), None)
    assert rc == 0, L.sqz_gpu_last_error()
    got = out[: n.value].cpu().numpy().view(np.uint32)
    assert got.size == want.size and (got == want).all()


def test_tokens_multi_bad_arguments():
    import ctypes as C, errno
    from sqz_b200 import _lib
    L = _lib.load()
    d = np.zeros(100, np.uint8)
    out = np.zeros(100, np.uint32)
    n = C.c_size_t()
    for devs in ([], [99], [0, -1]):
        arr = (C.c_int * max(len(devs), 1))(*devs)
        rc = L.sqz_gpu_tokens_multi(arr, len(devs), d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767,
                                    out.ctypes.data, out.size, C.byref(n), None)
        assert rc in (errno.EINVAL, errno.ENODEV), devs
    arr = (C.c_int * 1)(0)
    rc = L.sqz_gpu_tokens_multi(arr, 1, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767,
                                out.ctypes.data, 1, C.byref(n), None)
    assert rc == errno.E2BIG and n.value == 2                # a literal and one (99, 1) match


@pytest.mark.parametrize("mib,offset", [(7.3, 0), (9, 1 << 20), (11.5, 3276897)])
def test_shards_of_a_few_waves(mib, offset, oracle):
    """Between one and a few waves of tiles (7.3-11.5 MiB): the unsliced throughput shape (sqz_gpu.cu:
    slice_plan), partial last wave included: full table == oracle B, with and without a look-back halo."""
    from sqz_b200 import device
    n = int(mib * (1 << 20))
    d = corpus.synthetic(n, offset)
    oln, ods = oracle.match_table(d, 1 << 15, fast=True)
    ln, ds = sq.match_table(d)
    bad = np.nonzero((ln != oln) | (ds != ods))[0]
    assert bad.size == 0, (mib, bad[:5], ln[bad[:5]], oln[bad[:5]], ds[bad[:5]], ods[bad[:5]])
    # the same bytes as a shard in the middle of a larger buffer (halos on both sides, no edge tiles)
    first, cnt = 40000, n - 50000
    buf = torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    t = device.match_table(buf, first, cnt, 32767, 257)
    sl, sd = unpack(t)
    bad = np.nonzero((sl != oln[first:first + cnt]) | (sd != ods[first:first + cnt]))[0]
    assert bad.size == 0, (mib, bad[:5])
    tk = sq.tokens(d)
    ot, end = oracle.tokens_from_table(d, oln, ods)
    assert end == n and tk.size == ot.size and (tk == ot).all()


def test_large_device_shard_with_and_without_halos(oracle):
    """The device ABI on a 240 MiB shard (35 waves of tiles), from position 0 and as a shard with halos on
    both sides: full table == oracle B."""
    from sqz_b200 import device
    n = 240 << 20
    d = corpus.synthetic(n, 5 << 20)
    oln, ods = oracle.match_table(d, 1 << 15, fast=True)
    buf = torch.cat([torch.from_numpy(d).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    for first, cnt, back, ahead in ((0, n, 0, 0), (40000, n - 50000, 32767, 257)):
        t = device.match_table(buf, first, cnt, back, ahead)
        sl, sd = unpack(t)
        bad = np.nonzero((sl != oln[first:first + cnt]) | (sd != ods[first:first + cnt]))[0]
        assert bad.size == 0, (first, bad[:5], sl[bad[:5]], oln[first + bad[:5]], sd[bad[:5]], ods[first + bad[:5]])
        del t, sl, sd
