"""The decoder's copy phase on the GPU (lz_expand.cuh) at its seams, chains and size limits, against the
reference's byte-by-byte execution of the same tokens (tests/lz_reference.py):

- token counts at the warp, row and block seams of the length scan, and past 1024 scan blocks, where
  every thread of `scan_blocks` sums more than one block;
- rows and blocks of len-65535 matches (the widest row and block sums of `place_tokens`);
- token streams of rules the bitstream cannot carry (len up to 512, dist up to 65535, min_len 1 and 2,
  lazy parses);
- chains of pointer doubling that end 2^31 - 2 bytes back, the largest hop below the `kLanded` bit;
- bad tokens at every seam of `place_tokens`' offsets, literal words above 0xFF, wrong sizes;
- the device entry point on a side stream with a dirty, reused workspace;
- sqz_decompress_gpu at every window, on empty, tiny and corrupt streams."""
import ctypes as C
import errno

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

from lz_reference import execute, expand, stream_of_bytes, stream_of_count, stream_of_lengths
from test_gpu_expand import NAMES
from test_gpu_lazy import LAZY, stream

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

BLOCK = 2048                  # tokens per block of the length scan (expand::kScanBlock)
LIMIT = (1 << 31) - 1         # the largest output of one call


def gpu_expand(toks, nbytes, out=None):
    """(return code, out) of sqz_gpu_expand_tokens, called directly: the wrapper would raise, and would
    copy the output once more."""
    t = np.ascontiguousarray(toks, dtype=np.uint32)
    if out is None:
        out = np.empty(max(nbytes, 1), dtype=np.uint8)
    rc = _lib.load().sqz_gpu_expand_tokens(t.ctypes.data_as(_lib.u32p), t.size, out.ctypes.data_as(_lib.u8p), nbytes)
    return rc, out


def last_error() -> str:
    return (_lib.load().sqz_gpu_last_error() or b"").decode(errors="replace")


def assert_same(got, want, what):
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, (what, "bytes differ at", bad[:5], got[bad[:5]], want[bad[:5]])


def check(toks, nbytes, what):
    """sqz_gpu_expand_tokens == lz_execute on a valid stream."""
    want = expand(toks, nbytes)
    rc, got = gpu_expand(toks, nbytes)
    assert rc == 0, (what, rc, last_error())
    assert_same(got[:nbytes], want, what)


# ---- token counts at the seams of the length scan --------------------------------------------------

COUNTS = [1, 31, 32, 33, 255, 256, 257, 2047, 2048, 2049,
          BLOCK * 1024 - 1, BLOCK * 1024, BLOCK * 1024 + 1, 3 * BLOCK * 1024 + 5]
MIXES = [dict(), dict(lit=0.05, long=0.01, overlap=0.8), dict(lit=0.9, overlap=0.0), dict(lit=0.3, max_dist=7)]


@pytest.mark.parametrize("n_tokens", COUNTS)
def test_token_count_seams(n_tokens):
    blocks = (n_tokens + BLOCK - 1) // BLOCK
    if n_tokens > BLOCK * 1024:
        assert blocks > 1024               # scan_blocks: every thread sums more than one block
    mixes = MIXES if n_tokens < BLOCK * 1024 else MIXES[:1]
    for k, mix in enumerate(mixes):
        toks, n = stream_of_count(n_tokens * 8 + k, n_tokens, **mix)
        assert toks.size == n_tokens
        check(toks, n, (n_tokens, mix))


def test_rows_and_blocks_of_the_longest_matches():
    """One warp row (tokens 128..159 of block 0) and all 2048 tokens of block 1 are len-65535 matches,
    with literals around them: a row spans 2 MiB, a block 134 MB, the largest sums of place_tokens."""
    ln = np.zeros(3 * BLOCK + 100, np.int64)
    ln[128:160] = 65535
    ln[BLOCK:2 * BLOCK] = 65535
    ln[2 * BLOCK + 7::97] = 65535
    for seed, overlap in ((1, 0.3), (2, 1.0)):
        toks, n = stream_of_lengths(seed, ln, overlap)
        assert n > BLOCK * 65535
        check(toks, n, (seed, overlap))


# ---- token streams the bitstream cannot carry -------------------------------------------------------

WIDE_RULES = [(1 << 16, 3, 512, 65535), (1 << 16, 3, 300, 40000), (1 << 15, 2, 254, 32767), (1 << 15, 1, 8, 300)]


@pytest.mark.parametrize("rules", WIDE_RULES, ids=lambda r: "w%d_%d_%d_%d" % (r[0].bit_length() - 1, *r[1:]))
def test_rules_beyond_the_bitstream(rules, inputs):
    window, mn, mx, md = rules
    for name in NAMES + ["csrc.cat"]:
        d = inputs[name]
        assert sq.expand_tokens(sq.tokens(d, *rules), d.size) == d.tobytes(), (rules, name)
    d = corpus.synthetic(3 << 20, 777777)
    t = sq.tokens(d, *rules)
    ln, ds = t >> 16, t & 0xFFFF
    if mx > 257:                          # the stream really has what the bitstream cannot carry
        assert (ln > 257).any() and (ds[ln > 0] > 32767).any()
    if mn == 1:
        assert (ln == 1).any()
    assert sq.expand_tokens(t, d.size) == d.tobytes(), rules


@pytest.mark.parametrize("rules,flags", [((1 << 15, 3, 257, 32767), LAZY), ((1 << 15, 2, 254, 32767), LAZY),
                                         ((1 << 15, 2, 254, 32767), 0), ((1 << 10, 2, 31, 5), LAZY)])
def test_streamed_tokens(rules, flags, inputs):
    """The pipeline's tokens: lazy parses, min_len 2."""
    for d in [inputs[n] for n in ("laozi.txt", "x64.elf", "mandrill.bmp", "abc40")] + [corpus.synthetic(5 << 20, 31)]:
        t, _ = stream(d, 0, flags, rules)
        assert sq.expand_tokens(t, d.size) == d.tobytes(), (rules, flags, d.size)


# ---- chains at the size limit -----------------------------------------------------------------------

def _memory_or_skip():
    free, _ = torch.cuda.mem_get_info()
    if free < (11 << 30):
        pytest.skip("needs 11 GiB of free device memory (output and hops of a 2 GiB call)")
    avail = None
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    avail = int(line.split()[1]) << 10
    except OSError:
        pass
    if avail is not None and avail < (6 << 30):
        pytest.skip("needs 6 GiB of host memory (the output and the reference's)")


@pytest.mark.parametrize("prefix,dist", [(1, 1), (3, 3), (65535, 65535)])
def test_chains_at_the_size_limit(prefix, dist):
    """`prefix` literals, then len-65535 matches at `dist` up to 2^31 - 1 bytes.  With dist 1 the last
    byte's hop is 2^31 - 2, the largest below kLanded, reached after 31 rounds of plain doubling."""
    _memory_or_skip()
    lits = np.random.default_rng(prefix).integers(0, 256, prefix).astype(np.uint32)
    full, tail = divmod(LIMIT - prefix, 65535)
    toks = np.concatenate([lits, np.full(full, (65535 << 16) | dist, np.uint32),
                           np.array([(tail << 16) | dist] if tail else [], np.uint32)])
    rc, got = gpu_expand(toks, LIMIT, np.empty(LIMIT, np.uint8))
    assert rc == 0, last_error()
    step = 1 << 28
    if dist == 1:
        for lo in range(0, LIMIT, step):
            assert (got[lo:lo + step] == lits[0]).all(), lo
    else:
        code, want = execute(toks, LIMIT, np.empty(LIMIT, np.uint8))
        assert code == 0
        for lo in range(0, LIMIT, step):
            assert_same(got[lo:lo + step], want[lo:lo + step], (prefix, dist, lo))


def test_two_gib_and_more_are_refused_before_anything_is_allocated():
    """The host entry points refuse 2^31 bytes and more with EINVAL, not an allocation error."""
    L = _lib.load()
    toks = np.array([65, 66, 67], np.uint32)
    out = np.zeros(64, np.uint8)
    for nbytes in (1 << 31, 1 << 40):
        rc = L.sqz_gpu_expand_tokens(toks.ctypes.data_as(_lib.u32p), toks.size, out.ctypes.data_as(_lib.u8p), nbytes)
        assert rc == errno.EINVAL and "2 GiB" in last_error(), (nbytes, rc, last_error())
        # sqz_decompress_gpu on a stream whose header announces that size
        comp = np.frombuffer(sq.compress(b"AB", 15), np.uint8).copy()
        head = np.zeros(16, np.uint8)                      # the header's first word: the size
        bs = _lib.Bitstream()
        bs.data = head.ctypes.data_as(_lib.u8p)
        bs.capacity = head.size
        L.sqz_write_header(C.byref(bs), nbytes, 15)
        assert bs.error == 0 and bs.bytes == 8
        comp[:8] = head[:8]
        assert sq.read_header(comp) == (nbytes, 15)
        bs = _lib.Bitstream()
        bs.data = comp.ctypes.data_as(_lib.u8p)
        bs.capacity = bs.bytes = comp.size
        n, wb = C.c_uint64(), C.c_uint8()
        L.sqz_read_header(C.byref(bs), C.byref(n), C.byref(wb))
        s = _lib.State()
        L.sqz_init(C.byref(s))
        L.sqz_decompress_gpu(C.byref(s), C.byref(bs), out.ctypes.data_as(_lib.u8p), n.value)
        assert s.error == errno.EINVAL, (nbytes, s.error)
    for n_tokens, nbytes in ((3, 2), (1, 0), (0, 5)):      # more tokens than bytes; none for some bytes
        rc = L.sqz_gpu_expand_tokens(toks.ctypes.data_as(_lib.u32p), n_tokens, out.ctypes.data_as(_lib.u8p), nbytes)
        assert rc == errno.EINVAL, (n_tokens, nbytes)
    assert gpu_expand(toks[:0], 0)[0] == 0
    check(toks, 3, "after the refusals")


# ---- bad tokens at every seam -----------------------------------------------------------------------

N_LIT = 5000
SEAMS = [0, 1, 31, 32, 255, 256, 2047, 2048, 2049, N_LIT - 1]


@pytest.mark.parametrize("k", SEAMS)
def test_bad_tokens_at_every_seam(k):
    """An all-literal stream (output offset == token index) with token k replaced.  A len-3 match adds
    2 bytes, and the announced size is the changed stream's."""
    lits = np.random.default_rng(k).integers(0, 256, N_LIT).astype(np.uint32)
    cases = [((3 << 16) | (k + 1), N_LIT + 2, False),      # one byte before byte 0
             ((3 << 16) | 0, N_LIT + 2, False),            # dist 0
             (0x100 | int(lits[k]), N_LIT, False),          # a literal word above 0xFF
             (0xFF00 | int(lits[k]), N_LIT, False)]
    if k >= 1:
        cases.append(((3 << 16) | k, N_LIT + 2, True))     # reaches byte 0 exactly
    else:
        cases.append((int(lits[0]), N_LIT, True))
    for word, n, valid in cases:
        t = lits.copy()
        t[k] = word
        code, want = execute(t, n)
        rc, got = gpu_expand(t, n)
        if valid:
            assert code == 0 and rc == 0, (k, hex(word), rc, last_error())
            assert_same(got[:n], want[:n], (k, hex(word)))
            for m in (n - 1, n + 1):                       # the announced size off by one
                assert execute(t, m)[0] != 0
                rc, _ = gpu_expand(t, m)
                assert rc == errno.EINVAL, (k, hex(word), m)
                check(lits, N_LIT, ("after a refusal", k, m))
        else:
            assert code == 1 + k, (k, hex(word), code)
            assert rc == errno.EINVAL, (k, hex(word), rc)
            check(lits, N_LIT, ("after a refusal", k, hex(word)))


def test_symbol_words_are_refused(inputs):
    """Symbol words (SQZ_GPU_STREAM_SYMBOLS) are not tokens: the word of a match at dist 1..4 has
    bits 16..31 zero and would pass for a literal above 0xFF."""
    d = inputs["zeros4096"]
    w = sq.symbols_of_tokens(sq.tokens(d))
    assert (w >> 16 == 0).all() and (w > 0xFF).any()
    assert execute(w, w.size)[0] != 0
    with pytest.raises(sq.SqzError) as e:
        sq.expand_tokens(w, w.size)
    assert e.value.errno == errno.EINVAL


# ---- the device entry point -------------------------------------------------------------------------

def _expand_device(toks, n, work, stream_, device):
    """sqz_gpu_expand_tokens_device on `stream_`, output in a 0xAA-filled buffer 4096 bytes too long;
    the return code and the bytes are read after the stream is synchronised."""
    L = _lib.load()
    d_tok = torch.from_numpy(toks.view(np.int32)).to(device)
    out = torch.full((n + 4096,), 0xAA, dtype=torch.uint8, device=device)
    torch.cuda.synchronize(device)
    rc = L.sqz_gpu_expand_tokens_device(d_tok.data_ptr(), toks.size, out.data_ptr(), n, work.data_ptr(),
                                        stream_.cuda_stream)
    stream_.synchronize()
    assert rc == 0, last_error()
    got = out.cpu().numpy()
    assert_same(got[:n], expand(toks, n), ("device entry point", toks.size, n))
    assert (got[n:] == 0xAA).all(), "bytes past `bytes` were written"


def test_device_entry_point_on_a_side_stream():
    L = _lib.load()
    big, n_big = stream_of_count(21, 3 * BLOCK * 64 + 17, long=0.001, overlap=0.5)
    small, n_small = stream_of_count(22, 700)
    work = torch.full((L.sqz_gpu_expand_workspace(big.size, n_big),), 0xFF, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    assert side.cuda_stream != torch.cuda.default_stream().cuda_stream
    for toks, n in ((big, n_big), (small, n_small), (big, n_big)):   # the same workspace, dirty, again
        _expand_device(toks, n, work, side, "cuda")


def test_calls_keep_the_current_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    L = _lib.load()
    toks, n = stream_of_count(23, 10000)
    comp = sq.compress(corpus.fixtures()["laozi.txt"], 15)
    try:
        torch.cuda.set_device(1)
        work = torch.full((L.sqz_gpu_expand_workspace(toks.size, n),), 0xFF, dtype=torch.uint8, device="cuda:1")
        _expand_device(toks, n, work, torch.cuda.Stream(device=1), "cuda:1")
        assert torch.cuda.current_device() == 1
        check(toks, n, "host entry point on device 1")
        assert torch.cuda.current_device() == 1
        assert sq.decompress_gpu(comp) == sq.decompress(comp)
        assert torch.cuda.current_device() == 1
    finally:
        torch.cuda.set_device(0)


# ---- sqz_decompress_gpu -----------------------------------------------------------------------------

@pytest.mark.parametrize("wb", range(10, 16))
def test_decompress_gpu_at_every_window(wb, inputs):
    big = corpus.synthetic(20 << 20, 4242)
    for name, d in [(n, inputs[n]) for n in NAMES + ["csrc.cat", "empty"]] + [("synthetic", big)]:
        for lazy in (False, True):
            comp = sq.compress(d, wb, lazy=lazy)
            st = {}
            assert sq.decompress_gpu(comp, stats=st) == d.tobytes() == sq.decompress(comp), (name, wb, lazy)
            assert st["tokens"] == sq.decode_tokens(comp).size


def test_decompress_gpu_empty_and_one_byte():
    for d in (b"", b"x", b"\0", b"\xff"):
        comp = sq.compress(d, 15)
        assert sq.decompress_gpu(comp) == d == sq.decompress(comp)


def _outcome(fn, comp):
    try:
        return fn(comp)
    except sq.SqzError as e:
        return e.errno


def test_decompress_gpu_on_corrupt_streams(inputs):
    """Streams corrupted as test_codec.test_corrupt_streams_fail_cleanly corrupts them: the GPU path gives
    the host decoder's bytes or its errno."""
    d = inputs["laozi.txt"]
    comp = bytearray(sq.compress(d, 15))
    rng = np.random.default_rng(1)
    bad = 0
    for _ in range(40):
        c = bytearray(comp)
        for k in rng.integers(9, len(c), 3):
            c[k] ^= 1 << int(rng.integers(0, 8))
        want = _outcome(sq.decompress, bytes(c))
        assert _outcome(sq.decompress_gpu, bytes(c)) == want
        bad += isinstance(want, int)
    assert bad > 0
    truncated = bytes(comp[: len(comp) // 2 // 8 * 8])
    c = bytearray(comp)
    c[8] = 0xFF                                            # window byte out of range
    for c in (truncated, bytes(c)):
        want = _outcome(sq.decompress, c)
        assert isinstance(want, int) and _outcome(sq.decompress_gpu, c) == want


# ---- a seeded random sweep --------------------------------------------------------------------------

@pytest.mark.parametrize("seed", range(32))
def test_random_sweep(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(1 << 20, (8 << 20) + 1))
    mix = dict(lit=float(rng.uniform(0.05, 0.9)), long=float(10 ** rng.uniform(-5, -2)),
               overlap=float(rng.uniform(0, 1)), max_dist=int(rng.choice([4, 300, 32767, 65535])))
    toks = stream_of_bytes(seed, n, **mix)
    rc, got = gpu_expand(toks, n)
    assert rc == 0, f"seed {seed}: rc {rc} ({last_error()})"
    want = expand(toks, n)
    bad = np.flatnonzero(got[:n] != want)
    assert bad.size == 0, f"seed {seed} ({n} bytes, {mix}): bytes differ at {bad[:5]}"
