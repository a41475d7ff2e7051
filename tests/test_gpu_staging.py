"""Staging buffers kept between calls (sqz_gpu.cu: Stage and its park list): calls of every entry point,
of many shapes and rules, in one process take back each other's parked stages -- one up to four times
larger, one sized under other rules, one evicted, one whose last work may still be in flight, none after
sqz_gpu_release() -- and every result stays the oracle's."""
import ctypes as C

import numpy as np
import pytest

import sqz_b200 as sq
from sqz_b200 import _lib, corpus

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DEFAULT = (1 << 15, 3, 257, (1 << 15) - 1)
WIDE = (1 << 16, 3, 512, 65535)           # beyond what symbol words can carry
SMALL_WINDOW = (1 << 10, 3, 257, (1 << 10) - 1)


class Case:
    """An input under one set of rules, with the oracle's table and tokens."""

    def __init__(self, oracle, data, rules):
        self.d, self.rules = np.ascontiguousarray(data), rules
        window, mn, mx, md = rules
        self.ln, self.ds = oracle.match_table(self.d, window, fast=True, min_len=mn, max_len=mx, max_dist=md)
        self.tokens, end = oracle.tokens_from_table(self.d, self.ln, self.ds, mn)
        assert end == self.d.size


def stream(d, rules, symbols, read=None):
    """sqz_gpu_stream_* on device 0; `read` chunks at most, then the stream is closed."""
    L = _lib.load()
    st = C.c_void_p()
    rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, *rules, 0, 1 if symbols else 0)
    assert rc == 0, L.sqz_gpu_last_error()
    got = []
    try:
        while read is None or len(got) < read:
            p, n = _lib.u32p(), C.c_size_t()
            rc = L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n))
            assert rc == 0, L.sqz_gpu_last_error()
            if n.value == 0:
                break
            got.append(np.ctypeslib.as_array(p, shape=(n.value,)).copy())
    finally:
        L.sqz_gpu_stream_close(st)
    return got


def device_table(d, rules, stream_=None):
    from sqz_b200 import device
    buf = torch.zeros(d.size + 64, dtype=torch.uint8, device="cuda:0")
    buf[: d.size] = torch.from_numpy(d).cuda()
    window, mn, mx, md = rules
    if stream_ is None:
        return device.match_table(buf, 0, d.size, 0, 0, mn, mx, md)
    stream_.wait_stream(torch.cuda.current_stream())
    buf.record_stream(stream_)          # not handed out again before the search on stream_ has read it
    with torch.cuda.stream(stream_):
        return device.match_table(buf, 0, d.size, 0, 0, mn, mx, md)


def unpack(t):
    w = t.cpu().numpy().view(np.uint32)
    return (w >> 16).astype(np.uint16), (w & 0xFFFF).astype(np.uint16)


def check_table(c, ln, ds):
    bad = np.nonzero((ln != c.ln) | (ds != c.ds))[0]
    assert bad.size == 0, (c.d.size, c.rules, bad[:5])


def check_tokens(c, t):
    assert t.size == c.tokens.size and (t == c.tokens).all(), (c.d.size, c.rules)


def every_entry_point(c):
    check_table(c, *sq.match_table(c.d, *c.rules))
    check_tokens(c, sq.tokens(c.d, *c.rules))
    symbols = c.rules[2] <= 257 and c.rules[3] <= 32767
    got = np.concatenate(stream(c.d, c.rules, symbols))
    want = sq.symbols_of_tokens(c.tokens) if symbols else c.tokens
    assert got.size == want.size and (got == want).all(), (c.d.size, c.rules)
    check_tokens(c, sq.tokens_multi(c.d, [0, 0], *c.rules))
    check_table(c, *unpack(device_table(c.d, c.rules)))
    torch.cuda.synchronize()


def test_entry_points_share_parked_stages(oracle):
    """Sizes just over a power of two (stages of twice the capacity), a quarter of that (takes those, up to
    four times larger), below 1 MiB (the smallest capacity); window 2^10 after 2^15, max_len 512 /
    max_dist 65535 after the default rules; a release in between."""
    sq.release()
    big = corpus.synthetic((4 << 20) + 17, 4321)
    cases = [Case(oracle, big, DEFAULT),
             Case(oracle, big[: big.size // 4], DEFAULT),
             Case(oracle, big[: 300000], SMALL_WINDOW),
             Case(oracle, big[: big.size // 4], WIDE),
             Case(oracle, big[: 300000], DEFAULT)]
    for c in cases:
        every_entry_point(c)
    sq.release()
    every_entry_point(cases[1])
    sq.release()
    check_tokens(cases[0], sq.tokens(cases[0].d))


def test_more_shapes_than_are_kept(oracle):
    """More stages of different kinds and capacities than one device keeps (sixteen shards of one call among
    them), then the first shapes again: the oldest were freed on the way and the results stay exact."""
    sq.release()
    small = Case(oracle, corpus.synthetic(200000, 77), DEFAULT)
    large = Case(oracle, corpus.synthetic((5 << 20) + 3, 7 << 20), DEFAULT)    # capacity 8 Mi: no small stage fits
    for c in (small, large):
        check_table(c, *sq.match_table(c.d))
        check_tokens(c, sq.tokens(c.d))
        want = sq.symbols_of_tokens(c.tokens)
        got = np.concatenate(stream(c.d, DEFAULT, True))
        assert got.size == want.size and (got == want).all()
        check_table(c, *unpack(device_table(c.d, DEFAULT)))
        torch.cuda.synchronize()
    huge = corpus.synthetic(40 << 20, 3 << 20)                                  # against a fresh stage
    fresh = sq.tokens(huge)
    check_tokens(large, sq.tokens_multi(large.d, [0] * 16))
    assert (sq.tokens_multi(huge, [0, 0]) == fresh).all()
    check_table(small, *sq.match_table(small.d))
    check_table(large, *sq.match_table(large.d))
    sq.release()
    assert (sq.tokens(huge) == fresh).all()


def test_stage_given_back_while_its_work_may_run(oracle):
    """A stream of three chunks (2, 4, 2 MiB) closed after the first, then at once the one-shot call and
    another stream on an input of the same size; and the match workspace: two device calls on two streams
    without a wait in between must not share one."""
    sq.release()
    a = corpus.synthetic(8 << 20, 11 << 20)
    b = Case(oracle, corpus.synthetic(8 << 20, 21 << 20), DEFAULT)
    first = stream(a, DEFAULT, True, read=1)
    assert len(first) == 1 and first[0].size > 0
    check_tokens(b, sq.tokens(b.d))
    want = sq.symbols_of_tokens(b.tokens)
    got = np.concatenate(stream(b.d, DEFAULT, True))
    assert got.size == want.size and (got == want).all()
    c = Case(oracle, a, DEFAULT)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    t1 = device_table(c.d, DEFAULT, s1)
    t2 = device_table(b.d, DEFAULT, s2)
    torch.cuda.synchronize()
    check_table(c, *unpack(t1))
    check_table(b, *unpack(t2))
    sq.release()
    check_tokens(c, sq.tokens(c.d))
