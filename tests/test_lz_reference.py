"""The checker of the GPU copy phase, checked itself (no GPU): lz_execute (tests/c/lz_execute.c) gives back
the input from the oracle's tokens, agrees with an independent LZ77 expansion and with the host decoder,
and names the first bad token of a stream."""
import numpy as np
import pytest

import sqz_b200 as sq

from lz_reference import SHORT, execute, expand, stream_of_bytes, stream_of_count
from test_gpu_expand import NAMES, tokens_of
from test_gpu_shards import lz77_decode


@pytest.mark.parametrize("wb", [10, 15])
@pytest.mark.parametrize("name", NAMES + ["csrc.cat"])
def test_oracle_tokens_give_back_the_input(name, wb, inputs, oracle):
    d = inputs[name]
    assert (expand(tokens_of(oracle, d, wb), d.size) == d).all()


@pytest.mark.parametrize("seed", range(6))
def test_agrees_with_plain_lz77(seed):
    toks, n = stream_of_count(seed, 3000, long=0.01, overlap=0.5)
    assert (expand(toks, n) == lz77_decode(toks, n)).all(), seed
    toks = stream_of_bytes(seed, 50000 + seed, lit=0.2, long=0.02)
    assert (expand(toks, 50000 + seed) == lz77_decode(toks, 50000 + seed)).all(), seed


def test_generators_keep_their_promises():
    for seed in range(4):
        toks, n = stream_of_count(seed, 1000 + seed)
        assert toks.size == 1000 + seed
        assert execute(toks, n)[0] == 0
        for nbytes in (0, 1, 2, 65536 + seed, 1 << 20):
            t = stream_of_bytes(seed, nbytes, min_len=3, max_len=257, max_dist=32767)
            assert execute(t, nbytes)[0] == 0, (seed, nbytes)
            m = t[(t >> 16) != 0]
            assert ((m >> 16) >= 3).all() and ((m >> 16) <= 257).all() and ((m & 0xFFFF) <= 32767).all()
    # the heavy tail and the overlap are there: lengths up to 65535, and copies that read their own output
    toks, _ = stream_of_count(7, 200000, long=0.01, overlap=0.5)
    ln, ds = toks >> 16, toks & 0xFFFF
    assert ln.max() > 30000 and ((ln > 0) & (ds < ln)).sum() > 10000 and (ln == 1).any()


def test_bad_tokens_are_reported_at_their_index():
    lit = np.arange(10, dtype=np.uint32)
    cases = [(np.r_[lit, 0x100 | 7], 11, 11),               # a literal word above 0xFF (a symbol word)
             (np.r_[lit, 0x1FF, 1], 12, 11),
             (np.r_[lit, (3 << 16) | 0], 13, 11),           # dist 0
             (np.r_[lit, (3 << 16) | 11], 13, 11),          # one byte before byte 0
             (np.r_[(3 << 16) | 1, lit], 13, 1),            # a match as the first token
             (np.r_[lit, (5 << 16) | 2], 14, 11),           # past `bytes`
             (lit, 9, 10),                                  # a literal past `bytes`
             (np.r_[lit, (65535 << 16) | 10, 5], 65545, 12)]
    for toks, n, want in cases:
        assert execute(toks.astype(np.uint32), n)[0] == want, (toks[-3:], n)
    assert execute(lit, 11)[0] == SHORT
    assert execute(np.zeros(0, np.uint32), 1)[0] == SHORT
    assert execute(np.zeros(0, np.uint32), 0)[0] == 0
    code, out = execute(np.r_[lit, (3 << 16) | 10].astype(np.uint32), 13)   # reaches byte 0 exactly
    assert code == 0 and out[:13].tolist() == list(range(10)) + [0, 1, 2]


@pytest.mark.parametrize("seed", range(4))
def test_agrees_with_the_host_decoder(seed):
    """Within the bitstream's limits (len 3..257, dist <= 32767) the tokens survive the coder, and the
    host decoder's bytes are lz_execute's."""
    n = (1 << 18) + 977 * seed
    toks = stream_of_bytes(seed, n, lit=0.3, long=0.05, overlap=0.3, min_len=3, max_len=257, max_dist=32767)
    comp = sq.encode_tokens(toks, n, 15)
    back = sq.decode_tokens(comp)
    assert back.size == toks.size and (back == toks).all(), seed
    assert sq.decompress(comp) == expand(toks, n).tobytes(), seed
