"""The unmodified reference (oracle/_ref) where it was not built: its recorded answers.

tests/golden/reference_calls.json holds, for every call the suite makes to the reference, a digest
of the arguments and the length and FNV-1a-64 of what the reference returned.  RecordedReference
has Reference's methods: each computes its answer with this project's own code (the codec for
bitstreams, the oracle for match tables) and returns it only when it is the recorded one.  A test
that compares with the reference so compares with the reference's recorded answer, and its later
steps get real bytes and arrays to work on.

SQZ_RECORD_REFERENCE=<path> writes the answers of a run to <path> instead of checking them.  Record
only at a commit whose suite passes against the reference itself: the recording is taken to be the
reference's answers.
"""
from __future__ import annotations

import json
import os

import numpy as np

import sqz_b200 as sq
from oracle import _u8

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.json")


class RecordedReference:
    def __init__(self, oracle, record_to: str | None = None):
        self.oracle = oracle
        self.record_to = record_to
        self.calls = {}
        if not record_to:
            with open(PATH) as f:
                self.calls = json.load(f)["calls"]
        self.recorded = {}

    def _digest(self, a) -> str:
        if isinstance(a, (bytes, bytearray, memoryview)):
            a = np.frombuffer(a, np.uint8)
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a)
            return "%d:%016x" % (a.nbytes, self.oracle.fnv(a))
        if isinstance(a, tuple):
            return "(" + ",".join(self._digest(x) for x in a) + ")"
        return repr(a)

    def _answer(self, what: str, args: tuple, got):
        key = what + "(" + ",".join(self._digest(a) for a in args) + ")"
        have = self._digest(got)
        if self.record_to:
            self.recorded[key] = have
        else:
            assert key in self.calls, "no recorded reference answer for " + key
            assert have == self.calls[key], "%s: %s, the reference answered %s" % (key, have, self.calls[key])
        return got

    def save(self) -> None:
        if self.record_to and self.recorded:
            calls = {}
            if os.path.exists(self.record_to):
                with open(self.record_to) as f:
                    calls = json.load(f)["calls"]
            calls.update(self.recorded)
            with open(self.record_to, "w") as f:
                json.dump({"_about": "answers of the unmodified reference (oracle/_ref) to the calls of the test suite: "
                                     "call(argument digests) -> answer digest, a digest being byte length:FNV-1a-64; "
                                     "written by tests/recorded_reference.py",
                           "calls": dict(sorted(calls.items()))}, f, indent=0)
                f.write("\n")

    def compress(self, data, win_bits: int = 15, file_mode: bool = False) -> bytes:
        d = _u8(data)
        t, end = self.oracle.tokens_from_table(d, *self.oracle.match_table(d, 1 << win_bits, fast=True))
        assert end == d.size
        return self._answer("compress", (d, win_bits, file_mode),
                            sq.encode_tokens(t, d.size, win_bits, file_mode=file_mode))

    def decompress(self, comp) -> bytes:
        return self._answer("decompress", (comp,), sq.decompress(comp))

    def tokens(self, comp) -> np.ndarray:
        return self._answer("tokens", (comp,), sq.decode_tokens(comp))

    def encode_tokens(self, tokens, nbytes: int, win_bits: int = 15, file_mode: bool = False) -> bytes:
        t = np.ascontiguousarray(tokens, dtype=np.uint32)
        return self._answer("encode_tokens", (t, nbytes, win_bits, file_mode),
                            sq.encode_tokens(t, nbytes, win_bits, file_mode=file_mode))

    def bst_table(self, data, window: int, first: int = 0, count: int | None = None):
        d = _u8(data)
        got = self.oracle.match_table(d, 1 << 16, first, count, min_len=2, max_len=254, max_dist=window)
        return self._answer("bst_table", (d, window, first, count), got)
