"""Greedy, lazy and min-cost parse on several devices (sq.tokens_multi: sqz_gpu_tokens_multi_ex for greedy and
lazy, sqz_gpu_tokens_multi_cuts for min-cost, whose shards are cut at multiples of 16384).

* 1 GiB of the bench corpus (256 MiB when the host has less than 40 GB available, as the full-size test does)
  on 1, 2, 4 and 8 shards, one shard per device (shards share devices when the box has fewer): the three modes
  alternating, --runs calls each after one untimed call of each; host clock around the call, which returns
  after the last token copy has landed in pinned host memory.  Median, minimum and maximum rate, token counts.
* The min-cost kernel's device time per shard (sqz_gpu_mincost_kernel_seconds, CUDA events around each launch)
  on every shard count, taken in separate calls after the timed ones so that the events do not sit in them.
* The card's name and power limit, read in the same run.

Prints one JSON document; --out PATH writes it there as well.

    python tools/mincost_multi.py [--out profiles/r05_mincost_multi.json] [--runs 3]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sqz_b200 as sq  # noqa: E402
from sqz_b200 import _lib, corpus  # noqa: E402
from lazy_multi import card, summary  # noqa: E402

WINDOW, MIN_LEN, MAX_LEN, MAX_DIST = 1 << 15, 3, 257, 32767
MODES = {"greedy": 0, "lazy": _lib.STREAM_LAZY, "mincost": _lib.STREAM_MINCOST}


def input_bytes() -> int:
    try:
        import psutil
        if psutil.virtual_memory().available < (40 << 30):
            return 256 << 20
    except ImportError:
        pass
    return 1 << 30


class Multi:
    """One input into one pinned output buffer: greedy and lazy through sqz_gpu_tokens_multi_ex, min-cost through
    sqz_gpu_tokens_multi_cuts with the even cut at multiples of 16384."""

    def __init__(self, data: np.ndarray):
        self.L = _lib.load()
        self.data = data
        self.p_out = self.L.sqz_gpu_host_alloc(data.size * 4 + 16)
        if not self.p_out:
            raise SystemExit("pinned allocation failed")

    def __call__(self, devices, flags):
        devs = (C.c_int * len(devices))(*devices)
        n = C.c_size_t()
        per = (C.c_size_t * len(devices))()
        args = (self.data.ctypes.data_as(_lib.u8p), self.data.size, WINDOW, MIN_LEN, MAX_LEN, MAX_DIST, flags,
                self.p_out, self.data.size, C.byref(n), per)
        t0 = time.perf_counter()
        if flags & _lib.STREAM_MINCOST:
            what, rc = "sqz_gpu_tokens_multi_cuts", self.L.sqz_gpu_tokens_multi_cuts(devs, len(devices), None, *args)
        else:
            what, rc = "sqz_gpu_tokens_multi_ex", self.L.sqz_gpu_tokens_multi_ex(devs, len(devices), *args)
        dt = time.perf_counter() - t0
        if rc != 0:
            raise SystemExit("%s: %d %s" % (what, rc, self.L.sqz_gpu_last_error()))
        return dt, int(n.value), [int(x) for x in per]

    def close(self):
        self.L.sqz_gpu_host_free(self.p_out)


def alternate(run, runs, nbytes):
    """The three modes, untimed once, then alternating."""
    for flags in MODES.values():
        run(flags)
    times, tokens = {m: [] for m in MODES}, {}
    for _ in range(runs):
        for mode, flags in MODES.items():
            dt, tokens[mode], _ = run(flags)
            times[mode].append(dt)
    out = {m: dict(summary(times[m], nbytes), tokens=tokens[m]) for m in MODES}
    for m in ("lazy", "mincost"):
        out[m + "_over_greedy_median"] = out[m]["MBps_median"] / out["greedy"]["MBps_median"]
    return out


def kernel_times(run, calls):
    """Average device time of one min-cost launch (one per non-empty shard) over `calls` min-cost calls."""
    L = _lib.load()
    L.sqz_gpu_set_timing(1)
    try:
        L.sqz_gpu_mincost_kernel_seconds(1, None)
        for _ in range(calls):
            _, _, per = run(_lib.STREAM_MINCOST)
        launches = C.c_uint64()
        seconds = L.sqz_gpu_mincost_kernel_seconds(1, C.byref(launches))
    finally:
        L.sqz_gpu_set_timing(0)
        L.sqz_gpu_match_kernel_seconds(1, None)
    return {"mincost_kernel_ms_per_shard": 1e3 * seconds, "launches": int(launches.value), "calls": calls,
            "shard_tokens": per}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    args = ap.parse_args()
    doc = {"gpu": card(), "rules": "G1 (window 2^15, min_len 3, max_len 257, max_dist 32767)",
           "timing": "host clock around the multi-device call; tokens into pinned host memory"}
    n_dev = sq.device_count()
    data = corpus.synthetic(input_bytes(), 0)
    big = Multi(data)
    doc["bench_corpus"] = {"bytes": int(data.size), "order": "greedy, lazy and min-cost alternating, %d runs each "
                           "after one untimed call of each" % args.runs, "shards": {}}
    for world in (1, 2, 4, 8):
        devices = [g % n_dev for g in range(world)]
        row = alternate(lambda flags: big(devices, flags), args.runs, data.size)
        row["devices"] = devices
        row["mincost_kernel"] = kernel_times(lambda flags: big(devices, flags), 2)
        doc["bench_corpus"]["shards"][str(world)] = row
        print(world, json.dumps(row), flush=True)
    big.close()
    sq.release()

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
