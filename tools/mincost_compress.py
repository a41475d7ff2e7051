"""Greedy, lazy and min-cost parse (sqz_compress with struct sqz's `lazy` / `mincost`): compressed size and
best-of-3 time of every fixture, then the 256 MiB synthetic sample of bench.py's sqz_compress_e2e with the three
modes alternating, 3 runs each; and the device time of the min-cost kernel per 32 MiB chunk beside the match
search of the same chunks, from CUDA events (sqz_gpu_set_timing).  Prints one JSON document; --out PATH writes it
there as well.

    python tools/mincost_compress.py [--out profiles/r04_mincost.json] [--runs 3] [--sample-mib 256]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sqz_b200 as sq  # noqa: E402
from sqz_b200 import _lib, corpus  # noqa: E402
from lazy_compress import card  # noqa: E402

MODES = {"greedy": {}, "lazy": {"lazy": True}, "mincost": {"mincost": True}}


def timed(d, mode, stats=None, into=None):
    t0 = time.perf_counter()
    out = sq.compress(d, 15, stats=stats, into=into, **MODES[mode])
    return time.perf_counter() - t0, out


def kernel_times(sample, chunk):
    """Average device time of one min-cost launch and of one chunk's match search (both from CUDA events on the
    launching stream) over a stream of `chunk`-byte chunks with the min-cost flag, after one untimed pass."""
    L = _lib.load()
    d = np.ascontiguousarray(sample)

    def run():
        st = C.c_void_p()
        rc = L.sqz_gpu_stream_open(C.byref(st), 0, d.ctypes.data_as(_lib.u8p), d.size, 1 << 15, 3, 257, 32767, chunk,
                                   _lib.STREAM_SYMBOLS | _lib.STREAM_MINCOST)
        assert rc == 0, L.sqz_gpu_last_error()
        while True:
            p, n = _lib.u32p(), C.c_size_t()
            assert L.sqz_gpu_stream_next(st, C.byref(p), C.byref(n)) == 0, L.sqz_gpu_last_error()
            if n.value == 0:
                break
        L.sqz_gpu_stream_close(st)

    run()
    L.sqz_gpu_set_timing(1)
    try:
        L.sqz_gpu_mincost_kernel_seconds(1, None)
        L.sqz_gpu_match_kernel_seconds(1, None)
        run()
        k_mc, k_match = C.c_uint64(), C.c_uint64()
        t_mc = L.sqz_gpu_mincost_kernel_seconds(1, C.byref(k_mc))
        t_match = L.sqz_gpu_match_kernel_seconds(1, C.byref(k_match))
    finally:
        L.sqz_gpu_set_timing(0)
    return {"chunk_bytes": chunk, "chunks": int(k_mc.value), "mincost_kernel_ms": 1e3 * t_mc,
            "match_search_ms": 1e3 * t_match, "mincost_share_of_search_pct": 100.0 * t_mc / t_match,
            "mincost_ms_per_GiB": 1e3 * t_mc * (1 << 30) / chunk}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--sample-mib", type=int, default=256)
    args = ap.parse_args()
    doc = {"gpu": card(), "window": 1 << 15, "rules": "G1 (min_len 3, max_len 257, max_dist window - 1)",
           "coder_threads": "0 (automatic)", "files": {}}

    for name, d in corpus.all_files().items():
        row = {"bytes": int(d.size)}
        for mode in MODES:
            timed(d, mode)                                  # warm: pipeline buffers of this size
            best, size = 1e9, None
            for _ in range(args.runs):
                dt, out = timed(d, mode)
                best, size = min(best, dt), len(out)
            row[mode] = {"compressed_bytes": size, "seconds_best": best, "MBps": d.size / 1e6 / best}
        for mode in ("lazy", "mincost"):
            row[mode + "_size_change_pct"] = 100.0 * (row[mode]["compressed_bytes"] / row["greedy"]["compressed_bytes"] - 1)
        doc["files"][name] = row
        print(name, json.dumps(row), flush=True)

    sample = corpus.synthetic(args.sample_mib << 20, 0)
    doc["kernel"] = kernel_times(sample, 32 << 20)
    print("kernel", json.dumps(doc["kernel"]), flush=True)
    out_buf = np.empty(sq.capacity(sample.size), np.uint8)
    for mode in MODES:                                      # untimed, like bench.py's warm-up call
        timed(sample, mode, into=out_buf)
    runs = {m: [] for m in MODES}
    for _ in range(args.runs):
        for mode in MODES:
            st = {}
            dt, out = timed(sample, mode, stats=st, into=out_buf)
            runs[mode].append({"MBps": sample.size / 1e6 / dt, "seconds": dt, "tokens": st["tokens"],
                               "compressed_bytes": int(out.size), "search_wait_seconds": st["search_seconds"],
                               "entropy_seconds": st["entropy_seconds"]})
            print(mode, json.dumps(runs[mode][-1]), flush=True)
    _, blob = timed(sample, "mincost")
    e2e = {"sample": "corpus.synthetic(%d MiB, 0), the sample of bench.py's sqz_compress_e2e" % args.sample_mib,
           "order": "greedy, lazy and min-cost alternating, %d runs each after one untimed call of each" % args.runs,
           "runs": runs, "mincost_round_trip_identical": sq.decompress(blob) == sample.tobytes()}
    for mode in MODES:
        r = [x["MBps"] for x in runs[mode]]
        e2e[mode] = {"MBps_median": float(np.median(r)), "MBps_min": min(r), "MBps_max": max(r),
                     "tokens": runs[mode][0]["tokens"], "compressed_bytes": runs[mode][0]["compressed_bytes"]}
    doc["sqz_compress_e2e"] = e2e
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
