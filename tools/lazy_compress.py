"""Greedy against lazy parse (sqz_compress with struct sqz's `lazy` = 0 / 1): compressed size and time of every
fixture (best of 3), then the 256 MiB synthetic sample of bench.py's sqz_compress_e2e with the two modes
alternating, 3 runs each.  Prints one JSON document; --out PATH writes it there as well.

    python tools/lazy_compress.py [--out profiles/r03_lazy.json] [--runs 3] [--sample-mib 256]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sqz_b200 as sq  # noqa: E402
from sqz_b200 import corpus  # noqa: E402

MODES = {"greedy": False, "lazy": True}


def card() -> dict:
    if sq.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                        "--format=csv,noheader"], capture_output=True, text=True)
    f = [x.strip() for x in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return {"name": f[0] if f else None, "power_limit": f[1] if len(f) > 1 else None,
            "clocks_max_sm": f[2] if len(f) > 2 else None, "driver": f[3] if len(f) > 3 else None,
            "host_cores": os.cpu_count()}


def timed(d, lazy, stats=None, into=None):
    t0 = time.perf_counter()
    out = sq.compress(d, 15, lazy=lazy, stats=stats, into=into)
    return time.perf_counter() - t0, out


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
        for mode, lazy in MODES.items():
            timed(d, lazy)                                  # warm: pipeline buffers of this size
            best, size = 1e9, None
            for _ in range(args.runs):
                dt, out = timed(d, lazy)
                best, size = min(best, dt), len(out)
            row[mode] = {"compressed_bytes": size, "seconds_best": best, "MBps": d.size / 1e6 / best}
        row["size_change_pct"] = 100.0 * (row["lazy"]["compressed_bytes"] / row["greedy"]["compressed_bytes"] - 1)
        doc["files"][name] = row
        print(name, json.dumps(row), flush=True)

    sample = corpus.synthetic(args.sample_mib << 20, 0)
    out_buf = np.empty(sq.capacity(sample.size), np.uint8)
    for lazy in MODES.values():                             # untimed, like bench.py's warm-up call
        timed(sample, lazy, into=out_buf)
    runs = {m: [] for m in MODES}
    for _ in range(args.runs):
        for mode, lazy in MODES.items():
            st = {}
            dt, out = timed(sample, lazy, stats=st, into=out_buf)
            runs[mode].append({"MBps": sample.size / 1e6 / dt, "seconds": dt, "tokens": st["tokens"],
                               "compressed_bytes": int(out.size), "search_wait_seconds": st["search_seconds"],
                               "entropy_seconds": st["entropy_seconds"]})
            print(mode, json.dumps(runs[mode][-1]), flush=True)
    _, blob = timed(sample, True)
    e2e = {"sample": "corpus.synthetic(%d MiB, 0), the sample of bench.py's sqz_compress_e2e" % args.sample_mib,
           "order": "greedy and lazy alternating, %d runs each after one untimed call of each" % args.runs,
           "runs": runs, "lazy_round_trip_identical": sq.decompress(blob) == sample.tobytes()}
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
