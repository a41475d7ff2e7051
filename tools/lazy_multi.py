"""Greedy against lazy parse on several devices (sqz_gpu_tokens_multi_ex with flags 0 / SQZ_GPU_STREAM_LAZY).

* 1 GiB of the bench corpus on 1, 2, 4 and 8 shards, one shard per device (shards share devices when the box
  has fewer): the two modes alternating, --runs calls each after one untimed call of each; host clock around
  the call, which returns after the last token copy has landed in pinned host memory.  Token counts, and
  the encoded bytes of a 64 MiB prefix in both modes.
* The seam-word search (sqz_gpu_match_seam_device) on one shard of 1 GiB / 8 from the middle of the corpus,
  with CUDA events: its device time, beside that of the shard's table search and of its greedy and lazy exit
  maps, which is what it delays.
* x64.elf on 4 shards, where a fixed cost per shard would show: the same alternation, every run the mean of
  --small-calls calls.

Prints one JSON document; --out PATH writes it there as well.

    python tools/lazy_multi.py [--out profiles/r04_lazy_multi.json] [--runs 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sqz_b200 as sq  # noqa: E402
from sqz_b200 import _lib, corpus  # noqa: E402

WINDOW, MIN_LEN, MAX_LEN, MAX_DIST = 1 << 15, 3, 257, 32767
MODES = {"greedy": 0, "lazy": _lib.STREAM_LAZY}


def card() -> dict:
    if sq.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm,driver_version",
                        "--format=csv,noheader"], capture_output=True, text=True)
    rows = [[x.strip() for x in line.split(",")] for line in q.stdout.strip().splitlines()] if q.returncode == 0 else []
    return {"devices": sq.device_count(), "host_cores": os.cpu_count(),
            "cards": [{"index": r[0], "name": r[1], "power_limit": r[2], "clocks_max_sm": r[3], "driver": r[4]}
                      for r in rows if len(r) >= 5]}


class Multi:
    """sqz_gpu_tokens_multi_ex on one input into one pinned output buffer."""

    def __init__(self, data: np.ndarray):
        self.L = _lib.load()
        self.data = data
        self.p_out = self.L.sqz_gpu_host_alloc(data.size * 4 + 16)
        if not self.p_out:
            raise SystemExit("pinned allocation failed")

    def __call__(self, devices, flags):
        devs = (C.c_int * len(devices))(*devices)
        n = C.c_size_t()
        t0 = time.perf_counter()
        rc = self.L.sqz_gpu_tokens_multi_ex(devs, len(devices), self.data.ctypes.data_as(_lib.u8p), self.data.size,
                                            WINDOW, MIN_LEN, MAX_LEN, MAX_DIST, flags, self.p_out, self.data.size,
                                            C.byref(n), None)
        dt = time.perf_counter() - t0
        if rc != 0:
            raise SystemExit("sqz_gpu_tokens_multi_ex: %d %s" % (rc, self.L.sqz_gpu_last_error()))
        return dt, int(n.value)

    def close(self):
        self.L.sqz_gpu_host_free(self.p_out)


def summary(seconds, nbytes):
    r = [nbytes / 1e6 / s for s in seconds]
    return {"MBps_median": float(np.median(r)), "MBps_min": min(r), "MBps_max": max(r),
            "seconds": seconds}


def alternate(run, runs, nbytes, calls=1):
    """Both modes, untimed once, then alternating; every run the mean of `calls` calls."""
    for flags in MODES.values():
        run(flags)
    times, tokens = {m: [] for m in MODES}, {}
    for _ in range(runs):
        for mode, flags in MODES.items():
            total = 0.0
            for _ in range(calls):
                dt, tokens[mode] = run(flags)
                total += dt
            times[mode].append(total / calls)
    out = {m: dict(summary(times[m], nbytes), tokens=tokens[m]) for m in MODES}
    out["lazy_over_greedy_median"] = out["lazy"]["MBps_median"] / out["greedy"]["MBps_median"]
    return out


def seam_word_timing(world, reps):
    """CUDA-event times of one shard's seam word, table search and exit maps (torch only holds the memory)."""
    import torch
    L = _lib.load()
    total = 1 << 30
    n = total // world
    first = n * (world // 2)
    back, ahead = MAX_DIST, MAX_LEN
    host = corpus.synthetic(back + n + ahead, first - back)
    buf = torch.cat([torch.from_numpy(host).cuda(), torch.zeros(64, dtype=torch.uint8, device="cuda")])
    shard = buf.data_ptr() + back
    table = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    work = torch.empty(L.sqz_gpu_parse_workspace(n), dtype=torch.uint8, device="cuda")
    emap = torch.empty(512, dtype=torch.int16, device="cuda")
    s = torch.cuda.current_stream()

    def check(rc, what):
        if rc != 0:
            raise SystemExit("%s: %d %s" % (what, rc, L.sqz_gpu_last_error()))

    calls = {
        "match_table": lambda: check(L.sqz_gpu_match_table_device(shard, back, n, ahead, MIN_LEN, MAX_LEN, MAX_DIST,
                                                                  table.data_ptr(), s.cuda_stream), "table"),
        "seam_word": lambda: check(L.sqz_gpu_match_seam_device(shard, back, n, ahead, MIN_LEN, MAX_LEN, MAX_DIST,
                                                               table.data_ptr(), s.cuda_stream), "seam"),
        "exit_map_greedy": lambda: check(L.sqz_gpu_parse_exit_map_device_ex(table.data_ptr(), n, MIN_LEN, MAX_LEN, 0,
                                                                            work.data_ptr(), emap.data_ptr(),
                                                                            s.cuda_stream), "map"),
        "exit_map_lazy": lambda: check(L.sqz_gpu_parse_exit_map_device_ex(table.data_ptr(), n, MIN_LEN, MAX_LEN,
                                                                          _lib.STREAM_LAZY, work.data_ptr(),
                                                                          emap.data_ptr(), s.cuda_stream), "map"),
    }
    out = {"shard_positions": n, "shard_first": first, "launches_per_measurement": {}}
    for name, fn in calls.items():
        k = 3 if name == "match_table" else reps
        fn()                                              # warm: module load, parked workspace
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(k):
            fn()
        e1.record(s)
        e1.synchronize()
        out[name + "_ms"] = e0.elapsed_time(e1) / k
        out["launches_per_measurement"][name] = k
    w = int(table[n].item()) & 0xFFFFFFFF
    out["seam_word"] = {"len": w >> 16, "dist": w & 0xFFFF}
    out["note"] = ("seam_word_ms is back-to-back launches of the one-CTA search on an otherwise idle device: its "
                   "latency on the critical path before the shard's exit map, not a throughput")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--small-calls", type=int, default=20)
    args = ap.parse_args()
    doc = {"gpu": card(), "rules": "G1 (window 2^15, min_len 3, max_len 257, max_dist 32767)",
           "timing": "host clock around sqz_gpu_tokens_multi_ex; tokens into pinned host memory"}
    n_dev = sq.device_count()

    data = corpus.synthetic(int(args.gib * (1 << 30)), 0)
    big = Multi(data)
    doc["bench_corpus"] = {"bytes": int(data.size), "order": "greedy and lazy alternating, %d runs each after one "
                           "untimed call of each" % args.runs, "shards": {}}
    for world in (1, 2, 4, 8):
        devices = [g % n_dev for g in range(world)]
        row = alternate(lambda flags: big(devices, flags), args.runs, data.size)
        row["devices"] = devices
        doc["bench_corpus"]["shards"][str(world)] = row
        print(world, json.dumps(row), flush=True)
    big.close()
    sq.release()

    prefix = np.ascontiguousarray(data[: 64 << 20])
    del data
    devices = [g % n_dev for g in range(4)]
    enc = {}
    for mode, lazy in (("greedy", False), ("lazy", True)):
        toks = sq.tokens_multi(prefix, devices, lazy=lazy)
        comp = sq.encode_tokens(toks, prefix.size, 15)
        enc[mode] = {"tokens": int(toks.size), "encoded_bytes": len(comp)}
        if lazy:
            enc["lazy_round_trip_identical"] = sq.decompress(comp) == prefix.tobytes()
    enc["size_change_pct"] = 100.0 * (enc["lazy"]["encoded_bytes"] / enc["greedy"]["encoded_bytes"] - 1)
    doc["prefix_64MiB_encoded"] = enc
    print("prefix", json.dumps(enc), flush=True)

    doc["seam_word_one_shard"] = seam_word_timing(8, 200)
    print("seam", json.dumps(doc["seam_word_one_shard"]), flush=True)
    sq.release()

    elf = corpus.all_files()["x64.elf"]
    small = Multi(np.ascontiguousarray(elf))
    devices = [g % n_dev for g in range(4)]
    row = alternate(lambda flags: small(devices, flags), args.runs, elf.size, args.small_calls)
    row.update(devices=devices, bytes=int(elf.size), calls_per_run=args.small_calls)
    doc["x64_elf_4_shards"] = row
    small.close()
    print("x64.elf", json.dumps(row), flush=True)

    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
