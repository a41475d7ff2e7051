#!/usr/bin/env python
"""bench.py -- match-search throughput of sqz-b200 on B200, beside the reference CPU codec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size BYTES] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[4], SURVEY.md section 8d config 5): the 1 GiB synthetic corpus
-- the reference's six test/ files concatenated and repeated with seeded mutations -- cut into
N contiguous shards of 2^30/N bytes, one per GPU, each with a max_dist look-back halo and a
max_len look-ahead halo ("strong" scaling: the job is 1 GiB whatever N is).

A step = one pass of the hot path over the whole input: every rank computes the match table of
its shard (squeeze.h:338-358 at every i), the seams are resolved (one integer per seam: where the
previous shard's last token ends, squeeze.h:377-394), every rank parses its shard into tokens, and
the token arrays are concatenated in shard order on GPU 0.  No collective library is on that
path: the 1 KiB exit maps and the token counts cross a shared-memory mailbox on the host
(sqz_b200/shard.py), the tokens go peer-to-peer over NVLink into a CUDA-IPC-mapped buffer
(cudaMemcpyAsync, sized by their counts).  torch.distributed (NCCL) is used for the rendezvous,
the barriers around the timed region and the max-over-ranks of the timings only.  At N = 1 the
token array of the one shard is the concatenation.

`value` = input MB/s (1 MB = 1e6 B) of the whole job, inputs resident in HBM, timed with CUDA
events on the launching stream, max over ranks.  `e2e` = the same search through the host-buffer
C-ABI sqz_gpu_match_table() from pinned host memory to pinned host memory (every rank its shard),
host<->device copies inside the timed region.  `weak` (N > 1) = the round-1 layout, 1 GiB per GPU.

--impl reference times the UNMODIFIED reference codec (oracle/_ref, squeeze.compress)
on the host cores, on bounded samples of the same stream.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOW = 1 << 15
MIN_LEN, MAX_LEN, MAX_DIST = 3, 257, WINDOW - 1      # reference G1 rules, squeeze.h:13-15,342
SMEM_BYTES_PER_CLK_PER_SM = 128
METRIC = "match_search_input_MBps"
ROOFLINE_INPUTS = os.path.join(ROOT, "profiles", "r02_roofline_inputs.json")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def cc_count(g0: int, n: int, md: int) -> int:
    """Candidate-compares for positions [g0, g0+n): sum of min(i, max_dist)  (SURVEY 8d)."""
    a, b = g0, g0 + n
    k = min(max(md, a), b)              # positions below k have i < md
    tri = (k - 1) * k // 2 - (a - 1) * a // 2 if k > a else 0
    return tri + (b - k) * md


def roofline_inputs() -> dict:
    """Instruction and traffic counts of the dominant kernel, taken from the committed ncu capture
    of the kernel that is being benched (profiles/README.md says how it was made)."""
    try:
        with open(ROOFLINE_INPUTS) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.path = tempfile.mktemp(prefix="sqz_clocks_", suffix=".csv")
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "200"], stdout=self.fh, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if f[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            busy = [c for c in sm if c > 0.5 * max(sm)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm), power_w_max=max(power) if power else None)
        return out


# ----------------------------------------------------------------------------- reference arm
def reference_arm(args) -> None:
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import Oracle, Reference
    from sqz_b200 import corpus
    # oracle/_ref (the unmodified reference) when it was built; else the oracle's C restatement
    # of the same search + parse (kind "port"; it lacks the entropy stage, < 1 % of the time)
    kind = "reference" if Reference.available() else "port"
    cores = os.cpu_count() or 1
    slice_bytes = 128 << 10
    n_slices = 2 * cores
    total = args.size
    stride = max(total // n_slices, 1)
    slices = [corpus.synthetic(slice_bytes, (k * stride) // 4096 * 4096) for k in range(n_slices)]
    if kind == "port":
        Oracle.get().set_threads(1)

    def one_step() -> float:
        todo = list(range(n_slices))
        lock = threading.Lock()

        def worker():
            from oracle import Reference as R
            r = R(release=True) if kind == "reference" else None   # own handle; the C call releases the GIL
            while True:
                with lock:
                    if not todo:
                        return
                    k = todo.pop()
                if r is not None:
                    r.compress(slices[k], 15)
                else:
                    Oracle.get().tokens(slices[k], WINDOW)

        th = [threading.Thread(target=worker) for _ in range(cores)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        return time.perf_counter() - t0

    for _ in range(args.warmup):
        pass                                # a CPU loop has nothing to warm that matters; keep W for the record
    times = [one_step() for _ in range(args.steps)]
    sec = sum(times) / len(times)
    mbps = n_slices * slice_bytes / 1e6 / sec
    sample = ("%d slices x %d KiB of the synthetic stream, evenly spaced over %d MiB, one %s "
              "(window 2^15) per slice, work queue over %d threads; slices start with an empty window, "
              "which favours the reference by ~12%%"
              % (n_slices, slice_bytes >> 10, max(total >> 20, 1),
                 "squeeze.compress" if kind == "reference" else "oracle search+parse", cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": mbps, "unit": "MB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": mbps, "unit": "MB/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": mbps, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args) -> dict:
    return {
        "workload": "synthetic corpus (6 reference test/ files repeated + seeded mutations, SURVEY 8d config 5), "
                    "%d MiB in all, %d contiguous shard(s) of %d MiB with 32767 B / 257 B halos, window 2^15, "
                    "min_len 3, max_len 257, max_dist 32767"
                    % (args.size >> 20, args.gpus, (args.size // args.gpus) >> 20),
        "total_bytes": args.size, "bytes_per_gpu": args.size // args.gpus, "window": WINDOW, "min_len": MIN_LEN,
        "max_len": MAX_LEN, "max_dist": MAX_DIST, "parallelism": "shard%d" % args.gpus,
        "cache": "every shard (>= 128 MiB in, 4x that out) is larger than the 126 MB L2; no explicit flush",
    }


def dump_outputs(path: str, d_table, d_tokens) -> None:
    """What the last timed step handed its caller, as .npy files: the match table of rank 0's shard
    (length and distance per position) and the whole token stream.  Both are far larger than 64 MB,
    so fixed seeded samples of positions are written, with the positions themselves; the values are
    exact in float32 (16-bit length and distance) and float64 (32-bit tokens, positions)."""
    import torch
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0x53515A)

    def sample(n: int, k: int) -> np.ndarray:
        return np.arange(n) if n <= k else np.unique(rng.integers(0, n, k))

    pos = sample(d_table.numel(), 2 << 20)
    w = d_table[torch.from_numpy(pos).to(d_table.device)].cpu().numpy().view(np.uint32)
    at = sample(d_tokens.numel(), 1 << 20)
    tok = d_tokens[torch.from_numpy(at).to(d_tokens.device)].cpu().numpy().view(np.uint32)
    for name, a in (("match_position", pos.astype(np.float64)), ("match_len", (w >> 16).astype(np.float32)),
                    ("match_dist", (w & 0xFFFF).astype(np.float32)), ("token_index", at.astype(np.float64)),
                    ("token", tok.astype(np.float64)), ("token_count", np.array([d_tokens.numel()], np.float64))):
        np.save(os.path.join(path, name + ".npy"), a)


# ----------------------------------------------------------------------------- our arm
class DeviceArray:
    """A raw device allocation of the library seen as a CUDA array (torch.as_tensor wraps it)."""

    def __init__(self, ptr: int, n: int, typestr: str = "<i4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


def ours(args) -> None:
    import torch
    import torch.distributed as dist

    from sqz_b200 import _lib, corpus, shard
    L = _lib.load()
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run" % (args.gpus, world))
    if not torch.cuda.is_available() or L.sqz_gpu_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: sqz_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: whatever NCCL has to say (its version banner when the
        # box sets NCCL_DEBUG) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    def check(rc, what):
        if rc != 0:
            raise RuntimeError("%s failed: %d %s" % (what, rc, L.sqz_gpu_last_error()))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: int) -> int:
        if world == 1:
            return int(x)
        t = torch.tensor([int(x)], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    def pinned(nbytes, dtype):
        p = L.sqz_gpu_host_alloc(nbytes)
        if not p:
            raise MemoryError("sqz_gpu_host_alloc(%d)" % nbytes)
        buf = (C.c_uint8 * nbytes).from_address(p)
        return p, np.frombuffer(buf, dtype=dtype)

    stream = torch.cuda.current_stream()

    # ---- mailbox and gather buffer (N > 1): set up once, outside every timed region --------------
    mb, gather_ptr, gather_how, gather_base = None, 0, "single shard: its token array is the stream", None
    if world > 1:
        path = "/dev/shm/sqz_bench_%s_%s" % (os.environ.get("MASTER_PORT", "0"), os.environ.get("TORCHELASTIC_RUN_ID", "run"))
        if rank == 0:
            mb = shard.Mailbox(path, rank, world, create=True)
        dist.barrier()
        if rank != 0:
            mb = shard.Mailbox(path, rank, world, create=False)
        ok = 1
        if rank == 0:
            p = C.c_void_p()
            check(L.sqz_gpu_device_alloc(C.byref(p), 4 * args.size + 64), "sqz_gpu_device_alloc")
            gather_base = p.value
            handle = C.create_string_buffer(64)
            check(L.sqz_gpu_ipc_export(p, handle), "sqz_gpu_ipc_export")
            mb.put_blob(handle.raw)
            gather_ptr = p.value
        else:
            handle = mb.get_blob()[:64]
            p = C.c_void_p()
            rc = L.sqz_gpu_ipc_open(handle, C.byref(p))
            if rc != 0:
                ok = 0
                sys.stderr.write("rank %d: cudaIpcOpenMemHandle failed: %s\n" % (rank, L.sqz_gpu_last_error()))
            gather_ptr = p.value or 0
        t = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 1:
            gather_how = ("peer-to-peer cudaMemcpyAsync into a CUDA-IPC-mapped buffer on GPU 0, count x 4 bytes "
                          "per shard at the scanned offset")
        else:
            gather_ptr = 0
            gather_how = "unavailable: CUDA IPC mapping failed on this box, tokens stay on their GPUs"

    # ---- one leg: shard `me` of a `total`-byte stream, K timed steps -----------------------------
    seq = [0]

    def run_leg(total: int, me, steps: int, warmup: int, gather: bool, timed_kernel: bool):
        n, g0, back, ahead = me.n, me.first, me.back, me.ahead
        host = corpus.synthetic(back + n + ahead, g0 - back)
        d_data = torch.empty(back + n + ahead + 64, dtype=torch.uint8, device=dev)
        d_data[: back + n + ahead].copy_(torch.from_numpy(host))
        d_table = torch.empty(n, dtype=torch.int32, device=dev)
        d_tokens = torch.empty(n + 4, dtype=torch.int32, device=dev)
        d_work = torch.empty(L.sqz_gpu_parse_workspace(n), dtype=torch.uint8, device=dev)
        d_mwork = torch.empty(L.sqz_gpu_match_workspace(n), dtype=torch.uint8, device=dev)
        d_result = torch.zeros(2, dtype=torch.int64, device=dev)
        d_map = torch.zeros(512, dtype=torch.int16, device=dev)
        h_map = torch.zeros(512, dtype=torch.int16).pin_memory()
        h_result = torch.zeros(2, dtype=torch.int64).pin_memory()
        shard_ptr = d_data.data_ptr() + back
        state = {"count": 0, "offset": 0, "entry": 0}

        def step() -> None:
            s = stream.cuda_stream
            check(L.sqz_gpu_match_table_device_ws(shard_ptr, back, n, ahead, MIN_LEN, MAX_LEN, MAX_DIST,
                                                  d_table.data_ptr(), d_mwork.data_ptr(), s), "match_table")
            entry = 0
            if world > 1:
                # seam hand-off: every shard publishes overshoot(entry) for all entries (1 KiB); chaining
                # the earlier shards' maps gives this shard's entry.  Host mailbox, no collective.
                seq[0] += 1
                check(L.sqz_gpu_parse_exit_map_device(d_table.data_ptr(), n, MIN_LEN, MAX_LEN,
                                                      d_work.data_ptr(), d_map.data_ptr(), s), "exit_map")
                h_map.copy_(d_map, non_blocking=True)
                stream.synchronize()
                entry, _ = mb.entry(seq[0], h_map.numpy().view(np.uint16)[:MAX_LEN])
            check(L.sqz_gpu_parse_device(shard_ptr, d_table.data_ptr(), n, entry, MIN_LEN, MAX_LEN,
                                         d_tokens.data_ptr(), n, d_work.data_ptr(), d_result.data_ptr(), s), "parse")
            state["entry"] = entry
            if world > 1:
                h_result.copy_(d_result, non_blocking=True)
                stream.synchronize()
                count = int(h_result[0])
                at = mb.offset(seq[0], count)          # the earlier shards' counts
                state["count"], state["offset"] = count, at
                if gather and gather_ptr:
                    check(L.sqz_gpu_put_tokens(gather_ptr, at, d_tokens.data_ptr(), count, s), "put_tokens")

        for _ in range(warmup):
            step()
        barrier()
        sampler = None
        if timed_kernel:
            L.sqz_gpu_set_timing(1)
            L.sqz_gpu_match_kernel_seconds(1, None)
            sampler = ClockSampler(local)
            if rank == 0:
                sampler.start()
        launches0 = L.sqz_gpu_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for _ in range(steps):
            step()
        ev1.record(stream)
        barrier()
        sec = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3) / steps
        out = {"sec": sec, "launches": L.sqz_gpu_launch_count() - launches0, "host": host, "d_table": d_table,
               "d_tokens": d_tokens, "d_result": d_result, "state": state, "me": me, "d_data": d_data}
        if timed_kernel:
            nl = C.c_uint64()
            out["t_match"] = L.sqz_gpu_match_kernel_seconds(1, C.byref(nl))
            out["n_timed"] = int(nl.value)
            L.sqz_gpu_set_timing(0)
            out["clocks"] = sampler.stop() if rank == 0 else {}
        if world == 1:
            state["count"] = int(d_result[0].item())
        return out

    # ---- device-resident leg: the whole input, sharded (strong scaling) ----------------------------
    total = args.size
    plan = shard.plan(total, world, MAX_DIST, MAX_LEN)
    me = plan[rank]
    leg = run_leg(total, me, args.steps, args.warmup, gather=True, timed_kernel=True)
    n, g0, back, ahead = me.n, me.first, me.back, me.ahead
    host, d_table, sec, t_match, clocks = leg["host"], leg["d_table"], leg["sec"], leg["t_match"], leg["clocks"]
    n_tokens_mine = leg["state"]["count"]
    n_timed = leg["n_timed"]
    n_tokens = sum_over_ranks(n_tokens_mine)
    launches = sum_over_ranks(leg["launches"])
    t_match_max = max_over_ranks(t_match)
    if args.dump_outputs and rank == 0:
        if world == 1:
            toks = leg["d_tokens"][:n_tokens]
        elif gather_ptr:
            toks = torch.as_tensor(DeviceArray(gather_ptr, n_tokens), device=dev)
        else:
            raise SystemExit("--dump-outputs: the token stream was not gathered on GPU 0")
        dump_outputs(args.dump_outputs, d_table, toks)

    # visited candidate-compares: what the reference's scan really walks (it stops at the nearest
    # max_len candidate, squeeze.h:353); algorithmic CC ignores that early-out (SURVEY 8d)
    visited = 0
    for lo in range(0, n, 1 << 26):
        hi = min(lo + (1 << 26), n)
        w = d_table[lo:hi].to(torch.int64) & 0xFFFFFFFF
        ln, ds = w >> 16, w & 0xFFFF
        i = torch.arange(g0 + lo, g0 + hi, dtype=torch.int64, device=dev).clamp_(max=MAX_DIST)
        visited += int(torch.where(ln == MAX_LEN, ds, i).sum().item())
        del w, ln, ds, i
    visited = sum_over_ranks(visited)

    # ---- the benched table against the oracle (outside every timed region) -------------------------
    parity = {}
    try:
        from oracle import Oracle
        o = Oracle.get()
        win = min(16 << 20, n)
        mid = ((n - win) // 2) // 4096 * 4096
        b2 = min(back + mid, MAX_DIST)
        a2 = min(n + ahead - (mid + win), MAX_LEN)
        piece = np.ascontiguousarray(host[back + mid - b2: back + mid + win + a2])
        oln, ods = o.match_table(piece, WINDOW, first=b2, count=win, fast=True)
        tab = d_table[mid: mid + win].cpu().numpy().view(np.uint32)
        same = bool(((tab >> 16) == oln).all() and ((tab & 0xFFFF) == ods).all())
        rng = np.random.default_rng(1234 + rank)
        pos = rng.integers(0, n, 500)
        got = d_table[torch.from_numpy(pos).to(dev)].cpu().numpy().view(np.uint32)
        brute = 0
        for k, p in enumerate(pos.tolist()):
            lo_b = min(back + p, MAX_DIST)
            hi_b = min(n + ahead - p, MAX_LEN + 1)
            sl = host[back + p - lo_b: back + p + hi_b]
            # the slice ends before the data does: cap the oracle's run at max_len by the rules themselves
            bl, bd = o.best(np.ascontiguousarray(sl), lo_b, WINDOW)
            brute += int((bl, bd) == (int(got[k] >> 16), int(got[k] & 0xFFFF)))
        parity = {"window_bytes": int(win), "window_offset_in_shard": int(mid), "table_equals_oracle_B": same,
                  "brute_force_positions": 500, "brute_force_equal": brute,
                  "what": "the table this run was timed on, rank %d: every position of a %d MiB window against the "
                          "oracle's exact hash-chain search, 500 random positions against the restated reference loop "
                          "(squeeze.h:340-358)" % (rank, win >> 20)}
        assert same and brute == 500, "the benched table differs from the oracle: %r" % (parity,)
    except ImportError as e:
        parity = {"unavailable": repr(e)}

    # ---- N > 1: the gathered stream equals the single-GPU stream (outside every timed region) -----
    gathered = None
    if world > 1:
        barrier()
        mb.barrier(1)
        if rank == 0:
            whole = corpus.synthetic(total, 0)
            d_all = torch.empty(total + 64, dtype=torch.uint8, device=dev)
            d_all[:total].copy_(torch.from_numpy(whole))
            t_all = torch.empty(total, dtype=torch.int32, device=dev)
            k_all = torch.empty(total + 4, dtype=torch.int32, device=dev)
            w_all = torch.empty(L.sqz_gpu_parse_workspace(total), dtype=torch.uint8, device=dev)
            r_all = torch.zeros(2, dtype=torch.int64, device=dev)
            s = stream.cuda_stream
            check(L.sqz_gpu_match_table_device(d_all.data_ptr(), 0, total, 0, MIN_LEN, MAX_LEN, MAX_DIST, t_all.data_ptr(), s), "match_table")
            check(L.sqz_gpu_parse_device(d_all.data_ptr(), t_all.data_ptr(), total, 0, MIN_LEN, MAX_LEN, k_all.data_ptr(),
                                         total, w_all.data_ptr(), r_all.data_ptr(), s), "parse")
            torch.cuda.synchronize()
            single = int(r_all[0].item())
            gathered = {"single_gpu_tokens": single, "sharded_tokens": n_tokens, "how": gather_how,
                        "shard_tokens": mb.counts(seq[0])}
            if gather_ptr:
                got = torch.as_tensor(DeviceArray(gather_ptr, n_tokens), device=dev)
                gathered["identical_to_single_gpu_stream"] = bool(single == n_tokens and torch.equal(got, k_all[:single]))
                assert gathered["identical_to_single_gpu_stream"], "the gathered token stream differs from the 1-GPU stream"
            else:
                gathered["identical_to_single_gpu_stream"] = None
                assert single == n_tokens
            del d_all, t_all, k_all, w_all, whole
        mb.barrier(2)

    # ---- end-to-end leg (host buffers through the C-ABI), every rank its shard ----------------------
    span = back + n + ahead
    p_in, h_in = pinned(span, np.uint8)
    h_in[:] = host
    p_len, h_len = pinned(2 * span, np.uint16)
    p_dist, h_dist = pinned(2 * span, np.uint16)

    def e2e_step() -> None:
        check(L.sqz_gpu_match_table(C.cast(p_in, _lib.u8p), span, WINDOW, MIN_LEN, MAX_LEN, MAX_DIST,
                                    C.cast(p_len, _lib.u16p), C.cast(p_dist, _lib.u16p)), "sqz_gpu_match_table")

    for _ in range(min(args.warmup, 1)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    barrier()
    e2e_sec = max_over_ranks((time.perf_counter() - t0) / args.e2e_steps)
    tab = d_table[: 1 << 20].cpu().numpy().view(np.uint32)
    assert ((tab >> 16) == h_len[back: back + (1 << 20)]).all() and \
           ((tab & 0xFFFF) == h_dist[back: back + (1 << 20)]).all(), "host ABI and device ABI disagree"
    L.sqz_gpu_host_free(p_len); L.sqz_gpu_host_free(p_dist)
    del h_len, h_dist
    e2e_h2d = sum(s.back + s.n + s.ahead for s in plan)
    e2e_d2h = 4 * e2e_h2d

    # second end-to-end sample: the token stream, host to host, through the one-call entry points
    tok_e2e = None
    if world > 1:
        mb.barrier(3)
    if rank == 0:
        try:
            if world == 1:
                data_p, data_n = p_in, span
            else:
                data_p, whole_pin = pinned(total, np.uint8)
                whole_pin[:] = corpus.synthetic(total, 0)
                data_n = total
            p_tok, h_tok = pinned(4 * data_n + 64, np.uint32)
            cnt = C.c_size_t()
            devs = (C.c_int * world)(*range(world))

            def tok_step():
                if world == 1:
                    check(L.sqz_gpu_tokens(C.cast(data_p, _lib.u8p), data_n, WINDOW, MIN_LEN, MAX_LEN, MAX_DIST,
                                           C.cast(p_tok, _lib.u32p), data_n, C.byref(cnt)), "sqz_gpu_tokens")
                else:
                    check(L.sqz_gpu_tokens_multi(devs, world, C.cast(data_p, _lib.u8p), data_n, WINDOW, MIN_LEN, MAX_LEN,
                                                 MAX_DIST, p_tok, data_n, C.byref(cnt), None), "sqz_gpu_tokens_multi")
            tok_step()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                tok_step()
            dt = (time.perf_counter() - t0) / args.e2e_steps
            assert cnt.value == n_tokens, (cnt.value, n_tokens)
            tok_e2e = {"value": total / 1e6 / dt, "unit": "MB/s", "seconds": dt, "tokens": int(cnt.value),
                       "h2d_bytes_per_step": int(data_n), "d2h_bytes_per_step": int(4 * cnt.value),
                       "call": ("sqz_gpu_tokens" if world == 1 else "sqz_gpu_tokens_multi over %d devices from rank 0" % world)
                               + "(host pinned in, host pinned tokens out)"}
            L.sqz_gpu_host_free(p_tok)
            del h_tok
        except Exception as e:
            tok_e2e = {"value": None, "error": repr(e)}
    if world > 1:
        mb.barrier(4)

    # ---- weak-scaling leg (N > 1): the round-1 layout, every rank owns --size bytes ------------------
    weak = None
    if world > 1 and args.weak_steps > 0:
        del leg, d_table
        torch.cuda.empty_cache()
        wplan = shard.plan(total * world, world, MAX_DIST, MAX_LEN)
        wleg = run_leg(total * world, wplan[rank], args.weak_steps, 1, gather=False, timed_kernel=False)
        weak = {"value": total * world / 1e6 / wleg["sec"], "unit": "MB/s", "bytes_per_gpu": total,
                "ms_per_step": wleg["sec"] * 1e3, "steps": args.weak_steps, "warmup": 1,
                "note": "N x %d MiB, same step without the token gather" % (total >> 20)}
        del wleg

    if rank != 0:
        if world > 1:
            mb.close()
            dist.destroy_process_group()
        return

    # ---- by kind of data (N = 1): 64 MiB of text, ELF and image bytes each --------------------------
    per_kind = None
    if world == 1 and args.kind_bytes > 0:
        fx = corpus.fixtures()
        kinds = {"text": [fx["confucius.txt"], fx["laozi.txt"]], "elf": [fx["x64.elf"], fx["arm64.elf"]],
                 "image": [fx["mandrill.bmp"], fx["mandrill.png"]]}
        per_kind = {}
        size = args.kind_bytes
        kb = torch.zeros(size + 1024, dtype=torch.uint8, device=dev)
        kt = torch.empty(size, dtype=torch.int32, device=dev)
        kw = torch.empty(L.sqz_gpu_match_workspace(size), dtype=torch.uint8, device=dev)
        for name, parts in kinds.items():
            basek = np.concatenate(parts)
            data = np.tile(basek, size // basek.size + 1)[:size].copy()
            kb[:size].copy_(torch.from_numpy(data))
            best = 1e9
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record(stream)
                check(L.sqz_gpu_match_table_device_ws(kb.data_ptr(), 0, size, 0, MIN_LEN, MAX_LEN, MAX_DIST, kt.data_ptr(),
                                                      kw.data_ptr(), stream.cuda_stream), "match_table")
                e1.record(stream)
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) * 1e-3)
            per_kind[name] = {"value": size / 1e6 / best, "unit": "MB/s", "bytes": size, "ms": best * 1e3}
        del kb, kt, kw

    # ---- CPU baseline: the unmodified reference on one core, bounded sample -----
    cpu = None
    try:
        from oracle import Reference
        ref = Reference.get(release=True)
        # 8 slices spread evenly over the shard (its head alone is text and flatters the reference)
        slices, each = 8, max(args.cpu_sample // 8, 4096)
        secs = 0.0
        for k in range(slices):
            off = (g0 + k * (n // slices)) // 4096 * 4096
            ref.compress(corpus.synthetic(each, off), 15)
            secs += ref.last_seconds
        sample_bytes = slices * each
        cpu = {"value": sample_bytes / 1e6 / secs, "unit": "MB/s", "cores": 1, "kind": "reference",
               "sample": "%d slices x %d KiB spread evenly over the shard, each through the unmodified reference's "
                         "squeeze.compress (oracle/_ref, -O3 -DNDEBUG, window 2^15, empty window at the slice start), "
                         "%.1f s on 1 of %d host cores" % (slices, each >> 10, secs, os.cpu_count() or 1)}
    except Exception as e:  # the oracle is only the yardstick; never let it sink the measurement
        cpu = {"value": None, "unit": "MB/s", "cores": 0, "kind": "reference", "sample": "unavailable: %r" % (e,)}

    # ---- whole codec: sqz_compress (GPU search + serial host entropy stage), bounded sample ----
    comp = None
    try:
        import sqz_b200 as sq
        sample = np.ascontiguousarray(host[back: back + min(n, args.compress_sample)])
        # one untimed call first, like the W warm-up steps of the main metric: it allocates the
        # pipeline's pinned and device buffers (two slots of 32 MiB chunks), which later calls reuse,
        # and touches the caller's output buffer (the C API's caller owns it; sq.compress(into=...))
        out_buf = np.empty(sq.capacity(sample.size), np.uint8)
        warm = sample[: min(sample.size, (129 << 20))]
        t0 = time.perf_counter()
        sq.compress(warm, 15, into=out_buf)
        dt_warm = time.perf_counter() - t0
        st = {}
        t0 = time.perf_counter()
        blob = sq.compress(sample, 15, stats=st, into=out_buf)
        dt = time.perf_counter() - t0
        import os as _os
        cores = _os.cpu_count() or 1
        coder_threads = 1 if cores < 2 else 2 if cores < 8 else 4
        back_buf = np.empty(sample.size, np.uint8)
        back_buf[:] = 0                  # touched, like the output buffer of the compressor
        t0 = time.perf_counter()
        back_again = sq.decompress(blob, into=back_buf)
        dt_dec = time.perf_counter() - t0
        comp = {"value": sample.size / 1e6 / dt, "unit": "MB/s", "sample_bytes": int(sample.size),
                "compressed_bytes": len(blob), "seconds": dt, "search_wait_seconds": st["search_seconds"],
                "entropy_seconds": st["entropy_seconds"], "tokens": st["tokens"],
                "entropy_ns_per_token": st["entropy_seconds"] * 1e9 / max(st["tokens"], 1),
                "warmup": "one untimed sqz_compress of the first %d MiB (%.2f s: it allocates the pipeline's "
                          "pinned and device buffers and touches the output buffer)" % (warm.size >> 20, dt_warm),
                "decompress": {"value": sample.size / 1e6 / dt_dec, "unit": "MB/s", "seconds": dt_dec,
                               "round_trip_identical": bool(back_again.size == sample.size and (back_again == sample).all())},
                "host_threads": coder_threads + 1, "host_cores": cores,
                "note": "sqz_compress(host in, caller's host buffer out), coder_threads = 0 (automatic: on 8 cores "
                        "and more a model thread that counts symbols block-wise, three emitter threads working on "
                        "segments of 16 Ki tokens, the calling thread appending them in order); the GPU stream hands "
                        "over symbol words in 32 MiB chunks (SURVEY 8f N3) and is what the coder waits for now; "
                        "sqz_decompress is host only, one thread"}
    except Exception as e:
        comp = {"value": None, "error": repr(e)}

    ms_per_step = sec * 1e3
    value = total / 1e6 / sec
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    f_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    smem_peak = SMEM_BYTES_PER_CLK_PER_SM * sms * f_mhz * 1e6 / 1e9            # GB/s at the clock seen under load
    cc = cc_count(g0, n, MAX_DIST)                                             # this rank's launch
    cc_job = cc_count(0, total, MAX_DIST)
    achieved = cc * 4 / t_match / 1e9 if t_match > 0 else None
    # The bit-sliced kernel issues no load per candidate-compare, so the shared-memory figure can
    # exceed 1.  What binds it is the integer ALU pipe: 16 lanes/clk per SM sub-partition, i.e. half
    # a warp-instruction per clock.  The instruction count of its loop comes from the committed ncu
    # capture of this kernel (profiles/r02_roofline_inputs.json), not from a constant in this file.
    ri = roofline_inputs()
    alu_instr, cc_iter = ri.get("alu_instr_per_warp_iteration"), ri.get("cc_per_warp_iteration")
    alu_ceiling = 0.5 * 4 * sms * f_mhz * 1e6 * cc_iter / alu_instr if alu_instr and cc_iter else None      # CC/s
    quiet_instr = (ri.get("quiet_body") or {}).get("alu_instr_per_warp_iteration")
    quiet_ceiling = 0.5 * 4 * sms * f_mhz * 1e6 * cc_iter / quiet_instr if quiet_instr and cc_iter else None
    cc_per_s = cc / t_match if t_match > 0 else None
    traffic = None
    if ri.get("dram_bytes_per_input_byte") is not None:
        traffic = int(ri["dram_bytes_per_input_byte"] * n)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_bytes = n * (1 + 4)                                                    # input read + table write
    line = {
        "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args),
        "e2e": {"value": total / 1e6 / e2e_sec, "unit": "MB/s",
                "h2d_bytes_per_step": int(e2e_h2d), "d2h_bytes_per_step": int(e2e_d2h),
                "call": "sqz_gpu_match_table(host pinned in, host pinned len/dist out), every rank its shard",
                "steps": args.e2e_steps, "tokens": tok_e2e},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {
            "bound": "smem", "kernel": "match_table",
            "achieved": achieved, "peak": smem_peak, "unit": "GB/s",
            "frac": achieved / smem_peak if achieved else None,
            "traffic": traffic,
            "note": "algorithmic shared-memory bytes = 4 B per candidate-compare (SURVEY 8d), %d CC per launch "
                    "(rank 0's shard); peak = 128 B/clk/SM x %d SMs x %.0f MHz (SM clock sampled under this load); "
                    "north_star fixes the smem compare bound, HBM is shown in 'hbm'" % (cc, sms, f_mhz),
            "cc_per_launch": cc, "cc_per_step_all_ranks": cc_job, "visited_cc_per_step_all_ranks": visited,
            "visited_note": "what the reference's own scan walks: it stops at the nearest max_len candidate "
                            "(squeeze.h:353); %.2f %% of the algorithmic count" % (100.0 * visited / cc_job),
            "kernel_ms": t_match * 1e3, "kernel_ms_max_over_ranks": t_match_max * 1e3,
            "kernel_launches_timed": int(n_timed),
            "kernel_share_of_step": (t_match * 1e3) / ms_per_step if ms_per_step else None,
            "binding_resource": {
                "name": "integer ALU pipe (LOP3/SHF), 0.5 warp-instr/clk per SM sub-partition",
                "alu_instr_per_warp_iteration": alu_instr, "cc_per_warp_iteration": cc_iter,
                "ceiling_cc_per_s": alu_ceiling, "achieved_cc_per_s": cc_per_s,
                "frac": cc_per_s / alu_ceiling if cc_per_s and alu_ceiling else None,
                "alu_instr_per_warp_iteration_quiet_body": quiet_instr, "ceiling_cc_per_s_quiet_body": quiet_ceiling,
                "source": ri.get("source"), "captured_at_commit": ri.get("commit"),
                "note": "achieved counts the whole sqz_gpu_match_table_device call: bit-sliced kernel, edge tiles "
                        "and the finish kernel; the ceiling is that of the loop body with the need masks -- a warp "
                        "whose data is quiet (an image) runs the shorter body and can exceed it, which is why per_kind "
                        "shows image data above this ceiling's MB/s",
            },
            "traffic_note": ri.get("traffic_note"),
        },
        "hbm": {"achieved": hbm_bytes / t_match / 1e9 if t_match > 0 else None, "peak": hbm_peak, "unit": "GB/s",
                "frac": hbm_bytes / t_match / 1e9 / hbm_peak if t_match > 0 else None,
                "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback"},
        "parity_check": parity,
        "gather": gathered if gathered is not None else {"how": gather_how},
        "weak": weak,
        "per_kind": per_kind,
        "cpu_baseline": cpu,
        "sqz_compress_e2e": comp,
        "tokens_per_step": n_tokens,
    }
    emit(line)
    if world > 1:
        if gather_base:
            L.sqz_gpu_device_free(gather_base)
        mb.close(unlink=True)
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The one JSON line, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout carries exactly one JSON line.  Libraries that print there (NCCL's version banner when
    # the box sets NCCL_DEBUG, torchrun children) are pointed at stderr for the whole run.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=1 << 30, help="bytes of the whole job (cut into --gpus shards)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--weak-steps", type=int, default=1, help="timed steps of the weak-scaling leg (N > 1); 0 = skip")
    ap.add_argument("--kind-bytes", type=int, default=64 << 20, help="bytes per kind of the per_kind table (N = 1); 0 = skip")
    ap.add_argument("--cpu-sample", type=int, default=512 << 10)
    ap.add_argument("--compress-sample", type=int, default=256 << 20)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write samples of the last timed step's match table and token stream to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
