#!/usr/bin/env python
"""bench.py -- GiB/s of chunk + SHA-256 (+ probe) at 4 MiB average chunk (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (our CUDA path; N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   (CPU reference arm: the oracle on host cores)
    python bench.py ... --dump-outputs DIR                    (also writes the last timed step's chunk records as .npy,
                                                               so that two builds can be compared on the same inputs)

A "step" is one pass of the hot path (K1 scan -> K2 resolve -> K3 SHA-256 -> K4 probe) over one
batch = BASELINE config[1]: 1024 x 64 MiB synthetic files per GPU, resident in HBM, generated on
the device before the timed region (inputs are 64 GiB >> 126 MB L2, so no L2 flush is needed).
Steps are submitted asynchronously (the C ABI's submit/wait form) so the serial SHA-256 tail of
one batch's longest chunk overlaps the next batch; all K steps complete inside the timed region.
One JSON line on stdout (rank 0).  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

# 32 hardware work queues instead of the default 8: the engine keeps up to 28 CUDA streams busy and
# streams that alias one queue serialise (must be set before the CUDA context exists)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

GIB = float(1 << 30)
METRIC = "GiB/s chunked+SHA-256 at 4 MiB avg chunk; bit-exact boundaries/digests vs ref"


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def instr_ceiling(sm_total, sm_mhz, value_gbs):
    """Integer-pipe bound of SHA-256 on this GPU.  Every one of the chip's SMs runs SHA work (124 the bulk kernel, 24
    the long-chunk kernel), so the bound counts ALL of them: 64 ALU-pipe thread-instructions / clk / SM
    (profiles/r01_microbench.txt) over the ALU instructions per byte of the shipped kernel
    (profiles/r02_sass_mix.txt: loop of k_sha_tuned<2>, 1228 ALU-pipe instructions per 64 B block)."""
    if not sm_mhz:
        return None
    alu_per_block = 1228.0
    gbs = sm_total * 64 * float(sm_mhz) * 1e6 / (alu_per_block / 64.0) / 1e9
    return {"alu_pipe_GBps": gbs, "frac_of_alu_pipe": value_gbs / gbs if gbs else None, "sm_count": sm_total,
            "alu_instr_per_64B": alu_per_block,
            "source": "profiles/r02_sass_mix.txt (SASS count), profiles/r01_microbench.txt (64 thread-ops/clk/SM)"}


DUMP_LIMIT = 64_000_000   # bytes of array data --dump-outputs writes at most


def dump_outputs(out_dir, rec, known):
    """Writes the chunk records of one step as DIR/<field>.npy: row (index in the step's record list), stream and end_off
    as float64, digest (n x 32 bytes) and known as float32.  Above DUMP_LIMIT a fixed, seeded sample of rows is written."""
    n = len(rec)
    cap = DUMP_LIMIT // (3 * 8 + 32 * 4 + 4)
    rows = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    r = rec[rows]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("row", rows.astype(np.float64)), ("stream", r["stream"].astype(np.float64)),
                    ("end_off", r["end_off"].astype(np.float64)), ("digest", r["digest"].astype(np.float32)),
                    ("known", (np.asarray(known)[rows] != 0).astype(np.float32))):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def union_ms(intervals):
    """Total length of the union of [t0,t1] intervals (ms)."""
    tot, cur0, cur1 = 0.0, None, None
    for a, b in sorted(intervals):
        if cur0 is None:
            cur0, cur1 = a, b
        elif a <= cur1:
            cur1 = max(cur1, b)
        else:
            tot += cur1 - cur0
            cur0, cur1 = a, b
    if cur0 is not None:
        tot += cur1 - cur0
    return tot


# ------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle restatement on all host cores (the reference's
# own Go code cannot be built here: un-vendored module, no Go toolchain -- DESIGN.md).
# ------------------------------------------------------------------------------------------
def cpu_thread_candidates(cores: int):
    c = sorted({max(1, cores // 4), max(1, cores // 2), cores})
    return c


def cpu_pass(n_files: int, file_len: int, cores: int, repeats: int = 1, first_file: int = 0):
    """Times the oracle on `n_files` files; sweeps the thread count (a box may expose more logical
    CPUs than its quota / physical cores can feed) and returns the best: (GiB/s, seconds, threads)."""
    import oracle

    files = oracle.corpus_files(oracle.corpus(seed=2, file_len=file_len), first_file, n_files, threads=cores)
    cfg = oracle.config(4 << 20)
    best = None
    for th in cpu_thread_candidates(cores):
        for _ in range(repeats):
            t0 = time.perf_counter()
            oracle.chunk_digest_streams(cfg, files, threads=th)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, th)
    return n_files * file_len / best[0] / GIB, best[0], best[1]


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    file_len = args.file_mib << 20
    n_sample = max(cores, min(4 * cores, (8 << 30) // file_len))
    import oracle

    files = oracle.corpus_files(oracle.corpus(seed=2, file_len=file_len), 0, n_sample, threads=cores)
    cfg = oracle.config(4 << 20)
    # warm-up doubles as the thread-count pick (all the host threads it can USE, not merely see)
    best = None
    for th in cpu_thread_candidates(cores):
        t0 = time.perf_counter()
        oracle.chunk_digest_streams(cfg, files, threads=th)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, th)
    threads = best[1]
    for _ in range(max(0, args.warmup - 1)):
        oracle.chunk_digest_streams(cfg, files[:threads], threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rec = oracle.chunk_digest_streams(cfg, files, threads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rec, rec["flags"] & 1)
    val = n_sample * file_len * args.steps / dt / GIB
    sample = (f"{n_sample} x {args.file_mib} MiB files of the cfg2 corpus per step, one stream per task on "
              f"{threads} threads (best of {cpu_thread_candidates(cores)} on {cores} logical CPUs)")
    cores = threads
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
        "config": {"workload": f"cfg2: {args.files} x {args.file_mib} MiB files, 4 MiB avg chunk", "sample": sample},
        "cpu_baseline": {"value": val, "unit": "GiB/s", "cores": cores, "kind": "port", "sample": sample,
                         "sha": "SHA-NI" if oracle.lib().orc_have_shani() else "portable C",
                         "note": "restated CPU baseline (oracle/oracle.c), not the Go binary: the reference's "
                                 "arithmetic is the un-vendored Go module pbs-plus/pxar v0.19.2; no Go toolchain"},
        "e2e": {"value": val, "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------------
def cpu_legs_b1_b3():
    """BASELINE.md B1 / B3: the oracle on cfg1 (one 1 GiB stream, seed 1, 4 MiB average) with ONE thread -- whole path,
    scan only, SHA-256 only."""
    import oracle

    n = 1 << 30
    data = oracle.corpus_file(oracle.corpus(seed=1, file_len=n), 0)
    cfg = oracle.config(4 << 20)
    t0 = time.perf_counter(); rec = oracle.chunk_digest(cfg, data); t_all = time.perf_counter() - t0
    t0 = time.perf_counter(); ends = oracle.chunk_ends(cfg, data); t_scan = time.perf_counter() - t0
    t0 = time.perf_counter()
    s = 0
    for e in ends.tolist():
        oracle.sha256(data[s:e]); s = e
    t_sha = time.perf_counter() - t0
    assert rec["end_off"].tolist() == ends.tolist()
    return {"B1_chunk+sha_1thread_GiBps": n / t_all / GIB, "B3_scan_only_1thread_GiBps": n / t_scan / GIB,
            "B3_sha_only_1thread_GiBps": n / t_sha / GIB, "input": "cfg1: one 1 GiB stream (seed 1), 4 MiB average chunk",
            "chunks": int(len(rec)), "sha": "SHA-NI" if oracle.lib().orc_have_shani() else "portable C"}


def h2d_roofline(torch, host_arr, nbytes=8 << 30):
    """Measured pinned-host -> device copy bandwidth on THIS box in THIS run: the roofline of the e2e figure."""
    n = min(len(host_arr), nbytes)
    dst = torch.empty(n, dtype=torch.uint8, device="cuda")
    src = torch.from_numpy(np.asarray(host_arr[:n]))
    dst.copy_(src, non_blocking=True); torch.cuda.synchronize()
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); dst.copy_(src, non_blocking=True); e1.record(); e1.synchronize()
        best = max(best, n / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del dst
    return best


def run_distinct(args, eng, pg, torch, cfg, total_gib=768, batch_files=256, nbuf=7, early=True):
    """value_distinct: the same path over NON-REPEATING data (the cfg3 corpus): every batch is generated on the device,
    hashed ONCE, and its buffer is refilled as soon as the device no longer reads it -- with `early` (the default,
    PBSGPU_BATCH_EARLY_INPUT) that is when the bulk pass and the copy of the long chunks into the library's arena are done,
    without it only when the job's last 16 MiB chain ended.  Depth is bounded by HBM (nbuf x batch + arena), not by the
    number of steps -- the honest counterpart of the repeated-buffer headline.  A second context generates the
    next batches concurrently (its kernels share the GPU with the hashing); the wall time INCLUDES that generation."""
    import queue
    import threading
    from collections import deque

    file_len = args.file_mib << 20
    corp = pg.corpus(seed=3, file_len=file_len, block_len=4 << 20, run_blocks=8, dup_permille=300)
    known = eng.digest_set(1 << 21)
    gen = pg.Engine(eng.device)
    bufs = [torch.empty(batch_files * file_len, dtype=torch.uint8, device="cuda") for _ in range(nbuf)]
    off = np.arange(batch_files, dtype=np.uint64) * file_len
    ln = np.full(batch_files, file_len, dtype=np.uint64)
    n_batches = max(nbuf, (total_gib << 30) // (batch_files * file_len))
    # generation alone (one batch, nothing else running): what the overlapped generator costs the hashing at most
    gen.corpus_fill(corp, 0, batch_files, bufs[0], file_len)
    t0 = time.perf_counter(); gen.corpus_fill(corp, 0, batch_files, bufs[0], file_len); gen_alone = time.perf_counter() - t0
    free_q, full_q = queue.Queue(), queue.Queue()
    for b in range(nbuf):
        free_q.put(b)
    err = []

    def producer():
        try:
            for b in range(n_batches):
                slot = free_q.get()
                gen.corpus_fill(corp, b * batch_files, batch_files, bufs[slot], file_len)
                full_q.put((b, slot))
        except Exception as ex:  # pragma: no cover
            err.append(repr(ex))
        full_q.put(None)

    chunks = hits = 0
    pend_in, pend_out = deque(), deque()      # jobs whose input is still being read / whose records are not collected yet
    max_jobs = max(24, 2 * nbuf)

    def release_one():
        job, slot = pend_in.popleft()
        job.wait_input()                      # bulk pass + long-chunk gather done: the buffer can be refilled
        free_q.put(slot)

    def drain():
        nonlocal chunks, hits
        rec, _ = pend_out.popleft().wait()
        chunks += len(rec); hits += int((rec["flags"] & 1).sum())

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    th = threading.Thread(target=producer, daemon=True)
    th.start()
    done = False
    while not done or pend_in:
        item = None
        if not done:
            try:
                item = full_q.get(block=not pend_in)
            except queue.Empty:
                item = None
            else:
                if item is None:
                    done = True
        if item is not None:
            _, slot = item
            job = eng.submit(cfg, bufs[slot], off, ln, digest_set=known, early_input=early)   # corpus order: the set sees it in order
            pend_in.append((job, slot)); pend_out.append(job)
        while pend_in and pend_in[0][0].input_done():
            release_one()
        if pend_in and (item is None or len(pend_in) > nbuf - 2):
            release_one()                     # nothing to submit (or the generator is out of buffers): wait for the oldest input
        while len(pend_out) > max_jobs:
            drain()
    while pend_out:
        drain()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    th.join()
    gen.close()
    nbytes = n_batches * batch_files * file_len
    del bufs
    torch.cuda.empty_cache()
    if err:
        return {"value": None, "error": err[0]}
    return {"value": nbytes / wall / GIB, "unit": "GiB/s", "bytes": nbytes, "batches": n_batches,
            "batch_GiB": batch_files * file_len / GIB, "buffers": nbuf, "early_input": bool(early),
            "chunks": chunks, "known_chunks": hits,
            "hit_rate": hits / max(1, chunks), "seconds": wall,
            "generation_alone_GBps": batch_files * file_len / gen_alone / 1e9,
            "generation_share_if_serial": (n_batches * gen_alone) / wall,
            "workload": "cfg3 corpus (seed 3, 30 % duplicate 4 MiB blocks in runs of 8), every byte generated on the device and "
                        "hashed once; generation runs concurrently in a second context and is INSIDE the wall time"}


def expected_cfg4_hits(world, n_files, file_mib):
    """Known-chunk count of the first pass over the global cfg4 corpus, from a ONE-set run (profiles/r02_cfg4_expected.json,
    produced by `bench.py --workload cfg4verify`)."""
    p = ROOT / "profiles" / "r02_cfg4_expected.json"
    if not p.exists():
        return None
    try:
        for e in json.loads(p.read_text())["entries"]:
            if e["world"] == world and e["files_per_rank"] == n_files and e["file_mib"] == file_mib:
                return e
    except Exception:
        return None
    return None


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch

    import pbs_plus_b200 as pg

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev_t = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev_t)     # plumbing only: barrier, max over ranks, id broadcast
    eng = pg.Engine(local_rank, profiling=True)
    info = eng.device_info()
    sm_total = torch.cuda.get_device_properties(local_rank).multi_processor_count
    file_len = args.file_mib << 20
    n_files = args.files
    budget = info["free_mem"] - (6 << 30)
    while n_files * file_len > budget and n_files > 1:
        n_files //= 2
    reduced = n_files != args.files
    data = torch.empty(n_files * file_len, dtype=torch.uint8, device=dev_t)
    if world > 1:
        # cfg4 (BASELINE configs[3]): ONE corpus with duplicate runs (seed 3, 30 % of the 4 MiB blocks in runs of 8),
        # sharded by contiguous file ranges -- rank r holds files [r*n, (r+1)*n) -- so duplicate runs cross rank
        # boundaries and only the NCCL all-gather of the digests makes the KNOWN flags equal a single-GPU run
        corp = pg.corpus(seed=3, file_len=file_len, block_len=4 << 20, run_blocks=8, dup_permille=300)
        wl = (f"cfg4: {world} x {n_files} x {args.file_mib} MiB files of ONE duplicate-run corpus (seed 3, 30 % dup 4 MiB blocks, "
              f"runs of 8) sharded by file range, {args.avg_kib} KiB avg chunk, chunk+SHA-256 per rank + pbsgpu_set_allgather "
              f"(NCCL) of the digests every step, HBM-resident")
    else:
        corp = pg.corpus(seed=2, file_len=file_len)
        wl = (f"cfg2: {n_files} x {args.file_mib} MiB synthetic files per GPU (seed 2), {args.avg_kib} KiB avg "
              f"chunk (min avg/4, max 4*avg), chunk+SHA-256+probe, HBM-resident")
    eng.corpus_fill(corp, rank * n_files, n_files, data, file_len)
    off = np.arange(n_files, dtype=np.uint64) * file_len
    ln = np.full(n_files, file_len, dtype=np.uint64)
    cfg = pg.buzhash.NewConfig(args.avg_kib)  # default 4096: the reference's call (commit.go:303) = 4 MiB
    known = eng.digest_set(1 << 20)
    comm = None
    if world > 1:
        ident = [pg.NcclComm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0, device=dev_t)
        comm = pg.NcclComm(eng, ident[0], world, rank)       # the library's own communicator: the merge is C ABI, not torch
    launches = {"mine": 0}

    def submit():
        # N = 1: the probe is fused into the job (K4 on the job's stream).  N > 1: the probe needs the other ranks' digests
        return eng.submit(cfg, data, off, ln, digest_set=known if world == 1 else None)

    def finish(job):
        rec, t = job.wait()
        launches["mine"] += t["scan_launches"] + t["sha_launches"] + t["other_launches"]
        if world > 1:   # the ONE exchange step: pbsgpu_set_allgather (counts + padded digests over NCCL/NVLink, in-order insert)
            flags = known.allgather(comm, rec["digest"])
            launches["mine"] += 4    # compaction + make_keys + mark/probe + insert
        else:
            flags = (rec["flags"] & 1).astype(np.uint8)
        return rec, t, flags

    # ---- warm-up (untimed): W full steps, sequential, then one pipelined burst of K steps so that the
    # library's scratch pool (device + pinned buffers, events) is populated for K jobs in flight
    first_pass = None
    for _ in range(max(1, args.warmup)):
        r = finish(submit())
        if first_pass is None:
            first_pass = (len(r[0]), int(r[2].sum()))
    check = {"chunks_first_pass": first_pass[0], "known_first_pass": first_pass[1]}
    if world > 1:
        tot = torch.tensor(list(first_pass), dtype=torch.int64, device=dev_t)
        dist.all_reduce(tot)
        check = {"chunks_first_pass": int(tot[0].item()), "known_first_pass": int(tot[1].item()), "set_size": len(known)}
        # every replica holds the same set, and it accounts for every chunk: distinct = chunks - known
        if check["set_size"] != check["chunks_first_pass"] - check["known_first_pass"]:
            raise SystemExit(f"bench.py: rank {rank}: digest-set replica inconsistent: {check}")
        exp = expected_cfg4_hits(world, n_files, args.file_mib)
        check["expected_known_single_set"] = exp["known"] if exp else None
        if exp and (exp["known"] != check["known_first_pass"] or exp["chunks"] != check["chunks_first_pass"]):
            raise SystemExit(f"bench.py: cfg4 hit count differs from the single-set run: {check} vs {exp}")
        check["hit_rate_first_pass"] = check["known_first_pass"] / max(1, check["chunks_first_pass"])
    if not args.no_prewarm:
        for j in [submit() for _ in range(min(args.steps, args.inflight or args.steps))]:
            finish(j)
    # latency of ONE isolated batch (includes the serial tail of the longest chunk)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, t_iso, _ = finish(submit())
    torch.cuda.synchronize()
    iso_ms = (time.perf_counter() - t0) * 1e3

    # ---- timed region: exactly K steps
    launches["mine"] = 0
    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    from collections import deque
    q, results = deque(), []
    inflight = args.inflight if args.inflight > 0 else args.steps
    for _ in range(args.steps):
        if len(q) >= inflight:
            results.append(finish(q.popleft()))
        q.append(submit())
    while q:
        results.append(finish(q.popleft()))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev1.record()
    ev1.synchronize()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    if world > 1:
        tms = torch.tensor([ms], dtype=torch.float64, device=dev_t)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    step_bytes = n_files * file_len
    value = world * step_bytes * args.steps / (ms / 1e3) / GIB

    timings = [r[1] for r in results]
    n_chunks = int(timings[0]["chunks"])
    hit_last = float((results[-1][2] != 0).mean()) if len(results[-1][2]) else 0.0
    if hit_last != 1.0:
        raise SystemExit(f"bench.py: rank {rank}: a re-hashed step must find every digest known, got {hit_last}")
    sha_union = union_ms([(t["sha_t0"], t["sha_t1"]) for t in timings])
    scan_union = union_ms([(t["scan_t0"], t["scan_t1"]) for t in timings])
    peak, peak_src = measured_peaks()
    traffic = ncu_traffic() if (n_files == 1024 and args.file_mib == 64) else None
    # the roofline line follows from the SAME clock as `value`: algorithmic bytes of one step (per GPU) / ms_per_step
    step_gbs = step_bytes / (ms / args.steps / 1e3) / 1e9
    sha_gbs = step_bytes * args.steps / (sha_union / 1e3) / 1e9 if sha_union > 0 else 0.0
    scan_gbs = step_bytes * args.steps / (scan_union / 1e3) / 1e9 if scan_union > 0 else 0.0

    out = {
        "metric": METRIC, "value": value, "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic",
        "config": {
            "workload": wl,
            "reduced_to_fit_hbm": reduced, "chunks_per_step": n_chunks, "parallelism": f"files sharded x{world}",
            "l2": "inputs (>= 64 GiB) far exceed the 126 MB L2; no flush needed",
            "pipelining": "K steps submitted asynchronously over the SAME resident batch (13 stream slots, FIFO per slot); all "
                          "complete inside the timed region; see value_distinct for non-repeating data",
            "inflight": args.inflight or args.steps, "sm_partition(long,bulk,scan)": list(eng.partition_info()) + [eng.scan_partition_sms()],
            "known_hit_rate_last_step": hit_last, "first_pass_check": check,
        },
        "clocks": clocks,
        "gpu_launches": launches["mine"],
        "single_batch_latency_ms": iso_ms,
        "roofline": {
            "bound": "hbm", "kernel": "k_sha_tuned / k_sha_split (K3, dominant; instruction-bound integer work, see DESIGN.md)",
            "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
            "traffic": traffic["total"] if traffic else None, "traffic_detail": traffic,
            "algorithmic_bytes_per_launch": step_bytes, "peak_source": peak_src,
            "how": "algorithmic bytes of one step on one GPU (1 per input byte) / ms_per_step (the driver-checkable clock: "
                   "CUDA events around the K timed steps, max over ranks); all kernels of the step included",
            "kernel_intervals": {
                "what": "diagnostic: bytes of all K launches / union of their CUDA-event intervals on the launching streams",
                "sha_GBps": sha_gbs, "scan_GBps": scan_gbs, "sha_frac": sha_gbs / peak, "scan_frac": scan_gbs / peak},
            "instruction_ceiling": instr_ceiling(sm_total, clocks.get("sm_mhz"), step_gbs),
            "isolated_step_ms": {k: t_iso[k] for k in ("scan_ms", "sort_ms", "resolve_ms", "sha_ms", "sha_long_ms",
                                                        "sha_bulk_ms", "set_ms", "total_ms")},
        },
    }
    if args.timeline:
        out["timeline"] = [{k: round(float(t[k]), 2) for k in ("scan_t0", "scan_t1", "sha_t0", "sha_t1", "sha_long_ms", "sha_bulk_ms", "total_ms")}
                           for t in timings]
    # ---- untimed post-run parity check (VERDICT r1 next-1a): the record list of the LAST timed step equals the oracle's
    last_rec = results[-1][0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_rec, results[-1][2])
    if world == 1 and not args.no_verify and not reduced and args.avg_kib == 4096:
        import oracle
        t0 = time.perf_counter()
        ref = oracle.corpus_chunk_digest(oracle.config(4 << 20), oracle.corpus(seed=2, file_len=file_len), 0, n_files)
        ok = (len(ref) == len(last_rec) and ref["end_off"].tobytes() == last_rec["end_off"].tobytes()
              and ref["digest"].tobytes() == last_rec["digest"].tobytes() and ref["stream"].tobytes() == last_rec["stream"].tobytes())
        out["verify"] = {"equal_to_oracle": bool(ok), "records": int(len(ref)), "seconds": time.perf_counter() - t0,
                         "what": "every (stream, end offset, digest) of the last timed step vs oracle/ on the host cores (untimed)"}
        if not ok:
            print(json.dumps(out), flush=True)
            raise SystemExit("bench.py: GPU records differ from the oracle")
    # "next" rows measured beside the headline (never inside its timed region): K7, the commit walk's per-file
    # XXH3-64 (SURVEY 8 f2), over the same resident files through the blocking C call.
    try:
        eng.xxh3_batch(data, off, ln)
        t0 = time.perf_counter()
        hashes = eng.xxh3_batch(data, off, ln)
        dt = time.perf_counter() - t0
        try:
            import xxhash                     # independent implementation (libxxhash), when the box has it
            check_x = bool(int(hashes[0]) == xxhash.xxh3_64_intdigest(data[: file_len].cpu().numpy().tobytes()))
        except ImportError:
            check_x = None
        out["next_rows"] = {"f2_xxh3_file_hash": {
            "GBps": step_bytes / dt / 1e9, "frac_of_hbm_peak": step_bytes / dt / 1e9 / peak, "ms": dt * 1e3,
            "files": n_files, "file0_equals_libxxhash": check_x,
            "how": "wall time of one pbsgpu_xxh3_batch call over the step's resident files (incl. launch + D2H of the hashes)"}}
    except Exception as ex:   # an aid next to the headline: never fails the bench line
        out["next_rows"] = {"f2_xxh3_file_hash": {"error": repr(ex)}}
    del data
    torch.cuda.empty_cache()
    if world == 1 and not args.no_distinct:
        try:
            out["value_distinct"] = run_distinct(args, eng, pg, torch, cfg, total_gib=args.distinct_gib, nbuf=args.distinct_bufs,
                                                 batch_files=args.distinct_batch_files, early=bool(args.distinct_early))
        except Exception as ex:
            out["value_distinct"] = {"value": None, "error": repr(ex)}
        torch.cuda.empty_cache()
    if world > 1 and os.environ.get("PBSGPU_BENCH_CLOSE_COMM_BEFORE_E2E") and comm is not None:
        comm.close()
        comm = None
    if not args.no_e2e:
        # every rank runs the host-buffer path on its own GPU / PCIe link (rank r hashes its own files);
        # whole-job e2e = bytes of all ranks / slowest rank's time
        if args.e2e_files <= 0:
            args.e2e_files = 1024 if world == 1 else 512
        e2e = run_e2e(args, eng, cfg, pg, torch, first_file=rank * args.e2e_files)
        if world > 1:
            sec = torch.tensor([e2e.get("seconds") or 1e30], dtype=torch.float64, device=dev_t)
            dist.all_reduce(sec, op=dist.ReduceOp.MAX)
            if e2e.get("value") is not None and float(sec.item()) < 1e29:
                e2e["value"] = world * e2e["h2d_bytes_per_step"] * e2e["steps"] / float(sec.item()) / GIB
                e2e["h2d_bytes_per_step"] *= world
                e2e["d2h_bytes_per_step"] *= world
                e2e["seconds"] = float(sec.item())
                e2e["workload"] += f"; x{world} ranks, max over ranks"
            else:
                e2e = {"value": None, "unit": "GiB/s", "error": "a rank could not run the host-buffer path"}
        out["e2e"] = e2e
    if rank == 0:
        if not args.no_cpu:
            cores = os.cpu_count() or 1
            n_s = max(cores, min(2 * cores, (8 << 30) // file_len))
            v, dt, th = cpu_pass(n_s, file_len, cores, repeats=2)
            out["cpu_baseline"] = {
                "value": v, "unit": "GiB/s", "cores": th, "kind": "port",
                "sample": f"{n_s} x {args.file_mib} MiB files of the same corpus, one stream per task, {th} threads "
                          f"(best of {cpu_thread_candidates(cores)} on {cores} logical CPUs), best of 2 ({dt:.2f} s)",
                "note": "restated CPU baseline (oracle/oracle.c, SHA-NI), not the Go binary"}
            try:
                out["cpu_baseline"]["legs"] = cpu_legs_b1_b3()
            except Exception as ex:
                out["cpu_baseline"]["legs"] = {"error": repr(ex)}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()
    eng.close()


def run_cfg3(args):
    """BASELINE config[2]: a 10 TB synthetic corpus with 30 % duplicate 4 MiB blocks (runs of 8), streamed
    through HBM in 32 GiB batches (3 in flight) generated on the device; reports throughput and the hit rate.
    Not the default bench line (diagnostic / parity-at-scale run; see profiles/)."""
    import torch

    import pbs_plus_b200 as pg

    torch.cuda.set_device(0)
    eng = pg.Engine(0, profiling=False)
    file_len = args.file_mib << 20
    n_files = min(args.files, 512)                 # 32 GiB batches, NBUF of them in flight
    NBUF = 3
    total = int(args.total_tb * 1e12)
    n_batches = max(1, total // (n_files * file_len))
    corp = pg.corpus(seed=3, file_len=file_len, block_len=4 << 20, run_blocks=8, dup_permille=300)
    cfg = pg.buzhash.NewConfig(4096)
    known = eng.digest_set(4 << 20)
    bufs = [torch.empty(n_files * file_len, dtype=torch.uint8, device="cuda") for _ in range(NBUF)]
    off = np.arange(n_files, dtype=np.uint64) * file_len
    ln = np.full(n_files, file_len, dtype=np.uint64)
    jobs = [None] * NBUF
    chunks = hits = 0
    gen_s = 0.0

    def drain(slot):
        nonlocal chunks, hits
        if jobs[slot] is not None:
            rec, _ = jobs[slot].wait()
            flags = known.insert(rec["digest"])
            chunks += len(rec); hits += int((flags != 0).sum())
            jobs[slot] = None

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in range(n_batches):
        slot = b % NBUF
        drain(slot)                                # in order: the set sees batches in corpus order
        g0 = time.perf_counter()
        eng.corpus_fill(corp, b * n_files, n_files, bufs[slot], file_len)
        gen_s += time.perf_counter() - g0
        jobs[slot] = eng.submit(cfg, bufs[slot], off, ln)
    for k in range(NBUF):
        drain((n_batches + k) % NBUF)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    nbytes = n_batches * n_files * file_len
    print(json.dumps({
        "workload": f"cfg3: {nbytes / 1e12:.2f} TB corpus, 30% duplicate 4 MiB blocks in runs of 8, {n_batches} batches of "
                    f"{n_files} x {args.file_mib} MiB, 1 GPU", "bytes": nbytes, "chunks": chunks,
        "known_chunks": hits, "hit_rate": hits / max(1, chunks), "distinct_digests": len(known),
        "wall_s": wall, "generation_s": gen_s, "GiB_per_s_incl_generation": nbytes / wall / GIB,
        "GiB_per_s_excl_generation": nbytes / max(1e-9, wall - gen_s) / GIB}), flush=True)
    eng.close()


def run_e2e(args, eng, cfg, pg, torch, first_file=0):
    """Same metric through the public C-ABI call with HOST buffers: every step is one blocking
    pbsgpu_chunk_digest_batch call that copies that step's inputs from pinned host memory to the device
    (staged in 4 GiB groups, overlapped with the kernels) and returns the chunk records to the host.
    Two host threads with one context each issue the calls (the way a multi-worker Go caller would):
    while one call drains the serial SHA tail of its last group, the other call's copies use the link."""
    import threading

    file_len = args.file_mib << 20
    n = args.e2e_files
    workers = max(1, args.e2e_threads)
    engines = [eng] + [pg.Engine(eng.device) for _ in range(workers - 1)]
    host = None
    while host is None:
        try:
            host = eng.host_alloc(n * file_len)
        except Exception as e:   # not enough pinned memory on this host: halve the step
            if n <= 64:
                return {"value": None, "unit": "GiB/s", "error": str(e)}
            n //= 2
    # fill the pinned buffer with the same corpus (generated on the device, copied back once, untimed)
    tmp = torch.empty(n * file_len, dtype=torch.uint8, device="cuda")
    eng.corpus_fill(pg.corpus(seed=2, file_len=file_len), first_file, n, tmp, file_len)
    torch.from_numpy(np.asarray(host)).copy_(tmp)
    del tmp
    torch.cuda.empty_cache()
    off = np.arange(n, dtype=np.uint64) * file_len
    ln = np.full(n, file_len, dtype=np.uint64)
    h2d_peak = None
    try:
        h2d_peak = h2d_roofline(torch, host)
    except Exception:
        pass
    sets = [e.digest_set(1 << 16) for e in engines]
    for e, s in zip(engines, sets):
        e.chunk_digest_batch(cfg, host, off, ln, s)      # warm-up (also populates each context's pools)
    torch.cuda.synchronize()
    steps = max(workers, args.e2e_steps)
    nrec = [0] * workers
    errs = []

    def work(w):
        try:
            for _ in range(w, steps, workers):
                nrec[w] = len(engines[w].chunk_digest_batch(cfg, host, off, ln, sets[w]))
        except Exception as ex:   # pragma: no cover
            errs.append(repr(ex))

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(w,)) for w in range(workers)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    for s in sets:
        s.close()
    eng.host_free(host)
    for e in engines[1:]:
        e.close()
    if errs:
        return {"value": None, "unit": "GiB/s", "error": errs[0]}
    gbs = n * file_len * steps / dt / 1e9
    return {"value": n * file_len * steps / dt / GIB, "unit": "GiB/s", "h2d_bytes_per_step": int(n * file_len),
            "d2h_bytes_per_step": int(nrec[0] * 48), "steps": steps, "host_threads": workers, "seconds": dt,
            "roofline": {"bound": "pcie_h2d", "achieved": gbs, "peak": h2d_peak, "unit": "GB/s",
                         "frac": gbs / h2d_peak if h2d_peak else None,
                         "peak_source": "pinned host -> device copy of 8 GiB measured in this run on this box (best of 3, CUDA events)"},
            "workload": f"{n} x {args.file_mib} MiB files of the cfg2 corpus per step (one blocking C-ABI call) from "
                        f"pinned host memory; PCIe-bound", "timer": "host wall clock around the blocking C-ABI calls"}


def ncu_traffic():
    """dram bytes (read + write) per launch of EVERY kernel class of the step, from the committed ncu --set full
    summaries of one 64 GiB batch: K1 scan reads the input once, K3 (bulk + long-chunk kernel) reads it again."""
    import re
    files = {"K1_scan": ("r02_ncu_batch_k_scan_tuned.txt",), "K3_sha_bulk": ("r02_ncu_batch_k_sha_tuned.txt",), "K3_sha_long": ("r02_ncu_batch_k_sha_split.txt",)}
    out, tot = {}, 0.0
    for key, names in files.items():
        for name in names:
            p = ROOT / "profiles" / name
            if not p.exists():
                return None
            txt = p.read_text()
            b = 0.0
            for m in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                mm = re.search(m + r"\s+(\w+)\s+([0-9.]+)", txt)
                scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(mm.group(1)) if mm else None
                if scale is None:
                    return None
                b += float(mm.group(2)) * scale
            out[key] = b
            tot += b
    alg = 1024 * (64 << 20)
    out.update({"total": tot, "algorithmic": alg, "ratio_to_algorithmic": tot / alg,
                "source": "profiles/r02_ncu_batch_k_scan_tuned.txt + r02_ncu_batch_k_sha_tuned.txt + r02_ncu_batch_k_sha_split.txt (ncu --set full of one launch each inside `bench.py --steps 2`, one 64 GiB batch); "
                          "the input is read twice (K1, then K3): 2.0 x the algorithmic bytes; K7 (xxh3) is not part of the step"})
    return out


def run_cfg4verify(args):
    """ONE GPU, ONE digest set: the global cfg4 corpus of `--emulate-ranks` x `--files` files hashed shard after shard in
    global order.  Prints the entry bench.py's N > 1 arm compares its NCCL-merged hit count with
    (profiles/r02_cfg4_expected.json)."""
    import torch

    import pbs_plus_b200 as pg

    torch.cuda.set_device(0)
    eng = pg.Engine(0)
    file_len = args.file_mib << 20
    corp = pg.corpus(seed=3, file_len=file_len, block_len=4 << 20, run_blocks=8, dup_permille=300)
    cfg = pg.buzhash.NewConfig(4096)
    entries = []
    sub = 256                                   # files per batch
    buf = torch.empty(sub * file_len, dtype=torch.uint8, device="cuda")
    off = np.arange(sub, dtype=np.uint64) * file_len
    ln = np.full(sub, file_len, dtype=np.uint64)
    for world in [int(x) for x in args.emulate_ranks.split(",")]:
        known = eng.digest_set(1 << 20)
        chunks = hits = 0
        for b in range(world * args.files // sub):
            eng.corpus_fill(corp, b * sub, sub, buf, file_len)
            rec = eng.chunk_digest_batch(cfg, buf, off, ln, known)
            chunks += len(rec); hits += int((rec["flags"] & 1).sum())
        entries.append({"world": world, "files_per_rank": args.files, "file_mib": args.file_mib, "chunks": chunks, "known": hits,
                        "hit_rate": hits / max(1, chunks), "distinct": len(known)})
        known.close()
    print(json.dumps({"what": "cfg4 corpus (seed 3, 30 % dup 4 MiB blocks, runs of 8) through ONE set on one GPU, in global file order",
                      "entries": entries}), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--files", type=int, default=1024)
    ap.add_argument("--file-mib", type=int, default=64)
    ap.add_argument("--e2e-files", type=int, default=0, help="files per e2e step (0 = 1024 at N=1: the whole cfg2 batch per call; 512 per rank at N>1)")
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--e2e-threads", type=int, default=2)
    ap.add_argument("--avg-kib", type=int, default=4096, help="diagnostic only; the metric is quoted at 4096")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4verify"])
    ap.add_argument("--emulate-ranks", default="2,4,8", help="cfg4verify: world sizes to produce expected hit counts for")
    ap.add_argument("--timeline", action="store_true", help="add per-step kernel intervals (ms since context open) to the line")
    ap.add_argument("--no-verify", action="store_true", help="skip the untimed post-run comparison with the oracle")
    ap.add_argument("--no-distinct", action="store_true", help="skip the non-repeating-data figure (value_distinct)")
    ap.add_argument("--distinct-gib", type=int, default=768)
    ap.add_argument("--distinct-bufs", type=int, default=7, help="16 GiB input buffers of the value_distinct run")
    ap.add_argument("--distinct-batch-files", type=int, default=256, help="files (of --file-mib) per batch of the value_distinct run")
    ap.add_argument("--distinct-early", type=int, default=1, help="0: value_distinct without PBSGPU_BATCH_EARLY_INPUT")
    ap.add_argument("--total-tb", type=float, default=10.0, help="cfg3 only")
    ap.add_argument("--no-prewarm", action="store_true")
    ap.add_argument("--inflight", type=int, default=0,
                    help="max batches submitted but not yet waited for (0 = all K at once; the library's 13 "
                         "stream slots then queue them FIFO per stream, which keeps the GPU fed without the host)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the chunk records of the last timed step (rank 0's at N>1) as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload != "cfg2":
        ap.error("--dump-outputs needs the cfg2 workload (the timed steps)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload == "cfg3":
        if rank == 0:
            run_cfg3(args)
    elif args.workload == "cfg4verify":
        if rank == 0:
            run_cfg4verify(args)
    elif args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
