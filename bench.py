#!/usr/bin/env python3
"""bench.py -- haystack GB/s of the batched Aho-Corasick search on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2] [--impl ours|reference] [--mode strong|weak]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic haystacks.

  N = 1   BASELINE.json configs[1] (C2: 10k random 4-16 B alnum keys, 1M x 256 B haystacks, one key planted per
          haystack) -- the configuration the metric and the 30 % roofline target are quoted on.
  N > 1   BASELINE.json configs[4] (C5: 100k keys, 8M x 256 B haystacks): STRONG scaling, the 2 GiB batch is sharded
          over the N ranks through pyahocorasick_b200.distributed.scan_sharded's shard bounds, the flattened automaton
          is replicated, and the per-rank match counts are all-gathered over NCCL inside the timed region, off the
          compute stream.  Every rank checks its own count against what it planted.  (--mode weak: one C2-sized
          shard per rank, the round-1 behaviour.)

  value     haystack bytes / s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e       same metric through Automaton.find_all_batch() with a pinned HOST batch: H2D, kernel, D2H of count +
            records and the reference-order sort all inside the timed region; `variants` adds pageable host memory
            and a list of bytes objects
  roofline  the stream kernel alone: (haystack bytes + 12 B/match) / mean event-timed launch, against the measured
            HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the reference's own C extension (oracle/_ref) looping iter() over the whole batch, single thread (the
            reference holds the GIL), rank 0 at N=1; its match list is compared with the GPU's (parity_checked)
  latency   microseconds per Automaton.iter() call on ONE haystack of 256 B / 64 KiB / 16 MiB, ours vs the reference

--dump-outputs DIR writes what the last timed step returned (see dump_outputs) as DIR/<name>.npy, so that two builds can
be compared output for output: the workload is generated from fixed seeds, identical from run to run.

--impl reference times the reference extension on the host cores (one process per core, the pool created once, each
worker looping iter() over its slice of a bounded sample) and prints the same JSON shape.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD_DESC = {
    "C2": "C2: 10k random [4-16]B alnum keys, 1M x 256B haystacks, 1 planted key per haystack, seed 1001",
    "C3": "C3: 100k DNA 20-mers, 10M x 150B reads, 10% planted, seed 1003",
    "C4": "C4: 10k keys (C2 set), 64 x 16MiB haystacks, planted ~1 per 256B, seed 1004",
    "C5": "C5: 100k random [4-16]B alnum keys, 8M x 256B haystacks sharded over the GPUs, 1 planted key per haystack, seed 1005",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default=None, help="C2 (default at 1 GPU), C3, C4, C5 (default at N > 1)")
    ap.add_argument("--mode", default="strong", choices=["strong", "weak"], help="N > 1: shard one batch (strong) or one batch per rank (weak)")
    ap.add_argument("--scale", type=float, default=None, help="shrink the batch (debug only; invalidates the number)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="auto", choices=["auto", "filter", "dfa"])
    ap.add_argument("--cpu-sample", type=int, default=1_000_000, help="haystacks in the cpu_baseline sample (~10 s of CPU for C2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--variant", default="planted", choices=["planted", "sparse"], help="sparse = pure random haystacks (diagnostic)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's match records to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def default_scale(cfg, world):
    return {"C2": 1.0, "C3": 1.0, "C4": 1.0, "C5": 1.0 if world > 1 else 0.125}[cfg]


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- reference arm / cpu baseline
_W = {}          # per-worker state of the reference pool: the built automaton and this worker's haystacks


def _ref_build(keys):
    import oracle
    ref = oracle.ref_module("bytes")
    R = ref.Automaton(ref.STORE_INTS)
    for i, k in enumerate(keys):
        R.add_word(k, i)
    R.make_automaton()
    return R


def _pool_init(keys, rows, bounds, counter):
    """runs once in every worker: build the automaton, pick this worker's slice, turn it into bytes objects"""
    with counter.get_lock():
        me = counter.value
        counter.value += 1
    lo, hi = bounds[me]
    _W["R"] = _ref_build(keys)
    _W["hs"] = [r.tobytes() for r in rows[lo:hi]]
    _W["bytes"] = sum(len(h) for h in _W["hs"])


def _pool_step(min_seconds):
    """one measurement of one worker: loop iter() over its haystacks until min_seconds have passed (whole passes only)"""
    R, hs = _W["R"], _W["hs"]
    n = passes = 0
    t0 = time.perf_counter()
    while True:
        for h in hs:
            for _ in R.iter(h):
                n += 1
        passes += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            return dt, passes * _W["bytes"], n


def reference_single_thread(keys, rows, collect=False):
    """The reference's iter() looped over `rows` in THIS process.  Returns (seconds, matches, kind, records or None)."""
    import oracle
    if not oracle.ref_available("bytes"):
        # the reference did not travel: fall back to the C restatement (kind 'port')
        O = oracle.OracleAutomaton()
        for i, k in enumerate(keys):
            O.add_word(k, i)
        O.make_automaton()
        off = np.arange(rows.shape[0] + 1, dtype=np.int64) * rows.shape[1]
        t0 = time.perf_counter()
        rec = O.scan_batch_bytes(rows.reshape(-1), off)
        dt = time.perf_counter() - t0
        return dt, len(rec), "port", (np.asarray(rec, dtype=np.int64) if collect else None)
    R = _ref_build(keys)
    hs = [r.tobytes() for r in rows]
    out = [] if collect else None
    n = 0
    t0 = time.perf_counter()
    if collect:
        for i, h in enumerate(hs):
            for e, v in R.iter(h):
                out.append((i, e, v))
        n = len(out)
    else:
        for h in hs:
            for _ in R.iter(h):
                n += 1
    dt = time.perf_counter() - t0
    return dt, n, "reference", (np.asarray(out, dtype=np.int64).reshape(-1, 3) if collect else None)


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  One process per core
    (the reference holds the GIL: processes are the only way to use the cores); the pool is created ONCE, every
    worker builds the automaton once and then, per step, loops Automaton.iter() over its slice of a bounded sample
    for at least 0.25 s.  A step's rate is the sum of the workers' own rates (bytes they scanned / their own time):
    no worker waits for another, so a slow core costs its share and not the whole step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import oracle
    from pyahocorasick_b200 import synth
    cfg = args.config or "C2"
    if oracle.ref_available("bytes"):
        oracle.ref_module("bytes")                            # in the parent too: the driver records which .so files were loaded
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    per_core = {"C3": 2048}.get(cfg, 4096)                   # haystacks per core: ~1 MB
    full = {"C2": 1_000_000, "C3": 10_000_000, "C5": 8_000_000}.get(cfg, 1_000_000)
    step_rows = min(per_core * cores, full)
    if cfg == "C4":
        w = synth.make(cfg, scale=step_rows * 4096 / (64 * 16 * 1024 * 1024))
        rows_all = w.haystacks.reshape(-1, 4096)[:step_rows]
    else:
        w = synth.make(cfg, scale=step_rows / {"C2": 1e6, "C3": 1e7, "C5": 8e6}[cfg])
        rows_all = w.haystacks[:step_rows]
    step_rows = rows_all.shape[0]
    kind = "reference" if oracle.ref_available("bytes") else "port"
    min_s = 0.25
    # one thread alone, before the pool exists: what a core can do when nothing else runs
    alone = None
    if kind == "reference":
        R1 = _ref_build(w.keys)
        hs1 = [r.tobytes() for r in rows_all[:4096]]
        t0 = time.perf_counter()
        done = 0
        while time.perf_counter() - t0 < 1.0:
            for h in hs1:
                for _ in R1.iter(h):
                    pass
            done += 1
        alone = done * sum(len(h) for h in hs1) / (time.perf_counter() - t0)
        del R1, hs1
    rates, matches, single = [], 0, None
    t_region = time.perf_counter()
    if kind == "reference" and cores > 1:
        bounds = [(int(a[0]), int(a[-1]) + 1) if len(a) else (0, 0) for a in np.array_split(np.arange(step_rows), cores)]
        counter = mp.get_context("fork").Value("i", 0)
        with mp.get_context("fork").Pool(cores, initializer=_pool_init, initargs=(w.keys, rows_all, bounds, counter)) as pool:
            for s in range(args.warmup + args.steps):
                res = pool.map(_pool_step, [min_s] * cores, chunksize=1)
                if s >= args.warmup:
                    rates.append(sum(b / dt for dt, b, _ in res))
                    matches += sum(n for _, _, n in res)
                    best1 = max(b / dt for dt, b, _ in res)
                    single = best1 if single is None else max(single, best1)
        used = cores
    else:
        for s in range(args.warmup + args.steps):
            dt, n, kind, _ = reference_single_thread(w.keys, rows_all)
            if s >= args.warmup:
                rates.append(rows_all.size / dt)
                matches += n
        used, single = 1, max(rates) if rates else None
    t_region = time.perf_counter() - t_region
    val = float(np.mean(rates)) / 1e9
    line = {
        "impl": "reference", "metric": "haystack GB/s", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * min_s, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC[cfg], "sample": f"{step_rows} haystacks x {rows_all.shape[1]} B (bounded sample of the same generator), every worker loops its slice for >= {min_s} s per step"},
        "best_step_gbs": float(np.max(rates)) / 1e9, "worst_step_gbs": float(np.min(rates)) / 1e9, "timed_region_s": t_region,
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": used, "kind": kind,
                         "sample": f"{step_rows} x {rows_all.shape[1]} B, one process per core looping Automaton.iter(), sum of the workers' rates",
                         "best_worker_under_load_gbs": (single / 1e9) if single else None,
                         "single_thread_alone_gbs": (alone / 1e9) if alone else None,
                         "effective_cores": (val * 1e9 / alone) if alone else None},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- our arm
DUMP_LIMIT_BYTES = 64_000_000          # all files of one dump together, .npy headers included


def dump_outputs(out_dir, d_out, n_matches, suffix=""):
    """The records acb_scan_device() wrote (haystack, end_index, key_id), as float64 (exact for int32), in (haystack,
    end_index, key_id) order: the kernels append them in whatever order their atomics give.  When the three columns
    would pass DUMP_LIMIT_BYTES, a fixed seeded sample of the sorted rows is written instead (sample_rows.npy says
    which); match_count.npy always holds the full count."""
    rec = d_out[:n_matches].cpu().numpy().astype(np.int64)
    rec = rec[np.lexsort((rec[:, 2], rec[:, 1], rec[:, 0]))]
    os.makedirs(out_dir, exist_ok=True)
    cols = {"hay_id": rec[:, 0], "end_index": rec[:, 1], "key_id": rec[:, 2]}
    max_rows = (DUMP_LIMIT_BYTES - 4096) // (8 * (len(cols) + 1))
    if n_matches > max_rows:
        rows = np.sort(np.random.Generator(np.random.PCG64(0)).choice(n_matches, size=max_rows, replace=False))
        cols = {k: v[rows] for k, v in cols.items()}
        cols["sample_rows"] = rows
    cols["match_count"] = np.array([n_matches])
    for name, a in cols.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a.astype(np.float64))


def latency_block(A, keys, sizes=(256, 65536, 16 * 1024 * 1024)):
    """microseconds per Automaton.iter() call (all matches drained) on ONE haystack, ours vs the reference extension"""
    import oracle
    from pyahocorasick_b200 import synth
    rng = np.random.Generator(np.random.PCG64(77))
    R = _ref_build(keys) if oracle.ref_available("bytes") else None
    out = {}
    for sz in sizes:
        hay = synth.ALNUM[rng.integers(0, len(synth.ALNUM), size=sz)].tobytes()
        reps = 200 if sz <= 65536 else 5
        for _ in range(3):
            list(A.iter(hay))
        t0 = time.perf_counter()
        for _ in range(reps):
            n = sum(1 for _ in A.iter(hay))
        ours = (time.perf_counter() - t0) / reps * 1e6
        ref = None
        if R is not None:
            rr = max(1, reps // 5)
            t0 = time.perf_counter()
            for _ in range(rr):
                m = sum(1 for _ in R.iter(hay))
            ref = (time.perf_counter() - t0) / rr * 1e6
            assert m == n, (m, n)
        out[str(sz)] = {"ours_us": ours, "reference_us": ref, "matches": n}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    from pyahocorasick_b200 import _native as N
    from pyahocorasick_b200 import distributed as D
    from pyahocorasick_b200 import synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = args.config or ("C5" if world > 1 and args.mode == "strong" else "C2")
    strong = world > 1 and args.mode == "strong"
    scale = args.scale if args.scale is not None else default_scale(cfg, world)

    # ---- workload: same keys everywhere; strong: rank r builds rows [lo, hi) of the one global batch (the generator
    # is seeded per 64k-row block, so a shard never materialises the other ranks' rows); weak: its own batch -------------
    if strong:
        n_global = int(round({"C2": 1e6, "C3": 1e7, "C5": 8e6}[cfg] * scale))
        lo, hi = D.shard_bounds(n_global, world, rank)
        w = synth.make_rows(cfg, lo, hi, planted=(args.variant == "planted"))
    else:
        w = synth.make(cfg, scale=scale, planted=(args.variant == "planted"))
        if world > 1 and rank > 0:                     # different haystack bytes per rank, same shape
            rng = np.random.Generator(np.random.PCG64(9000 + rank))
            hay = synth.random_haystacks(rng, synth.DNA if cfg == "C3" else synth.ALNUM, *w.haystacks.shape)
            synth.plant(rng, hay, w.keys, np.arange(hay.shape[0]) if cfg != "C3" else np.nonzero(rng.random(hay.shape[0]) < 0.1)[0])
            w.haystacks = hay
            w.planted_hay = None
    A = synth.build_automaton(w.keys)
    L = N.lib()
    tb = A._ensure_table(local)
    n_hay, stride = w.haystacks.shape
    total = int(w.haystacks.size)

    pinned = torch.empty(w.haystacks.shape, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[...] = w.haystacks
    d_hay = pinned.cuda(non_blocking=True)
    d_cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
    cap = max(4 * n_hay, 1 << 20)
    d_out = torch.empty((cap, 3), dtype=torch.int32, device="cuda")
    gathered = torch.zeros(world, dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    algo = N.ALGOS[args.algo]
    # the count all-gather runs on its own stream, ordered after the scan by an event: the next scan does not wait for it
    side = torch.cuda.Stream() if world > 1 else None
    d_cnt_side = torch.zeros(1, dtype=torch.int64, device="cuda") if world > 1 else None

    def step():
        d_cnt.zero_()
        N.check(L.acb_scan_device(tb, d_hay.data_ptr(), total, None, n_hay, stride, d_out.data_ptr(), cap, d_cnt.data_ptr(), stream, algo))
        if world > 1:
            d_cnt_side.copy_(d_cnt)                    # snapshot on the compute stream; the side stream gathers the snapshot
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(side):
                side.wait_event(ev)
                dist.all_gather_into_tensor(gathered, d_cnt_side)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # strong scaling: the same global batch on ONE GPU (rank 0, untimed extra, the other ranks wait), so that the line
    # carries its own single-GPU reference point for this configuration (the N=1 bench line is C2, a different workload)
    single = None
    if strong:
        if rank == 0:
            wf = synth.make_rows(cfg, 0, n_global, planted=(args.variant == "planted"))
            d_full = torch.from_numpy(wf.haystacks).cuda()
            nf, tot_f = wf.haystacks.shape[0], int(wf.haystacks.size)
            capf = max(4 * nf, 1 << 20)
            d_out_f = torch.empty((capf, 3), dtype=torch.int32, device="cuda")
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for i in range(3 + 5):
                if i == 3:
                    e0.record()
                d_cnt.zero_()
                N.check(L.acb_scan_device(tb, d_full.data_ptr(), tot_f, None, nf, stride, d_out_f.data_ptr(), capf, d_cnt.data_ptr(), stream, algo))
            e1.record()
            torch.cuda.synchronize()
            single = {"gbs": tot_f / (e0.elapsed_time(e1) / 5 * 1e-3) / 1e9, "ms_per_step": e0.elapsed_time(e1) / 5,
                      "matches": int(d_cnt.item()), "what": "the whole global batch on one GPU (rank 0, before the timed region)"}
            del d_full, d_out_f, wf
            torch.cuda.empty_cache()
        barrier()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    n_matches = int(d_cnt.item())
    # per-rank result check: every planted occurrence of this rank's rows must be there (a lower bound on the count),
    # and at N > 1 rank 0 checks the gathered counts against the sum
    planted_lb = int(len(w.planted_hay)) if getattr(w, "planted_hay", None) is not None else 0
    assert n_matches >= planted_lb, f"rank {rank}: {n_matches} matches < {planted_lb} planted occurrences"
    if world > 1:
        cnts = gathered.cpu().numpy()
        assert int(cnts[rank]) == n_matches, (rank, cnts.tolist(), n_matches)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    launches0 = L.acb_launch_count()
    # ---- timed region: K steps, CUDA events on the launching stream -------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    ev0.record()
    for i in range(args.steps):
        d_cnt.zero_()
        kev[i][0].record()
        N.check(L.acb_scan_device(tb, d_hay.data_ptr(), total, None, n_hay, stride, d_out.data_ptr(), cap, d_cnt.data_ptr(), stream, algo))
        kev[i][1].record()
        if world > 1:
            d_cnt_side.copy_(d_cnt)
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(side):
                side.wait_event(ev)
                dist.all_gather_into_tensor(gathered, d_cnt_side)
    if world > 1:
        torch.cuda.current_stream().wait_stream(side)   # the last gather belongs to the timed region
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    if args.dump_outputs:
        last = int(d_cnt.item())
        if last > cap:
            raise SystemExit(f"rank {rank}: {last} matches do not fit the {cap}-record buffer, nothing to dump")
        dump_outputs(args.dump_outputs, d_out, last, f"_rank{rank}" if world > 1 else "")
    launches = L.acb_launch_count() - launches0
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    tot_bytes = torch.tensor([total], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_bytes, op=dist.ReduceOp.SUM)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = int(tot_bytes.item()) / (ms_step * 1e-3) / 1e9
    total_matches = int(gathered.sum().item()) if world > 1 else n_matches

    # ---- e2e: the public API with host batches --------------------------------------------------
    e2e = None
    if not args.no_e2e:
        def time_api(batch, reps):
            for _ in range(2):
                m = A.find_all_batch(batch, algo=args.algo)
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                m = A.find_all_batch(batch, algo=args.algo)
                if world > 1:
                    c = torch.tensor([len(m)], dtype=torch.int64, device="cuda")
                    dist.all_gather_into_tensor(gathered, c)
            barrier()
            dt = (time.perf_counter() - t0) / reps
            tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()), m
        e2e_steps = max(3, min(args.steps, 10))
        dt, m = time_api(pinned.numpy(), e2e_steps)
        assert len(m) == n_matches, (len(m), n_matches)
        e2e = {"value": int(tot_bytes.item()) / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(tot_bytes.item()),
               "d2h_bytes_per_step": world * (8 + 12 * len(m)), "ms_per_step": dt * 1e3, "steps": e2e_steps,
               "includes": "H2D of the batch from pinned host memory, kernel, D2H of count+records, reference-order sort"}
        if world == 1:
            dt_pg, m2 = time_api(np.array(w.haystacks, copy=True), 3)            # ordinary (pageable) numpy memory
            n_list = min(n_hay, 200_000)
            as_list = [r.tobytes() for r in w.haystacks[:n_list]]                # what a drop-in user most naturally has
            dt_ls, m3 = time_api(as_list, 3)
            e2e["variants"] = {"pageable_ndarray_gbs": total / dt_pg / 1e9,
                               "list_of_bytes_gbs": n_list * stride / dt_ls / 1e9, "list_of_bytes_n": n_list}
            assert len(m2) == n_matches

    # clocks under load: the timed region is only a few ms long, so keep the same step running for another
    # ~0.5 s (untimed) while nvidia-smi samples SM clock and throttle reasons every 50 ms
    t_end = time.perf_counter() + 0.5
    while time.perf_counter() < t_end:
        for _ in range(50):
            step()
        torch.cuda.synchronize()
    clk = clocks.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel ------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    algo_bytes = total + 12 * n_matches
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(cfg)
        except Exception:
            traffic = None
    kernel_name = "acb_dfa_kernel"
    if args.algo != "dfa":      # the PAIR placement (gram 4, stride 1: C2 / C4 key sets) has its own kernel
        kernel_name = "acb_pair_kernel" if (A.filter_shape()["filter_flags"] & 2) else "acb_stream_kernel"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "kernel": kernel_name,
                "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": algo_bytes}

    # ---- CPU baseline + full parity check of its match list (rank 0, N=1 only) ------------------
    cpu, parity_checked = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ns = min(args.cpu_sample, n_hay)
        rows = w.haystacks[:ns]
        dt, nm, kind, ref_rec = reference_single_thread(w.keys, rows, collect=True)
        cpu = {"value": rows.size / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": kind,
               "sample": f"first {ns} haystacks of the batch ({rows.size / 1e6:.1f} MB), Automaton.iter() loop, {dt:.1f} s",
               "matches_per_s": nm / dt, "host_cores_available": os.cpu_count()}
        # the reference's (haystack, end_index, value) list IS the parity oracle (BASELINE.md section 2): compare it,
        # record for record and in the reference's order, with what the GPU path returns for the same haystacks
        m = A.find_all_batch(w.haystacks[:ns], algo=args.algo)
        got = np.stack([m.hay_id.astype(np.int64), m.end_index.astype(np.int64), np.asarray(m.values(), dtype=np.int64)], axis=1)
        if got.shape != ref_rec.shape or not np.array_equal(got, ref_rec):
            raise SystemExit(f"PARITY FAILURE: GPU records differ from the {kind} on the first {ns} haystacks "
                             f"({got.shape[0]} vs {ref_rec.shape[0]} records)")
        parity_checked = int(ref_rec.shape[0])

    latency = None
    if rank == 0 and world == 1 and not args.no_latency:
        latency = latency_block(A, w.keys)

    if rank == 0:
        line = {
            "metric": "haystack GB/s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD_DESC[cfg] + ("" if args.variant == "planted" else " [SPARSE variant: no planted keys]") + ("" if scale == default_scale(cfg, world) else f" [SCALED x{scale}: not a valid bench number]"),
                       "n_haystacks_per_gpu": n_hay, "haystack_bytes": stride, "n_keys": len(w.keys),
                       "l2": f"batch {total / 1e6:.0f} MB per GPU > 126 MB L2, no flush needed" if total > 126e6 else "batch smaller than L2",
                       "algo": args.algo,
                       "parallelism": (f"one batch sharded x{world} (strong scaling)" if strong else f"one batch per rank x{world} (weak scaling)") + ", NCCL all-gather of match counts on a side stream" if world > 1 else "single GPU"},
            "matches_per_s": total_matches / (ms_step * 1e-3), "matches_per_step": total_matches,
            "results_verified": {"per_rank_planted_lower_bound": True, "gathered_counts_consistent": world > 1,
                                 "sum_equals_single_gpu_count": (single["matches"] == total_matches) if single else None},
            "strong_scaling": ({"single_gpu": single, "efficiency_vs_single_gpu": value / (world * single["gbs"])} if single else None),
            "parity_checked": parity_checked, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "latency": latency,
            "gpu_launches": int(launches), "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
