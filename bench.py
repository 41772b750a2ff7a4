"""bench.py -- BASELINE.json metric: SSE chunks/sec & JSON GB/s at 4096 streams x 512 deltas (64 B).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

One "step" = one pass of the hot path over one batch (SURVEY 8(d) C3: 4096 streams x 512 delta
events of 64 B + a usage event + [DONE] per stream, one event per network chunk).  Under torchrun
every rank runs its own 4096-stream batch on its own GPU (streams shard with no cross-GPU
dependency: weak scaling, no collective on the data path).

value   : chunks/s with inputs resident in HBM (kernels only, CUDA events on the launching stream)
e2e     : the same through the host-buffer C-ABI call (pinned host -> device -> host inside the
          timed region) plus the read-back of the usage records
roofline: algorithmic bytes (128 B per 64-B event) / summed kernel time, vs MEASURED_PEAKS.json
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

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_STREAMS, N_EVENTS, EVENT_BYTES = 4096, 512, 64
ALGO_BYTES_PER_EVENT = 128          # 64 read + 64 re-emitted (SURVEY 8(d))
METRIC, UNIT = "sse_chunks_per_sec", "chunks/s"


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed ncu capture."""
    p = ROOT / "profiles" / "traffic.json"
    try:
        return json.loads(p.read_text())["traffic_bytes_per_launch"]
    except Exception:
        return None


# ---- CPU reference arm: the reference's OWN code (oracle/_ref via oracle/ref_arm.py), else the oracle port ------------------
def _port_worker(args):
    seed, n_streams, n_events = args
    from llmapigateway_b200.synth import sse_batch
    from oracle.sse_oracle import run_stream
    b = sse_batch(n_streams=n_streams, n_events=n_events, seed=seed)
    streams = [b.stream_chunks(s) for s in range(n_streams)]
    t0 = time.perf_counter()
    for chunks in streams:
        relay, tap = run_stream(chunks)
        assert not relay.failed and len(tap.rows) == 1
    return time.perf_counter() - t0


def cpu_arm(variant: str, procs: int, n_streams: int, n_events: int, seed: int = 3):
    """`n_streams` C3 streams split over `procs` processes -> (events/s, kind).  kind "reference": the unmodified reference modules
    from oracle/_ref (make_llm_request + ChunkProcessorThread through httpx.MockTransport, BASELINE.md B1/B2); kind "port": the
    oracle restatement (only when oracle/_ref did not travel to this box)."""
    from oracle import ref_arm
    if ref_arm.ref_root() is not None:
        ev, _, _ = ref_arm.run_config3(variant, procs, n_streams, n_events, seed)
        return ev, "reference"
    import multiprocessing as mp
    per = max(1, n_streams // procs)
    with mp.get_context("fork").Pool(procs) as pool:
        times = pool.map(_port_worker, [(seed + i, per, n_events) for i in range(procs)])
    return procs * per * n_events / max(times), "port"


def cpu_baseline_block(n_events: int, budget_s: float = 25.0):
    """BASELINE.md section 3: B1 (faithful: pure-Python parser standing in for json5) and B2 (generous: C json) on one core (how the
    reference runs) and on all the cores this process may use.  Samples are sized from a short probe to fit `budget_s`."""
    from oracle import ref_arm
    cores = ref_arm.effective_cores()
    probe, kind = cpu_arm("B2", 1, 8, n_events)
    per_core = max(8, min(256, int(probe * budget_s / 4 / n_events / 4)))       # streams per core for ~budget/4 s per variant
    out = {"cores": cores, "kind": kind, "unit": UNIT}
    for name, variant, procs in (("B2_N", "B2", cores), ("B2_1", "B2", 1), ("B1_N", "B1", cores), ("B1_1", "B1", 1)):
        n = per_core * procs if variant == "B2" else max(procs, per_core * procs // 2)
        ev, _ = cpu_arm(variant, procs, n, n_events)
        out[name] = {"value": ev, "streams": n, "procs": procs}
    out["value"] = out["B2_N"]["value"]
    out["sample"] = (f"C3 streams of {n_events} x {EVENT_BYTES} B events (+ usage event, [DONE]) through the reference's own make_llm_request + ChunkProcessorThread "
                     f"(httpx.MockTransport, no sockets): {out['B2_N']['streams']} streams over {cores} processes for the headline value (B2 = json5.loads -> C json.loads, generous); "
                     f"B1 = pure-Python parser standing in for json5; *_1 = one process (how the reference is deployed)") if kind == "reference" else \
                    f"oracle port (oracle/_ref absent), {cores} processes"
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi polled every 20 ms by ONE child process for the whole measured part of the run."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.idx, self.samples, self.loaded, self.reasons = gpu_index, [], [], set()
        self.max_mhz, self.proc = None, None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx), "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                try:
                    mhz = float(f[0]); self.max_mhz = float(f[1])
                except Exception:
                    continue
                self.samples.append(mhz)
                if len(f) > 6 and f[6].isdigit() and int(f[6]) > 0:
                    self.loaded.append(mhz)
                for n, v in zip(self.NAMES, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)

    def summary(self):
        s = sorted(self.loaded or self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "samples_under_load": len(self.loaded)}


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores, same config/metric/unit.
    A step = the whole C3 configuration (4096 x 512 events) when a probe says K + W steps fit in a few minutes, else a bounded
    sample of it (stated in `config`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_arm
    cores = ref_arm.effective_cores()
    probe, kind = cpu_arm("B2", cores, 8 * cores, N_EVENTS)
    steps_total = args.warmup + args.steps
    full_s = N_STREAMS * N_EVENTS / probe
    n_streams = N_STREAMS if full_s * steps_total <= 240 else max(cores, int(N_STREAMS * 240 / (full_s * steps_total)) // cores * cores)
    vals = []
    for i in range(steps_total):
        t0 = time.perf_counter()
        v, _ = cpu_arm("B2", cores, n_streams, N_EVENTS, seed=3 + 100 * i)
        if i >= args.warmup:
            vals.append((v, time.perf_counter() - t0))
    value = float(np.mean([v for v, _ in vals]))
    ms = n_streams * N_EVENTS / value * 1e3
    sample = (f"{n_streams} of {N_STREAMS} streams x {N_EVENTS} events of {EVENT_BYTES} B per step over {cores} processes; "
              + ("the UNMODIFIED reference (oracle/_ref): make_llm_request relay + ChunkProcessorThread tap through httpx.MockTransport, json5.loads -> C json.loads (B2, generous)"
                 if kind == "reference" else "oracle port (oracle/_ref absent)"))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "C3: 4096 concurrent SSE streams x 512 data: deltas (64 B each), parse/normalise/re-emit",
                       "streams_per_step": n_streams, "events_per_stream": N_EVENTS, "same_config": n_streams == N_STREAMS},
            "json_gbs": value * EVENT_BYTES / 1e9,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


def run_reference_side(args):
    """`--impl reference --config c4|c5`: the reference's own code for that configuration on this box's host cores (oracle/_ref),
    on a bounded sample sized for a few minutes."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import ref_arm
    cores = ref_arm.effective_cores()
    if args.config == "c4":
        n_total = 8192
        ids = list(range(0, n_total, max(1, n_total // (16 * cores))))[:16 * cores]
        vals = []
        for i in range(args.warmup + args.steps):
            v, slowest, served = ref_arm.run_config4("B2", cores, ids, n_total, N_EVENTS)
            if i >= args.warmup:
                vals.append(v)
        value = float(np.mean(vals))
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": len(ids) * N_EVENTS / value * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": "C4: 3-deep fallback rule chain, 20% injected upstream failure, 8192 concurrent streams", "streams_per_step": len(ids), "same_config": False},
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
                                 "sample": f"{len(ids)} of 8192 streams per step over {cores} processes: the UNMODIFIED chat.py:20 chat_completions (oracle/_ref) + make_llm_request + ChunkProcessorThread tap, MockTransport upstream, json5.loads -> C json.loads"},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    else:
        n = min(args.records, 1_000_000)
        r = ref_arm.run_config5(n)
        q = [r[k] for k in ("hour_window_s", "hour_all_s", "day_window_s", "day_all_s")]
        value = n * len(q) / sum(q)
        line = {"impl": "reference", "metric": "usage_rollup_records_per_sec", "value": value, "unit": "records/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0,
                "ms_per_step": sum(q) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": {"workload": "C5: usage-stats rollup", "records": n, "same_config": n == args.records, "queries": r},
                "cpu_baseline": {"value": value, "unit": "records/s", "cores": 1, "kind": "reference",
                                 "sample": f"{n} rows in a SQLite file, the UNMODIFIED TokensUsageDB.get_aggregated_usage (tokens_usage_db.py:222) for hour/day, endpoint window and whole table; load time {r['load_s']:.1f} s not counted"},
                "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


_RESULT_FD = None


def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    return world, rank, local, dev, barrier, max_over_ranks, sum_over_ranks


def run_c4(args):
    """BASELINE configs[3]: 8 192 concurrent streaming requests, a 3-rule fallback chain each, every upstream attempt failing
    independently with p = 0.2 (SURVEY 8(d) C4).  Streams go to GPUs by shard_of(stream_id, N) (strong scaling: the total is
    fixed); no collective on the data path.  One step = the whole walk of this rank's requests through ChainBatch: request scan,
    per-round body rewrite with the attempt's plan, one SSE step per round over what the upstreams streamed, error details of
    the failed first events, usage rows of the served streams -- HOST buffers in, host buffers out (this config has no
    device-resident form: the walk is host-driven by design, SURVEY 8(e))."""
    import torch.distributed as dist
    import llmapigateway_b200 as L
    from llmapigateway_b200 import chat, rewrite, synth
    from llmapigateway_b200.gateway import shard_of
    world, rank, local, dev, barrier, max_over_ranks, sum_over_ranks = _dist_setup()
    S, E = (8192 if args.streams == N_STREAMS else args.streams), args.events
    W, K = max(args.warmup, 3), args.steps
    providers, rules, fallback_provider = synth.chain_world()
    os.environ.setdefault("ALPHA_KEY_ENV", "sk-alpha-from-env")
    up = synth.ChainUpstream(S, E, seed=4, p_fail=0.2)
    mine = np.array([i for i in range(S) if shard_of(i, world) == rank])
    all_bodies = synth.chain_request_bodies(S, seed=4)
    bodies = [all_bodies[i] for i in mine]
    n = len(mine)
    eng = L.Engine(device=local, max_streams=max(n, 1), max_step_chunks=n * (E + 2) + 64, max_step_bytes=n * (E * EVENT_BYTES + 512) + 4096)
    import httpx
    mode = "httpx028" if tuple(int(x) for x in httpx.__version__.split(".")[:2]) >= (0, 28) else "httpx027"
    plans = rewrite.RulePlans(rules, fallback_provider=fallback_provider, stream_mode=mode)
    eng.load_rules(plans)
    up.prepare(mine, 3, alloc=eng.alloc_pinned)
    walker = chat.ChainBatch(eng, plans, providers, rules)
    sampler = ClockSampler(local)
    if rank == 0:                                   # (one poller for the box: nvidia-smi takes a driver lock every sample)
        sampler.start()
    for _ in range(W):
        out = walker.run(bodies, None, up, stream_ids=mine)
    barrier()
    l0 = eng.launch_count()
    times = []
    for _ in range(K):
        barrier()
        t0 = time.perf_counter()
        out = walker.run(bodies, None, up, stream_ids=mine)
        eng.sync()
        times.append(time.perf_counter() - t0)
    barrier()
    launches = eng.launch_count() - l0
    if rank == 0:
        sampler.stop()
    # correctness of the timed configuration (not timed): served-by round == first non-failing attempt, bytes == the upstream's
    kind = up.kind[:3, mine]
    first_ok = np.where((kind == 0).any(axis=0), (kind == 0).argmax(axis=0), -1)
    assert np.array_equal(out.served_round, first_ok.astype(np.int32)), "served-by round differs from the injected failure schedule"
    b = up.batch; co = b.chunk_off.astype(np.int64)
    for k in range(0, n, max(1, n // 64)):
        if first_ok[k] >= 0:
            s = int(mine[k]); lo, hi = int(co[b.seg_chunk[s]]), int(co[b.seg_chunk[s + 1]])
            assert out.emitted(k) == b.data[lo:hi].tobytes()
    step_s = max_over_ranks(float(np.mean(times)))
    relayed = sum_over_ranks(float(out.chunks_relayed))
    delta_events = sum_over_ranks(float((first_ok >= 0).sum() * E))
    attempts = sum_over_ranks(float(out.attempts))
    failed503 = sum_over_ranks(float((first_ok < 0).sum()))
    per_gpu = delta_events / world / step_s
    in_bytes = sum(int(a.data.size) for _, a in up.prepared.values()) + sum(len(x) for x in bodies)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = _peaks()
    value = delta_events / step_s
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": step_s * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "C4: 3-deep fallback rule chain, 20% injected upstream failure, 8192 concurrent streams sharded across the GPUs by shard_of(stream_id, N)",
                       "streams_total": S, "streams_rank0": n, "events_per_stream": E, "p_fail": 0.2, "failure_kinds": ["http500+text", "first event error", "first event detail"],
                       "counts": "chunks = the 64-B delta events of the streams that were served (the usage event and [DONE] of each are relayed too, not counted)",
                       "l2": "inputs larger than L2 at N<=2 (270 MB per walk); host buffers every step, nothing cached on the device between steps",
                       "parallelism": f"streams sharded x{world}, no collective"},
            "chunks_relayed_incl_tail": relayed, "attempts": attempts, "walk_phases_ms_rank0": {k: round(v * 1e3, 3) for k, v in out.timings.items()}, "exhausted_503": failed503, "per_gpu_chunks_per_s": per_gpu,
            "json_gbs": value * EVENT_BYTES / 1e9, "clocks": sampler.summary(), "gpu_launches": int(launches),
            "e2e": {"value": value, "unit": UNIT, "ms_per_step": step_s * 1e3, "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": in_bytes,
                    "note": "the walk is host-driven: `value` IS the end-to-end number (pinned host buffers -> device -> pinned host buffers every round)"},
            "roofline": {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None, "peak_source": peak_src,
                         "note": "host-driven walk: PCIe and Python control bound, see the C3 line for the kernel roofline"}}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_c5(args):
    """BASELINE configs[4]: usage-stats rollup of 10 M extracted usage records -> per-hour / per-day x model aggregation, 1 vs N GPUs.
    Records are partitioned by contiguous row ranges over the ranks (strong scaling); every rank accumulates its records into a
    dense (bucket x model) table of 64-bit integer cells, ONE all-reduce(sum) over that table is the exchange step (SURVEY 8(e)),
    rank 0 compacts the rows.  A step = the `hour` and the `day` rollup, each over the window the stats endpoint asks for
    (stats.py:46-55: 24 h / 2 weeks) AND over the whole table (no window: the worst case for the table size)."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from datetime import datetime, timedelta
    import llmapigateway_b200 as L
    from llmapigateway_b200 import usage as U
    world, rank, local, dev, barrier, max_over_ranks, sum_over_ranks = _dist_setup()
    n = args.records
    W, K = max(args.warmup, 3), args.steps
    end = datetime(2026, 9, 21, 6, 57, 17, 47518)
    ts, models, tok, cost = U.synth_usage_columns(n, seed=5, end=end)
    names = sorted({m for m in models if m is not None})
    lo, hi = rank * n // world, (rank + 1) * n // world
    eng = L.Engine(device=local, max_streams=64, max_step_chunks=1024, max_step_bytes=1 << 20)
    stream = torch.cuda.Stream(device=dev)
    eng.set_stream(stream.cuda_stream)
    tab = U.UsageTable(eng)
    tab.load_columns(ts[lo:hi], list(models[lo:hi]), *[t[lo:hi] for t in tok], cost[lo:hi], names=names)
    tab._upload()
    t_min, t_max = int(ts.min()), int(ts.max())
    nm = len(names) + 1
    lib = tab._lib
    queries = []
    for period in ("hour", "day"):
        s0, e0 = U.stats_window(period, end)
        for label, start, stop in ((period + "_window", s0, e0), (period + "_all", None, None)):
            p = U.PERIODS[period]
            qlo = max(t_min, U.to_us(start)) if start is not None else t_min
            qhi = min(t_max, U.to_us(stop)) if stop is not None else t_max
            b0 = int(lib.lgw_rollup_bucket_of(qlo, p)); b1 = int(lib.lgw_rollup_bucket_of(qhi, p))
            nb = b1 - b0 + 1 + (25 if period == "hour" else 1)
            queries.append(dict(label=label, period=period, start=start, end=stop, b0=b0, nb=nb, groups=nb * nm,
                                table=torch.zeros(nb * nm * U.ROLLUP_CELLS, dtype=torch.int64, device=dev),
                                inexact=torch.zeros(nb * nm, dtype=torch.int32, device=dev), oob=torch.zeros(2, dtype=torch.int32, device=dev)))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def one(q, timed=None):
        with torch.cuda.stream(stream):
            q["table"].zero_(); q["inexact"].zero_(); q["oob"].zero_()
            flush.fill_(1)                                 # evict L2 (not timed)
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record(stream)
            tab.accumulate(q["period"], q["start"], q["end"], q["b0"], q["nb"], nm, C.c_void_p(q["table"].data_ptr()),
                           C.c_void_p(q["inexact"].data_ptr()), C.c_void_p(q["oob"].data_ptr()))
            e1.record(stream)
            if world > 1:
                dist.all_reduce(q["table"], op=dist.ReduceOp.SUM)
                dist.all_reduce(q["inexact"], op=dist.ReduceOp.MAX)
            rows = tab.emit(q["b0"], q["nb"], nm, C.c_void_p(q["table"].data_ptr()), C.c_void_p(q["inexact"].data_ptr()), pinned=True) if rank == 0 else None
            e2.record(stream)
        torch.cuda.synchronize(dev)
        if timed is not None:
            timed.append((e0.elapsed_time(e1), e0.elapsed_time(e2)))
        return rows

    sampler = ClockSampler(local); sampler.start()
    for _ in range(W):
        for q in queries:
            one(q)
    barrier()
    l0 = eng.launch_count()
    per_q = {q["label"]: [] for q in queries}
    rows_of = {}
    for _ in range(K):
        for q in queries:
            barrier()
            r = one(q, per_q[q["label"]])
            rows_of[q["label"]] = r.copy() if r is not None else None      # (not timed: the pinned row buffer is reused by the next rollup)
    barrier()
    launches = eng.launch_count() - l0
    sampler.stop()
    res = {}
    for q in queries:
        acc = max_over_ranks(float(np.mean([t[0] for t in per_q[q["label"]]])))
        tot = max_over_ranks(float(np.mean([t[1] for t in per_q[q["label"]]])))
        res[q["label"]] = dict(groups=q["groups"], accum_ms=acc, total_ms=tot, records_per_s=n / (tot / 1e3),
                               accum_gbs_rank=40.0 * (hi - lo) / (acc / 1e3) / 1e9, path="privatised (shared memory)" if q["groups"] <= 2560 else "global 64-bit reductions")
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # correctness of the timed configuration (not timed): conservation against the host columns
    for q in queries:
        rows = rows_of[q["label"]]
        sel = np.ones(n, bool)
        if q["start"] is not None:
            sel = (ts >= U.to_us(q["start"])) & (ts <= U.to_us(q["end"]))
        assert int(rows["count"].sum()) == int(sel.sum()), (q["label"], int(rows["count"].sum()), int(sel.sum()))
        assert int(rows["prompt_tokens"].sum()) == int(tok[0][sel].astype(np.int64).sum())
        assert int(rows["cached_tokens"].sum()) == int(tok[4][sel].astype(np.int64).sum())
    peak, peak_src = _peaks()
    step_ms = sum(r["total_ms"] for r in res.values())
    head = res["day_window"]
    value = n * len(res) / (step_ms / 1e3)
    achieved = head["accum_gbs_rank"]
    line = {"metric": "usage_rollup_records_per_sec", "value": value, "unit": "records/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": "C5: usage-stats rollup, 10M extracted usage records -> per-hour/day x model aggregation (SURVEY 8(d) C5: 400-day window, 64 models Zipf 1.1 + 1% NULL)",
                       "records_total": n, "records_rank0": hi - lo, "step": "4 rollups: hour and day, each over the stats endpoint's window (24 h / 2 weeks) and over the whole table",
                       "l2": "flushed: 256 MiB written on the stream before every rollup (not timed)", "parallelism": f"row ranges x{world}; one all-reduce(sum) of the dense table per rollup"},
            "rollups": res, "clocks": sampler.summary(), "gpu_launches": int(launches),
            "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(sum(len(rows_of[q["label"]]) for q in queries) * U.ROW_DTYPE.itemsize),
                    "note": "records are device-resident by design (ingested once, queried many times); the result rows are copied to the host inside the timed region"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "kernel": "k_rollup_accum_smem + k_rollup_merge on the `day` window (40 B algorithmic per record, SURVEY 8(d)); the other rollups are in `rollups`"}}
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTE_SAMPLE = 1 << 21          # re-emitted byte positions in the dump (seeded, fixed for a given input size)
DUMP_MAX_STREAMS = 4096             # streams whose verdicts, states and usage records are dumped (all of them at the default size)
DUMP_MAX_BYTES = 64 << 20


def _c3_outputs(eng, batch_set, dev) -> dict:
    """What a caller of the device step holds after one step, as float arrays: the re-emitted bytes (a seeded sample of
    positions), each stream's segment verdict, and each stream's state with the usage record the tap extracted."""
    import torch
    from llmapigateway_b200._abi import KIND_FLOAT, KIND_INT
    from llmapigateway_b200.engine import SEG_DTYPE
    b, h, d = batch_set
    rng = np.random.default_rng(0)
    n_bytes, n_streams = int(b.data.size), int(b.seg_slot.size)
    pos = np.unique(rng.integers(0, n_bytes, size=min(n_bytes, DUMP_BYTE_SAMPLE)))
    out = {"out_bytes_pos": pos.astype(np.float64),
           "out_bytes": d["out"][torch.from_numpy(pos).to(dev)].cpu().numpy().astype(np.float32)}
    sel = np.arange(n_streams) if n_streams <= DUMP_MAX_STREAMS else np.sort(rng.choice(n_streams, DUMP_MAX_STREAMS, replace=False))
    out["stream_index"] = sel.astype(np.float64)
    segs = d["segs"].cpu().numpy().view(SEG_DTYPE)[sel]
    for f in SEG_DTYPE.names:
        out["seg_" + f] = segs[f].astype(np.float64)
    st = np.ctypeslib.as_array(eng.state(b.seg_slot[sel]))
    for f in st.dtype.names:
        if f != "rec":
            out["state_" + f] = st[f].astype(np.float64)
    rec = st["rec"]
    for f in ("prompt_tokens", "completion_tokens", "total_tokens", "reasoning_tokens", "cached_tokens", "cost", "model_val", "provider_val"):
        bits, kind = rec[f]["bits"], rec[f]["kind"]
        val = np.zeros(len(sel))                    # 0 where the value is not a number (string, null, absent ...): `_kind` says which
        val[kind == KIND_INT] = bits[kind == KIND_INT]
        val[kind == KIND_FLOAT] = bits[kind == KIND_FLOAT].view(np.float64)
        out["usage_" + f] = val
        out["usage_" + f + "_kind"] = kind.astype(np.float64)
    for f in ("model", "provider"):
        raw = rec[f].view(np.uint8).reshape(len(sel), -1)
        live = np.arange(raw.shape[1])[None, :] < rec[f + "_len"][:, None]       # bytes past the length are not part of the value
        out["usage_" + f + "_bytes"] = np.where(live, raw, 0).astype(np.float32)
        out["usage_" + f + "_len"] = rec[f + "_len"].astype(np.float64)
    out["usage_str_flags"] = rec["str_flags"].astype(np.float64)
    out["usage_exotic"] = rec["exotic"].astype(np.float64)
    return out


def _write_outputs(path: str, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"dump of {total} bytes exceeds {DUMP_MAX_BYTES}"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def _emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--streams", type=int, default=N_STREAMS)
    ap.add_argument("--events", type=int, default=N_EVENTS)
    ap.add_argument("--mode", type=int, default=0, help="0 bulk kernel (default), 1 exact sequential path")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="c3", choices=["c3", "c4", "c5"],
                    help="c3 (default): BASELINE configs[2], the headline; c4: 3-deep fallback chain with 20 %% injected failure, 8192 streams "
                         "sharded over the GPUs (strong scaling); c5: usage rollup of 10 M records, 1 vs N GPUs")
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="c3: write what the last timed step computed as DIR/<name>.npy (float32/float64, at most 64 MB in all; "
                         "a seeded sample of the re-emitted bytes), so that two builds can be compared output for output; "
                         "e.g. bench_outputs/<build> (git-ignored)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != "c3" or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for the default configuration (--config c3 --impl b200)")
    # stdout carries exactly one line, the JSON result: everything else that writes to fd 1 during the run (NCCL's
    # version banner, library chatter of child processes) is sent to stderr
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference_arm(args) if args.config == "c3" else run_reference_side(args)
    if args.config == "c4":
        return run_c4(args)
    if args.config == "c5":
        return run_c5(args)

    import torch
    import torch.distributed as dist
    import llmapigateway_b200 as L
    from llmapigateway_b200 import _abi
    from llmapigateway_b200.engine import SEG_DTYPE
    from llmapigateway_b200.synth import sse_batch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the engine has no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    from llmapigateway_b200 import numa
    numa_info = numa.bind_to_gpu_node(local)        # pinned staging buffers on the GPU's own NUMA node (before anything is allocated)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    S, E = args.streams, args.events
    W, K = max(args.warmup, 3), args.steps

    eng = L.Engine(device=local, max_streams=S, max_step_chunks=S * (E + 2) + 8, max_step_bytes=S * (E * EVENT_BYTES + 512))
    eng.set_mode(args.mode)
    # two alternating input sets: every step touches 2 x 128 MiB of HBM that the previous step evicted from L2
    sets = []
    for k in range(2):
        b = sse_batch(n_streams=S, n_events=E, seed=3 + 1000 * k + rank)
        pin = lambda a: torch.from_numpy(a).pin_memory()
        h = {"data": pin(b.data), "chunk_off": pin(b.chunk_off), "seg_chunk": pin(b.seg_chunk), "seg_slot": pin(b.seg_slot)}
        d = {n: t.to(dev) for n, t in h.items()}
        d["out"] = torch.empty_like(d["data"])
        d["segs"] = torch.empty(S * SEG_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        h["out"] = torch.empty(b.data.size, dtype=torch.uint8).pin_memory()
        sets.append((b, h, d))
    stream = torch.cuda.Stream(device=dev)
    eng.set_stream(stream.cuda_stream)
    status = np.full(S, 200, dtype=np.int32)
    n_chunks = sets[0][0].n_chunks

    def device_step(k):
        b, h, d = sets[k % 2]
        eng.open(b.seg_slot, status)           # stream table reset (tiny kernel)
        eng.step_device(d["data"].data_ptr(), int(b.data.size), d["chunk_off"].data_ptr(), n_chunks, d["seg_chunk"].data_ptr(),
                        d["seg_slot"].data_ptr(), S, d["out"].data_ptr(), d["segs"].data_ptr())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- value: device-resident ------------------------------------------------------------------
    sampler = ClockSampler(local); sampler.start()
    for k in range(W):
        device_step(k); eng.sync()
    # keep the GPU under the same load for ~0.4 s before the timed steps so that the clock sampler
    # (20 ms period) sees clocks and throttle reasons under this very workload; not timed
    t_load = time.perf_counter(); k_load = 0
    while time.perf_counter() - t_load < 0.4:
        device_step(k_load); k_load += 1
        if k_load % 16 == 0:
            eng.sync()
    eng.sync()
    barrier()
    l0 = eng.launch_count()
    chained_ms = 0.0      # engine events around the three kernels of a step (chained with programmatic dependent launches)
    step_ms = []
    # Between timed steps (not timed): 256 MiB written on the same stream.  It evicts L2 (126 MB) and keeps the GPU busy
    # while the host enqueues the step's launches, so the timed region is the device's work, not the host's launch latency
    # (a serving loop enqueues step k+1 while step k runs).
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    t_wall0 = time.perf_counter()
    for k in range(K):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b, h, d = sets[k % 2]
        with torch.cuda.stream(stream):
            flush.fill_(k & 1)
        eng.open(b.seg_slot, status)
        with torch.cuda.stream(stream):
            e0.record(stream)
            eng.step_device(d["data"].data_ptr(), int(b.data.size), d["chunk_off"].data_ptr(), n_chunks, d["seg_chunk"].data_ptr(),
                            d["seg_slot"].data_ptr(), S, d["out"].data_ptr(), d["segs"].data_ptr())
            e1.record(stream)
        eng.sync()
        step_ms.append(e0.elapsed_time(e1))
        chained_ms += eng.last_step_ms()["relay"]        # (chained launches: the total of the step's kernels comes back here)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = eng.launch_count() - l0
    outputs = _c3_outputs(eng, sets[(K - 1) % 2], dev) if args.dump_outputs and rank == 0 else None     # (before anything reuses the set)
    dev_ms = float(np.sum(step_ms))
    if world > 1:
        t = torch.tensor([dev_ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); dev_ms = float(t.item())
    ms_per_step = dev_ms / K
    events_total = world * S * E
    value = events_total / (ms_per_step / 1e3)

    # per-kernel breakdown: the same step with CUDA events between the kernels (back-to-back launches, not timed into `value`)
    kern = {"prime": 0.0, "relay": 0.0, "commit": 0.0}
    eng.set_kernel_timing(True)
    KB = 5
    for k in range(KB + 1):
        b, h, d = sets[k % 2]
        with torch.cuda.stream(stream):
            flush.fill_(k & 1)
        eng.open(b.seg_slot, status)
        eng.step_device(d["data"].data_ptr(), int(b.data.size), d["chunk_off"].data_ptr(), n_chunks, d["seg_chunk"].data_ptr(),
                        d["seg_slot"].data_ptr(), S, d["out"].data_ptr(), d["segs"].data_ptr())
        eng.sync()
        if k:
            ms = eng.last_step_ms()
            for n in kern:
                kern[n] += ms[n] / KB
    eng.set_kernel_timing(False)
    counters = eng.debug_counters()

    # correctness spot check of the timed configuration (not timed)
    b, h, d = sets[KB % 2]                              # the set of the last step that ran (the breakdown loop's last)
    torch.cuda.synchronize(dev)
    assert torch.equal(d["out"], d["data"]), "re-emitted bytes differ from the input of committed streams"
    st = eng.state(b.seg_slot[:4])
    for s in range(4):
        assert _abi.usage_rec_to_dict(st[s].rec) == b.truths[s].expected_row()

    # ---- e2e: host buffers through the C-ABI call ---------------------------------------------------
    e2e_ms = []
    for k in range(2 + min(K, 5)):
        b, h, d = sets[k % 2]
        barrier()
        t0 = time.perf_counter()
        eng.open(b.seg_slot, status)
        res = eng.step(h["data"].numpy(), h["chunk_off"].numpy(), h["seg_chunk"].numpy(), h["seg_slot"].numpy(), out=h["out"].numpy())
        states = eng.close(b.seg_slot)
        barrier()
        if k >= 2:
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
    e2e_step = float(np.mean(e2e_ms))
    assert np.array_equal(h["out"].numpy(), h["data"].numpy()), "end-to-end: re-emitted host bytes differ from the input of committed streams"
    assert _abi.usage_rec_to_dict(states[5].rec) == b.truths[5].expected_row()
    e2e_direct = eng.last_step_direct()
    if world > 1:
        t = torch.tensor([e2e_step], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_step = float(t.item())
    e2e_value = events_total / (e2e_step / 1e3)
    n_bytes = int(sets[0][0].data.size)
    h2d = n_bytes + 4 * (n_chunks + 1) + 4 * (S + 1) + 4 * S + 8 * S
    d2h = n_bytes + S * SEG_DTYPE.itemsize + S * 440

    # ---- the same end-to-end call in "verdicts only" mode (out_bytes = NULL: the caller relays its own copy of the chunks, as
    # StreamBatcher(relay_from="host") does); a side measurement -- the headline `e2e` above downloads the re-emitted bytes --------
    e2e_vo = None
    try:
        if world > 1:                       # a single-GPU side figure: the multi-GPU lines carry the headline numbers only
            raise StopIteration
        vo_ms = []
        for k in range(2 + min(K, 5)):
            b, h, d = sets[k % 2]
            barrier()
            t0 = time.perf_counter()
            eng.open(b.seg_slot, status)
            res = eng.step(h["data"].numpy(), h["chunk_off"].numpy(), h["seg_chunk"].numpy(), h["seg_slot"].numpy(), relay_from_host=True)
            states = eng.close(b.seg_slot)
            barrier()
            if k >= 2:
                vo_ms.append((time.perf_counter() - t0) * 1e3)
        vo_step = float(np.mean(vo_ms))
        assert bool((res.segs["emit_chunk_begin"].astype(np.int64) == np.asarray(b.seg_chunk[:-1], dtype=np.int64)).all()), "verdicts-only: a committed stream does not relay from its first chunk"
        assert res.out.ctypes.data == h["data"].numpy().ctypes.data, "verdicts-only: the relayed bytes must be the caller's own buffer"
        assert _abi.usage_rec_to_dict(states[5].rec) == b.truths[5].expected_row()
        if world > 1:
            t = torch.tensor([vo_step], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); vo_step = float(t.item())
        e2e_vo = {"value": events_total / (vo_step / 1e3), "unit": UNIT, "ms_per_step": vo_step, "h2d_bytes_per_step": h2d,
                  "d2h_bytes_per_step": S * SEG_DTYPE.itemsize + S * 440,
                  "note": "lgw_sse_step with out_bytes = NULL: the relayed bytes are the caller's own (request_handler.py:141-142 yields the original chunk); "
                          "the kernels and the device-side re-emit are unchanged, only the download of the bytes is left out. NOT the headline e2e."}
    except StopIteration:
        e2e_vo = None
    except Exception as ex:
        e2e_vo = {"error": repr(ex)}

    # ---- transcript tap (SURVEY 8(f) rank 3), same C3 batch, device resident; a side measurement, not part of `value` -----------
    text_tap = None
    if world == 1:
        try:
            eng.enable_transcripts()
            t_ms = []
            for k in range(4):
                b, h, d = sets[k % 2]
                eng.open(b.seg_slot, status)
                eng.step_device(d["data"].data_ptr(), int(b.data.size), d["chunk_off"].data_ptr(), n_chunks, d["seg_chunk"].data_ptr(),
                                d["seg_slot"].data_ptr(), S, d["out"].data_ptr(), d["segs"].data_ptr())
                eng.sync()
                st_text = eng.step_transcript()
                if k:
                    t_ms.append(eng.transcript_last_ms())
            raw = b.data.tobytes()[:E * EVENT_BYTES]              # stream 0 of the last set: its text is the 8 content bytes of every delta
            want = b"".join(raw[i * EVENT_BYTES + 49:i * EVENT_BYTES + 57] for i in range(E))
            assert st_text.segment(0) == want, "transcript of stream 0 differs from its content bytes"
            assert int(st_text.seg_off[-1]) == S * E * 8 and not (st_text.flags & _abi.TF_SEQUENTIAL).any()
            tm = float(np.mean(t_ms))
            text_tap = {"ms": tm, "kernels": "k_text_extract + k_text_scan + k_text_pack", "text_bytes": int(st_text.seg_off[-1]),
                        "input_gbs": int(b.data.size) / (tm / 1e3) / 1e9, "note": "every event parsed again with the full machine, one chunk per lane"}
        except Exception as ex:
            text_tap = {"error": repr(ex)}

    sampler.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = _peaks()
    kern_step = dict(kern)
    kernel_ms = chained_ms / K                      # device time of the step's kernels as launched in the timed region
    algo = S * E * ALGO_BYTES_PER_EVENT
    achieved = algo / (kernel_ms / 1e3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "C3: 4096 concurrent SSE streams x 512 data: deltas (64 B each), parse/normalise/re-emit",
                   "streams_per_gpu": S, "events_per_stream": E, "event_bytes": EVENT_BYTES, "events_per_chunk": 1,
                   "extra_chunks_per_stream": "1 usage event + data: [DONE] (not counted)", "parallelism": f"streams sharded x{world}, no collective",
                   "l2": "flushed: 256 MiB written on the stream before every timed step (not timed), plus two alternating input/output sets (268 MB per step; L2 = 126 MB)",
                   "mode": "bulk" if args.mode == 0 else "sequential"},
        "json_gbs": value * EVENT_BYTES / 1e9,
        "kernel_ms": {"step_chained": kernel_ms, "back_to_back": kern_step, "back_to_back_sum": sum(kern_step.values())},
        "segments": counters,
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_step, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "json_gbs": e2e_value * EVENT_BYTES / 1e9,
                "path": ("direct: the bulk kernel's TMA loads/stores move the bytes over PCIe themselves (LGW_DIRECT)" if e2e_direct
                         else "pinned host buffers, 8 slices: upload of slice k+1 | kernels of slice k | download of slice k-1 on three streams"),
                "numa": numa_info, "pcie_peak_note": "copy engines alone, 134 MB each way at once: 2.78 ms (48.7 GB/s per direction; 55 GB/s one direction alone), measured with tools/exp_e2e.py on this pool"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": _traffic(), "peak_source": peak_src,
                     "kernel": "k_prime2 + k_relay2 + k_commit2 (the whole step: CUDA events around the three kernels as launched in the timed region, "
                               "chained with programmatic dependent launches; 128 B algorithmic per 64-B event; usage-field extraction is inside: "
                               "k_relay2 locates the fields of every stream's usage event, k_commit2 reads them out)"},
        "wall_s_timed_loop": t_wall,
    }
    if e2e_vo is not None:
        line["e2e_verdicts_only"] = e2e_vo
    if text_tap is not None:
        line["transcript_tap"] = text_tap
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_block(E)
    if world == 1 and not args.no_cpu_baseline:
        # the other built rows of SURVEY 8 on their own configurations (C2 bodies, C5 rollup at 2M records), same box, same run
        try:
            sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))   # (spawned CPU workers import it by name)
            import bench_rows as br
            eng2 = L.Engine(max_streams=64, max_step_chunks=1024, max_step_bytes=1 << 20, device=local)
            line["other_rows"] = br.bench_bodies(eng2, 1024, reps=10) + br.bench_rollup(eng2, 2_000_000)
            eng2.close_engine()
        except Exception as ex:                                    # never lose the headline line to a side measurement
            line["other_rows"] = {"error": repr(ex)}
    if outputs is not None:
        _write_outputs(args.dump_outputs, outputs)
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
