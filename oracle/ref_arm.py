"""The reference's OWN code as the CPU arm -- TEST INFRASTRUCTURE (bench.py's cpu_baseline / --impl reference legs only).

Drives, unmodified, from oracle/_ref (a copy of the reference made by oracle/build_ref.py):
  llm_gateway_core/services/request_handler.py:8     make_llm_request(..., is_streaming=True)  -- stream_generator,
        priming loop, combined_generator (loop A) over an httpx.MockTransport upstream (no sockets)
  llm_gateway_core/middleware/chat_logging.py:69     ChunkProcessorThread.run (loop B) + get_token_usage :233 on the
        relayed chunks, write_log replaced by a recorder (the DB-row point, :54)
i.e. BASELINE.md section 3's B1/B2 variants.  `json5` is not installed in this image (no network):
  B2 "generous": json5.loads -> the stdlib's C json.loads
  B1 "faithful": json5.loads -> the stdlib's PURE-PYTHON decoder (json.decoder with py_scanstring / py_make_scanner), the
                 closest stand-in available for a pure-Python recursive-descent parser (the real json5 is slower still)
Logging is left at the reference's default (INFO records are formatted and dropped by a NullHandler: no console I/O).
"""
from __future__ import annotations

import asyncio
import copy
import json
import logging
import os
import queue
import sys
import tempfile
import time
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF_DIR = HERE / "_ref"


def ref_root() -> Path | None:
    return REF_DIR if (REF_DIR / "llm_gateway_core" / "services" / "request_handler.py").exists() else None


def _pure_python_loads():
    import json.decoder as jd
    import json.scanner as js

    class PyDecoder(jd.JSONDecoder):
        def __init__(self, **kw):
            super().__init__(**kw)
            self.parse_string = jd.py_scanstring
            self.parse_object = jd.JSONObject
            self.parse_array = jd.JSONArray
            self.scan_once = js.py_make_scanner(self)

    dec = PyDecoder()
    return dec.decode


def install_json5(variant: str):
    shim = types.ModuleType("json5")
    loads = json.loads if variant == "B2" else _pure_python_loads()
    shim.loads = lambda s, **kw: loads(s)
    shim.load = lambda fp, **kw: json.loads(fp.read())
    shim.dumps = lambda o, **kw: json.dumps(o)
    shim.JSONDecodeError = json.JSONDecodeError
    shim.__doc__ = f"stand-in for the missing json5 package ({variant})"
    sys.modules["json5"] = shim


_mods = {}


def load(variant: str):
    """Import the reference modules from oracle/_ref with the json5 stand-in of `variant`."""
    if _mods.get("variant") == variant:
        return _mods["rh"], _mods["cl"]
    root = ref_root()
    if root is None:
        raise RuntimeError("reference sources not available (oracle/_ref missing: run oracle/build_ref.py next to a reference checkout)")
    install_json5(variant)
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    for h in list(logging.getLogger().handlers):
        logging.getLogger().removeHandler(h)
    logging.getLogger().addHandler(logging.NullHandler())
    logging.getLogger().setLevel(logging.INFO)            # the reference's default level: records are built, not printed
    os.environ.setdefault("LOG_CHAT_ENABLED", "true")
    for name in [m for m in sys.modules if m.startswith("llm_gateway_core")]:
        del sys.modules[name]
    import llm_gateway_core.db.tokens_usage_db as tdb
    tmp = Path(tempfile.mkdtemp(prefix="lgw_ref_")) / "tokens_usage.db"

    def _init(self, db_filename: str = "tokens_usage.db"):      # tokens_usage_db.py:17-25 hard-codes <root>/db
        self.db_path = tmp
        self._init_db()

    tdb.TokensUsageDB.__init__ = _init
    import llm_gateway_core.services.request_handler as rh
    import llm_gateway_core.middleware.chat_logging as cl
    _mods.update(variant=variant, rh=rh, cl=cl)
    return rh, cl


class _NoWaitQueue(queue.Queue):
    def get(self, block=True, timeout=None):      # chat_logging.py:94 waits 5 s for the next chunk; the stream is over
        return super().get(block=False)


def run_streams(streams: list[list[bytes]], variant: str = "B2", with_tap: bool = True):
    """All `streams` (lists of network chunks) through the reference, one after the other on this core (the reference is a
    single event loop).  Returns (seconds, n_events_relayed_bytes, rows)."""
    import httpx
    rh, cl = load(variant)
    rows = []
    real_write = cl.write_log
    cl.write_log = lambda h, b, accum, usage: rows.append(copy.copy(usage))
    real_client = httpx.AsyncClient
    cur = {"chunks": None}

    class _Body(httpx.AsyncByteStream):
        async def __aiter__(self):
            for c in cur["chunks"]:
                yield c

    def handler(request):
        return httpx.Response(200, headers={"content-type": "text/event-stream"}, stream=_Body())

    rh.httpx.AsyncClient = lambda **kw: real_client(transport=httpx.MockTransport(handler), **kw)
    n_bytes = 0

    async def go():
        nonlocal n_bytes
        for chunks in streams:
            cur["chunks"] = chunks
            resp, err = await rh.make_llm_request("http://upstream.test/v1/chat/completions", {}, {"model": "m", "messages": []}, True)
            assert resp is not None, err
            out = []
            try:
                async for c in resp.body_iterator:
                    out.append(c)
            except UnboundLocalError:              # request_handler.py:144 when no usage was seen
                pass
            n_bytes += sum(len(c) for c in out)
            if with_tap and out:
                t = cl.ChunkProcessorThread({}, "", True)
                t.queue = _NoWaitQueue()
                for c in out:
                    t.enqueue_chunk(c)
                t.run()

    t0 = time.perf_counter()
    try:
        asyncio.run(go())
    finally:
        rh.httpx.AsyncClient = real_client
        cl.write_log = real_write
    return time.perf_counter() - t0, n_bytes, rows


def effective_cores() -> int:
    """CPUs this process may really use: the affinity mask, capped by the cgroup's cpu.max quota."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def _worker(args):
    variant, seed, n_streams, n_events, stream_lo = args
    sys.path.insert(0, str(HERE.parent))
    from llmapigateway_b200.synth import sse_batch
    b = sse_batch(n_streams=n_streams, n_events=n_events, seed=seed, slot_base=stream_lo)
    streams = [b.stream_chunks(s) for s in range(n_streams)]
    secs, n_bytes, rows = run_streams(streams, variant)
    assert len(rows) == n_streams and n_bytes == int(b.data.size)
    return secs


def run_config3(variant: str, procs: int, n_streams: int, n_events: int = 512, seed: int = 3):
    """`n_streams` C3 streams split evenly over `procs` processes (BASELINE.md B?-N).  Returns (events/s, slowest process s, wall s)."""
    import multiprocessing as mp
    per = [n_streams // procs + (1 if i < n_streams % procs else 0) for i in range(procs)]
    jobs, lo = [], 0
    for i, n in enumerate(per):
        if n:
            jobs.append((variant, seed + 7919 * i, n, n_events, lo)); lo += n
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    if len(jobs) == 1:
        times = [_worker(jobs[0])]
    else:
        with ctx.Pool(len(jobs)) as pool:
            times = pool.map(_worker, jobs)
    wall = time.perf_counter() - t0
    return n_streams * n_events / max(times), max(times), wall


# ---- config 4: the reference's own endpoint body (chat.py:20 chat_completions) over the failure-injecting upstream --------------
def load_chat(variant: str = "B2"):
    """chat.py imported unmodified from oracle/_ref: ModelRotationDB's file redirected to a temp dir (model_rotation_db.py:15-22
    hard-codes <root>/db), api/v1/models.py (loads config files at import; not on this path) replaced by an empty router."""
    import types
    load(variant)
    import llm_gateway_core.db.model_rotation_db as mdb
    tmp = Path(tempfile.mkdtemp(prefix="lgw_rot_")) / "rotation.db"

    def _init(self, db_filename: str = "llmgateway_rotation.db"):
        self.db_path = tmp
        self._init_db()

    mdb.ModelRotationDB.__init__ = _init
    from fastapi import APIRouter
    stub = types.ModuleType("llm_gateway_core.api.v1.models")
    stub.router = APIRouter()
    sys.modules["llm_gateway_core.api.v1.models"] = stub
    import llm_gateway_core.api.v1.chat as chat
    return chat


def _c4_worker(args):
    variant, ids, n_total, n_events = args
    import types
    import httpx
    sys.path.insert(0, str(HERE.parent))
    from llmapigateway_b200 import synth
    chat = load_chat(variant)
    rh, cl = _mods["rh"], _mods["cl"]
    providers, rules, fallback_provider = synth.chain_world()
    chat.settings.fallback_provider = fallback_provider
    os.environ.setdefault("ALPHA_KEY_ENV", "sk-alpha-from-env")
    loader = types.SimpleNamespace(providers_config=providers, fallback_rules=rules)
    up = synth.ChainUpstream(n_total, n_events, seed=4, p_fail=0.2, lazy=True)
    bodies = synth.chain_request_bodies(n_total, seed=4)
    cl.write_log = lambda h, b, accum, usage: None
    state = {"sid": 0, "attempt": 0}

    class _Body(httpx.AsyncByteStream):
        def __init__(self, chunks):
            self.chunks = chunks

        async def __aiter__(self):
            for c in self.chunks:
                yield c

    def handler(request):
        ans = up.stream_chunks(state["sid"], state["attempt"])
        state["attempt"] += 1
        if isinstance(ans, tuple):
            return httpx.Response(ans[0], content=ans[1])
        return httpx.Response(200, headers={"content-type": "text/event-stream"}, stream=_Body(ans))

    real_client = httpx.AsyncClient
    rh.httpx.AsyncClient = lambda **kw: real_client(transport=httpx.MockTransport(handler), **kw)
    served = [0]

    class Req:
        def __init__(self, body):
            self._b = body
            self.headers = {}
            self.app = types.SimpleNamespace(state=types.SimpleNamespace(config_loader=loader))

        async def body(self):
            return self._b

    async def go():
        from fastapi import HTTPException
        for sid in ids:
            state["sid"], state["attempt"] = int(sid), 0
            try:
                resp = await chat.chat_completions(Req(bodies[int(sid)]))
            except HTTPException:
                continue
            out = []
            try:
                async for c in resp.body_iterator:
                    out.append(c)
            except UnboundLocalError:
                pass
            t = cl.ChunkProcessorThread({}, "", True)          # chat_logging.py tap of the relayed stream
            t.queue = _NoWaitQueue()
            for c in out:
                t.enqueue_chunk(c)
            t.run()
            served[0] += 1

    t0 = time.perf_counter()
    try:
        asyncio.run(go())
    finally:
        rh.httpx.AsyncClient = real_client
    return time.perf_counter() - t0, served[0]


def run_config4(variant: str, procs: int, ids, n_total: int = 8192, n_events: int = 512):
    """The streams `ids` of config 4 through the unmodified chat_completions, split over `procs` processes.
    -> (delta events relayed per second, slowest process seconds, served streams)."""
    import multiprocessing as mp
    ids = list(ids)
    parts = [ids[i::procs] for i in range(procs)]
    jobs = [(variant, p, n_total, n_events) for p in parts if p]
    if len(jobs) == 1:
        res = [_c4_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(len(jobs)) as pool:
            res = pool.map(_c4_worker, jobs)
    served = sum(r[1] for r in res)
    slowest = max(r[0] for r in res)
    return served * n_events / slowest, slowest, served


# ---- config 5: TokensUsageDB.get_aggregated_usage (tokens_usage_db.py:222) on a SQLite file of the same records -----------------------
def run_config5(n_rows: int, periods=("hour", "day")):
    """-> dict(load_s, per query seconds).  The reference has one process and SQLite is single-threaded per connection."""
    import sqlite3
    from datetime import datetime, timedelta
    sys.path.insert(0, str(HERE.parent))
    from llmapigateway_b200 import usage as U
    load("B2")
    import llm_gateway_core.db.tokens_usage_db as tdb
    db = tdb.TokensUsageDB()
    end = datetime(2026, 9, 21, 6, 57, 17, 47518)
    ts, models, tok, cost = U.synth_usage_columns(n_rows, seed=5, end=end)
    epoch = datetime(1970, 1, 1)
    t0 = time.perf_counter()
    conn = sqlite3.connect(db.db_path)
    conn.executemany("INSERT INTO tokens_usage (timestamp, prompt_tokens, completion_tokens, total_tokens, reasoning_tokens, cached_tokens, cost, model, provider)"
                     " VALUES (?,?,?,?,?,?,?,?,NULL)",
                     (((epoch + timedelta(microseconds=int(ts[i]))).isoformat(), int(tok[0][i]), int(tok[1][i]), int(tok[2][i]), int(tok[3][i]), int(tok[4][i]),
                       float(cost[i]), models[i]) for i in range(n_rows)))
    conn.commit(); conn.close()
    out = {"load_s": time.perf_counter() - t0, "rows": n_rows}
    for period in periods:
        s0, e0 = U.stats_window(period, end)
        t0 = time.perf_counter(); r1 = db.get_aggregated_usage(period, start_date=s0, end_date=e0); out[period + "_window_s"] = time.perf_counter() - t0
        t0 = time.perf_counter(); r2 = db.get_aggregated_usage(period); out[period + "_all_s"] = time.perf_counter() - t0
        out[period + "_groups"] = (len(r1), len(r2))
    return out
