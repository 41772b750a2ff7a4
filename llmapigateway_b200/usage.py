"""Usage records on the device and their rollup -- the host-side mirror of
llm_gateway_core/db/tokens_usage_db.py (TokensUsageDB) for rows a10/a11 of SURVEY.md section 8:

  UsageTable.insert_usage(d)         <- TokensUsageDB.insert_usage          (:119-162)
  UsageTable.get_aggregated_usage()  <- TokensUsageDB.get_aggregated_usage  (:222-304)  [GPU kernel]
  stats_window(period, now)          <- llm_gateway_core/api/v1/stats.py:46-55

Records live as SoA columns (40 B/record) in HBM; `model` is dictionary-encoded at ingest and
ranked in byte order so that ascending rank == the SQL's `model ASC`.  Every accumulator of the
rollup is an integer (see csrc/rollup.cuh), so per-GPU partial tables merge with a plain sum.
A group whose cost the fixed-point sum cannot hold (flag `inexact`) is answered on the host from
the host copy of its records, the way SQLite sums them (`sqlite_sum`).
"""
from __future__ import annotations

import ctypes as C
import math
from datetime import datetime, timedelta

import numpy as np

from . import _native

PERIODS = {"hour": 0, "day": 1, "week": 2, "month": 3}
_EPOCH = datetime(1970, 1, 1)
ROLLUP_CELLS = 10

ROW_DTYPE = np.dtype([("bucket", "<i8"), ("model_rank", "<i4"), ("inexact", "<u4"), ("prompt_tokens", "<i8"),
                      ("completion_tokens", "<i8"), ("total_tokens", "<i8"), ("reasoning_tokens", "<i8"),
                      ("cached_tokens", "<i8"), ("cost", "<f8"), ("count", "<i8")])
assert ROW_DTYPE.itemsize == 72


def to_us(dt: datetime) -> int:
    return (dt - _EPOCH) // timedelta(microseconds=1)


def period_label(period: str, bucket: int) -> str:
    """strftime(fmt, timestamp) of tokens_usage_db.py:242-250 for a bucket index."""
    if period == "hour":                      # bucket = day * 24 + hour of day (csrc/rollup.cuh)
        return (_EPOCH + timedelta(days=bucket // 24)).strftime("%Y-%m-%d") + " %02d:00:00" % (bucket % 24)
    if period == "day":
        return (_EPOCH + timedelta(days=bucket)).strftime("%Y-%m-%d")
    if period == "week":
        return "%04d-W%02d" % (bucket // 64, bucket % 64)
    return "%04d-%02d" % (bucket // 12, bucket % 12 + 1)


def sqlite_sum(costs) -> float | None:
    """SUM(cost) of SQLite >= 3.43 over REAL values in scan order (Kahan-Babuska-Neumaier).  A NaN was stored as NULL and is
    skipped; no value left gives NULL (None); a NaN result is NULL too.  A NaN error term is dropped, which is how [inf, 1.0]
    sums to inf; an infinite one is not, so a sum that overflows, [1e308, 1e308], is inf + -inf = NULL."""
    s = err = 0.0
    seen = False
    for r in costs:
        if r != r:
            continue
        seen = True
        t = s + r
        err += (s - t) + r if abs(s) > abs(r) else (r - t) + s
        s = t
    if not seen:
        return None
    out = s if math.isnan(err) else s + err
    return None if math.isnan(out) else out


def _bucket_span_us(period: str, bucket: int) -> tuple[int, int]:
    """[lo, hi) in microseconds holding every timestamp whose bucket_of() is `bucket`, with the one-day slack of SQLite's
    millisecond roll (csrc/rollup.cuh: a record can land in the bucket of the next day)."""
    day = 86400 * 10**6
    if period == "hour":
        return (bucket - 24) * 3600 * 10**6, (bucket + 1) * 3600 * 10**6
    if period == "day":
        return (bucket - 1) * day, (bucket + 1) * day
    if period == "month":
        y, m = divmod(bucket, 12)
        first = to_us(datetime(y, m + 1, 1))
        nxt = to_us(datetime(y + 1, 1, 1) if m == 11 else datetime(y, m + 2, 1))
        return first - day, nxt
    y, w = divmod(bucket, 64)                 # %W = (day of year + 7 - weekday) / 7: day of year in [7w - 7, 7w + 5]
    jan1 = to_us(datetime(y, 1, 1))
    return jan1 + (7 * w - 8) * day, jan1 + (7 * w + 6) * day


def stats_window(period: str, now: datetime):
    """stats.py:46-55: (start_date, end_date) the stats endpoint asks for."""
    delta = {"hour": timedelta(hours=24), "day": timedelta(weeks=2), "week": timedelta(weeks=15), "month": timedelta(days=365)}[period]
    return now - delta, now


class UsageTable:
    """Device-resident usage records + GPU rollup.  `engine` is an llmapigateway_b200.Engine."""

    COLS = ("ts_us", "model_rank", "prompt_tokens", "completion_tokens", "total_tokens", "reasoning_tokens", "cached_tokens", "cost")
    DTYPES = (np.int64, np.int32, np.int32, np.int32, np.int32, np.int32, np.int32, np.float64)

    def __init__(self, engine):
        self.eng = engine
        self._lib = _native.load()
        self._host = {c: np.zeros(0, dtype=d) for c, d in zip(self.COLS, self.DTYPES)}
        self._models: list[str | None] = []      # per record, until encoded
        self._providers: list[str | None] = []   # per record (listing only; the rollup does not group by provider)
        self._dev = None                          # (n, {col: device ptr}, names)
        self._pending_rows: list[tuple] = []
        self.rejected = 0                         # records insert_usage refused (see there)

    # -- ingest ------------------------------------------------------------------------------------
    def insert_usage(self, tokens_usage: dict, timestamp: datetime | None = None):
        """One record, same dict shape as the reference's insert_usage (:136-143).  Like the reference (:155-159) this never
        raises: a value SQLite would have stored as NULL (JSON null), as REAL/TEXT (a non-integer where a count belongs), or
        that no INTEGER column of the device table can hold (|v| >= 2^31) makes the record unusable for the integer rollup
        and the row is REJECTED (counted in `rejected`), never half-inserted."""
        ts = to_us(timestamp or datetime.now())
        g = tokens_usage.get
        try:
            counts = []
            for k in ("prompt_tokens", "completion_tokens", "total_tokens", "reasoning_tokens", "cached_tokens"):
                v = g(k, 0)
                if v is None:
                    v = 0                                              # SUM() skips NULL
                if isinstance(v, bool) or not isinstance(v, int):
                    if isinstance(v, float) and v.is_integer():
                        v = int(v)
                    else:
                        raise ValueError(k)
                if not -(1 << 31) <= v < (1 << 31):
                    raise OverflowError(k)
                counts.append(v)
            cost = g("cost", 0.0)
            cost = 0.0 if cost is None else float(cost)
            model, provider = g("model"), g("provider")
            if model is not None and not isinstance(model, str):
                model = str(model)
        except Exception:
            self.rejected += 1
            return False
        self._pending_rows.append((ts, model, *counts, cost, provider))
        self._dev = None
        return True

    def load_columns(self, ts_us, models, prompt, completion, total, reasoning, cached, cost, names=None):
        """Bulk ingest of columns (models: sequence of str|None).  `names`: the model dictionary to encode against when several
        tables (one per GPU) are merged -- every rank must rank the models identically (sorted by UTF-8 bytes, NULL first)."""
        self._fixed_names = sorted(set(names), key=lambda s: s.encode("utf-8")) if names is not None else None
        self._host = {"ts_us": np.ascontiguousarray(ts_us, np.int64), "model_rank": None,
                      "prompt_tokens": np.ascontiguousarray(prompt, np.int32), "completion_tokens": np.ascontiguousarray(completion, np.int32),
                      "total_tokens": np.ascontiguousarray(total, np.int32), "reasoning_tokens": np.ascontiguousarray(reasoning, np.int32),
                      "cached_tokens": np.ascontiguousarray(cached, np.int32), "cost": np.ascontiguousarray(cost, np.float64)}
        self._models = list(models)
        self._providers = [None] * len(self._models)
        self._pending_rows = []
        self._dev = None

    def _materialise(self):
        if self._pending_rows:
            cols = list(zip(*self._pending_rows))
            h = self._host
            fresh = {"ts_us": np.concatenate([h["ts_us"], np.array(cols[0], np.int64)]), "model_rank": None}     # built completely
            for k, name in enumerate(self.COLS[2:7]):                                                           # before anything
                fresh[name] = np.concatenate([h[name], np.array(cols[2 + k], np.int32)])                        # is replaced
            fresh["cost"] = np.concatenate([h["cost"], np.array(cols[7], np.float64)])
            self._host = fresh
            self._models = list(self._models) + list(cols[1])
            self._providers = list(self._providers) + list(cols[8])
            self._pending_rows = []
        names = getattr(self, "_fixed_names", None) or sorted({m for m in self._models if m is not None}, key=lambda s: s.encode("utf-8"))
        rank = {m: i + 1 for i, m in enumerate(names)}
        rank[None] = 0
        self._host["model_rank"] = np.fromiter((rank[m] for m in self._models), dtype=np.int32, count=len(self._models))
        self._names = [None] + names

    def _free_device(self):
        """Give the device copy of the columns back (an insert makes it stale; without this every re-upload would leak the last one)."""
        ptrs, self._dev_ptrs = getattr(self, "_dev_ptrs", None), None
        self._dev = None
        if ptrs and getattr(self.eng, "_h", None):
            for p in ptrs.values():
                self._lib.lgw_device_free(self.eng._h, p)

    def close(self):
        self._free_device()

    def _upload(self):
        if self._dev is not None:
            return
        self._free_device()
        self._materialise()
        n = int(self._host["ts_us"].size)
        ptrs = {}
        self._dev_ptrs = ptrs                     # (registered before the first allocation: a failed upload frees what it got)
        for c in self.COLS:
            a = self._host[c]
            p = C.c_void_p()
            self.eng._ck(self._lib.lgw_device_alloc(self.eng._h, max(a.nbytes, 8), C.byref(p)), "device_alloc")
            self.eng._ck(self._lib.lgw_device_upload(self.eng._h, p, a.ctypes.data_as(C.c_void_p), a.nbytes), "device_upload")
            ptrs[c] = p
        self._dev = (n, ptrs)

    def __len__(self):
        return int(self._host["ts_us"].size) + len(self._pending_rows)

    # -- rollup ---------------------------------------------------------------------------------------
    def geometry(self, period: str, start: datetime | None, end: datetime | None):
        self._materialise() if self._host.get("model_rank") is None or self._pending_rows else None
        ts = self._host["ts_us"]
        p = PERIODS[period]
        lo = int(ts.min()) if ts.size else 0
        hi = int(ts.max()) if ts.size else 0
        if start is not None:
            lo = max(lo, to_us(start))
        if end is not None:
            hi = min(hi, to_us(end))
        if hi < lo:
            hi = lo
        b0 = int(self._lib.lgw_rollup_bucket_of(lo, p)); b1 = int(self._lib.lgw_rollup_bucket_of(hi, p))
        slack = 25 if period == "hour" else 1            # SQLite's millisecond rounding can push a record one day ahead
        return b0, b1 - b0 + 1 + slack, len(self._names)

    def accumulate(self, period: str, start, end, bucket0: int, n_buckets: int, n_models: int, d_table, d_inexact, d_oob):
        """Add this table's records into a caller-owned dense device table (multi-GPU merge)."""
        self._upload()
        n, ptr = self._dev
        self.eng._ck(self._lib.lgw_usage_rollup_accum(
            self.eng._h, ptr["ts_us"], ptr["model_rank"], ptr["prompt_tokens"], ptr["completion_tokens"], ptr["total_tokens"],
            ptr["reasoning_tokens"], ptr["cached_tokens"], ptr["cost"], n, PERIODS[period],
            int(start is not None), to_us(start) if start is not None else 0, int(end is not None), to_us(end) if end is not None else 0,
            bucket0, n_buckets, n_models, d_table, d_inexact, d_oob), "usage_rollup_accum")

    def emit(self, bucket0: int, n_buckets: int, n_models: int, d_table, d_inexact, pinned: bool = False) -> np.ndarray:
        """Rows of a dense device table (this GPU's, or the all-reduced sum of every GPU's), time_period DESC, model ASC.
        pinned=True: the rows land in a page-locked buffer owned by this table (grown on demand, REUSED by the next pinned emit:
        consume or copy them first) -- a full `hour` table over 400 days is 45 MB of rows, 10 ms into pageable memory, < 1 ms pinned."""
        groups = n_buckets * n_models
        if pinned:
            need = groups * ROW_DTYPE.itemsize
            buf = getattr(self, "_pinned_rows", None)
            if buf is None or buf.size < need:
                buf = self._pinned_rows = self.eng.alloc_pinned(need)
            rows = buf[:need].view(ROW_DTYPE)
        else:
            rows = np.zeros(groups, dtype=ROW_DTYPE)
        n_rows = C.c_uint64(0)
        self.eng._ck(self._lib.lgw_usage_rollup_emit(self.eng._h, d_table, d_inexact, bucket0, n_buckets, n_models,
                                                     rows.ctypes.data_as(C.c_void_p), groups, C.byref(n_rows)), "usage_rollup_emit")
        return rows[:n_rows.value]

    def _row_dict(self, period: str, r, cost) -> dict:
        return {"time_period": period_label(period, int(r["bucket"])), "model": self._names[int(r["model_rank"])],
                "prompt_tokens": int(r["prompt_tokens"]), "completion_tokens": int(r["completion_tokens"]),
                "total_tokens": int(r["total_tokens"]), "reasoning_tokens": int(r["reasoning_tokens"]),
                "cached_tokens": int(r["cached_tokens"]), "cost": cost, "count": int(r["count"])}

    def rows_to_dicts(self, period: str, rows) -> list[dict]:
        """Dicts of emitted rows (e.g. of a table all-reduced over ranks).  A row flagged `inexact` is refused with ValueError:
        its cost is not the sum of its records, and the records that would give the right answer may live on other ranks."""
        bad = np.flatnonzero(rows["inexact"])
        if bad.size:
            r = rows[bad[0]]
            raise ValueError("%d rollup row(s) hold a cost the fixed-point sum cannot represent (first: %s, model %r)"
                             % (bad.size, period_label(period, int(r["bucket"])), self._names[int(r["model_rank"])]))
        return [self._row_dict(period, r, float(r["cost"])) for r in rows]

    def rollup_rows(self, period: str, start: datetime | None = None, end: datetime | None = None) -> np.ndarray:
        """Rows (ROW_DTYPE) ordered time_period DESC, model ASC."""
        self._upload()
        b0, nb, nm = self.geometry(period, start, end)
        groups = nb * nm
        lib, h = self._lib, self.eng._h
        tab, inx, oob = C.c_void_p(), C.c_void_p(), C.c_void_p()
        for p, nbytes in ((tab, groups * ROLLUP_CELLS * 8), (inx, groups * 4), (oob, 8)):
            self.eng._ck(lib.lgw_device_alloc(h, nbytes, C.byref(p)), "device_alloc")
            self.eng._ck(lib.lgw_device_zero(h, p, nbytes), "device_zero")
        try:
            self.accumulate(period, start, end, b0, nb, nm, tab, inx, oob)
            rows = np.zeros(groups, dtype=ROW_DTYPE)
            n_rows = C.c_uint64(0)
            self.eng._ck(lib.lgw_usage_rollup_emit(h, tab, inx, b0, nb, nm, rows.ctypes.data_as(C.c_void_p), groups, C.byref(n_rows)), "usage_rollup_emit")
            lost = np.zeros(1, np.uint32)
            self.eng._ck(lib.lgw_device_download(h, lost.ctypes.data_as(C.c_void_p), oob, 4), "device_download")
            # records outside the table are exactly those the window excludes only when no window was given; never expected
            assert int(lost[0]) == 0 or start is not None or end is not None, "records fell outside the rollup table"
            return rows[:n_rows.value]
        finally:
            for p in (tab, inx, oob):
                lib.lgw_device_free(h, p)

    def get_aggregated_usage(self, period: str, start_date: datetime | None = None, end_date: datetime | None = None) -> list[dict]:
        """Same result shape and order as TokensUsageDB.get_aggregated_usage (:289-291); [] for a bad period (:296-298)."""
        if period not in PERIODS:
            return []
        if len(self) == 0:
            return []
        rows = self.rollup_rows(period, start_date, end_date)
        cost = rows["cost"].tolist()
        for j in np.flatnonzero(rows["inexact"]).tolist():
            cost[j] = sqlite_sum(self._group_costs(period, start_date, end_date, int(rows["bucket"][j]), int(rows["model_rank"][j])))
        return [self._row_dict(period, r, c) for r, c in zip(rows, cost)]

    def _group_costs(self, period: str, start: datetime | None, end: datetime | None, bucket: int, model_rank: int) -> list[float]:
        """Costs of one group's records from the host columns, in insertion order (SQLite's scan order within a group).
        numpy narrows the records to the model and a time span around the bucket; bucket_of() decides the rest."""
        h = self._host
        ts = h["ts_us"]
        lo, hi = _bucket_span_us(period, bucket)
        sel = (h["model_rank"] == model_rank) & (ts >= lo) & (ts < hi)
        if start is not None:
            sel &= ts >= to_us(start)
        if end is not None:
            sel &= ts <= to_us(end)
        p = PERIODS[period]
        keep = [i for i in np.flatnonzero(sel).tolist() if self._lib.lgw_rollup_bucket_of(int(ts[i]), p) == bucket]
        return h["cost"][keep].tolist()

    # -- record listing: /v1/api/usage-records (stats.py:69-87) ---------------------------------------------
    def get_total_records_count(self) -> int:
        """tokens_usage_db.py:200-220"""
        return len(self)

    def get_latest_usage_records(self, limit: int = 25, offset: int = 0) -> list[dict]:
        """tokens_usage_db.py:69-117: newest first (`ORDER BY timestamp DESC LIMIT ? OFFSET ?`), same keys.  Host
        side: a page of 25 rows out of the host copy of the columns is not GPU work.  Records with equal
        timestamps come in insertion order (SQLite leaves their order unspecified)."""
        self._materialise()
        h = self._host
        n = int(h["ts_us"].size)
        if limit < 0:
            limit = n                                           # SQLite: a negative LIMIT means no limit
        order = np.argsort(-h["ts_us"], kind="stable")[max(offset, 0):max(offset, 0) + limit]
        out = []
        for i in order:
            i = int(i)
            out.append({"id": i + 1, "timestamp": (_EPOCH + timedelta(microseconds=int(h["ts_us"][i]))).isoformat(),
                        "prompt_tokens": int(h["prompt_tokens"][i]), "completion_tokens": int(h["completion_tokens"][i]),
                        "total_tokens": int(h["total_tokens"][i]), "reasoning_tokens": int(h["reasoning_tokens"][i]),
                        "cached_tokens": int(h["cached_tokens"][i]), "cost": float(h["cost"][i]),
                        "model": self._models[i], "provider": self._providers[i]})
        return out

    def last_ms(self):
        ms = (C.c_float * 2)()
        self.eng._ck(self._lib.lgw_rollup_last_ms(self.eng._h, C.byref(ms)), "rollup_last_ms")
        return {"accum": ms[0], "emit": ms[1]}


def synth_usage_columns(n: int, seed: int = 5, end: datetime = datetime(2026, 9, 21, 6, 57, 17, 47518), days: int = 400, n_models: int = 64):
    """SURVEY 8(d) C5: timestamps uniform over a 400-day window, 64 model names (Zipf s=1.1) + 1% NULL,
    token ints < 2^17, cost = k x 1e-6."""
    rng = np.random.default_rng([seed, n])
    ts = to_us(end) - rng.integers(0, days * 86400 * 10**6, n, dtype=np.int64)
    w = 1.0 / np.arange(1, n_models + 1) ** 1.1
    mid = rng.choice(n_models, size=n, p=w / w.sum())
    names = np.array(["provider-%02d/model-%02d" % (i % 7, i) for i in range(n_models)], dtype=object)
    models = names[mid]
    models[rng.random(n) < 0.01] = None
    tok = [rng.integers(0, 2**17, n, dtype=np.int32) for _ in range(5)]
    cost = rng.integers(0, 10**6, n).astype(np.float64) * 1e-6
    return ts, models, tok, cost
