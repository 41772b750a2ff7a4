"""GPU: the rollup's cost sums through the C ABI on hostile costs -- NaN, infinities, values the 128-bit fixed point cannot
hold, runs of values with bits below 2^-80, signed zeros and a group at the per-record bound -- on both accumulation paths.
Unflagged rows must be math.fsum of their group bit for bit; a group is flagged exactly when it holds a record the fixed
point cannot represent; get_aggregated_usage answers flagged groups exactly like SQLite."""
import math
from datetime import datetime, timedelta

import numpy as np
import pytest

from llmapigateway_b200.usage import _EPOCH, PERIODS, UsageTable, stats_window, synth_usage_columns, to_us
from oracle import rollup_oracle as ro
from test_rollup_cost_cpu import TOP, representable, same
from test_rollup_gpu import _iso, _ulps

pytestmark = pytest.mark.gpu
NOW = datetime(2026, 9, 21, 6, 57, 17, 47518)

# groups of their own (one model each, all records in one hour inside every stats window)
HOSTILE_GROUPS = {
    "hostile/nan-only": [math.nan] * 3,
    "hostile/inf-and-one": [math.inf, 1.0],
    "hostile/inf-minus-inf": [math.inf, -math.inf],
    "hostile/1e308-twice": [1e308, 1e308],
    "hostile/1e15": [1e15],
    "hostile/wrap": [2.0 ** 46, 2.0 ** 46],
    "hostile/1e-12-run": [1e-12] * 40,
    "hostile/minus-zero": [-0.0] * 3,
    "hostile/at-bound": [TOP] * 9 + [-2.0 ** -80],
    "hostile/over-bound": [2.0 ** 15, 1.0],
}
# scattered over ordinary records (their groups also hold ordinary costs)
SCATTERED = [math.nan, math.inf, -math.inf, 1e-12, 1e-300, 5e-324, -0.0, 1e14, 2.0 ** 46, TOP, -TOP, 2.0 ** -80]


@pytest.fixture(scope="module")
def engine():
    import llmapigateway_b200 as L
    e = L.Engine(max_streams=64, max_step_chunks=1024, max_step_bytes=1 << 20)
    yield e
    e._lib.lgw_rollup_set_path(e._h, 0)
    e.close_engine()


@pytest.fixture(scope="module")
def data():
    n = 200_000
    ts, models, tok, cost = synth_usage_columns(n, seed=17, end=NOW)
    models = list(models)
    rng = np.random.default_rng(17)
    recent = np.flatnonzero(ts >= to_us(NOW - timedelta(days=14)))
    for k, i in enumerate(rng.choice(recent, 240, replace=False).tolist()):
        cost[i] = SCATTERED[k % len(SCATTERED)]
    for i in rng.choice(n, 60, replace=False).tolist():
        cost[i] = SCATTERED[i % len(SCATTERED)]
    hour = to_us(NOW - timedelta(hours=3))
    extra = [(hour + 1000 * k, m, c) for m, cs in HOSTILE_GROUPS.items() for k, c in enumerate(cs)]
    ts = np.concatenate([ts, np.array([x[0] for x in extra], np.int64)])
    models += [x[1] for x in extra]
    tok = [np.concatenate([t, np.full(len(extra), 7, np.int32)]) for t in tok]
    cost = np.concatenate([cost, np.array([x[2] for x in extra])])
    conn = ro.make_db([(_iso(ts[i]), int(tok[0][i]), int(tok[1][i]), int(tok[2][i]), int(tok[3][i]), int(tok[4][i]), float(cost[i]), models[i], "P")
                       for i in range(ts.size)])
    rep = np.array([representable(c) for c in cost.tolist()])
    return ts, models, tok, cost, conn, rep


def _windows(period):
    return ((None, None), stats_window(period, NOW))


def _groups(bucket, rank, n_models, ts, s, e):
    """{bucket * n_models + rank: record indices in insertion order} of the records inside the window"""
    sel = np.ones(ts.size, bool)
    if s is not None:
        sel &= ts >= to_us(s)
    if e is not None:
        sel &= ts <= to_us(e)
    idx = np.flatnonzero(sel)
    key = bucket[idx] * n_models + rank[idx]
    order = np.argsort(key, kind="stable")
    key, idx = key[order], idx[order]
    starts = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
    ends = np.r_[starts[1:], key.size]
    return {int(key[a]): idx[a:b] for a, b in zip(starts.tolist(), ends.tolist())}


def test_cost_sums_on_both_paths(engine, data):
    ts, models, tok, cost, conn, rep = data
    t = UsageTable(engine)
    t.load_columns(ts, models, *tok, cost)
    t._materialise()
    rank = t._host["model_rank"]
    nm = len(t._names)
    n_flagged = 0
    for period, p in PERIODS.items():
        bucket = np.array([t._lib.lgw_rollup_bucket_of(x, p) for x in ts.tolist()], np.int64)
        for s, e in _windows(period):
            engine._lib.lgw_rollup_set_path(engine._h, 0)
            a = t.rollup_rows(period, s, e)
            engine._lib.lgw_rollup_set_path(engine._h, 1)
            b = t.rollup_rows(period, s, e)
            engine._lib.lgw_rollup_set_path(engine._h, 0)
            assert len(a) == len(b) > 0 and a.tobytes() == b.tobytes(), (period, s)
            groups = _groups(bucket, rank, nm, ts, s, e)
            keys = (a["bucket"] * nm + a["model_rank"]).tolist()
            assert sorted(keys) == sorted(groups)
            for r, k in zip(a, keys):
                idx = groups[k]
                assert bool(r["inexact"]) == (not rep[idx].all()), (period, s, k, cost[idx])
                if r["inexact"]:
                    n_flagged += 1
                else:
                    assert float(r["cost"]).hex() == math.fsum(cost[idx].tolist()).hex(), (period, s, k)
                assert int(r["count"]) == idx.size
            got, want = t.get_aggregated_usage(period, s, e), ro.aggregated_usage(conn, period, s, e)
            assert len(got) == len(want) == len(a)
            for g, w, r in zip(got, want, a):
                for f in ("time_period", "model", "prompt_tokens", "completion_tokens", "total_tokens", "reasoning_tokens", "cached_tokens", "count"):
                    assert g[f] == w[f], (f, g, w)
                if r["inexact"]:
                    assert same(g["cost"], w["cost"]), (period, s, g, w)
                else:
                    assert _ulps(g["cost"], w["cost"]) <= 4, (g, w)
            for m, cs in HOSTILE_GROUPS.items():                       # the named groups are all in every window
                row = [g for g in got if g["model"] == m]
                assert len(row) == 1 and row[0]["count"] == len(cs), (m, row)
    assert n_flagged > 8 * 8                  # 8 flagged named groups in each of 8 rollups, and the groups of scattered costs


def test_insert_usage_gives_the_same_answer(engine, data):
    ts, models, tok, cost, conn, rep = data
    bulk = UsageTable(engine)
    bulk.load_columns(ts, models, *tok, cost)
    one = UsageTable(engine)
    names = ("prompt_tokens", "completion_tokens", "total_tokens", "reasoning_tokens", "cached_tokens")
    for i in range(ts.size):
        d = {f: int(tok[k][i]) for k, f in enumerate(names)}
        d["cost"] = float(cost[i])
        d["model"] = models[i]
        assert one.insert_usage(d, timestamp=_EPOCH + timedelta(microseconds=int(ts[i])))
    for period in PERIODS:
        for s, e in _windows(period):
            got, want = one.get_aggregated_usage(period, s, e), bulk.get_aggregated_usage(period, s, e)
            assert len(got) == len(want) > 0
            for g, w in zip(got, want):
                assert {k: v for k, v in g.items() if k != "cost"} == {k: v for k, v in w.items() if k != "cost"}
                assert same(g["cost"], w["cost"]), (g, w)
    bulk.close(); one.close()
