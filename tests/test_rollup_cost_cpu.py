"""CPU: the rollup's exact cost arithmetic (csrc/rollup.cuh cost_to_limbs / limbs_to_cost, host build of the same code the
kernels run) against exact references -- fractions.Fraction for representability and rounding, math.fsum (the correctly
rounded exact sum) for sums -- and the host answer for flagged groups (usage.sqlite_sum over usage.UsageTable._group_costs)
against SQLite's own SUM(cost) through the reference's statement."""
import math
import random
import sqlite3
from datetime import datetime, timedelta
from fractions import Fraction

import numpy as np
import pytest

import host_machine as hm
from llmapigateway_b200.usage import PERIODS, UsageTable, _bucket_span_us, period_label, sqlite_sum, synth_usage_columns, to_us
from oracle import rollup_oracle as ro

BOUND = 2 ** 15                     # |cost| of one exactly summed record (rollup.cuh cost_to_limbs)
MAX_COUNT = 2 ** 32 - 1             # records of one group the 128-bit sum is guaranteed to hold
TOP = math.nextafter(2.0 ** 15, 0)  # the largest representable magnitude
NOW = datetime(2026, 9, 21, 6, 57, 17, 47518)


def representable(c: float) -> bool:
    return math.isfinite(c) and abs(Fraction(c)) < BOUND and (Fraction(c) * 2 ** 80).denominator == 1


def cells_of(x: Fraction, count: int = 1):
    """the four cells a group of `count` records of value x holds: count x the two's complement limbs of x * 2^80"""
    v = int(x * 2 ** 80) % 2 ** 128
    return [count * ((v >> (32 * k)) & 0xFFFFFFFF) for k in range(4)]


def same(a, b) -> bool:
    """equal floats with equal signs of zero, or both None"""
    return (a is None and b is None) or (a is not None and b is not None and a.hex() == b.hex())


# ---- cost_to_limbs: which doubles are exact ---------------------------------------------------------------------------------

EDGES = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 2.0 ** -80, -2.0 ** -80, 2.0 ** -81, 3 * 2.0 ** -81, 2.0 ** -79 + 2.0 ** -80,
         2.0 ** -28 + 2.0 ** -80, 2.0 ** -27 + 2.0 ** -79, 2.0 ** -27 + 2.0 ** -80 * 3, 1.0, 1 + 2.0 ** -52, 0.1, 1e-6, 1e-7, 1e-8, 1e-12, 1e-25,
         TOP, -TOP, 2.0 ** 15, -2.0 ** 15, math.nextafter(2.0 ** 15, math.inf), 2.0 ** 14, 2.0 ** 46, 2.0 ** 47, 1e14, 1e15, 1e300, 1.7976931348623157e308,
         math.inf, -math.inf, math.nan, -math.nan]


def test_cost_to_limbs_is_exact_exactly_when_the_value_is_representable():
    rng = random.Random(7)
    values = list(EDGES)
    for e in range(2048):                                   # every biased exponent, full and trimmed mantissas, both signs
        for _ in range(6):
            z = rng.choice((0, rng.randrange(53), 52))
            m = rng.getrandbits(52) >> z << z
            bits = (rng.getrandbits(1) << 63) | (e << 52) | m
            values.append(float(np.array(bits, np.uint64).view(np.float64)))
    for _ in range(20000):                                  # the exponents where the answer turns: around 2^-80 and 2^15
        lead = rng.randrange(-90, 20)
        p = rng.randrange(1, 54)
        values.append(rng.choice((1, -1)) * math.ldexp(rng.getrandbits(p) | (1 << (p - 1)), lead - p + 1))
    n_exact = 0
    for c in values:
        ok, limbs = hm.cost_to_limbs(c)
        assert ok == representable(c), (c, c.hex(), ok)
        if ok:
            n_exact += 1
            assert list(limbs) == cells_of(Fraction(c)), (c, limbs)
    assert 5000 < n_exact < len(values) - 5000


# ---- sums: bit for bit the correctly rounded exact sum ------------------------------------------------------------------

def _costs(rng, n):
    """n representable costs: leading bits in a random window of [2^-80, 2^15), a random number of significant bits, both
    signs; a third of the lists cancel (half of them is the negated other half, shuffled in)"""
    lo = int(rng.integers(-80, 15))
    hi = int(rng.integers(lo, 15)) + 1
    lead = rng.integers(lo, hi, n)
    prec = rng.integers(1, np.minimum(53, lead + 81) + 1)
    m = np.floor(np.ldexp(1.0 + rng.random(n), prec - 1))
    c = np.ldexp(m, lead - prec + 1) * rng.choice((-1.0, 1.0), n)
    if n >= 2 and rng.random() < 1 / 3:
        k = n // 2
        c[k:2 * k] = -c[:k][rng.permutation(k)]
        rng.shuffle(c)
    return c


def test_fixed_point_sums_equal_fsum_bit_for_bit():
    rng = np.random.default_rng(20261017)
    lens = np.exp(rng.uniform(0, math.log(5000), 100_000)).astype(np.int64).clip(1, 5000)
    lens[:1000] = 1
    lens[1000:2000] = 5000
    for n in lens.tolist():
        c = _costs(rng, n)
        ok, cells = hm.sum_costs(c)
        want = math.fsum(c.tolist())
        assert ok, c
        got = hm.limbs_to_cost(cells)
        assert got.hex() == want.hex(), (n, got, want)


@pytest.mark.parametrize("costs, want", [
    ([2.0 ** 14, 2.0 ** -39], 2.0 ** 14),                                         # a tie: to even (down)
    ([2.0 ** 14 + 2.0 ** -38, 2.0 ** -39], 2.0 ** 14 + 2.0 ** -37),               # a tie: to even (up)
    ([2.0 ** 14, 2.0 ** -39, 2.0 ** -80], 2.0 ** 14 + 2.0 ** -38),                # one LSB of the fixed point breaks the tie (sticky)
    ([2.0 ** 14, 2.0 ** -39, -2.0 ** -80], 2.0 ** 14),
    ([2.0 ** 14 + 2.0 ** -38, 2.0 ** -39, -2.0 ** -80], 2.0 ** 14 + 2.0 ** -38),
    ([-2.0 ** 14, -2.0 ** -39], -2.0 ** 14),
    ([-2.0 ** 14 - 2.0 ** -38, -2.0 ** -39], -2.0 ** 14 - 2.0 ** -37),
    ([-2.0 ** 14, -2.0 ** -39, -2.0 ** -80], -2.0 ** 14 - 2.0 ** -38),
    ([TOP, 2.0 ** -80], TOP),
    ([TOP, TOP], 2 * TOP),
    ([1.0, 2.0 ** -53], 1.0), ([1.0, 2.0 ** -53, 2.0 ** -80], 1 + 2.0 ** -52),
    ([TOP, -TOP], 0.0), ([-0.0], 0.0), ([-0.0, -0.0], 0.0), ([2.0 ** -80, -2.0 ** -80], 0.0),
    ([2.0 ** -80] * 3, 3 * 2.0 ** -80), ([-2.0 ** -80], -2.0 ** -80),
])
def test_ties_and_sticky_bits(costs, want):
    ok, cells = hm.sum_costs(costs)
    assert ok
    got = hm.limbs_to_cost(cells)
    assert got.hex() == want.hex() == math.fsum(costs).hex(), (got, want)


@pytest.mark.parametrize("costs", [[2.0 ** 46, 2.0 ** 46], [1e14, 1e14], [-2.0 ** 46, -2.0 ** 46, -2.0 ** 46], [1e15], [1e300], [2.0 ** 15],
                                   [math.inf, 1.0], [math.nan], [1e-12, 2e-12], [1e-25] * 3])
def test_costs_the_fixed_point_cannot_hold_are_flagged(costs):
    """Each record below the old bound of 2^47, [2^46, 2^46] wrapped the 128-bit cell to -2^47 without a flag."""
    ok, cells = hm.sum_costs(costs)
    assert not ok, (costs, hm.limbs_to_cost(cells))


@pytest.mark.parametrize("x", [Fraction(2 ** 40) + Fraction(1, 2 ** 13), Fraction(2 ** 40 + Fraction(1, 2 ** 12)) + Fraction(1, 2 ** 13),
                               Fraction(2 ** 40) + Fraction(1, 2 ** 13) + Fraction(1, 2 ** 80), Fraction(2 ** 126 + 2 ** 73 - 1, 2 ** 80),
                               Fraction(2 ** 126 + 2 ** 73, 2 ** 80), Fraction(2 ** 126 + 2 ** 73 + 1, 2 ** 80), Fraction(2 ** 126 + 3 * 2 ** 73, 2 ** 80)])
def test_limbs_to_cost_rounds_half_to_even_far_from_one_record(x):
    for v in (x, -x):
        assert hm.limbs_to_cost(cells_of(v)) == float(v), v


def test_limbs_to_cost_at_the_bound():
    """The largest sums an unflagged group can hold: 2^32 - 1 records of the largest magnitude, and random counts of random
    representable records, both signs; the cells are what the kernels' 64-bit additions of the limbs leave."""
    rng = np.random.default_rng(3)
    cases = [(TOP, MAX_COUNT), (-TOP, MAX_COUNT), (2.0 ** -80, MAX_COUNT), (-2.0 ** -80, MAX_COUNT), (TOP, 1), (1.0, MAX_COUNT)]
    cases += [(float(c), int(k)) for c, k in zip(_costs(rng, 4000), rng.integers(1, MAX_COUNT + 1, 4000))]
    for c, k in cases:
        ok, limbs = hm.cost_to_limbs(c)
        assert ok, c
        cells = [k * l for l in limbs]
        assert all(x < 2 ** 64 for x in cells)              # no 64-bit cell wraps
        assert hm.limbs_to_cost(cells) == float(Fraction(c) * k), (c, k)
    rnd = random.Random(5)
    for _ in range(20000):                                  # any 128-bit value the cells can carry
        v = Fraction(rnd.getrandbits(rnd.randrange(1, 128)) * rnd.choice((1, -1)), 2 ** 80)
        assert hm.limbs_to_cost(cells_of(v)) == float(v), v


# ---- flagged groups: SQLite's SUM(REAL), restated ---------------------------------------------------------------------

needs_ksum = pytest.mark.skipif(sqlite3.sqlite_version_info < (3, 43), reason="SQLite before 3.43 sums REAL without compensation")

HOSTILE = [1e308, -1e308, math.inf, -math.inf, math.nan, 1e16, -1e16, 1e-300, 5e-324, 1e14, -0.0, 1e-12, -1e-12, 2.0 ** 46, 2.0 ** 15]


def _hostile_costs(rng: random.Random, n: int) -> list[float]:
    share = rng.choice((0.0, 0.2, 0.6, 1.0))
    return [rng.choice(HOSTILE) if rng.random() < share else rng.choice((1, -1)) * 10.0 ** rng.uniform(-20, 20) for _ in range(n)]


@needs_ksum
def test_sqlite_sum_restatement_matches_sqlite():
    rng = random.Random(11)
    days, models = 100, ["m%03d" % i for i in range(200)]           # 20 000 groups of the `day` rollup
    rows = []
    for d in range(days):
        for m in models:
            n = rng.choice((1, 1, 2, 3, 5, 8, rng.randrange(1, 60)))
            for c in _hostile_costs(rng, n):
                ts = datetime(2026, 1, 1) + timedelta(days=d, seconds=rng.randrange(23 * 3600))
                rows.append((ts.isoformat(), 1, 2, 3, 0, 0, c, m, "P"))
    rng.shuffle(rows)                                                # SQLite scans a group in insertion order
    groups = {}
    for r in rows:
        groups.setdefault((r[0][:10], r[7]), []).append(r[6])
    got = ro.aggregated_usage(ro.make_db(rows), "day")
    assert len(got) == len(groups) == days * len(models)
    n_none = 0
    for g in got:
        want = sqlite_sum(groups[(g["time_period"], g["model"])])
        assert same(g["cost"], want), (g, groups[(g["time_period"], g["model"])])
        n_none += g["cost"] is None
    assert n_none > 100


@pytest.mark.parametrize("costs, want", [([math.nan], None), ([math.nan, math.nan], None), ([math.inf, 1.0], math.inf), ([math.inf, -math.inf], None),
                                         ([1e308, 1e308], None),             # the sum overflows, its error term is -inf: inf + -inf
                                         ([2.0 ** 46, 2.0 ** 46], 2.0 ** 47), ([1e14, 1e14], 2e14),
                                         ([1e-12, 2e-12], 3e-12), ([1e-25] * 3, 3.0000000000000002e-25), ([-0.0], 0.0), ([], None)])
def test_sqlite_sum_on_the_rows_of_the_issue(costs, want):
    assert same(sqlite_sum(costs), want)


def _table(n, seed, days):
    """a CPU-side UsageTable (no engine: only the host columns and bucket_of) with hostile costs and SQLite's roll quirks"""
    ts, models, tok, cost = synth_usage_columns(n, seed=seed, end=NOW, days=days)
    rng = random.Random(seed)
    for i in range(0, n, 7):
        cost[i] = rng.choice(HOSTILE)
    quirks = [datetime(2025, 12, 31, 23, 59, 59, 999999), datetime(2026, 8, 31, 23, 59, 59, 999600), datetime(2026, 6, 30, 23, 59, 59, 999500),
              datetime(2026, 8, 30, 23, 59, 59, 999999), datetime(2026, 9, 6, 23, 59, 59, 999999), datetime(2026, 9, 7, 0, 0, 0)]
    for k, q in enumerate(quirks * 5):
        ts[n - 1 - k] = to_us(q)
    t = UsageTable(engine=None)
    t.load_columns(ts, models, *tok, cost)
    t._materialise()
    return t, ts, models, tok, cost


def test_bucket_span_holds_every_timestamp_of_its_bucket():
    lib = UsageTable(engine=None)._lib
    rng = random.Random(9)
    samples = [datetime(1999, 12, 31, 23, 59, 59, 999999), datetime(2026, 1, 31, 23, 59, 59, 999999), datetime(2024, 2, 29, 23, 59, 59, 999999),
               datetime(2027, 1, 3, 23, 59, 59, 999999), datetime(2027, 1, 4), datetime(2026, 12, 31, 23, 59, 59, 999500)]
    samples += [datetime(1990, 1, 1) + timedelta(seconds=rng.randrange(60 * 365 * 86400), microseconds=rng.choice((0, 999999, rng.randrange(10**6))))
                for _ in range(20000)]
    for dt in samples:
        us = to_us(dt)
        for period, p in PERIODS.items():
            lo, hi = _bucket_span_us(period, int(lib.lgw_rollup_bucket_of(us, p)))
            assert lo <= us < hi, (dt, period)


@needs_ksum
def test_host_answer_for_flagged_groups_matches_sqlite():
    """What get_aggregated_usage puts in a flagged row -- sqlite_sum over _group_costs -- computed for EVERY group of every period
    and window, against SQLite's statement over the same rows; and _group_costs against a plain scan of all records."""
    n = 6000
    t, ts, models, tok, cost = _table(n, seed=13, days=40)
    conn = ro.make_db([((datetime(1970, 1, 1) + timedelta(microseconds=int(ts[i]))).isoformat(), int(tok[0][i]), int(tok[1][i]), int(tok[2][i]),
                        int(tok[3][i]), int(tok[4][i]), float(cost[i]), models[i], "P") for i in range(n)])
    rank = t._host["model_rank"]
    for period, p in PERIODS.items():
        bucket = np.array([t._lib.lgw_rollup_bucket_of(int(x), p) for x in ts.tolist()], np.int64)
        for s, e in ((None, None), (NOW - timedelta(days=14), NOW), (NOW - timedelta(days=20), None), (None, NOW - timedelta(days=30))):
            sel = np.ones(n, bool)
            if s is not None:
                sel &= ts >= to_us(s)
            if e is not None:
                sel &= ts <= to_us(e)
            groups = {}
            for i in np.flatnonzero(sel).tolist():
                groups.setdefault((int(bucket[i]), int(rank[i])), []).append(i)
            want = ro.aggregated_usage(conn, period, s, e)
            assert len(want) == len(groups) > 0
            for w, (b, r) in zip(want, sorted(groups, key=lambda k: (-k[0], k[1]))):
                idx = groups[(b, r)]
                got = t._group_costs(period, s, e, b, r)
                assert [x.hex() for x in got] == [float(cost[i]).hex() for i in idx], (period, b, r)
                assert (w["time_period"], w["model"]) == (period_label(period, b), t._names[r])
                assert same(w["cost"], sqlite_sum(got)), (period, s, e, w, got)
