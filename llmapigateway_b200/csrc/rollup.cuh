// Usage-stats rollup (SURVEY.md row a11): GROUP BY strftime(fmt, timestamp), model with SUM x5,
// SUM(cost), COUNT(*) -- llm_gateway_core/db/tokens_usage_db.py:222-304 (SQL at :268-286).
//
// Records are SoA in HBM, 40 B each: int64 timestamp (microseconds of the naive local datetime the
// reference writes at :135), int32 model rank (0 = NULL, else 1 + rank of the name in byte order,
// so ascending rank == SQL "model ASC"), 5 x int32 token counts, fp64 cost.
//
// Every accumulator is an integer, so partial tables from several GPUs merge with a plain sum in
// any order: token sums/count are int64; cost is summed EXACTLY as a 128-bit fixed-point number
// (LSB 2^-80) held as four 32-bit limbs in 64-bit cells, then rounded once to double (correctly
// rounded, half to even: tests/test_rollup_cost_cpu.py pins it bit for bit against math.fsum).
// A record is representable when it is finite, |c| < 2^15 and c * 2^80 is an integer; a group of
// fewer than 2^32 such records cannot leave the 128-bit range (2^32 * 2^15 * 2^80 = 2^127), nor can a
// 64-bit limb cell overflow.  A group holding any other record, or 2^32 records or more, is flagged
// `inexact`; the host answers those groups from its own copy of the records, like SQLite
// (usage.py: sqlite_sum).  SQLite's SUM(REAL) is a compensated sum, so unflagged groups agree
// with it to an ulp or so (tests allow 4 ulp).
//
// Bucket index (monotone in time, so descending index == "time_period DESC"):
//   hour  : day * 24 + hour-of-day          day : days since 1970-01-01   (day: see date_days)
//   week  : year * 64 + %W  (%W = week of year, Monday first, 00-53: SQLite/C strftime)
//   month : year * 12 + (month - 1)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define LGW_RHD __host__ __device__ __forceinline__
#else
#define LGW_RHD inline
#endif

namespace lgw {

enum RollupPeriod : int { RP_HOUR = 0, RP_DAY = 1, RP_WEEK = 2, RP_MONTH = 3 };
#define LGW_ROLLUP_CELLS 10          /* 5 token sums, count, 4 cost limbs */

// floor division for possibly negative numerators
LGW_RHD int64_t fdiv(int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; }

// civil date from days since 1970-01-01 (proleptic Gregorian; H. Hinnant's algorithm)
LGW_RHD void civil_from_days(int64_t z, int64_t& y, int& m, int& d) {
    z += 719468;
    const int64_t era = fdiv(z, 146097);
    const int64_t doe = z - era * 146097;
    const int64_t yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    y = yoe + era * 400;
    const int64_t doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const int64_t mp = (5 * doy + 2) / 153;
    d = (int)(doy - (153 * mp + 2) / 5 + 1);
    m = (int)(mp < 10 ? mp + 3 : mp - 9);
    if (m <= 2) ++y;
}
LGW_RHD int64_t days_from_civil(int64_t y, int m, int d) {
    y -= m <= 2;
    const int64_t era = fdiv(y, 400);
    const int64_t yoe = y - era * 400;
    const int64_t doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
    const int64_t doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
    return era * 146097 + doe - 719468;
}

// SQLite 3.45 date.c quirks, reproduced on purpose (the oracle IS SQLite, same library on the GPU box):
//  * the seconds field is rounded to milliseconds inside the Julian-day value, (int64)(s*1000 + 0.5),
//    so 23:59:59.9995+ becomes 24:00:00.000 of the same parsed date ("roll");
//  * Y-M-D stay as parsed unless D > 28, in which case isDate() re-derives them from the Julian day
//    (normalisation of dates like Feb 31) -- a rolled 31st becomes the 1st of the next month;
//  * %H is always the parsed hour;  %W takes the weekday from the (rolled) Julian day but the day of
//    year from the parsed date relative to Jan 1 of the year in use.
// '1999-12-31T23:59:59.999999' therefore formats as '2000-01-01 23:00:00' / '2000-W00', while
// '2026-03-01T23:59:59.999999' (a Sunday) stays '2026-03-01 23:00:00' but gets '2026-W09'.
LGW_RHD int64_t bucket_of(int64_t ts_us, int period) {
    const int64_t secs = fdiv(ts_us, 1000000);
    const int64_t us = ts_us - secs * 1000000;
    const int64_t pdays = fdiv(secs, 86400);                          // parsed date
    const int64_t tod = secs - pdays * 86400;                         // parsed time of day, seconds
    const int64_t sec_in_min = tod % 60;
    const double s = (double)(sec_in_min * 1000000 + us) / 1e6;      // what the parser makes of "SS.ffffff"
    const int64_t ms = (int64_t)(s * 1000.0 + 0.5);
    const bool roll = (tod - sec_in_min) * 1000 + ms >= 86400000;
    int64_t y; int m, d;
    civil_from_days(pdays, y, m, d);
    int64_t udays = pdays;                                            // date in use for %Y %m %d
    if (roll && d > 28) { udays = pdays + 1; civil_from_days(udays, y, m, d); }
    if (period == RP_HOUR) return udays * 24 + tod / 3600;
    if (period == RP_DAY) return udays;
    if (period == RP_MONTH) return y * 12 + (m - 1);
    int64_t nday = pdays - days_from_civil(y, 1, 1);                  // trunc((x.iJD - jan1.iJD + 12h) / 1d)
    if (nday < 0) nday = 0;
    const int64_t wdays = pdays + (roll ? 1 : 0);
    const int wd = (int)((((wdays % 7) + 7) % 7 + 3) % 7);            // Monday = 0; 1970-01-01 was a Thursday
    return y * 64 + (nday + 7 - wd) / 7;
}

// ---- exact cost accumulation ---------------------------------------------------------------------
// double -> signed 128-bit fixed point with LSB 2^-80, as four 32-bit limbs (two's complement).
// returns false when the value cannot be represented exactly (bits below 2^-80, |c| >= 2^15, NaN/Inf).
LGW_RHD bool cost_to_limbs(double c, uint32_t limb[4]) {
    uint64_t b; memcpy(&b, &c, 8);
    const int E = (int)((b >> 52) & 0x7FF);
    uint64_t M = b & 0x000FFFFFFFFFFFFFull;
    const bool neg = b >> 63;
    limb[0] = limb[1] = limb[2] = limb[3] = 0;
    if (E == 0x7FF) return false;
    if (E == 0) { if (M == 0) return true; return false; }            // subnormals: far below 2^-80
    M |= 1ull << 52;
    const int shift = E - 1075 + 80;                                  // value * 2^80 = M * 2^shift
    bool exact = true;
    uint64_t lo, hi;
    if (shift >= 0) {
        if (shift > 42) return false;                                 // |value| >= 2^15: 2^32 records could wrap the 128-bit sum
        if (shift == 0) { lo = M; hi = 0; }
        else { lo = M << shift; hi = M >> (64 - shift); }
    } else {
        const int r = -shift;
        if (r >= 53) { lo = 0; hi = 0; exact = false; }
        else { exact = (M & ((1ull << r) - 1)) == 0; lo = M >> r; hi = 0; }
    }
    if (neg) { lo = ~lo + 1; hi = ~hi + (lo == 0 ? 1 : 0); }
    limb[0] = (uint32_t)lo; limb[1] = (uint32_t)(lo >> 32); limb[2] = (uint32_t)hi; limb[3] = (uint32_t)(hi >> 32);
    return exact;
}

// four 64-bit cells of summed limbs -> one double, rounded half-to-even
LGW_RHD double limbs_to_cost(const uint64_t cell[4]) {
    // carry-propagate into a 128-bit two's complement value (mod 2^128)
    uint64_t c0 = cell[0];
    uint64_t c1 = cell[1] + (c0 >> 32);
    uint64_t c2 = cell[2] + (c1 >> 32);
    uint64_t c3 = cell[3] + (c2 >> 32);
    uint64_t lo = (c0 & 0xFFFFFFFFull) | (c1 << 32);
    uint64_t hi = (c2 & 0xFFFFFFFFull) | (c3 << 32);
    const bool neg = hi >> 63;
    if (neg) { lo = ~lo + 1; hi = ~hi + (lo == 0 ? 1 : 0); }
    if ((lo | hi) == 0) return 0.0;
    // top 64 significant bits + sticky
    int top;                      // index of the highest set bit (0..127)
    if (hi) { top = 127; while (!((hi >> (top - 64)) & 1)) --top; }
    else { top = 63; while (!((lo >> top) & 1)) --top; }
    uint64_t sig; bool sticky = false;
    if (top >= 64) {
        const int s = top - 63;                                       // drop s low bits (1..64)
        sig = s == 64 ? hi : (hi << (64 - s)) | (lo >> s);
        sticky = s == 64 ? lo != 0 : (lo & ((1ull << s) - 1)) != 0;
    } else sig = lo << (63 - top);
    // sig has its top bit at 63; value = sig * 2^(top - 63 - 80)
    uint64_t kept = sig >> 11;
    const uint64_t half = (sig >> 10) & 1, rest = sig & 0x3FF;
    int e2 = top - 80;                                                // exponent of the leading bit
    if (half && (rest || sticky || (kept & 1))) { ++kept; if (kept >> 53) { kept >>= 1; ++e2; } }
    const uint64_t bits = ((uint64_t)(e2 + 1023) << 52) | (kept & 0x000FFFFFFFFFFFFFull) | (neg ? 1ull << 63 : 0);
    double d; memcpy(&d, &bits, 8);
    return d;
}

struct RollupRow {               // == lgw_rollup_row
    int64_t bucket;
    int32_t model_rank; uint32_t inexact;
    int64_t prompt_tokens, completion_tokens, total_tokens, reasoning_tokens, cached_tokens;
    double cost;
    int64_t count;
};

#if defined(__CUDACC__)
struct RollupArgs {
    const int64_t* ts_us; const int32_t* model_rank;
    const int32_t* tok[5]; const double* cost;
    uint64_t n;
    int period; int64_t start_us, end_us; int has_start, has_end;
    int64_t bucket0; uint32_t n_buckets, n_models;       // dense table geometry: [n_buckets][n_models][CELLS]
    unsigned long long* table; uint32_t* inexact;        // inexact: per group flag (cost bits lost)
    uint32_t* oob;                                        // records whose bucket fell outside the table (must stay 0)
};

// one record per thread per trip; all table updates are 64-bit integer reductions (RED.ADD, no return)
__global__ void __launch_bounds__(256) k_rollup_accum(RollupArgs a) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (uint64_t)gridDim.x * blockDim.x) {
        const int64_t ts = __ldg(a.ts_us + i);
        if ((a.has_start && ts < a.start_us) || (a.has_end && ts > a.end_us)) continue;     // tokens_usage_db.py:255-266
        const int64_t b = bucket_of(ts, a.period) - a.bucket0;
        const uint32_t mr = (uint32_t)__ldg(a.model_rank + i);
        if (b < 0 || b >= (int64_t)a.n_buckets || mr >= a.n_models) { atomicAdd(a.oob, 1u); continue; }
        const uint64_t g = (uint64_t)b * a.n_models + mr;
        unsigned long long* cell = a.table + g * LGW_ROLLUP_CELLS;
#pragma unroll
        for (int k = 0; k < 5; ++k) atomicAdd(cell + k, (unsigned long long)(long long)__ldg(a.tok[k] + i));
        atomicAdd(cell + 5, 1ull);
        uint32_t limb[4];
        if (!cost_to_limbs(__ldg(a.cost + i), limb)) a.inexact[g] = 1;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (limb[k]) atomicAdd(cell + 6 + k, (unsigned long long)limb[k]);
    }
}

// ---- block-privatised accumulation (tables that fit in shared memory: every window the stats endpoint asks for, stats.py:46-55) ----
// Each block keeps the whole table in shared memory as 32-bit (lo, hi) halves, cell-major ([cell][group]: lanes of a warp that hit
// different groups hit different banks).  A 64-bit add is one native 32-bit shared atomic on `lo` plus -- only on a carry or a
// negative addend -- one on `hi`.  At the end the block stores its partial table to global scratch (plain coalesced stores) and
// k_rollup_merge folds the partials into the caller's table: no global atomics at all.
#define LGW_ROLLUP_SMEM_GROUPS 2560u                                  // 2560 x (10 x 8 + 4) B = 215 040 B (+ 8 KiB of queues; records are indexed with 32 bits)
LGW_RHD size_t rollup_smem_bytes(uint32_t groups) { return (size_t)groups * (LGW_ROLLUP_CELLS * 8 + 4) + 32u * 64u * 4u; }   // + the warps' index queues

__device__ __forceinline__ void smem_add64(uint32_t* lo, uint32_t* hi, uint32_t v, uint32_t sign_ext) {
    const uint32_t old = atomicAdd(lo, v);
    const uint32_t up = sign_ext + ((old + v) < old ? 1u : 0u);      // carry out of the low half + the addend's own high half
    if (up) atomicAdd(hi, up);
}

// one record into the block's table (all 32 lanes of the caller are expected to be here together: see the queue below)
__device__ __forceinline__ uint32_t rollup_smem_record(const RollupArgs& a, uint64_t i, int64_t ts, uint32_t G, uint32_t* lo, uint32_t* hi, uint32_t* flag) {
    const int64_t b = bucket_of(ts, a.period) - a.bucket0;
    const uint32_t mr = (uint32_t)__ldg(a.model_rank + i);
    if (b < 0 || b >= (int64_t)a.n_buckets || mr >= a.n_models) return 1u;
    const uint32_t g = (uint32_t)b * a.n_models + mr;
    int32_t v[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) v[k] = __ldg(a.tok[k] + i);
    const double cost = __ldg(a.cost + i);
#pragma unroll
    for (int k = 0; k < 5; ++k) smem_add64(lo + k * G + g, hi + k * G + g, (uint32_t)v[k], v[k] < 0 ? 0xFFFFFFFFu : 0u);
    smem_add64(lo + 5 * G + g, hi + 5 * G + g, 1u, 0u);
    uint32_t limb[4];
    if (!cost_to_limbs(cost, limb)) flag[g] = 1;
#pragma unroll
    for (int k = 0; k < 4; ++k) if (limb[k]) smem_add64(lo + (6 + k) * G + g, hi + (6 + k) * G + g, limb[k], 0u);
    return 0u;
}

// Records that pass the window filter are first QUEUED per warp (their indices, 64-entry ring in shared memory, positions from a
// ballot prefix) and handled 32 at a time by the whole warp: with a 2-week window over 400 days 3.5 % of the records pass, and
// without the queue 68 % of the warp trips would run the bucket / load / atomics path for one or two lanes.
#define LGW_ROLLUP_QUEUE 64u
__global__ void __launch_bounds__(1024, 1) k_rollup_accum_smem(RollupArgs a, unsigned long long* __restrict__ partial, uint32_t* __restrict__ partial_flag) {
    extern __shared__ uint32_t sm[];
    const uint32_t G = a.n_buckets * a.n_models;
    uint32_t* lo = sm;                                                // [CELLS][G]
    uint32_t* hi = sm + (size_t)LGW_ROLLUP_CELLS * G;                 // [CELLS][G]
    uint32_t* flag = hi + (size_t)LGW_ROLLUP_CELLS * G;               // [G]
    uint32_t* queue = flag + G + (threadIdx.x >> 5) * LGW_ROLLUP_QUEUE;   // this warp's ring of record indices
    for (uint32_t k = threadIdx.x; k < G * (2 * LGW_ROLLUP_CELLS + 1); k += blockDim.x) sm[k] = 0;
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
    uint32_t oob = 0, head = 0, tail = 0;                             // (head, tail: the same in every lane of the warp)
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t first = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t trips = a.n > (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u) ? (a.n - ((uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) + 4 * stride - 1) / (4 * stride) : 0;
    for (uint64_t t = 0; t < trips; ++t) {                            // (a warp-uniform trip count: the ballots below need all 32 lanes)
        const uint64_t i0 = first + t * 4 * stride;
        int64_t tsv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const uint64_t i = i0 + u * stride; tsv[u] = i < a.n ? __ldg(a.ts_us + i) : INT64_MIN; }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint64_t i = i0 + u * stride;
            const int64_t ts = tsv[u];
            const bool in = i < a.n && !((a.has_start && ts < a.start_us) || (a.has_end && ts > a.end_us));     // tokens_usage_db.py:255-266
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, in);
            if (in) queue[(tail + __popc(m & lt)) & (LGW_ROLLUP_QUEUE - 1u)] = (uint32_t)i;
            tail += __popc(m);
            __syncwarp();
            if (tail - head >= 32u) {
                const uint64_t j = queue[(head + lane) & (LGW_ROLLUP_QUEUE - 1u)];
                oob += rollup_smem_record(a, j, __ldg(a.ts_us + j), G, lo, hi, flag);
                head += 32u;
                __syncwarp();
            }
        }
    }
    if (lane < tail - head) {
        const uint64_t j = queue[(head + lane) & (LGW_ROLLUP_QUEUE - 1u)];
        oob += rollup_smem_record(a, j, __ldg(a.ts_us + j), G, lo, hi, flag);
    }
    if (oob) atomicAdd(a.oob, oob);
    __syncthreads();
    unsigned long long* mine = partial + (size_t)blockIdx.x * LGW_ROLLUP_CELLS * G;
    for (uint32_t k = threadIdx.x; k < G * LGW_ROLLUP_CELLS; k += blockDim.x) mine[k] = (unsigned long long)lo[k] | ((unsigned long long)hi[k] << 32);
    for (uint32_t k = threadIdx.x; k < G; k += blockDim.x) partial_flag[(size_t)blockIdx.x * G + k] = flag[k];
}

// table[g][cell] += sum over blocks of partial[block][cell][g] (64-bit wrap-around sums: exact two's complement).  blockIdx.y picks
// one of LGW_ROLLUP_MERGE_SLICES interleaved sets of blocks, so that the (independent, pipelined) loads of a thread stay few.
#define LGW_ROLLUP_MERGE_SLICES 16u
__global__ void __launch_bounds__(256) k_rollup_merge(const unsigned long long* __restrict__ partial, const uint32_t* __restrict__ partial_flag, uint32_t n_blocks,
                                                      uint32_t G, unsigned long long* table, uint32_t* inexact) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;         // index into [cell][g]
    const uint32_t slice = blockIdx.y;
    if (k < G * LGW_ROLLUP_CELLS) {
        unsigned long long s = 0;
#pragma unroll 4
        for (uint32_t b = slice; b < n_blocks; b += LGW_ROLLUP_MERGE_SLICES) s += partial[(size_t)b * LGW_ROLLUP_CELLS * G + k];
        const uint32_t cell = k / G, g = k % G;
        if (s) atomicAdd(table + (size_t)g * LGW_ROLLUP_CELLS + cell, s);
    }
    if (k < G) {
        uint32_t f = 0;
        for (uint32_t b = slice; b < n_blocks; b += LGW_ROLLUP_MERGE_SLICES) f |= partial_flag[(size_t)b * G + k];
        if (f) inexact[k] = 1;
    }
}

// ---- compaction: groups with count > 0, in "time_period DESC, model ASC" order, over as many blocks as the table needs --------------
// pass 1 counts the occupied groups of every 1024-position tile (output order), pass 2 scans the tile counts, pass 3 writes.
LGW_RHD uint64_t rollup_group_at(uint64_t j, uint32_t n_buckets, uint32_t n_models) {
    const uint64_t bdesc = j / n_models, mr = j % n_models;
    return (uint64_t)(n_buckets - 1 - bdesc) * n_models + mr;
}

__global__ void __launch_bounds__(1024) k_rollup_count(const unsigned long long* __restrict__ table, uint32_t n_buckets, uint32_t n_models, uint32_t* __restrict__ tile_count) {
    const uint64_t total = (uint64_t)n_buckets * n_models;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t has = j < total && table[rollup_group_at(j, n_buckets, n_models) * LGW_ROLLUP_CELLS + 5] != 0;
    const uint32_t c = __syncthreads_count(has);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = c;
}

__global__ void __launch_bounds__(1024) k_rollup_scan(uint32_t* tile_count, uint32_t n_tiles, unsigned long long* n_rows) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (uint32_t start = 0; start < n_tiles; start += blockDim.x) {
        const uint32_t k = start + threadIdx.x;
        const uint32_t v = k < n_tiles ? tile_count[k] : 0;
        uint32_t x = v;                                               // inclusive warp scan
        const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d); if (lane >= (uint32_t)d) x += y; }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        uint32_t before = 0, all = 0;
        for (uint32_t w = 0; w < 32; ++w) { const uint32_t s = warp_sums[w]; if (w < warp) before += s; all += s; }
        if (k < n_tiles) tile_count[k] = base + before + x - v;       // exclusive offset of the tile
        __syncthreads();
        if (threadIdx.x == 0) base += all;
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_rows = base;
}

__global__ void __launch_bounds__(1024) k_rollup_write(const unsigned long long* __restrict__ table, const uint32_t* __restrict__ inexact, uint32_t n_buckets, uint32_t n_models,
                                                       int64_t bucket0, const uint32_t* __restrict__ tile_off, RollupRow* rows, unsigned long long rows_cap) {
    __shared__ uint32_t warp_sums[32];
    const uint64_t total = (uint64_t)n_buckets * n_models;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t g = 0; uint32_t has = 0;
    if (j < total) { g = rollup_group_at(j, n_buckets, n_models); has = table[g * LGW_ROLLUP_CELLS + 5] != 0; }
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, has);
    if (lane == 0) warp_sums[warp] = __popc(ballot);
    __syncthreads();
    uint32_t before = 0;
    for (uint32_t w = 0; w < warp; ++w) before += warp_sums[w];
    const unsigned long long pos = (unsigned long long)tile_off[blockIdx.x] + before + __popc(ballot & ((1u << lane) - 1));
    if (has && pos < rows_cap) {
        const unsigned long long* c = table + g * LGW_ROLLUP_CELLS;
        RollupRow r;
        r.bucket = bucket0 + (int64_t)(g / n_models); r.model_rank = (int32_t)(g % n_models);
        r.inexact = inexact[g] | (uint32_t)(c[5] >> 32 != 0);          // >= 2^32 records: the cost cells may have wrapped
        r.prompt_tokens = (int64_t)c[0]; r.completion_tokens = (int64_t)c[1]; r.total_tokens = (int64_t)c[2];
        r.reasoning_tokens = (int64_t)c[3]; r.cached_tokens = (int64_t)c[4]; r.count = (int64_t)c[5];
        uint64_t cells[4] = {c[6], c[7], c[8], c[9]};
        r.cost = limbs_to_cost(cells);
        rows[pos] = r;
    }
}
#endif

}  // namespace lgw
