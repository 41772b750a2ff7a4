"""One rank of the 2-rank rollup merge test (tests/test_rollup_gpu.py): this rank's half of the records is accumulated on the GPU
into a dense table, the tables are summed across ranks (NCCL all-reduce when every rank has its own GPU, else gloo over host
copies of the device tables), rank 0 compacts the merged table on the GPU and compares with SQLite over ALL records."""
import ctypes as C
import os
import sys
from datetime import datetime, timedelta
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))


def main():
    import torch
    import torch.distributed as dist
    import llmapigateway_b200 as L
    from llmapigateway_b200 import usage as U
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    ndev = torch.cuda.device_count()
    own_gpu = ndev >= world
    local = rank if own_gpu else 0
    torch.cuda.set_device(local)
    dist.init_process_group("nccl" if own_gpu else "gloo")
    dev = torch.device("cuda", local)
    NOW = datetime(2026, 9, 21, 6, 57, 17, 47518)
    n = 200_000
    ts, models, tok, cost = U.synth_usage_columns(n, seed=11, end=NOW)
    names = sorted({m for m in models if m is not None})
    flagged = n - 1                                         # one record of rank 1's half the fixed-point cost sum cannot hold
    ts[flagged], models[flagged], cost[flagged] = U.to_us(NOW - timedelta(days=1)), names[0], float("inf")
    if rank == 1:
        names_local_missing = names[-1]                     # rank 1 never sees the rarest model: the shared dictionary must still line up
        keep = np.array([m != names_local_missing for m in models])
    lo, hi = rank * n // world, (rank + 1) * n // world
    eng = L.Engine(device=local, max_streams=64, max_step_chunks=1024, max_step_bytes=1 << 20)
    tab = U.UsageTable(eng)
    tab.load_columns(ts[lo:hi], list(models[lo:hi]), *[t[lo:hi] for t in tok], cost[lo:hi], names=names)
    tab._upload()
    nm = len(names) + 1
    failures = 0
    for period, start, end in (("day", NOW - timedelta(weeks=2), NOW), ("hour", None, None), ("month", None, None)):
        p = U.PERIODS[period]
        qlo = max(int(ts.min()), U.to_us(start)) if start is not None else int(ts.min())
        qhi = min(int(ts.max()), U.to_us(end)) if end is not None else int(ts.max())
        b0 = int(tab._lib.lgw_rollup_bucket_of(qlo, p)); b1 = int(tab._lib.lgw_rollup_bucket_of(qhi, p))
        nb = b1 - b0 + 1 + (25 if period == "hour" else 1)
        table = torch.zeros(nb * nm * U.ROLLUP_CELLS, dtype=torch.int64, device=dev)
        inexact = torch.zeros(nb * nm, dtype=torch.int32, device=dev)
        oob = torch.zeros(2, dtype=torch.int32, device=dev)
        tab.accumulate(period, start, end, b0, nb, nm, C.c_void_p(table.data_ptr()), C.c_void_p(inexact.data_ptr()), C.c_void_p(oob.data_ptr()))
        eng.sync()
        if own_gpu:
            dist.all_reduce(table, op=dist.ReduceOp.SUM); dist.all_reduce(inexact, op=dist.ReduceOp.MAX)
        else:
            h_t, h_i = table.cpu(), inexact.cpu()
            dist.all_reduce(h_t, op=dist.ReduceOp.SUM); dist.all_reduce(h_i, op=dist.ReduceOp.MAX)
            table.copy_(h_t); inexact.copy_(h_i)
        torch.cuda.synchronize(dev)
        if rank == 0:
            from oracle import rollup_oracle as ro
            from test_rollup_gpu import _compare, _iso
            rows = tab.emit(b0, nb, nm, C.c_void_p(table.data_ptr()), C.c_void_p(inexact.data_ptr()))
            conn = ro.make_db([(_iso(ts[i]), int(tok[0][i]), int(tok[1][i]), int(tok[2][i]), int(tok[3][i]), int(tok[4][i]), float(cost[i]), models[i], "P") for i in range(n)])
            want = ro.aggregated_usage(conn, period, start, end)
            # the merged row of the flagged record's group carries the flag, and rows_to_dicts refuses to print its cost
            key = (U.period_label(period, int(tab._lib.lgw_rollup_bucket_of(int(ts[flagged]), p))), names[0])
            bad = np.flatnonzero(rows["inexact"])
            assert [(U.period_label(period, int(rows["bucket"][j])), tab._names[int(rows["model_rank"][j])]) for j in bad] == [key], (period, bad)
            try:
                tab.rows_to_dicts(period, rows)
                raise AssertionError("rows_to_dicts printed a flagged row")
            except ValueError:
                pass
            assert [w["cost"] for w in want if (w["time_period"], w["model"]) == key] == [float("inf")]
            _compare(tab.rows_to_dicts(period, np.delete(rows, bad)), [w for w in want if (w["time_period"], w["model"]) != key])
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("ROLLUP_MERGE_OK nccl" if own_gpu else "ROLLUP_MERGE_OK gloo")


if __name__ == "__main__":
    main()
