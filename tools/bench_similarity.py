#!/usr/bin/env python
"""Similarity search (Engine.db_similarity / db_similarity_batch) on the C5 database of tools/bench_configs.py: 10^7
records of 24..31 nt and its 64 queries.  For each of the 12 methods: 64 single-query calls, then the same 64 queries
as one batch, alternated; device ms (last_kernel_ms, summed over the single calls) and wall ms, top-k k = 10, no
all_scores.  Then one query alone through both paths (the batch path's one-query case), and the 64-query batch through
MultiEngine() on every visible GPU.  The batch rows are checked against the single-query results (== on the bits) and
two queries against oracle/ir_oracle.py on a prefix of the database.  One JSON line per measurement; the card's name
and power limit come first.
    python tools/bench_similarity.py [--records N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench_configs as BC  # noqa: E402
from bench_range import card  # noqa: E402

R = BC.R
K = 10


def same_bits(a, b):
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prefix", type=int, default=2000, help="records checked against the oracle")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    f = open(args.out, "a") if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if f:
            f.write(line + "\n"); f.flush()
    emit(card())
    from oracle import ir_oracle as IO
    codes, off, lens, qs, Q, db = BC.c5_data(args.records, 64)
    eng = R.Engine(0)
    eng.set_timing(True)
    eng.db_load(db)
    n = args.records
    batch = {}
    try:
        for method in IO.METHODS:
            sd, sw, bd, bw, od, ob = [], [], [], [], [], []
            for r in range(args.reps + 1):                 # round 0 warms both paths up
                t0 = time.perf_counter(); dev = 0.0; single = []
                for q in qs:
                    single.append(eng.db_similarity(q, method, k=K, want_scores=False)); dev += eng.last_kernel_ms()
                t1 = time.perf_counter()
                _, bi, bs = eng.db_similarity_batch(qs, method, k=K, want_scores=False); bdev = eng.last_kernel_ms()
                t2 = time.perf_counter()
                eng.db_similarity(qs[0], method, k=K, want_scores=False); o1 = eng.last_kernel_ms()
                eng.db_similarity_batch(qs[:1], method, k=K, want_scores=False); b1 = eng.last_kernel_ms()
                if r:
                    sd.append(dev); sw.append((t1 - t0) * 1e3); bd.append(bdev); bw.append((t2 - t1) * 1e3); od.append(o1); ob.append(b1)
            assert np.array_equal(bi, np.stack([s[1] for s in single])) and same_bits(bs, np.stack([s[2] for s in single])), method
            batch[method] = (bi, bs)
            emit({"db": "c5", "records": n, "queries": 64, "method": method, "k": K,
                  "single64_device_ms": float(np.median(sd)), "single64_wall_ms": float(np.median(sw)),
                  "batch64_device_ms": float(np.median(bd)), "batch64_wall_ms": float(np.median(bw)),
                  "device_speedup": float(np.median(sd) / np.median(bd)), "wall_speedup": float(np.median(sw) / np.median(bw)),
                  "one_query_single_device_ms": float(np.median(od)), "one_query_batch_device_ms": float(np.median(ob)),
                  "reps": args.reps, "single64_device_ms_all": sd, "batch64_device_ms_all": bd})
        # every row of a batch with all_scores == the single call, and two queries against the oracle on a prefix
        for method in IO.METHODS:
            alls, _, _ = eng.db_similarity_batch([qs[0], qs[63]], method)
            for j, qi in enumerate((0, 63)):
                one, _, _ = eng.db_similarity(qs[qi], method)
                assert same_bits(alls[j], one), method
                docs = [R.decode(codes[off[i]:off[i + 1]]) for i in range(args.prefix)]
                want = IO.search(R.decode(qs[qi]), docs, method)
                assert same_bits(alls[j, :args.prefix], want), method
        emit({"db": "c5", "oracle_checked_queries": [0, 63], "prefix": args.prefix, "batch_rows_equal_single": True, "ok": True})
    finally:
        eng.db_free()
    me = R.MultiEngine()
    try:
        me.db_load(db)
        for method in IO.METHODS:
            ts = []
            for r in range(args.reps + 1):
                t0 = time.perf_counter(); _, mi, ms = me.db_similarity_batch(qs, method, k=K, want_scores=False); t1 = time.perf_counter()
                if r:
                    ts.append((t1 - t0) * 1e3)
            assert np.array_equal(mi, batch[method][0]) and same_bits(ms, batch[method][1]), method
            emit({"db": "c5", "records": n, "queries": 64, "method": method, "k": K, "gpus": me.n_devices,
                  "multi_batch64_wall_ms": float(np.median(ts)), "equal_to_one_engine": True, "multi_batch64_wall_ms_all": ts})
    finally:
        me.close()


if __name__ == "__main__":
    main()
