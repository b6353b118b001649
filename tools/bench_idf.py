#!/usr/bin/env python
"""Similarity search over idf and tf-idf vectors (Engine.db_similarity_batch(vector_type=...)) on the C5 database of
tools/bench_configs.py: 10^7 records of 24..31 nt and its 64 queries.  Reports the document-frequency table build (first
call after db_load, device ms and wall ms), then per vector type x the six vector measures one 64-query batch (top-k
k = 10, no all_scores), device ms (last_kernel_ms) and wall ms, beside the 'tf' batch of the same method in the same run;
then the same batches through MultiEngine() on every visible GPU.  The table is checked against tests/_idf_oracle.py in
full, and two queries' scores against the oracle on a prefix of the database under the verified table.  One JSON line per
measurement; the card's name and power limit come first.
    python tools/bench_idf.py [--records N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import bench_configs as BC  # noqa: E402
from bench_range import card  # noqa: E402

R = BC.R
K = 10
METHODS = ["cosine", "pearson", "euclidian_distance", "manhattan_distance", "tanimoto_distance", "dice_dist"]


def same_bits(a, b):
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--prefix", type=int, default=2000, help="records whose scores are checked against the oracle")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    f = open(args.out, "a") if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if f:
            f.write(line + "\n"); f.flush()
    emit(card())
    import _idf_oracle as IDF
    codes, off, lens, qs, Q, db = BC.c5_data(args.records, 64)
    n = args.records
    eng = R.Engine(0)
    eng.set_timing(True)
    eng.db_load(db)
    res = {}
    try:
        t0 = time.perf_counter(); df, idf = eng.db_idf_table(); t1 = time.perf_counter()
        emit({"db": "c5", "records": n, "idf_table_build_device_ms": eng.last_kernel_ms(), "idf_table_build_wall_ms": (t1 - t0) * 1e3})
        # the table against the oracle in full (np.cumsum over every record in collection order)
        df_want, idf_want = IDF.table_codes(codes, off)
        table_ok = same_bits(df.reshape(-1), df_want) and same_bits(idf.reshape(-1), idf_want)
        emit({"db": "c5", "idf_table_equals_oracle": table_ok})
        assert table_ok
        for method in METHODS:
            for vt in ("tf", "idf", "tf-idf"):
                dev, wall = [], []
                for r in range(args.reps + 1):           # round 0 warms up
                    t0 = time.perf_counter()
                    _, bi, bs = eng.db_similarity_batch(qs, method, k=K, want_scores=False, vector_type=vt)
                    t1 = time.perf_counter()
                    if r:
                        dev.append(eng.last_kernel_ms()); wall.append((t1 - t0) * 1e3)
                res[(vt, method)] = (bi, bs)
                emit({"db": "c5", "records": n, "queries": 64, "method": method, "vector_type": vt, "k": K,
                      "batch64_device_ms": float(np.median(dev)), "batch64_wall_ms": float(np.median(wall)),
                      "reps": args.reps, "batch64_device_ms_all": dev})
        pre = [R.decode(codes[off[i]:off[i + 1]]) for i in range(args.prefix)]
        for vt in ("idf", "tf-idf"):
            B = IDF.vectors(pre, vt, idf.reshape(-1))
            A = IDF.vectors([R.decode(qs[0]), R.decode(qs[63])], vt, idf.reshape(-1))
            for method in METHODS:
                alls, _, _ = eng.db_similarity_batch([qs[0], qs[63]], method, vector_type=vt)
                for j in range(2):
                    assert same_bits(alls[j, :args.prefix], IDF.scores(method, A[j], B)), (vt, method)
        emit({"db": "c5", "oracle_checked_queries": [0, 63], "prefix": args.prefix, "ok": True})
    finally:
        eng.db_free()
    me = R.MultiEngine()
    try:
        me.db_load(db)
        t0 = time.perf_counter(); mdf, midf = me.db_idf_table(); t1 = time.perf_counter()
        assert same_bits(mdf, df) and same_bits(midf, idf)
        emit({"db": "c5", "records": n, "gpus": me.n_devices, "multi_idf_table_build_wall_ms": (t1 - t0) * 1e3, "equal_to_one_engine": True})
        for method in METHODS:
            for vt in ("tf", "idf", "tf-idf"):
                ts = []
                for r in range(args.reps + 1):
                    t0 = time.perf_counter(); _, mi, ms = me.db_similarity_batch(qs, method, k=K, want_scores=False, vector_type=vt); t1 = time.perf_counter()
                    if r:
                        ts.append((t1 - t0) * 1e3)
                assert np.array_equal(mi, res[(vt, method)][0]) and same_bits(ms, res[(vt, method)][1]), (vt, method)
                emit({"db": "c5", "records": n, "queries": 64, "method": method, "vector_type": vt, "k": K, "gpus": me.n_devices,
                      "multi_batch64_wall_ms": float(np.median(ts)), "equal_to_one_engine": True, "multi_batch64_wall_ms_all": ts})
    finally:
        me.close()


if __name__ == "__main__":
    main()
