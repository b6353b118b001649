#!/usr/bin/env python
"""Appending records to the loaded C5 database (Engine.db_append) against reloading it.  The C5 database of
tools/bench_configs.py (10^7 records of 24..31 nt) is loaded with its last X records held back, X = 500, 10^4, 10^6,
and the X records are appended: wall ms of db_append without and with a built idf table (the table is then continued
over the X records).  Alternated with it in the same run: what a reload of the grown collection costs -- pack of the
whole collection (from the symbol codes; and once, from Python strings, what ir._Resident did before appends), db_load,
and the full idf table build.  After the last repetition of each X the appended database is checked against the fresh
load: stored order and tiers (db_layout), one 64-query top-k (k = 10) and one 64-query tf-idf cosine batch, and the idf
table, bit for bit.  One JSON line per measurement; the card's name and power limit come first.
    python tools/bench_append.py [--records N] [--reps R] [--out FILE]"""
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
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind != "f":
        return bool(a.shape == b.shape and np.array_equal(a, b))
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def part(codes, off, i0, i1):
    return codes[off[i0]:off[i1]], off[i0:i1 + 1] - off[i0]


def wall(f):
    t0 = time.perf_counter()
    out = f()
    return (time.perf_counter() - t0) * 1e3, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tails", default="500,10000,1000000")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    f = open(args.out, "a") if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if f:
            f.write(line + "\n"); f.flush()
    emit(card())
    n = args.records
    codes, off, lens, qs, Q, db = BC.c5_data(n, 64)
    # the collection as Python strings, packed once the way ir._Resident reloads it (pack(list of str))
    text = R.encoding._DEC[codes].tobytes().decode()
    strs = [text[off[i]:off[i + 1]] for i in range(n)]
    ms, _ = wall(lambda: R.pack(strs, bits=4))
    emit({"db": "c5", "records": n, "pack_from_str_wall_ms": ms})
    del strs, text
    eng, ref = R.Engine(0), R.Engine(0)
    for e in (eng, ref):
        e.set_costs(BC.DEFAULT)
    eng.db_load(db); eng.db_search_topk(Q, K); eng.db_similarity_batch(qs, "cosine", k=K, want_scores=False, vector_type="tf-idf")  # warm-up
    for X in (int(x) for x in args.tails.split(",")):
        head = R.pack(part(codes, off, 0, n - X), bits=4)
        tail_ms, tail = wall(lambda: R.pack(part(codes, off, n - X, n), bits=4))
        res = {"append_wall_ms": [], "append_idf_wall_ms": [], "pack_wall_ms": [], "load_wall_ms": [], "idf_build_wall_ms": []}
        for r in range(args.reps):
            eng.db_load(head)
            res["append_wall_ms"].append(wall(lambda: eng.db_append(tail))[0])
            eng.db_load(head); eng.db_idf_table()
            res["append_idf_wall_ms"].append(wall(lambda: eng.db_append(tail))[0])
            ms, full = wall(lambda: R.pack((codes, off), bits=4))
            res["pack_wall_ms"].append(ms)
            res["load_wall_ms"].append(wall(lambda: ref.db_load(full))[0])
            res["idf_build_wall_ms"].append(wall(lambda: ref.db_idf_table())[0])
        out = {"db": "c5", "records": n, "appended": X, "reps": args.reps, "pack_tail_wall_ms": tail_ms}
        out.update({k + "_median": float(np.median(v)) for k, v in res.items()})
        out.update(res)
        emit(out)
        # eng holds head + tail with a continued table, ref the fresh load of the whole collection with a fresh table
        la, lb = eng.db_layout(), ref.db_layout()
        layout_ok = all(same_bits(x, y) for x, y in zip(la, lb))
        ta, tb = eng.db_idf_table(), ref.db_idf_table()
        table_ok = same_bits(ta[0], tb[0]) and same_bits(ta[1], tb[1])
        ga, gb = eng.db_search_topk(Q, K), ref.db_search_topk(Q, K)
        topk_ok = same_bits(ga[0], gb[0]) and same_bits(ga[1], gb[1])
        va = eng.db_similarity_batch(qs, "cosine", k=K, want_scores=False, vector_type="tf-idf")
        vb = ref.db_similarity_batch(qs, "cosine", k=K, want_scores=False, vector_type="tf-idf")
        tfidf_ok = same_bits(va[1], vb[1]) and same_bits(va[2], vb[2])
        emit({"db": "c5", "appended": X, "layout_equal": layout_ok, "idf_table_equal": table_ok, "topk64_equal": topk_ok,
              "tfidf_cosine64_equal": tfidf_ok, "tier_end": [int(x) for x in la[1]]})
        assert layout_ok and table_ok and topk_ok and tfidf_ok, X


if __name__ == "__main__":
    main()
