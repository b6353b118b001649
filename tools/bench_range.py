#!/usr/bin/env python
"""Range search (Engine.db_search_range) on the C5 database of tools/bench_configs.py: 10^7 records of 24..31 nt,
64 queries mutated at 10 %, default costs.  For each bound: hits, device ms (last_kernel_ms), wall ms and cells/s,
with db_search_topk(k=10) on the same batch, the two alternated in one loop.  Then the c5i variant (1 % IUPAC
records: the fp64 tail).  Two queries per database are checked against the oracle over the whole database.
One JSON line per measurement; the card's name and power limit come first.
    python tools/bench_range.py [--records N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bench_configs as BC  # noqa: E402

R = BC.R
BOUNDS = (0.0, 1.0, 2.0, 4.0)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:                       # noqa: BLE001
        return {"gpu": "unknown", "error": repr(ex)}


def run(eng, n_rec, iupac, reps, emit):
    from oracle import oracle as O
    codes, off, lens, qs, Q, db = BC.c5_data(n_rec, 64, iupac)
    cells = float(np.array([len(q) for q in qs], np.float64).sum() * lens.astype(np.float64).sum())
    eng.set_costs(BC.DEFAULT); eng.set_timing(True)
    eng.db_load(db)
    try:
        res = {}
        for b in BOUNDS:
            rt, rk, tt, tk = [], [], [], []
            for r in range(reps + 1):                  # round 0 warms both paths up
                t0 = time.perf_counter(); res[b] = eng.db_search_range(Q, b); t1 = time.perf_counter()
                k_range, mode = eng.last_kernel_ms(), eng.last_mode
                t2 = time.perf_counter(); eng.db_search_topk(Q, 10); t3 = time.perf_counter()
                if r:
                    rt.append((t1 - t0) * 1e3); rk.append(k_range); tt.append((t3 - t2) * 1e3); tk.append(eng.last_kernel_ms())
            emit({"db": "c5i" if iupac else "c5", "records": n_rec, "queries": 64, "max_dist": b, "hits": int(res[b][0][-1]),
                  "mode": mode, "range_device_ms": float(np.median(rk)), "range_wall_ms": float(np.median(rt)),
                  "range_device_gcups": cells / (np.median(rk) * 1e-3) * 1e-9,
                  "topk10_device_ms": float(np.median(tk)), "topk10_wall_ms": float(np.median(tt)),
                  "topk10_device_gcups": cells / (np.median(tk) * 1e-3) * 1e-9, "reps": reps,
                  "range_device_ms_all": rk, "topk10_device_ms_all": tk})
    finally:
        eng.db_free()
    for qi in (0, 63):                                  # the oracle over the whole database
        qc = qs[qi]
        d = O.distance_batch(np.tile(qc, n_rec), np.arange(n_rec + 1, dtype=np.int64) * qc.shape[0], codes, off, BC.DEFAULT)
        for b in BOUNDS:
            o, i, dist = res[b]
            want = np.flatnonzero(d <= b)
            assert np.array_equal(i[o[qi]:o[qi + 1]], want), (iupac, qi, b)
            assert np.array_equal(dist[o[qi]:o[qi + 1]], d[want]), (iupac, qi, b)
    emit({"db": "c5i" if iupac else "c5", "oracle_checked_queries": [0, 63], "bounds": list(BOUNDS), "ok": True})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=10_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    f = open(args.out, "a") if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if f:
            f.write(line + "\n"); f.flush()
    emit(card())
    eng = R.Engine(0)
    run(eng, args.records, False, args.reps, emit)
    run(eng, args.records, True, args.reps, emit)


if __name__ == "__main__":
    main()
