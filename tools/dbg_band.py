#!/usr/bin/env python
"""Band against tape layout of the int16x2 distance kernel (k_dist_band16 / k_dist_twin16), both forced with
RSD_DIST_BAND, on device-resident batches: C2-shaped pairs (ACGU, lengths U[100, 300], user_costs) at several batch
sizes and batches of 1.5-4 kb pairs.  Prints the kernel time of each (median of 5 after 2 warm-ups) and checks that
both layouts give the same distances.  This is where RSD_BAND_MIN_PAIRS comes from.

    python tools/dbg_band.py [--sizes 1000,10000,...]"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as G  # noqa: E402

G.build()
import torch  # noqa: E402
import rna_sequence_diff_patch_b200 as R  # noqa: E402
from rna_sequence_diff_patch_b200 import cost_tables  # noqa: E402


def batch(rng, n, lo, hi):
    la = rng.integers(lo, hi + 1, size=n); lb = rng.integers(lo, hi + 1, size=n)
    oa = np.zeros(n + 1, np.int64); ob = np.zeros(n + 1, np.int64)
    np.cumsum(la, out=oa[1:]); np.cumsum(lb, out=ob[1:])
    ca = rng.integers(0, 4, size=int(oa[-1])).astype(np.uint8); cb = rng.integers(0, 4, size=int(ob[-1])).astype(np.uint8)
    return R.pack((ca, oa), bits=2), R.pack((cb, ob), bits=2), float((la.astype(np.float64) * lb).sum())


def time_layout(eng, A, B, band, reps=5, warm=2):
    os.environ["RSD_DIST_BAND"] = "1" if band else "0"
    t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (A.words, A.start, A.len, B.words, B.start, B.len)]
    out = torch.zeros(A.n, dtype=torch.float64, device="cuda")
    ms = []
    for k in range(warm + reps):
        eng.distance_batch_dev(*[x.data_ptr() for x in t], A.n, A.max_len, B.max_len, 2, A.symmask | B.symmask,
                               out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        if k >= warm:
            ms.append(eng.last_kernel_ms())
    del os.environ["RSD_DIST_BAND"]
    return float(np.median(ms)), float(min(ms)), float(max(ms)), out.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,10000,30000,60000,100000,150000,250000,400000,1000000")
    ap.add_argument("--long", default="1500:4000,2000:3000,3000:1500,4000:1000", help="length:pairs of the long batches")
    args = ap.parse_args()
    eng = R.Engine(0)
    eng.set_costs(cost_tables.user_costs())
    eng.set_timing(True)
    rng = np.random.default_rng(20260002)
    shapes = [(int(n), 100, 300) for n in args.sizes.split(",") if n]
    shapes += [(int(k), int(L), int(L)) for L, k in (x.split(":") for x in args.long.split(",") if x)]
    for n, lo, hi in shapes:
        A, B, cells = batch(rng, n, lo, hi)
        tt, tlo, thi, dt = time_layout(eng, A, B, False)
        tb, blo, bhi, db = time_layout(eng, A, B, True)
        same = np.array_equal(dt, db)
        print(f"{n:8d} pairs len {lo}-{hi}: tape {tt:8.3f} ms [{tlo:.3f}, {thi:.3f}] = {cells / tt * 1e-6:7.0f} GCUPS | "
              f"band {tb:8.3f} ms [{blo:.3f}, {bhi:.3f}] = {cells / tb * 1e-6:7.0f} GCUPS | band/tape {tb / tt:.3f} | "
              f"equal {same}", flush=True)
        assert same


if __name__ == "__main__":
    main()
