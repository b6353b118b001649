#!/usr/bin/env python
"""Host paths of the pair-batch and search calls on one build: for every call, the launch_count() delta, the numeric
mode, a digest of the results, the RSD_TRACE lines with their times blanked (chunk counts, band vs tape, long-batch
layout) and, with timing on, last_kernel_ms() (median of 5 after a warm-up).  Run it on two builds and diff the logs:
everything but the `ms` lines must match.

    python tools/dbg_host_paths.py [--root TREE]        (TREE: the build to load, default this checkout)

Calls: chunked distance_batch (canonical and explicit start[]), distance_batch_codes, distance_batch_dev, the general
kernels (forced int32, fp64 under the default costs), 200 pairs of 7 kb through distance_batch (packed and raw codes)
and script_batch (both routed to the panel kernels), a chunked script_batch (RSD_SCRIPT_BUDGET_WORDS), and top-k and
range searches whose queries form two groups (A/C/G/U queries and queries with ambiguity codes)."""
import argparse
import dataclasses
import hashlib
import os
import re
import sys
import tempfile

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))
import __graft_entry__ as G  # noqa: E402

G.build()
import torch  # noqa: E402
import rna_sequence_diff_patch_b200 as R  # noqa: E402
from rna_sequence_diff_patch_b200 import cost_tables  # noqa: E402

I32, F64 = 2, 3      # RSD_MODE_I32 / RSD_MODE_F64 (include/rsd.h)


def batch(rng, n, lo, hi, n_sym=4):
    la = rng.integers(lo, hi + 1, size=n); lb = rng.integers(lo, hi + 1, size=n)
    oa = np.zeros(n + 1, np.int64); ob = np.zeros(n + 1, np.int64)
    np.cumsum(la, out=oa[1:]); np.cumsum(lb, out=ob[1:])
    ca = rng.integers(0, n_sym, size=int(oa[-1])).astype(np.uint8); cb = rng.integers(0, n_sym, size=int(ob[-1])).astype(np.uint8)
    return (ca, oa, la.astype(np.int32)), (cb, ob, lb.astype(np.int32))


def digest(x):
    h = hashlib.sha256()
    for a in (x if isinstance(x, (list, tuple)) else [x]):
        if isinstance(a, dict):
            for k in sorted(a):
                h.update(np.ascontiguousarray(a[k]).tobytes())
        else:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def traced(fn):
    """fn() with RSD_TRACE=1 (and timing on, for the chunk lines) and the library's stderr captured -> (result, trace lines
    with times blanked)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        os.environ["RSD_TRACE"] = "1"
        try:
            res = fn()
            torch.cuda.synchronize()
        finally:
            del os.environ["RSD_TRACE"]
            os.dup2(saved, 2); os.close(saved)
        f.seek(0)
        lines = f.read().decode(errors="replace").splitlines()
    lines = [re.sub(r"\d+\.\d+( ?(ms|us))?", "#", ln) for ln in lines if ln.startswith("[rsd trace]")]
    return res, lines


def run(eng, name, fn, env=None):
    for k, v in (env or {}).items():
        os.environ[k] = v
    eng.set_timing(True)
    try:
        res, lines = traced(fn)
        fn()                                         # warm-up
        ms, launches = [], set()
        for _ in range(5):
            l0 = eng.launch_count()
            again = fn()
            torch.cuda.synchronize()
            ms.append(eng.last_kernel_ms())
            launches.add(eng.launch_count() - l0)
        eng.set_timing(False)
    finally:
        for k in (env or {}):
            del os.environ[k]
    same = digest(res) == digest(again)
    print(f"== {name}: mode {eng.last_mode} launches {sorted(launches)} results {digest(res)} traced==untraced {same}")
    for ln in lines:
        print("   ", ln)
    print(f"   ms {float(np.median(ms)):.4f}", flush=True)


def main():
    rng = np.random.default_rng(20261022)
    eng = R.Engine(0)
    user, default = cost_tables.user_costs(), cost_tables.default_costs()
    print("device", torch.cuda.get_device_name(0), flush=True)

    # the bench's C2 shape: the host calls cut it into chunks, the small ones on the tape layout, the large ones on the band
    (ca, oa, la), (cb, ob, lb) = batch(rng, 1_000_000, 100, 300)
    A, B = R.pack((ca, oa), bits=2), R.pack((cb, ob), bits=2)
    Ae, Be = dataclasses.replace(A, canonical=False), dataclasses.replace(B, canonical=False)
    eng.set_costs(user)
    run(eng, "distance_batch canonical", lambda: eng.distance_batch(A, B))
    run(eng, "distance_batch explicit start", lambda: eng.distance_batch(Ae, Be))
    run(eng, "distance_batch_codes", lambda: eng.distance_batch_codes(ca, la, cb, lb, bits=2, symmask=0xF))
    t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (A.words, A.start, A.len, B.words, B.start, B.len)]
    out = torch.empty(A.n, dtype=torch.float64, device="cuda")

    def dev():
        eng.distance_batch_dev(*[x.data_ptr() for x in t], A.n, A.max_len, B.max_len, 2, A.symmask | B.symmask,
                               out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return out.cpu().numpy()
    run(eng, "distance_batch_dev", dev)
    run(eng, "distance_batch forced int32 (k_dist_gen<int, 2>)", lambda: eng.distance_batch(A, B, force_mode=I32))
    A4, B4 = A.repack(4), B.repack(4)
    run(eng, "distance_batch forced int32, 4 bit (k_dist_gen<int, 4>)", lambda: eng.distance_batch(A4, B4, force_mode=I32))
    run(eng, "distance_batch forced fp64 (k_dist_gen<double, 2>)", lambda: eng.distance_batch(A, B, force_mode=F64))
    (ia, ioa, _), (ib, iob, _) = batch(rng, 50_000, 100, 300, n_sym=15)
    IA, IB = R.pack((ia, ioa), bits=4), R.pack((ib, iob), bits=4)
    eng.set_costs(default)
    run(eng, "distance_batch IUPAC, default costs (k_dist_gen<double, 4>)", lambda: eng.distance_batch(IA, IB))

    # 200 pairs of 7 kb: routed to the panel kernels by the distance and the script calls
    (lc, loa, lla), (lcb, lob, llb) = batch(rng, 200, 6800, 7200)
    LA, LB = R.pack((lc, loa), bits=2), R.pack((lcb, lob), bits=2)
    run(eng, "distance_batch 200 x 7 kb (routed)", lambda: eng.distance_batch(LA, LB))
    run(eng, "distance_batch explicit start 200 x 7 kb (routed)",
        lambda: eng.distance_batch(dataclasses.replace(LA, canonical=False), dataclasses.replace(LB, canonical=False)))
    run(eng, "distance_batch_codes 200 x 7 kb (routed)", lambda: eng.distance_batch_codes(lc, lla, lcb, llb, bits=2, symmask=0xF))
    run(eng, "script_batch 200 x 7 kb (routed)", lambda: eng.script_batch(LA, LB))
    run(eng, "script_batch 200 x 7 kb, RSD_SCRIPT_NO_LONG", lambda: eng.script_batch(LA, LB), {"RSD_SCRIPT_NO_LONG": "1"})

    # chunked script batch: a direction-word budget of 2 * 10^5 words cuts 3000 pairs into tens of chunks
    (sa, soa, _), (sb, sob, _) = batch(rng, 3000, 100, 300)
    SA, SB = R.pack((sa, soa), bits=2), R.pack((sb, sob), bits=2)
    run(eng, "script_batch chunked", lambda: eng.script_batch(SA, SB), {"RSD_SCRIPT_BUDGET_WORDS": "200000"})
    run(eng, "script_batch round trip", lambda: eng.script_batch(SA, SB, check_roundtrip=True))

    # search: A/C/G/U database, queries with and without ambiguity codes (two query groups)
    (dc, do, _), _ = batch(rng, 60_000, 100, 300)
    eng.db_load(R.pack((dc, do), bits=4))
    (qc, qo, _), _ = batch(rng, 12, 150, 250)
    qc = qc.copy()
    for q in range(8, 12):                                 # the last four queries carry every ambiguity code (4..14)
        qc[qo[q] + 5:qo[q] + 16] = np.arange(4, 15)
    Q = R.pack((qc, qo), bits=4)
    run(eng, "db_search_topk two groups", lambda: eng.db_search_topk(Q, 10))
    run(eng, "db_search_range two groups", lambda: eng.db_search_range(Q, 60.0))
    eng.close()


main()
