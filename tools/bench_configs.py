#!/usr/bin/env python
"""Measure BASELINE configs 3, 4 and 5 (bench.py covers config 2, the headline).  One JSON line per
config on stdout; used for profiles/ and DESIGN.md, not by the driver.
    python tools/bench_configs.py [--c3-pairs N] [--c5-records N] [--which c3,c4,c5[,c5i]]   (c5i: C5 with 1 % IUPAC records, fp64)"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as G  # noqa: E402

G.build()
import rna_sequence_diff_patch_b200 as R  # noqa: E402

DROPIN = os.path.join(ROOT, "rna-sequence-diff-patch_b200", "dropin")
DEFAULT = __import__('rna_sequence_diff_patch_b200.cost_tables', fromlist=['x']).default_costs()


def mutate_batch(rng, codes, off, alpha=4, p_sub=0.05, p_ins=0.025, p_del=0.025, lo=1000, hi=2000):
    """vectorised per-base mutation of a concatenated batch, each result clipped into [lo, hi]"""
    out_c, out_l = [], []
    for p in range(len(off) - 1):
        a = codes[off[p]:off[p + 1]]
        r = rng.random(a.shape[0])
        sub = rng.integers(0, alpha, size=a.shape[0], dtype=np.uint8)
        x = np.where(r < p_sub, sub, a)
        keep = ~((r >= p_sub) & (r < p_sub + p_del))
        reps = np.where(r > 1 - p_ins, 2, 1) * keep
        y = np.repeat(x, reps)
        dup = np.repeat(np.arange(a.shape[0]), reps)
        second = np.concatenate([[False], dup[1:] == dup[:-1]])
        y[second] = rng.integers(0, alpha, size=int(second.sum()), dtype=np.uint8)
        if y.shape[0] > hi: y = y[:hi]
        if y.shape[0] < lo: y = np.concatenate([y, rng.integers(0, alpha, size=lo - y.shape[0], dtype=np.uint8)])
        out_c.append(y); out_l.append(y.shape[0])
    o = np.zeros(len(out_l) + 1, np.int64); np.cumsum(out_l, out=o[1:])
    return np.concatenate(out_c), o


def c3(eng, n_pairs, reps=3):
    rng = np.random.default_rng(20260003)
    la = rng.integers(1000, 2001, size=n_pairs)
    oa = np.zeros(n_pairs + 1, np.int64); np.cumsum(la, out=oa[1:])
    ca = rng.integers(0, 4, size=int(oa[-1]), dtype=np.uint8)
    cb, ob = mutate_batch(rng, ca, oa)
    indep = np.arange(n_pairs) % 10 == 0
    for p in np.nonzero(indep)[0]:
        cb[ob[p]:ob[p + 1]] = rng.integers(0, 4, size=int(ob[p + 1] - ob[p]), dtype=np.uint8)
    A, B = R.pack((ca, oa)), R.pack((cb, ob))
    cells = float((np.diff(oa) * np.diff(ob)).sum())
    eng.set_costs(DEFAULT); eng.set_timing(True)
    import ctypes as C
    from rna_sequence_diff_patch_b200 import _lib
    lib = R.load_library()
    max_ops = int((A.len.astype(np.int64) + B.len).max())
    def pinned(shape, dtype):                     # page-locked output buffers (rsd_host_alloc), like a serving caller would use
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p(); _lib.check(lib.rsd_host_alloc(C.byref(ptr), n))
        return np.frombuffer((C.c_uint8 * n).from_address(ptr.value), dtype=dtype).reshape(shape)
    for P in (A, B):                              # page-locked inputs as well
        for name in ("words", "start", "len"):
            src = getattr(P, name); dst = pinned(src.shape, src.dtype); dst[...] = src; setattr(P, name, dst)
    op = pinned((n_pairs, max_ops), np.uint8); n_ops = pinned((n_pairs,), np.int32); dist = pinned((n_pairs,), np.float64)
    ok = pinned((n_pairs,), np.uint8); mode = C.c_int()
    ts, kms = [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        _lib.check(lib.rsd_script_patch_check_batch(
            eng.ctx, _lib.ptr(A.words, C.c_uint32), _lib.ptr(A.start, C.c_int64), _lib.ptr(A.len, C.c_int32), A.words.shape[0],
            _lib.ptr(B.words, C.c_uint32), _lib.ptr(B.start, C.c_int64), _lib.ptr(B.len, C.c_int32), B.words.shape[0],
            n_pairs, A.bits, A.symmask | B.symmask, 0, max_ops, _lib.ptr(op, C.c_uint8), None, None,
            _lib.ptr(n_ops, C.c_int32), _lib.ptr(dist, C.c_double), _lib.ptr(ok, C.c_uint8), C.byref(mode)))
        if r:
            ts.append(time.perf_counter() - t0); kms.append(eng.last_kernel_ms())
    assert ok.all()
    # a sample of the scripts against the oracle (op codes, counts, distances): first 64 pairs and 64 spread over the batch
    from oracle import oracle as O
    sample = np.unique(np.concatenate([np.arange(min(64, n_pairs)), np.linspace(0, n_pairs - 1, 64).astype(np.int64)]))
    sa = np.concatenate([ca[oa[p]:oa[p + 1]] for p in sample]); sb = np.concatenate([cb[ob[p]:ob[p + 1]] for p in sample])
    soa = np.concatenate([[0], np.cumsum([oa[p + 1] - oa[p] for p in sample])]).astype(np.int64)
    sob = np.concatenate([[0], np.cumsum([ob[p + 1] - ob[p] for p in sample])]).astype(np.int64)
    w_ops, _, _, w_cnt, w_dist = O.script_batch(sa, soa, sb, sob, DEFAULT)
    for x, p in enumerate(sample):
        assert n_ops[p] == w_cnt[x] and dist[p] == w_dist[x], f"C3 pair {p}: count / distance differ from the oracle"
        assert np.array_equal(op[p, :n_ops[p]], w_ops[x, :w_cnt[x]]), f"C3 pair {p}: script differs from the oracle"
    t, k = float(np.mean(ts)), float(np.mean(kms)) * 1e-3
    # HBM streams of the script path (SURVEY 8d): 2-bit direction codes written once by the forward kernel (16 rows per
    # 32-bit word, columns padded to the 32-column strips), packed inputs read, op bytes written
    la_, lb_ = np.diff(oa), np.diff(ob)
    dir_bytes = float((((la_ + 15) // 16) * (((lb_ + 31) // 32) * 32) * 4).sum())
    in_bytes = float(A.words.nbytes + B.words.nbytes + 2 * n_pairs * 12)
    hbm = {"direction_bytes_written": dir_bytes, "packed_input_bytes": in_bytes, "op_bytes_written": float(n_ops.sum()),
           "achieved_gbs_over_device_time": (dir_bytes + in_bytes + float(n_ops.sum())) / k * 1e-9, "peak_gbs": 6552.6}
    return {"config": "C3", "hbm_streams": hbm, "pairs": n_pairs, "cells": cells, "mode": mode.value,
            "e2e_pairs_per_s": n_pairs / t, "e2e_gcups": cells / t * 1e-9, "e2e_s": t,
            "device_pairs_per_s": n_pairs / k, "device_gcups": cells / k * 1e-9, "device_s": k,
            "roundtrip_ok": bool(ok.all()), "oracle_checked_pairs": int(sample.shape[0]), "output": "op bytes + n_ops + dist + ok (oi/oj derivable by prefix sum), pinned host buffers"}


def c4(eng, L=50000, reps=3, batch_pairs=24):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _synth import c4_pair                      # the pair whose oracle script digest is committed (tests/golden/c4_digest.json)
    a, b = c4_pair(m=L)
    eng.set_costs(DEFAULT); eng.set_timing(True)
    ts, kms = [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        res = eng.long_pair(a, b)
        if r:
            ts.append(time.perf_counter() - t0); kms.append(eng.last_kernel_ms())
    cells = float(L) * b.shape[0]
    t, k = float(np.mean(ts)), float(np.mean(kms)) * 1e-3
    fwd = []
    for r in range(reps + 1):
        eng.long_pair(a, b, want_script=False)
        if r:
            fwd.append(eng.last_kernel_ms())
    kf = float(np.mean(fwd)) * 1e-3
    digest_ok = None
    if L == 50000:
        import hashlib
        rec = json.load(open(os.path.join(ROOT, "tests", "golden", "c4_digest.json")))["c4_default_costs"]
        sha = lambda x, dt: hashlib.sha256(np.ascontiguousarray(x, dtype=dt).tobytes()).hexdigest()
        digest_ok = bool(res["dist"] == float.fromhex(rec["dist"]) and sha(res["op"], np.uint8) == rec["op_sha256"]
                         and sha(res["oi"], np.int32) == rec["oi_sha256"] and sha(res["oj"], np.int32) == rec["oj_sha256"])
        assert digest_ok, "C4 script differs from the oracle digest"
    # the batch form (BASELINE config 4 names "long pairs"): K pairs of the same shape in one rsd_long_pairs call;
    # pair 0 is the digest pair, every script is checked as a valid path whose cost equals the reported distance
    batch = None
    if batch_pairs > 1:
        pairs = [c4_pair(seed=20260004 + q, m=L) for q in range(batch_pairs)]
        bt, bk, bf = [], [], []
        for r in range(reps + 1):
            t0 = time.perf_counter()
            out = eng.long_pairs(pairs)
            if r:
                bt.append(time.perf_counter() - t0); bk.append(eng.last_kernel_ms()); bf.append(eng.long_forward_ms())
        bcells = float(sum(float(x.shape[0]) * y.shape[0] for x, y in pairs))
        assert out[0]["dist"] == res["dist"] and np.array_equal(out[0]["op"], res["op"]) and np.array_equal(out[0]["oj"], res["oj"])
        for (x, y), o in zip(pairs, out):
            op, oi, oj = o["op"], o["oi"], o["oj"]
            assert oi[-1] == x.shape[0] and oj[-1] == y.shape[0]
            upd = op == 2
            assert float((op != 2).sum() + (x[oi[upd] - 1] != y[oj[upd] - 1]).sum()) == o["dist"], "script cost != distance"
            assert np.array_equal(y[oj[op != 1] - 1], y), "patching A with the script does not give B"
        batch = {"pairs": batch_pairs, "cells": bcells, "device_s": float(np.mean(bk)) * 1e-3, "device_gcups": bcells / (float(np.mean(bk)) * 1e-3) * 1e-9,
                 "forward_s": float(np.mean(bf)) * 1e-3, "forward_gcups": bcells / (float(np.mean(bf)) * 1e-3) * 1e-9,
                 "e2e_s": float(np.mean(bt)), "e2e_gcups": bcells / float(np.mean(bt)) * 1e-9,
                 "checked": "pair 0 == the single-pair result (oracle digest); every script: valid path, cost == distance, patch(A) == B"}
    return {"config": "C4", "batch": batch, "script_equals_oracle_digest": digest_ok, "forward_only_device_s": kf, "forward_only_gcups": cells / kf * 1e-9, "m": L, "n": int(b.shape[0]), "cells": cells, "mode": res["mode"], "dist": res["dist"],
            "n_ops": int(res["op"].shape[0]), "e2e_gcups": cells / t * 1e-9, "e2e_s": t,
            "device_gcups": cells / k * 1e-9, "device_s": k}


def c1(eng):
    """BASELINE config 1: the named test_input.xml pairs through the StringEditDistance surface (wagnerFisher ->
    create_paths -> generate_es -> patching, and the reverse script), compared with what the unmodified reference
    returned for them (tests/golden/ref_golden.json: G2-G5 of SURVEY Appendix B); wall time per pair."""
    from rna_sequence_diff_patch_b200 import sed
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_golden.json")))
    times = []
    for name, c in g["xml_named"].items():
        costs = g["user_costs" if c["user"] else "default_costs"]
        t0 = time.perf_counter()
        dp = sed.wagner_fisher(c["a"], c["b"], costs, engine=eng)
        paths = sed.create_paths(dp)
        es = sed.generate_es(paths[0], c["a"], c["b"])
        code, out = sed.patching(es, c["a"])
        rcode, back = sed.patching(sed.generate_rev_es(es), c["b"])
        times.append(time.perf_counter() - t0)
        assert dp[len(dp) - 1][len(dp[0]) - 1].value == c["distance"] and len(paths) == c["n_paths"], name
        assert es == c["es"][0] and [code, out] == c["patch0"] and [rcode, back] == c["rev_patch0"], name
        assert sed.edit_script(c["a"], c["b"], costs, engine=eng) == es
    return {"config": "C1", "pairs": len(times), "ms_per_pair_all_steps": float(np.mean(times[1:]) * 1e3) if len(times) > 1 else float(times[0] * 1e3),
            "checked": "distance, number of co-optimal paths, ES of paths[0], patch and reverse-patch results == the reference's (golden)"}


def x2(eng, L=1_000_000):
    """One pair whose direction matrix (2 bit per cell: 250 GB at 10^6 x 10^6) exceeds the device: the row-block /
    panel-range overflow path of rsd_long_pair.  No CPU oracle at 10^12 cells: the script is checked as a valid path
    whose cost equals the reported distance, patch(A) == B, and the distance-only call (no directions, two alternating
    checkpoint rows) must give the same number."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _synth import c4_pair
    a, b = c4_pair(seed=20260042, m=L)
    eng.set_costs(DEFAULT); eng.set_timing(True)
    os.environ["RSD_TRACE"] = "1"
    t0 = time.perf_counter(); res = eng.long_pair(a, b); t_first = time.perf_counter() - t0       # includes the one-time cudaMalloc of the pool
    del os.environ["RSD_TRACE"]
    t0 = time.perf_counter(); res = eng.long_pair(a, b); t_script = time.perf_counter() - t0; dev_script = eng.last_kernel_ms() * 1e-3
    t0 = time.perf_counter(); d_only = eng.long_pair(a, b, want_script=False)["dist"]; t_dist = time.perf_counter() - t0; dev_dist = eng.last_kernel_ms() * 1e-3
    op, oi, oj = res["op"], res["oi"], res["oj"]
    assert oi[-1] == a.shape[0] and oj[-1] == b.shape[0]
    di = np.diff(np.concatenate([[0], oi])); dj = np.diff(np.concatenate([[0], oj]))
    assert np.array_equal(di, (op != 0).astype(np.int64)) and np.array_equal(dj, (op != 1).astype(np.int64)), "not a path"
    upd = op == 2
    assert float((op != 2).sum() + (a[oi[upd] - 1] != b[oj[upd] - 1]).sum()) == res["dist"] == d_only, "script cost != distance"
    assert np.array_equal(b[oj[op != 1] - 1], b), "patching A with the script does not give B"
    cells = float(a.shape[0]) * b.shape[0]
    return {"config": "x2-overflow", "m": int(a.shape[0]), "n": int(b.shape[0]), "cells": cells, "dist": res["dist"], "n_ops": int(op.shape[0]),
            "first_call_wall_s": t_first, "script_wall_s": t_script, "script_device_s": dev_script, "script_gcups_device": cells / dev_script * 1e-9,
            "distance_only_wall_s": t_dist, "distance_only_device_s": dev_dist, "distance_only_gcups_device": cells / dev_dist * 1e-9,
            "direction_matrix_bytes": cells / 4, "checked": "valid path, cost == distance == distance-only pass, patch(A) == B"}


def c5_data(n_rec, nq=64, iupac=False):
    """The single-process C5 database (24..31 nt, ACGU with one N per 1000 symbols) and nq queries (records with 10 %
    of their symbols redrawn) -> (codes, off, lens, query codes list, Q packed, db packed)."""
    rng = np.random.default_rng(20260005)
    lens = rng.integers(24, 32, size=n_rec)
    off = np.zeros(n_rec + 1, np.int64); np.cumsum(lens, out=off[1:])
    codes = rng.integers(0, 4, size=int(off[-1]), dtype=np.uint8)
    codes[rng.random(codes.shape[0]) < 1e-3] = 14
    if iupac:                                           # SURVEY 8d: second run, 1 % of the records drawn from all 15 symbols
        full = np.repeat(rng.random(n_rec) < 0.01, lens)   #   -> non-dyadic default costs (0.66 / 0.83) -> fp64 reference-order kernels
        codes[full] = rng.integers(0, 15, size=int(full.sum()), dtype=np.uint8)
    qs, qo = [], [0]
    for r in rng.integers(0, n_rec, size=nq):
        s = codes[off[r]:off[r + 1]].copy()
        hit = rng.random(s.shape[0]) < 0.1
        s[hit] = rng.integers(0, 4, size=int(hit.sum()), dtype=np.uint8)
        qs.append(s); qo.append(qo[-1] + s.shape[0])
    Q = R.pack((np.concatenate(qs), np.array(qo, np.int64)), bits=4)
    db = R.pack((codes, off), bits=4)
    return codes, off, lens, qs, Q, db


def c5(eng, n_rec, nq=64, k=10, reps=3, iupac=False):
    codes, off, lens, qs, Q, db = c5_data(n_rec, nq, iupac)
    eng.set_costs(DEFAULT); eng.set_timing(True)
    eng.db_load(db)
    cells = float(sum(len(q) for q in qs)) * 0 + float(np.add.outer(np.array([len(q) for q in qs]), np.zeros(1)).sum() * 0)
    cells = float(np.array([len(q) for q in qs], np.float64).sum() * lens.astype(np.float64).sum())
    ts, kms = [], []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        idx, sc = eng.db_search_topk(Q, k)
        if r:
            ts.append(time.perf_counter() - t0); kms.append(eng.last_kernel_ms())
    # every query's top-k against the oracle on a prefix of the database small enough for the CPU (the GPU result on
    # that prefix comes from a second, small load), plus two queries on the whole database
    from oracle import oracle as O
    for qi in (0, nq - 1):
        wi, ws = O.search_topk(O.decode(qs[qi]), codes, off, DEFAULT, k)
        assert np.array_equal(idx[qi], wi) and np.array_equal(sc[qi], ws), f"C5 query {qi} differs from the oracle"
    # the other scorers of search_collection on the same database (8f rank 4): one query, all scores + top-k on device
    sim = {}
    if iupac:
        eng.db_free()
        t, kk = float(np.mean(ts)), float(np.mean(kms)) * 1e-3
        return {"config": "C5-iupac", "records": n_rec, "queries": nq, "k": k, "cells": cells, "mode": eng.last_mode,
                "e2e_gcups": cells / t * 1e-9, "e2e_s": t, "device_gcups": cells / kk * 1e-9, "device_s": kk}
    db_bytes = float(db.words.nbytes + n_rec * (8 + 4 + 8 + 8))           # words + start + len + perm read, score written
    for method in ("set_jaccard_similarity", "multi_dice_similarity", "cosine", "pearson"):
        ms = []
        for r in range(3):
            eng.db_similarity(qs[0], method, k=k, want_scores=False)
            if r:
                ms.append(eng.last_kernel_ms())
        m = float(np.mean(ms))
        sim[method] = {"ms_per_query": m, "records_per_s": n_rec / (m * 1e-3), "hbm_gbs_algorithmic": db_bytes / (m * 1e-3) * 1e-9}
    eng.db_free()
    t, kk = float(np.mean(ts)), float(np.mean(kms)) * 1e-3
    return {"config": "C5", "similarity_search": sim, "records": n_rec, "queries": nq, "k": k, "cells": cells, "mode": eng.last_mode,
            "e2e_gcups": cells / t * 1e-9, "e2e_s": t, "device_gcups": cells / kk * 1e-9, "device_s": kk,
            "top1_scores_head": sc[:3, 0].tolist()}


def c2_iupac(eng, n_pairs, reps=3):
    """The reference's own default workload shape (timing.py:12-15: 15-letter strings, default costs.json) at C2
    lengths: non-dyadic costs -> the fp64 kernel in the reference's operation order.  Device-resident timing."""
    import torch
    rng = np.random.default_rng(20260002)
    la = rng.integers(100, 301, size=n_pairs); lb = rng.integers(100, 301, size=n_pairs)
    oa = np.zeros(n_pairs + 1, np.int64); ob = np.zeros(n_pairs + 1, np.int64)
    np.cumsum(la, out=oa[1:]); np.cumsum(lb, out=ob[1:])
    ca = rng.integers(0, 15, size=int(oa[-1]), dtype=np.uint8); cb = rng.integers(0, 15, size=int(ob[-1]), dtype=np.uint8)
    A, B = R.pack((ca, oa)), R.pack((cb, ob))
    eng.set_costs(DEFAULT); eng.set_timing(True)
    dev = torch.device("cuda", eng.device)
    d = {k: torch.from_numpy(v).to(dev) for k, v in dict(aw=A.words, as_=A.start, al=A.len, bw=B.words, bs=B.start, bl=B.len).items()}
    out = torch.zeros(n_pairs, dtype=torch.float64, device=dev)
    kms = []
    for r in range(reps + 1):
        eng.distance_batch_dev(d["aw"].data_ptr(), d["as_"].data_ptr(), d["al"].data_ptr(), d["bw"].data_ptr(), d["bs"].data_ptr(),
                               d["bl"].data_ptr(), n_pairs, A.max_len, B.max_len, 4, A.symmask | B.symmask, out.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        if r:
            kms.append(eng.last_kernel_ms())
    from oracle import oracle as O
    n_chk = min(n_pairs, 4000)
    want = O.distance_batch(ca[:oa[n_chk]], oa[:n_chk + 1].copy(), cb[:ob[n_chk]], ob[:n_chk + 1].copy(), DEFAULT)
    assert np.array_equal(out[:n_chk].cpu().numpy(), want), "fp64 distances differ from the oracle"
    cells = float((la * lb).sum()); k = float(np.mean(kms)) * 1e-3
    return {"pairs": n_pairs, "mode": eng.last_mode, "device_gcups": cells / k * 1e-9, "kernel_ms": k * 1e3, "oracle_checked_pairs": n_chk}


C5_BLOCKS = 64          # the synthetic database is generated in 64 independently seeded blocks so that a rank builds only its shard


def c5_block(b, records):
    """Records [records*b/64, records*(b+1)/64) of the C5 database: ocu.fa-shaped (24..31 nt, ACGU, one N per 1000 symbols)."""
    rng = np.random.default_rng([20260005, b])
    n = records * (b + 1) // C5_BLOCKS - records * b // C5_BLOCKS
    lens = rng.integers(24, 32, size=n)
    total = int(lens.sum())
    codes = rng.integers(0, 4, size=total, dtype=np.uint8)
    codes[rng.integers(0, total, size=rng.binomial(total, 1e-3))] = 14
    return codes, lens


def c5_queries(records, nq):
    """The query batch: records of block 0 with 10 % of their symbols redrawn (the same on every rank)."""
    codes, lens = c5_block(0, records)
    off = np.concatenate([[0], np.cumsum(lens)])
    rng = np.random.default_rng([20260005, 1000])
    qs = []
    for r in rng.integers(0, lens.shape[0], size=nq):
        s = codes[off[r]:off[r + 1]].copy()
        hit = rng.random(s.shape[0]) < 0.1
        s[hit] = rng.integers(0, 4, size=int(hit.sum()), dtype=np.uint8)
        qs.append(s)
    return qs


def c5_sharded(eng, rank, world, dev, records=10_000_000, nq=64, k=10, steps=10, warmup=3, check_queries=2):
    """BASELINE config 5 as north_star states it: the database sharded contiguously over the ranks (one per GPU),
    the query batch on every rank, a local exact top-k per shard, ONE NCCL all_gather of the packed (index, score)
    lists, merge with the same key.  Strong scaling: the database size is fixed.  Timed on the device (CUDA events,
    max over ranks); rank 0 checks the merged lists of `check_queries` queries against the oracle over the WHOLE
    database after the timed region.  Returns the dict for bench.py's other_configs (None on ranks > 0)."""
    import torch
    import torch.distributed as dist
    b_lo, b_hi = C5_BLOCKS * rank // world, C5_BLOCKS * (rank + 1) // world
    parts = [c5_block(b, records) for b in range(b_lo, b_hi)]
    codes = np.concatenate([p[0] for p in parts]); lens = np.concatenate([p[1] for p in parts])
    off = np.zeros(lens.shape[0] + 1, np.int64); np.cumsum(lens, out=off[1:])
    base = records * b_lo // C5_BLOCKS                              # global index of this shard's first record
    shard = R.pack((codes, off), bits=4)
    shard.symmask |= (1 << 14) | 0xF                                # one numeric mode on every rank
    qs = c5_queries(records, nq)
    Q = R.pack((np.concatenate(qs), np.concatenate([[0], np.cumsum([len(q) for q in qs])]).astype(np.int64)), bits=4)
    eng.set_costs(DEFAULT)
    eng.set_timing(False)
    eng.db_load(shard, global_index_base=base)
    try:
        qd = {n: torch.from_numpy(v).to(dev) for n, v in dict(w=Q.words, s=Q.start, l=Q.len).items()}
        local = torch.zeros((2, nq, k), dtype=torch.int64, device=dev)          # [0] indices, [1] fp64 scores (as bits)
        gathered = torch.zeros((world, 2, nq, k), dtype=torch.int64, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        launches0 = eng.launch_count()

        def step():
            eng.db_search_topk_dev(qd["w"].data_ptr(), qd["s"].data_ptr(), qd["l"].data_ptr(), nq, Q.max_len, 4, Q.symmask | 0xF | (1 << 14),
                                   k, local[0].data_ptr(), local[1].data_ptr(), stream)
            if world > 1:
                dist.all_gather_into_tensor(gathered, local)          # the one collective of the path: Q*k*16 bytes per rank
            else:
                gathered[0].copy_(local)

        for _ in range(max(warmup, 1)):
            step()
        torch.cuda.synchronize()
        launches_per_step = eng.launch_count() - launches0
        launches_per_step //= max(warmup, 1)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record(); e1.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        sym = torch.tensor([float(lens.sum())], dtype=torch.float64, device=dev)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
            dist.all_reduce(sym, op=dist.ReduceOp.SUM)
        mode = eng.last_mode
        if rank != 0:
            return None
        g = gathered.cpu().numpy()
        from rna_sequence_diff_patch_b200.engine import topk_merge
        mi, msc = topk_merge(np.ascontiguousarray(g[:, 0]), np.ascontiguousarray(g[:, 1]).view(np.float64))
        cells = float(sum(len(q) for q in qs)) * float(sym.item())
        res = {"records": records, "queries": nq, "k": k, "n_gpus": world, "scaling": "strong",
               "gcups": cells * steps / (ms * 1e-3) * 1e-9, "ms_per_query_batch": ms / steps, "mode": mode,
               "collective": "one all_gather_into_tensor of Q*k*16 B per rank (NCCL)" if world > 1 else "none (one shard)",
               "launches_per_batch": int(launches_per_step), "shard_records": int(lens.shape[0])}
        # oracle over the whole database (rank 0 rebuilds the blocks it did not hold)
        if check_queries:
            from oracle import oracle as O
            allp = [c5_block(b, records) for b in range(C5_BLOCKS)]
            ac = np.concatenate([p[0] for p in allp]); al = np.concatenate([p[1] for p in allp])
            ao = np.zeros(al.shape[0] + 1, np.int64); np.cumsum(al, out=ao[1:])
            for qi in list(range(nq))[:check_queries]:
                wi, ws = O.search_topk(O.decode(qs[qi]), ac, ao, DEFAULT, k)
                assert np.array_equal(mi[qi], wi) and np.array_equal(msc[qi], ws), f"sharded top-k of query {qi} differs from the oracle"
            res["oracle_checked_queries"] = check_queries
        return res
    finally:
        eng.db_free()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--which", default="c3,c4,c5")
    ap.add_argument("--c3-pairs", type=int, default=100000)
    ap.add_argument("--c5-records", type=int, default=10_000_000)
    ap.add_argument("--c5-iupac-queries", type=int, default=8)
    ap.add_argument("--x2-len", type=int, default=1_000_000)
    args = ap.parse_args()
    eng = R.Engine(0)
    for w in args.which.split(","):
        t0 = time.perf_counter()
        res = {"c3": lambda: c3(eng, args.c3_pairs), "c4": lambda: c4(eng), "c5": lambda: c5(eng, args.c5_records),
               "c5i": lambda: c5(eng, args.c5_records, nq=args.c5_iupac_queries, reps=2, iupac=True),
               "c2i": lambda: c2_iupac(eng, 200_000, reps=2), "c4s": lambda: c4(eng, reps=1, batch_pairs=8),
               "x2": lambda: x2(eng, args.x2_len), "c1": lambda: c1(eng)}[w]()
        res["wall_incl_datagen_s"] = time.perf_counter() - t0
        print(json.dumps(res), flush=True)
