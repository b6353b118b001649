#!/usr/bin/env python
"""Randomised parity fuzz of the CUDA paths against the C oracle (test infrastructure, not the product):
random alphabets, cost tables (shipped, random dyadic, random decimal), length mixes (empties, tiny,
100-300, kb-sized, skewed), batch sizes on both sides of the chunking threshold, forced numeric modes.
Everything is compared with `==`.  Prints one line per round and a summary; exit code 1 on any mismatch.

    python tools/fuzz_gpu.py [--seconds 120] [--seed 1]"""
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
from oracle import oracle as O  # noqa: E402
from oracle import ir_oracle as IO  # noqa: E402

DROPIN = os.path.join(ROOT, "rna-sequence-diff-patch_b200", "dropin")
DEFAULT = __import__('rna_sequence_diff_patch_b200.cost_tables', fromlist=['x']).default_costs()
USER = __import__('rna_sequence_diff_patch_b200.cost_tables', fromlist=['x']).user_costs()
SYM = "AGCUYRWSKMDVHBN"


def random_costs(rng, kind):
    if kind == "default":
        return DEFAULT
    if kind == "user":
        return USER
    c = {"insert": 0, "delete": 0, "update": {a: {b: 0.0 for b in SYM} for a in SYM}}
    if kind == "dyadic":
        q = float(rng.choice([1.0, 0.5, 0.25]))
        pick = lambda: float(rng.integers(1, 13)) * q
    elif kind == "int":
        pick = lambda: float(rng.integers(1, 6))
    else:
        pick = lambda: float(np.round(rng.uniform(0.05, 3.0), int(rng.integers(1, 4))))
    c["insert"], c["delete"] = pick(), pick()
    for a in SYM:
        for b in SYM:
            c["update"][a][b] = pick()
    return c


def random_lengths(rng, n, kind):
    if kind == "tiny":
        return rng.integers(0, 6, size=n)
    if kind == "short":
        return rng.integers(0, 41, size=n)
    if kind == "c2":
        return rng.integers(100, 301, size=n)
    if kind == "kb":
        return rng.integers(600, 2200, size=n)
    if kind == "skew":
        L = rng.integers(1, 60, size=n)
        big = rng.random(n) < 0.03
        L[big] = rng.integers(400, 3000, size=int(big.sum()))
        return L
    return rng.integers(0, 700, size=n)                      # "wide"


def make(rng, lens, alpha):
    off = np.zeros(lens.shape[0] + 1, np.int64); np.cumsum(lens, out=off[1:])
    al = np.array([SYM.index(ch) for ch in alpha], np.uint8)
    return al[rng.integers(0, len(al), size=int(off[-1]))], off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=120)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    rng = np.random.default_rng(args.seed)
    eng, ref = R.Engine(0), None
    t_end = time.time() + args.seconds
    rounds = bad = 0
    cells = 0.0
    while time.time() < t_end:
        rounds += 1
        alpha = [SYM[:4], SYM[:4], SYM[:4] + "N", SYM, SYM[:2], "ACGUYR"][int(rng.integers(0, 6))]
        ckind = ["default", "user", "dyadic", "int", "decimal"][int(rng.integers(0, 5))]
        lkind = ["tiny", "short", "c2", "kb", "skew", "wide"][int(rng.integers(0, 6))]
        what = ["dist", "dist", "script", "search", "long", "sim", "range", "simb", "append"][int(rng.integers(0, 9))]
        costs = random_costs(rng, ckind)
        eng.set_costs(costs)
        force = int(rng.choice([0, 0, 0, 2, 3]))
        try:
            if what == "dist":
                budget = 3e8 if lkind != "kb" else 1.5e9
                n = int(rng.choice([1, 7, 300, 5000, 66000, 150000]))
                la, lb = random_lengths(rng, n, lkind), random_lengths(rng, n, lkind)
                while float((la.astype(np.float64) * lb).sum()) > budget and n > 1:
                    n //= 2; la, lb = la[:n], lb[:n]
                ca, oa = make(rng, la, alpha); cb, ob = make(rng, lb, alpha)
                knobs = {}
                if rng.random() < 0.6: knobs["RSD_DIST_BAND"] = str(rng.choice([0, 1]))     # int16x2 layout: band / tape
                os.environ.update(knobs)
                try:
                    got = eng.distance_batch(R.pack((ca, oa)), R.pack((cb, ob)), force_mode=force)
                finally:
                    for kname in knobs: del os.environ[kname]
                want = O.distance_batch(ca, oa, cb, ob, costs)
                ok = np.array_equal(got, want)
                cells += float((la.astype(np.float64) * lb).sum())
                desc = f"dist n={n} mode={eng.last_mode} knobs={knobs}"
            elif what == "script":
                n = int(rng.choice([1, 5, 200, 2000]))
                if lkind in ("kb", "wide", "skew"):
                    n = min(n, 60)
                la, lb = random_lengths(rng, n, lkind), random_lengths(rng, n, lkind)
                ca, oa = make(rng, la, alpha); cb, ob = make(rng, lb, alpha)
                if rng.random() < 0.5 and n > 1:                 # homologous pairs: long tie runs
                    cb, ob = ca.copy(), oa.copy()
                    hit = rng.random(cb.shape[0]) < 0.08
                    al = np.array([SYM.index(ch) for ch in alpha], np.uint8)
                    cb[hit] = al[rng.integers(0, len(al), size=int(hit.sum()))]
                res = eng.script_batch(R.pack((ca, oa)), R.pack((cb, ob)), force_mode=force if force != 2 else 0, check_roundtrip=True)
                ops, oi, oj, cnt, dist = O.script_batch(ca, oa, cb, ob, costs)
                ok = np.array_equal(res["dist"], dist) and np.array_equal(res["n_ops"], cnt) and bool(res["ok"].all())
                for p in range(n):
                    k = cnt[p]
                    ok = ok and np.array_equal(res["op"][p, :k], ops[p, :k]) and np.array_equal(res["oi"][p, :k], oi[p, :k]) \
                        and np.array_equal(res["oj"][p, :k], oj[p, :k])
                cells += float((np.diff(oa).astype(np.float64) * np.diff(ob)).sum())
                desc = f"script n={n} mode={eng.last_mode}"
            elif what == "sim":
                n = int(rng.choice([1, 40, 400]))
                lens = rng.integers(0, int(rng.choice([8, 40, 300])), size=n)
                cd, od = make(rng, lens, alpha)
                docs = [O.decode(cd[od[k]:od[k + 1]]) for k in range(n)]
                q = O.decode(make(rng, np.array([int(rng.integers(0, 40))]), alpha)[0])
                bits = 2 if (set(alpha) <= set("AGCU") and rng.random() < 0.5) else 4
                eng.db_load(R.pack((cd, od), bits=bits))
                ok = True
                try:
                    for method in rng.choice(IO.METHODS, size=3, replace=False):
                        got, _, _ = eng.db_similarity(R.encode(q), str(method))
                        qa = IO.represent(q, str(method))
                        want = np.zeros(n)
                        for k2, d2 in enumerate(docs):
                            try:
                                want[k2] = IO.score(str(method), qa, IO.represent(d2, str(method)))
                            except ZeroDivisionError:          # set measures of two empty sequences: the reference raises, the device returns NaN
                                want[k2] = np.nan
                        ok = ok and bool(np.array_equal(np.isnan(got), np.isnan(want))
                                         and np.array_equal(got[~np.isnan(got)].view(np.uint64), want[~np.isnan(want)].view(np.uint64)))
                finally:
                    eng.db_free()
                desc = f"sim n={n} bits={bits} qlen={len(q)} mode=0"
            elif what == "simb":
                # a similarity query batch (rsd_db_similarity_batch) with a random query count and RSD_SIM_QBATCH, top-k too
                n = int(rng.choice([1, 40, 400, 5000]))
                lens = rng.integers(0, int(rng.choice([8, 40, 300])), size=n)
                cd, od = make(rng, lens, alpha)
                docs = [O.decode(cd[od[k]:od[k + 1]]) for k in range(n)]
                nq = int(rng.integers(1, 80))
                cq, oq = make(rng, rng.integers(0, 40, size=nq), alpha)
                queries = [O.decode(cq[oq[q]:oq[q + 1]]) for q in range(nq)]
                method = str(rng.choice(IO.METHODS))
                k = int(rng.choice([0, 1, 7, 128]))
                bits = 2 if (set(alpha) <= set("AGCU") and rng.random() < 0.5) else 4
                knobs = {"RSD_SIM_QBATCH": str(int(rng.integers(1, 20)))} if rng.random() < 0.7 else {}
                eng.db_load(R.pack((cd, od), bits=bits))
                os.environ.update(knobs)
                try:
                    alls, idx, sc = eng.db_similarity_batch((cq, oq), method, k)
                finally:
                    for kname in knobs: del os.environ[kname]
                    eng.db_free()
                dreps = [IO.represent(d2, method) for d2 in docs]
                ok = alls.shape == (nq, n)
                for q in range(nq):
                    qa = IO.represent(queries[q], method)
                    want = np.zeros(n)
                    for k2, d2 in enumerate(dreps):
                        try:
                            want[k2] = IO.score(method, qa, d2)
                        except ZeroDivisionError:              # set measures of two empty sequences: the device returns NaN
                            want[k2] = np.nan
                    ok = ok and bool(np.array_equal(np.isnan(alls[q]), np.isnan(want))
                                     and np.array_equal(alls[q][~np.isnan(want)].view(np.uint64), want[~np.isnan(want)].view(np.uint64)))
                    valid = np.flatnonzero(~np.isnan(want))
                    top = valid[np.argsort(-want[valid], kind="stable")][:k]
                    wi = np.full(k, -1, np.int64); ws = np.zeros(k); wi[:top.shape[0]] = top; ws[:top.shape[0]] = want[top]
                    ok = ok and np.array_equal(idx[q], wi) and np.array_equal(sc[q], ws)
                desc = f"simb n={n} q={nq} method={method} k={k} bits={bits} knobs={knobs}"
            elif what == "long":
                m, n2 = int(rng.integers(1, 5000)), int(rng.integers(1, 5000))
                al = np.array([SYM.index(ch) for ch in alpha], np.uint8)
                a1 = al[rng.integers(0, len(al), size=m)]
                if rng.random() < 0.5:                           # homologous: the interesting tie structure
                    keep = rng.random(m) > 0.03
                    b1 = a1[keep].copy()
                    hit = rng.random(b1.shape[0]) < 0.05
                    b1[hit] = al[rng.integers(0, len(al), size=int(hit.sum()))]
                    if b1.shape[0] == 0:
                        b1 = a1[:1].copy()
                else:
                    b1 = al[rng.integers(0, len(al), size=n2)]
                # second-generation path with random planner knobs: rings, panel width, a memory budget / CTA limit that
                # forces the row-block x panel-range overflow path, a widened steps field (modular-key wrap regime)
                knobs = {}
                if rng.random() < 0.5: knobs["RSD_LONG_C"] = str(rng.choice([4, 8, 16]))
                if rng.random() < 0.4: knobs["RSD_LONG_BUDGET_MB"] = str(rng.choice([2, 3, 6]))
                if rng.random() < 0.3: knobs["RSD_LONG_MAXCTAS"] = str(rng.choice([1, 2, 7]))
                if rng.random() < 0.3: knobs["RSD_LONG_S"] = str(rng.choice([18, 20, 21]))
                if rng.random() < 0.3: knobs["RSD_LONG_RINGS"] = str(rng.choice([1, 2, 3]))
                os.environ.update(knobs)
                try:
                    fm = force if force != 2 else 0
                    if rng.random() < 0.5:
                        res = eng.long_pair(a1, b1, force_mode=fm)
                        extra = []
                    else:                                        # a batch: this pair plus two short companions
                        comp = [(al[rng.integers(0, len(al), size=int(rng.integers(0, 900)))], al[rng.integers(0, len(al), size=int(rng.integers(0, 900)))]) for _ in range(2)]
                        out = eng.long_pairs([(a1, b1)] + comp, force_mode=fm)
                        res, extra = out[0], list(zip(out[1:], comp))
                finally:
                    for kname in knobs: del os.environ[kname]
                ops, oi, oj, d = O.canonical_script(O.decode(a1), O.decode(b1), costs)
                ok = res["dist"] == d and np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)
                for r2, (a2, b2) in extra:
                    if a2.shape[0] == 0 or b2.shape[0] == 0:
                        ok = ok and r2["op"].shape[0] == a2.shape[0] + b2.shape[0]
                        continue
                    o2, i2, j2, d2 = O.canonical_script(O.decode(a2), O.decode(b2), costs)
                    ok = ok and r2["dist"] == d2 and np.array_equal(r2["op"], o2) and np.array_equal(r2["oi"], i2) and np.array_equal(r2["oj"], j2)
                cells += float(m) * b1.shape[0]
                desc = f"long {m}x{b1.shape[0]} mode={eng.last_mode} knobs={knobs} batch={len(extra) + 1}"
            elif what == "range":
                n = int(rng.choice([1, 50, 3000, 40000]))
                lens = rng.integers(0 if rng.random() < 0.3 else 20, int(rng.choice([32, 33, 60])), size=n)
                cd, od = make(rng, lens, alpha)
                nq = int(rng.choice([1, 3, 70]))
                ql = rng.integers(1, int(rng.choice([32, 65])), size=nq)
                cq, oq = make(rng, ql, alpha)
                D = np.stack([O.distance_batch(np.tile(cq[oq[q]:oq[q + 1]], n), np.arange(n + 1, dtype=np.int64) * int(ql[q]), cd, od, costs)
                              for q in range(nq)])
                # the bound from the oracle's own distances: an occurring D, the double below it, 0 or inf
                v = float(rng.choice(D.ravel()))
                bound = [v, float(np.nextafter(v, -np.inf)) if v > 0 else 0.0, 0.0, float("inf")][int(rng.choice([0, 0, 1, 1, 2, 3]))]
                eng.db_load(R.pack((cd, od), bits=4))
                try:
                    off, idx, dist = eng.db_search_range(R.pack((cq, oq), bits=4), bound, force_mode=0 if force == 2 else force)
                finally:
                    eng.db_free()
                ok = off[0] == 0
                for q in range(nq):
                    w = np.flatnonzero(D[q] <= bound)
                    ok = ok and np.array_equal(idx[off[q]:off[q + 1]], w) and np.array_equal(dist[off[q]:off[q + 1]], D[q, w])
                cells += float(ql.sum()) * float(lens.sum())
                desc = f"range n={n} q={nq} max_dist={bound!r} hits={int(off[-1])} mode={eng.last_mode}"
            elif what == "append":
                # a collection split at random into a load and 1-3 appends (some empty, some of other alphabets, so the
                # tiers move); everything compared with a fresh load of the whole collection
                n = int(rng.choice([1, 50, 3000, 40000]))
                lens = rng.integers(0 if rng.random() < 0.3 else 20, int(rng.choice([32, 33, 60])), size=n)
                cuts = np.sort(rng.integers(0, n + 1, size=int(rng.integers(1, 4))))
                bounds = [0, *cuts.tolist(), n]
                parts = [make(rng, lens[a:b], alpha if rng.random() < 0.7 else str(rng.choice([SYM, "ACGUYR", "YR", SYM[:4] + "N"])))
                         for a, b in zip(bounds[:-1], bounds[1:])]
                cd = np.concatenate([c for c, _ in parts]); od = np.zeros(n + 1, np.int64); np.cumsum(lens, out=od[1:])
                nq = int(rng.integers(1, 5)); k = int(rng.choice([1, 6, 10, 128]))
                ql = rng.integers(1, int(rng.choice([32, 65])), size=nq)
                cq, oq = make(rng, ql, alpha)
                Qp = R.pack((cq, oq), bits=4)
                method = str(rng.choice(IO.METHODS))
                ref = ref or R.Engine(0)                        # the fresh load
                ref.set_costs(costs)
                idf_first = rng.random() < 0.5
                bound = float(rng.choice([1.0, 4.0, np.inf]))
                got, want = [], []
                for e, pieces in ((eng, parts), (ref, [(cd, od)])):
                    e.db_load(R.pack(pieces[0], bits=4))
                    try:
                        if idf_first:
                            e.db_idf_table()
                        for p in pieces[1:]:
                            e.db_append(R.pack(p, bits=4))
                        out = [e.db_layout(), e.db_search_topk(Qp, k, want_scores=True), e.db_search_range(Qp, bound),
                               e.db_similarity_batch([cq[oq[q]:oq[q + 1]] for q in range(nq)], method, k=10)]
                        if method in IO.METHODS[6:]:
                            out.append(e.db_similarity_batch([cq[oq[q]:oq[q + 1]] for q in range(nq)], method, k=10, vector_type="tf-idf"))
                            out.append(e.db_idf_table())
                    finally:
                        e.db_free()
                    (got if e is eng else want).append(out)
                flat = lambda xs: [np.asarray(a) for x in xs for y in x for a in (y if isinstance(y, tuple) else (y,)) if a is not None]
                fg, fw = flat(got[0]), flat(want[0])
                diff = [i for i, (a, b) in enumerate(zip(fg, fw)) if a.shape != b.shape or a.tobytes() != b.tobytes()]
                ok = len(fg) == len(fw) and not diff
                cells += float(ql.sum()) * float(lens.sum())
                desc = (f"append n={n} parts={[b - a for a, b in zip(bounds[:-1], bounds[1:])]} q={nq} k={k} {method} "
                        f"idf_first={idf_first} max_dist={bound}" + (f" differing outputs {diff}" if diff else ""))
            else:
                n = int(rng.choice([1, 50, 3000, 40000]))
                lens = rng.integers(0 if rng.random() < 0.3 else 20, int(rng.choice([32, 33, 60])), size=n)
                cd, od = make(rng, lens, alpha)
                nq = int(rng.integers(1, 5)); k = int(min(rng.choice([1, 6, 10, 50]), max(n, 1)))
                ql = rng.integers(1, int(rng.choice([32, 65, 90])), size=nq)
                cq, oq = make(rng, ql, alpha)
                eng.db_load(R.pack((cd, od), bits=4))
                try:
                    idx, sc, alls = eng.db_search_topk(R.pack((cq, oq), bits=4), k, want_scores=True)
                finally:
                    eng.db_free()
                ok = True
                for q in range(nq):
                    wi, ws, wall = O.search_topk(O.decode(cq[oq[q]:oq[q + 1]]), cd, od, costs, k, want_scores=True)
                    ok = ok and np.array_equal(idx[q, :len(wi)], wi) and np.array_equal(sc[q, :len(ws)], ws) and np.array_equal(alls[q], wall)
                cells += float(ql.sum()) * float(lens.sum())
                desc = f"search n={n} q={nq} k={k} mode={eng.last_mode}"
        except R.RsdError as e:
            ok, desc = True, f"{what} rejected: {e}"             # e.g. a forced mode the costs do not allow
        bad += 0 if ok else 1
        print(f"[{rounds:4d}] {'ok ' if ok else 'BAD'} alpha={alpha:<15} costs={ckind:<8} len={lkind:<6} force={force} {desc}", flush=True)
    print(json.dumps({"rounds": rounds, "mismatches": bad, "cells_checked": cells, "seed": args.seed}))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
