"""Batched and multi-GPU similarity search (rsd_db_similarity_batch, rsd_multi_db_similarity): every row of a query
batch equals the single-query search bit for bit, on every database layout, query batch size, chunk boundary and shard
layout the host path produces; the drop-in session shares one resident copy between wf_score and the other measures.
Every comparison is `==` on the bits, NaN where NaN is expected."""
import json
import math
import os

import numpy as np
import pytest

from oracle import ir_oracle as IO
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KMAX = 128                     # RSD_TOPK_MAX
SEED = 4096                    # the seed chunk of the similarity top-k
MAIN = 1 << 20                 # its main chunk
SET_METHODS = ["set_intersection_similarity", "set_jaccard_similarity", "set_dice_similarity"]
VECTOR_METHODS = ["cosine", "pearson", "euclidian_distance", "manhattan_distance", "tanimoto_distance", "dice_dist"]
RSD_EINVAL = 1


@pytest.fixture(scope="module")
def R():
    import __graft_entry__ as G
    G.build()
    import rna_sequence_diff_patch_b200 as R
    assert R.load_library().rsd_device_count() > 0
    return R


@pytest.fixture(scope="module")
def eng(R):
    return R.Engine(0)


@pytest.fixture(scope="module")
def gir():
    with open(os.path.join(ROOT, "tests", "golden", "ref_golden_ir.json")) as f:
        return json.load(f)


def unhex(xs):
    return np.array([math.nan if x == "nan" else float.fromhex(x) for x in xs], dtype=np.float64)


def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def oracle_rows(queries, docs, method):
    """ir_oracle scores, one row per query; the set measures of two empty sequences (0 / 0 in Python: the reference
    raises) are NaN, as on the device"""
    reps = [IO.represent(d, method) for d in docs]
    out = np.zeros((len(queries), len(docs)))
    for q, query in enumerate(queries):
        a = IO.represent(query, method)
        for j, b in enumerate(reps):
            try:
                out[q, j] = IO.score(method, a, b)
            except ZeroDivisionError:
                out[q, j] = math.nan
    return out


def topk_of(scores, k):
    """Per row: the first k of the stable descending sort of the non-NaN scores, padded with index -1 / score 0.0"""
    scores = np.atleast_2d(scores)
    idx = np.full((scores.shape[0], k), -1, np.int64)
    sc = np.zeros((scores.shape[0], k), np.float64)
    for q, row in enumerate(scores):
        valid = np.flatnonzero(~np.isnan(row))
        top = valid[np.argsort(-row[valid], kind="stable")][:k]
        idx[q, :top.shape[0]] = top
        sc[q, :top.shape[0]] = row[top]
    return idx, sc


def single_rows(R, eng, queries, method, k=0):
    """Engine.db_similarity query by query -> (scores [Q, n], idx [Q, k], score [Q, k])"""
    rows = [eng.db_similarity(R.encode(q), method, k=k) for q in queries]
    return np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows]), np.stack([r[2] for r in rows])


class qbatch:
    """RSD_SIM_QBATCH for the duration of a block"""
    def __init__(self, v): self.v = v
    def __enter__(self): os.environ["RSD_SIM_QBATCH"] = str(self.v)
    def __exit__(self, *a): del os.environ["RSD_SIM_QBATCH"]


# ---------------------------------------------------------------------------------------------------------------------
# the reference's recorded scores and the oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_golden_queries_in_one_batch(R, eng, gir):
    eng.db_load(R.pack(gir["docs"], bits=4))
    try:
        for method in IO.METHODS:
            alls, idx, sc = eng.db_similarity_batch([R.encode(q) for q in gir["queries"]], method, k=5)
            assert alls.shape == (len(gir["queries"]), len(gir["docs"]))
            for q, query in enumerate(gir["queries"]):
                want = unhex(gir["scores"][query][method])
                assert same_bits(alls[q], want), (query, method)
                wi, ws = topk_of(want, 5)
                assert np.array_equal(idx[q], wi[0]) and same_bits(sc[q], ws[0]), (query, method)
    finally:
        eng.db_free()


def test_layouts_and_awkward_queries_match_oracle_and_single_calls(R, eng):
    """2-bit ACGU, 4-bit IUPAC and mixed databases; the batch holds an empty query, a one-symbol query and an
    ambiguity-heavy one among ordinary ones"""
    rng = np.random.default_rng(41)
    acgu = ["".join(rng.choice(list("AGCU"), size=int(L))) for L in rng.integers(0, 70, size=300)]
    iupac = ["".join(rng.choice(list(IO.SYMBOLS), size=int(L))) for L in rng.integers(0, 50, size=300)]
    for docs, bits in ((acgu, 2), (iupac, 4), (acgu + iupac, 4)):
        queries = ["", "G", "NNRYKMSWBDHVNRY", docs[3], docs[17], "ACGUNNRY" * 4]
        eng.db_load(R.pack(docs, bits=bits))
        try:
            for method in IO.METHODS:
                alls, idx, sc = eng.db_similarity_batch((np.concatenate([R.encode(q) for q in queries]),
                                                         np.cumsum([0] + [len(q) for q in queries])), method, k=9)
                s_all, s_idx, s_sc = single_rows(R, eng, queries, method, k=9)
                assert same_bits(alls, s_all) and np.array_equal(idx, s_idx) and same_bits(sc, s_sc), (method, bits)
                assert same_bits(alls, oracle_rows(queries, docs, method)), (method, bits)
        finally:
            eng.db_free()


def test_empty_query_scores(R, eng):
    """an empty query gives what rsd_db_similarity gives: 0 for the set measures, NaN for the vector measures"""
    docs = ["ACGU", "G", "NNRA"]
    eng.db_load(R.pack(docs, bits=4))
    try:
        alls, _, _ = eng.db_similarity_batch([np.zeros(0, np.uint8), R.encode("AG")], "set_jaccard_similarity")
        assert np.array_equal(alls[0], np.zeros(3))
        alls, _, _ = eng.db_similarity_batch([np.zeros(0, np.uint8)], "cosine")
        assert np.isnan(alls).all()
        alls, idx, sc = eng.db_similarity_batch([], "cosine", k=4)
        assert alls.shape == (0, 3) and idx.shape == (0, 4) and sc.shape == (0, 4)
    finally:
        eng.db_free()


def test_small_query_batches_equal_the_default(R, eng):
    """RSD_SIM_QBATCH=3: 100 queries in 34 passes, the last one partial, == one run with the default batch"""
    rng = np.random.default_rng(42)
    docs = ["".join(rng.choice(list("AGCUN"), size=int(L))) for L in rng.integers(0, 60, size=5000)]
    queries = [R.encode("".join(rng.choice(list("AGCUNRY"), size=int(L)))) for L in rng.integers(0, 40, size=100)]
    eng.db_load(R.pack(docs, bits=4))
    try:
        for method in ("set_dice_similarity", "multi_jaccard_similarity", "cosine", "pearson", "euclidian_distance"):
            want = eng.db_similarity_batch(queries, method, k=KMAX)
            with qbatch(3):
                got = eng.db_similarity_batch(queries, method, k=KMAX)
            assert same_bits(got[0], want[0]) and np.array_equal(got[1], want[1]) and same_bits(got[2], want[2]), method
            assert np.array_equal(want[1][17], eng.db_similarity(queries[17], method, k=KMAX)[1])
    finally:
        eng.db_free()


@pytest.mark.parametrize("bits", [2, 4])
def test_tf_hand_off_in_a_batch(R, eng, bits):
    """ACGU records of 60000 symbols (the last the per-thread kernel counts) and 60001 (the first it hands to the warp
    kernel), a 65537-symbol run, records of length 0 and 1 and (4 bit) ambiguity codes at either end"""
    rng = np.random.default_rng(60100 + bits)
    acgu = lambda n: "".join(rng.choice(list("ACGU"), size=n))
    docs = [acgu(60000), acgu(60001), "A" * 65537, "", "G", acgu(40), acgu(333)]
    if bits == 4:
        docs += ["R" + acgu(99), acgu(99) + "Y", "N" + acgu(5000), acgu(5000) + "D"]
    queries = [acgu(50), "A" * 40, "ACGUNRYACGUACGUSWKM" + acgu(20), "", "C"]
    eng.db_load(R.pack(docs, bits=bits))
    try:
        for m in VECTOR_METHODS:
            alls, _, _ = eng.db_similarity_batch([R.encode(q) for q in queries], m)
            assert same_bits(alls, oracle_rows(queries, docs, m)), (m, bits)
            assert same_bits(alls, single_rows(R, eng, queries, m)[0]), (m, bits)
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# top-k across the chunk boundaries
# ---------------------------------------------------------------------------------------------------------------------
def chunk_of(i):
    return 0 if i < SEED else 1 if i < SEED + MAIN else 2


def record_masks(codes, off):
    lens = np.diff(off)
    masks = np.zeros(lens.shape[0], np.int64)
    ne = lens > 0
    masks[ne] = np.bitwise_or.reduceat(np.left_shift(np.uint16(1), codes.astype(np.uint16)), off[:-1][ne])
    return masks


def test_topk_ties_cut_in_a_different_chunk_per_query(R, eng):
    """4096 + 2^20 + 50000 records, each holding A, C, G and U and at most one of Y, N, R: 200 + 10 + 0 Y records, 60 +
    100 + 0 N records and 20 + 30 + 150 R records in the seed, main and last chunk.  Query ACGU+Y, ACGU+N and ACGU+R
    score those records 1.0 under the set measures (the rest less), so the 128th and 129th best tie, and the cut falls
    in the seed chunk for the first query, in the main chunk for the second and in the last chunk for the third."""
    rng = np.random.default_rng(43)
    n = SEED + MAIN + 50_000
    lens = rng.integers(8, 17, size=n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    codes = rng.integers(0, 4, size=int(off[-1]), dtype=np.uint8)
    for c in range(4):
        codes[off[:-1] + c] = c
    spans = [np.arange(0, SEED), np.arange(SEED, SEED + MAIN), np.arange(SEED + MAIN, n)]
    free = [s.copy() for s in spans]
    for sym, counts in ((4, (200, 10, 0)), (14, (60, 100, 0)), (5, (20, 30, 150))):      # Y, N, R
        for ch, cnt in enumerate(counts):
            pick = rng.choice(free[ch], cnt, replace=False)
            free[ch] = np.setdiff1d(free[ch], pick)
            codes[off[pick] + 4] = sym
    queries = ["ACGUY" * 4, "ACGUN" * 4, "ACGUR" * 4]
    masks = record_masks(codes, off)
    uniq, inv = np.unique(masks, return_inverse=True)
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        for m in SET_METHODS[1:]:
            want = np.stack([np.array([IO.score(m, IO.set_mask(q), int(u)) for u in uniq], np.float64)[inv] for q in queries])
            cuts = []
            for q in range(3):
                ranked = topk_of(want[q], KMAX + 1)[0][0]
                assert want[q, ranked[KMAX - 1]] == want[q, ranked[KMAX]] == 1.0, (m, q)
                tied = np.flatnonzero(want[q] == 1.0)
                assert len({chunk_of(i) for i in tied}) >= 2, "the tied records must span two chunks"
                cuts.append(chunk_of(ranked[KMAX - 1]))
            assert cuts == [0, 1, 2], cuts
            wi, ws = topk_of(want, KMAX)
            alls, idx, sc = eng.db_similarity_batch([R.encode(q) for q in queries], m, k=KMAX)
            assert same_bits(alls, want), m
            assert np.array_equal(idx, wi) and same_bits(sc, ws), m
            for q in range(3):
                _, si, ss = eng.db_similarity(R.encode(queries[q]), m, k=KMAX, want_scores=False)
                assert np.array_equal(si, idx[q]) and same_bits(ss, sc[q]), (m, q)
    finally:
        eng.db_free()


def test_k_above_the_rankable_records_pads(R, eng):
    docs = ["", "ACGUAGG", "G", "CCCAAAUU", "", "GUGUGAC", "A", "ACGUNNRY", "UUAAC"]
    queries = ["ACGUUGCA", "G", "GGGAAAC"]
    eng.db_load(R.pack(docs, bits=4))
    try:
        for m in ("cosine", "pearson", "tanimoto_distance"):
            want = oracle_rows(queries, docs, m)
            alls, idx, sc = eng.db_similarity_batch([R.encode(q) for q in queries], m, k=12)
            wi, ws = topk_of(want, 12)
            assert same_bits(alls, want) and np.array_equal(idx, wi) and same_bits(sc, ws), m
            for q in range(len(queries)):
                n_ok = int(np.count_nonzero(~np.isnan(want[q])))
                assert n_ok < 12 and (idx[q, n_ok:] == -1).all() and (sc[q, n_ok:] == 0.0).all()
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# several shards: MultiEngine
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("devices,n_docs", [([0, 0, 0], 5000), ([0] * 8, 700)])
def test_multi_engine_equals_one_engine(R, eng, devices, n_docs):
    """contiguous shards on one GPU; with 8 shards of about 90 records every shard has fewer than k = 128 rankable
    records (and the records of length 0 and 1 are not rankable under the vector measures)"""
    rng = np.random.default_rng(44 + len(devices))
    docs = ["".join(rng.choice(list("AGCUNRY"), size=int(L))) for L in rng.integers(0, 40, size=n_docs)]
    queries = [R.encode(q) for q in (docs[5], "", "A", "ACGUNNRYACGU", docs[n_docs // 2])]
    P = R.pack(docs, bits=4)
    me = R.MultiEngine(devices)
    try:
        me.db_load(P)
        eng.db_load(P)
        try:
            for m in ("set_jaccard_similarity", "multi_dice_similarity", "cosine", "pearson", "manhattan_distance"):
                for k in (0, 10, KMAX):
                    want = eng.db_similarity_batch(queries, m, k=k)
                    got = me.db_similarity_batch(queries, m, k=k)
                    assert same_bits(got[0], want[0]) and np.array_equal(got[1], want[1]) and same_bits(got[2], want[2]), (m, k)
                alls, idx, sc = me.db_similarity(queries[0], m, k=7)
                w = eng.db_similarity(queries[0], m, k=7)
                assert same_bits(alls, w[0]) and np.array_equal(idx, w[1]) and same_bits(sc, w[2]), m
        finally:
            eng.db_free()
            me.db_free()
    finally:
        me.close()


def test_similarity_collection_on_a_multi_engine(R, gir):
    from rna_sequence_diff_patch_b200 import ir
    me = R.MultiEngine([0, 0])
    try:
        q = gir["queries"][0]
        for m in IO.METHODS:
            res = ir.similarity_collection(q, gir["docs"], m, engine=me)
            assert [s for s, _ in res] == gir["docs"]
            assert same_bits(np.array([v for _, v in res]), unhex(gir["scores"][q][m])), m
    finally:
        ir.release_collection()
        me.close()


# ---------------------------------------------------------------------------------------------------------------------
# the drop-in session: one resident copy for wf_score and the other measures
# ---------------------------------------------------------------------------------------------------------------------
def test_search_threads_load_the_collection_once(R, gir, golden, dropin, monkeypatch):
    from rna_sequence_diff_patch_b200 import engine as E
    from rna_sequence_diff_patch_b200 import ir
    docs = gir["docs"]
    assert all(d == d.upper() for d in docs)
    loads = []
    for cls in (E.Engine, E.MultiEngine):
        orig = cls.db_load
        monkeypatch.setattr(cls, "db_load", lambda self, db, *a, _o=orig, **kw: (loads.append(db.n), _o(self, db, *a, **kw))[1])
    IR = dropin.IR

    class Coll:
        def find(self, flt): return iter([{"sequence": s} for s in docs])
    q = gir["queries"][1]
    # what the callbacks receive: the wf_score list, and per sequence the NaN-skipping mean over the methods
    qc = O.encode(q)
    c, o = O.concat(docs)
    d = O.distance_batch(np.tile(qc, len(docs)), np.arange(len(docs) + 1, dtype=np.int64) * len(qc), c, o, golden["default_costs"])
    wf = [(s, 1 / (1 + float(x))) for s, x in zip(docs, d)]
    # Python floats, as the drop-in holds them: sum() adds exact floats with compensation, numpy scalars without
    per = [[(s, float(v)) for s, v in zip(docs, unhex(gir["scores"][q][m]))] for m in ("cosine", "set_jaccard_similarity")] + [wf]
    rows = [dict(p) for p in per]
    order = list(dict.fromkeys(docs))
    mean = []
    for s in order:
        vals = [r[s] for r in rows if r[s] == r[s]]
        mean.append((s, sum(vals) / len(vals) if vals else float("nan")))
    cwd = os.getcwd()
    os.chdir(dropin.cwd)
    try:
        ir.release_collection()
        for _ in range(2):
            got = {}
            IR.create_search_threads([IR.cosine, IR.set_jaccard_similarity, IR.wf_score], q, 'tf', Coll(),
                                     on_search_done=lambda r: got.__setitem__("mean", r), on_wf_done=lambda r: got.__setitem__("wf", r))
            assert got["wf"] == wf
            assert [s for s, _ in got["mean"]] == [s for s, _ in mean]
            assert same_bits(np.array([v for _, v in got["mean"]]), np.array([v for _, v in mean]))
    finally:
        os.chdir(cwd)
        ir.release_collection()
    assert loads == [len(docs)], loads


# ---------------------------------------------------------------------------------------------------------------------
# arguments
# ---------------------------------------------------------------------------------------------------------------------
def test_argument_errors(R, eng):
    import ctypes as C
    lib = R.load_library()
    i64p, f64p, u8p = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_uint8)
    eng.db_load(R.pack(["ACGU", "GGA"], bits=4))
    me = R.MultiEngine([0, 0])
    try:
        me.db_load(R.pack(["ACGU", "GGA"], bits=4))
        for target in (eng, me):
            with pytest.raises(R.RsdError) as ei:
                target.db_similarity_batch([R.encode("AC")], "nope")
            assert ei.value.code == RSD_EINVAL
            for method, k in ((12, 0), (-1, 0), (0, KMAX + 1), (0, -1)):
                with pytest.raises(R.RsdError) as ei:
                    target.db_similarity_batch([R.encode("AC")], method, k=k)
                assert ei.value.code == RSD_EINVAL, (method, k)
            with pytest.raises(R.RsdError) as ei:
                target.db_similarity_batch((np.array([0, 15, 1], np.uint8), np.array([0, 3], np.int64)), "cosine")
            assert ei.value.code == RSD_EINVAL and "not a symbol" in str(ei.value)
            for off in ([0, 2, 1], [1, 2, 3], [0, -1, 3]):
                with pytest.raises(R.RsdError) as ei:
                    target.db_similarity_batch((np.array([0, 1, 2], np.uint8), np.array(off, np.int64)), "cosine")
                assert ei.value.code == RSD_EINVAL, off
        codes = np.array([0, 1], np.uint8); off = np.array([0, 2], np.int64)
        idx = np.zeros(4, np.int64); sc = np.zeros(4)
        for fn, h in ((lib.rsd_db_similarity_batch, eng.ctx), (lib.rsd_multi_db_similarity, me._h)):
            assert fn(h, codes.ctypes.data_as(u8p), off.ctypes.data_as(i64p), 1, 0, 4, None, None, None) == RSD_EINVAL
            assert fn(h, None, off.ctypes.data_as(i64p), 1, 0, 4, idx.ctypes.data_as(i64p), sc.ctypes.data_as(f64p), None) == RSD_EINVAL
            assert fn(h, None, None, 0, 0, 4, None, None, None) == 0                # no queries: nothing to do
    finally:
        eng.db_free()
        me.close()
