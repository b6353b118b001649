"""Similarity search over idf and tf-idf vectors (rsd_db_idf_table, rsd_db_vector_similarity_batch and their rsd_multi
forms): the document-frequency table equals the sequential sum in collection order, and every score equals the
reference's (golden file) or its host restatement (tests/_idf_oracle.py) bit for bit, NaN where NaN is expected."""
import json
import math
import os
import pickle

import numpy as np
import pytest

import _idf_oracle as IDF
from oracle import ir_oracle as IO

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VECTOR_METHODS = IO.METHODS[6:]
VTS = ("idf", "tf-idf")
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


def topk_of(scores, k):
    scores = np.atleast_2d(scores)
    idx = np.full((scores.shape[0], k), -1, np.int64)
    sc = np.zeros((scores.shape[0], k), np.float64)
    for q, row in enumerate(scores):
        valid = np.flatnonzero(~np.isnan(row))
        top = valid[np.argsort(-row[valid], kind="stable")][:k]
        idx[q, :top.shape[0]] = top
        sc[q, :top.shape[0]] = row[top]
    return idx, sc


def mixed_docs(n, seed):
    """mostly A/G/C/U records with ambiguity codes interleaved: store order (length, tier) != collection order"""
    rng = np.random.default_rng(seed)
    docs = []
    for i in range(n):
        s = rng.choice(list("AGCU"), size=int(rng.integers(20, 61)))
        if i % 7 == 3:
            for p in rng.integers(0, s.shape[0], size=int(rng.integers(1, 3))):
                s[p] = rng.choice(list(IO.SYMBOLS[4:]))
        docs.append("".join(s))
    return docs


def check_all(R, e, docs, queries, k=0, methods=VECTOR_METHODS):
    """every vector type x method against the oracle (scores, and top-k when k > 0)"""
    _, idf = IDF.table(docs)
    for vt in VTS:
        B, A = IDF.vectors(docs, vt, idf), IDF.vectors(queries, vt, idf)
        for method in methods:
            want = np.stack([IDF.scores(method, a, B) for a in A])
            alls, idx, sc = e.db_similarity_batch([R.encode(q) for q in queries], method, k=k, vector_type=vt)
            assert same_bits(alls, want), (vt, method)
            if k:
                wi, ws = topk_of(want, k)
                assert np.array_equal(idx, wi) and same_bits(sc, ws), (vt, method)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the reference's recorded vectors and scores
# ---------------------------------------------------------------------------------------------------------------------
def test_golden_table_and_scores_engine_and_multi(R, eng, gir):
    small = gir["idf_docs"]
    qs = list(gir["idf_scores"])
    me = R.MultiEngine([0, 0, 0])
    try:
        for e in (eng, me):
            e.db_load(R.pack(small, bits=4))
            df, idf = e.db_idf_table()
            for s, v in gir["idf"].items():
                assert same_bits(IDF.idf_vector(s, idf.reshape(-1)).reshape(-1), unhex(v)), s
            for vt in VTS:
                for method in VECTOR_METHODS:
                    alls, _, _ = e.db_similarity_batch([R.encode(q) for q in qs], method, vector_type=vt)
                    for j, q in enumerate(qs):
                        assert same_bits(alls[j], unhex(gir["idf_scores"][q][vt][method])), (type(e).__name__, q, vt, method)
            e.db_free()
    finally:
        me.close()


class _Coll:
    def __init__(self, docs): self.docs = docs
    def find(self, _): return iter(self.docs)
    def count_documents(self, _): return len(self.docs)


def test_golden_through_dropin_search_collection(R, gir):
    """documents as the importer writes them (stored 'tf', no 'idf'): the GPU path, the reference's scores"""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "rna-sequence-diff-patch_b200", "dropin"))
    import IRMethods as IR
    from rna_sequence_diff_patch_b200 import ir as _ir
    from rna_sequence_diff_patch_b200 import measures as M
    small = gir["idf_docs"]
    coll = _Coll([{"sequence": s, "tf": pickle.dumps(M.convert_to_tf_vector(s))} for s in small])
    calls = []
    real = _ir.similarity_collection
    _ir.similarity_collection = lambda *a, **kw: calls.append(kw.get("vector_type")) or real(*a, **kw)
    try:
        for q, per_vt in gir["idf_scores"].items():
            for vt, per_m in per_vt.items():
                for name, want in per_m.items():
                    res = IR.search_collection(q, vt, coll, getattr(IR, name))
                    assert [s for s, _ in res] == small
                    assert same_bits(np.array([v for _, v in res]), unhex(want)), (q, vt, name)
    finally:
        _ir.similarity_collection = real
        _ir.release_collection()
    assert calls and set(calls) == set(VTS)


# ---------------------------------------------------------------------------------------------------------------------
# 2. collection order decides the df bits
# ---------------------------------------------------------------------------------------------------------------------
def test_order_sensitive_table_and_scores(R, eng):
    docs = mixed_docs(20000, 3)
    df_want, idf_want = IDF.table(docs)
    qs = mixed_docs(64, 4)[:60] + ["ACGUN", "YRWSKMDVHBN", "", "A"]
    me = R.MultiEngine([0, 0, 0])
    try:
        for e in (eng, me):
            e.db_load(R.pack(docs, bits=4))
            df, idf = e.db_idf_table()
            assert same_bits(df.reshape(-1), df_want) and same_bits(idf.reshape(-1), idf_want), type(e).__name__
        # the check is meaningful: most sums differ from an order-free sum
        V = IDF.values(docs)
        assert sum(math.fsum(V[:, p]) != df_want[p] for p in range(225)) > 50
        check_all(R, eng, docs, qs, k=10)
        check_all(R, me, docs, qs[:8], k=10)
    finally:
        eng.db_free()
        me.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. shapes
# ---------------------------------------------------------------------------------------------------------------------
def test_awkward_records_both_packings(R, eng):
    rng = np.random.default_rng(9)
    acgu = ["".join(rng.choice(list("AGCU"), size=int(L))) for L in rng.integers(0, 50, size=200)]
    acgu += ["", "A", "G", "".join(rng.choice(list("AGCU"), size=60001))]              # thread path and worklist
    iupac = acgu[:150] + ["N", "NNNNNN", "NN", "".join(rng.choice(list(IO.SYMBOLS), size=61000))]
    iupac += ["".join(rng.choice(list(IO.SYMBOLS), size=int(L))) for L in rng.integers(0, 40, size=60)]
    qs = ["ACGUUGCA", "", "U", "NNYRW", "ACGUN" * 5, "".join(rng.choice(list(IO.SYMBOLS), size=30))]
    for docs, bits in ((acgu, 2), (acgu, 4), (iupac, 4)):
        eng.db_load(R.pack(docs, bits=bits))
        try:
            assert R.pack(docs, bits=bits).bits == bits
            check_all(R, eng, docs, qs, k=7)
        finally:
            eng.db_free()


def test_one_record_collection_is_never_ranked(R, eng):
    eng.db_load(R.pack(["ACGUAC"], bits=4))
    try:
        df, idf = eng.db_idf_table()
        own = IDF.presence("ACGUAC").reshape(15, 15)
        assert (df[own] == 1).all() and not idf[own].any()   # df = N at the record's own bigrams: its vectors are 0
        assert idf[~own].any()                                 # other bigrams have df 0 or < 1
        for vt in VTS:
            for method in ("cosine", "pearson"):               # 0 / 0 for every query
                alls, idx, sc = eng.db_similarity_batch([R.encode("ACGUAC"), R.encode("GGN")], method, k=3, vector_type=vt)
                assert np.isnan(alls).all() and (idx == -1).all(), (vt, method)
        check_all(R, eng, ["ACGUAC"], ["ACGUAC", "GGN"], k=3)
    finally:
        eng.db_free()


def test_topk_128_ties_qbatch_and_single_calls(R, eng):
    base = mixed_docs(300, 5)
    docs = [base[i % 40] for i in range(3000)]                 # many exact ties
    qs = [base[i] for i in range(0, 40, 4)] + ["NNNN"]
    eng.db_load(R.pack(docs, bits=4))
    try:
        check_all(R, eng, docs, qs, k=128)
        for vt in VTS:
            for method in VECTOR_METHODS:
                ref = eng.db_similarity_batch([R.encode(q) for q in qs], method, k=128, vector_type=vt)
                os.environ["RSD_SIM_QBATCH"] = "3"
                try:
                    got = eng.db_similarity_batch([R.encode(q) for q in qs], method, k=128, vector_type=vt)
                finally:
                    del os.environ["RSD_SIM_QBATCH"]
                assert same_bits(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and same_bits(got[2], ref[2])
                for j, q in enumerate(qs[:3]):
                    one = eng.db_similarity(R.encode(q), method, k=128, vector_type=vt)
                    assert same_bits(one[0], ref[0][j]) and np.array_equal(one[1], ref[1][j]) and same_bits(one[2], ref[2][j])
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# 4. the cached table follows the loaded database
# ---------------------------------------------------------------------------------------------------------------------
def test_table_follows_reload_and_free(R, eng):
    a, b = mixed_docs(500, 6), mixed_docs(700, 7)
    eng.db_load(R.pack(a, bits=4))
    eng.db_similarity_batch([R.encode(a[0])], "cosine", vector_type="idf")
    eng.db_load(R.pack(b, bits=4))
    df, idf = eng.db_idf_table()
    assert same_bits(df.reshape(-1), IDF.table(b)[0])
    check_all(R, eng, b, [a[0], b[1]], methods=["cosine"])
    eng.db_free()
    for call in (lambda: eng.db_idf_table(), lambda: eng.db_similarity_batch([R.encode("ACG")], "cosine", vector_type="tf-idf")):
        with pytest.raises(R.RsdError) as ei:
            call()
        assert ei.value.code == RSD_EINVAL
    eng.db_load(R.pack(a, bits=4), global_index_base=5)
    try:
        with pytest.raises(R.RsdError) as ei:
            eng.db_idf_table()
        assert ei.value.code == RSD_EINVAL and "global_index_base" in str(ei.value)
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# 5. emulated shards
# ---------------------------------------------------------------------------------------------------------------------
def test_multi_equals_single(R, eng):
    docs = mixed_docs(3000, 8) + ["", "N", "".join(["ACGU"] * 16000)]
    qs = [R.encode(q) for q in mixed_docs(12, 9) + ["YRN"]]
    eng.db_load(R.pack(docs, bits=4))
    try:
        want_t = eng.db_idf_table()
        want = {(vt, m): eng.db_similarity_batch(qs, m, k=20, vector_type=vt) for vt in VTS for m in VECTOR_METHODS}
    finally:
        eng.db_free()
    for devices in ([0, 0, 0], [0] * 8):
        me = R.MultiEngine(devices)
        try:
            me.db_load(R.pack(docs, bits=4))
            t = me.db_idf_table()
            assert same_bits(t[0], want_t[0]) and same_bits(t[1], want_t[1]), devices
            for (vt, m), w in want.items():
                got = me.db_similarity_batch(qs, m, k=20, vector_type=vt)
                assert same_bits(got[0], w[0]) and np.array_equal(got[1], w[1]) and same_bits(got[2], w[2]), (devices, vt, m)
        finally:
            me.close()


# ---------------------------------------------------------------------------------------------------------------------
# 6. argument errors
# ---------------------------------------------------------------------------------------------------------------------
def test_argument_errors(R, eng):
    import ctypes as C
    from rna_sequence_diff_patch_b200._lib import ptr
    eng.db_load(R.pack(["ACGU", "GGA"], bits=4))
    try:
        for kw in (dict(method="cosine", vector_type="bm25"), dict(method="cosine", vector_type=3),
                   dict(method="cosine", vector_type=-1), dict(method="set_jaccard_similarity", vector_type="idf"),
                   dict(method="multi_dice_similarity", vector_type="tf-idf"), dict(method="cosine", vector_type="idf", k=129),
                   dict(method="cosine", vector_type="idf", k=-1)):
            with pytest.raises(R.RsdError) as ei:
                eng.db_similarity_batch([R.encode("ACG")], **kw)
            assert ei.value.code == RSD_EINVAL, kw
        lib = R.load_library()
        codes = np.array([0, 1, 15], np.uint8); off = np.array([0, 3], np.int64)
        idx = np.zeros(1, np.int64); sc = np.zeros(1, np.float64)
        rc = lib.rsd_db_vector_similarity_batch(eng.ctx, ptr(codes, C.c_uint8), ptr(off, C.c_int64), 1, 1, 6, 1,
                                                ptr(idx, C.c_int64), ptr(sc, C.c_double), None)
        assert rc == RSD_EINVAL and b"not a symbol" in lib.rsd_last_error()
    finally:
        eng.db_free()
