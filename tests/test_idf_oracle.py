"""The host restatement of the idf / tf-idf search (tests/_idf_oracle.py) against measures.py and the reference's
recorded vectors and scores (CPU only)."""
import json
import math
import os
import random

import numpy as np
import pytest

import _idf_oracle as IDF
from oracle import ir_oracle as IO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VECTOR_METHODS = IO.METHODS[6:]


@pytest.fixture(scope="module")
def gir():
    with open(os.path.join(ROOT, "tests", "golden", "ref_golden_ir.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def M():
    from rna_sequence_diff_patch_b200 import measures
    return measures


def unhex(xs):
    return np.array([math.nan if x == "nan" else float.fromhex(x) for x in xs], dtype=np.float64)


def same_bits(a, b):
    a, b = np.asarray(a, np.float64).reshape(-1), np.asarray(b, np.float64).reshape(-1)
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def test_golden_vectors_and_scores(gir):
    small = gir["idf_docs"]
    _, idf = IDF.table(small)
    for s, v in gir["idf"].items():
        assert same_bits(IDF.idf_vector(s, idf), unhex(v)), s
    for key, rec in gir["idf_pairlist"].items():
        a, b = key.split("|")
        _, t = IDF.table([a, b])
        assert same_bits(IDF.idf_vector(a, t), unhex(rec["idf_a"]))
        assert same_bits(IDF.vectors([a], "tf-idf", t), unhex(rec["tfidf_a"]))
        assert same_bits(IDF.vectors([b], "tf-idf", t), unhex(rec["tfidf_b"]))
    for q, per_vt in gir["idf_scores"].items():
        for vt, per_m in per_vt.items():
            for name, want in per_m.items():
                assert same_bits(IDF.search([q], small, vt, name, idf)[0], unhex(want)), (q, vt, name)


def test_values_table_and_scores_match_measures(M):
    rnd = random.Random(11)
    docs = []
    for _ in range(60):                                   # mostly ACGU with ambiguity codes, some all-IUPAC, short ones
        s = rnd.choices(IO.SYMBOLS[:4], k=rnd.randint(0, 40))
        for _ in range(rnd.randint(0, 3)):
            if s:
                s[rnd.randrange(len(s))] = rnd.choice(IO.SYMBOLS[4:])
        docs.append("".join(s))
    docs += ["".join(rnd.choices(IO.SYMBOLS, k=n)) for n in (1, 2, 9, 30)] + ["NNNN", ""]
    V = IDF.values(docs)
    for j, d in enumerate(docs[::7]):
        for p in range(0, 225, 4):
            pair = IO.SYMBOLS[p // 15] + IO.SYMBOLS[p % 15]
            assert V[7 * j, p] == M.compare_pair_to_seq(pair, d, is_document=False), (pair, d)
    _, idf = IDF.table(docs)
    for s in docs[::5] + ["ACGUN", "YRWSKMDVHBN"]:             # the last two: bigrams with df == 0
        assert same_bits(IDF.idf_vector(s, idf), M.convert_to_idf_vector(s, list_of_docs=docs)), s
    for vt in ("idf", "tf-idf"):
        B = IDF.vectors(docs, vt, idf)
        for q in ("ACGUACGGA", "NRYAC"):
            a = IDF.vectors([q], vt, idf)[0]
            for name in VECTOR_METHODS:
                want = [IO.score(name, a, b) for b in B]
                assert same_bits(IDF.scores(name, a, B), want), (vt, q, name)


def test_fused_chain_is_not_the_plain_product():
    """The restatement's tf-idf is the fused chain: on these vectors it differs from a multiply-then-add chain"""
    rnd = random.Random(5)
    docs = ["".join(rnd.choices(IO.SYMBOLS, k=rnd.randint(2, 200))) for _ in range(50)]
    _, idf = IDF.table(docs)
    tf = np.stack([IO.tf_vector(s) for s in docs]); iv = np.stack([IDF.idf_vector(s, idf) for s in docs])
    fused = IDF.dot_fma(tf, iv)
    plain = np.zeros_like(fused)
    for r in range(len(docs)):
        for i in range(15):
            for j in range(15):
                acc = 0.0
                for k in range(15):
                    acc = acc + tf[r, i, k] * iv[r, k, j]
                plain[r, i, j] = acc
    assert not np.array_equal(fused, plain)
    assert np.allclose(fused, plain, rtol=1e-14, atol=0)


def test_table_of_codes_equals_table_of_strings():
    rnd = random.Random(3)
    docs = ["".join(rnd.choices(IO.SYMBOLS[:4] if i % 5 else IO.SYMBOLS, k=rnd.randint(0, 30))) for i in range(3000)]
    codes = np.array([c for d in docs for c in IO.codes_of(d)], np.uint8)
    off = np.zeros(len(docs) + 1, np.int64); np.cumsum([len(d) for d in docs], out=off[1:])
    want = IDF.table(docs)
    got = IDF.table_codes(codes, off, chunk=700)
    assert same_bits(got[0], want[0]) and same_bits(got[1], want[1])
