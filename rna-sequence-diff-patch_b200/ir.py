"""ir.py — the search side of the reference's IRMethods.py on top of the CUDA engine.

Mirrors: wf_score IR:435-440, the wf_score branch of search_collection IR:443-447,466-477 (one
batched GPU scan of the collection instead of one wagnerFisher call per document), and the
stable descending top-k of performance.py:12-15 / gui.py:573,593; every document within a distance bound
(range_collection, which the reference lacks); and the other scorers of
search_collection — set / multiset / TF-vector measures, IR:49-389 — as one GPU pass over the collection
(similarity_collection)."""
from __future__ import annotations

import weakref
from operator import itemgetter

import numpy as np

from . import sed
from .encoding import pack
from .engine import get_search_engine


def wf_score(seq1: str, seq2: str, costs: dict) -> float:
    """IR:435-440: 1 / (1 + D[m][n])."""
    return 1 / (1 + sed.distance(seq1, seq2, costs))


def _validate_collection(query: str, sequences, costs: dict):
    """The reference raises KeyError for the first (document, row symbol, column symbol) whose update cost is not in
    the table (SED:87 through IR:437).  One pass over the distinct symbols of the whole collection decides whether
    any document can fail; only then is the per-document check (which finds the reference's first error) run."""
    upd = costs["update"]
    doc_syms = set().union(*map(set, sequences)) if len(sequences) < 64 else set("".join(sequences))
    clean = True
    for c1 in set(query):
        row = upd.get(c1)
        for c2 in doc_syms:
            if c2.lower() != c1.lower() and (row is None or c2 not in row):
                clean = False
    if not clean:
        for s in sequences:
            sed._validate_and_encode(query, s, costs)


class _Resident:
    """The collection each engine holds, as loaded by score_collection / range_collection / similarity_collection: a
    session that searches the same collection again (gui.py:532-600: every search re-reads collection.find({})) pays
    rsd_db_load once per engine.  The copy is keyed on its content (the documents after the case rule of the measure
    that loaded them), so wf_score (upper case) and the other measures (as stored) share it when the collection has no
    lower-case letters.  A collection that only grew (gui.py's imports, fa_import.py: records added at the end) has its
    new documents appended to the held copy instead of being reloaded."""
    held = weakref.WeakKeyDictionary()      # engine -> (load generation, documents as given, upper, documents as loaded)

    @classmethod
    def load(cls, eng, sequences, upper: bool):
        h = cls.held.get(eng)
        if h is not None and h[0] == getattr(eng, "_db_gen", 0) and h[2] == upper and h[1] == sequences:
            return
        content = _upper(sequences) if upper else sequences
        if h is not None and h[0] == getattr(eng, "_db_gen", 0):
            if h[3] == content:
                return
            n = len(h[3])
            if n < len(content) and content[:n] == h[3]:
                eng.db_append(pack(content[n:], bits=4))
                cls.held[eng] = (eng._db_gen, sequences, upper, content)
                return
        cls.held.pop(eng, None)
        eng.db_load(pack(content, bits=4))
        cls.held[eng] = (eng._db_gen, sequences, upper, content)

    @classmethod
    def drop(cls):
        for eng, (gen, *_) in list(cls.held.items()):
            if gen == getattr(eng, "_db_gen", 0):
                eng.db_free()
        cls.held.clear()


def _upper(sequences):
    return [s.upper() for s in sequences]


def release_collection():
    """Free the device copies of the collection kept by the searches (optional; the next search reloads)."""
    _Resident.drop()


def score_collection(query: str, sequences, costs: dict, engine=None):
    """[(sequence, wf_score(query, sequence))] in collection order — what
    search_collection(query, _, collection, wf_score) returns (IR:469-477): one pass over the collection, sharded
    over every visible GPU (one process, NCCL gather of the top-k lists; the per-document scores come back per shard)."""
    sequences = list(sequences)
    if not sequences:
        return []
    eng = engine or get_search_engine()
    eng.set_costs(costs)
    _validate_collection(query, sequences, costs)
    _Resident.load(eng, sequences, upper=True)
    _, _, scores = eng.db_search_topk(pack([query.upper()], bits=4), k=1, want_scores=True)
    return [(s, float(v)) for s, v in zip(sequences, scores[0])]


def range_collection(query: str, sequences, max_dist: float, costs: dict, engine=None):
    """[(index, sequence, D)] for every sequence of the collection with D = distance(query, sequence) <= max_dist
    (inclusive), in collection order — the wf_score scan of search_collection (IR:466-477) filtered on the distance
    instead of ranked, with D exact rather than recovered from 1 / (1 + D)."""
    sequences = list(sequences)
    if not sequences:
        return []
    eng = engine or get_search_engine()
    eng.set_costs(costs)
    _validate_collection(query, sequences, costs)
    _Resident.load(eng, sequences, upper=True)
    _, idx, dist = eng.db_search_range(pack([query.upper()], bits=4), max_dist)
    return [(int(i), sequences[i], float(d)) for i, d in zip(idx, dist)]


SIM_METHODS = ("set_intersection_similarity", "set_jaccard_similarity", "set_dice_similarity",
               "multi_intersection_similarity", "multi_jaccard_similarity", "multi_dice_similarity",
               "cosine", "pearson", "euclidian_distance", "manhattan_distance", "tanimoto_distance", "dice_dist")


def similarity_collection(query: str, sequences, method: str, engine=None, vector_type: str = "tf"):
    """[(sequence, method(query, sequence))] in collection order for one of SIM_METHODS — what
    search_collection(query, vector_type, collection, <method>) returns (IR:449-477), one GPU pass.  The documents'
    stored 'tf' vectors are rebuilt from the sequences on the device (they are convert_to_tf_vector(sequence),
    fa_import.py:49).  vector_type 'idf' / 'tf-idf' (the six vector measures only; IR:458-465) scores the idf / tf-idf
    vectors of IR:189-225 over these sequences as the whole collection.  Unknown symbols raise KeyError (the reference:
    KeyError IR:106 / ValueError IR:155).  Sharded over every visible GPU like score_collection."""
    if method not in SIM_METHODS:
        raise ValueError(f"unknown similarity method {method!r}")
    if vector_type not in ("tf", "idf", "tf-idf"):
        raise ValueError(f"unknown vector type {vector_type!r}")
    if method not in SIM_METHODS[6:]:
        vector_type = "tf"               # the set / multiset measures have no vector type (IR:449-454)
    sequences = list(sequences)
    if not sequences:
        return []
    from .encoding import encode
    eng = engine or get_search_engine()
    qc = encode(query)
    _Resident.load(eng, sequences, upper=False)
    scores, _, _ = eng.db_similarity(qc, method, vector_type=vector_type)
    return [(s, float(v)) for s, v in zip(sequences, scores)]


def top_k(scores, k):
    """performance.py:12-15 — stable, so ties keep collection order."""
    return sorted(scores, key=itemgetter(1), reverse=True)[0:k]
