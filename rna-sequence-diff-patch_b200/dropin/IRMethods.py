"""Drop-in for the reference's IRMethods.py (put this directory first on sys.path).

Every public name of the reference module exists here with the same signature, so its importers work
unchanged: gui.py:18-22 (21 names), timing.py:4 (`from IRMethods import *`), performance.py:3,
fa_import.py:5.  What runs where:

  * wf_score (IR:435-440) and search_collection (IR:443-477) with method == wf_score, a set / multiset
    measure, or a vector measure on the stored 'tf' vectors: ONE GPU pass over the collection (librsd.so).
  * the representations (convert_to_*) and the twelve measures called on ONE pair of pre-built sets /
    vectors (gui.py:455-500, timing.py): host objects by nature (Python sets, numpy arrays) —
    rna_sequence_diff_patch_b200/measures.py, same values as the reference.  A measure called on two
    SEQUENCES (str) scores that pair on the GPU instead.
  * search_collection with vector_type 'idf' / 'tf-idf' (IR:458-465) and a vector measure: ONE GPU pass too
    when every document is laid out as the reference's importer writes it -- a stored 'tf' vector and no stored
    'idf' (fa_import.py:30-36,49) -- the collection's document-frequency table is built on the device and the
    vectors are rebuilt from the sequences.  Any other collection keeps the host branch, like the reference:
    one with stored 'idf' vectors (only a caller's own update_idfs writes them, and they may be stale) is scored
    from those, and a document that lacks the stored 'idf' / 'tf' vector gets it computed from its sequence (the
    reference would raise KeyError there).
  * create_search_threads (IR:480-515): one GPU scan per method, no fork, no second WF pass, no pandas."""
import math  # noqa: F401  (module-level names of the reference module, visible to `from IRMethods import *`)
import os
import pickle
import sys
import time  # noqa: F401
from multiprocessing import Manager, Process  # noqa: F401
from operator import itemgetter  # noqa: F401

import numpy as np  # noqa: F401

try:
    import pandas as pd  # noqa: F401
except Exception:  # pragma: no cover - pandas is optional here (the reference needs it, IR:7)
    pd = None

_HERE = os.path.dirname(os.path.abspath(__file__))
if _HERE not in sys.path:
    sys.path.insert(0, _HERE)

import StringEditDistance as _SED  # noqa: E402  (the drop-in next to this file)
from StringEditDistance import wagnerFisher  # noqa: E402,F401
from rna_sequence_diff_patch_b200 import ir as _ir  # noqa: E402
from rna_sequence_diff_patch_b200 import measures as _m  # noqa: E402
from rna_sequence_diff_patch_b200.measures import (  # noqa: E402,F401
    ambiguity_vectors, ambiguous_nucleotides, base_nucleotides, compare_pair_to_seq, convert_to_idf_vector,
    convert_to_multi_set, convert_to_set, convert_to_tf_vector, create_and_start_threads, create_tf_idf_vector,
    get_base_possibilities, intersection, nucleotides, possibilities, time_method)


def wf_score(seq1, seq2, user_cost=False):
    return _ir.wf_score(seq1, seq2, _SED.user_costs if user_cost else _SED.default_costs)


def _measure(host_fn):
    """The object callers pass as `method`: pre-built sets / vectors -> the host measure (the reference's call,
    gui.py:462-500); two sequences -> that pair scored on the GPU."""
    name = host_fn.__name__

    def fn(a, b, return_dict=None):
        if isinstance(a, str) and isinstance(b, str):
            val = _ir.similarity_collection(a, [b], name)[0][1]
            if return_dict is None:
                return val
            return_dict[host_fn.return_key] = val
            return None
        return host_fn(a, b, return_dict)
    fn.__name__ = fn.__qualname__ = name
    fn.__doc__ = host_fn.__doc__
    fn.host = host_fn
    return fn


set_intersection_similarity = _measure(_m.set_intersection_similarity)
set_jaccard_similarity = _measure(_m.set_jaccard_similarity)
set_dice_similarity = _measure(_m.set_dice_similarity)
multi_intersection_similarity = _measure(_m.multi_intersection_similarity)
multi_jaccard_similarity = _measure(_m.multi_jaccard_similarity)
multi_dice_similarity = _measure(_m.multi_dice_similarity)
cosine = _measure(_m.cosine)
pearson = _measure(_m.pearson)
euclidian_distance = _measure(_m.euclidian_distance)
manhattan_distance = _measure(_m.manhattan_distance)
tanimoto_distance = _measure(_m.tanimoto_distance)
dice_dist = _measure(_m.dice_dist)
_SET_MULTI = (set_intersection_similarity, set_jaccard_similarity, set_dice_similarity,
              multi_intersection_similarity, multi_jaccard_similarity, multi_dice_similarity)
_VECTOR = (cosine, pearson, euclidian_distance, manhattan_distance, tanimoto_distance, dice_dist)


def perform_methods(a, b, do_cosine=False, do_pearson=False, do_euclidian_distance=False, do_manhattan_distance=False,
                    do_tanimoto_distance=False, do_dice_dist=False):
    """IR:421-432."""
    wanted = (do_cosine, do_pearson, do_euclidian_distance, do_manhattan_distance, do_tanimoto_distance, do_dice_dist)
    return create_and_start_threads([m for m, on in zip(_VECTOR, wanted) if on], a, b)


def _doc_vector(doc, key, build):
    return pickle.loads(doc[key]) if key in doc else build(doc['sequence'])


def search_collection(query, vector_type, collection, method, return_dict=None, callback=None):
    """IR:443-477.  wf_score always uses the default costs (IR:470)."""
    if method is wf_score:
        scores = _ir.score_collection(query, [doc['sequence'] for doc in collection.find({})], _SED.default_costs)
    elif method in _SET_MULTI or (method in _VECTOR and vector_type == 'tf'):
        scores = _ir.similarity_collection(query, [doc['sequence'] for doc in collection.find({})], method.__name__)
    elif method in _VECTOR and all('tf' in doc and 'idf' not in doc for doc in collection.find({})):
        scores = _ir.similarity_collection(query, [doc['sequence'] for doc in collection.find({})], method.__name__,
                                           vector_type='idf' if vector_type == 'idf' else 'tf-idf')
    elif method in _VECTOR:
        def idf_of(s):
            return convert_to_idf_vector(s, collection)
        if vector_type == 'idf':                                                   # IR:458-460
            vector1 = convert_to_idf_vector(query, collection)

            def convert(doc):
                return _doc_vector(doc, 'idf', idf_of)
        else:                                                                      # IR:461-464
            vector1 = create_tf_idf_vector(query, collection)

            def convert(doc):
                return np.dot(_doc_vector(doc, 'tf', convert_to_tf_vector), _doc_vector(doc, 'idf', idf_of))
        scores = [(doc['sequence'], method.host(vector1, convert(doc))) for doc in collection.find({})]
    else:
        # any other callable: the reference's generic loop over the stored 'tf' vectors (IR:455-457,466-470)
        vector1 = convert_to_tf_vector(query)
        scores = [(doc['sequence'], method(vector1, _doc_vector(doc, 'tf', convert_to_tf_vector)))
                  for doc in collection.find({})]
    if callback is not None:
        callback(scores)
    elif return_dict is not None:
        return_dict[method.__name__] = scores
    else:
        return scores


def create_search_threads(methods_to_execute, query, vector_type, collection, on_search_done=None, on_wf_done=None):
    """IR:480-515: one GPU scan of the collection per method instead of a forked process per method plus
    a second, separate WF pass (IR:487-491,511-515); no pandas (the reference's DataFrame.append, IR:501, no
    longer exists).  The callbacks receive what the reference passes them: a list of (sequence, mean score
    over the methods) — duplicates collapse like the reference's dict, the mean skips NaN like
    DataFrame.mean (IR:501-505) — and the raw wf_score list."""
    per_method = [search_collection(query, vector_type, collection, m) for m in methods_to_execute]
    if on_search_done is not None:
        order, rows = [], []
        seen = set()
        for scores in per_method:
            row = {}
            for seq, sc in scores:
                if seq not in seen:
                    seen.add(seq)
                    order.append(seq)
                row[seq] = sc
            rows.append(row)
        final = []
        for seq in order:
            vals = [r[seq] for r in rows if seq in r and r[seq] == r[seq]]
            final.append((seq, sum(vals) / len(vals) if vals else float('nan')))
        on_search_done(final)
    if wf_score in methods_to_execute and on_wf_done is not None:
        on_wf_done(per_method[list(methods_to_execute).index(wf_score)])


def top_k(scores, k):
    return _ir.top_k(scores, k)
