"""Engine — the Python face of librsd.so (include/rsd.h).

One Engine = one rsd_ctx = one GPU.  The CUDA context is created by the first compute call in
the calling process, so an Engine created before a fork() must not be used in the child:
get_engine() keeps one Engine per (pid, device)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import check, ptr
from .encoding import SYMBOLS, PackedSeqs, encode, pack

_f64, _i32, _i64, _u8, _u32 = C.c_double, C.c_int32, C.c_int64, C.c_uint8, C.c_uint32


def costs_to_arrays(costs: dict):
    """{'insert','delete','update':{src:{dst:cost}}} (costs.json, SED:6-18) -> (ins, del, sub[225]).
    Missing table entries stay 0; they are unreachable unless the caller feeds such symbols."""
    sub = np.zeros(225, dtype=np.float64)
    upd = costs["update"]
    for a, ch_a in enumerate(SYMBOLS):
        row = upd.get(ch_a)
        if row is None:
            continue
        for b, ch_b in enumerate(SYMBOLS):
            if a != b and ch_b in row:
                sub[a * 15 + b] = float(row[ch_b])
    return float(costs["insert"]), float(costs["delete"]), sub


def _db_query(Q: PackedSeqs, db_bits: int) -> PackedSeqs:
    """The repacking rule of the database searches: 2-bit queries go to 4 bits for a 4-bit database."""
    Q = Q.repack(db_bits) if Q.bits != db_bits and db_bits == 4 else Q
    if Q.bits != db_bits:
        raise ValueError("query symbols do not fit the database packing; reload the database with bits=4")
    return Q


def _sim_method(method) -> int:
    if isinstance(method, str):
        if method not in Engine.SIM_METHODS:
            raise _lib.RsdError(_lib.RSD_EINVAL, f"unknown similarity method {method!r}")
        return Engine.SIM_METHODS.index(method)
    return int(method)


def _sim_queries(queries):
    """A similarity query batch -> (codes uint8, offsets int64[q+1]): a (codes, offsets) tuple as pack takes it, or a
    list of code arrays (or of strings, encoded)."""
    if isinstance(queries, tuple):
        codes, off = queries
        return np.ascontiguousarray(codes, np.uint8), np.ascontiguousarray(off, np.int64)
    parts = [encode(x) if isinstance(x, str) else np.asarray(x, np.uint8).reshape(-1) for x in queries]
    off = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([p.shape[0] for p in parts], out=off[1:])
    codes = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    return np.ascontiguousarray(codes, np.uint8), off


VECTOR_TYPES = {"tf": 0, "idf": 1, "tf-idf": 2}          # search_collection's vector_type (IR:455-465); 1, 2 = RSD_VEC_*


def _vector_type(vector_type) -> int:
    if isinstance(vector_type, str):
        if vector_type not in VECTOR_TYPES:
            raise _lib.RsdError(_lib.RSD_EINVAL, f"unknown vector type {vector_type!r}")
        return VECTOR_TYPES[vector_type]
    return int(vector_type)


def _sim_entry(tf_fn, vec_fn, vector_type):
    """The entry point of a similarity batch: the 'tf' one, or the idf / tf-idf one with the vector type bound."""
    vt = _vector_type(vector_type)
    if vt == 0:
        return tf_fn
    return lambda h, codes, off, nq, method, k, idx, sc, alls: vec_fn(h, codes, off, nq, vt, method, k, idx, sc, alls)


def _idf_table(fn, h):
    """Calls rsd_db_idf_table / rsd_multi_db_idf_table -> (df [15, 15], idf [15, 15])."""
    df = np.zeros((15, 15), np.float64); idf = np.zeros((15, 15), np.float64)
    check(fn(h, ptr(df, _f64), ptr(idf, _f64)))
    return df, idf


def _similarity_batch(fn, h, db_n: int, queries, method, k: int, want_scores: bool):
    """Calls rsd_db_similarity_batch / rsd_multi_db_similarity -> (all_scores [q, n] | None, top_idx [q, k], top_score [q, k])."""
    codes, off = _sim_queries(queries)
    nq = off.shape[0] - 1
    cc = codes if codes.shape[0] else np.zeros(1, np.uint8)
    alls = np.zeros((nq, db_n), np.float64) if want_scores else None
    idx = np.full((nq, max(k, 1)), -1, np.int64); sc = np.zeros((nq, max(k, 1)), np.float64)
    check(fn(h, ptr(cc, _u8), ptr(off, _i64), nq, _sim_method(method), int(k), ptr(idx, _i64), ptr(sc, _f64),
             ptr(alls, _f64) if want_scores and db_n and nq else None))
    return alls, idx[:, :k], sc[:, :k]


def _search_range(fn, h, Q: PackedSeqs, max_dist: float, force_mode: int, guess: int):
    """Calls a range entry point (rsd_db_search_range / rsd_multi_db_search_range) with room for `guess` hits; when the
    hits do not fit (RSD_ERANGE, hit_off complete), once more with the exact total."""
    nq = Q.n
    off = np.zeros(nq + 1, np.int64)
    mode = C.c_int()
    for attempt in range(2):
        cap = max(int(guess), 1)
        idx = np.empty(cap, np.int64); dist = np.empty(cap, np.float64)
        rc = fn(h, ptr(Q.words, _u32), ptr(Q.start, _i64), ptr(Q.len, _i32), nq, Q.words.shape[0], Q.bits, Q.symmask,
                float(max_dist), force_mode, cap, ptr(off, _i64), ptr(idx, _i64), ptr(dist, _f64), C.byref(mode))
        if rc == _lib.RSD_ERANGE and attempt == 0:
            guess = int(off[nq])
            continue
        check(rc)
        total = int(off[nq])
        return (off, idx[:total], dist[:total]), mode.value


class Engine:
    def __init__(self, device: int = 0):
        self._lib = _lib.load_library()
        self._ctx = C.c_void_p()
        check(self._lib.rsd_create(device, C.byref(self._ctx)))
        self.device = device
        self.pid = os.getpid()
        self.last_mode = 0
        self._costs_key = None

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.rsd_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            if os.getpid() == self.pid:
                self.close()
        except Exception:
            pass

    # ---- costs ---------------------------------------------------------------------------------
    def set_costs(self, costs: dict):
        """Snapshot a cost dict (the reference reads its global dict at call time, SED:87,95-97)."""
        ins, dele, sub = costs_to_arrays(costs)
        key = (ins, dele, sub.tobytes())
        if key != self._costs_key:
            check(self._lib.rsd_set_costs(self._ctx, ins, dele, ptr(sub, _f64)))
            self._costs_key = key

    def classify(self, symmask: int, max_m: int, max_n: int, force_mode: int = 0):
        mode, k = C.c_int(), C.c_int()
        check(self._lib.rsd_classify(self._ctx, symmask, max_m, max_n, force_mode, C.byref(mode), C.byref(k)))
        return mode.value, k.value

    # ---- batched distance ------------------------------------------------------------------------
    @staticmethod
    def _common_bits(*ps: PackedSeqs):
        bits = 2 if all(p.bits == 2 for p in ps) else 4
        return [p.repack(bits) for p in ps], bits

    def distance_batch(self, A: PackedSeqs, B: PackedSeqs, force_mode: int = 0, out: np.ndarray | None = None):
        """out[p] = D[m][n] of (A[p] -> B[p]) as fp64 (== wagnerFisher(...)[-1][-1].value)."""
        if A.n != B.n:
            raise ValueError("A and B must hold the same number of sequences")
        (A, B), bits = self._common_bits(A, B)
        if out is None:
            out = np.zeros(A.n, dtype=np.float64)
        mode = C.c_int()
        # a batch in rsd_pack's layout keeps its start[] on the host: the device rebuilds it from the lengths
        check(self._lib.rsd_distance_batch(
            self._ctx, ptr(A.words, _u32), None if A.canonical else ptr(A.start, _i64), ptr(A.len, _i32), A.words.shape[0],
            ptr(B.words, _u32), None if B.canonical else ptr(B.start, _i64), ptr(B.len, _i32), B.words.shape[0],
            A.n, A.max_len, B.max_len, bits, A.symmask | B.symmask, force_mode, ptr(out, _f64), C.byref(mode)))
        self.last_mode = mode.value
        return out

    def distance_batch_codes(self, a_codes: np.ndarray, a_len: np.ndarray, b_codes: np.ndarray, b_len: np.ndarray,
                             bits: int = 4, symmask: int = 0, force_mode: int = 0, out: np.ndarray | None = None):
        """Distances straight from raw symbol codes (uint8, sequences concatenated in pair order) and int32
        lengths: the codes are packed on the device, chunk by chunk, under the kernels of earlier chunks."""
        n = int(a_len.shape[0])
        if int(b_len.shape[0]) != n:
            raise ValueError("a_len and b_len must have the same length")
        a_codes = np.ascontiguousarray(a_codes, np.uint8); b_codes = np.ascontiguousarray(b_codes, np.uint8)
        a_len = np.ascontiguousarray(a_len, np.int32); b_len = np.ascontiguousarray(b_len, np.int32)
        if out is None:
            out = np.zeros(n, dtype=np.float64)
        pad = np.zeros(1, np.uint8)
        mode = C.c_int()
        check(self._lib.rsd_distance_batch_codes(
            self._ctx, ptr(a_codes if a_codes.size else pad, _u8), ptr(a_len, _i32),
            ptr(b_codes if b_codes.size else pad, _u8), ptr(b_len, _i32), n,
            int(a_len.max(initial=0)), int(b_len.max(initial=0)), bits, symmask, force_mode, ptr(out, _f64), C.byref(mode)))
        self.last_mode = mode.value
        return out

    def distance_batch_dev(self, a_words, a_start, a_len, b_words, b_start, b_len, n_pairs, max_m, max_n, bits,
                           symmask, out, stream, force_mode: int = 0):
        """Device-pointer variant (ints = device addresses, stream = cudaStream_t handle); async."""
        mode = C.c_int()
        check(self._lib.rsd_distance_batch_dev(self._ctx, a_words, a_start, a_len, b_words, b_start, b_len,
                                               n_pairs, max_m, max_n, bits, symmask, force_mode, out,
                                               C.byref(mode), stream))
        self.last_mode = mode.value
        return mode.value

    # ---- one pair, whole matrix --------------------------------------------------------------------
    def matrix(self, a_codes: np.ndarray, b_codes: np.ndarray):
        m, n = int(a_codes.shape[0]), int(b_codes.shape[0])
        vals = np.zeros((m + 1, n + 1), dtype=np.float64)
        mask = np.zeros((m + 1, n + 1), dtype=np.uint8)
        a = np.ascontiguousarray(a_codes, dtype=np.uint8) if m else np.zeros(1, np.uint8)
        b = np.ascontiguousarray(b_codes, dtype=np.uint8) if n else np.zeros(1, np.uint8)
        check(self._lib.rsd_matrix(self._ctx, ptr(a, _u8), m, ptr(b, _u8), n, ptr(vals, _f64), ptr(mask, _u8)))
        return vals, mask

    # ---- batched canonical scripts -------------------------------------------------------------------
    def script_batch(self, A: PackedSeqs, B: PackedSeqs, force_mode: int = 0, check_roundtrip: bool = False):
        """-> dict(op uint8[n,max_ops], oi, oj int32[n,max_ops], n_ops int32[n], dist f64[n][, ok uint8[n]]).
        Ops run origin->sink; (oi, oj) = matrix cell entered (reference indices are oi-1 / oj-1)."""
        if A.n != B.n:
            raise ValueError("A and B must hold the same number of sequences")
        (A, B), bits = self._common_bits(A, B)
        n = A.n
        max_ops = max(int((A.len.astype(np.int64) + B.len).max()) if n else 0, 1)
        op = np.zeros((n, max_ops), np.uint8); oi = np.zeros((n, max_ops), np.int32)
        oj = np.zeros((n, max_ops), np.int32); n_ops = np.zeros(n, np.int32); dist = np.zeros(n, np.float64)
        mode = C.c_int()
        args = [self._ctx, ptr(A.words, _u32), ptr(A.start, _i64), ptr(A.len, _i32), A.words.shape[0],
                ptr(B.words, _u32), ptr(B.start, _i64), ptr(B.len, _i32), B.words.shape[0],
                n, bits, A.symmask | B.symmask, force_mode, max_ops,
                ptr(op, _u8), ptr(oi, _i32), ptr(oj, _i32), ptr(n_ops, _i32), ptr(dist, _f64)]
        res = dict(op=op, oi=oi, oj=oj, n_ops=n_ops, dist=dist)
        if check_roundtrip:
            ok = np.zeros(n, np.uint8)
            check(self._lib.rsd_script_patch_check_batch(*args, ptr(ok, _u8), C.byref(mode)))
            res["ok"] = ok
        else:
            check(self._lib.rsd_script_batch(*args, C.byref(mode)))
        self.last_mode = mode.value
        return res

    def patch_batch(self, scripts: dict, A: PackedSeqs, B: PackedSeqs, X: PackedSeqs):
        """patching(es_p, x_p) for scripts from script_batch -> (out codes uint8[n,max_out], out_len, err).
        Every script must be a path of its pair (A_p -> B_p), like those of script_batch and their reverses
        (eswire.rev_packed with A and B swapped): RsdError RSD_EINVAL otherwise, before any device work.  Hand-edited
        scripts go through sed.patching."""
        (A, B, X), bits = self._common_bits(A, B, X)
        n = A.n
        op, oi, oj, n_ops = scripts["op"], scripts["oi"], scripts["oj"], scripts["n_ops"]
        max_ops = op.shape[1]
        max_out = max(int((X.len.astype(np.int64) + n_ops).max()) if n else 0, 1)
        out = np.zeros((n, max_out), np.uint8); out_len = np.zeros(n, np.int32); err = np.zeros(n, np.int32)
        check(self._lib.rsd_patch_batch(
            self._ctx, ptr(op, _u8), ptr(oi, _i32), ptr(oj, _i32), ptr(n_ops, _i32), max_ops,
            ptr(A.words, _u32), ptr(A.start, _i64), ptr(A.len, _i32), A.words.shape[0],
            ptr(B.words, _u32), ptr(B.start, _i64), ptr(B.len, _i32), B.words.shape[0],
            ptr(X.words, _u32), ptr(X.start, _i64), ptr(X.len, _i32), X.words.shape[0],
            n, bits, max_out, ptr(out, _u8), ptr(out_len, _i32), ptr(err, _i32)))
        return out, out_len, err

    # ---- database search ------------------------------------------------------------------------------
    def db_load(self, db: PackedSeqs, global_index_base: int = 0):
        check(self._lib.rsd_db_load(self._ctx, ptr(db.words, _u32), ptr(db.start, _i64), ptr(db.len, _i32),
                                    db.n, db.words.shape[0], db.bits, db.symmask, global_index_base))
        self._db_n = db.n
        self._db_bits = db.bits
        self._db_gen = getattr(self, "_db_gen", 0) + 1      # lets callers that keep a database resident notice a reload

    def db_free(self):
        check(self._lib.rsd_db_free(self._ctx))
        self._db_gen = getattr(self, "_db_gen", 0) + 1

    def db_append(self, db: PackedSeqs):
        """Append db's records (same packing as the loaded database) after the loaded ones: the database then answers
        every search exactly as a db_load of the concatenation would, and a built idf table is continued, not rebuilt."""
        check(self._lib.rsd_db_append(self._ctx, ptr(db.words, _u32), ptr(db.start, _i64), ptr(db.len, _i32),
                                      db.n, db.words.shape[0], db.bits, db.symmask))
        self._db_n += db.n
        self._db_gen += 1

    def db_layout(self):
        """The stored order of the loaded database -> (perm int64[n_db]: global index of stored record r,
        tier_end int64[16], tier_mask uint32[16])."""
        n = C.c_int64()
        check(self._lib.rsd_db_layout(self._ctx, C.byref(n), None, None, None))
        perm = np.zeros(max(n.value, 1), np.int64); te = np.zeros(16, np.int64); tm = np.zeros(16, np.uint32)
        check(self._lib.rsd_db_layout(self._ctx, C.byref(n), ptr(perm, _i64), ptr(te, _i64), ptr(tm, _u32)))
        return perm[:n.value], te, tm

    def db_search_topk(self, Q: PackedSeqs, k: int, want_scores: bool = False, force_mode: int = 0):
        """-> (top_idx int64[q,k], top_score f64[q,k][, all_scores f64[q, n_db]])."""
        Q = _db_query(Q, self._db_bits)
        nq = Q.n
        idx = np.zeros((nq, k), np.int64); sc = np.zeros((nq, k), np.float64)
        alls = np.zeros((nq, self._db_n), np.float64) if want_scores else None
        mode = C.c_int()
        check(self._lib.rsd_db_search_topk(self._ctx, ptr(Q.words, _u32), ptr(Q.start, _i64), ptr(Q.len, _i32), nq,
                                           Q.words.shape[0], Q.bits, Q.symmask, k, force_mode,
                                           ptr(idx, _i64), ptr(sc, _f64),
                                           ptr(alls, _f64) if want_scores else None, C.byref(mode)))
        self.last_mode = mode.value
        return (idx, sc, alls) if want_scores else (idx, sc)

    def db_search_range(self, Q: PackedSeqs, max_dist: float, force_mode: int = 0):
        """Every database record within max_dist (inclusive) of each query, with its exact distance D (the fp64 value of
        distance_batch(query, record)) -> CSR (offsets int64[q+1], idx int64[total], dist f64[total]): the hits of query q
        are idx[offsets[q]:offsets[q+1]], by global index ascending.  max_dist = inf returns every record."""
        Q = _db_query(Q, self._db_bits)
        res, self.last_mode = _search_range(self._lib.rsd_db_search_range, self._ctx, Q, max_dist, force_mode,
                                            getattr(self, "_range_total", Q.n * 256))
        self._range_total = int(res[0][-1])
        return res

    def db_search_topk_dev(self, q_words, q_start, q_len, n_queries, max_qlen, bits, q_symmask, k, top_idx, top_score,
                           stream, force_mode: int = 0):
        mode = C.c_int()
        check(self._lib.rsd_db_search_topk_dev(self._ctx, q_words, q_start, q_len, n_queries, max_qlen, bits,
                                               q_symmask, k, force_mode, top_idx, top_score, C.byref(mode), stream))
        self.last_mode = mode.value
        return mode.value

    # ---- other scorers of search_collection (set / multiset / TF-vector measures) ---------------------------
    SIM_METHODS = ("set_intersection_similarity", "set_jaccard_similarity", "set_dice_similarity",
                   "multi_intersection_similarity", "multi_jaccard_similarity", "multi_dice_similarity",
                   "cosine", "pearson", "euclidian_distance", "manhattan_distance", "tanimoto_distance", "dice_dist")

    def db_similarity(self, query_codes: np.ndarray, method, k: int = 0, want_scores: bool = True, vector_type="tf"):
        """IR:443-477 for the measures of IR:49-389 against the loaded database; vector_type 'idf' / 'tf-idf' (vector
        measures only) scores the idf / tf-idf vectors of IR:189-225 instead of the TF matrices (IR:458-465).
        -> (all_scores f64[n_db] | None, top_idx int64[k], top_score f64[k])."""
        if _vector_type(vector_type) != 0:
            alls, idx, sc = self.db_similarity_batch([np.asarray(query_codes, np.uint8)], method, k, want_scores, vector_type)
            return (alls[0] if want_scores else None), idx[0], sc[0]
        mid = _sim_method(method)
        q = np.ascontiguousarray(query_codes, np.uint8)
        qq = q if q.shape[0] else np.zeros(1, np.uint8)
        alls = np.zeros(self._db_n, np.float64) if want_scores else None
        idx = np.full(max(k, 1), -1, np.int64); sc = np.zeros(max(k, 1), np.float64)
        check(self._lib.rsd_db_similarity(self._ctx, ptr(qq, _u8), int(q.shape[0]), mid, int(k), ptr(idx, _i64), ptr(sc, _f64),
                                          ptr(alls, _f64) if want_scores and self._db_n else None))
        return alls, idx[:k], sc[:k]

    def db_similarity_batch(self, queries, method, k: int = 0, want_scores: bool = True, vector_type="tf"):
        """db_similarity for a batch of queries in one pass over the database per query batch: `queries` is a list of
        code arrays or a (codes, offsets) tuple, as pack takes it.  Row q equals db_similarity(queries[q], ...) bit for bit.
        -> (all_scores f64[q, n_db] | None, top_idx int64[q, k], top_score f64[q, k])."""
        fn = _sim_entry(self._lib.rsd_db_similarity_batch, self._lib.rsd_db_vector_similarity_batch, vector_type)
        return _similarity_batch(fn, self._ctx, getattr(self, "_db_n", 0), queries, method, k, want_scores)

    def db_idf_table(self):
        """The document frequencies and idf values of the loaded database (IR:189-216), built on the device on first use
        after db_load -> (df f64[15, 15], idf f64[15, 15]).  A database loaded with global_index_base != 0 is refused."""
        return _idf_table(self._lib.rsd_db_idf_table, self._ctx)

    def topk_merge(self, idx: np.ndarray, score: np.ndarray):
        return topk_merge(idx, score)

    # ---- long pair ----------------------------------------------------------------------------------------
    def long_pair(self, a_codes: np.ndarray, b_codes: np.ndarray, want_script: bool = True, force_mode: int = 0):
        m, n = int(a_codes.shape[0]), int(b_codes.shape[0])
        a = np.ascontiguousarray(a_codes, np.uint8) if m else np.zeros(1, np.uint8)
        b = np.ascontiguousarray(b_codes, np.uint8) if n else np.zeros(1, np.uint8)
        max_ops = m + n + 1 if want_script else 1
        op = np.empty(max_ops, np.uint8); oi = np.empty(max_ops, np.int32); oj = np.empty(max_ops, np.int32)     # only [:n_ops] is handed out
        n_ops = C.c_int64(); dist = C.c_double(); mode = C.c_int()
        check(self._lib.rsd_long_pair(self._ctx, ptr(a, _u8), m, ptr(b, _u8), n, force_mode, int(want_script), max_ops,
                                      ptr(op, _u8), ptr(oi, _i32), ptr(oj, _i32), C.byref(n_ops), C.byref(dist),
                                      C.byref(mode)))
        self.last_mode = mode.value
        k = n_ops.value
        return dict(dist=dist.value, op=op[:k], oi=oi[:k], oj=oj[:k], mode=mode.value)

    def long_pairs(self, pairs, want_script: bool = True, force_mode: int = 0):
        """A batch of long pairs [(a_codes, b_codes), ...] in as few launches as the device memory allows
        (rsd_long_pairs); -> list of dicts like long_pair."""
        K = len(pairs)
        if K == 0:
            return []
        A = [np.ascontiguousarray(a, np.uint8) if a.shape[0] else np.zeros(1, np.uint8) for a, _ in pairs]
        B = [np.ascontiguousarray(b, np.uint8) if b.shape[0] else np.zeros(1, np.uint8) for _, b in pairs]
        m = np.array([a.shape[0] for a, _ in pairs], np.int64); n = np.array([b.shape[0] for _, b in pairs], np.int64)
        max_ops = (m + n + 1) if want_script else np.ones(K, np.int64)
        # np.empty: only [:n_ops] is handed out, and calloc of 72 recycled 100 - 400 KB chunks costs several ms per call
        op = [np.empty(int(k), np.uint8) for k in max_ops]
        oi = [np.empty(int(k), np.int32) for k in max_ops]; oj = [np.empty(int(k), np.int32) for k in max_ops]
        parr = lambda xs: (C.c_void_p * K)(*[x.ctypes.data for x in xs])
        n_ops = np.zeros(K, np.int64); dist = np.zeros(K, np.float64); mode = (C.c_int * K)()
        check(self._lib.rsd_long_pairs(self._ctx, K, parr(A), ptr(m, _i64), parr(B), ptr(n, _i64), force_mode, int(want_script),
                                       ptr(np.ascontiguousarray(max_ops, np.int64), _i64), parr(op), parr(oi), parr(oj),
                                       ptr(n_ops, _i64), ptr(dist, _f64), mode))
        self.last_mode = mode[0]
        return [dict(dist=float(dist[k]), op=op[k][:n_ops[k]], oi=oi[k][:n_ops[k]], oj=oj[k][:n_ops[k]], mode=mode[k]) for k in range(K)]

    def long_forward_ms(self) -> float:
        return float(self._lib.rsd_long_forward_ms(self._ctx))

    # ---- introspection -----------------------------------------------------------------------------------
    def launch_count(self) -> int:
        return int(self._lib.rsd_launch_count(self._ctx))

    def set_timing(self, on: bool):
        check(self._lib.rsd_set_timing(self._ctx, int(on)))

    def last_kernel_ms(self) -> float:
        return float(self._lib.rsd_last_kernel_ms(self._ctx))

    def ubench(self, which: int) -> float:
        v = C.c_double()
        check(self._lib.rsd_ubench(self._ctx, which, C.byref(v)))
        return v.value

    @property
    def ctx(self):
        return self._ctx


class MultiEngine:
    """Database search over several GPUs from one process (include/rsd.h, rsd_multi_*): contiguous shards, the
    query batch on every device, local top-k, one NCCL all-gather of the lists, merge.  Same search interface as
    Engine (set_costs / db_load / db_search_topk / db_search_range / db_similarity[_batch] / db_idf_table / db_free), so
    ir.score_collection and ir.similarity_collection run on either."""

    def __init__(self, devices=None):
        self._lib = _lib.load_library()
        self._h = C.c_void_p()
        if devices is None:
            check(self._lib.rsd_multi_create(None, 0, C.byref(self._h)))
        else:
            arr = (C.c_int * len(devices))(*devices)
            check(self._lib.rsd_multi_create(arr, len(devices), C.byref(self._h)))
        self.n_devices = int(self._lib.rsd_multi_device_count(self._h))
        self.pid = os.getpid()
        self.last_mode = 0
        self._costs_key = None
        self._db_gen = 0
        self._db_n = 0
        self._db_bits = 4

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.rsd_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            if os.getpid() == self.pid:
                self.close()
        except Exception:
            pass

    def set_costs(self, costs: dict):
        ins, dele, sub = costs_to_arrays(costs)
        key = (ins, dele, sub.tobytes())
        if key != self._costs_key:
            check(self._lib.rsd_multi_set_costs(self._h, ins, dele, ptr(sub, _f64)))
            self._costs_key = key

    def db_load(self, db: PackedSeqs):
        check(self._lib.rsd_multi_db_load(self._h, ptr(db.words, _u32), ptr(db.start, _i64), ptr(db.len, _i32), db.n,
                                          db.words.shape[0], db.bits, db.symmask))
        self._db_n, self._db_bits = db.n, db.bits
        self._db_gen += 1

    def db_free(self):
        check(self._lib.rsd_multi_db_free(self._h))
        self._db_gen += 1

    def db_append(self, db: PackedSeqs):
        """Engine.db_append over the whole database: the records go to the last shard (no rebalancing)."""
        check(self._lib.rsd_multi_db_append(self._h, ptr(db.words, _u32), ptr(db.start, _i64), ptr(db.len, _i32), db.n,
                                            db.words.shape[0], db.bits, db.symmask))
        self._db_n += db.n
        self._db_gen += 1

    def db_search_topk(self, Q: PackedSeqs, k: int, want_scores: bool = False, force_mode: int = 0):
        Q = _db_query(Q, self._db_bits)
        nq = Q.n
        idx = np.zeros((nq, max(k, 1)), np.int64); sc = np.zeros((nq, max(k, 1)), np.float64)
        alls = np.zeros((nq, self._db_n), np.float64) if want_scores else None
        mode = C.c_int()
        check(self._lib.rsd_multi_db_search_topk(self._h, ptr(Q.words, _u32), ptr(Q.start, _i64), ptr(Q.len, _i32), nq,
                                                 Q.words.shape[0], Q.bits, Q.symmask, k, force_mode, ptr(idx, _i64), ptr(sc, _f64),
                                                 ptr(alls, _f64) if want_scores else None, C.byref(mode)))
        self.last_mode = mode.value
        idx, sc = idx[:, :k], sc[:, :k]
        return (idx, sc, alls) if want_scores else (idx, sc)

    def db_search_range(self, Q: PackedSeqs, max_dist: float, force_mode: int = 0):
        """Engine.db_search_range over the whole sharded database."""
        Q = _db_query(Q, self._db_bits)
        res, self.last_mode = _search_range(self._lib.rsd_multi_db_search_range, self._h, Q, max_dist, force_mode,
                                            getattr(self, "_range_total", Q.n * 256))
        self._range_total = int(res[0][-1])
        return res

    def db_similarity(self, query_codes: np.ndarray, method, k: int = 0, want_scores: bool = True, vector_type="tf"):
        """Engine.db_similarity over the whole sharded database."""
        alls, idx, sc = self.db_similarity_batch([np.asarray(query_codes, np.uint8)], method, k, want_scores, vector_type)
        return (alls[0] if want_scores else None), idx[0], sc[0]

    def db_similarity_batch(self, queries, method, k: int = 0, want_scores: bool = True, vector_type="tf"):
        """Engine.db_similarity_batch over the whole sharded database."""
        fn = _sim_entry(self._lib.rsd_multi_db_similarity, self._lib.rsd_multi_db_vector_similarity, vector_type)
        return _similarity_batch(fn, self._h, self._db_n, queries, method, k, want_scores)

    def db_idf_table(self):
        """Engine.db_idf_table over the whole sharded database: the sums run through the shards in order."""
        return _idf_table(self._lib.rsd_multi_db_idf_table, self._h)

    def launch_count(self) -> int:
        return int(self._lib.rsd_multi_launch_count(self._h))


def topk_merge(idx: np.ndarray, score: np.ndarray):
    """idx/score: [n_shards, n_queries, k] -> merged ([n_queries, k], [n_queries, k]) with the key
    (score descending, global index ascending) — the reduction after the NCCL gather."""
    lib = _lib.load_library()
    g, nq, k = idx.shape
    idx = np.ascontiguousarray(idx, np.int64); score = np.ascontiguousarray(score, np.float64)
    oi = np.zeros((nq, k), np.int64); os_ = np.zeros((nq, k), np.float64)
    check(lib.rsd_topk_merge(ptr(idx, _i64), ptr(score, _f64), g, nq, k, ptr(oi, _i64), ptr(os_, _f64)))
    return oi, os_


_engines: dict = {}


def get_engine(device: int = 0) -> Engine:
    """Process-local singleton (fork-safe: keyed by pid)."""
    key = (os.getpid(), device)
    e = _engines.get(key)
    if e is None:
        e = _engines[key] = Engine(device)
    return e


_multi: dict = {}


def get_search_engine():
    """What search_collection runs on: every visible GPU when there is more than one (MultiEngine, one process),
    else the process-local Engine."""
    lib = _lib.load_library()
    if lib.rsd_device_count() <= 1:
        return get_engine()
    e = _multi.get(os.getpid())
    if e is None:
        e = _multi[os.getpid()] = MultiEngine()
    return e
