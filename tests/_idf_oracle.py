"""Host restatement of the reference's idf and tf-idf vectors (IRMethods.py IR:189-225) and of the six vector measures
over a whole collection, fast enough for tens of thousands of records.  TEST INFRASTRUCTURE ONLY.  Pinned to
measures.py and to tests/golden/ref_golden_ir.json by tests/test_idf_oracle.py.

  compare_pair_to_seq (IR:225-252) depends only on the set of literal bigrams of the document: the largest product
  wa * wb over the expansions (a, b) of the pair whose bigram occurs, 0 when none does.
  df[p] = the sequential fp64 sum of those values in collection order (IR:205-212) = the last row of np.cumsum.
  idf[p] = 0 if df[p] == 0 else math.log(N / df[p], 10).
  tf-idf = np.dot(tf, idf), which BLAS evaluates per element as a fused multiply-add chain over k = 0..14 ascending
  from +0.0; Python has no math.fma, so a few lines of C (built on first use into a temporary directory) run it."""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess
import tempfile

import numpy as np

from oracle import ir_oracle as IO

W = IO.W


def possibilities(s: int):
    """IR:255-287 on codes: (symbols, probabilities)."""
    if s < 4:
        syms, probs = [s], [1]
        for x in range(4, 15):
            if W[x][s] != 0:
                syms.append(x); probs.append(float(W[x][s]))
        return syms, probs
    syms = [b for b in range(4) if W[s][b] != 0]
    return syms + [s], [1 / len(syms)] * len(syms) + [1]


def expansions():
    """Per pair p = a * 15 + b: [(bigram, wa * wb)] over possibilities(a) x possibilities(b)."""
    out = []
    for p in range(225):
        sa, pa = possibilities(p // 15)
        sb, pb = possibilities(p % 15)
        out.append([(x * 15 + y, wx * wy) for x, wx in zip(sa, pa) for y, wy in zip(sb, pb)])
    return out


_EXP = expansions()


def presence(seq: str) -> np.ndarray:
    """bool[225]: the literal bigrams of seq"""
    cs = IO.codes_of(seq)
    p = np.zeros(225, bool)
    for a, b in zip(cs[:-1], cs[1:]):
        p[a * 15 + b] = True
    return p


def values(docs) -> np.ndarray:
    """[N, 225]: compare_pair_to_seq(p, doc) for every document and pair"""
    P = np.stack([presence(d) for d in docs]) if len(docs) else np.zeros((0, 225), bool)
    V = np.zeros((P.shape[0], 225))
    for p, ex in enumerate(_EXP):
        col = V[:, p]
        for e, w in ex:
            np.maximum(col, np.where(P[:, e], w, 0.0), out=col)
    return V


def table(docs):
    """(df [225], idf [225]) of the collection `docs` in this order"""
    V = values(docs)
    df = np.cumsum(V, axis=0)[-1] if V.shape[0] else np.zeros(225)
    return df, _idf_of(df, len(docs))


def _idf_of(df, n):
    return np.array([0.0 if d == 0 else math.log(n / d, 10) for d in df])


def table_codes(codes: np.ndarray, off: np.ndarray, chunk: int = 1 << 18):
    """table() of a collection given as symbol codes (record i = codes[off[i]:off[i+1]]), for millions of records: the
    values of each chunk come from its distinct presence sets, and np.cumsum continues from the previous chunk's sums."""
    n = off.shape[0] - 1
    ex = [(np.array([e for e, _ in x]), np.array([w for _, w in x])) for x in _EXP]
    df = np.zeros(225)
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        c = codes[off[r0]:off[r1]].astype(np.int64)
        rec = np.repeat(np.arange(r1 - r0), np.diff(off[r0:r1 + 1]))
        inner = rec[:-1] == rec[1:]                             # bigrams inside one record
        P = np.zeros((r1 - r0, 225), bool)
        P[rec[:-1][inner], (c[:-1] * 15 + c[1:])[inner]] = True
        U, inv = np.unique(np.packbits(P, axis=1), axis=0, return_inverse=True)
        PU = np.unpackbits(U, axis=1, count=225).astype(bool)
        VU = np.zeros((PU.shape[0], 225))
        for p, (e, w) in enumerate(ex):
            VU[:, p] = np.max(np.where(PU[:, e], w[None, :], 0.0), axis=1)
        V = np.concatenate([df[None, :], VU[inv.reshape(-1)]])
        df = np.cumsum(V, axis=0)[-1]
    return df, _idf_of(df, n)


def idf_vector(seq: str, idf: np.ndarray) -> np.ndarray:
    return np.where(presence(seq), idf, 0.0).reshape(15, 15)


_SRC = r"""
#include <math.h>
/* c[n][15][15] = a[n] . b[n], each element a fused multiply-add chain over k = 0..14 from +0.0 */
void mm_fma(const double *a, const double *b, double *c, long n) {
  for (long r = 0; r < n; ++r, a += 225, b += 225, c += 225)
    for (int i = 0; i < 15; ++i) for (int j = 0; j < 15; ++j) {
      double acc = 0.0;
      for (int k = 0; k < 15; ++k) acc = fma(a[i * 15 + k], b[k * 15 + j], acc);
      c[i * 15 + j] = acc;
    }
}
"""
_lib = None


def _mm():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="idf_oracle_")
        src, so = os.path.join(d, "mm.c"), os.path.join(d, "mm.so")
        with open(src, "w") as f:
            f.write(_SRC)
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o", so, src, "-lm"])
        _lib = C.CDLL(so)
        _lib.mm_fma.restype = None
        _lib.mm_fma.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long]
    return _lib


def dot_fma(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """[n, 15, 15] x [n, 15, 15] -> [n, 15, 15], the fused chain per element"""
    a = np.ascontiguousarray(a, np.float64).reshape(-1, 225)
    b = np.ascontiguousarray(b, np.float64).reshape(-1, 225)
    c = np.zeros_like(a)
    if a.shape[0]:
        _mm().mm_fma(a.ctypes.data, b.ctypes.data, c.ctypes.data, a.shape[0])
    return c.reshape(-1, 15, 15)


def vectors(seqs, vector_type: str, idf: np.ndarray) -> np.ndarray:
    """[n, 15, 15]: the idf or tf-idf vectors of seqs under the table idf"""
    iv = np.stack([idf_vector(s, idf) for s in seqs]) if len(seqs) else np.zeros((0, 15, 15))
    if vector_type == "idf":
        return iv
    tf = np.stack([IO.tf_vector(s) for s in seqs]) if len(seqs) else np.zeros((0, 15, 15))
    return dot_fma(tf, iv)


def scores(method: str, a: np.ndarray, B: np.ndarray) -> np.ndarray:
    """IR:290-389 of the query vector a against every row of B ([n, 15, 15]), with the reference's numpy arithmetic:
    np.sum over a row is the same pairwise sum as over the 15 x 15 matrix."""
    a = a.reshape(225); B = B.reshape(-1, 225)
    with np.errstate(all="ignore"):
        if method == "pearson":
            a = a - np.average(a)
            B = B - np.average(B, axis=1)[:, None]
        if method == "euclidian_distance":
            return 1 / (1 + np.sqrt(np.sum(np.square(a - B), axis=1)))
        if method == "manhattan_distance":
            return 1 / (1 + np.sqrt(np.sum(np.abs(a - B), axis=1)))
        num = np.sum(np.multiply(a, B), axis=1)
        a_sq, b_sq = np.sum(np.square(a)), np.sum(np.square(B), axis=1)
        if method in ("cosine", "pearson"):
            return num / np.sqrt(a_sq * b_sq)
        if method == "tanimoto_distance":
            return num / (a_sq + b_sq - num)
        if method == "dice_dist":
            return 2 * num / (a_sq + b_sq)
    raise ValueError(method)


def search(queries, docs, vector_type: str, method: str, idf=None) -> np.ndarray:
    """[len(queries), len(docs)]: search_collection(query, vector_type, docs, method) scores; idf: the table of docs
    (computed when not given)"""
    if idf is None:
        idf = table(docs)[1]
    B = vectors(docs, vector_type, idf)
    A = vectors(queries, vector_type, idf)
    return np.stack([scores(method, a, B) for a in A]) if len(queries) else np.zeros((0, len(docs)))
