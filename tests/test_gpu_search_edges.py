"""GPU parity of the database searches' exact top-k where ties cross chunk, tier and shard boundaries (DESIGN §3, §4).

Both searches order their results by score descending, then collection index ascending, and no single kernel owns
that order.  rsd_db_load stores the records sorted by (symbol tier, length); the search scans the stored order in
chunks (a 4096-record seed chunk, then main chunks; the int16x2 prefix first, the fp64 tail after it);
k_topk_fold merges each chunk's candidates into the running list and raises the threshold tau = (score, index); and a
record of a later chunk gets in only through the filter `s > ts || (s == ts && g <= ti)`.

Each test builds a database in which tied records straddle such a boundary, with the smaller collection indices on
the later side, and asserts that layout (from a host restatement of the store order) before it compares every
result with the oracle using ==.  If the store order or the chunking changes, the precondition fails instead of the
test passing vacuously."""
import numpy as np
import pytest

from oracle import ir_oracle as IO
from oracle import oracle as O

pytestmark = pytest.mark.gpu

I16X2, F64 = 1, 3
KMAX = 128                     # RSD_TOPK_MAX
SEED = 4096                    # the seed chunk of both searches
MAIN_SEARCH = 1 << 21          # the largest main chunk of the edit-distance search
MAIN_SIM = 1 << 20             # the main chunk of the similarity search
L = 28                         # storm query length
VECTOR_METHODS = ["cosine", "pearson", "euclidian_distance", "manhattan_distance", "tanimoto_distance", "dice_dist"]
SET_METHODS = ["set_intersection_similarity", "set_jaccard_similarity", "set_dice_similarity"]


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


# ---------------------------------------------------------------------------------------------------------------------
# host restatements and checks
# ---------------------------------------------------------------------------------------------------------------------
def record_masks(codes, off):
    """bit c set = symbol c occurs in the record"""
    lens = np.diff(off)
    masks = np.zeros(lens.shape[0], np.int64)
    ne = lens > 0
    if ne.any():
        masks[ne] = np.bitwise_or.reduceat(np.left_shift(np.uint16(1), codes.astype(np.uint16)), off[:-1][ne])
    return masks


def stored_order(codes, off):
    """rsd_db_load's store order: stable sort by (tier, length).  A record's tier is the rank of its rarest symbol,
    the symbols ranked by how many records hold them; the first tiers are merged up to the one that brings the
    prefix to half of the records.  -> the collection index of each stored record"""
    lens = np.diff(off)
    n = lens.shape[0]
    masks = record_masks(codes, off)
    holds = np.array([np.count_nonzero((masks >> b) & 1) for b in range(16)])
    rank = np.empty(16, np.int64)
    rank[np.argsort(-holds, kind="stable")] = np.arange(16)
    tier = np.zeros(n, np.int64)
    for b in range(16):
        tier = np.where((masks >> b) & 1, np.maximum(tier, rank[b]), tier)
    r0 = 0
    while r0 < 15 and 2 * np.count_nonzero(tier <= r0) < n:
        r0 += 1
    return np.lexsort((lens, np.maximum(tier - r0, 0)))


def topk_of(scores, k):
    """Per row: the first k of the stable descending sort of the non-NaN scores (performance.py:12-15), padded with
    index -1 / score 0.0."""
    scores = np.atleast_2d(scores)
    idx = np.full((scores.shape[0], k), -1, np.int64)
    sc = np.zeros((scores.shape[0], k), np.float64)
    for q, row in enumerate(scores):
        valid = np.flatnonzero(~np.isnan(row))
        top = valid[np.argsort(-row[valid], kind="stable")][:k]
        idx[q, :top.shape[0]] = top
        sc[q, :top.shape[0]] = row[top]
    return idx, sc


def oracle_scores(queries, codes, off, costs):
    """oracle.search_topk's score of every record, one row per query"""
    return np.stack([O.search_topk(q, codes, off, costs, 1, want_scores=True)[2] for q in queries])


def assert_tie_displaced(row, stored, boundary, k):
    """The precondition of a tie test at one chunk boundary: the k-th and (k+1)-th best records tie; the records
    stored before `boundary` already fill a top-k list whose last key has that score, so tau holds that score once
    they are folded; and a record stored after the boundary with the same score and a smaller collection index belongs
    to the true top-k.  Only the equal-score branch of the filter lets it in."""
    ranked = topk_of(row, k + 1)[0][0]
    assert ranked[k] >= 0 and row[ranked[k - 1]] == row[ranked[k]], "the k-th and (k+1)-th entries must tie"
    before = np.sort(stored[:boundary])
    first = before[np.argsort(-row[before], kind="stable")][:k]
    assert first.shape[0] == k and row[first[-1]] == row[ranked[k - 1]], "the records before the boundary must fill the list with ties"
    after = np.zeros(row.shape[0], bool)
    after[stored[boundary:]] = True
    top = ranked[:k]
    late = top[after[top] & (row[top] == row[first[-1]]) & (top < first[-1])]
    assert late.shape[0] > 0, "no tied record after the boundary has a smaller index than tau"


def same_bits(a, b):
    return bool(np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


# ---------------------------------------------------------------------------------------------------------------------
# the tie storm: records at distance exactly 1 from two queries, spread over lengths L-1, L, L+1
# ---------------------------------------------------------------------------------------------------------------------
def variant(rng, q, kind):
    """q (ACGU codes) at distance exactly 1 under ins = del = sub = 1 (and C -> D = 1): one edit"""
    if kind == "D":                                              # one C of the query became D: an fp64-tail record
        v = q.copy(); v[rng.choice(np.flatnonzero(q == 2))] = 10
        return v
    p = int(rng.integers(0, q.shape[0]))
    if kind == "sub":
        v = q.copy(); v[p] = (v[p] + rng.integers(1, 4)) % 4
        return v
    if kind == "del":
        return np.delete(q, p)
    return np.insert(q, p, rng.integers(0, 4)).astype(np.uint8)


class Storm:
    """Random ACGU fillers of lengths 20-32 around two queries A and B of length L = 28, plus
    - at the smallest indices (the first tenth of the collection): 60 insertions (L+1) then 64 substitutions (L) of
      A, 70 + 70 of B, and 4 exact copies of A: with the copies, exactly KMAX records of A score >= 0.5 there;
    - from 55 % of the collection on: 200 deletions (L-1), 100 substitutions and 100 insertions of each query.
    Few fillers are shorter than L, so the deletions (large indices) sit in the seed chunk and fill its top-k list
    with ties, and the insertions (smallest indices) come in the last chunks: they displace them through g <= ti.
    The KMAX-th key of A is the last low-index tie, the (KMAX+1)-th lies past the middle, so that cut crosses every
    shard boundary of 2, 3 or 8 shards.  n_d = (a, b) adds, at the smallest indices of all, records with one C of
    A / B turned into D; they store after every ACGU record: the fp64 tail."""

    def __init__(self, seed, n, n_long, n_d=(0, 0), n_short=1500, n_prev=500):
        rng = np.random.default_rng(seed)
        q = []
        while len(q) < 2:
            s = rng.integers(0, 4, size=L, dtype=np.uint8)
            if (s == 2).sum() >= 2:
                q.append(s)
        a, b = q
        lens = np.full(n, L, np.int64)
        lens[:n_short] = rng.integers(20, L - 1, size=n_short)
        lens[n_short:n_short + n_prev] = L - 1
        lens[n_short + n_prev:n_short + n_prev + n_long] = rng.integers(L + 1, 33, size=n_long)
        lens = rng.permutation(lens)
        low_kinds = ([(a, "D")] * n_d[0] + [(b, "D")] * n_d[1] + [(a, "ins")] * 60 + [(b, "ins")] * 70
                     + [(a, "sub")] * 64 + [(b, "sub")] * 70 + [(a, "copy")] * 4)
        high_kinds = [(x, kind) for x in (a, b) for kind, cnt in (("del", 200), ("sub", 100), ("ins", 100)) for _ in range(cnt)]
        low = np.sort(rng.choice(n // 10, size=len(low_kinds), replace=False))
        high = rng.choice(np.arange(int(0.55 * n), n), size=len(high_kinds), replace=False)
        special = {}
        for pos, (x, kind) in zip(np.concatenate([low, high]), low_kinds + high_kinds):
            special[int(pos)] = x.copy() if kind == "copy" else variant(rng, x, kind)
            lens[pos] = special[int(pos)].shape[0]
        off = np.zeros(n + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        codes = rng.integers(0, 4, size=int(off[-1]), dtype=np.uint8)
        for pos, v in special.items():
            codes[off[pos]:off[pos + 1]] = v
        self.codes, self.off, self.n = codes, off, n
        self.d_records = np.sort(low[:sum(n_d)])
        self.queries = [O.decode(a), O.decode(b)]
        self.stored = stored_order(codes, off)
        self._scores = {}

    def scores(self, queries, costs):
        """oracle scores of the given queries (cached per query)"""
        for q in queries:
            if q not in self._scores:
                self._scores[q] = oracle_scores([q], self.codes, self.off, costs)[0]
        return np.stack([self._scores[q] for q in queries])


@pytest.fixture(scope="module")
def storm(golden):
    """about 10^5 records: one seed chunk and one main chunk; n - 4096 is not a multiple of 32"""
    s = Storm(20261020, 100_003, n_long=20_000)
    s.scores(s.queries, golden["default_costs"])
    return s


@pytest.fixture(scope="module")
def storm_big(golden):
    """about 2.2 * 10^6 records: the insertions are stored past seed + the largest main chunk"""
    s = Storm(20261021, 2_200_000, n_long=60_000)
    s.scores(s.queries, golden["default_costs"])
    return s


def check_storm_layout(s, costs, boundaries):
    """the scores the storm promises, and the tie displacements at every boundary for A at k = KMAX and B at k = 1
    and KMAX"""
    sc = s.scores(s.queries, costs)
    for row in sc:
        assert np.count_nonzero(row == 0.5) >= 3 * KMAX
    assert np.count_nonzero(sc[0] == 1.0) == 4 and np.count_nonzero(sc[1] == 1.0) == 0
    for boundary in boundaries:
        assert_tie_displaced(sc[0], s.stored, boundary, KMAX)
        assert_tie_displaced(sc[1], s.stored, boundary, KMAX)
        assert_tie_displaced(sc[1], s.stored, boundary, 1)
    return sc


def search_and_check(R, eng, s, queries, k, costs, force_mode=0, mode=None):
    eng.set_costs(costs)
    want = s.scores(queries, costs)
    wi, ws = topk_of(want, k)
    eng.db_load(R.pack((s.codes, s.off), bits=4))
    try:
        idx, sc, alls = eng.db_search_topk(R.pack(queries, bits=4), k, want_scores=True, force_mode=force_mode)
        if mode is not None:
            assert eng.last_mode == mode
    finally:
        eng.db_free()
    assert np.array_equal(alls, want)
    for q in range(len(queries)):
        assert np.array_equal(idx[q], wi[q]) and np.array_equal(sc[q], ws[q]), (q, k)
    return idx, sc


# ---------------------------------------------------------------------------------------------------------------------
# 1 + 2: the storm through the int16x2 search kernel, the general path and a tiered database
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, KMAX])
def test_storm_fast_path(R, eng, golden, storm, k):
    costs = golden["default_costs"]
    sc = check_storm_layout(storm, costs, [SEED])
    wi, ws = O.search_topk(storm.queries[0], storm.codes, storm.off, costs, k)      # topk_of is the oracle's own cut
    assert np.array_equal(topk_of(sc[0], k)[0][0], wi) and np.array_equal(topk_of(sc[0], k)[1][0], ws)
    search_and_check(R, eng, storm, storm.queries, k, costs, mode=I16X2)


@pytest.mark.parametrize("k", [1, KMAX])
def test_storm_fast_path_across_main_chunks(R, eng, golden, storm_big, k):
    check_storm_layout(storm_big, golden["default_costs"], [SEED, SEED + MAIN_SEARCH])
    search_and_check(R, eng, storm_big, storm_big.queries, k, golden["default_costs"], mode=I16X2)


@pytest.mark.parametrize("k", [1, KMAX])
def test_storm_general_path(R, eng, golden, storm, k):
    """force_mode = 3: the seed chunk of the general path, then k_score_filter_pairs over n - 4096 records (not a
    multiple of 32, so the warps at the seams hold two queries)"""
    costs = golden["default_costs"]
    check_storm_layout(storm, costs, [SEED])
    assert (storm.n - SEED) % 32 != 0
    queries = storm.queries + [storm.queries[0][:-2] + "GG"]
    search_and_check(R, eng, storm, queries, k, costs, force_mode=F64, mode=F64)


@pytest.fixture(scope="module")
def tiered(golden):
    """the storm with 37 + 29 records at distance 1 through C -> D at the smallest indices: the fp64 tail"""
    s = Storm(20261022, 100_003, n_long=20_000, n_d=(37, 29))
    s.scores(s.queries, golden["default_costs"])
    return s


@pytest.mark.parametrize("k", [1, KMAX])
def test_tiered_tail_ties_displace_the_fast_prefix(R, eng, golden, tiered, k):
    """The int16x2 kernel takes the ACGU prefix, the general kernels the D records stored after it; their ties have
    the smallest indices, so they must displace the prefix's through k_score_filter_pairs' g <= ti.  The tail holds
    66 records and the batch 3 queries, so warps of the filter hold two queries."""
    costs = golden["default_costs"]
    s = tiered
    n_acgu = s.n - s.d_records.shape[0]
    assert np.array_equal(np.sort(s.stored[n_acgu:]), s.d_records), "the D records must store after every ACGU record"
    assert s.d_records.shape[0] % 32 != 0
    queries = s.queries + [s.queries[1][:-1] + "A"]
    sc = s.scores(queries, costs)
    assert (sc[:2, s.d_records] == 0.5).sum() == s.d_records.shape[0]
    assert_tie_displaced(sc[0], s.stored, n_acgu, KMAX)          # A's best are its copies: its ties cut at KMAX only
    assert_tie_displaced(sc[1], s.stored, n_acgu, k)
    search_and_check(R, eng, s, queries, k, costs, mode=F64)


# ---------------------------------------------------------------------------------------------------------------------
# 3: shards and MultiEngine
# ---------------------------------------------------------------------------------------------------------------------
def multi_bounds(lens, G):
    """rsd_multi_db_load's contiguous shards: shard g ends at the last record whose length prefix sum is <= total * (g+1) / G"""
    csum = np.cumsum(lens.astype(np.float64))
    total = float(csum[-1])
    cuts = [0] + [int(np.searchsorted(csum, total * (g + 1) / G, side="right")) for g in range(G - 1)] + [lens.shape[0]]
    return list(zip(cuts[:-1], cuts[1:]))


def assert_cut_crosses(bounds, kth, next_):
    shard_of = lambda i: next(g for g, (lo, hi) in enumerate(bounds) if lo <= i < hi)
    assert shard_of(kth) != shard_of(next_), (bounds, kth, next_)


def test_sharded_storm_ties_across_shards(R, eng, golden, storm):
    from rna_sequence_diff_patch_b200.dist_search import shard_bounds, slice_packed
    from rna_sequence_diff_patch_b200.engine import topk_merge
    costs = golden["default_costs"]
    want = storm.scores(storm.queries, costs)
    wi, ws = topk_of(want, KMAX)
    ranked = topk_of(want[0], KMAX + 1)[0][0]
    assert want[0, ranked[KMAX - 1]] == want[0, ranked[KMAX]] == 0.5
    db = R.pack((storm.codes, storm.off), bits=4)
    Q = R.pack(storm.queries, bits=4)
    eng.set_costs(costs)
    for world in (2, 3, 8):
        bounds = shard_bounds(db.len, world)
        assert_cut_crosses(bounds, ranked[KMAX - 1], ranked[KMAX])
        li, ls = [], []
        for lo, hi in bounds:
            eng.db_load(slice_packed(db, lo, hi), global_index_base=lo)
            try:
                i, s = eng.db_search_topk(Q, KMAX)
            finally:
                eng.db_free()
            li.append(i); ls.append(s)
        mi, ms = topk_merge(np.stack(li), np.stack(ls))
        assert np.array_equal(mi, wi) and np.array_equal(ms, ws), world
    assert_cut_crosses(multi_bounds(db.len, 3), ranked[KMAX - 1], ranked[KMAX])
    me = R.MultiEngine([0, 0, 0])
    try:
        me.set_costs(costs)
        me.db_load(db)
        idx, sc, alls = me.db_search_topk(Q, KMAX, want_scores=True)
        assert me.last_mode == I16X2
        assert np.array_equal(alls, want)
        assert np.array_equal(idx, wi) and np.array_equal(sc, ws)
        me.db_free()
    finally:
        me.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4: rsd_db_search_topk_dev
# ---------------------------------------------------------------------------------------------------------------------
def search_dev(eng, Q, k, force_mode=0):
    """rsd_db_search_topk_dev on torch device tensors, on a side stream that is synchronised before the read"""
    import torch
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (Q.words, Q.start, Q.len)]
        idx = torch.full((Q.n, max(k, 1)), -7, dtype=torch.int64, device="cuda")
        sc = torch.full((Q.n, max(k, 1)), -7.0, dtype=torch.float64, device="cuda")
    mode = eng.db_search_topk_dev(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), Q.n, Q.max_len, Q.bits, Q.symmask, k,
                                  idx.data_ptr(), sc.data_ptr(), side.cuda_stream, force_mode)
    side.synchronize()
    return idx.cpu().numpy(), sc.cpu().numpy(), mode


def storm_queries(s, n, seed):
    """A, B, then n - 2 copies of them with one to three substitutions: every query meets integer-distance ties"""
    rng = np.random.default_rng(seed)
    out = list(s.queries)
    while len(out) < n:
        q = O.encode(s.queries[len(out) % 2]).copy()
        pos = rng.choice(L, size=int(rng.integers(1, 4)), replace=False)
        q[pos] = (q[pos] + rng.integers(1, 4, size=pos.shape[0])) % 4
        out.append(O.decode(q))
    return out


def test_search_topk_dev(R, eng, golden, storm):
    """130 queries (three batches of 64, the last one partial) at k = KMAX; then a batch mixing ambiguous and plain
    queries, which the device entry point does not regroup: all of it goes through the general kernels."""
    costs = golden["default_costs"]
    check_storm_layout(storm, costs, [SEED])
    queries = storm_queries(storm, 130, 7)
    # D and H cost 0.66 / 0.83 against A under the default table: not dyadic, no int16x2 kernel for these batches
    mixed = [queries[0], queries[0][:3] + "D" + queries[0][4:], queries[1], queries[2][:-1] + "H", queries[3]]
    eng.set_costs(costs)
    eng.db_load(R.pack((storm.codes, storm.off), bits=4))
    try:
        Q = R.pack(queries, bits=4)
        idx, sc, mode = search_dev(eng, Q, KMAX)
        assert mode == I16X2
        hi, hs = eng.db_search_topk(Q, KMAX)
        Qm = R.pack(mixed, bits=4)
        midx, msc, mmode = search_dev(eng, Qm, KMAX)
        assert mmode == F64
        mhi, mhs = eng.db_search_topk(Qm, KMAX)
        with pytest.raises(R.RsdError):
            search_dev(eng, Q, 0)
    finally:
        eng.db_free()
    assert np.array_equal(idx, hi) and np.array_equal(sc, hs)
    wi, ws = topk_of(storm.scores(queries, costs), KMAX)
    for q in range(len(queries)):
        assert np.array_equal(idx[q], wi[q]) and np.array_equal(sc[q], ws[q]), q
    assert np.array_equal(midx, mhi) and np.array_equal(msc, mhs)
    wi, ws = topk_of(storm.scores(mixed, costs), KMAX)
    assert np.array_equal(midx, wi) and np.array_equal(msc, ws)


# ---------------------------------------------------------------------------------------------------------------------
# 5: k limits and empties
# ---------------------------------------------------------------------------------------------------------------------
def test_k_above_the_limit_is_rejected(R, eng, golden, storm):
    eng.set_costs(golden["default_costs"])
    eng.db_load(R.pack((storm.codes, storm.off[:2001].copy()), bits=4))
    try:
        Q = R.pack(storm.queries, bits=4)
        for force_mode in (0, F64):
            eng.db_search_topk(Q, KMAX, force_mode=force_mode)
            with pytest.raises(R.RsdError):
                eng.db_search_topk(Q, KMAX + 1, force_mode=force_mode)
        eng.db_similarity(O.encode(storm.queries[0]), "cosine", k=KMAX)
        with pytest.raises(R.RsdError):
            eng.db_similarity(O.encode(storm.queries[0]), "cosine", k=KMAX + 1)
    finally:
        eng.db_free()


def small_search(R, eng, costs, docs, queries, k, force_mode=0):
    c, o = O.concat(docs)
    eng.set_costs(costs)
    eng.db_load(R.pack(docs, bits=4))
    try:
        idx, sc, alls = eng.db_search_topk(R.pack(queries, bits=4), k, want_scores=True, force_mode=force_mode)
        mode = eng.last_mode
    finally:
        eng.db_free()
    want = oracle_scores(queries, c, o, costs)
    assert np.array_equal(alls, want)
    for q, query in enumerate(queries):
        wi, ws = O.search_topk(query, c, o, costs, k)
        assert np.array_equal(idx[q], wi) and np.array_equal(sc[q], ws), q
    return idx, sc, mode


def test_k_above_the_record_count_pads(R, eng, golden):
    docs = ["ACGUACGUAC", "GGGCCCAUAU", "ACGUACGUAC", "", "UUUUA"]
    for force_mode, mode in ((0, I16X2), (F64, F64)):
        idx, sc, got_mode = small_search(R, eng, golden["default_costs"], docs, ["ACGUACGUAG", "GGCCAU"], 12, force_mode)
        assert got_mode == mode
        assert (idx[:, 5:] == -1).all() and (sc[:, 5:] == 0.0).all() and (idx[:, :5] >= 0).all()


def test_empty_records_and_queries(R, eng, golden):
    """a stored record of length 0 and a zero-length query inside a batch on the int16x2 kernel; a batch of only
    zero-length queries, which the int16x2 kernel cannot take (it needs a query row), on the general path"""
    rng = np.random.default_rng(5)
    docs = ["", "ACGU"] + ["".join(rng.choice(list("ACGU"), size=int(n))) for n in rng.integers(0, 33, size=300)] + [""]
    costs = golden["default_costs"]
    assert sum(d == "" for d in docs) >= 3
    _, _, mode = small_search(R, eng, costs, docs, ["", docs[7], "", "ACGUAGCU"], 20)
    assert mode == I16X2
    _, _, mode = small_search(R, eng, costs, docs, ["", ""], 20)
    assert mode != I16X2
    _, _, mode = small_search(R, eng, costs, docs, [""], 5)
    assert mode != I16X2


# ---------------------------------------------------------------------------------------------------------------------
# 6: where k_sim_tf_thread hands records to the warp kernel k_sim_tf
# ---------------------------------------------------------------------------------------------------------------------
def tf_search(queries, docs, methods):
    """ir_oracle.search with each record's representation computed once"""
    tfs = [IO.tf_vector(d) for d in docs]
    return {(q, m): np.array([IO.score(m, IO.represent(q, m), v) for v in tfs], np.float64) for q in queries for m in methods}


@pytest.mark.parametrize("bits", [2, 4])
def test_tf_thread_and_warp_kernels_split_at_60000_symbols(R, eng, bits):
    """ACGU records of 60000 symbols (the last one the per-thread kernel counts in uint16) and 60001 (the first one it
    hands over), a 65537-symbol run of one symbol whose bigram count passes 2^16, records whose only ambiguity code is
    first or last, and records of length 0 and 1 (all-zero TF matrix) — all six vector measures, bit for bit"""
    rng = np.random.default_rng(60000 + bits)
    acgu = lambda n: "".join(rng.choice(list("ACGU"), size=n))
    docs = [acgu(60000), acgu(60001), "A" * 65537, "", "G", acgu(40), acgu(333)]
    if bits == 4:
        docs += ["R" + acgu(99), acgu(99) + "Y", "N" + acgu(5000), acgu(5000) + "D"]
    lens = [len(d) for d in docs]
    assert 60000 in lens and 60001 in lens and max(lens) >= 65537
    assert IO.tf_vector("A" * 65537)[0, 0] == 65536                     # wraps to 0 in a 16-bit counter
    queries = [acgu(50), "A" * 40, "ACGUNRYACGUACGUSWKM" + acgu(20)]
    want = tf_search(queries, docs, VECTOR_METHODS)
    eng.db_load(R.pack(docs, bits=bits))
    try:
        for q in queries:
            for m in VECTOR_METHODS:
                got, _, _ = eng.db_similarity(R.encode(q), m)
                assert same_bits(got, want[q, m]), (q[:8], m, bits, got, want[q, m])
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# 7: similarity ranking across three chunks, with the list not yet full after the seed, and with k above the
#    number of rankable records
# ---------------------------------------------------------------------------------------------------------------------
def test_set_measures_ties_across_three_chunks(R, eng):
    """k = KMAX over 4096 + 2^20 + 50000 records.  Every record holds A, C, G and U; 160 also hold N, spread over the
    three chunks, and two in the last chunk hold N and R as well: the cut falls inside a massive tie in the third
    chunk."""
    rng = np.random.default_rng(72)
    n = SEED + MAIN_SIM + 50_000
    lens = rng.integers(8, 17, size=n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    codes = rng.integers(0, 4, size=int(off[-1]), dtype=np.uint8)
    for c in range(4):                                                    # A, G, C and U in every record
        codes[off[:-1] + c] = c
    c2, c3 = SEED + MAIN_SIM, n
    with_n = np.concatenate([rng.choice(SEED, 50, replace=False), rng.choice(np.arange(SEED, c2), 50, replace=False),
                             rng.choice(np.arange(c2, c3), 60, replace=False)])
    codes[off[with_n] + 4] = 14                                           # N
    best = rng.choice(np.setdiff1d(np.arange(c2, c3), with_n), 2, replace=False)
    codes[off[best] + 4] = 14; codes[off[best] + 5] = 5                   # N and R
    query = "ACGUNR" + "ACGU" * 5
    qmask = IO.set_mask(query)
    masks = record_masks(codes, off)
    uniq, inv = np.unique(masks, return_inverse=True)
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        for m in SET_METHODS:
            want = np.array([IO.score(m, qmask, int(u)) for u in uniq], np.float64)[inv]
            wi, ws = topk_of(want, KMAX)
            ranked = topk_of(want, KMAX + 1)[0][0]
            assert want[ranked[KMAX - 1]] == want[ranked[KMAX]]
            assert ((wi[0] < SEED).any() and ((wi[0] >= SEED) & (wi[0] < c2)).any() and (ranked[KMAX - 1] >= c2)
                    and (wi[0, :2] >= c2).all()), "the top-k must draw from all three chunks"
            got, idx, sc = eng.db_similarity(R.encode(query), m, k=KMAX)
            assert same_bits(got, want), m
            assert np.array_equal(idx, wi[0]) and np.array_equal(sc, ws[0]), m
    finally:
        eng.db_free()


def test_pearson_list_not_full_after_the_seed(R, eng):
    """The first 4096 records give 40 non-NaN Pearson scores (the rest have length 0 or 1: all-zero TF matrix, 0/0),
    so the list is not full after the seed fold; the true top-k ends in negative scores from later records (bigrams
    disjoint from the query's).  tau must stay at 'accept all' until the list is full."""
    rng = np.random.default_rng(73)
    acgu = lambda n: "".join(rng.choice(list("ACGU"), size=n))
    gu = lambda n: "".join(rng.choice(list("GU"), size=n))
    seed = ["" if i % 2 else "C" for i in range(SEED)]
    for i in rng.choice(SEED, 40, replace=False):
        seed[i] = acgu(int(rng.integers(20, 41)))
    later = ["A" if i % 3 else "" for i in range(2000)]
    kinds = rng.permutation(["p"] * 30 + ["n"] * 600 + ["x"] * 1370)
    for i, kind in enumerate(kinds):
        if kind == "p":
            later[i] = acgu(int(rng.integers(20, 41)))
        elif kind == "n":
            later[i] = gu(int(rng.integers(20, 41)))
    docs = seed + later
    query = "AC" * 15
    want = IO.search(query, docs, "pearson")
    assert np.count_nonzero(~np.isnan(want[:SEED])) < KMAX
    wi, ws = topk_of(want, KMAX)
    assert (wi[0] >= 0).all() and (ws[0, -1] < 0) and (wi[0][ws[0] < 0] >= SEED).all()
    eng.db_load(R.pack(docs, bits=4))
    try:
        got, idx, sc = eng.db_similarity(R.encode(query), "pearson", k=KMAX)
    finally:
        eng.db_free()
    assert same_bits(got, want)
    assert np.array_equal(idx, wi[0]) and np.array_equal(sc, ws[0])


def test_k_above_the_rankable_records_pads(R, eng):
    """NaN scores are never ranked; the list pads with -1 / 0.0"""
    docs = ["", "ACGUAGG", "G", "CCCAAAUU", "", "GUGUGAC", "A", "ACGUNNRY", "UUAAC"]
    query = "ACGUUGCA"
    eng.db_load(R.pack(docs, bits=4))
    try:
        for m in ("cosine", "pearson", "tanimoto_distance"):
            want = IO.search(query, docs, m)
            n_ok = int(np.count_nonzero(~np.isnan(want)))
            assert 0 < n_ok < 12
            got, idx, sc = eng.db_similarity(R.encode(query), m, k=12)
            wi, ws = topk_of(want, 12)
            assert same_bits(got, want)
            assert np.array_equal(idx, wi[0]) and np.array_equal(sc, ws[0]), m
            assert (idx[n_ok:] == -1).all() and (sc[n_ok:] == 0.0).all()
    finally:
        eng.db_free()
