"""Range search over the resident database (rsd_db_search_range, rsd_multi_db_search_range, Engine.db_search_range).

For each query: every record with D(query, record) <= max_dist, D being the fp64 distance the oracle computes for
(source = query, destination = record), in collection order, with D itself.  Every GPU result is compared with the
oracle using ==: the oracle's distances of all records, filtered and kept in index order.  The bounds come from the
oracle's own distance multiset, an occurring D and the double just below it, so both sides of the inclusive edge
are hit."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_search_edges import Storm

gpu = pytest.mark.gpu
I16X2, F64 = 1, 3
ERANGE = 6
IUPAC = "YRWSKMDVHB"


@pytest.fixture(scope="module")
def R():
    import __graft_entry__ as G
    G.build()
    import rna_sequence_diff_patch_b200 as R
    return R


@pytest.fixture(scope="module")
def eng(R):
    assert R.load_library().rsd_device_count() > 0
    return R.Engine(0)


# ---------------------------------------------------------------------------------------------------------------------
# the oracle side
# ---------------------------------------------------------------------------------------------------------------------
def oracle_dist(queries, codes, off, costs):
    """D of every (query, record) pair, one row per query"""
    n = off.shape[0] - 1
    rows = []
    for q in queries:
        qc = O.encode(q)
        rows.append(O.distance_batch(np.tile(qc, n), np.arange(n + 1, dtype=np.int64) * qc.shape[0], codes, off, costs))
    return np.stack(rows) if rows else np.zeros((0, n))


def range_of(D, max_dist):
    """-> (offsets, idx, dist): per row the records with D <= max_dist, by index"""
    off, idx, dist = [0], [], []
    for row in D:
        h = np.flatnonzero(row <= max_dist)
        idx.append(h); dist.append(row[h]); off.append(off[-1] + h.shape[0])
    cat = lambda xs, t: np.concatenate(xs).astype(t) if xs else np.zeros(0, t)
    return np.array(off, np.int64), cat(idx, np.int64), cat(dist, np.float64)


def assert_same(got, want, what=""):
    (go, gi, gd), (wo, wi, wd) = got, want
    assert np.array_equal(go, wo), what
    assert np.array_equal(gi, wi), what
    assert np.array_equal(gd.view(np.uint64), wd.view(np.uint64)), what          # bit-identical distances


def edge_bounds(D, picks):
    """occurring distances and the doubles just below them"""
    vals = np.unique(D)
    out = []
    for v in picks(vals):
        out += [float(v), float(np.nextafter(v, -np.inf))]
    return out


def family_db(seed, n, lo, hi, alphabet="ACGU", n_queries=64, p_mut=0.08, extra=None):
    """n random records of lengths lo..hi over `alphabet`, and queries that are mutated copies of records (so that
    small bounds have hits)"""
    rng = np.random.default_rng(seed)
    recs = ["".join(rng.choice(list(alphabet), size=int(rng.integers(lo, hi + 1)))) for _ in range(n)]
    if extra:
        extra(rng, recs)
    queries = []
    for _ in range(n_queries):
        s = list(recs[int(rng.integers(0, n))])
        for i in range(len(s)):
            if rng.random() < p_mut:
                s[i] = str(rng.choice(list("ACGU")))
        queries.append("".join(s)[:hi])
    codes, off = O.concat(recs)
    return recs, codes, off, queries


def search(R, eng, codes, off, queries, costs, bounds, force_mode=0, mode=None, D=None):
    """every bound through Engine.db_search_range against the oracle; -> the oracle's distance matrix"""
    eng.set_costs(costs)
    if D is None:
        D = oracle_dist(queries, codes, off, costs)
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        Q = R.pack(queries, bits=4)
        for b in bounds:
            got = eng.db_search_range(Q, b, force_mode=force_mode)
            if mode is not None:
                assert eng.last_mode == mode, b
            assert_same(got, range_of(D, b), b)
    finally:
        eng.db_free()
    return D


# ---------------------------------------------------------------------------------------------------------------------
# 1 - 5: the kernels and the query grouping
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def acgun(golden):
    """about 10^5 ACGU+N records of 24-31 nt, 64 queries; default costs (N: 0.75, so int16x2 at k = 2)"""
    recs, codes, off, queries = family_db(20261101, 100_000, 24, 31, alphabet="ACGUACGUACGUN")
    D = oracle_dist(queries, codes, off, golden["default_costs"])
    return codes, off, queries, D


@gpu
def test_fast_path(R, eng, golden, acgun):
    codes, off, queries, D = acgun
    costs = golden["default_costs"]
    eng.set_costs(costs)
    assert eng.classify(0x400F, 31, 31) == (2, 2)
    bounds = [0.0, 1.0, 2.5] + edge_bounds(D, lambda v: [v[v > 2.5][0], v[v > 4][0]])
    search(R, eng, codes, off, queries, costs, bounds, mode=I16X2, D=D)
    assert range_of(D, 1.0)[0][-1] > 0 and range_of(D, 2.5)[0][-1] > range_of(D, 1.0)[0][-1]     # the small bounds do have hits
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        Q = R.pack(queries, bits=4)
        for b in bounds:
            a = eng.db_search_range(Q, b)
            g = eng.db_search_range(Q, b, force_mode=F64)
            assert eng.last_mode == F64
            assert_same(g, a, b)
    finally:
        eng.db_free()


@gpu
def test_scaled_integer_mode(R, eng, golden):
    """every cost 0.75: the int16x2 kernel at k = 2; bounds at multiples of 0.75 and just below them"""
    costs = {"insert": 0.75, "delete": 0.75,
             "update": {a: {b: 0.75 for b in golden["default_costs"]["update"][a]} for a in golden["default_costs"]["update"]}}
    recs, codes, off, queries = family_db(20261102, 20_000, 20, 32, n_queries=16)
    eng.set_costs(costs)
    assert eng.classify(0xF, 32, 32) == (1, 2)
    bounds = []
    for j in (0, 1, 2, 3, 5, 8):
        bounds += [0.75 * j, float(np.nextafter(0.75 * j, -np.inf))]
    bounds = [b for b in bounds if b >= 0]
    search(R, eng, codes, off, queries, costs, bounds, mode=I16X2)


@gpu
def test_tiered_fp64_tail(R, eng, golden):
    """1 % of the records carry an IUPAC symbol (non-dyadic 0.66 / 0.83 under the default table): they store after
    the ACGU prefix and go through the general kernels in fp64; bounds at their non-dyadic distances"""
    def sprinkle(rng, recs):
        for i in rng.choice(len(recs), size=len(recs) // 100, replace=False):
            s = list(recs[i]); s[int(rng.integers(0, len(s)))] = str(rng.choice(list(IUPAC))); recs[i] = "".join(s)
    recs, codes, off, queries = family_db(20261103, 100_000, 24, 31, n_queries=32, extra=sprinkle)
    costs = golden["default_costs"]
    D = oracle_dist(queries, codes, off, costs)
    tail = np.array([any(c in IUPAC for c in r) for r in recs])
    frac = D[:, tail][(D[:, tail] * 4) != np.floor(D[:, tail] * 4)]
    assert frac.shape[0] > 0
    nd = np.unique(frac)
    bounds = [float(nd[0]), float(np.nextafter(nd[0], -np.inf)), float(nd[nd.shape[0] // 3]), float(np.nextafter(nd[nd.shape[0] // 3], -np.inf))]
    search(R, eng, codes, off, queries, costs, bounds, mode=F64, D=D)
    h = range_of(D, bounds[2])
    assert tail[h[1]].any() and (~tail[h[1]]).any()              # hits from the fp64 tail and from the int16x2 prefix


@gpu
def test_general_path(R, eng, golden):
    recs, codes, off, queries = family_db(20261104, 3_000, 40, 300, n_queries=8, p_mut=0.05)
    costs = golden["user_costs"]
    D = oracle_dist(queries, codes, off, costs)
    bounds = [0.0] + edge_bounds(D, lambda v: [v[v.shape[0] // 50], v[v.shape[0] // 5]]) + [np.inf]
    search(R, eng, codes, off, queries, costs, bounds, D=D)


@gpu
def test_mixed_query_batch_keeps_caller_order(R, eng, golden, acgun):
    """ambiguous queries (IUPAC: the general kernels) interleaved with plain ones (the int16x2 kernel): the two
    groups run separately and the hits come back in caller order"""
    codes, off, queries, _ = acgun
    n = off.shape[0] - 1
    sel = np.arange(0, n, 7)                                       # a smaller database keeps the fp64 oracle quick
    recs = [O.decode(codes[off[i]:off[i + 1]]) for i in sel]
    codes2, off2 = O.concat(recs)
    mixed = []
    for i, q in enumerate(queries[:12]):
        mixed.append(q if i % 2 == 0 else q[:5] + IUPAC[i % len(IUPAC)] + q[6:])
    costs = golden["default_costs"]
    D = oracle_dist(mixed, codes2, off2, costs)
    bounds = edge_bounds(D, lambda v: [v[v > 3][0], v[v > 6][0]])
    search(R, eng, codes2, off2, mixed, costs, bounds, mode=F64, D=D)


# ---------------------------------------------------------------------------------------------------------------------
# 6, 7, 9: order, agreement with top-k, shards
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def storm(golden):
    """the tie storm of test_gpu_search_edges: records at distance 1 of two queries at the smallest and at the largest
    indices, with lengths L-1, L, L+1, so the smallest-index hits are stored last"""
    s = Storm(20261020, 100_003, n_long=20_000)
    s.D = oracle_dist(s.queries, s.codes, s.off, golden["default_costs"])
    return s


@gpu
def test_order_when_the_store_order_differs(R, eng, golden, storm):
    s = storm
    h = range_of(s.D, 1.0)
    pos = np.empty(s.n, np.int64); pos[s.stored] = np.arange(s.n)
    for q in range(2):
        hits = h[1][h[0][q]:h[0][q + 1]]
        assert hits.shape[0] > 500
        assert (np.diff(pos[hits]) < 0).any(), "the layout must store some hit with a smaller index after a larger one"
    search(R, eng, s.codes, s.off, s.queries, golden["default_costs"], [1.0, float(np.nextafter(1.0, -np.inf)), 2.0], mode=I16X2, D=s.D)


@gpu
def test_agrees_with_topk(R, eng, golden, acgun):
    """for every query with >= 128 hits: its hits by (D asc, index asc) start with db_search_topk(k=128)"""
    codes, off, queries, D = acgun
    eng.set_costs(golden["default_costs"])
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        Q = R.pack(queries, bits=4)
        ro, ri, rd = eng.db_search_range(Q, 12.0)
        ti, ts = eng.db_search_topk(Q, 128)
    finally:
        eng.db_free()
    checked = 0
    for q in range(len(queries)):
        i, d = ri[ro[q]:ro[q + 1]], rd[ro[q]:ro[q + 1]]
        if i.shape[0] < 128:
            continue
        o = np.lexsort((i, d))[:128]
        assert np.array_equal(i[o], ti[q]), q
        assert np.array_equal(1.0 / (1.0 + d[o]), ts[q]), q
        checked += 1
    assert checked >= 8


@gpu
def test_shards(R, eng, golden, storm):
    """2, 3 and 8 emulated shards (global_index_base) and MultiEngine([0, 0, 0]): the hits of the storm lie at the
    smallest and the largest indices, so a query's hits cross every shard boundary"""
    from rna_sequence_diff_patch_b200.dist_search import shard_bounds, slice_packed
    s = storm
    costs = golden["default_costs"]
    want = range_of(s.D, 1.0)
    db = R.pack((s.codes, s.off), bits=4)
    Q = R.pack(s.queries, bits=4)
    eng.set_costs(costs)
    for world in (2, 3, 8):
        bounds = shard_bounds(db.len, world)
        parts = []
        for lo, hi in bounds:
            eng.db_load(slice_packed(db, lo, hi), global_index_base=lo)
            try:
                parts.append(eng.db_search_range(Q, 1.0))
            finally:
                eng.db_free()
        for q in range(2):                                        # each query's hits lie on both sides of every boundary
            hits = want[1][want[0][q]:want[0][q + 1]]
            assert all((hits < lo).any() and (hits >= lo).any() for lo, _ in bounds[1:]), world
        off, idx, dist = [0], [], []
        for q in range(2):
            for o, i, d in parts:
                idx.append(i[o[q]:o[q + 1]]); dist.append(d[o[q]:o[q + 1]])
            off.append(sum(x.shape[0] for x in idx))
        assert_same((np.array(off), np.concatenate(idx), np.concatenate(dist)), want, world)
    me = R.MultiEngine([0, 0, 0])
    try:
        me.set_costs(costs)
        me.db_load(db)
        assert_same(me.db_search_range(Q, 1.0), want, "multi")
        assert me.last_mode == I16X2
        me.db_free()
    finally:
        me.close()


# ---------------------------------------------------------------------------------------------------------------------
# 8: capacity
# ---------------------------------------------------------------------------------------------------------------------
def c_range(R, ctx, Q, max_dist, cap, force_mode=0, fn="rsd_db_search_range"):
    """the C entry point with a caller-chosen cap -> (rc, hit_off, hit_idx, hit_dist)"""
    lib = R.load_library()
    off = np.full(Q.n + 1, -7, np.int64)
    idx = np.zeros(max(cap, 1), np.int64); dist = np.zeros(max(cap, 1), np.float64)
    p = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    rc = getattr(lib, fn)(ctx, p(Q.words, C.c_uint32), p(Q.start, C.c_int64), p(Q.len, C.c_int32), Q.n, Q.words.shape[0],
                          Q.bits, Q.symmask, max_dist, force_mode, cap, p(off, C.c_int64), p(idx, C.c_int64),
                          p(dist, C.c_double), None)
    return rc, off, idx, dist


@gpu
def test_capacity(R, eng, golden, acgun):
    codes, off, queries, D = acgun
    n = off.shape[0] - 1
    want = range_of(D, np.inf)
    assert want[0][-1] == 64 * n and 64 * n > (1 << 20)          # more hits than the device buffer starts with
    eng.set_costs(golden["default_costs"])
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        Q = R.pack(queries, bits=4)
        eng.__dict__.pop("_range_total", None)                     # first guess 64 * 256: the wrapper's retry
        assert_same(eng.db_search_range(Q, np.inf), want, "inf")
        assert_same(eng.db_search_range(Q, np.inf), want, "inf again")
        small = range_of(D, 6.0)
        rc, o, _, _ = c_range(R, eng.ctx, Q, 6.0, int(small[0][-1]) - 1)
        assert rc == ERANGE and str(int(small[0][-1])) in R.load_library().rsd_last_error().decode()
        assert np.array_equal(o, small[0])
        rc, o, i, d = c_range(R, eng.ctx, Q, 6.0, int(small[0][-1]))
        assert rc == 0
        assert_same((o, i, d), small, "exact cap")
        eng.__dict__["_range_total"] = 1
        assert_same(eng.db_search_range(Q, 6.0), small, "retry")
    finally:
        eng.db_free()


# ---------------------------------------------------------------------------------------------------------------------
# 10 - 12: edges, argument checks, self-join
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_edges(R, eng, golden):
    costs = golden["default_costs"]
    eng.set_costs(costs)
    recs = ["ACGU", "", "GGAUCC", "ACGUACGUAC", "N"]
    codes, off = O.concat(recs)
    Q = R.pack(["ACGA", "", "ACGUN"], bits=4)
    search(R, eng, codes, off, ["ACGA", "", "ACGUN"], costs, [0.0, 1.0, 3.0, np.inf])
    # empty database
    eng.db_load(R.pack((np.zeros(0, np.uint8), np.zeros(1, np.int64)), bits=4))
    try:
        o, i, d = eng.db_search_range(Q, np.inf)
        assert o.tolist() == [0, 0, 0, 0] and i.shape == (0,) and d.shape == (0,)
        o, i, d = eng.db_search_range(R.pack([], bits=4), 1.0)    # n_queries = 0
        assert o.tolist() == [0] and i.shape == (0,)
    finally:
        eng.db_free()
    # no database loaded
    with pytest.raises(R.RsdError) as ei:
        eng.db_search_range(Q, 1.0)
    assert ei.value.code == 1
    # a query packing that differs from the database's
    eng.db_load(R.pack(["ACGU", "GGAU"], bits=2))
    try:
        rc, _, _, _ = c_range(R, eng.ctx, R.pack(["ACGU"], bits=4), 1.0, 16)
        assert rc == 1 and "packing" in R.load_library().rsd_last_error().decode()
    finally:
        eng.db_free()
    # force_mode = 1 where the int16x2 kernel cannot take the whole database (records > 32 symbols)
    eng.db_load(R.pack(["ACGU" * 10, "ACG"], bits=4))
    try:
        with pytest.raises(R.RsdError) as ei:
            eng.db_search_range(R.pack(["ACGU"], bits=4), 1.0, force_mode=I16X2)
        assert ei.value.code == 1
    finally:
        eng.db_free()


def test_bad_bounds_fail_without_a_device(R):
    """NaN and negative bounds are rejected before the device is touched (CPU only)"""
    lib = R.load_library()
    ctx = C.c_void_p()
    assert lib.rsd_create(0, C.byref(ctx)) == 0
    try:
        Q = R.pack(["ACGU"], bits=4)
        for b in (float("nan"), -1.0, -0.5e-300):
            rc, _, _, _ = c_range(R, ctx, Q, b, 4)
            assert rc == 1 and "max_dist" in lib.rsd_last_error().decode()
        eng = R.Engine(0)
        eng._db_bits = 4
        for b in (float("nan"), -1.0):
            with pytest.raises(R.RsdError) as ei:
                eng.db_search_range(Q, b)
            assert ei.value.code == 1
    finally:
        lib.rsd_destroy(ctx)


@gpu
def test_self_join_is_symmetric(R, eng, golden):
    """2000 records joined against themselves under a symmetric table with ins = del: the hit relation is symmetric,
    with equal distances both ways, and holds the diagonal at D = 0"""
    costs = golden["default_costs"]
    upd = costs["update"]
    assert costs["insert"] == costs["delete"]
    assert all(upd[a][b] == upd[b][a] for a in "ACGU" for b in "ACGU" if a != b)
    rng = np.random.default_rng(20261112)
    seeds = ["".join(rng.choice(list("ACGU"), size=int(rng.integers(22, 31)))) for _ in range(40)]
    recs = []
    for _ in range(2000):
        s = list(seeds[int(rng.integers(0, 40))])
        for i in range(len(s)):
            if rng.random() < 0.1:
                s[i] = str(rng.choice(list("ACGU")))
        recs.append("".join(s))
    codes, off = O.concat(recs)
    D = search(R, eng, codes, off, recs, costs, [4.0])
    eng.db_load(R.pack((codes, off), bits=4))
    try:
        o, i, d = eng.db_search_range(R.pack(recs, bits=4), 4.0)
    finally:
        eng.db_free()
    q = np.repeat(np.arange(2000), np.diff(o))
    pairs = dict(zip(zip(q.tolist(), i.tolist()), d.tolist()))
    assert all(pairs.get((r, s)) == v for (s, r), v in pairs.items())
    assert all(pairs.get((r, r)) == 0.0 for r in range(2000))
    assert len(pairs) > 2000 * 3
