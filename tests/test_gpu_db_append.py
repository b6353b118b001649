"""Appending records to the loaded database (rsd_db_append, rsd_multi_db_append, Engine / MultiEngine.db_append): the
stored order equals rsd_db_load's for the concatenation (checked against a numpy restatement through rsd_db_layout),
and every search -- edit-distance top-k and range, the twelve similarity measures, the idf / tf-idf vector types and
the idf table -- answers bit for bit what a fresh load of the concatenation answers."""
import ctypes as C

import numpy as np
import pytest

import _idf_oracle as IDF
from oracle import ir_oracle as IO

pytestmark = pytest.mark.gpu

RSD_EINVAL = 1
VTS = ("idf", "tf-idf")
SEED_CHUNK = 4096              # the seed chunk of the edit-distance search
SEARCH_CHUNK = 1 << 21         # its largest main chunk
IDF_CHUNK = 1 << 20            # the chunk of the idf table build and of the similarity passes


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
def ref(R):
    return R.Engine(0)


# ---------------------------------------------------------------------------------------------------------------------
# host restatement of the stored order
# ---------------------------------------------------------------------------------------------------------------------
def layout_of(codes, off):
    """rsd_db_load's stored order of the collection: per-record symbol masks, holds[b] = records holding symbol b,
    symbols ranked by holds (stable), tier = rank of the rarest symbol, the first tiers merged up to half of the
    records (r0), stable sort by (merged tier, length, index).  -> (perm, tier_end[16], tier_mask[16], r0)"""
    lens = np.diff(off)
    n = lens.shape[0]
    masks = np.zeros(n, np.int64)
    ne = lens > 0
    if ne.any():
        masks[ne] = np.bitwise_or.reduceat(np.left_shift(np.uint16(1), codes.astype(np.uint16)), off[:-1][ne])
    holds = np.array([np.count_nonzero((masks >> b) & 1) for b in range(16)])
    order = np.argsort(-holds, kind="stable")
    rank = np.empty(16, np.int64)
    rank[order] = np.arange(16)
    tier = np.zeros(n, np.int64)
    for b in range(16):
        tier = np.where((masks >> b) & 1, np.maximum(tier, rank[b]), tier)
    cum = np.cumsum(np.bincount(tier, minlength=16))
    r0 = 0
    while r0 < 15 and 2 * cum[r0] < n:
        r0 += 1
    acc, mask = 0, []
    for r in range(16):
        if holds[order[r]] > 0:
            acc |= 1 << int(order[r])
        mask.append(acc)
    sel = [min(15, t + r0) for t in range(16)]
    perm = np.lexsort((np.arange(n), lens, np.maximum(tier - r0, 0)))
    return perm, cum[sel].astype(np.int64), np.array(mask, np.uint32)[sel], r0


def check_layout(eng, codes, off, base=0):
    perm, te, tm = eng.db_layout()
    wp, wte, wtm, r0 = layout_of(codes, off)
    assert np.array_equal(perm, wp + base)
    assert np.array_equal(te, wte) and np.array_equal(tm, wtm)
    return te, tm, r0


# ---------------------------------------------------------------------------------------------------------------------
# results against a fresh load
# ---------------------------------------------------------------------------------------------------------------------
def same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool(a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
                and np.array_equal(a[~np.isnan(a)].view(np.uint64), b[~np.isnan(b)].view(np.uint64)))


def assert_same_results(R, a, b, queries, costs, bits=4, idf=True, sims=True):
    """every search of engine a equals engine b's bit for bit (NaN where NaN)"""
    a.set_costs(costs); b.set_costs(costs)
    Q = R.pack(queries, bits=bits)
    for k in (1, 10, 128):
        ga, gb = a.db_search_topk(Q, k, want_scores=True), b.db_search_topk(Q, k, want_scores=True)
        assert np.array_equal(ga[0], gb[0]) and same_bits(ga[1], gb[1]) and same_bits(ga[2], gb[2]), k
    for bound in (2.0, 6.5, float("inf")):
        ra, rb = a.db_search_range(Q, bound), b.db_search_range(Q, bound)
        assert all(np.array_equal(x, y) for x, y in zip(ra[:2], rb[:2])) and same_bits(ra[2], rb[2]), bound
    qc = [R.encode(q) for q in queries]
    if sims:
        for method in IO.METHODS:
            ga, gb = a.db_similarity_batch(qc, method, k=10), b.db_similarity_batch(qc, method, k=10)
            assert same_bits(ga[0], gb[0]) and np.array_equal(ga[1], gb[1]) and same_bits(ga[2], gb[2]), method
    if idf:
        for vt in VTS:
            for method in IO.METHODS[6:]:
                ga = a.db_similarity_batch(qc, method, k=10, vector_type=vt)
                gb = b.db_similarity_batch(qc, method, k=10, vector_type=vt)
                assert same_bits(ga[0], gb[0]) and np.array_equal(ga[1], gb[1]) and same_bits(ga[2], gb[2]), (vt, method)
        ta, tb = a.db_idf_table(), b.db_idf_table()
        assert same_bits(ta[0], tb[0]) and same_bits(ta[1], tb[1])


def assert_table(eng, codes, off):
    df, idf = eng.db_idf_table()
    wdf, widf = IDF.table_codes(codes, off)
    assert same_bits(df.reshape(-1), wdf) and same_bits(idf.reshape(-1), widf)


def seqs_of(rng, n, alphabet="AGCU", lo=0, hi=40, dup=0.3, pool=None):
    """n random records; a share `dup` drawn from a small pool, so scores tie"""
    pool = pool or ["".join(rng.choice(list(alphabet), size=int(m))) for m in rng.integers(lo, hi + 1, size=20)]
    out = []
    for _ in range(n):
        if rng.random() < dup:
            out.append(pool[int(rng.integers(len(pool)))])
        else:
            out.append("".join(rng.choice(list(alphabet), size=int(rng.integers(lo, hi + 1)))))
    return out


def codes_of(R, seqs):
    from rna_sequence_diff_patch_b200.encoding import concat
    return concat(seqs)


def fresh(R, ref, seqs, bits=4, base=0):
    ref.db_load(R.pack(seqs, bits=bits), global_index_base=base)
    return ref


# ---------------------------------------------------------------------------------------------------------------------
# 1: the layout oracle pins rsd_db_load, then load + append
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bits", [2, 4])
def test_layout_after_load_and_append(R, eng, bits):
    rng = np.random.default_rng(11 + bits)
    alphas = ["AGCU", "AG", "C"] if bits == 2 else ["AGCU", "AGCUN", "AGCUYR", "YR"]

    def mixed(n, hi):                                   # records of several alphabets, so they fall in several tiers
        out = sum((seqs_of(rng, n // len(alphas), a, 0, hi) for a in alphas), [])
        return [out[i] for i in rng.permutation(len(out))]
    docs = mixed(3000, 60)
    eng.db_load(R.pack(docs, bits=bits))
    te0, _, _ = check_layout(eng, *codes_of(R, docs))
    assert np.unique(te0).shape[0] > 1
    more = mixed(1800, 70)
    eng.db_append(R.pack(more, bits=bits))
    check_layout(eng, *codes_of(R, docs + more))
    assert eng._db_n == len(docs) + len(more)


# ---------------------------------------------------------------------------------------------------------------------
# 3: after one append, several, an empty one, and on a database loaded with no records
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bits", [2, 4])
def test_appends_equal_a_fresh_load(R, eng, ref, golden, bits):
    rng = np.random.default_rng(30 + bits)
    alpha = "AGCU" if bits == 2 else "AGCUN"
    pool = ["".join(rng.choice(list(alpha), size=int(m))) for m in rng.integers(4, 31, size=12)]
    queries = [pool[0], pool[3], "ACGUACGUAC", ""]
    docs = seqs_of(rng, 800, alpha, 0, 32, 0.4, pool)
    eng.db_load(R.pack(docs, bits=bits))
    eng.db_idf_table()                                               # built before the appends: continued
    for n_add in (300, 0, 1, 2500, 64):
        more = seqs_of(rng, n_add, alpha, 0, 32, 0.4, pool)
        eng.db_append(R.pack(more, bits=bits))
        docs = docs + more
        check_layout(eng, *codes_of(R, docs))
        assert_same_results(R, eng, fresh(R, ref, docs, bits), queries, golden["default_costs"], bits)
    assert_table(eng, *codes_of(R, docs))


def test_append_to_an_empty_database(R, eng, ref, golden):
    rng = np.random.default_rng(41)
    eng.db_load(R.pack([], bits=4))
    assert eng.db_layout()[0].shape == (0,)
    docs = []
    for n_add in (0, 700, 300):
        more = seqs_of(rng, n_add, "AGCUYR", 0, 30)
        eng.db_append(R.pack(more, bits=4))
        docs = docs + more
    check_layout(eng, *codes_of(R, docs))
    assert_same_results(R, eng, fresh(R, ref, docs), ["ACGUAGCU", docs[5]], golden["default_costs"])
    assert_table(eng, *codes_of(R, docs))


# ---------------------------------------------------------------------------------------------------------------------
# 2: appends that change the tiering
# ---------------------------------------------------------------------------------------------------------------------
def test_append_reranks_symbols_and_moves_r0(R, eng, ref, golden):
    """mostly ACGU with a few IUPAC records; the append brings enough Y / R records to outrank U and move the cut"""
    rng = np.random.default_rng(51)
    docs = seqs_of(rng, 2000, "AGC", 3, 30, 0) + seqs_of(rng, 100, "AGCUYR", 3, 30, 0)
    eng.db_load(R.pack(docs, bits=4))
    _, tm0, r00 = check_layout(eng, *codes_of(R, docs))
    more = seqs_of(rng, 3000, "YR", 3, 30, 0) + seqs_of(rng, 500, "AGCUYRN", 3, 30, 0)
    eng.db_append(R.pack(more, bits=4))
    docs = docs + more
    _, tm1, r01 = check_layout(eng, *codes_of(R, docs))
    assert r01 != r00 and tm1[0] != tm0[0]
    assert_same_results(R, eng, fresh(R, ref, docs), ["AGCAGC", "YRYRYR", "ACGUN"], golden["default_costs"])


def test_append_longer_than_32_drops_the_fast_prefix(R, eng, ref, golden):
    """the int16x2 thread-per-record prefix needs every record within 32 symbols: one longer record ends it"""
    rng = np.random.default_rng(52)
    docs = seqs_of(rng, 3000, "AGCUN", 1, 32)
    eng.db_load(R.pack(docs, bits=4))
    more = ["ACGU" * 10] + seqs_of(rng, 50, "AGCU", 1, 32)
    eng.db_append(R.pack(more, bits=4))
    docs = docs + more
    check_layout(eng, *codes_of(R, docs))
    assert_same_results(R, eng, fresh(R, ref, docs), ["ACGUACGU", "ACGU" * 9, "ACGUN"], golden["default_costs"])


def test_append_of_symbols_the_database_did_not_hold(R, eng, ref, golden):
    rng = np.random.default_rng(53)
    docs = seqs_of(rng, 1500, "AGCU", 0, 30)
    eng.db_load(R.pack(docs, bits=4))
    more = seqs_of(rng, 400, "YRWSKM", 1, 30)
    eng.db_append(R.pack(more, bits=4))
    docs = docs + more
    check_layout(eng, *codes_of(R, docs))
    assert_same_results(R, eng, fresh(R, ref, docs), ["ACGUAC", "YRWSKM"], golden["default_costs"])


# ---------------------------------------------------------------------------------------------------------------------
# 4, 5: the idf table across its 2^20 chunk, the search across its 2^21 chunk and the 4096-record seed chunk
# ---------------------------------------------------------------------------------------------------------------------
def big_collection(rng, n, lo=8, hi=31):
    lens = rng.integers(lo, hi + 1, size=n)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    codes = rng.integers(0, 4, size=int(off[-1]), dtype=np.uint8)
    codes[rng.random(codes.shape[0]) < 0.002] = 14                     # N: a small general-path tail
    return codes, off


def part(codes, off, i0, i1):
    return codes[off[i0]:off[i1]], off[i0:i1 + 1] - off[i0]


@pytest.mark.parametrize("built_before", [True, False])
def test_idf_continued_across_its_chunk(R, eng, ref, built_before):
    rng = np.random.default_rng(61)
    n0, n = IDF_CHUNK - 700, IDF_CHUNK + 900
    codes, off = big_collection(rng, n)
    eng.db_load(R.pack(part(codes, off, 0, n0), bits=4))
    if built_before:
        assert_table(eng, *part(codes, off, 0, n0))
    eng.db_append(R.pack(part(codes, off, n0, n), bits=4))
    assert_table(eng, codes, off)
    ref.db_load(R.pack((codes, off), bits=4))
    qc = [codes[off[i]:off[i + 1]] for i in (3, n - 2)]
    for vt in VTS:
        for method in ("cosine", "pearson"):
            ga = eng.db_similarity_batch(qc, method, k=20, vector_type=vt)
            gb = ref.db_similarity_batch(qc, method, k=20, vector_type=vt)
            assert same_bits(ga[0], gb[0]) and np.array_equal(ga[1], gb[1]) and same_bits(ga[2], gb[2]), (vt, method)


@pytest.mark.parametrize("n0,n", [(SEED_CHUNK - 100, SEED_CHUNK + 300), (SEARCH_CHUNK - 500, SEARCH_CHUNK + 1500)])
def test_append_across_search_chunks(R, eng, ref, golden, n0, n):
    rng = np.random.default_rng(n0)
    codes, off = big_collection(rng, n)
    eng.db_load(R.pack(part(codes, off, 0, n0), bits=4))
    eng.db_append(R.pack(part(codes, off, n0, n - 7), bits=4))
    eng.db_append(R.pack(part(codes, off, n - 7, n), bits=4))
    check_layout(eng, codes, off)
    ref.db_load(R.pack((codes, off), bits=4))
    queries = [R.decode(codes[off[i]:off[i + 1]]) for i in (0, n0 + 3, n - 1)]
    assert_same_results(R, eng, ref, queries, golden["default_costs"], idf=False, sims=n < SEED_CHUNK * 2)


# ---------------------------------------------------------------------------------------------------------------------
# 6: a shard loaded with global_index_base != 0
# ---------------------------------------------------------------------------------------------------------------------
def test_append_continues_the_global_index(R, eng, ref, golden):
    rng = np.random.default_rng(71)
    base = 10_000
    docs = seqs_of(rng, 900, "AGCUN", 0, 30)
    eng.db_load(R.pack(docs, bits=4), global_index_base=base)
    more = seqs_of(rng, 400, "AGCUN", 0, 30)
    eng.db_append(R.pack(more, bits=4))
    docs = docs + more
    check_layout(eng, *codes_of(R, docs), base=base)
    fresh(R, ref, docs, base=base)
    assert_same_results(R, eng, ref, ["ACGUN", docs[950]], golden["default_costs"], idf=False)
    idx, _ = eng.db_search_topk(R.pack([docs[1200]], bits=4), 3)
    assert idx[0, 0] == base + 1200 or docs[idx[0, 0] - base] == docs[1200]


# ---------------------------------------------------------------------------------------------------------------------
# 7: MultiEngine: the appends go to the last shard; every device gets the continued idf table
# ---------------------------------------------------------------------------------------------------------------------
def test_multi_engine_appends(R, ref, golden):
    rng = np.random.default_rng(81)
    pool = ["".join(rng.choice(list("AGCUN"), size=int(m))) for m in rng.integers(4, 30, size=10)]
    docs = seqs_of(rng, 3000, "AGCUN", 0, 30, 0.3, pool)
    me = R.MultiEngine([0, 0, 0])
    try:
        me.db_load(R.pack(docs, bits=4))
        me.db_idf_table()
        for n_add in (500, 0, 1200):
            more = seqs_of(rng, n_add, "AGCUNYR", 0, 30, 0.3, pool)
            me.db_append(R.pack(more, bits=4))
            docs = docs + more
            assert_same_results(R, me, fresh(R, ref, docs), [pool[1], "ACGUAGCUN", "YRYR"], golden["default_costs"])
        assert_table(me, *codes_of(R, docs))
    finally:
        me.close()


# ---------------------------------------------------------------------------------------------------------------------
# 8: refusals leave the database as it was
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals(R, eng, golden):
    lib = R.load_library()
    rng = np.random.default_rng(91)
    docs = seqs_of(rng, 500, "AGCU", 0, 30)
    good = R.pack(seqs_of(rng, 20, "AGCU", 1, 30), bits=2)
    P = lambda a, t: a.ctypes.data_as(C.POINTER(t))

    def call(p, n=None, n_words=None, bits=None, symmask=None, words=True, start=True, length=True, ctx=None):
        return lib.rsd_db_append(ctx or eng._ctx, P(p.words, C.c_uint32) if words else None, P(p.start, C.c_int64) if start else None,
                                 P(p.len, C.c_int32) if length else None, p.n if n is None else n,
                                 p.words.shape[0] if n_words is None else n_words, p.bits if bits is None else bits,
                                 p.symmask if symmask is None else symmask)

    empty = R.Engine(0)
    assert call(good, ctx=empty._ctx) == RSD_EINVAL                   # no database loaded
    eng.set_costs(golden["default_costs"])
    eng.db_load(R.pack(docs, bits=2))
    Q = R.pack(["ACGUACGU", docs[3]], bits=2)
    before = (eng.db_layout(), eng.db_search_topk(Q, 10, want_scores=True), eng.db_idf_table())
    neg = R.pack(["ACGU", "GG"], bits=2); neg.len = neg.len.copy(); neg.len[1] = -1
    out = R.pack(["ACGU", "GG"], bits=2); out.start = out.start.copy(); out.start[1] = out.words.shape[0]
    cases = [call(good, bits=4), call(good, symmask=0x4F), call(neg), call(out), call(good, n_words=0),
             call(good, words=False), call(good, start=False), call(good, length=False), call(good, n=-1)]
    assert cases == [RSD_EINVAL] * len(cases)
    assert call(good, n=0, words=False, start=False, length=False) == 0        # an empty batch changes nothing
    after = (eng.db_layout(), eng.db_search_topk(Q, 10, want_scores=True), eng.db_idf_table())
    for x, y in zip(before, after):
        for u, v in zip(x, y):
            assert same_bits(u, v)
    assert lib.rsd_multi_db_append(None, None, None, None, 0, 0, 4, 0) == RSD_EINVAL


# ---------------------------------------------------------------------------------------------------------------------
# 9: ir._Resident appends the documents a collection gained instead of reloading it
# ---------------------------------------------------------------------------------------------------------------------
class Counted:
    """instance-level wrappers that count db_load / db_append"""

    def __init__(self, eng):
        self.loads = self.appends = 0
        load, append = eng.db_load, eng.db_append

        def db_load(*a, **k):
            self.loads += 1
            return load(*a, **k)

        def db_append(*a, **k):
            self.appends += 1
            return append(*a, **k)
        eng.db_load, eng.db_append = db_load, db_append


def test_resident_appends_a_grown_collection(R, golden):
    from rna_sequence_diff_patch_b200 import ir
    costs = golden["default_costs"]
    rng = np.random.default_rng(101)
    e, f = R.Engine(0), R.Engine(0)
    cnt = Counted(e)

    def same(x, y):                                     # [(sequence, score)] lists, NaN where NaN
        return [u for u, _ in x] == [u for u, _ in y] and same_bits([v for _, v in x], [v for _, v in y])

    def fresh_ir(fn, *args, **kw):
        f.db_free()                                                                   # a new generation: f reloads
        return fn(*args, engine=f, **kw)
    try:
        # the upper-case rule (score_collection, range_collection)
        L = seqs_of(rng, 1200, "AGCUY", 0, 30)
        assert same(ir.score_collection("ACGUAG", L[:700], costs, engine=e), fresh_ir(ir.score_collection, "ACGUAG", L[:700], costs))
        assert (cnt.loads, cnt.appends) == (1, 0)
        assert same(ir.score_collection("ACGUAG", L, costs, engine=e), fresh_ir(ir.score_collection, "ACGUAG", L, costs))
        assert (cnt.loads, cnt.appends) == (1, 1)
        assert ir.range_collection("ACGUAG", L, 4.0, costs, engine=e) == fresh_ir(ir.range_collection, "ACGUAG", L, 4.0, costs)
        assert (cnt.loads, cnt.appends) == (1, 1)
        # the as-stored rule (similarity_collection): not a prefix of the held upper-case copy -> a reload, then appends
        U = seqs_of(rng, 1500, "AGCUN", 0, 30)
        for vt in ("tf", "tf-idf"):
            a = ir.similarity_collection("ACGUAG", U[:900], "cosine", engine=e, vector_type=vt)
            assert same(a, fresh_ir(ir.similarity_collection, "ACGUAG", U[:900], "cosine", vector_type=vt))
        assert (cnt.loads, cnt.appends) == (2, 1)
        for n in (1400, 1500):
            for vt in ("tf-idf", "idf"):
                a = ir.similarity_collection("ACGUAG", U[:n], "pearson", engine=e, vector_type=vt)
                assert same(a, fresh_ir(ir.similarity_collection, "ACGUAG", U[:n], "pearson", vector_type=vt))
        assert (cnt.loads, cnt.appends) == (2, 3)
        assert same(ir.score_collection("ACGUAG", U, costs, engine=e), fresh_ir(ir.score_collection, "ACGUAG", U, costs))
        assert (cnt.loads, cnt.appends) == (2, 3)                                     # upper(U) == U: held as is
        changed = ["UUUU"] + U[1:] + ["GGGA"]                                          # an earlier record changed: reload
        assert same(ir.similarity_collection("ACGUAG", changed, "dice_dist", engine=e),
                    fresh_ir(ir.similarity_collection, "ACGUAG", changed, "dice_dist"))
        assert (cnt.loads, cnt.appends) == (3, 3)
    finally:
        ir._Resident.held.pop(e, None); ir._Resident.held.pop(f, None)


def test_dropin_search_collection_appends(R, dropin):
    """the reference's call site: an import adds records at the end of the collection, and the next
    search_collection appends them to the resident copy instead of reloading it"""

    class Coll:
        def __init__(self, docs):
            self.docs = docs

        def find(self, _q):
            return [{"sequence": s} for s in self.docs]

    from rna_sequence_diff_patch_b200 import ir
    eng = R.get_search_engine()
    rng = np.random.default_rng(111)
    coll = Coll(seqs_of(rng, 400, "AGCU", 1, 30))
    dropin.IR.search_collection("ACGUAGC", "tf", coll, dropin.IR.wf_score)
    cnt = Counted(eng)
    f = R.Engine(0)
    try:
        for _ in range(2):
            coll.docs = coll.docs + seqs_of(rng, 500, "AGCUN", 1, 30)                  # fa_import.py: 500 per run
            got = dropin.IR.search_collection("ACGUAGC", "tf", coll, dropin.IR.wf_score)
            f.db_free()                                                                 # f: a fresh load each time
            assert got == ir.score_collection("ACGUAGC", coll.docs, dropin.SED.default_costs, engine=f)
        assert (cnt.loads, cnt.appends) == (0, 2)
    finally:
        del eng.db_load, eng.db_append
        ir._Resident.held.pop(f, None)
