"""GPU parity at the edges of the numeric modes (DESIGN §2).

The library is exact because the host picks a narrow integer kernel only while every value it holds fits its type.
Each test here puts a batch on the last shape (or table) inside such a bound and on the first one outside, checks the
mode chosen on both sides, compares every result with the oracle with ==, and, where the oracle's distances give the
peak value the kernel held, asserts that the batch came within 10 % of the bound.  The edges are found with the host
classifier (Engine.classify) or, for the two bounds it does not expose, with the formulas restated in tests/_edges.py,
so a loosened bound moves the test to the shape that overflows."""
import numpy as np
import pytest

import _edges as E
from _synth import mutate_codes
from oracle import oracle as O

pytestmark = pytest.mark.gpu

I16X2, I32, F64 = 1, 2, 3
N_LIMIT = 65000.0              # int16x2: N = -H' in an unsigned 16-bit lane
H_LIMIT = 2147483000.0         # int32 distance kernels: |H'|
NEAR = 0.9                     # how close to the bound an inside batch must come


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


def rand_str(rng, L, alphabet):
    al = np.array(list(alphabet))
    return "".join(al[rng.integers(0, len(al), size=L)])


def homolog(rng, s, L, alphabet):
    """s with 5 % substitutions, 2.5 % insertions and 2.5 % deletions, trimmed or padded to L symbols"""
    idx = np.array([alphabet.index(ch) for ch in s], np.uint8)
    t = "".join(alphabet[c] for c in mutate_codes(rng, idx, alpha=len(alphabet)))
    return (t + rand_str(rng, max(0, L - len(t)), alphabet))[:L]


def edge_batch(rng, m, n, alphabet, n_small=8):
    """pairs of the shape (m, n) where the values peak (N = i*del + j*ins - D is largest where D is small): one pair
    of identical sequences (a prefix of the other when m != n), two homologous pairs and a random one; then small
    random pairs, empty sequences included"""
    base = rand_str(rng, max(m, n), alphabet)
    a, b = [base[:m]], [base[:n]]
    for _ in range(2):
        s = rand_str(rng, m, alphabet)
        a.append(s); b.append(homolog(rng, s, n, alphabet))
    a.append(rand_str(rng, m, alphabet)); b.append(rand_str(rng, n, alphabet))
    for _ in range(n_small):
        a.append(rand_str(rng, int(rng.integers(0, min(m, 200) + 1)), alphabet))
        b.append(rand_str(rng, int(rng.integers(0, min(n, 200) + 1)), alphabet))
    return a, b


def oracle_dist(a, b, costs):
    ac, ao = O.concat(a); bc, bo = O.concat(b)
    return O.distance_batch(ac, ao, bc, bo, costs)


def peak(a, b, d, costs, k):
    """the largest m*del + n*ins - D over the batch, scaled by 2^k: -H' (int16x2: N) at the last cell of each pair"""
    la = np.array([len(x) for x in a], np.float64); lb = np.array([len(x) for x in b], np.float64)
    return float(((la * costs["delete"] + lb * costs["insert"] - d) * 2.0 ** k).max())


def symmask_of(alphabet):
    return sum(1 << c for c in set(E.codes_of(alphabet)))


def dev_distances(R, eng, A, B, n_pairs, max_m, max_n, symmask):
    """rsd_distance_batch_dev on torch device tensors, on a side stream that is synchronised before the read"""
    import torch
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t = [torch.from_numpy(np.ascontiguousarray(x if x.size else np.zeros(1, x.dtype))).cuda()
             for x in (A.words, A.start, A.len, B.words, B.start, B.len)]
        out = torch.full((max(n_pairs, 1),), -1.0, dtype=torch.float64, device="cuda")
    mode = eng.distance_batch_dev(*[x.data_ptr() for x in t], n_pairs, max_m, max_n, A.bits, symmask, out.data_ptr(),
                                  side.cuda_stream)
    side.synchronize()
    return out.cpu().numpy(), mode


def check_entry_points(R, eng, a, b, costs, mode, monkeypatch):
    """distance_batch, distance_batch_codes and distance_batch_dev (exact max_m / max_n, both overstated, n_pairs of
    1 and 0) equal the oracle; each reports `mode` for the batch as it stands.  -> the oracle's distances"""
    monkeypatch.setenv("RSD_DIST_NO_LONG", "1")          # pairs of >= 6144 symbols stay on the batch kernels
    eng.set_costs(costs)
    want = oracle_dist(a, b, costs)
    bits = 2 if set("".join(a + b)) <= set("AGCU") else 4
    A, B = R.pack(a, bits=bits), R.pack(b, bits=bits)
    symmask = A.symmask | B.symmask
    n = len(a)
    got = eng.distance_batch(A, B)
    assert eng.last_mode == mode
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
    ac, ao = O.concat(a); bc, bo = O.concat(b)
    got = eng.distance_batch_codes(ac, np.diff(ao).astype(np.int32), bc, np.diff(bo).astype(np.int32), bits=bits,
                                   symmask=symmask)
    assert eng.last_mode == mode
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
    got, m = dev_distances(R, eng, A, B, n, A.max_len, B.max_len, symmask)
    assert m == mode
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
    # lengths overstated by the caller (allowed): the mode may move across the edge, the distances must not change
    got, _ = dev_distances(R, eng, A, B, n, 2 * A.max_len + 7, B.max_len + 64, symmask)
    assert np.array_equal(got, want), np.flatnonzero(got != want)[:8]
    got, _ = dev_distances(R, eng, A, B, 1, A.max_len, B.max_len, symmask)
    assert got[0] == want[0]
    got, m = dev_distances(R, eng, A, B, 0, A.max_len, B.max_len, symmask)
    assert m == mode and got[0] == -1.0                     # nothing written
    return want


# ---------------------------------------------------------------------------------------------------------------------
# k_dist_twin16: the byte table of v = ins + del - sub, and N = -H' < 65000 in both orientations
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 2])
def test_twin16_byte_table_edge(R, eng, monkeypatch, k):
    """ins + del = 127 (x 2^-k): v = 127 still fits the sign-extended byte, the substitutions spread v over 0..127;
    the longest square batch the table allows, one symbol longer, and the same batch with ins + del = 128"""
    rng = np.random.default_rng(100 + k)
    inside, outside = E.v_table(k), E.v_table(k, ins_del=(64, 64))
    eng.set_costs(inside)
    assert eng.classify(0xF, 1, 1) == (I16X2, k)
    e = E.last_inside(lambda x: eng.classify(0xF, x, x)[0] == I16X2, 1, 1 << 20)
    a, b = edge_batch(rng, e, e, "AGCU")
    d = check_entry_points(R, eng, a, b, inside, I16X2, monkeypatch)
    assert peak(a, b, d, inside, k) >= NEAR * N_LIMIT
    a1, b1 = edge_batch(rng, e + 1, e + 1, "AGCU")
    check_entry_points(R, eng, a1, b1, inside, I32, monkeypatch)
    eng.set_costs(outside)
    assert eng.classify(0xF, 1, 1) == (I32, k)
    check_entry_points(R, eng, a, b, outside, I32, monkeypatch)


@pytest.mark.parametrize("which", ["default_costs", "user_costs"])
def test_twin16_length_edge(R, eng, golden, monkeypatch, which):
    """the shipped tables on A/G/C/U: the longest square batch that keeps N < 65000 (32 466 / 12 960), and one longer"""
    costs = golden[which]
    rng = np.random.default_rng(7 if which == "user_costs" else 8)
    eng.set_costs(costs)
    e = E.last_inside(lambda x: eng.classify(0xF, x, x)[0] == I16X2, 1, 1 << 20)
    k = eng.classify(0xF, e, e)[1]
    a, b = edge_batch(rng, e, e, "AGCU")
    d = check_entry_points(R, eng, a, b, costs, I16X2, monkeypatch)
    assert peak(a, b, d, costs, k) >= NEAR * N_LIMIT
    a, b = edge_batch(rng, e + 1, e + 1, "AGCU")
    check_entry_points(R, eng, a, b, costs, I32, monkeypatch)


@pytest.mark.parametrize("ins,dele,m", [(27, 100, 40), (100, 27, 200)])
def test_twin16_asymmetric_edge(R, eng, monkeypatch, ins, dele, m):
    """m rows fixed, n grows: (27, 100) is bounded by the swapped orientation, (100, 27) by the stored one — the
    kernel may take either (plan_swap), so both must fit.  N <= min(m, n) * (ins + del) here: no closeness check."""
    costs = E.table(ins, dele, E.SUBS_V)
    rng = np.random.default_rng(ins)
    eng.set_costs(costs)
    e = E.last_inside(lambda n: eng.classify(0xF, m, n)[0] == I16X2, m, 1 << 20)
    a, b = edge_batch(rng, m, e, "AGCU")
    check_entry_points(R, eng, a, b, costs, I16X2, monkeypatch)
    a, b = edge_batch(rng, m, e + 1, "AGCU")
    check_entry_points(R, eng, a, b, costs, I32, monkeypatch)


# ---------------------------------------------------------------------------------------------------------------------
# k_dist_gen<int>: |H'| < 2147483000, the scale 2^k (k <= 16) and scaled costs below 2^30
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alphabet", ["AGCU", "AGCUNRY"])
def test_int32_magnitude_edge(R, eng, monkeypatch, alphabet):
    """every cost 2^20, 2-bit and 4-bit packing: the longest square batch whose |H'| fits an int32, and one longer"""
    costs = E.uniform(2.0 ** 20)
    mask = symmask_of(alphabet)
    rng = np.random.default_rng(len(alphabet))
    eng.set_costs(costs)
    e = E.last_inside(lambda x: eng.classify(mask, x, x)[0] == I32, 1, 1 << 20)
    a, b = edge_batch(rng, e, e, alphabet)
    d = check_entry_points(R, eng, a, b, costs, I32, monkeypatch)
    assert peak(a, b, d, costs, 0) >= NEAR * H_LIMIT
    a, b = edge_batch(rng, e + 1, e + 1, alphabet)
    check_entry_points(R, eng, a, b, costs, F64, monkeypatch)


@pytest.mark.parametrize("name,mode,k", [("K16_SMALL", I16X2, 16), ("K16_WIDE", I32, 16), ("K17", F64, 0),
                                         ("DEAR_IN", I32, 0), ("DEAR_OUT", F64, 0)])
def test_scale_and_cost_width_edges(R, eng, monkeypatch, name, mode, k):
    """costs in units of 2^-16 (the finest scale) run on the integer kernels; one cost of 2^-17 goes to fp64.  A
    substitution of 2^30 - 1 still fits the int32 tables, 2^30 does not."""
    costs = getattr(E, name)
    eng.set_costs(costs)
    assert eng.classify(0xF, 300, 300) == (mode, k)
    a, b = edge_batch(np.random.default_rng(len(name)), 300, 300, "AGCU")
    check_entry_points(R, eng, a, b, costs, mode, monkeypatch)


# ---------------------------------------------------------------------------------------------------------------------
# k_script_fwd<false>: (cost << S | steps) keys below 2^30, else k_script_fwd<true>
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [1000, 2000])
def test_script_key_edge(R, eng, monkeypatch, m):
    """ins = del = sub = c on m x m pairs: the largest c whose keys fit (by the restated bound) runs int32 keys and
    the next one fp64, while distance_batch stays int32 for both; scripts equal the oracle's canonical scripts"""
    monkeypatch.setenv("RSD_SCRIPT_NO_LONG", "1")
    fits = lambda c: E.script_key_bound(E.uniform(c), "AGCU", 0, m, m)[0] < E.SCRIPT_KEY_LIMIT
    c0 = E.last_inside(fits, 1, 1 << 20)
    rng = np.random.default_rng(m)
    a, b = edge_batch(rng, m, m, "AGCU", n_small=6)
    A, B = R.pack(a), R.pack(b)
    ac, ao = O.concat(a); bc, bo = O.concat(b)
    for c, want_mode in ((c0, I32), (c0 + 1, F64)):
        costs = E.uniform(float(c))
        eng.set_costs(costs)
        res = eng.script_batch(A, B, check_roundtrip=True)
        assert eng.last_mode == want_mode, (c, eng.last_mode)
        ops, oi, oj, cnt, dist = O.script_batch(ac, ao, bc, bo, costs)
        assert np.array_equal(res["dist"], dist) and np.array_equal(res["n_ops"], cnt) and res["ok"].all()
        for p in range(len(a)):
            kk = cnt[p]
            assert np.array_equal(res["op"][p, :kk], ops[p, :kk]), (c, p)
            assert np.array_equal(res["oi"][p, :kk], oi[p, :kk]) and np.array_equal(res["oj"][p, :kk], oj[p, :kk]), (c, p)
        assert np.array_equal(eng.distance_batch(A, B), dist) and eng.last_mode == I32
        if want_mode == I32:
            S = E.script_key_bound(costs, "AGCU", 0, m, m)[1]
            assert peak(a, b, dist, costs, S) >= NEAR * E.SCRIPT_KEY_LIMIT


# ---------------------------------------------------------------------------------------------------------------------
# k_long2: 32-bit modular keys while (64 maxc + 128) << S < 2^30, else the exact-double kernels
# ---------------------------------------------------------------------------------------------------------------------
LONG_SUBS = [0, 700, 1500, 2045, 2100, 2500, 3000, 4090, 350, 1023, 1800, 4000]      # |sub - ins - del| <= 2045
_long_oracle = {}


def long_pairs_3000():
    rng = np.random.default_rng(3000)
    a, b = edge_batch(rng, 3000, 3000, "AGCU", n_small=0)
    return [(np.array(E.codes_of(x), np.uint8), np.array(E.codes_of(y), np.uint8)) for x, y in zip(a, b)]


@pytest.mark.parametrize("lanes", [4, 8, 16])
def test_long_pair_key32_edge(R, eng, monkeypatch, capfd, lanes):
    """3000 x 3000 (S = 13): maxc = 2045 (ins 1022, del 1023) is the largest the 32-bit keys allow and runs k_long2
    (4 / 8 / 16 columns per lane); maxc = 2046 runs the exact-double fallback.
    The path shows in the RSD_TRACE output: only k_long2 batches print a 'long batch:' line."""
    monkeypatch.setenv("RSD_TRACE", "1")
    monkeypatch.setenv("RSD_LONG_C", str(lanes))
    pairs = long_pairs_3000()
    for (ins, dele), want32 in (((1022, 1023), True), ((1023, 1023), False)):
        costs = E.table(ins, dele, LONG_SUBS)
        assert all(E.long_key32_ok(costs, "AGCU", 0, a.shape[0], b.shape[0]) == want32 for a, b in pairs)
        eng.set_costs(costs)
        capfd.readouterr()
        res = eng.long_pairs(pairs)
        err = capfd.readouterr().err
        assert ("long batch:" in err) == want32, err[-400:]
        for p, (r, (a, b)) in enumerate(zip(res, pairs)):
            key = (ins, dele, p)
            if key not in _long_oracle:
                _long_oracle[key] = O.canonical_script(O.decode(a), O.decode(b), costs)
            ops, oi, oj, d = _long_oracle[key]
            assert r["mode"] == I32
            assert r["dist"] == d, (ins, dele, p)
            assert np.array_equal(r["op"], ops) and np.array_equal(r["oi"], oi) and np.array_equal(r["oj"], oj), (ins, dele, p)


# ---------------------------------------------------------------------------------------------------------------------
# k_search_twin16: <= 7 symbols, queries <= 64, records <= 32, v <= 127
# ---------------------------------------------------------------------------------------------------------------------
def search_check(R, eng, costs, recs, queries, want_mode, k=10):
    eng.set_costs(costs)
    codes, off = O.concat(recs)
    eng.db_load(R.pack(recs, bits=4))
    try:
        idx, sc, alls = eng.db_search_topk(R.pack(queries, bits=4), k, want_scores=True)
        mode = eng.last_mode
    finally:
        eng.db_free()
    assert mode == want_mode, (mode, want_mode)
    for q, query in enumerate(queries):
        wi, ws, wa = O.search_topk(query, codes, off, costs, k, want_scores=True)
        assert np.array_equal(alls[q], wa), q
        assert np.array_equal(idx[q], wi) and np.array_equal(sc[q], ws), q


def search_db(rng, n, alphabet, hi=32):
    recs = [rand_str(rng, int(L), alphabet) for L in rng.integers(20, hi + 1, size=n)]
    recs[0] = rand_str(rng, hi, alphabet)
    return recs


def int_table(rng):
    """integer costs over every symbol: dyadic with v <= 6, so only the symbol count and the lengths decide"""
    upd = {a: {b: (0.0 if a == b else float(rng.integers(1, 5))) for b in E.SYM} for a in E.SYM}
    return {"insert": 2.0, "delete": 3.0, "update": upd}


def test_search_fast_prefix_symbol_edge(R, eng):
    """7 distinct symbols keep the int16x2 search kernel, an 8th (W) in the query sends every record to the general
    kernels; W in a few records sends only those"""
    rng = np.random.default_rng(77)
    costs = int_table(rng)
    recs = search_db(rng, 3000, "AGCUNRY")
    qs = [recs[5], recs[100][:25], rand_str(rng, 30, "AGCUNRY")]
    assert len(set("".join(recs + qs))) == 7
    search_check(R, eng, costs, recs, qs, I16X2)
    search_check(R, eng, costs, recs, qs[:2] + [qs[2][:10] + "W" + qs[2][11:]], I32)
    recs_w = recs + [rand_str(rng, 28, "AGCUNRYW") for _ in range(5)]
    search_check(R, eng, costs, recs_w, qs, I32)


def test_search_fast_prefix_length_edges(R, eng):
    """queries of 64 symbols keep the fast kernel, 65 do not; records of 32 keep it, one record of 33 does not"""
    rng = np.random.default_rng(64)
    costs = int_table(rng)
    recs = search_db(rng, 3000, "AGCUN")
    q64 = (recs[3] + recs[4] + rand_str(rng, 64, "AGCUN"))[:64]
    qs = [q64, recs[7], rand_str(rng, 40, "AGCUN")]
    search_check(R, eng, costs, recs, qs, I16X2)
    search_check(R, eng, costs, recs, [q64 + "A"] + qs[1:], I32)
    search_check(R, eng, costs, recs + [rand_str(rng, 33, "AGCUN")], qs, I32)


def test_search_fast_prefix_v_edge(R, eng):
    """v = ins + del - sub = 127 keeps the fast kernel (scores spread over the whole byte table), 128 does not"""
    rng = np.random.default_rng(127)
    recs = search_db(rng, 3000, "AGCUN")
    qs = [recs[11], recs[12][:20] + rand_str(rng, 40, "AGCUN"), rand_str(rng, 64, "AGCUN")]
    search_check(R, eng, E.v_table(), recs, qs, I16X2)
    search_check(R, eng, E.v_table(ins_del=(64, 64)), recs, qs, I32)


# ---------------------------------------------------------------------------------------------------------------------
# fp64 kernels: borders are products i*del, j*ins (as in the reference), not running sums
# ---------------------------------------------------------------------------------------------------------------------
FP = E.table(0.1, 0.3, [0.2, 0.7, 0.35, 0.6, 0.15, 0.9, 0.25, 0.55, 0.05, 0.8, 0.45, 0.65], other=0.3)


def border_pairs(rng, alphabet, core_lo, core_hi, prefix_lens):
    """b = P + a (the best path may insert P along row 0) and a = P + b (deletes along column 0), P of the given
    lengths, then random and empty pairs"""
    a, b = [], []
    for L in prefix_lens:
        s = rand_str(rng, int(rng.integers(core_lo, core_hi + 1)), alphabet)
        a.append(s); b.append(rand_str(rng, L, alphabet) + s)
        a.append(rand_str(rng, L, alphabet) + s); b.append(s)
    for _ in range(10):
        a.append(rand_str(rng, int(rng.integers(0, core_hi)), alphabet)); b.append(rand_str(rng, int(rng.integers(0, core_hi)), alphabet))
    a += ["", rand_str(rng, 17, alphabet)]; b += [rand_str(rng, 23, alphabet), ""]
    return a, b


def assert_products_matter(a, b, d, costs):
    """some pair's distance is exactly a border product that differs from the running sum"""
    ins, dele = costs["insert"], costs["delete"]
    di, dd = set(E.border_sums_differ(ins, 4096)), set(E.border_sums_differ(dele, 4096))
    hit = [p for p in range(len(a)) if (len(b[p]) - len(a[p]) in di and d[p] == (len(b[p]) - len(a[p])) * ins)
           or (len(a[p]) - len(b[p]) in dd and d[p] == (len(a[p]) - len(b[p])) * dele)]
    assert hit


def test_fp64_borders_distance_and_script(R, eng):
    rng = np.random.default_rng(1)
    lens = [6, 10, 17, 33, 64, 150]
    assert set(lens) <= set(E.border_sums_differ(0.1, 200)) & set(E.border_sums_differ(0.3, 200))
    eng.set_costs(FP)
    for alphabet in ("AGCU", "AGCUN"):
        a, b = border_pairs(rng, alphabet, 5, 200, lens)
        want = oracle_dist(a, b, FP)
        assert_products_matter(a, b, want, FP)
        A, B = R.pack(a), R.pack(b)
        assert np.array_equal(eng.distance_batch(A, B), want) and eng.last_mode == F64
        assert np.array_equal(eng.distance_batch(A, B, force_mode=F64), want) and eng.last_mode == F64
        res = eng.script_batch(A, B, check_roundtrip=True)
        assert eng.last_mode == F64
        ops, oi, oj, cnt, dist = O.script_batch(*O.concat(a), *O.concat(b), FP)
        assert np.array_equal(res["dist"], dist) and np.array_equal(res["n_ops"], cnt) and res["ok"].all()
        for p in range(len(a)):
            kk = cnt[p]
            assert np.array_equal(res["op"][p, :kk], ops[p, :kk]) and np.array_equal(res["oi"][p, :kk], oi[p, :kk]), p


def test_fp64_borders_long_pair_and_matrix(R, eng):
    rng = np.random.default_rng(2)
    eng.set_costs(FP)
    a, b = border_pairs(rng, "AGCU", 1500, 2500, [33, 1000])
    a, b = a[:4], b[:4]
    for x, y in zip(a, b):
        r = eng.long_pair(np.array(E.codes_of(x), np.uint8), np.array(E.codes_of(y), np.uint8))
        ops, oi, oj, d = O.canonical_script(x, y, FP)
        assert r["mode"] == F64 and r["dist"] == d
        assert np.array_equal(r["op"], ops) and np.array_equal(r["oi"], oi) and np.array_equal(r["oj"], oj)
    assert_products_matter(a, b, oracle_dist(a, b, FP), FP)
    x = rand_str(rng, 200, "AGCUN")
    for xa, yb in ((x, rand_str(rng, 40, "AGCUN") + x), (rand_str(rng, 26, "AGCUN") + x, x)):
        vals, mask = eng.matrix(np.array(E.codes_of(xa), np.uint8), np.array(E.codes_of(yb), np.uint8))
        wv, wm = O.matrix(xa, yb, FP)
        assert np.array_equal(vals, wv) and np.array_equal(mask, wm)
        assert vals[0, -1] == (len(yb)) * FP["insert"] and vals[-1, 0] == len(xa) * FP["delete"]


def test_fp64_borders_search_general_path(R, eng):
    rng = np.random.default_rng(3)
    qs = [rand_str(rng, 12, "AGCU") for _ in range(3)]
    recs = search_db(rng, 2000, "AGCU")
    for q in qs:
        for L in (6, 10, 17, 20):
            recs.append(rand_str(rng, L, "AGCU") + q)
            recs.append(q + rand_str(rng, L, "AGCU"))
    search_check(R, eng, FP, recs, qs + [recs[-1]], F64)
