"""GPU parity: batches of long pairs (rsd_long_pairs: rings of CTAs) and the linear-space overflow path (row blocks
from checkpoint rows x panel ranges) vs the oracle's canonical script (= create_paths(dp)[0], SED:228-271)."""
import numpy as np
import pytest

from _synth import mutate_codes
from oracle import oracle as O

pytestmark = pytest.mark.gpu


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


def make_pairs(seed, shapes, alpha=4):
    rng = np.random.default_rng(seed)
    out = []
    for m, n in shapes:
        a = rng.integers(0, alpha, size=m, dtype=np.uint8)
        if m and n and abs(m - n) < m // 4:
            b = mutate_codes(rng, a, alpha=alpha)
            b = np.concatenate([b, rng.integers(0, alpha, size=max(0, n - b.shape[0]), dtype=np.uint8)])[:n]
        else:
            b = rng.integers(0, alpha, size=n, dtype=np.uint8)
        out.append((a, b))
    return out


def check(res, a, b, costs, script=True):
    ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), costs)
    assert res["dist"] == d
    if script:
        assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)


SHAPES = [(3000, 3100), (2000, 2500), (1000, 5000), (17, 4000), (4000, 33), (2047, 2049), (1, 1), (640, 640), (3333, 129)]


@pytest.mark.parametrize("rings", [1, 2, 4, 9])
def test_batch_of_pairs_vs_oracle(R, eng, golden, monkeypatch, rings):
    monkeypatch.setenv("RSD_LONG_RINGS", str(rings))
    pairs = make_pairs(100 + rings, SHAPES)
    for costs in (golden["default_costs"], golden["user_costs"]):
        eng.set_costs(costs)
        res = eng.long_pairs(pairs)
        assert len(res) == len(pairs)
        for r, (a, b) in zip(res, pairs):
            assert r["mode"] == 2
            check(r, a, b, costs)
    # distance only
    res = eng.long_pairs(pairs, want_script=False)
    for r, (a, b) in zip(res, pairs):
        check(r, a, b, costs, script=False)


def test_batch_with_empty_and_mixed_alphabets(R, eng, golden):
    """empty sides are answered on the host (border row / column, SED:146-182); an ACGU+N pair puts the whole call on
    the x4 dyadic scale of the default table; next to a full-IUPAC pair (0.66 / 0.83: not dyadic) only that pair goes to
    the fp64 kernel, the ACGU pair keeps the integer keys of its own symbols"""
    costs = golden["default_costs"]
    eng.set_costs(costs)
    e = np.zeros(0, np.uint8)
    pairs = make_pairs(5, [(900, 1000), (1500, 1400)])
    rng = np.random.default_rng(6)
    with_n = rng.integers(0, 4, size=1200, dtype=np.uint8); with_n[::37] = 14
    pairs.append((with_n, mutate_codes(rng, with_n)))
    res = eng.long_pairs(pairs + [(pairs[0][0], e), (e, pairs[0][1]), (e, e)])
    for r, (a, b) in zip(res[:3], pairs):
        assert r["mode"] == 2
        check(r, a, b, costs)
    assert res[3]["dist"] == 900.0 and res[3]["op"].tolist() == [1] * 900
    assert res[4]["dist"] == 1000.0 and res[4]["op"].tolist() == [0] * 1000 and res[4]["oj"].tolist() == list(range(1, 1001))
    assert res[5]["dist"] == 0.0 and res[5]["op"].shape[0] == 0
    iupac = make_pairs(8, [(800, 820)], alpha=15)
    res = eng.long_pairs(pairs[:1] + iupac)
    assert res[0]["mode"] == 2 and res[1]["mode"] == 3
    check(res[0], *pairs[0], costs)
    check(res[1], *iupac[0], costs)


@pytest.mark.parametrize("budget_mb,maxctas", [(4, 0), (2, 0), (0, 3), (2, 5), (3, 1)])
def test_overflow_path_row_blocks_and_panel_ranges(R, eng, golden, monkeypatch, budget_mb, maxctas):
    """RSD_LONG_BUDGET_MB forces the row-block path (checkpoint rows, recomputation bottom to top), RSD_LONG_MAXCTAS the
    panel ranges: distance and script must equal the oracle's, i.e. the one-launch result."""
    if budget_mb:
        monkeypatch.setenv("RSD_LONG_BUDGET_MB", str(budget_mb))
    if maxctas:
        monkeypatch.setenv("RSD_LONG_MAXCTAS", str(maxctas))
    shapes = [(5000, 5000), (3001, 4100), (4097, 1500), (700, 6000)]
    pairs = make_pairs(321, shapes)
    for costs in (golden["default_costs"], golden["user_costs"]):
        eng.set_costs(costs)
        for a, b in pairs:
            check(eng.long_pair(a, b), a, b, costs)
            check(eng.long_pair(a, b, want_script=False), a, b, costs, script=False)
        res = eng.long_pairs(pairs)                      # blocked pairs run alone inside a batch call
        for r, (a, b) in zip(res, pairs):
            check(r, a, b, costs)


def test_overflow_path_in_the_wrap_regime(R, eng, golden, monkeypatch):
    """checkpoint rows hold keys modulo 2^32: with a widened steps field (RSD_LONG_S) they wrap several times between
    the blocks of a 3 k x 3 k matrix"""
    monkeypatch.setenv("RSD_LONG_S", "21")
    monkeypatch.setenv("RSD_LONG_BUDGET_MB", "2")
    costs = golden["user_costs"]
    eng.set_costs(costs)
    for a, b in make_pairs(77, [(3000, 3000), (2500, 3300)]):
        res = eng.long_pair(a, b)
        assert res["mode"] == 2
        check(res, a, b, costs)
        check(eng.long_pair(a, b, want_script=False), a, b, costs, script=False)


def test_overflow_budget_too_small_is_an_error(R, eng, golden, monkeypatch):
    monkeypatch.setenv("RSD_LONG_BUDGET_MB", "0")
    eng.set_costs(golden["default_costs"])
    (a, b), = make_pairs(1, [(2000, 2000)])
    monkeypatch.setenv("RSD_LONG_BUDGET_MB", "0")
    with pytest.raises(R.RsdError):
        # 0 MB: nothing fits, not even 32-row blocks
        eng.long_pair(a, b)


def test_overflow_path_equals_one_launch_at_60kb(R, eng, golden, monkeypatch):
    """60 kb x 60 kb, beyond what the CPU oracle does in test time: the row-block / panel-range path must return the
    distance and script of the one-launch path (itself pinned to the oracle digest at 50 kb), for budgets that give
    3 and 12 row blocks and for panel ranges of 100 CTAs."""
    from _synth import c4_pair
    a, b = c4_pair(seed=6060, m=60000)
    eng.set_costs(golden["default_costs"])
    ref = eng.long_pair(a, b)
    assert ref["oi"][-1] == a.shape[0] and ref["oj"][-1] == b.shape[0]
    for env in ({"RSD_LONG_BUDGET_MB": "500"}, {"RSD_LONG_BUDGET_MB": "120"}, {"RSD_LONG_MAXCTAS": "100"},
                {"RSD_LONG_BUDGET_MB": "300", "RSD_LONG_MAXCTAS": "77"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        res = eng.long_pair(a, b)
        assert res["dist"] == ref["dist"]
        assert np.array_equal(res["op"], ref["op"]) and np.array_equal(res["oi"], ref["oi"]) and np.array_equal(res["oj"], ref["oj"])
        assert eng.long_pair(a, b, want_script=False)["dist"] == ref["dist"]
        for k in env:
            monkeypatch.delenv(k)


def _long_batches(err):
    return sum("long batch:" in line for line in err.splitlines())


@pytest.mark.parametrize("script", [True, False])
def test_mixed_symbol_batch_runs_each_pair_on_its_own_symbols(R, eng, golden, monkeypatch, capfd, script):
    """A call's cost tables cover the symbols of all its pairs.  A pair that does not fit the 32-bit keys on those tables
    is planned again on its own symbols: it runs on k_long2 when it fits there (one RSD_TRACE 'long batch:' line per
    k_long2 batch), and only a pair that does not fit alone goes to the exact-double / fp64 kernel."""
    monkeypatch.setenv("RSD_TRACE", "1")
    # (a) default table: the full-IUPAC pair is not dyadic (fp64); each ACGU pair runs alone on k_long2
    costs = golden["default_costs"]
    acgu = make_pairs(31, [(3000, 3100), (2000, 2100)])
    iupac = make_pairs(32, [(1500, 1600)], alpha=15)
    eng.set_costs(costs)
    capfd.readouterr()
    res = eng.long_pairs(acgu + iupac, want_script=script)
    err = capfd.readouterr().err
    assert [r["mode"] for r in res] == [2, 2, 3]
    assert _long_batches(err) == 2, err[-600:]
    for r, (a, b) in zip(res, acgu + iupac):
        check(r, a, b, costs, script=script)
    # (b) integer table where substitutions involving N cost thousands: the ACGU+N pair needs the exact-double kernel
    # (still integer keys: mode 2), the ACGU pair fits the 32-bit keys of its own symbols
    def sub(x, y):
        return 0.0 if x == y else 4000.0 + (x + y).count("A") if "N" in (x, y) else 1.0
    big_n = {"insert": 1.0, "delete": 1.0, "update": {x: {y: sub(x, y) for y in O.SYMBOLS} for x in O.SYMBOLS}}
    rng = np.random.default_rng(33)
    (a0, b0), = make_pairs(34, [(3000, 3000)])
    with_n = rng.integers(0, 4, size=2500, dtype=np.uint8); with_n[::41] = 14
    pairs = [(a0, b0), (with_n, mutate_codes(rng, with_n))]
    eng.set_costs(big_n)
    capfd.readouterr()
    res = eng.long_pairs(pairs, want_script=script)
    err = capfd.readouterr().err
    assert [r["mode"] for r in res] == [2, 2]
    assert _long_batches(err) == 1, err[-600:]
    for r, (a, b) in zip(res, pairs):
        check(r, a, b, big_n, script=script)
