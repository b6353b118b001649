"""GPU parity: the long-pair path (panel wavefront + traceback) vs the oracle and via properties."""
import hashlib
import json
import os

import numpy as np
import pytest

from _synth import c4_pair, mutate_codes
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


def apply_script(op, oj, b):
    """closed-form patch on the host: destination symbols of the non-delete ops"""
    keep = op != 1
    return b[oj[keep] - 1]


@pytest.mark.parametrize("shape", [(3000, 3000), (5000, 777), (300, 4100), (1, 700), (257, 256), (2049, 2048)])
def test_long_pair_vs_oracle(R, eng, golden, shape):
    rng = np.random.default_rng(sum(shape))
    m, n = shape
    a = rng.integers(0, 4, size=m, dtype=np.uint8)
    b = mutate_codes(rng, a)[:n] if m == n else rng.integers(0, 4, size=n, dtype=np.uint8)
    for costs, modes in ((golden["default_costs"], (0, 3)), (golden["user_costs"], (0,))):
        eng.set_costs(costs)
        ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), costs)
        for force in modes:
            res = eng.long_pair(a, b, force_mode=force)
            assert res["mode"] == (3 if force == 3 else 2)
            assert res["dist"] == d
            assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)


def test_long_pair_iupac_fp64(R, eng, golden):
    rng = np.random.default_rng(77)
    a = rng.integers(0, 15, size=2500, dtype=np.uint8)
    b = mutate_codes(rng, a, alpha=15, p_sub=0.1)
    eng.set_costs(golden["default_costs"])
    res = eng.long_pair(a, b)
    assert res["mode"] == 3
    ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), golden["default_costs"])
    assert res["dist"] == d and np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi)


def test_empty_sides(R, eng, golden):
    eng.set_costs(golden["user_costs"])
    a = np.array([0, 1, 2], np.uint8); e = np.zeros(0, np.uint8)
    r = eng.long_pair(a, e)
    assert r["dist"] == 9.0 and r["op"].tolist() == [1, 1, 1] and r["oi"].tolist() == [1, 2, 3]
    r = eng.long_pair(e, a)
    assert r["dist"] == 6.0 and r["op"].tolist() == [0, 0, 0] and r["oj"].tolist() == [1, 2, 3]


def _sha(arr, dt):
    return hashlib.sha256(np.ascontiguousarray(arr, dtype=dt).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def c4_digest():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "c4_digest.json")) as f:
        return json.load(f)


def _check_digest(res, rec):
    assert res["dist"] == float.fromhex(rec["dist"])
    assert res["op"].shape[0] == rec["n_ops"]
    assert _sha(res["op"], np.uint8) == rec["op_sha256"], "canonical script differs from the oracle's (ops)"
    assert _sha(res["oi"], np.int32) == rec["oi_sha256"] and _sha(res["oj"], np.int32) == rec["oj_sha256"]


def test_c4_canonical_script_equals_oracle_digest(R, eng, golden, c4_digest):
    """50 kb x 50 kb (BASELINE config 4), where the kernel's keys are carried modulo 2^32 and wrap: the whole
    canonical script (= create_paths(dp)[0], SED:228-271) must equal the oracle's, recorded as SHA-256 by
    tests/golden/make_golden_c4.py; both cost tables, plus every other kernel variant on the default one."""
    a, b = c4_pair()
    for name in ("default_costs", "user_costs"):
        eng.set_costs(golden[name])
        res = eng.long_pair(a, b)
        assert res["mode"] == 2
        _check_digest(res, c4_digest["c4_" + name])
    rng = np.random.default_rng(20260044)
    a2 = rng.integers(0, 4, size=30000, dtype=np.uint8); b2 = rng.integers(0, 4, size=50000, dtype=np.uint8)
    _check_digest(eng.long_pair(a2, b2), c4_digest["random_30k_50k_user_costs"])


def test_c4_other_kernel_variants_equal_oracle_digest(R, eng, golden, c4_digest, monkeypatch):
    a, b = c4_pair()
    eng.set_costs(golden["default_costs"])
    for env in ({"RSD_LONG_WIDE": "1"}, {"RSD_LONG_C": "8"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        _check_digest(eng.long_pair(a, b), c4_digest["c4_default_costs"])
        for k in env:
            monkeypatch.delenv(k)
    _check_digest(eng.long_pair(a, b, force_mode=3), c4_digest["c4_default_costs"])     # fp64 kernel, same script


def test_30k_pair_vs_oracle_in_the_wrap_regime(R, eng, golden):
    """30 kb x 30 kb: i*del + j*ins passes 2^(31-S) (S = 16) half-way through the matrix, so the second half runs
    on wrapped keys; compared with the oracle run here (about 6 s of CPU)."""
    rng = np.random.default_rng(30030)
    a = rng.integers(0, 4, size=30000, dtype=np.uint8)
    b = mutate_codes(rng, a, p_sub=0.08, p_ins=0.04, p_del=0.04)
    costs = golden["user_costs"]
    eng.set_costs(costs)
    ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), costs)
    res = eng.long_pair(a, b)
    assert res["mode"] == 2 and res["dist"] == d
    assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)


@pytest.mark.parametrize("S", [19, 21])
def test_forced_wide_steps_field_wraps_small_matrices(R, eng, golden, monkeypatch, S):
    """RSD_LONG_S widens the steps field so the modular keys wrap after 2^(31-S) border units: at S = 21 a
    3 k x 3 k matrix wraps six times (user costs: del 3, ins 2) — every (cost, steps) comparison still has to
    order the candidates like the oracle."""
    monkeypatch.setenv("RSD_LONG_S", str(S))
    for seed, (m, n) in enumerate([(3000, 3000), (2500, 3300), (1200, 4000)]):
        rng = np.random.default_rng(900 + seed)
        a = rng.integers(0, 4, size=m, dtype=np.uint8)
        b = mutate_codes(rng, a)[:n] if seed == 0 else rng.integers(0, 4, size=n, dtype=np.uint8)
        for costs in (golden["user_costs"], golden["default_costs"]):
            eng.set_costs(costs)
            ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), costs)
            res = eng.long_pair(a, b)
            assert res["mode"] == 2 and res["dist"] == d
            assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)


def test_c4_shape_properties(R, eng, golden):
    """50 kb x 50 kb: size-independent properties next to the digest — (i) the script is a valid path whose cost
    equals the reported distance, (ii) patching A with it gives B, (iii) the distance agrees with the batched
    distance kernel (independent code path)."""
    a, b = c4_pair()
    eng.set_costs(golden["default_costs"])
    res = eng.long_pair(a, b)
    op, oi, oj = res["op"], res["oi"], res["oj"]
    assert oi[-1] == a.shape[0] and oj[-1] == b.shape[0]
    di = np.diff(np.concatenate([[0], oi])); dj = np.diff(np.concatenate([[0], oj]))
    assert np.array_equal(di, (op != 0).astype(np.int64)) and np.array_equal(dj, (op != 1).astype(np.int64))
    upd = op == 2
    cost = float((op != 2).sum() + (a[oi[upd] - 1] != b[oj[upd] - 1]).sum())
    assert cost == res["dist"]
    assert np.array_equal(apply_script(op, oj, b), b)
    off_a = np.array([0, a.shape[0]], np.int64); off_b = np.array([0, b.shape[0]], np.int64)
    d = eng.distance_batch(R.pack((a, off_a)), R.pack((b, off_b)))
    assert d[0] == res["dist"]


def test_wide_key_fallback_paths_agree(R, eng, golden, monkeypatch):
    """The 32-bit key kernel (k_long2) is the default; the double-carried integer key kernel is the fallback, forced
    here through RSD_LONG_WIDE and reached naturally by costs too large for the 32-bit bound."""
    rng = np.random.default_rng(77)
    a = rng.integers(0, 4, size=2600, dtype=np.uint8)
    b = mutate_codes(rng, a)
    costs = golden["default_costs"]
    eng.set_costs(costs)
    ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), costs)
    fast = eng.long_pair(a, b)
    monkeypatch.setenv("RSD_LONG_WIDE", "1")
    wide = eng.long_pair(a, b)
    monkeypatch.delenv("RSD_LONG_WIDE")
    for res in (fast, wide):
        assert res["mode"] == 2 and res["dist"] == d
        assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)
    # integer costs in the thousands: (32 * maxc + 64) << S exceeds 2^30 -> the wide kernel is chosen by the library
    big = {"insert": 3000.0, "delete": 2500.0,
           "update": {x: {y: (0.0 if x == y else 4100.0 + 7 * ((ord(x) + 3 * ord(y)) % 11)) for y in "AGCUYRWSKMDVHBN"} for x in "AGCUYRWSKMDVHBN"}}
    eng.set_costs(big)
    ops, oi, oj, d = O.canonical_script(O.decode(a), O.decode(b), big)
    res = eng.long_pair(a, b)
    assert res["mode"] == 2 and res["dist"] == d
    assert np.array_equal(res["op"], ops) and np.array_equal(res["oi"], oi) and np.array_equal(res["oj"], oj)
