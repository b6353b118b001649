"""GPU parity of the band layout of the int16x2 distance kernel (k_dist_band16, DESIGN §4).

The band kernel computes only the diagonal band of cells an optimal path can reach, so its distances must equal the
oracle's and the tape kernel's (k_dist_twin16) with ==.  Each case forces the layout with RSD_DIST_BAND and reads the
RSD_TRACE line of the band launch to know which kernel ran.  The shapes aim at the places the band can go wrong: a band
of width zero, optima along the band's edge, loose bounds, both orientations of the plan, warps that mix row counts,
the ends of the word buffers and the chunked host paths."""
import numpy as np
import pytest

import _edges as E
from oracle import oracle as O

pytestmark = pytest.mark.gpu

I16X2 = 1
SYM = "AGCU"


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


def rand_str(rng, L):
    return "".join(np.array(list(SYM))[rng.integers(0, 4, size=L)])


def dev_distances(eng, A, B, symmask):
    import torch
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        # device buffers of exactly the packed words: no padding after the last sequence
        t = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (A.words, A.start, A.len, B.words, B.start, B.len)]
        out = torch.full((A.n,), -1.0, dtype=torch.float64, device="cuda")
    eng.distance_batch_dev(*[x.data_ptr() for x in t], A.n, A.max_len, B.max_len, A.bits, symmask, out.data_ptr(),
                           side.cuda_stream)
    side.synchronize()
    return out.cpu().numpy()


def run(R, eng, a, b, costs, band, monkeypatch, capfd, entries=("batch", "codes", "dev")):
    """distances of every entry point with the layout forced -> (list of arrays, whether every launch was the band kernel,
    whether any was)"""
    monkeypatch.setenv("RSD_DIST_NO_LONG", "1")
    monkeypatch.setenv("RSD_TRACE", "1")
    monkeypatch.setenv("RSD_DIST_BAND", "1" if band else "0")
    eng.set_costs(costs)
    A, B = R.pack(a, bits=2), R.pack(b, bits=2)
    symmask = A.symmask | B.symmask
    capfd.readouterr()
    outs = []
    for e in entries:
        if e == "batch":
            outs.append(eng.distance_batch(A, B))
        elif e == "codes":
            ac, ao = O.concat(a); bc, bo = O.concat(b)
            outs.append(eng.distance_batch_codes(ac, np.diff(ao).astype(np.int32), bc, np.diff(bo).astype(np.int32),
                                                 bits=2, symmask=symmask))
        else:
            outs.append(dev_distances(eng, A, B, symmask))
        assert eng.last_mode == I16X2
    err = capfd.readouterr().err
    return outs, err.count("k_dist_band16:")


def check(R, eng, a, b, costs, monkeypatch, capfd, expect_band=True, entries=("batch", "codes", "dev")):
    """every entry point, band forced and tape forced, equals the oracle"""
    ac, ao = O.concat(a); bc, bo = O.concat(b)
    want = O.distance_batch(ac, ao, bc, bo, costs)
    got_band, n_band = run(R, eng, a, b, costs, True, monkeypatch, capfd, entries)
    got_tape, n_tape = run(R, eng, a, b, costs, False, monkeypatch, capfd, entries)
    assert n_tape == 0
    assert (n_band > 0) == expect_band, n_band
    for g in got_band + got_tape:
        assert np.array_equal(g, want), np.flatnonzero(g != want)[:8]
    return want


@pytest.mark.parametrize("which", ["user_costs", "default_costs"])
def test_band_c2_batch(R, eng, monkeypatch, capfd, which):
    """the bench distribution: ACGU, lengths U[100, 300]; 70 000 pairs so the host entry points cut it into chunks"""
    from rna_sequence_diff_patch_b200 import cost_tables
    costs = getattr(cost_tables, which)()
    eng.set_costs(costs)
    if eng.classify(0xF, 300, 300)[0] != I16X2:
        pytest.skip("table not exact in int16x2")
    rng = np.random.default_rng(11)
    n = 70000 if which == "user_costs" else 8000
    la = rng.integers(100, 301, size=n); lb = rng.integers(100, 301, size=n)
    a = [rand_str(rng, int(x)) for x in la]
    b = [rand_str(rng, int(x)) for x in lb]
    check(R, eng, a, b, costs, monkeypatch, capfd)


def related_batch(rng, m, n_pairs=96):
    """identical pairs (q = 0), one indel, a rotation (the diagonal bound is loose, the optimum uses long gaps),
    a prefix and random pairs, all of about m symbols"""
    a, b = [], []
    for k in range(n_pairs):
        s = rand_str(rng, m)
        kind = k % 6
        if kind == 0:
            t = s
        elif kind == 1:                                   # one deletion
            p = int(rng.integers(0, m)); t = s[:p] + s[p + 1:]
        elif kind == 2:                                   # one insertion
            p = int(rng.integers(0, m + 1)); t = s[:p] + rand_str(rng, 1) + s[p:]
        elif kind == 3:                                   # rotation
            p = int(rng.integers(1, m)); t = s[p:] + s[:p]
        elif kind == 4:
            t = s[: int(rng.integers(1, m))]
        else:
            t = rand_str(rng, int(rng.integers(m // 2, 2 * m)))
        a.append(s); b.append(t)
    return a, b


@pytest.mark.parametrize("m", [33, 150, 257])
def test_band_related_pairs(R, eng, monkeypatch, capfd, m):
    from rna_sequence_diff_patch_b200 import cost_tables
    costs = cost_tables.user_costs()
    a, b = related_batch(np.random.default_rng(m), m)
    check(R, eng, a, b, costs, monkeypatch, capfd)


def test_band_identical_only(R, eng, monkeypatch, capfd):
    """every pair identical: every band has width zero (q = 0), D = 0"""
    from rna_sequence_diff_patch_b200 import cost_tables
    rng = np.random.default_rng(3)
    a = [rand_str(rng, int(x)) for x in rng.integers(1, 400, size=200)]
    d = check(R, eng, a, list(a), cost_tables.user_costs(), monkeypatch, capfd)
    assert not d.any()


@pytest.mark.parametrize("swap", [False, True])
def test_band_100_vs_300(R, eng, monkeypatch, capfd, swap):
    """m = 100 against n = 300 and the reverse: the plan takes the orientation with less strip padding"""
    from rna_sequence_diff_patch_b200 import cost_tables
    rng = np.random.default_rng(100 + swap)
    a = [rand_str(rng, 100) for _ in range(130)]
    b = [rand_str(rng, 300) if k % 2 else a[k] + rand_str(rng, 200) for k in range(130)]
    if swap:
        a, b = b, a
    check(R, eng, a, b, cost_tables.user_costs(), monkeypatch, capfd)


@pytest.mark.parametrize("ins,dele", [(2, 3), (5, 1)])
def test_band_v_zero(R, eng, monkeypatch, capfd, ins, dele):
    """every substitution costs ins + del (v = 0): many optimal paths, some along the band's edge"""
    costs = E.table(ins, dele, [ins + dele] * 12)
    a, b = related_batch(np.random.default_rng(ins), 120)
    check(R, eng, a, b, costs, monkeypatch, capfd)


@pytest.mark.parametrize("ins,dele", [(0, 3), (2, 0)])
def test_band_zero_gap_cost_routes_to_tape(R, eng, monkeypatch, capfd, ins, dele):
    """ins = 0 or del = 0 leaves the band unbounded: the forced band layout falls back to the tape kernel"""
    costs = E.table(ins, dele, [0, 1, 2, 1, 2, 0, 2, 1, 1, 1, 0, 1])
    a, b = related_batch(np.random.default_rng(ins + 7), 90)
    check(R, eng, a, b, costs, monkeypatch, capfd, expect_band=False)


@pytest.mark.parametrize("n_pairs", [1, 3, 63, 65, 129])
def test_band_odd_twins(R, eng, monkeypatch, capfd, n_pairs):
    """one shape, an odd number of pairs: the last group has no twin; 65 and 129 leave a warp task partly empty"""
    from rna_sequence_diff_patch_b200 import cost_tables
    rng = np.random.default_rng(n_pairs)
    a = [rand_str(rng, 140) for _ in range(n_pairs)]
    b = [rand_str(rng, 170) for _ in range(n_pairs)]
    check(R, eng, a, b, cost_tables.user_costs(), monkeypatch, capfd)


def test_band_mixed_warp(R, eng, monkeypatch, capfd):
    """one strip class (161-192 columns) with neighbouring row counts and different n in one warp task; a short
    pair last in both word buffers, so the rows of longer pairs run past its end.  This checks the results of such a
    warp.  It cannot see whether the kernel's code loads of those rows stay inside the words buffer (the clamp to
    the pair's last word): an over-read of a few words lands in the same allocation and its codes are never used, so
    it neither faults nor changes a value."""
    from rna_sequence_diff_patch_b200 import cost_tables
    rng = np.random.default_rng(5)
    la = list(rng.integers(100, 111, size=77)) + [3]
    lb = list(rng.integers(161, 193, size=77)) + [170]
    a = [rand_str(rng, int(x)) for x in la]
    b = [rand_str(rng, int(x)) for x in lb]
    b[-1] = a[-1] * 56 + "AG"
    check(R, eng, a, b, cost_tables.user_costs(), monkeypatch, capfd)
    check(R, eng, b, a, cost_tables.user_costs(), monkeypatch, capfd)


def edge_pairs(rng, m, n, k=6):
    """pairs of the shape (m, n) where N peaks: a prefix pair, homologs and a random pair"""
    base = rand_str(rng, max(m, n))
    a, b = [base[:m]], [base[:n]]
    for _ in range(k):
        s = rand_str(rng, m)
        t = list(s[:n].ljust(n, "A"))
        for p in rng.integers(0, n, size=max(1, n // 50)):
            t[p] = SYM[int(rng.integers(0, 4))]
        a.append(s); b.append("".join(t))
    a.append(rand_str(rng, m)); b.append(rand_str(rng, n))
    return a, b


def test_band_length_edge(R, eng, monkeypatch, capfd):
    """the longest square batch int16x2 holds where that is inside the band kernel's strip classes (<= 4096 columns)"""
    costs = E.table(64, 63, E.SUBS_V)
    eng.set_costs(costs)
    e = E.last_inside(lambda x: eng.classify(0xF, x, x)[0] == I16X2, 1, 1 << 20)
    assert e <= 4096, e
    a, b = edge_pairs(np.random.default_rng(9), e, e)
    check(R, eng, a, b, costs, monkeypatch, capfd)


@pytest.mark.parametrize("ins,dele,m", [(27, 100, 40), (100, 27, 200)])
def test_band_asymmetric_edge(R, eng, monkeypatch, capfd, ins, dele, m):
    """m rows fixed, n at the last length int16x2 holds in both orientations"""
    costs = E.table(ins, dele, E.SUBS_V)
    eng.set_costs(costs)
    e = E.last_inside(lambda n: eng.classify(0xF, m, n)[0] == I16X2, m, 1 << 20)
    assert e <= 4096, e
    a, b = edge_pairs(np.random.default_rng(ins), m, e)
    check(R, eng, a, b, costs, monkeypatch, capfd)
