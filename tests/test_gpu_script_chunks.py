"""The batched script path (rsd_ctx::script_pipeline behind rsd_script_batch and rsd_script_patch_check_batch) when its
direction words are cut into several chunks of pairs.

The path keeps 2 bits per cell of direction words on the device.  When a batch's words exceed a budget (70 % of the free
device memory), it runs plan -> k_script_fwd -> k_traceback -> k_finalize once per chunk: direction offsets restart at 0,
the temporary op rows are sized for the largest chunk and reused, each chunk re-plans in the same plan slot, and each
chunk's op / oi / oj rows go back on the copy stream while the next chunk computes (the events of that hand-off are a
ring of 16).  How many chunks a call runs therefore depends on the free memory of the device at the time of the call.
RSD_SCRIPT_BUDGET_WORDS sets the budget of one call, so these tests run the chunked layouts on small batches.

Each test first checks, from the RSD_TRACE line of the call, that the call ran the number of chunks the split rule
(chunk_starts, restated below) gives; then it compares every result with == against the C oracle and against the same
call without the budget, which runs as one chunk."""
import ctypes as C
import re

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_script import mutate, rand_seqs

gpu = pytest.mark.gpu

KNOB = "RSD_SCRIPT_BUDGET_WORDS"
RING = 16                        # RSD_MAX_CHUNKS: the copy stream's ev_done events are reused after this many chunks
_u8, _i32, _i64, _u32, _f64 = C.c_uint8, C.c_int32, C.c_int64, C.c_uint32, C.c_double


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
# the split rule of script_pipeline
# ---------------------------------------------------------------------------------------------------------------------
def words_of(m, n, cols):
    """direction words of an m x n pair: 16 rows per word, columns padded to whole lanes of `cols` (32 in the int32 mode,
    16 in fp64); 0 when a side is empty (the planner answers such pairs without the forward kernel)"""
    return -(-m // 16) * (-(-n // cols) * cols)


class TooSmall(Exception):
    pass


def chunk_starts(m, n, cols, max_ops, budget):
    """-> the first pair of every chunk.  A new chunk starts at pair p when the current one holds words and its words,
    p's words and the temporary op rows of its pairs up to p ((p - start + 1) * max_ops bytes) exceed the budget;
    TooSmall(p) when pair p alone does not fit"""
    starts, acc = [0], 0
    for p in range(len(m)):
        w = words_of(int(m[p]), int(n[p]), cols)
        if acc > 0 and acc + w + (p - starts[-1] + 1) * max_ops // 4 > budget:
            starts.append(p)
            acc = 0
        if w + max_ops // 4 > budget:
            raise TooSmall(p)
        acc += w
    return starts


def test_split_rule_restatement():
    """the restated rule on hand-counted cases (no device needed)"""
    assert words_of(0, 500, 32) == words_of(500, 0, 32) == 0
    assert words_of(17, 33, 32) == 2 * 64 and words_of(17, 33, 16) == 2 * 48 and words_of(16, 32, 32) == 32
    w = words_of(1500, 1500, 32)                                        # 94 * 1504
    assert chunk_starts([1500] * 6, [1500] * 6, 32, 3000, 3 * w + 2250) == [0, 3]      # 3 pairs: 3 * 3000 // 4 op words
    assert chunk_starts([1500] * 6, [1500] * 6, 32, 3000, 3 * w + 2249) == [0, 2, 4]
    assert chunk_starts([0, 1500, 0], [1500, 1500, 0], 32, 3000, w + 750) == [0, 2]   # trivial pairs add only op rows
    with pytest.raises(TooSmall) as ei:
        chunk_starts([10, 1500], [10, 1500], 32, 3000, w + 749)
    assert ei.value.args == (1,)


# ---------------------------------------------------------------------------------------------------------------------
# data: C3-shaped pairs per numeric mode and cost table, the oracle's scripts computed once
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = {            # alphabet, packing, script mode, scale k of the integer mode
    "acgu-2bit": ("AGCU", 2, 2, None),
    "acgun-4bit-int32-k2": ("AGCUAGCUAGCUN", 4, 2, 2),
    "iupac15-4bit-fp64": ("AGCUYRWSKMDVHBN", 4, 3, None),
}
DATASETS = [(s, t) for s in SHAPES for t in ("default", "user")]
N_PAIRS = 250

_data = {}


class Data:
    def __init__(self, R, a, b, bits, mode, costs):
        self.a, self.b, self.bits, self.mode, self.costs = a, b, bits, mode, costs
        self.cols = 16 if mode == 3 else 32
        self.m = np.array([len(s) for s in a]); self.n = np.array([len(s) for s in b])
        self.A, self.B = R.pack(a, bits=bits), R.pack(b, bits=bits)
        ac, ao = O.concat(a); bc, bo = O.concat(b)
        self.want = O.script_batch(ac, ao, bc, bo, costs)              # op, oi, oj, n_ops, dist
        self.words = np.array([words_of(int(x), int(y), self.cols) for x, y in zip(self.m, self.n)])

    def max_ops(self, idx):
        return max(int((self.m[idx] + self.n[idx]).max()), 1)


def dataset(R, eng, golden, shape, table):
    key = (shape, table)
    if key not in _data:
        alphabet, bits, mode, k = SHAPES[shape]
        rng = np.random.default_rng(20261022 + DATASETS.index(key))
        a = rand_seqs(rng, N_PAIRS, 1000, 2000, alphabet)
        b = [mutate(rng, s, list(alphabet))[:2000] if p % 10 else rand_seqs(rng, 1, 1000, 2000, alphabet)[0]
             for p, s in enumerate(a)]
        d = Data(R, a, b, bits, mode, golden[f"{table}_costs"])
        if k is not None:
            eng.set_costs(d.costs)
            assert eng.classify(d.A.symmask | d.B.symmask, d.A.max_len, d.B.max_len, force_mode=2) == (2, k)
        _data[key] = d
    eng.set_costs(_data[key].costs)
    return _data[key]


def layout(d, name):
    """-> (pairs of the batch, budget, chunk starts) of a named layout"""
    idx = np.arange(len(d.a))
    mo = d.max_ops(idx)
    whole = int(d.words.sum()) + len(idx) * mo // 4
    if name == "two":
        budget = whole * 6 // 10
    elif name in ("uneven", "threshold", "threshold-1"):
        budget = whole * 28 // 100
        if name != "uneven":
            # the threshold of the first split: at this budget its pair joins the first chunk, one word below it does not
            s1 = chunk_starts(d.m, d.n, d.cols, mo, budget)[1]
            budget = int(d.words[:s1 + 1].sum()) + (s1 + 1) * mo // 4 - (name == "threshold-1")
            assert chunk_starts(d.m, d.n, d.cols, mo, budget)[1] == s1 + (name == "threshold")
    elif name == "ring":
        budget = whole // 40
    elif name == "one-per-pair":
        # pairs of more than half the largest pair's words: no two of them fit a budget of one pair plus its op rows
        idx = np.flatnonzero(2 * d.words > d.words.max())
        mo = d.max_ops(idx)
        budget = int(d.words[idx].max()) + mo // 4
    starts = chunk_starts(d.m[idx], d.n[idx], d.cols, mo, budget)
    sizes = np.diff(starts + [len(idx)])
    assert {"two": len(starts) == 2, "uneven": 3 <= len(starts) <= 5 and len(set(sizes)) > 1,
            "ring": len(starts) > 2 * RING, "one-per-pair": (sizes == 1).all() and len(idx) > 100,
            "threshold": len(starts) > 2, "threshold-1": len(starts) > 2}[name], (name, sizes)
    return idx, budget, starts


# ---------------------------------------------------------------------------------------------------------------------
# calls, the trace, comparisons
# ---------------------------------------------------------------------------------------------------------------------
_TRACE = re.compile(r"\[rsd trace\] script: .* (\d+) chunk\(s\)")


def traced(monkeypatch, capfd, budget, fn, trace=True):
    """fn() with the budget knob set (None: unset) and RSD_TRACE on or off -> (result, [chunk count of each script call])"""
    for k, v in ((KNOB, budget), ("RSD_TRACE", 1 if trace else None)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))
    capfd.readouterr()
    res = fn()
    counts = [int(c) for c in _TRACE.findall(capfd.readouterr().err)]
    monkeypatch.delenv(KNOB, raising=False)
    monkeypatch.delenv("RSD_TRACE", raising=False)
    return res, counts


def op_only(R, eng, A, B, max_ops):
    """rsd_script_patch_check_batch through ctypes with oi = oj = NULL, as tools/bench_configs.py calls it for C3"""
    lib, p_ = R.load_library(), R._lib.ptr
    n = A.n
    op = np.zeros((n, max_ops), np.uint8); n_ops = np.zeros(n, np.int32); dist = np.zeros(n, np.float64)
    ok = np.zeros(n, np.uint8); mode = C.c_int()
    R._lib.check(lib.rsd_script_patch_check_batch(
        eng.ctx, p_(A.words, _u32), p_(A.start, _i64), p_(A.len, _i32), A.words.shape[0],
        p_(B.words, _u32), p_(B.start, _i64), p_(B.len, _i32), B.words.shape[0],
        n, A.bits, A.symmask | B.symmask, 0, max_ops, p_(op, _u8), None, None, p_(n_ops, _i32), p_(dist, _f64),
        p_(ok, _u8), C.byref(mode)))
    eng.last_mode = mode.value
    return dict(op=op, n_ops=n_ops, dist=dist, ok=ok)


def entry_call(R, eng, entry, A, B, max_ops):
    if entry == "script":
        return lambda: eng.script_batch(A, B)
    if entry == "roundtrip":
        return lambda: eng.script_batch(A, B, check_roundtrip=True)
    assert entry == "op-only"
    return lambda: op_only(R, eng, A, B, max_ops)


def check_oracle(res, want, idx):
    """n_ops, dist and the rows up to n_ops == the oracle's (pairs idx of its batch); ok, where returned, all set"""
    op, oi, oj, cnt, dist = want
    assert np.array_equal(res["n_ops"], cnt[idx]) and np.array_equal(res["dist"], dist[idx])
    for q, p in enumerate(idx):
        k = cnt[p]
        for key, rows in (("op", op), ("oi", oi), ("oj", oj)):
            if key in res:
                assert np.array_equal(res[key][q, :k], rows[p, :k]), (p, key)
    if "ok" in res:
        assert res["ok"].all()


def check_same(x, y):
    assert x.keys() == y.keys()
    assert np.array_equal(x["n_ops"], y["n_ops"]) and np.array_equal(x["dist"], y["dist"])
    if "ok" in x:
        assert np.array_equal(x["ok"], y["ok"])
    for key in ("op", "oi", "oj"):
        if key in x:
            for p, k in enumerate(x["n_ops"]):
                assert np.array_equal(x[key][p, :k], y[key][p, :k]), (p, key)


def run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, n_chunks, entry, A, B):
    """the call under the budget (traced: n_chunks chunks; == the oracle), again untraced (the trace synchronises the
    stream after the kernels; the unsynchronised run must agree), then without the budget (one chunk: the forced calls
    left the measured budget alone; == the chunked results) -> (chunked, one-chunk results)"""
    fn = entry_call(R, eng, entry, A, B, d.max_ops(idx))
    res, counts = traced(monkeypatch, capfd, budget, fn)
    assert counts == [n_chunks]
    assert eng.last_mode == d.mode
    check_oracle(res, d.want, idx)
    again, counts = traced(monkeypatch, capfd, budget, fn, trace=False)
    assert counts == []
    check_same(again, res)
    one, counts = traced(monkeypatch, capfd, None, fn)
    assert counts == [1]
    check_same(one, res)
    return res, one


# ---------------------------------------------------------------------------------------------------------------------
# 1. layouts x numeric modes x cost tables
# ---------------------------------------------------------------------------------------------------------------------
LAYOUTS = ["two", "uneven", "one-per-pair", "ring", "threshold", "threshold-1"]


@gpu
@pytest.mark.parametrize("layout_name", LAYOUTS)
@pytest.mark.parametrize("shape,table", DATASETS, ids=[f"{s}-{t}" for s, t in DATASETS])
def test_chunk_layouts(R, eng, golden, monkeypatch, capfd, shape, table, layout_name):
    """Engine.script_batch on 250 pairs of 1-2 kb (90 % homologous) in 2 chunks, 3-5 uneven chunks, one pair per chunk,
    more than 32 chunks (the ring of 16 copy events wraps twice) and a budget at the threshold of a split and one word
    below it; the patch of the chunked scripts == the patch of the one-chunk scripts (== B)"""
    d = dataset(R, eng, golden, shape, table)
    idx, budget, starts = layout(d, layout_name)
    A, B = (d.A, d.B) if len(idx) == len(d.a) else (R.pack([d.a[p] for p in idx], bits=d.bits),
                                                    R.pack([d.b[p] for p in idx], bits=d.bits))
    res, one = run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, len(starts), "script", A, B)
    out, out_len, err = eng.patch_batch(res, A, B, A)
    ref = eng.patch_batch(one, A, B, A)
    assert not err.any()
    for x, y in zip((out, out_len, err), ref):
        assert np.array_equal(x, y)
    for q, p in enumerate(idx):
        assert R.decode(out[q, :out_len[q]]) == d.b[p], p


# ---------------------------------------------------------------------------------------------------------------------
# 2. the round-trip entry point, with all rows and with op rows only
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("layout_name", ["uneven", "ring"])
@pytest.mark.parametrize("entry", ["roundtrip", "op-only"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_roundtrip_entry_points(R, eng, golden, monkeypatch, capfd, shape, entry, layout_name):
    """rsd_script_patch_check_batch chunked: through Engine.script_batch(check_roundtrip=True) (op, oi, oj rows cross
    per chunk) and through ctypes with oi = oj = NULL (only op rows cross): every round trip ok, scripts == the oracle"""
    d = dataset(R, eng, golden, shape, "default")
    idx, budget, starts = layout(d, layout_name)
    run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, len(starts), entry, d.A, d.B)


# ---------------------------------------------------------------------------------------------------------------------
# 3. mid-length pairs: a single pair fills a chunk
# ---------------------------------------------------------------------------------------------------------------------
_mid = {}


@gpu
@pytest.mark.parametrize("entry", ["roundtrip", "no-long"])
@pytest.mark.parametrize("shape", ["acgu-2bit", "iupac15-4bit-fp64"])
def test_mid_length_pairs(R, eng, golden, monkeypatch, capfd, shape, entry):
    """10 pairs of 4.2-6 kb (more than 128 strips of 32 columns: the planner's class of single-group tasks) through the
    round-trip entry point, which never routes to the panel kernels, and through script_batch with RSD_SCRIPT_NO_LONG=1;
    budgets of the largest pair alone (its words plus its op rows fill the budget exactly) and of about three pairs"""
    if shape not in _mid:
        alphabet, bits, mode, _ = SHAPES[shape]
        rng = np.random.default_rng(4206)
        a = rand_seqs(rng, 10, 4200, 6000, alphabet)
        b = [mutate(rng, s, list(alphabet))[:6000] if p % 10 else rand_seqs(rng, 1, 4200, 6000, alphabet)[0]
             for p, s in enumerate(a)]
        _mid[shape] = Data(R, a, b, bits, mode, golden["default_costs"])
    d = _mid[shape]
    eng.set_costs(d.costs)
    assert min(map(len, d.b)) > 128 * 32
    if entry == "no-long":
        monkeypatch.setenv("RSD_SCRIPT_NO_LONG", "1")
    idx = np.arange(len(d.a))
    mo = d.max_ops(idx)
    big = int(np.argmax(d.words))
    lone = int(d.words[big]) + mo // 4
    for budget in (lone, (int(d.words.sum()) + len(idx) * mo // 4) // 3):
        starts = chunk_starts(d.m, d.n, d.cols, mo, budget)
        assert len(starts) >= 3
        if budget == lone:
            assert big in starts and big + 1 in starts + [len(idx)]
        run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, len(starts),
                    "roundtrip" if entry == "roundtrip" else "script", d.A, d.B)


# ---------------------------------------------------------------------------------------------------------------------
# 4. trivial pairs: no direction words, but op rows
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["empty-source", "empty-destination", "both-empty"])
def test_trivial_pairs_at_chunk_edges(R, eng, golden, monkeypatch, capfd, kind):
    """Pairs with an empty side add no direction words but their op rows count toward the temporary-op term.  Nine
    1500 x 1500 pairs P and four trivial pairs E as  E P P P | E P P P | P P P E | E : a trivial pair first in the batch,
    first in a chunk, last in a chunk and alone in the last chunk; every call == the oracle"""
    rng = np.random.default_rng(44)
    L = 1500
    pattern = "EPPPEPPPPPPEE"
    a, b = [], []
    for c in pattern:
        s = rand_seqs(rng, 1, L, L, "AGCU")[0]
        if c == "P":
            a.append(s); b.append((mutate(rng, s, "AGCU") + s)[:L])
        else:
            a.append("" if kind != "empty-destination" else s)
            b.append("" if kind != "empty-source" else s)
    d = Data(R, a, b, 2, 2, golden["default_costs"])
    eng.set_costs(d.costs)
    idx = np.arange(len(a))
    mo = d.max_ops(idx)
    assert mo == 2 * L
    budget = 3 * words_of(L, L, 32) + mo                   # three P plus the op rows of four pairs fill a chunk exactly
    starts = chunk_starts(d.m, d.n, d.cols, mo, budget)
    assert starts == [0, 4, 8, 12]
    E = [p for p, c in enumerate(pattern) if c == "E"]
    assert E == [0, 4, 11, 12]
    for entry in ("script", "roundtrip", "op-only"):
        run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, len(starts), entry, d.A, d.B)


# ---------------------------------------------------------------------------------------------------------------------
# 5. a budget below one pair
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_budget_below_one_pair_is_an_error(R, eng, golden, monkeypatch, capfd):
    """One word less than the largest pair's words plus max_ops / 4: RsdError RSD_ENOMEM naming that pair (its first
    occurrence).  The engine's next calls, chunked and unchunked, are still correct, and the unchunked one runs as one
    chunk"""
    d = dataset(R, eng, golden, "acgu-2bit", "default")
    idx = np.arange(len(d.a))
    mo = d.max_ops(idx)
    big = int(np.argmax(d.words))
    budget = int(d.words[big]) + mo // 4 - 1
    with pytest.raises(TooSmall) as ei:
        chunk_starts(d.m, d.n, d.cols, mo, budget)
    assert ei.value.args == (big,)
    for entry in ("script", "roundtrip"):
        monkeypatch.setenv(KNOB, str(budget))
        with pytest.raises(R.RsdError) as ei:
            entry_call(R, eng, entry, d.A, d.B, mo)()
        assert ei.value.code == R._lib.RSD_ENOMEM and f"pair {big} needs" in str(ei.value), str(ei.value)
    monkeypatch.delenv(KNOB)
    _, budget, starts = layout(d, "uneven")
    run_chunked(R, eng, monkeypatch, capfd, d, idx, budget, len(starts), "script", d.A, d.B)
