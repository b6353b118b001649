"""The batched patch (rsd_patch_batch, Engine.patch_batch) and the on-device round-trip check
(rsd_script_patch_check_batch: k_script_fwd -> k_traceback -> k_finalize) at C3 shapes, and the path rule of the patch.

k_finalize scans a script in blocks of 256 ops and carries the consumed-source / produced-destination counts from block
to block; it patches with the closed form out = (destination symbols of the non-delete ops) ++ x[len(source):], which
is the reference's sequential patching (SED:380-457) exactly when the script is a path of its pair.  Every result is
compared with ==: against the C oracle's closed form (O.patch_closed_codes) and, on samples that cover every variant,
against sed.patching on the reference's op dicts.  Each test first asserts the layout it is about."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_script import mutate, rand_seqs

gpu = pytest.mark.gpu
OK, EINVAL, ENODEV = 0, 1, 2
BLOCK = 256                      # ops per block of k_finalize's scan, and the stride of its tail loop
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


@pytest.fixture(scope="module")
def sed():
    from rna_sequence_diff_patch_b200 import sed
    return sed


def codes(s):
    return O.encode(s) if s else np.zeros(0, np.uint8)


def rows(scripts, p):
    k = int(scripts["n_ops"][p])
    return scripts["op"][p, :k], scripts["oi"][p, :k], scripts["oj"][p, :k]


def es_of(sed, op, oi, oj, a, b):
    """the reference's op dicts of a packed script; an empty side is only indexed (at -1) by ops that never read it"""
    return sed.es_from_packed(op, oi, oj, a or "A", b or "A")


def check_patch(R, out, out_len, err, scripts, a, b, xs, sed=None, sample=()):
    """err / out_len / out of every pair == the oracle's closed form; nothing written past out_len; on `sample` also
    == sed.patching on the op dicts"""
    for p in range(len(a)):
        op, oi, oj = rows(scripts, p)
        code, want = O.patch_closed_codes(op, oi, oj, codes(a[p]), codes(b[p]), codes(xs[p]))
        assert err[p] == code, (p, err[p], code)
        assert out_len[p] == want.shape[0], p
        assert np.array_equal(out[p, :out_len[p]], want), p
        if code >= 0:
            assert not out[p, out_len[p]:].any(), p
    for p in sample:
        op, oi, oj = rows(scripts, p)
        assert sed.patching(es_of(sed, op, oi, oj, a[p], b[p]), xs[p]) == (int(err[p]), R.decode(out[p, :out_len[p]])), p


def raw_patch(R, ctx, op, oi, oj, n_ops, A, B, X, max_out):
    """rsd_patch_batch through ctypes with oi / oj optional (None = NULL) and a caller-chosen max_out -> (rc, out,
    out_len, err)"""
    lib = R.load_library()
    n = A.n
    out = np.zeros((n, max_out), np.uint8); out_len = np.zeros(n, np.int32); err = np.zeros(n, np.int32)
    p = R._lib.ptr
    rc = lib.rsd_patch_batch(ctx, p(op, _u8), None if oi is None else p(oi, _i32), None if oj is None else p(oj, _i32),
                             p(n_ops, _i32), op.shape[1],
                             p(A.words, _u32), p(A.start, _i64), p(A.len, _i32), A.words.shape[0],
                             p(B.words, _u32), p(B.start, _i64), p(B.len, _i32), B.words.shape[0],
                             p(X.words, _u32), p(X.start, _i64), p(X.len, _i32), X.words.shape[0],
                             n, A.bits, max_out, p(out, _u8), p(out_len, _i32), p(err, _i32))
    return rc, out, out_len, err


# ---------------------------------------------------------------------------------------------------------------------
# 1-2. C3 shapes: about 400 pairs of 1-2 kb, 90 % homologous, 10 % unrelated
# ---------------------------------------------------------------------------------------------------------------------
SHAPES = {            # alphabet, packing, script mode, scale k of the integer mode
    "acgu-2bit": ("AGCU", 2, 2, 0),
    "acgun-4bit-int32-k2": ("AGCUAGCUAGCUN", 4, 2, 2),
    "iupac15-4bit-fp64": ("AGCUYRWSKMDVHBN", 4, 3, None),
}
TAILS = (1, 255, 256, 257, 700)
FLIPS = (0, 255, 256, -1)
N_VARIANTS = 1 + len(TAILS) + len(FLIPS) + 3


def x_variant(rng, a, v, alphabet):
    """v-th patch input for source a: a; a + tail; a with one symbol changed; a[:-1], a[:m-300], ''"""
    if v == 0:
        return a
    v -= 1
    if v < len(TAILS):
        return a + "".join(rng.choice(list(alphabet), size=TAILS[v]))
    v -= len(TAILS)
    if v < len(FLIPS):
        i = FLIPS[v] % len(a)
        return a[:i] + next(c for c in alphabet if c != a[i]) + a[i + 1:]
    return (a[:-1], a[:len(a) - 300], "")[v - len(FLIPS)]


_c3_cache = {}


@pytest.fixture
def c3(R, eng, golden, request):
    """(alphabet, bits, mode, k) of the shape, sources a, destinations b, packed A / B, their scripts from script_batch"""
    name = request.param
    if name not in _c3_cache:
        alphabet, bits, mode, k = SHAPES[name]
        rng = np.random.default_rng(20261021 + list(SHAPES).index(name))
        a = rand_seqs(rng, 400, 1000, 2000, alphabet)
        b = [mutate(rng, s, list(alphabet))[:2000] if p % 10 else rand_seqs(rng, 1, 1000, 2000, alphabet)[0]
             for p, s in enumerate(a)]
        A, B = R.pack(a), R.pack(b)
        assert A.bits == B.bits == bits
        eng.set_costs(golden["default_costs"])
        scripts = eng.script_batch(A, B)
        assert eng.last_mode == mode
        if k is not None:
            assert eng.classify(A.symmask | B.symmask, A.max_len, B.max_len, force_mode=2) == (2, k)
        _c3_cache[name] = (SHAPES[name], a, b, A, B, scripts)
    return _c3_cache[name]


@gpu
@pytest.mark.parametrize("c3", list(SHAPES), indirect=True)
def test_c3_shapes_patch_every_variant(R, eng, sed, c3):
    """every pair patched with one of 13 inputs x, rotating: the source itself, tails across the 256-thread stride of
    the tail loop, a changed symbol in the first, second and last block, shorter inputs and the empty string"""
    (alphabet, bits, mode, k), a, b, A, B, scripts = c3
    rng = np.random.default_rng(7 + bits)
    xs = [x_variant(rng, s, p % N_VARIANTS, alphabet) for p, s in enumerate(a)]
    n_ops = scripts["n_ops"]
    assert (n_ops > BLOCK).all() and (n_ops > 4 * BLOCK).mean() > 0.9         # every script spans several blocks
    tails = np.array([len(x) - len(s) for x, s in zip(xs, a)])
    assert {257, 700} <= set(tails.tolist()) and (tails == 256).any()
    out, out_len, err = eng.patch_batch(scripts, A, B, R.pack(xs, bits=bits))
    assert {0, 1, -1} == set(err.tolist())
    check_patch(R, out, out_len, err, scripts, a, b, xs, sed, range(3 * N_VARIANTS))


@gpu
@pytest.mark.parametrize("c3", list(SHAPES), indirect=True)
def test_c3_shapes_roundtrip_bytes(R, eng, c3):
    """patch(script, A) is B byte for byte; the fused round-trip entry point returns the scripts of script_batch, also
    when called with oi = oj = NULL as the C3 benchmark does"""
    (alphabet, bits, mode, k), a, b, A, B, scripts = c3
    assert (scripts["n_ops"] > BLOCK).all()
    out, out_len, err = eng.patch_batch(scripts, A, B, A)
    assert not err.any()
    for p in range(len(a)):
        assert out_len[p] == len(b[p]) and R.decode(out[p, :out_len[p]]) == b[p], p
        assert not out[p, out_len[p]:].any(), p

    checked = eng.script_batch(A, B, check_roundtrip=True)
    assert eng.last_mode == mode and checked["ok"].all()
    assert np.array_equal(checked["n_ops"], scripts["n_ops"]) and np.array_equal(checked["dist"], scripts["dist"])
    for p in range(len(a)):
        for key in (0, 1, 2):                                   # op, oi, oj
            assert np.array_equal(rows(checked, p)[key], rows(scripts, p)[key]), (p, key)

    lib = R.load_library()
    n, max_ops = A.n, scripts["op"].shape[1]
    op = np.zeros((n, max_ops), np.uint8); n_ops = np.zeros(n, np.int32); dist = np.zeros(n, np.float64)
    ok = np.zeros(n, np.uint8); mode_out = C.c_int()
    p_ = R._lib.ptr
    R._lib.check(lib.rsd_script_patch_check_batch(
        eng.ctx, p_(A.words, _u32), p_(A.start, _i64), p_(A.len, _i32), A.words.shape[0],
        p_(B.words, _u32), p_(B.start, _i64), p_(B.len, _i32), B.words.shape[0],
        n, bits, A.symmask | B.symmask, 0, max_ops, p_(op, _u8), None, None, p_(n_ops, _i32), p_(dist, _f64), p_(ok, _u8),
        C.byref(mode_out)))
    assert mode_out.value == mode and ok.all()
    assert np.array_equal(n_ops, scripts["n_ops"]) and np.array_equal(dist, scripts["dist"])
    for p in range(n):
        assert np.array_equal(op[p, :n_ops[p]], rows(scripts, p)[0]), p


# ---------------------------------------------------------------------------------------------------------------------
# 3-4. empty sides, reversed scripts
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_empty_sides(R, eng, golden, sed):
    """m = 0 (all INS), n = 0 (all DEL) and both empty, short and over several blocks, each with x in
    {'', 'A', a, a + tail}"""
    rng = np.random.default_rng(31)
    a, b, xs = [], [], []
    for L in (1, 7, 300, 700):
        s, t = rand_seqs(rng, 2, L, L, "AGCU")
        for sa, sb in (("", t), (s, ""), ("", "")):
            for x in ("", "A", sa, sa + "".join(rng.choice(list("AGCU"), size=300))):
                a.append(sa); b.append(sb); xs.append(x)
    eng.set_costs(golden["default_costs"])
    A, B = R.pack(a, bits=2), R.pack(b, bits=2)
    scripts = eng.script_batch(A, B)
    for p in range(len(a)):
        op, oi, oj = rows(scripts, p)
        assert op.shape[0] == len(a[p]) + len(b[p]) and set(op.tolist()) <= ({0} if not a[p] else {1})
    assert (scripts["n_ops"] > BLOCK).any() and (scripts["n_ops"] == 0).any()
    out, out_len, err = eng.patch_batch(scripts, A, B, R.pack(xs, bits=2))
    assert {0, 1, -1} == set(err.tolist())
    check_patch(R, out, out_len, err, scripts, a, b, xs, sed, range(len(a)))


@gpu
def test_reversed_scripts(R, eng, golden, sed):
    """eswire.rev_packed turns B back into A: patch_batch(A=B, B=A, X=B) == A with code 0; with a tail and with a
    changed symbol == sed.patching(generate_rev_es(es), x); C3-sized pairs and short ones"""
    from rna_sequence_diff_patch_b200 import eswire
    rng = np.random.default_rng(32)
    a = rand_seqs(rng, 24, 1000, 2000, "AGCU") + rand_seqs(rng, 48, 1, 300, "AGCU")
    b = [mutate(rng, s, "AGCU")[:2000] if p % 6 else rand_seqs(rng, 1, 1, 2000, "AGCU")[0] for p, s in enumerate(a)]
    eng.set_costs(golden["default_costs"])
    A, B = R.pack(a, bits=2), R.pack(b, bits=2)
    fwd = eng.script_batch(A, B)
    n, max_ops = len(a), fwd["op"].shape[1]
    rev = dict(op=np.zeros((n, max_ops), np.uint8), oi=np.zeros((n, max_ops), np.int32),
               oj=np.zeros((n, max_ops), np.int32), n_ops=fwd["n_ops"].copy())
    for p in range(n):
        k = int(fwd["n_ops"][p])
        rev["op"][p, :k], rev["oi"][p, :k], rev["oj"][p, :k] = eswire.rev_packed(*rows(fwd, p))
    assert (fwd["n_ops"][:24] > 4 * BLOCK).all() and (rev["op"] == 0).any() and (rev["op"] == 1).any()

    out, out_len, err = eng.patch_batch(rev, B, A, B)
    assert not err.any()
    for p in range(n):
        assert R.decode(out[p, :out_len[p]]) == a[p], p

    xs = [s + "".join(rng.choice(list("AGCU"), size=300)) if p % 2 else s[:-1] + ("G" if s[-1] != "G" else "A")
          for p, s in enumerate(b)]
    out, out_len, err = eng.patch_batch(rev, B, A, R.pack(xs, bits=2))
    assert (err == 1).all()
    check_patch(R, out, out_len, err, rev, b, a, xs)
    for p in range(n):
        es = sed.es_from_packed(*rows(fwd, p), a[p], b[p])
        assert sed.patching(sed.generate_rev_es(es), xs[p]) == (1, R.decode(out[p, :out_len[p]])), p


# ---------------------------------------------------------------------------------------------------------------------
# 5. the reference's hand-edited scripts
# ---------------------------------------------------------------------------------------------------------------------
def sides_of(es):
    """(A, B) of a script: the source characters of its non-inserts, the destination characters of its non-deletes"""
    return ("".join(e["source"]["character"] for e in es if e["operation"] != "insert"),
            "".join(e["destination"]["character"] for e in es if e["operation"] != "delete"))


def is_path(es):
    """plain restatement of the path rule: the source index of every delete / update and the destination index of
    every insert / update is the cell the path enters minus one (the indices sed.patching reads)"""
    ci = cj = 0
    for e in es:
        o = e["operation"]
        ci += o != "insert"
        cj += o != "delete"
        if o != "insert" and e["source"]["index"] != ci - 1:
            return False
        if o != "delete" and e["destination"]["index"] != cj - 1:
            return False
    return (ci, cj) == tuple(map(len, sides_of(es)))


@gpu
def test_reference_hand_edited_scripts(R, eng):
    """golden['patch_odd'] (make_golden.py): the reference's scripts, a third of them reversed, patched onto inputs with
    tails, changed and missing symbols; case t was shuffled when t % 11 == 5.  Paths, in one batch, give the recorded
    output; every other script is refused with RSD_EINVAL"""
    import json
    import os
    from rna_sequence_diff_patch_b200 import eswire
    with open(os.path.join(os.path.dirname(__file__), "golden", "ref_golden.json")) as f:
        cases = json.load(f)["patch_odd"]
    assert len(cases) == 120
    path = [is_path(c["es"]) for c in cases]
    assert all(ok for t, ok in enumerate(path) if t % 11 != 5)
    assert not all(ok for t, ok in enumerate(path) if t % 11 == 5)

    def batch(cs):
        packed = [eswire.es_to_packed(c["es"]) for c in cs]
        max_ops = max(len(c["es"]) for c in cs)
        s = dict(op=np.zeros((len(cs), max_ops), np.uint8), oi=np.zeros((len(cs), max_ops), np.int32),
                 oj=np.zeros((len(cs), max_ops), np.int32), n_ops=np.array([len(c["es"]) for c in cs], np.int32))
        for p, (op, oi, oj) in enumerate(packed):
            k = op.shape[0]
            s["op"][p, :k], s["oi"][p, :k], s["oj"][p, :k] = op, oi, oj
        ab = [sides_of(c["es"]) for c in cs]
        return s, R.pack([x for x, _ in ab], bits=4), R.pack([y for _, y in ab], bits=4), R.pack([c["x"] for c in cs], bits=4)

    good = [c for c, ok in zip(cases, path) if ok]
    out, out_len, err = eng.patch_batch(*batch(good))
    for p, c in enumerate(good):
        assert [int(err[p]), R.decode(out[p, :out_len[p]])] == c["out"], p
    for c in (c for c, ok in zip(cases, path) if not ok):
        with pytest.raises(R.RsdError) as ei:
            eng.patch_batch(*batch([c]))
        assert ei.value.code == EINVAL and "pair 0 op" in str(ei.value)


# ---------------------------------------------------------------------------------------------------------------------
# 6. long pairs
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_long_pair_scripts(R, eng, golden, sed):
    """six pairs of 4-9 kb: script_batch routes them to rsd_long_pairs; their scripts patch A and A + 300 symbols like
    the oracle; the round-trip entry point (never routed: the tape kernel) returns the same scripts, all ok"""
    rng = np.random.default_rng(36)
    a = rand_seqs(rng, 6, 4500, 9000, "AGCU")
    b = [mutate(rng, s, "AGCU") if p != 4 else rand_seqs(rng, 1, 4200, 9000, "AGCU")[0] for p, s in enumerate(a)]
    assert min(map(len, a + b)) >= 4096
    eng.set_costs(golden["default_costs"])
    A, B = R.pack(a), R.pack(b)
    launches0 = eng.launch_count()
    scripts = eng.script_batch(A, B)
    assert eng.launch_count() - launches0 <= 4                  # one forward launch, traceback, emit
    checked = eng.script_batch(A, B, check_roundtrip=True)
    assert checked["ok"].all()
    assert np.array_equal(checked["n_ops"], scripts["n_ops"]) and np.array_equal(checked["dist"], scripts["dist"])
    for p in range(len(a)):
        for key in (0, 1, 2):
            assert np.array_equal(rows(checked, p)[key], rows(scripts, p)[key]), (p, key)
    for xs in (a, [s + "".join(rng.choice(list("AGCU"), size=300)) for s in a]):
        out, out_len, err = eng.patch_batch(scripts, A, B, R.pack(xs, bits=2))
        check_patch(R, out, out_len, err, scripts, a, b, xs, sed, (0, 4))
        assert (err == (0 if xs is a else 1)).all()


# ---------------------------------------------------------------------------------------------------------------------
# 7. refusals, with or without a device
# ---------------------------------------------------------------------------------------------------------------------
SUBJECT_OPS = [2, 1, 2, 0, 0, 2, 2, 1, 2, 0, 2, 2, 0, 2, 1, 2]          # UPD, DEL and INS; 12 source / 13 destination symbols


def test_patch_refuses_scripts_that_are_not_paths(R):
    """Each script that is not a path of its pair is refused with RSD_EINVAL before the device is touched, naming the
    pair and the op; a path with oi = oj = NULL gets past the check (RSD_ENODEV without a device, RSD_OK with one).

    Were the check to regress, these calls would reach k_finalize, so every refused script stays inside the buffers:
    it is off by exactly one op or index from a path; it is pair 0 of three, never the last pair; max_out leaves 8
    symbols of slack, so an extra insert lands inside the pair's own slot; and the pair's lengths (12 and 13) are not
    multiples of the 16 / 8 symbols of a 2- / 4-bit word, so a read one symbol past either sequence stays inside the
    sequence's last packed word."""
    lib = R.load_library()
    on_gpu = lib.rsd_device_count() > 0
    rng = np.random.default_rng(37)
    ops = np.array(SUBJECT_OPS, np.uint8)
    m, n = int((ops != 0).sum()), int((ops != 1).sum())
    assert (m, n) == (12, 13)
    a = ["".join(rng.choice(list("AGCU"), size=L)) for L in (m, 9, 5)]
    b = ["".join(rng.choice(list("AGCU"), size=L)) for L in (n, 9, 6)]
    A, B = R.pack(a, bits=2), R.pack(b, bits=2)
    fill = [np.array([2] * 9, np.uint8), np.array([2] * 5 + [0], np.uint8)]       # the other two pairs: paths
    max_ops = len(ops) + 2

    def script(subject):
        op = np.zeros((3, max_ops), np.uint8); oi = np.zeros((3, max_ops), np.int32); oj = np.zeros((3, max_ops), np.int32)
        for p, o in enumerate([subject] + fill):
            op[p, :len(o)] = o
            oi[p, :len(o)] = np.cumsum(o != 0); oj[p, :len(o)] = np.cumsum(o != 1)
        n_ops = np.array([len(subject)] + [len(o) for o in fill], np.int32)
        return op, oi, oj, n_ops

    cases = {                    # name -> (op row, None or (index array, op, change)); oi / oj are passed with the latter
        "one INS too many": (np.append(ops, 0), None),
        "one DEL too many": (np.append(ops, 1), None),
        "one INS too few": (np.delete(ops, np.flatnonzero(ops == 0)[-1]), None),
        "op code 3": (np.where(np.arange(len(ops)) == 5, 3, ops).astype(np.uint8), None),
        "wrong oi on a DEL": (ops, ("oi", 7, +1)),
        "wrong oj on an UPD": (ops, ("oj", 8, -1)),
    }
    assert ops[7] == 1 and ops[8] == 2 and ops[5] == 2
    ctx = C.c_void_p()
    assert lib.rsd_create(0, C.byref(ctx)) == 0
    try:
        max_out = max(len(x) for x in a) + max(len(y) for y in b) + 8
        for name, (subject, wrong) in cases.items():
            op, oi, oj, n_ops = script(subject)
            if wrong:
                key, t, d = wrong
                dict(oi=oi, oj=oj)[key][0, t] += d
            rc, *_ = raw_patch(R, ctx, op, oi if wrong else None, oj if wrong else None, n_ops, A, B, A, max_out)
            msg = lib.rsd_last_error().decode()
            assert rc == EINVAL and "pair 0 " in msg and ("op" in msg), (name, rc, msg)
        op, oi, oj, n_ops = script(ops)
        rc, out, out_len, err = raw_patch(R, ctx, op, None, None, n_ops, A, B, A, max_out)
        assert rc == (OK if on_gpu else ENODEV), lib.rsd_last_error().decode()
        if on_gpu:
            assert not err.any() and all(R.decode(out[p, :out_len[p]]) == b[p] for p in range(3))
        # the same refusal through Engine.patch_batch
        op, oi, oj, n_ops = script(ops)
        oj[0, 8] += 1
        with pytest.raises(R.RsdError) as ei:
            R.Engine(0).patch_batch(dict(op=op, oi=oi, oj=oj, n_ops=n_ops), A, B, A)
        assert ei.value.code == EINVAL and "pair 0 op 8 (UPD)" in str(ei.value)
    finally:
        lib.rsd_destroy(ctx)
