"""Cost tables and restated bounds for the mode-edge tests (tests/test_gpu_mode_edges.py, tests/test_abi.py).

Each narrow kernel is exact only while every value it holds fits its type; the host classifier (rsd_ctx::classify,
script_pipeline, rsd_long_pairs) picks it from thresholds on the costs and lengths.  The tables here sit on those
thresholds, and the formulas restate the two bounds that rsd_classify does not expose."""
import itertools
import math

SYM = "AGCUYRWSKMDVHBN"

# the 12 off-diagonal A/G/C/U substitutions of the v-edge tables (row-major, diagonal skipped): with ins + del = 127
# they give v = max(0, ins + del - sub) = 127, 126, 125, 114, 87, 63, 37, 1, 0, 0, 0, 0 and |w| <= 127
SUBS_V = [0, 1, 2, 13, 40, 64, 90, 126, 127, 128, 200, 254]


def table(ins, dele, acgu_subs=None, other=1.0):
    """{'insert','delete','update'}: `other` for every substitution, then the A/G/C/U block from acgu_subs."""
    upd = {a: {b: (0.0 if a == b else float(other)) for b in SYM} for a in SYM}
    if acgu_subs is not None:
        it = iter(acgu_subs)
        for a in "AGCU":
            for b in "AGCU":
                if a != b:
                    upd[a][b] = float(next(it))
    return {"insert": float(ins), "delete": float(dele), "update": upd}


def uniform(c):
    """insert, delete and every substitution cost c."""
    return table(c, c, other=c)


def v_table(k=0, ins_del=(64, 63)):
    """int16x2 byte-table edge: ins + del = 127 (v = 127 fits the sign-extended byte), 128 does not.  k = 2 gives the
    same scaled table in quarter units (15.75 / 16 -> 63 / 64)."""
    s = 2.0 ** -k
    return table(ins_del[0] * s, ins_del[1] * s, [x * s for x in SUBS_V])


# the unit tables of the k (scale) edge: k = 16 when every cost is a multiple of 2^-16 and one of them is odd
K16_SMALL = table(31 / 65536, 33 / 65536, [(2 * i + 1) / 65536 for i in range(12)])          # int16x2, k = 16
K16_WIDE = table(1 + 2.0 ** -16, 1.0, [(2 * i + 1) / 65536 for i in range(12)])             # int32, k = 16
K17 = table(1 + 2.0 ** -16, 1.0, [2.0 ** -17] + [(2 * i + 1) / 65536 for i in range(11)])   # k would be 17: fp64
DEAR_IN = table(1.0, 1.0, [2.0 ** 30 - 1] * 12)        # largest scaled cost an int32 table holds
DEAR_OUT = table(1.0, 1.0, [2.0 ** 30] * 12)           # one more: fp64


def codes_of(symbols):
    return [SYM.index(ch) for ch in symbols]


def scaled_costs(costs, symbols, k):
    """(ins, del, {(a, b): sub}) scaled by 2^k, over the substitutions between the given symbols."""
    s = 2.0 ** k
    subs = {(a, b): costs["update"][a][b] * s for a in symbols for b in symbols if a != b}
    return costs["insert"] * s, costs["delete"] * s, subs


def ceil_log2(v):
    return max(0, math.ceil(math.log2(v)))


def script_key_bound(costs, symbols, k, max_m, max_n):
    """script_pipeline (rsd_api.cu): int32 (cost, steps) keys, key = cost << S | steps, are used while this bound is
    below 1073741000; -> (bound, S)."""
    ins, dele, subs = scaled_costs(costs, symbols, k)
    maxabsw = max([ins + dele] + [abs(v - ins - dele) for v in subs.values()])
    S = ceil_log2(max_m + max_n + 66)
    return (max_m * dele + (max_n + 64) * ins + maxabsw + 2.0) * 2.0 ** S + (max_m + max_n + 66), S


SCRIPT_KEY_LIMIT = 1073741000.0


def long_key32_ok(costs, symbols, k, m, n):
    """rsd_long_pairs (rsd_long.inl): a pair runs on the 32-bit modular keys of k_long2 when 32 rows of drift,
    (64 maxc + 128) << S, stay below 2^30; maxc = the largest |scaled cost| among ins, del and w = sub - ins - del."""
    ins, dele, subs = scaled_costs(costs, symbols, k)
    maxc = max([ins, dele, ins + dele] + [abs(v - ins - dele) for v in subs.values()])
    S = ceil_log2(m + n + 66)
    return S <= 24 and (int(64 * maxc + 128) << S) < (1 << 30)


def border_sums_differ(c, upto):
    """the lengths i <= upto at which i * c (how the fp64 kernels and the reference fill the borders) differs from
    c added i times"""
    return [i for i, s in enumerate(itertools.accumulate([c] * upto), start=1) if s != i * c]


def last_inside(inside, lo, hi):
    """the largest x in [lo, hi) with inside(x), for inside(lo) true and inside(hi) false (a monotone predicate)"""
    assert inside(lo) and not inside(hi), (lo, hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if inside(mid):
            lo = mid
        else:
            hi = mid
    return lo
