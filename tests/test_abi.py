"""The C-ABI library loads and exports exactly what include/rsd.h declares (CPU only: no compute)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as G
    G.build()
    import rna_sequence_diff_patch_b200 as R
    return R


def header_functions():
    txt = open(os.path.join(ROOT, "include", "rsd.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(rsd_[a-z0-9_]+)\s*\(", txt)))


def test_header_and_library_agree(built):
    from rna_sequence_diff_patch_b200 import _lib
    names = header_functions()
    assert len(names) >= 25
    lib = ctypes.CDLL(built.library_path())
    for n in names:
        assert hasattr(lib, n), f"{n} declared in rsd.h but not exported by librsd.so"
    assert sorted(_lib.SIGNATURES) == names, "ctypes SIGNATURES and rsd.h differ"


def test_loads_without_gpu_and_fails_loudly(built):
    import json
    lib = built.load_library()
    assert lib.rsd_abi_version() == 1
    if lib.rsd_device_count() == 0:
        eng = built.Engine(0)
        eng.set_costs(__import__('rna_sequence_diff_patch_b200.cost_tables', fromlist=['x']).default_costs())
        p = built.pack(["ACGU", "GGA"])
        with pytest.raises(built.RsdError) as ei:
            eng.distance_batch(p, p)
        assert ei.value.code == 2 and "no CPU fallback" in str(ei.value)


def test_pack_roundtrip_and_symmask(built):
    import numpy as np
    from rna_sequence_diff_patch_b200.encoding import unpack, concat
    seqs = ["ACGU", "", "GGAUUUCAGGAUUUCAGGAUUUCAG", "N", "AGCUYRWSKMDVHBN" * 3]
    for bits in (4,):
        p = built.pack(seqs, bits=bits)
        codes, off = unpack(p)
        c2, o2 = concat(seqs)
        assert np.array_equal(codes, c2) and np.array_equal(off, o2)
        assert p.symmask == 0x7FFF
    p2 = built.pack(["ACGU", "UUGA"])
    assert p2.bits == 2 and p2.symmask == 0xF
    with pytest.raises(KeyError):
        built.pack(["ACGT"])
    with pytest.raises(built.RsdError):
        built.pack(["ACGN"], bits=2)


def test_classifier_modes(built, default_costs, user_costs):
    eng = built.Engine(0)
    eng.set_costs(default_costs)
    assert eng.classify(0xF, 300, 300) == (1, 0)            # ACGU, all costs 1 -> int16x2
    assert eng.classify(0x7FFF, 300, 300)[0] == 3           # 0.66 / 0.83 present -> fp64
    assert eng.classify(0x400F, 31, 31) == (2, 2)           # ACGU+N: 0.75 -> x4, int32
    assert eng.classify(0xF, 50000, 50000)[0] == 2          # too long for int16
    eng.set_costs(user_costs)
    assert eng.classify(0xF, 300, 300) == (1, 0)
    with pytest.raises(built.RsdError):
        eng.classify(0x7FFF, 10, 10, force_mode=2)          # int forced on non-dyadic costs
    bad = {"insert": -1.0, "delete": 1.0, "update": default_costs["update"]}
    with pytest.raises(built.RsdError) as ei:
        eng.set_costs(bad)
    assert ei.value.code == 5


def test_classifier_edges(built, default_costs, user_costs):
    """The documented edges of the narrow kernels, last shape inside and first shape outside: a bound that tightens
    sends exact work to a slower kernel, which no parity test notices.  (mode, k): 1 int16x2, 2 int32, 3 fp64."""
    import _edges as E
    eng = built.Engine(0)
    cases = [
        (E.v_table(), 0xF, [((478, 478), (1, 0)), ((479, 479), (2, 0))]),            # v = 127 fits the byte table
        (E.v_table(ins_del=(64, 64)), 0xF, [((10, 10), (2, 0))]),                     # v = 128 does not
        (E.v_table(k=2), 0xF, [((478, 478), (1, 2)), ((479, 479), (2, 2))]),          # the same after a x4 scale
        (E.v_table(k=2, ins_del=(64, 64)), 0xF, [((10, 10), (2, 2))]),
        (default_costs, 0xF, [((32466, 32466), (1, 0)), ((32467, 32467), (2, 0))]),   # N < 65000
        (user_costs, 0xF, [((12960, 12960), (1, 0)), ((12961, 12961), (2, 0))]),
        # asymmetric: the first is bounded by the swapped orientation, the second by the stored one
        (E.table(27, 100, E.SUBS_V), 0xF, [((40, 2017), (1, 0)), ((40, 2018), (2, 0))]),
        (E.table(100, 27, E.SUBS_V), 0xF, [((200, 530), (1, 0)), ((200, 531), (2, 0))]),
        (E.uniform(2.0 ** 20), 0xF, [((990, 990), (2, 0)), ((991, 991), (3, 0))]),    # |H'| < 2147483000
        (E.uniform(2.0 ** 20), 0x7FFF, [((990, 990), (2, 0)), ((991, 991), (3, 0))]),
        (E.K16_SMALL, 0xF, [((300, 300), (1, 16))]),
        (E.K16_WIDE, 0xF, [((300, 300), (2, 16))]),
        (E.K17, 0xF, [((300, 300), (3, 0))]),
        (E.DEAR_IN, 0xF, [((300, 300), (2, 0))]),                                      # scaled costs < 2^30
        (E.DEAR_OUT, 0xF, [((300, 300), (3, 0))]),
    ]
    for costs, symmask, shapes in cases:
        eng.set_costs(costs)
        for (m, n), want in shapes:
            assert eng.classify(symmask, m, n) == want, (costs["insert"], costs["delete"], symmask, m, n)


def test_topk_merge_host(built):
    import numpy as np
    eng = built.Engine(0)
    idx = np.array([[[0, 3, 5]], [[10, 11, -1]]], dtype=np.int64)          # 2 shards, 1 query, k=3
    sc = np.array([[[0.9, 0.5, 0.5]], [[0.9, 0.5, 0.0]]], dtype=np.float64)
    oi, os_ = eng.topk_merge(idx, sc)
    assert oi.tolist() == [[0, 10, 3]] and os_.tolist() == [[0.9, 0.9, 0.5]]
