"""Long pairs in one call (rsd_long_pairs): wall / device time of K 50 kb pairs for ring counts and panel widths."""
import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as G; G.build()
import rna_sequence_diff_patch_b200 as R
from rna_sequence_diff_patch_b200 import cost_tables
from _synth import c4_pair
import torch
L = int(os.environ.get("L", 50000))
pairs = [c4_pair(seed=20260004 + k, m=L) for k in range(int(os.environ.get("NPAIRS", 16)))]
eng = R.Engine(0); eng.set_costs(cost_tables.default_costs()); eng.set_timing(True)
single = eng.long_pair(*pairs[0])
# (pairs, rings, columns per lane); 0 = the library's own choice
configs = [(1, 0, 0), (1, 1, 4), (1, 1, 8), (1, 1, 16), (2, 0, 0), (2, 2, 8), (2, 2, 16), (4, 0, 0), (4, 4, 8), (4, 4, 16), (8, 0, 0), (8, 8, 8), (8, 8, 16),
           (12, 0, 0), (12, 12, 8), (12, 12, 16), (16, 0, 0), (16, 16, 8), (16, 16, 16)]
if os.environ.get("CONFIGS"):
    configs = [tuple(int(x) for x in c.split(":")) for c in os.environ["CONFIGS"].split(",")]
for K, rings, C in configs:
    for name, v in (("RSD_LONG_RINGS", rings), ("RSD_LONG_C", C)):
        if v: os.environ[name] = str(v)
        else: os.environ.pop(name, None)
    cells = sum(float(a.shape[0]) * b.shape[0] for a, b in pairs[:K])
    for want in (False, True):
        best = 1e9; fwd = 0
        for rep in range(3):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            res = eng.long_pairs(pairs[:K], want_script=want)
            dt = time.perf_counter() - t0
            if dt < best: best, fwd, dev = dt, eng.long_forward_ms(), eng.last_kernel_ms()
        ok = all(r["dist"] == single["dist"] for r in res[:1]) and (not want or np.array_equal(res[0]["op"], single["op"]))
        print(f"K={K} rings={rings} C={C} script={want}: wall {best * 1e3:.2f} ms, device {dev:.2f} ms, forward {fwd:.2f} ms = {cells / fwd * 1e-6:.0f} GCUPS fwd, "
              f"{cells / dev * 1e-6:.0f} GCUPS device; pair0 ok={ok}", flush=True)
