#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 weighted Wagner–Fischer engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2-iupac]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY 8d "C2"): 1,000,000 synthetic RNA pairs per GPU, lengths
iid uniform in [100,300], alphabet ACGU iid uniform, costs = the shipped user_costs.json, distance
only.  One step = one pass of the hot path (rsd_distance_batch) over the whole batch.
Metric: GCUPS = 1e-9 * sum(m*n) / seconds (interior cells only).

  value     inputs resident in HBM (rsd_distance_batch_dev on torch's current stream), CUDA events
  e2e       the same through the host C-ABI call rsd_distance_batch with pinned HOST buffers:
            H2D of the packed batch and D2H of the distances inside the timed region
  roofline  dominant kernel (k_dist_twin16) timed with CUDA events on its own stream inside the
            library; bound = INT32 ALU issue rate (SURVEY 8d: 5 integer ops per cell), peak measured
            in this run with rsd_ubench (IADD3 issue rate); a secondary HBM figure is added
  cpu_baseline  the C oracle port (oracle/wf_oracle.c, pthreads over all host cores) on a bounded
            sample of the same pairs

Multi-GPU (torchrun, one rank per GPU): pairs are independent, every rank runs its own batch of
the same shape (weak scaling), no data-path collective; value = all ranks' cells / max-over-ranks time.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEEDS = {"c2": 20260002, "c2-iupac": 20260002}
L2_FLUSH_BYTES = 512 << 20
DUMP_BYTES = 60 << 20              # data written by --dump-outputs: with its .npy header, under 64 * 10^6 bytes
DUMP_SEED = 20260099


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(directory, distances):
    """Write what the timed path returned in its last step, the float64 distance of every pair, to
    DIR/distances.npy, so that two builds run with the same arguments can be compared output for output.  A batch
    larger than DUMP_BYTES is cut to a fixed, seeded sample of its pairs (kept in pair order)."""
    n_max = DUMP_BYTES // distances.itemsize
    if distances.shape[0] > n_max:
        keep = np.sort(np.random.default_rng(DUMP_SEED).choice(distances.shape[0], n_max, replace=False))
        distances = distances[keep]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "distances.npy"), np.ascontiguousarray(distances, dtype=np.float64))


def gen_pairs(n_pairs: int, seed: int, alphabet_size: int):
    """(codes_a, off_a, codes_b, off_b) uint8 codes 0..alphabet_size-1 (table order AGCU...)."""
    rng = np.random.default_rng(seed)
    la = rng.integers(100, 301, size=n_pairs, dtype=np.int64)
    lb = rng.integers(100, 301, size=n_pairs, dtype=np.int64)
    oa = np.zeros(n_pairs + 1, np.int64); ob = np.zeros(n_pairs + 1, np.int64)
    np.cumsum(la, out=oa[1:]); np.cumsum(lb, out=ob[1:])
    ca = rng.integers(0, alphabet_size, size=int(oa[-1]), dtype=np.uint8)
    cb = rng.integers(0, alphabet_size, size=int(ob[-1]), dtype=np.uint8)
    return ca, oa, cb, ob


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe; NVML in-process, nvidia-smi as fallback)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.via = "nvidia-smi"

    def _nvml(self):
        """The same NVML fields nvidia-smi prints, read in-process: a 35 ms timed region gets dozens of samples
        instead of the one a 50 ms nvidia-smi call can deliver."""
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        bits = [pynvml.nvmlClocksEventReasonHwSlowdown if hasattr(pynvml, "nvmlClocksEventReasonHwSlowdown") else pynvml.nvmlClocksThrottleReasonHwSlowdown,
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown, pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                pynvml.nvmlClocksThrottleReasonSwPowerCap]
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        self.via = "nvml (in-process, 2 ms period)"
        while not self.stop_flag.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.samples.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b in bits])
            self.stop_flag.wait(0.002)

    def run(self):
        try:
            self._nvml()
            return
        except Exception:  # noqa: BLE001  (no pynvml / NVML error: fall back to the nvidia-smi recipe)
            pass
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if len(s) >= 6 and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 6 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for s in self.samples if len(s) >= 6 for k in range(4) if s[2 + k] == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "via": self.via}


def cpu_baseline(ca, oa, cb, ob, costs, target_s=12.0, nthreads=0):
    """C oracle port on a bounded prefix of the same pairs; -> (gcups, cores, description, seconds)."""
    from oracle import oracle as O
    O.build()
    cores = nthreads or O.num_threads()

    def run(n):
        a = ca[: oa[n]]; b = cb[: ob[n]]
        t0 = time.perf_counter()
        O.distance_batch(a, oa[: n + 1].copy(), b, ob[: n + 1].copy(), costs, nthreads=cores)
        dt = time.perf_counter() - t0
        cells = float(((oa[1: n + 1] - oa[:n]) * (ob[1: n + 1] - ob[:n])).sum())
        return cells, dt

    n_total = len(oa) - 1
    n0 = min(2000, n_total)
    cells, dt = run(n0)
    n = int(min(n_total, max(n0, n0 * target_s / max(dt, 1e-6))))
    cells, dt = run(n)
    return cells / dt * 1e-9, cores, f"first {n} pairs of the workload, C oracle port, {cores} threads", dt


def _pyref_init(ref_dir):
    """Pool initialiser: import the unmodified reference once per worker (it reads its cost files from the CWD and
    prints a self-test at import, SED:6-18,463-471)."""
    import contextlib
    import io
    os.chdir(ref_dir)
    sys.path.insert(0, ref_dir)
    with contextlib.redirect_stdout(io.StringIO()):
        import StringEditDistance  # noqa: F401


def _pyref_pair(args):
    import StringEditDistance as S
    a, b = args
    dp = S.wagnerFisher(a, b, True)
    return float(dp[len(dp) - 1][len(dp[0]) - 1].value)


def python_reference_baseline(ca, oa, cb, ob, n_pairs=768, want=None):
    """The reference's own pure-Python wagnerFisher (baseline/_ref/StringEditDistance.py, unmodified) on the first
    n_pairs pairs of the workload, one spawn-pool worker per host core; -> dict for the JSON line."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "StringEditDistance.py")):
        return {"unavailable": "baseline/_ref/StringEditDistance.py is absent (run `python __graft_entry__.py build` where /root/reference exists)"}
    import multiprocessing as mp
    sym = np.frombuffer(b"AGCUYRWSKMDVHBN", dtype=np.uint8)
    pairs = [(sym[ca[oa[p]:oa[p + 1]]].tobytes().decode(), sym[cb[ob[p]:ob[p + 1]]].tobytes().decode()) for p in range(n_pairs)]
    cores = os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores, initializer=_pyref_init, initargs=(ref_dir,)) as pool:
        pool.map(_pyref_pair, pairs[:cores])                      # warm: every worker has imported the module
        t0 = time.perf_counter()
        got = pool.map(_pyref_pair, pairs, chunksize=1)
        dt = time.perf_counter() - t0
    cells = float(((oa[1: n_pairs + 1] - oa[:n_pairs]) * (ob[1: n_pairs + 1] - ob[:n_pairs])).sum())
    res = {"value": cells / dt * 1e-9, "unit": "GCUPS", "cores": cores, "kind": "reference",
           "sample": f"first {n_pairs} pairs of the workload through the unmodified StringEditDistance.wagnerFisher "
                     f"(pure Python, spawn pool of {cores} workers, {dt:.1f} s)"}
    if want is not None:
        res["matches_gpu"] = bool(np.array_equal(np.array(got), want[:n_pairs]))
    return res


def _claim_stdout():
    """Keep stdout for the single JSON line: libraries (NCCL prints its version banner there) get stderr."""
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def bind_near_gpu(index):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs next to its GPU, as NVML reports
    them — with 8 ranks the host->device copies otherwise cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        import torch
        pr = torch.cuda.get_device_properties(index)
        try:
            h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0".encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception as e:  # noqa: BLE001
        log(f"[bench] no CPU affinity for GPU {index}: {e}")
        return None


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c2-iupac"])
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the C3/C4/C5 side measurements")
    ap.add_argument("--c5-records", type=int, default=10_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the distances of the last device-resident step to DIR/distances.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    costs = __import__('rna_sequence_diff_patch_b200.cost_tables', fromlist=['x']).user_costs()
    alpha = 4 if args.workload == "c2" else 15
    config = {"workload": f"C2: {args.pairs} pairs/GPU, len U[100,300], "
                          f"{'ACGU (2-bit)' if alpha == 4 else '15-letter IUPAC (4-bit)'}, user_costs.json, distance only",
              "pairs_per_gpu": args.pairs, "seed": SEEDS[args.workload],
              "l2": f"flushed between timed steps by writing a {L2_FLUSH_BYTES >> 20} MiB buffer",
              "parallelism": f"pairs sharded over {world} rank(s), no collective"}

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        ca, oa, cb, ob = gen_pairs(args.pairs, SEEDS[args.workload] + 0, alpha)
        vals = []
        for s in range(args.warmup + args.steps):
            g, cores, desc, dt = cpu_baseline(ca, oa, cb, ob, costs, target_s=max(2.0, 60.0 / max(1, args.steps + args.warmup)))
            if s >= args.warmup:
                vals.append((g, dt))
        v = float(np.mean([g for g, _ in vals])) if vals else 0.0
        ms = float(np.mean([dt for _, dt in vals]) * 1e3) if vals else 0.0
        print(file=out, flush=True, *[json.dumps({
            "impl": "reference", "metric": "GCUPS", "value": v, "unit": "GCUPS", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "GCUPS", "cores": cores, "kind": "port", "sample": desc,
                             "note": "the reference is pure Python and cannot travel to the GPU box; this is the C "
                                     "restatement of its algorithm (oracle/wf_oracle.c), pinned to it by tests/golden"},
            "cpu_baseline_python": python_reference_baseline(ca, oa, cb, ob),
            "e2e": {"value": v, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0})])
        return

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist
    import __graft_entry__ as G
    G.build()
    import rna_sequence_diff_patch_b200 as R

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_near_gpu(local_rank) if world > 1 else None      # pinned buffers are first-touched after this
    if numa:
        config["host"] = f"each rank runs on the {numa} CPUs NVML lists next to its GPU (pinned buffers first-touched there)"

    ca, oa, cb, ob = gen_pairs(args.pairs, SEEDS[args.workload] + rank, alpha)
    cells = float(((oa[1:] - oa[:-1]) * (ob[1:] - ob[:-1])).sum())
    t0 = time.perf_counter()
    A = R.pack((ca, oa)); B = R.pack((cb, ob))
    log(f"[rank {rank}] packed {args.pairs} pairs ({A.bits}-bit) in {time.perf_counter() - t0:.2f}s; cells/step={cells:.3e}")
    eng = R.Engine(local_rank)
    eng.set_costs(costs)
    eng.set_timing(True)
    symmask = A.symmask | B.symmask
    max_m, max_n = A.max_len, B.max_len

    # pinned host copies (the e2e path reads these) and device-resident copies (the `value` path)
    def pin(x):
        t = torch.from_numpy(x).pin_memory()
        return t
    hp = {k: pin(v) for k, v in dict(aw=A.words, as_=A.start, al=A.len, bw=B.words, bs=B.start, bl=B.len).items()}
    dp = {k: v.to(dev, non_blocking=True) for k, v in hp.items()}
    out_dev = torch.zeros(args.pairs, dtype=torch.float64, device=dev)
    out_host = torch.zeros(args.pairs, dtype=torch.float64).pin_memory()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def step_dev():
        eng.distance_batch_dev(dp["aw"].data_ptr(), dp["as_"].data_ptr(), dp["al"].data_ptr(),
                               dp["bw"].data_ptr(), dp["bs"].data_ptr(), dp["bl"].data_ptr(),
                               args.pairs, max_m, max_n, A.bits, symmask, out_dev.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)

    import ctypes as C
    from rna_sequence_diff_patch_b200 import _lib
    lib = R.load_library()

    def cptr(t, typ):
        return C.cast(t.data_ptr(), C.POINTER(typ))

    def step_e2e():
        # packed words + lengths from pinned host memory; the batch has rsd_pack's layout, so start[] stays on the
        # host (NULL) and is rebuilt on the device from the lengths
        mode = C.c_int()
        _lib.check(lib.rsd_distance_batch(
            eng.ctx, cptr(hp["aw"], C.c_uint32), None, cptr(hp["al"], C.c_int32), A.words.shape[0],
            cptr(hp["bw"], C.c_uint32), None, cptr(hp["bl"], C.c_int32), B.words.shape[0],
            args.pairs, max_m, max_n, A.bits, symmask, 0, cptr(out_host, C.c_double), C.byref(mode)))

    hc = {"ca": pin(ca), "cb": pin(cb)}                    # raw symbol codes, 1 byte per symbol (what the CPU arm consumes)
    out_codes = torch.zeros(args.pairs, dtype=torch.float64).pin_memory()

    def step_codes():
        mode = C.c_int()
        _lib.check(lib.rsd_distance_batch_codes(
            eng.ctx, cptr(hc["ca"], C.c_uint8), cptr(hp["al"], C.c_int32), cptr(hc["cb"], C.c_uint8), cptr(hp["bl"], C.c_int32),
            args.pairs, max_m, max_n, A.bits, symmask, 0, cptr(out_codes, C.c_double), C.byref(mode)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------
    for _ in range(args.warmup):
        step_dev()
    torch.cuda.synchronize()
    launches0 = eng.launch_count()
    sampler = ClockSampler(local_rank); sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    barrier()
    for s in range(args.steps):
        flush.fill_(s & 0xFF)                       # L2 flush, outside the events
        ev[s][0].record()
        step_dev()
        ev[s][1].record()
        ev[s][1].synchronize()
        kernel_ms.append(eng.last_kernel_ms())
    barrier()
    launches_per_step = (eng.launch_count() - launches0) / max(1, args.steps)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = float(sum(step_ms))
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        c = torch.tensor([cells], dtype=torch.float64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        cells_all = float(c.item())
    else:
        cells_all = cells
    value = cells_all * args.steps / (total_ms * 1e-3) * 1e-9
    mode_used = eng.last_mode
    check_dev = out_dev.cpu().numpy()

    # ---- end to end through the host C-ABI call ---------------------------------------------------
    for _ in range(max(1, min(args.warmup, 2))):
        step_e2e()
    barrier()
    e2e_s = 0.0
    for s in range(args.steps):
        flush.fill_(s & 0xFF); torch.cuda.synchronize()
        t0 = time.perf_counter()
        step_e2e()
        e2e_s += time.perf_counter() - t0
    barrier()
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = cells_all * args.steps / e2e_s * 1e-9
    h2d = int(sum(hp[k].numel() * hp[k].element_size() for k in ("aw", "al", "bw", "bl")))
    d2h = int(out_host.numel() * 8)
    assert np.array_equal(out_host.numpy(), check_dev), "host and device entry points disagree"

    # ---- the same from raw symbol codes (ingest included: the codes are packed on the device) -------------
    for _ in range(2):
        step_codes()
    barrier()
    codes_s = 0.0
    for s in range(args.steps):
        flush.fill_(s & 0xFF); torch.cuda.synchronize()
        t0 = time.perf_counter()
        step_codes()
        codes_s += time.perf_counter() - t0
    barrier()
    if world > 1:
        t = torch.tensor([codes_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        codes_s = float(t.item())
    sampler.stop_flag.set(); sampler.join(timeout=2)
    assert np.array_equal(out_codes.numpy(), check_dev), "rsd_distance_batch_codes disagrees with the packed entry points"
    e2e_codes = {"value": cells_all * args.steps / codes_s * 1e-9, "unit": "GCUPS", "ms_per_step": codes_s / args.steps * 1e3,
                 "h2d_bytes_per_step": int(hc["ca"].numel() + hc["cb"].numel() + 8 * args.pairs), "d2h_bytes_per_step": d2h,
                 "what": "rsd_distance_batch_codes: 1 byte per symbol from pinned host memory, packed on the device per chunk"}

    # ---- BASELINE config 5 at every N: 10^7-record database sharded over the ranks, ONE all_gather per batch ----
    c5s = None
    if not args.no_extras:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs as BC
            c5s = BC.c5_sharded(eng, rank, world, dev, records=args.c5_records, steps=args.steps, warmup=args.warmup)
        except Exception as ex:                      # side measurements must never break the contract line
            c5s = {"error": repr(ex)}
        eng.set_costs(costs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel -----------------------------------------------------------
    kms = float(np.mean(kernel_ms))
    peaks = {}
    for name, which in (("iadd3", 0), ("viaddmnmx_s16x2", 2), ("prmt", 3), ("mix_cell", 7), ("dadd", 4), ("imad", 5)):
        try:
            peaks[name] = eng.ubench(which) * 1e-12
        except Exception as e:                      # pragma: no cover
            peaks[name] = None
            log("ubench failed:", e)
    peak = peaks["iadd3"]
    achieved = cells * 5.0 / (kms * 1e-3) * 1e-12          # Tiop/s, 5 integer ops per cell (SED:95-106)
    mp = {}
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(mp.get("hbm_gbs", 6650.0))
    alg_bytes = h2d + d2h
    roofline = {"bound": "int32_alu", "kernel": "k_dist_twin16<32>" if mode_used == 1 else ("k_dist_gen<int>" if mode_used == 2 else "k_dist_gen<double>"),
                "achieved": achieved, "peak": peak, "unit": "Tiop/s", "frac": achieved / peak if peak else None,
                "ops_per_cell": 5, "kernel_ms": kms, "kernel_gcups": cells / (kms * 1e-3) * 1e-9,
                "peak_source": "rsd_ubench IADD3 issue rate measured in this run (MEASURED_PEAKS.json has no INT32 entry)",
                "note": "frac > 1 is possible: DPX VIADDMNMX fuses add+min and the S16x2 forms update two cells per instruction",
                "issue_peaks_Tops": peaks, "traffic": None,
                "hbm": {"achieved": alg_bytes / (kms * 1e-3) * 1e-9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": alg_bytes / (kms * 1e-3) * 1e-9 / hbm_peak, "algorithmic_bytes": alg_bytes,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in mp else "fallback 6650"}}

    cpu = None
    if not args.no_cpu_baseline:
        g, cores, desc, dt = cpu_baseline(ca, oa, cb, ob, costs)
        cpu = {"value": g, "unit": "GCUPS", "cores": cores, "kind": "port", "sample": desc + f" ({dt:.1f} s)"}
        from oracle import oracle as O
        n_chk = 20000
        want = O.distance_batch(ca[: oa[n_chk]], oa[: n_chk + 1].copy(), cb[: ob[n_chk]], ob[: n_chk + 1].copy(), costs)
        assert np.array_equal(check_dev[:n_chk], want), "GPU distances differ from the oracle"
    cpu_py = None if args.no_cpu_baseline else python_reference_baseline(ca, oa, cb, ob, want=check_dev)
    if cpu_py is not None and cpu_py.get("matches_gpu") is False:
        raise AssertionError("GPU distances differ from the unmodified Python reference")

    # ---- side measurements of the other BASELINE configs (reduced sizes, N=1 only; full sizes: tools/bench_configs.py)
    extras = None
    if world == 1 and not args.no_extras:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_configs as BC
            e3 = BC.c3(eng, 20000, reps=2); e4 = BC.c4(eng, reps=2); e2i = BC.c2_iupac(eng, 200_000, reps=3)
            e5i = BC.c5(eng, 2_000_000, nq=64, reps=2, iupac=True); e1 = BC.c1(eng)
            extras = {"c1_xml_pairs_dropin_surface": e1,
                      "c3_script_patch_roundtrip": {"pairs": e3["pairs"], "pairs_per_s_device": e3["device_pairs_per_s"],
                                                    "gcups_device": e3["device_gcups"], "pairs_per_s_e2e": e3["e2e_pairs_per_s"],
                                                    "roundtrip_ok": e3["roundtrip_ok"], "oracle_checked_pairs": e3["oracle_checked_pairs"]},
                      "c4_long_pair_50kb": {"gcups_device": e4["device_gcups"], "ms_device": e4["device_s"] * 1e3,
                                            "forward_only_ms": e4["forward_only_device_s"] * 1e3, "n_ops": e4["n_ops"],
                                            "script_equals_oracle_digest": e4["script_equals_oracle_digest"],
                                            "roofline_frac_5ops": e4["device_gcups"] * 5e-3 / peak if peak else None,
                                            "batch": dict(e4["batch"], roofline_frac_5ops=e4["batch"]["device_gcups"] * 5e-3 / peak if peak else None) if e4.get("batch") else None},
                      "c5_iupac_mixed": dict(e5i, note="C5 second run (SURVEY 8d) at 2*10^6 records: 1 % of the records drawn from all 15 symbols; the int16x2 kernel "
                                                         "scores the common-alphabet prefix of the stored order, the fp64 kernels the IUPAC records; queries that carry "
                                                         "non-dyadic symbols form their own group; two queries checked against the oracle on the whole database"),
                      "c2_iupac_fp64": dict(e2i, roofline_frac_dadd=(e2i["device_gcups"] * 5e-3 / peaks["dadd"]) if peaks.get("dadd") else None,
                                            note="15-letter alphabet, default costs.json (0.66 / 0.83 ...): fp64 kernel in the reference's "
                                                 "operation order; 5 fp64-pipe ops per cell (3 DADD + 2 compares) against the measured DADD issue peak")}
        except Exception as ex:                      # side measurements must never break the contract line
            extras = {"error": repr(ex)}
    if c5s and "gcups" in c5s and peak:
        c5s["roofline_frac_5ops"] = c5s["gcups"] * 5e-3 / peak          # 5 integer ops per cell against the IADD3 issue peak
        c5s["roofline_frac_1alu_per_cell"] = c5s["gcups"] * 1e-3 / peak  # the kernel's own ceiling: one alu-pipe instruction per cell
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if mode_used == 1 and args.pairs == tj.get("pairs"):
            traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline["traffic"] = traffic
    roofline["traffic_source"] = "profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel at this size" if traffic else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, check_dev)          # rank 0's batch

    print(file=out, flush=True, *[json.dumps({
        "metric": "GCUPS", "value": value, "unit": "GCUPS", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {1: "s16x2", 2: "s32", 3: "f64"}[mode_used], "data": "synthetic",
        "config": config, "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_python": cpu_py,
        "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s / args.steps * 1e3},
        "e2e_from_codes": e2e_codes,
        "gpu_launches": int(round(launches_per_step * args.steps)), "launches_per_step": launches_per_step,
        "clocks": sampler.summary(), "other_configs": dict(extras or {}, c5_sharded_search=c5s) if (extras or c5s) else None})])
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
