// k_plan.cuh — device-side work planning for the systolic warp kernels.
//
// A pair (m source symbols, n destination symbols) needs ns = ceil(n / C) lanes ("strips" of C
// matrix columns held in registers).  Pairs are binned by (ns, m) with a counting sort.  The strips
// of the G groups of one warp task are laid end to end on a *tape* of 32*P lane slots which the warp
// walks in P passes; a group whose strips straddle a pass boundary hands its boundary column from
// lane 31 of one pass to lane 0 of the next through a small per-warp scratch column.  (P, G) is
// chosen per ns to minimise idle lanes: e.g. ns = 7 -> 9 groups on 2 passes (63 of 64 slots) instead
// of 4 groups on one (28 of 32); ns = 47 -> 2 groups on 3 passes (94 of 96) instead of 1 on 2 (47/64).
//   * "twin" bins put two pairs of identical (ns, m) into one group — the int16x2 kernels carry
//     one pair in each half of every register;
//   * pairs with more than RSD_NSQ_MAX strips form one class of single-group tasks.
// Bins are numbered heaviest first so the persistent kernels hand out the long tasks first.
#pragma once
#include <cooperative_groups.h>
#include "rsd_common.cuh"

#define RSD_MQ_MAX 2048                   // m is binned exactly below MQ-1, clamped above; MQ <= this
#define RSD_NSQ_MAX 128                   // ns is binned exactly up to here; longer pairs share class NSQ_MAX+1
#define RSD_NB_MAX ((RSD_NSQ_MAX + 2) * RSD_MQ_MAX)
#define RSD_PLAN_COPIES 8                 // privatised bin counters: the L2 serialises atomics per address
#ifndef RSD_TAPE_GAIN
#define RSD_TAPE_GAIN 108                 // extra passes must buy this much utilisation (percent of the shortest layout)
#endif

struct PlanView {
    int *pair_bin;        // [n_pairs] bin of each pair, -1 = trivial (m == 0 or n == 0)
    int *bin_cnt;         // [COPIES][NB_MAX] privatised counters (copy = warp index & 7)
    int *bin_cursor;      // [COPIES][NB_MAX] per-copy cursors, preset to the copy's first rank inside its bin
    int *bin_group_off;   // [NB + 1] exclusive scan of groups per bin
    int *bin_warp_off;    // [NSC + 1] exclusive scan of warp tasks per strip class (tasks are cut from a class's whole group list)
    int2 *groups;         // [n_pairs] {pair A, pair B or -1}
    int *totals;          // {n_groups, n_tasks}
    int *work_counter;    // persistent-kernel ticket
    int C;                // columns per lane
    int allow_twin;
    int m_shift;          // rows are binned as m >> m_shift: 0 (exact) when twins need equal m, coarser otherwise
    int MQ;               // row bins per class for this call: min((max_m >> m_shift) + 2, RSD_MQ_MAX)
    int NSC;              // strip classes for this call: min(max_ns, RSD_NSQ_MAX + 1); classes 1..NSC
    int NB;               // NSC * MQ
    int band;             // tasks for k_dist_band16: 32 groups each, no tape (every class <= RSD_NSQ_MAX)
    unsigned long long *dbg;
};

// Twin plans may process a pair with the roles of the two sequences swapped (columns = the source): the
// distance is the same number with ins/del exchanged and the substitution table transposed, and the
// orientation with fewer strip-padding cells is taken: m * (n + pad(n))  vs  n * (m + pad(m)).
__host__ __device__ __forceinline__ bool plan_swap(int m, int n, int C) {
    const int pn = (n + C - 1) / C * C - n, pm = (m + C - 1) / C * C - m;
    return (long long)n * pm < (long long)m * pn;
}
__host__ __device__ __forceinline__ int plan_nsq(int ns) { return ns > RSD_NSQ_MAX ? RSD_NSQ_MAX + 1 : ns; }
__device__ __forceinline__ int plan_bin(int m, int n, const PlanView &pv) {
    const int nsq = plan_nsq((n + pv.C - 1) / pv.C);
    const int ms = m >> pv.m_shift;
    const int mq = ms < pv.MQ - 1 ? ms : pv.MQ - 1;
    return (pv.NSC - nsq) * pv.MQ + (pv.MQ - 1 - mq);
}
__device__ __forceinline__ int bin_nsq(int bin, const PlanView &pv) { return pv.NSC - bin / pv.MQ; }
__device__ __forceinline__ int bin_mq(int bin, const PlanView &pv) { return pv.MQ - 1 - bin % pv.MQ; }
__device__ __forceinline__ bool bin_twin(int bin, const PlanView &pv) {
    return pv.allow_twin && bin_nsq(bin, pv) <= RSD_NSQ_MAX && bin_mq(bin, pv) < pv.MQ - 1;
}

// groups per task G and passes P for groups of ns strips: maximise the lane-slot utilisation
// G*ns / (32*P).  Passes with a boundary hand-off run a slightly heavier row loop, so extra passes
// are only taken when they buy at least 8 % more utilisation than the shortest layout.
__host__ __device__ __forceinline__ void tape_shape(int nsq, int &P, int &G) {
    if (nsq > RSD_NSQ_MAX) { P = 0; G = 1; return; }          // P depends on the pair: computed in the kernel
    const int pmin = (nsq + 31) >> 5;
    const int pmax = nsq <= 32 ? 4 : (pmin + 4 < 8 ? 8 : pmin + 4);
    const int g0 = (32 * pmin) / nsq;
    int bp = pmin, bg = g0;
    for (int p = pmin + 1; p <= pmax; ++p) {
        const int g = (32 * p) / nsq;
        if ((long long)g * bp > (long long)bg * p) { bp = p; bg = g; }      // g/p > bg/bp
    }
    // utilisation ratio best/shortest = (bg/bp) / (g0/pmin) >= 1.08 ?
    if ((long long)bg * pmin * 100 < (long long)g0 * bp * RSD_TAPE_GAIN) { bp = pmin; bg = g0; }
    P = bp; G = bg;
}

// groups per task and passes of the layout the plan is cut for
__host__ __device__ __forceinline__ void task_shape(const PlanView &pv, int nsq, int &P, int &G) {
    if (pv.band) { P = 1; G = 32; return; }
    tape_shape(nsq, P, G);
}

// trivial pairs are answered here: D = n*ins (m == 0) or m*del (n == 0) — one fp64 multiply,
// like the reference's border rows (SED:159,177).
// -> the pair's bin (-1: answered here)
__device__ __forceinline__ int plan_count_one(const int32_t *__restrict__ a_len, const int32_t *__restrict__ b_len, int64_t p,
                                              const PlanView &pv, double ins, double del, double *out) {
    int m = a_len[p], n = b_len[p];
    if (m == 0 || n == 0) {
        pv.pair_bin[p] = -1;
        if (out) out[p] = m == 0 ? __dmul_rn((double)n, ins) : __dmul_rn((double)m, del);
        return -1;
    }
    if (pv.allow_twin && plan_swap(m, n, pv.C)) { const int t = m; m = n; n = t; }
    int bin = plan_bin(m, n, pv);
    pv.pair_bin[p] = bin;
    return bin;
}

// one block of 1024 threads walks the bins in coalesced chunks of 1024; (groups, tasks) are scanned
// together as one 64-bit value with warp shuffles (three barriers per chunk)
__device__ __forceinline__ void plan_scan_block(const PlanView &pv) {      // one block of 1024 threads
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_total;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    unsigned long long carry = 0ull;                     // same value in every thread
    for (int base = 0; base < pv.NB; base += 1024) {
        const int b = base + t;
        unsigned long long v = 0ull;
        int c = 0;
        if (b < pv.NB) {
#pragma unroll
            for (int k = 0; k < RSD_PLAN_COPIES; ++k) {
                const int ck = pv.bin_cnt[(size_t)k * RSD_NB_MAX + b];
                pv.bin_cursor[(size_t)k * RSD_NB_MAX + b] = c;              // this copy's first rank inside the bin
                if (ck) pv.bin_cnt[(size_t)k * RSD_NB_MAX + b] = 0;         // leave the counters zeroed for the next plan
                c += ck;
            }
            if (c) {
                const int groups = bin_twin(b, pv) ? (c + 1) >> 1 : c;
                v = (unsigned long long)groups << 32;
            }
        }
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(RSD_FULL, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_warp[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const unsigned long long x = s_warp[lane];
            unsigned long long xi = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(RSD_FULL, xi, o);
                if (lane >= o) xi += y;
            }
            s_warp[lane] = xi - x;                       // exclusive offset of each warp
            if (lane == 31) s_total = xi;
        }
        __syncthreads();
        const unsigned long long excl = carry + s_warp[wid] + (inc - v);
        if (b < pv.NB) {
            pv.bin_group_off[b] = (int)(excl >> 32);
            // a twin bin with an odd count leaves its last group without a partner
            if ((c & 1) && bin_twin(b, pv)) pv.groups[(int)(excl >> 32) + (c >> 1)].y = -1;
        }
        carry += s_total;
        __syncthreads();
    }
    // Warp tasks are cut from the group list of a whole strip class (all row bins of one ns, rows descending), G groups
    // each, not bin by bin: a bin's last, partly filled task used to cost half a task per bin on average — a quarter of
    // the work of a 74 k-pair chunk spread over 2000 (ns, m) bins.  The groups of a task now may differ a little in m
    // (neighbouring bins); every lane keeps its own row count.  bin_warp_off[0 .. NSC] holds the task offsets per class.
    if (t == 0) pv.bin_group_off[pv.NB] = (int)(carry >> 32);
    __syncthreads();
    if (t == 0) {
        int tasks = 0;
        for (int ci = 0; ci < pv.NSC; ++ci) {
            pv.bin_warp_off[ci] = tasks;
            const int groups = pv.bin_group_off[(ci + 1) * pv.MQ] - pv.bin_group_off[ci * pv.MQ];
            int P, G;
            task_shape(pv, pv.NSC - ci, P, G);
            tasks += (groups + G - 1) / G;
        }
        pv.bin_warp_off[pv.NSC] = tasks;
        pv.totals[0] = (int)(carry >> 32); pv.totals[1] = tasks;
        *pv.work_counter = 0;
    }
}

// rank r of pair p inside its bin (any assignment of distinct ranks will do)
__device__ __forceinline__ void plan_fill_one(int64_t p, int bin, int r, const PlanView &pv) {
    int *g = reinterpret_cast<int *>(pv.groups);
    if (bin_twin(bin, pv)) g[2 * (pv.bin_group_off[bin] + (r >> 1)) + (r & 1)] = (int)p;
    else pv.groups[pv.bin_group_off[bin] + r] = make_int2((int)p, -1);
}

// The whole plan as ONE cooperative launch (count -> grid sync -> scan by block 0 -> grid sync -> fill):
// three dependent tiny kernels cost ~0.1 ms of launch latency per call, two grid syncs a few microseconds.
__global__ void __launch_bounds__(1024) k_plan_all(const int32_t *__restrict__ a_len, const int32_t *__restrict__ b_len,
                                                   int64_t n_pairs, PlanView pv, double ins, double del, double *out) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long t0 = 0, t1 = 0, t2 = 0, t3 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    // Counter updates are aggregated per warp: the lanes that hit the same bin (MATCH.ANY) send one atomic with their
    // number.  Batches of one shape — the (query, record) pairs of a database search: 6 * 10^6 pairs in a handful of
    // bins — otherwise serialise on a few addresses (2.3 ms per plan, ncu); mixed batches lose nothing.
    const int lane = threadIdx.x & 31;
    const size_t copy = (size_t)((threadIdx.x >> 5) & (RSD_PLAN_COPIES - 1)) * RSD_NB_MAX;
    for (int64_t p0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); p0 < n_pairs; p0 += stride) {
        const int64_t p = p0 + lane;
        const int bin = p < n_pairs ? plan_count_one(a_len, b_len, p, pv, ins, del, out) : -1;
        const unsigned peers = __match_any_sync(RSD_FULL, bin);
        if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&pv.bin_cnt[copy + bin], __popc(peers));
    }
    grid.sync();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (blockIdx.x == 0) plan_scan_block(pv);
    grid.sync();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t2));
    for (int64_t p0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); p0 < n_pairs; p0 += stride) {
        const int64_t p = p0 + lane;
        const int bin = p < n_pairs ? pv.pair_bin[p] : -1;
        const unsigned peers = __match_any_sync(RSD_FULL, bin);
        const int leader = __ffs(peers) - 1;
        int base = 0;
        if (bin >= 0 && lane == leader) base = atomicAdd(&pv.bin_cursor[copy + bin], __popc(peers));
        base = __shfl_sync(RSD_FULL, base, leader);
        if (bin >= 0) plan_fill_one(p, bin, base + __popc(peers & ((1u << lane) - 1u)), pv);
    }
    if (pv.dbg) {                                   // RSD_TRACE: phase times
        grid.sync();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t3));
        if (blockIdx.x == 0 && threadIdx.x == 0) { pv.dbg[0] = t1 - t0; pv.dbg[1] = t2 - t1; pv.dbg[2] = t3 - t2; }
    }
}

// ---- one warp task (warp-uniform part), decoded by every lane --------------------------------
struct TapeTask {
    int ns;            // strips per group; 0 = class of longer pairs (take it from the pair)
    int P;             // passes (0 = from the pair)
    int gfirst;        // index of the task's first group in pv.groups
    int ng;            // groups in this task
};

__device__ __forceinline__ TapeTask plan_decode(const PlanView &pv, int W) {
    int lo = 0, hi = pv.NSC;                       // largest strip class ci with bin_warp_off[ci] <= W
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(&pv.bin_warp_off[mid]) <= W) lo = mid; else hi = mid;
    }
    const int ci = lo;
    const int nsq = pv.NSC - ci;
    int P, G;
    task_shape(pv, nsq, P, G);
    const int gbase = __ldg(&pv.bin_group_off[ci * pv.MQ]);
    const int gcount = __ldg(&pv.bin_group_off[(ci + 1) * pv.MQ]) - gbase;
    const int wl = W - __ldg(&pv.bin_warp_off[ci]);
    TapeTask t;
    t.ns = nsq > RSD_NSQ_MAX ? 0 : nsq;
    t.P = P;
    t.gfirst = gbase + wl * G;
    t.ng = min(G, gcount - wl * G);
    return t;
}

// ---- what one lane does in one pass of a task -------------------------------------------------
struct LaneSlot {
    int pA, pB;        // pair indices (pB == pA when the group has no twin)
    bool hasB;
    bool on;           // the slot holds a strip
    int s;             // strip index inside its group
    int sk;            // row skew of this lane in this pass (lanes of one group run one row apart)
    bool lead;         // s == 0: the matrix border is the left neighbour
    bool from_scratch; // lane 0 continuing a group that started in the previous pass
    bool to_scratch;   // lane 31 whose group continues in the next pass
};

__device__ __forceinline__ LaneSlot tape_slot(const PlanView &pv, const TapeTask &tt, int ns, int pass, int lane) {
    LaneSlot ls;
    const int q = pass * 32 + lane;
    const int g = q / ns;
    ls.s = q - g * ns;
    ls.on = g < tt.ng;
    const int q0 = max(g * ns, pass * 32);          // first slot of this group inside this pass
    ls.sk = q - q0;
    ls.lead = ls.s == 0;
    ls.from_scratch = ls.on && lane == 0 && ls.s > 0;
    ls.to_scratch = ls.on && lane == 31 && ls.s < ns - 1;
    ls.pA = ls.pB = -1; ls.hasB = false;
    if (ls.on) {
        const int2 gp = pv.groups[tt.gfirst + g];
        ls.pA = gp.x; ls.hasB = gp.y >= 0; ls.pB = ls.hasB ? gp.y : gp.x;
    }
    return ls;
}
