// k_search.cuh — query batch vs resident database shard with exact top-k (BASELINE config 5).
//
// Replaces (reference): the wf_score scan of search_collection IR:466-477 (one wagnerFisher per
// document, IR:435-440) and the stable descending sort + [:k] of performance.py:12-15.
//
// Fast kernel (records <= 32 symbols, <= 7 distinct symbols incl. the queries', dyadic costs):
//   one thread = two database records (lo / hi half of every register, uint16 N = -H' values, max
//   form as in k_dist_twin16), the record right-aligned in 32 column registers and left-padded with
//   a PAD symbol whose v = 0 keeps N at the border value 0 — so the answer is always in column
//   register 31.
//   The query symbol of a row is uniform over the whole grid: its 8-byte row of the compact cost
//   table comes from shared memory with one broadcast LDS.64, and each packed cell is
//   PRMT (both records' v) + IMAD (packed add, fma pipe) + VIMNMX3.U16x2.
//   The record's selector registers are built once and reused for every query of the batch.
// Two epilogues share that body (template RANGE):
// Top-k: a candidate passes when its key (score desc, global index asc) is not worse than the
//   current k-th best key of its query (tau).  tau starts at "accept all" and is tightened after
//   every chunk by k_topk_fold, which also keeps the running top-k list.  The final order is a
//   total order on (score, index), so the result does not depend on atomic ordering.
// Range: every record whose scaled integer distance is <= floor(max_dist * 2^k) is appended as (key, D),
//   key = (query in batch << 32) | (global index - base); no threshold state, no fold.  The append order
//   depends on the atomics, so each batch's hits are sorted by key on the device (cub radix sort).
#pragma once
#include <type_traits>
#include "k_dist.cuh"

#define RSD_TOPK_MAX 128

struct SearchTab {               // per query-batch constants
    int ins, del;                // scaled
    double inv_scale;
    uint32_t compact_lut_lo, compact_lut_hi;   // 16 x 4-bit: original code -> compact index (7 = PAD / absent)
};

struct TopkState {
    double *tau_s; int64_t *tau_i;         // [Q] current k-th best key (score, index); index LLONG_MAX = accept all on ties
    double *best_s; int64_t *best_i;       // [Q][k] running top-k, sorted
    double *cand_s; int64_t *cand_i;       // [Q][cap] candidates of the current chunk
    int *cand_n;                           // [Q]
    int64_t cap;
    int k;
};

// hits of a range search (one query batch): the count may pass cap, the batch then reruns with a larger buffer
struct RangeHits {
    unsigned long long *keys;              // [cap] (query in batch << 32) | (global index - base)
    double *dist;                          // [cap] D
    unsigned long long *n;                 // hits appended (may exceed cap)
    int64_t cap;
    int thr;                               // fast kernel: floor(max_dist * 2^k), clamped to INT_MAX
    double max_dist;                       // general path: compared with the fp64 distance
};

// rowtab[q][i] = 8 bytes: v(query symbol i of q, compact symbol 0..6) = max(0, -w) <= 127; byte 7 (PAD) = 0
template <bool RANGE>
__global__ void __launch_bounds__(128)
k_search_twin16(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start,
                const int32_t *__restrict__ db_len, int64_t rec0, int64_t n_rec, int db_bits,
                const int64_t *__restrict__ perm, int64_t global_base, const uint2 *__restrict__ rowtab, int QROWS, const int32_t *__restrict__ q_len, int n_queries,
                SearchTab tab, TopkState tk, double *__restrict__ all_scores, int64_t all_stride, uint32_t one, RangeHits rh) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint2 *s_rows = reinterpret_cast<uint2 *>(smem_raw);                     // [n_queries][QROWS]
    double *s_tau = reinterpret_cast<double *>(s_rows + (size_t)n_queries * QROWS);
    long long *s_taui = reinterpret_cast<long long *>(s_tau + n_queries);
    int *s_qlen = reinterpret_cast<int *>(s_taui + n_queries);
    for (int k = threadIdx.x; k < n_queries * QROWS; k += blockDim.x) s_rows[k] = rowtab[k];
    for (int k = threadIdx.x; k < n_queries; k += blockDim.x) {
        if constexpr (!RANGE) { s_tau[k] = tk.tau_s[k]; s_taui[k] = tk.tau_i[k]; }
        s_qlen[k] = q_len[k];
    }
    __syncthreads();

    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t rA0 = rec0 + 2 * t;
    const bool live = rA0 < rec0 + n_rec;                     // dead threads idle through the loops (warp votes below)
    const int64_t rA = live ? rA0 : rec0, rB = rA + 1;
    const bool hasB = live && rB < rec0 + n_rec;
    const int nA = db_len[rA], nB = hasB ? db_len[rB] : nA;
    // the database is stored sorted by length, so the records of a warp share (almost always) one
    // length: columns left of the longest record are padding for every lane and are skipped, two at a time
    int cskip = 32 - max(nA, nB);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cskip = min(cskip, __shfl_xor_sync(RSD_FULL, cskip, o));
    const uint32_t *wA = db_words + db_start[rA];
    const uint32_t *wB = hasB ? db_words + db_start[rB] : wA;
    const uint64_t lut = ((uint64_t)tab.compact_lut_hi << 32) | tab.compact_lut_lo;

    // selectors: nibbles [idx A][8|idx A -> sign][idx B][8|idx B -> sign], both index the same 8-byte row
    uint32_t sel[32];
    {
        const int per = 32 / db_bits;
        uint32_t cwA = 0, cwB = 0;
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const int jA = c - (32 - nA), jB = c - (32 - nB);
            uint32_t ia = 7u, ib = 7u;                                       // PAD
            if (jA >= 0) {
                if (jA % per == 0 || c == 32 - nA) cwA = __ldg(wA + jA / per);
                const uint32_t code = (cwA >> ((jA % per) * db_bits)) & ((1u << db_bits) - 1u);
                ia = (uint32_t)(lut >> (4 * code)) & 7u;
            }
            if (jB >= 0) {
                if (jB % per == 0 || c == 32 - nB) cwB = __ldg(wB + jB / per);
                const uint32_t code = (cwB >> ((jB % per) * db_bits)) & ((1u << db_bits) - 1u);
                ib = (uint32_t)(lut >> (4 * code)) & 7u;
            }
            sel[c] = 0x8080u + ia * 0x11u + ib * 0x1100u;
        }
    }
    const int baseA = nA * tab.ins, baseB = nB * tab.ins;
    // gridDim.y > 1 (the short seeding chunk) splits the query batch over blockIdx.y to shorten the pass
    const int q_lo = (int)((long long)n_queries * blockIdx.y / gridDim.y), q_hi = (int)((long long)n_queries * (blockIdx.y + 1) / gridDim.y);

    // One copy of the query loop per number of skipped padding columns (0, 2, .. 16): the column loop is
    // fully unrolled from SKIP on, with no per-row tests.
    auto run_queries = [&](auto skip_tag) {
        constexpr int SKIP = decltype(skip_tag)::value;
        for (int q = q_lo; q < q_hi; ++q) {
            uint32_t H[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) H[c] = 0u;
            const int m = s_qlen[q];
            const uint2 *rows = s_rows + (size_t)q * QROWS;
#pragma unroll 2
            for (int i = 0; i < m; ++i) {
                const uint2 r = rows[i];
                // skipped columns hold the border value 0 and hand 0 to the first computed column
                uint32_t left = 0u, diag = 0u;
#pragma unroll
                for (int c = SKIP; c < 32; ++c) {
                    const uint32_t v = prmt(r.x, r.y, sel[c]);
                    const uint32_t x = add_fma(v, diag, one);
                    diag = H[c];
                    H[c] = max3u16x2(x, H[c], left);
                    left = H[c];
                }
            }
            const int dA = m * tab.del + baseA - (int)(H[31] & 0xffffu);
            const int dB = m * tab.del + baseB - (int)(H[31] >> 16);
            if constexpr (RANGE) {
                const bool cA = live && dA <= rh.thr, cB = hasB && dB <= rh.thr;
                const unsigned mA = __ballot_sync(RSD_FULL, cA), mB = __ballot_sync(RSD_FULL, cB);
                if (mA | mB) {
                    const int lane_id = threadIdx.x & 31;
                    unsigned long long base = 0;
                    if (lane_id == 0) base = atomicAdd(rh.n, (unsigned long long)(__popc(mA) + __popc(mB)));
                    base = __shfl_sync(RSD_FULL, base, 0);
                    const unsigned below = (1u << lane_id) - 1u;
                    const unsigned long long qk = (unsigned long long)q << 32;
                    if (cA) {
                        const unsigned long long slot = base + __popc(mA & below);
                        if (slot < (unsigned long long)rh.cap) { rh.keys[slot] = qk | (unsigned long long)(perm[rA] - global_base); rh.dist[slot] = __dmul_rn((double)dA, tab.inv_scale); }
                    }
                    if (cB) {
                        const unsigned long long slot = base + __popc(mA) + __popc(mB & below);
                        if (slot < (unsigned long long)rh.cap) { rh.keys[slot] = qk | (unsigned long long)(perm[rB] - global_base); rh.dist[slot] = __dmul_rn((double)dB, tab.inv_scale); }
                    }
                }
                continue;
            }
            // IR:440  score = 1 / (1 + cost)
            const double sA = __ddiv_rn(1.0, __dadd_rn(1.0, __dmul_rn((double)dA, tab.inv_scale)));
            const double sB = __ddiv_rn(1.0, __dadd_rn(1.0, __dmul_rn((double)dB, tab.inv_scale)));
            const long long gA = perm[rA], gB = perm[rB < rec0 + n_rec ? rB : rA];
            if (all_scores && live) {
                all_scores[(size_t)q * all_stride + (gA - global_base)] = sA;
                if (hasB) all_scores[(size_t)q * all_stride + (gB - global_base)] = sB;
            }
            if (tk.k > 0) {
                // candidates are appended with one atomic per warp (ballot + rank): in the seeding chunk every record is a
                // candidate of every query, and 4096 same-address atomics per query were 3/4 of that launch (ncu: 177 us)
                const double ts = s_tau[q]; const long long ti = s_taui[q];
                const bool cA = live && (sA > ts || (sA == ts && gA <= ti));
                const bool cB = hasB && (sB > ts || (sB == ts && gB <= ti));
                const unsigned mA = __ballot_sync(RSD_FULL, cA), mB = __ballot_sync(RSD_FULL, cB);
                if (mA | mB) {
                    const int lane_id = threadIdx.x & 31;
                    int base = 0;
                    if (lane_id == 0) base = atomicAdd(&tk.cand_n[q], __popc(mA) + __popc(mB));
                    base = __shfl_sync(RSD_FULL, base, 0);
                    const unsigned below = (1u << lane_id) - 1u;
                    if (cA) {
                        const int slot = base + __popc(mA & below);
                        if (slot < tk.cap) { tk.cand_s[(size_t)q * tk.cap + slot] = sA; tk.cand_i[(size_t)q * tk.cap + slot] = gA; }
                    }
                    if (cB) {
                        const int slot = base + __popc(mA) + __popc(mB & below);
                        if (slot < tk.cap) { tk.cand_s[(size_t)q * tk.cap + slot] = sB; tk.cand_i[(size_t)q * tk.cap + slot] = gB; }
                    }
                }
            }
        }
    };
    switch (min(cskip, 16) >> 1) {          // warp-uniform
        case 0: run_queries(std::integral_constant<int, 0>{}); break;
        case 1: run_queries(std::integral_constant<int, 2>{}); break;
        case 2: run_queries(std::integral_constant<int, 4>{}); break;
        case 3: run_queries(std::integral_constant<int, 6>{}); break;
        case 4: run_queries(std::integral_constant<int, 8>{}); break;
        case 5: run_queries(std::integral_constant<int, 10>{}); break;
        case 6: run_queries(std::integral_constant<int, 12>{}); break;
        case 7: run_queries(std::integral_constant<int, 14>{}); break;
        default: run_queries(std::integral_constant<int, 16>{}); break;
    }
}

__global__ void k_topk_init(TopkState tk, int n_queries) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n_queries) return;
    tk.tau_s[q] = -INFINITY; tk.tau_i[q] = 0x7fffffffffffffffLL;  // accept everything
    tk.cand_n[q] = 0;
    for (int r = 0; r < tk.k; ++r) { tk.best_s[(size_t)q * tk.k + r] = 0.0; tk.best_i[(size_t)q * tk.k + r] = -1; }
}

// key order: a before b  <=>  score_a > score_b, or equal scores and index_a < index_b
__device__ __forceinline__ bool key_before(double sa, long long ia, double sb, long long ib) {
    return sa > sb || (sa == sb && ia < ib);
}

// One CTA per query: merge this chunk's candidates into the running sorted top-k, update tau.
// k rounds of "best remaining candidate" (block argbest), each inserted into the sorted list.
__global__ void __launch_bounds__(256) k_topk_fold(TopkState tk) {
    const int q = blockIdx.x;
    const int tid = threadIdx.x;
    __shared__ double s_bs[RSD_TOPK_MAX]; __shared__ long long s_bi[RSD_TOPK_MAX];
    __shared__ double r_s[256]; __shared__ long long r_i[256]; __shared__ int r_pos[256];
    const int k = tk.k;
    const int n = (int)min((int64_t)tk.cand_n[q], tk.cap);
    for (int r = tid; r < k; r += 256) { s_bs[r] = tk.best_s[(size_t)q * k + r]; s_bi[r] = tk.best_i[(size_t)q * k + r]; }
    __syncthreads();
    double *cs = tk.cand_s + (size_t)q * tk.cap; int64_t *ci = tk.cand_i + (size_t)q * tk.cap;
    // every thread keeps the best of its own (strided) candidates; after a round only the winner's owner rescans
    double bs = -2.0; long long bi = 0x7fffffffffffffffLL; int bp = -1;
    auto rescan = [&]() {
        bs = -2.0; bi = 0x7fffffffffffffffLL; bp = -1;
        for (int c = tid; c < n; c += 256) {
            const long long idx = ci[c];
            if (idx == -2) continue;                         // taken in an earlier round
            const double s = cs[c];
            if (bp < 0 || key_before(s, idx, bs, bi)) { bs = s; bi = idx; bp = c; }
        }
    };
    rescan();
    for (int round = 0; round < k; ++round) {
        r_s[tid] = bs; r_i[tid] = bi; r_pos[tid] = bp;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (tid < o) {
                const int ob = r_pos[tid + o];
                if (ob >= 0 && (r_pos[tid] < 0 || key_before(r_s[tid + o], r_i[tid + o], r_s[tid], r_i[tid]))) {
                    r_s[tid] = r_s[tid + o]; r_i[tid] = r_i[tid + o]; r_pos[tid] = ob;
                }
            }
            __syncthreads();
        }
        const int wp = r_pos[0];
        if (wp < 0) break;                                   // no candidates left
        const double ws = r_s[0]; const long long wi = r_i[0];
        __syncthreads();
        // insert into the sorted list if it beats the current last entry (or the list has a free slot)
        const bool list_full = s_bi[k - 1] >= 0;
        const bool better = !list_full || key_before(ws, wi, s_bs[k - 1], s_bi[k - 1]);
        __syncthreads();
        if (!better) break;                                  // candidates come out best-first: nothing further can enter
        if (tid == 0) {
            // duplicates (same global index already in the list) cannot occur: every record is scanned once
            int pos = k - 1;
            while (pos > 0 && (s_bi[pos - 1] < 0 || key_before(ws, wi, s_bs[pos - 1], s_bi[pos - 1]))) {
                s_bs[pos] = s_bs[pos - 1]; s_bi[pos] = s_bi[pos - 1]; --pos;
            }
            s_bs[pos] = ws; s_bi[pos] = wi;
        }
        if (tid == (wp & 255)) { ci[wp] = -2; rescan(); }    // the owner of the winner marks it taken and refreshes its best
        __syncthreads();
    }
    __syncthreads();
    for (int r = tid; r < k; r += 256) { tk.best_s[(size_t)q * k + r] = s_bs[r]; tk.best_i[(size_t)q * k + r] = s_bi[r]; }
    if (tid == 0) {
        tk.cand_n[q] = 0;
        if (s_bi[k - 1] >= 0) { tk.tau_s[q] = s_bs[k - 1]; tk.tau_i[q] = s_bi[k - 1]; }
    }
}


// rowtab[q][i] from the packed queries: byte b < 7 = v(query symbol, compact symbol b), byte 7 = 0 (PAD)
__global__ void k_build_rowtab(const uint32_t *__restrict__ q_words, const int64_t *__restrict__ q_start,
                               const int32_t *__restrict__ q_len, int n_queries, int bits, int QROWS,
                               const IntCosts *__restrict__ ic, uint32_t compact_syms_lo, uint32_t compact_syms_hi,
                               uint2 *__restrict__ rowtab) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_queries * QROWS) return;
    const int q = idx / QROWS, i = idx % QROWS;
    uint2 r = make_uint2(0u, 0u);
    if (i < q_len[q]) {
        const uint32_t a = pk_get(q_words, q_start[q], i, bits);
        const uint64_t syms = ((uint64_t)compact_syms_hi << 32) | compact_syms_lo;   // 7 x 4-bit original codes
        uint64_t v = 0;
        for (int b = 0; b < 7; ++b) {
            const uint32_t sym = (uint32_t)(syms >> (4 * b)) & 15u;
            v |= (uint64_t)(uint8_t)max(0, -ic->w[a][sym]) << (8 * b);
        }
        r = make_uint2((uint32_t)v, (uint32_t)(v >> 32));
    }
    rowtab[idx] = r;
}

// General path, a whole group of queries at once: pair p = (query q_base + p / n_rec, record rec0 + p % n_rec) as the
// (start, len) views the systolic distance kernels take.
__global__ void k_fill_pairs_view(const int64_t *__restrict__ q_start, const int32_t *__restrict__ q_len, int q_base, int n_q,
                                  const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len, int64_t rec0, int64_t n_rec,
                                  int64_t *__restrict__ a_start, int32_t *__restrict__ a_len, int64_t *__restrict__ b_start, int32_t *__restrict__ b_len) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (int64_t)n_q * n_rec) return;
    const int q = q_base + (int)(p / n_rec); const int64_t r = rec0 + p % n_rec;
    a_start[p] = q_start[q]; a_len[p] = q_len[q];
    b_start[p] = db_start[r]; b_len[p] = db_len[r];
}

// ... and their distances (produced by the systolic distance kernels, any mode) -> scores, optional all_scores rows, and
// the candidates of each of the n_q queries
__global__ void k_score_filter_pairs(const double *__restrict__ dist, int64_t rec0, int64_t n_rec, const int64_t *__restrict__ perm,
                                     int64_t global_base, int q_base, int n_q, TopkState tk, double *__restrict__ all_scores, int64_t all_stride) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (int64_t)n_q * n_rec) return;
    const int q = q_base + (int)(p / n_rec); const int64_t r = p % n_rec;
    const double s = __ddiv_rn(1.0, __dadd_rn(1.0, dist[p]));
    const long long g = perm[rec0 + r];
    if (all_scores) all_scores[(size_t)q * all_stride + (g - global_base)] = s;
    if (tk.k > 0) {
        const double ts = tk.tau_s[q]; const long long ti = tk.tau_i[q];
        if (s > ts || (s == ts && g <= ti)) {
            // one atomic per (warp, query): the candidates of a warp almost always belong to one query
            const unsigned act = __activemask();
            const unsigned peers = __match_any_sync(act, q);
            const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
            int base = 0;
            if (lane == leader) base = atomicAdd(&tk.cand_n[q], __popc(peers));
            base = __shfl_sync(peers, base, leader);
            const int slot = base + __popc(peers & ((1u << lane) - 1u));
            if (slot < tk.cap) { tk.cand_s[(size_t)q * tk.cap + slot] = s; tk.cand_i[(size_t)q * tk.cap + slot] = g; }
        }
    }
}

// ... or, in a range search, the pairs within max_dist (fp64 compare: the distance of an integer mode is exactly
// d / 2^k, so d / 2^k <= max_dist decides as d <= floor(max_dist * 2^k) would).  q_base is the query in the batch.
__global__ void k_range_filter_pairs(const double *__restrict__ dist, int64_t rec0, int64_t n_rec, const int64_t *__restrict__ perm,
                                     int64_t global_base, int q_base, int n_q, RangeHits rh) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (int64_t)n_q * n_rec) return;
    const double d = dist[p];
    if (!(d <= rh.max_dist)) return;
    const int q = q_base + (int)(p / n_rec); const int64_t r = p % n_rec;
    // one atomic per (warp, query), as in k_score_filter_pairs
    const unsigned peers = __match_any_sync(__activemask(), q);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(rh.n, (unsigned long long)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    const unsigned long long slot = base + __popc(peers & ((1u << lane) - 1u));
    if (slot < (unsigned long long)rh.cap) {
        rh.keys[slot] = ((unsigned long long)q << 32) | (unsigned long long)(perm[rec0 + r] - global_base);
        rh.dist[slot] = d;
    }
}

// after the sort by key: idx[i] = global index of hit i; off[q] = first hit of query q of the batch (off[n_q] = n)
__global__ void k_range_split(const unsigned long long *__restrict__ keys, int64_t n, int n_q, int64_t global_base,
                              int64_t *__restrict__ idx, int64_t *__restrict__ off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (int64_t)(keys[i] & 0xffffffffull) + global_base;
    if (i <= n_q) {
        const unsigned long long want = (unsigned long long)i << 32;
        int64_t lo = 0, hi = n;
        while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (keys[mid] < want) lo = mid + 1; else hi = mid; }
        off[i] = lo;
    }
}
