// k_sim.cuh — set / multiset / TF-vector similarity of one query against the loaded database
// (SURVEY 8f rank 4; reference IRMethods.py IR:49-389 driven by search_collection IR:443-477).
//
// The reference computes these measures with numpy, so "identical results" means re-creating numpy's
// arithmetic: every product / sum / square root below is a single correctly rounded fp64 operation
// (__dmul_rn, __dadd_rn, ... — no fma contraction), and reductions over the 15x15 TF matrix follow
// numpy's pairwise summation for 225 contiguous doubles: two blocks (elements 0..111 and 112..224), in
// each block eight strided accumulators r[j] += x[8g + j], combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
// the 225th element added last to the second block, then block1 + block2.
//
//   k_sim_query   one warp: representations of the query (symbol mask, 4-vector, TF matrix, centred TF
//                 matrix and their norms) -> SimQuery in global memory
//   k_sim_small   one thread per record: set_* and multi_* measures (a mask and four sequential sums)
//   k_sim_tf_thread  one thread per record made of A, G, C, U only: 16 bigram counts, the 225-term sums unrolled
//   k_sim_tf      one warp per record (records with ambiguity codes): TF matrix in shared memory, the vector measures
//
// Query batches (rsd_db_similarity_batch): the same arithmetic, each record rebuilt once per batch and scored against
// every query of it; scores [Q][stride] in record order.
//   k_sim_query_batch        one warp per query -> SimQuery[q]
//   k_sim_small_batch        one thread per record: its mask and four sums once, then every query (constants in shared memory)
//   k_sim_tf_thread_batch    one thread per A/G/C/U record: 16 bigram counts in registers, the record-only sums once, the
//                            query TF vectors staged in shared memory RSD_SIM_QT at a time
//   k_sim_tf_batch           one warp per worklist record: TF matrix in shared memory once, then every query
//   k_sim_filter_batch       the top-k candidates of one score range, query = blockIdx.y
#pragma once
#include "../../include/rsd.h"
#include "rsd_common.cuh"

#define RSD_SIM_COUNT 12          // the RSD_SIM_* method ids are declared in include/rsd.h

#define RSD_TF 225

struct SimQuery {
    double tf[RSD_TF];       // IR:147-186
    double tfc[RSD_TF];      // tf - average(tf)  (IR:309-314)
    double tf_sq, tfc_sq;    // sum(tf^2), sum(tfc^2)
    double ms[4];            // IR:95-107
    double ms_sum;           // np.sum(ms)
    uint32_t mask;           // IR:49-51
};

// IR:20-46: probability of each base (A, G, C, U) behind every symbol; the bases are unit vectors
__device__ const double c_simW[16][4] = {
    {1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1},
    {0, 0, 0.5, 0.5}, {0.5, 0.5, 0, 0}, {0.5, 0, 0, 0.5}, {0, 0.5, 0.5, 0}, {0, 0.5, 0, 0.5}, {0.5, 0, 0.5, 0},
    {0.33, 0.33, 0, 0.33}, {0.33, 0.33, 0.33, 0}, {0.33, 0, 0.33, 0.33}, {0, 0.33, 0.33, 0.33},
    {0.25, 0.25, 0.25, 0.25}, {0, 0, 0, 0}};

// numpy's pairwise sum of f(0..224), evaluated by the 32 lanes of a warp; every lane returns the total
template <typename F>
__device__ __forceinline__ double np_sum225(F f) {
    const int lane = threadIdx.x & 31;
    const int base = (lane >> 3 & 1) * 112, j = lane & 7;
    double r = 0.0;
    if (lane < 16) {
        r = f(base + j);
        for (int g = 1; g < 14; ++g) r = __dadd_rn(r, f(base + 8 * g + j));
    }
    r = __dadd_rn(r, __shfl_down_sync(RSD_FULL, r, 1));       // lanes 0,2,4,6 (+8): r0+r1, r2+r3, ...
    r = __dadd_rn(r, __shfl_down_sync(RSD_FULL, r, 2));       // lanes 0,4 (+8)
    r = __dadd_rn(r, __shfl_down_sync(RSD_FULL, r, 4));       // lanes 0, 8: the two block sums
    const double b1 = __shfl_sync(RSD_FULL, r, 0);
    double b2 = __shfl_sync(RSD_FULL, r, 8);
    b2 = __dadd_rn(b2, f(224));
    return __dadd_rn(b1, b2);
}

// TF matrix of one sequence into v[225] (shared memory, one warp); get(i) returns the code of symbol i
template <typename G>
__device__ __forceinline__ void tf_build(double *v, int len, G get) {
    const int lane = threadIdx.x & 31;
    for (int e = lane; e < RSD_TF; e += 32) v[e] = 0.0;
    __syncwarp();
    for (int i = 0; i + 1 < len; ++i) {
        const int cur = get(i), nxt = get(i + 1);
        if (lane == 0) v[cur * 15 + nxt] = __dadd_rn(v[cur * 15 + nxt], 1.0);                    // IR:156
        if (nxt >= 4) {                                                                          // IR:176-184
            if (lane < 16) {
                const int k = lane >> 2, jj = lane & 3;
                v[k * 15 + jj] = __dadd_rn(v[k * 15 + jj], __dmul_rn(c_simW[cur][k], c_simW[nxt][jj]));
            }
        } else if (cur >= 4) {                                                                   // IR:171-174
            if (lane < 4) v[lane * 15 + nxt] = __dadd_rn(v[lane * 15 + nxt], c_simW[cur][lane]);
        }
        __syncwarp();
    }
}

// the representations of one query (one warp; v = 225 doubles of shared memory)
__device__ __forceinline__ void sim_query_build(double *v, const uint8_t *__restrict__ q, int len, SimQuery *out) {
    const int lane = threadIdx.x;
    tf_build(v, len, [&](int i) { return (int)q[i]; });
    const double total = np_sum225([&](int e) { return v[e]; });
    const double avg = __ddiv_rn(total, 225.0);                                                  // np.average
    for (int e = lane; e < RSD_TF; e += 32) { out->tf[e] = v[e]; out->tfc[e] = __dadd_rn(v[e], -avg); }
    const double sq = np_sum225([&](int e) { return __dmul_rn(v[e], v[e]); });
    const double csq = np_sum225([&](int e) { const double x = __dadd_rn(v[e], -avg); return __dmul_rn(x, x); });
    if (lane == 0) {
        out->tf_sq = sq; out->tfc_sq = csq;
        uint32_t mask = 0; double c[4] = {0.0, 0.0, 0.0, 0.0};
        for (int i = 0; i < len; ++i) {
            const int s = q[i];
            mask |= 1u << s;
            for (int k = 0; k < 4; ++k) c[k] = __dadd_rn(c[k], c_simW[s][k]);
        }
        out->mask = mask;
        for (int k = 0; k < 4; ++k) out->ms[k] = c[k];
        out->ms_sum = __dadd_rn(__dadd_rn(__dadd_rn(c[0], c[1]), c[2]), c[3]);
    }
}

__global__ void __launch_bounds__(32) k_sim_query(const uint8_t *__restrict__ q, int len, SimQuery *out) {
    __shared__ double v[RSD_TF];
    sim_query_build(v, q, len, out);
}

// one CTA per query of a batch: query q is codes[off[q] .. off[q+1]) -> out[q]
__global__ void __launch_bounds__(32) k_sim_query_batch(const uint8_t *__restrict__ codes, const int64_t *__restrict__ off, SimQuery *out) {
    __shared__ double v[RSD_TF];
    const int q = blockIdx.x;
    sim_query_build(v, codes + off[q], (int)(off[q + 1] - off[q]), out + q);
}

// One thread per stored record: set_* (IR:54-91) and multi_* (IR:110-145) measures.
__global__ void __launch_bounds__(256)
k_sim_small(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
            int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
            const SimQuery *__restrict__ Q, int method, double *__restrict__ scores) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int len = db_len[r];
    const int64_t st = db_start[r];
    uint32_t mask = 0; double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
    const bool multi = method >= RSD_SIM_MULTI_INTERSECTION;
    for (int i = 0; i < len; ++i) {
        const uint32_t s = pk_get(db_words, st, i, db_bits);
        mask |= 1u << s;
        if (multi) {
            c0 = __dadd_rn(c0, c_simW[s][0]); c1 = __dadd_rn(c1, c_simW[s][1]);
            c2 = __dadd_rn(c2, c_simW[s][2]); c3 = __dadd_rn(c3, c_simW[s][3]);
        }
    }
    double out;
    if (!multi) {
        const double inter = (double)__popc(mask & Q->mask);
        if (method == RSD_SIM_SET_INTERSECTION) out = inter;
        else if (method == RSD_SIM_SET_JACCARD) out = __ddiv_rn(inter, (double)__popc(mask | Q->mask));
        else out = __ddiv_rn(__dmul_rn(2.0, inter), (double)(__popc(mask) + __popc(Q->mask)));
    } else {
        // IR:110-116: sim = 0; sim += min(ca[k], cb[k]) for k = 0..3
        double sim = fmin(Q->ms[0], c0);
        sim = __dadd_rn(sim, fmin(Q->ms[1], c1));
        sim = __dadd_rn(sim, fmin(Q->ms[2], c2));
        sim = __dadd_rn(sim, fmin(Q->ms[3], c3));
        const double both = __dadd_rn(Q->ms_sum, __dadd_rn(__dadd_rn(__dadd_rn(c0, c1), c2), c3));
        if (method == RSD_SIM_MULTI_INTERSECTION) out = sim;
        else if (method == RSD_SIM_MULTI_JACCARD) out = __ddiv_rn(sim, __dadd_rn(both, -sim));
        else out = __ddiv_rn(__dmul_rn(2.0, sim), both);
    }
    scores[perm[r] - global_base] = out;
}

// One warp per stored record: vector measures on the TF matrices (IR:290-389); a = query, b = record.
__global__ void __launch_bounds__(128)
k_sim_tf(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
         int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
         const SimQuery *__restrict__ Q, int method, double *__restrict__ scores,
         const int *__restrict__ worklist, const int *__restrict__ worklist_n) {
    __shared__ double s_a[RSD_TF];
    __shared__ double s_v[4][RSD_TF];
    if (worklist) n_rec = *worklist_n;               // only the records the per-thread kernel deferred
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const double *qa = method == RSD_SIM_PEARSON ? Q->tfc : Q->tf;
    for (int e = threadIdx.x; e < RSD_TF; e += blockDim.x) s_a[e] = qa[e];
    __syncthreads();
    const double a_sq = method == RSD_SIM_PEARSON ? Q->tfc_sq : Q->tf_sq;
    double *v = s_v[wib];
    const int64_t n_warps = (int64_t)gridDim.x * 4;
    for (int64_t rr = (int64_t)blockIdx.x * 4 + wib; rr < n_rec; rr += n_warps) {
        const int64_t r = worklist ? (int64_t)worklist[rr] : rr;
        const int len = db_len[r];
        const int64_t st = db_start[r];
        tf_build(v, len, [&](int i) { return (int)pk_get(db_words, st, i, db_bits); });
        if (method == RSD_SIM_PEARSON) {
            const double avg = __ddiv_rn(np_sum225([&](int e) { return v[e]; }), 225.0);
            for (int e = lane; e < RSD_TF; e += 32) v[e] = __dadd_rn(v[e], -avg);
            __syncwarp();
        }
        double out;
        if (method == RSD_SIM_EUCLIDEAN || method == RSD_SIM_MANHATTAN) {
            const double d = method == RSD_SIM_EUCLIDEAN
                ? np_sum225([&](int e) { const double x = __dadd_rn(s_a[e], -v[e]); return __dmul_rn(x, x); })
                : np_sum225([&](int e) { return fabs(__dadd_rn(s_a[e], -v[e])); });
            out = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(d)));
        } else {
            const double num = np_sum225([&](int e) { return __dmul_rn(s_a[e], v[e]); });
            const double b_sq = np_sum225([&](int e) { return __dmul_rn(v[e], v[e]); });
            if (method == RSD_SIM_COSINE || method == RSD_SIM_PEARSON) out = __ddiv_rn(num, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
            else if (method == RSD_SIM_TANIMOTO) out = __ddiv_rn(num, __dadd_rn(__dadd_rn(a_sq, b_sq), -num));
            else out = __ddiv_rn(__dmul_rn(2.0, num), __dadd_rn(a_sq, b_sq));
        }
        if (lane == 0) scores[perm[r] - global_base] = out;
        __syncwarp();
    }
}

// numpy's pairwise sum of f(0..224) evaluated by ONE thread (fully unrolled, so f sees compile-time indices)
template <typename F>
__device__ __forceinline__ double np_sum225_thread(F f) {
    double blk[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        double r[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = f(112 * h + j);
#pragma unroll
        for (int g = 1; g < 14; ++g)
#pragma unroll
            for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], f(112 * h + 8 * g + j));
        blk[h] = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    }
    blk[1] = __dadd_rn(blk[1], f(224));
    return __dadd_rn(blk[0], blk[1]);
}

// One THREAD per stored record, for records made of A, G, C, U only (the bulk of a real database): their TF matrix
// is 16 bigram counts in the top-left 4 x 4 corner, every other entry is exactly 0, so the matrix never has to be
// materialised — the 225-term sums are unrolled with the 16 counts in registers.  Records that contain an
// ambiguity code (or are too long for 16-bit counters) are appended to a worklist for k_sim_tf.
__global__ void __launch_bounds__(128)
k_sim_tf_thread(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
                int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
                const SimQuery *__restrict__ Q, int method, double *__restrict__ scores,
                int *__restrict__ worklist, int *__restrict__ worklist_n) {
    __shared__ double s_a[RSD_TF];
    __shared__ uint16_t s_cnt[16][128];
    const double *qa = method == RSD_SIM_PEARSON ? Q->tfc : Q->tf;
    for (int e = threadIdx.x; e < RSD_TF; e += blockDim.x) s_a[e] = qa[e];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int tid = threadIdx.x;
    const int len = db_len[r];
    const int64_t st = db_start[r];
    bool plain = len <= 60000;
#pragma unroll
    for (int e = 0; e < 16; ++e) s_cnt[e][tid] = 0;
    if (plain && len > 0) {
        uint32_t prev = pk_get(db_words, st, 0, db_bits);
        plain = prev < 4u;
        for (int i = 1; i < len && plain; ++i) {
            const uint32_t cur = pk_get(db_words, st, i, db_bits);
            if (cur >= 4u) { plain = false; break; }
            s_cnt[prev * 4 + cur][tid] += 1;                                   // IR:156
            prev = cur;
        }
    }
    if (!plain) { worklist[atomicAdd(worklist_n, 1)] = (int)r; return; }
    double b[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) b[e] = (double)s_cnt[e][tid];
    auto bv = [&](int e) -> double {                                           // entry e of the record's TF matrix
        const int row = e / 15, col = e % 15;
        return (row < 4 && col < 4) ? b[row * 4 + col] : 0.0;
    };
    const double a_sq = method == RSD_SIM_PEARSON ? Q->tfc_sq : Q->tf_sq;
    double out;
    if (method == RSD_SIM_PEARSON) {
        // np.average of the count matrix: the counts are small integers, so their sum is exact whatever the order
        const double avg = __ddiv_rn((double)(len > 0 ? len - 1 : 0), 225.0);
        const double num = np_sum225_thread([&](int e) { return __dmul_rn(s_a[e], __dadd_rn(bv(e), -avg)); });
        const double b_sq = np_sum225_thread([&](int e) { const double x = __dadd_rn(bv(e), -avg); return __dmul_rn(x, x); });
        out = __ddiv_rn(num, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
    } else if (method == RSD_SIM_EUCLIDEAN) {
        const double d = np_sum225_thread([&](int e) { const double x = __dadd_rn(s_a[e], -bv(e)); return __dmul_rn(x, x); });
        out = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(d)));
    } else if (method == RSD_SIM_MANHATTAN) {
        const double d = np_sum225_thread([&](int e) { return fabs(__dadd_rn(s_a[e], -bv(e))); });
        out = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(d)));
    } else {
        const double num = np_sum225_thread([&](int e) { return __dmul_rn(s_a[e], bv(e)); });
        const double b_sq = np_sum225_thread([&](int e) { return __dmul_rn(bv(e), bv(e)); });
        if (method == RSD_SIM_COSINE) out = __ddiv_rn(num, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
        else if (method == RSD_SIM_TANIMOTO) out = __ddiv_rn(num, __dadd_rn(__dadd_rn(a_sq, b_sq), -num));
        else out = __ddiv_rn(__dmul_rn(2.0, num), __dadd_rn(a_sq, b_sq));
    }
    scores[perm[r] - global_base] = out;
}

// Candidates of one score range for the top-k fold (same key as the edit-distance search: score desc,
// global index asc).  NaN scores (the reference's 0/0) compare false and are never ranked.
__global__ void k_sim_filter(const double *__restrict__ scores, int64_t r0, int64_t n, int64_t global_base, TopkState tk) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double s = scores[r0 + r];
    const long long g = global_base + r0 + r;
    const double ts = tk.tau_s[0]; const long long ti = tk.tau_i[0];
    if (s > ts || (s == ts && g <= ti)) {
        const int slot = atomicAdd(&tk.cand_n[0], 1);
        if (slot < tk.cap) { tk.cand_s[slot] = s; tk.cand_i[slot] = g; }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// query batches
// ------------------------------------------------------------------------------------------------------------------
#define RSD_SIM_QB 64             // queries per batch at most (the host may take fewer: RSD_SIM_QBATCH, device memory)
#define RSD_SIM_QT 8              // query TF vectors in shared memory at a time (k_sim_tf_thread_batch)

// The set / multiset measures of one record (mask, c0..c3) against one query, as k_sim_small computes them.
__device__ __forceinline__ double sim_small_score(int method, uint32_t mask, double c0, double c1, double c2, double c3,
                                                  uint32_t qmask, const double *qms) {
    if (method < RSD_SIM_MULTI_INTERSECTION) {
        const double inter = (double)__popc(mask & qmask);
        if (method == RSD_SIM_SET_INTERSECTION) return inter;
        if (method == RSD_SIM_SET_JACCARD) return __ddiv_rn(inter, (double)__popc(mask | qmask));
        return __ddiv_rn(__dmul_rn(2.0, inter), (double)(__popc(mask) + __popc(qmask)));
    }
    double sim = fmin(qms[0], c0);
    sim = __dadd_rn(sim, fmin(qms[1], c1));
    sim = __dadd_rn(sim, fmin(qms[2], c2));
    sim = __dadd_rn(sim, fmin(qms[3], c3));
    const double both = __dadd_rn(qms[4], __dadd_rn(__dadd_rn(__dadd_rn(c0, c1), c2), c3));
    if (method == RSD_SIM_MULTI_INTERSECTION) return sim;
    if (method == RSD_SIM_MULTI_JACCARD) return __ddiv_rn(sim, __dadd_rn(both, -sim));
    return __ddiv_rn(__dmul_rn(2.0, sim), both);
}

// One thread per stored record, nq queries: set_* and multi_* measures.
__global__ void __launch_bounds__(256)
k_sim_small_batch(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
                  int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
                  const SimQuery *__restrict__ Q, int nq, int method, double *__restrict__ scores, int64_t stride) {
    __shared__ uint32_t s_mask[RSD_SIM_QB];
    __shared__ double s_ms[RSD_SIM_QB][5];                    // ms[0..3], ms_sum
    for (int i = threadIdx.x; i < nq; i += blockDim.x) {
        s_mask[i] = Q[i].mask;
        for (int j = 0; j < 4; ++j) s_ms[i][j] = Q[i].ms[j];
        s_ms[i][4] = Q[i].ms_sum;
    }
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int len = db_len[r];
    const int64_t st = db_start[r];
    uint32_t mask = 0; double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
    const bool multi = method >= RSD_SIM_MULTI_INTERSECTION;
    for (int i = 0; i < len; ++i) {
        const uint32_t s = pk_get(db_words, st, i, db_bits);
        mask |= 1u << s;
        if (multi) {
            c0 = __dadd_rn(c0, c_simW[s][0]); c1 = __dadd_rn(c1, c_simW[s][1]);
            c2 = __dadd_rn(c2, c_simW[s][2]); c3 = __dadd_rn(c3, c_simW[s][3]);
        }
    }
    double *out = scores + (perm[r] - global_base);
    for (int q = 0; q < nq; ++q) out[(size_t)q * stride] = sim_small_score(method, mask, c0, c1, c2, c3, s_mask[q], s_ms[q]);
}

// One THREAD per A/G/C/U record, nq queries (k_sim_tf_thread for a batch).  The record's 16 bigram counts stay in
// registers and its own terms are computed once: b_sq for cosine / Tanimoto / Dice, the average and the centred b_sq for
// Pearson.  Per query only the sums that involve it run: num, or the Euclidean / Manhattan distance sum.
//
// num of cosine / Tanimoto / Dice adds only the 16 corner products: the other 209 terms are query TF entry * 0.  Query TF
// entries are sums of counts and products of the non-negative weights c_simW, so >= 0 and finite, and each of those
// terms is +0; every partial sum of the pairwise order is then >= +0, and adding +0 to it changes nothing.  The 16
// corner products keep their accumulator and their place in the order (np_sum225_thread with a compile-time test).
// Pearson's query vector is centred (negative entries) and the Euclidean / Manhattan terms are not zero: full sums.
__global__ void __launch_bounds__(128)
k_sim_tf_thread_batch(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
                      int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
                      const SimQuery *__restrict__ Q, int nq, int method, double *__restrict__ scores, int64_t stride,
                      int *__restrict__ worklist, int *__restrict__ worklist_n) {
    __shared__ double s_a[RSD_SIM_QT][RSD_TF];
    __shared__ double s_asq[RSD_SIM_QT];
    __shared__ uint16_t s_cnt[16][128];
    const int tid = threadIdx.x;
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + tid;
    const bool pearson = method == RSD_SIM_PEARSON;
    bool plain = false;
    int len = 0;
    if (r < n_rec) {
        len = db_len[r];
        const int64_t st = db_start[r];
        plain = len <= 60000;
#pragma unroll
        for (int e = 0; e < 16; ++e) s_cnt[e][tid] = 0;
        if (plain && len > 0) {
            uint32_t prev = pk_get(db_words, st, 0, db_bits);
            plain = prev < 4u;
            for (int i = 1; i < len && plain; ++i) {
                const uint32_t cur = pk_get(db_words, st, i, db_bits);
                if (cur >= 4u) { plain = false; break; }
                s_cnt[prev * 4 + cur][tid] += 1;                               // IR:156
                prev = cur;
            }
        }
        if (!plain) worklist[atomicAdd(worklist_n, 1)] = (int)r;
    }
    double b[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) b[e] = plain ? (double)s_cnt[e][tid] : 0.0;
    auto corner = [](int e) { return e / 15 < 4 && e % 15 < 4; };
    auto bv = [&](int e) -> double { return corner(e) ? b[e / 15 * 4 + e % 15] : 0.0; };
    double avg = 0.0, b_sq = 0.0;
    if (plain) {
        if (pearson) {
            avg = __ddiv_rn((double)(len > 0 ? len - 1 : 0), 225.0);                  // the counts sum exactly (k_sim_tf_thread)
            b_sq = np_sum225_thread([&](int e) { const double x = __dadd_rn(bv(e), -avg); return __dmul_rn(x, x); });
        } else if (method == RSD_SIM_COSINE || method == RSD_SIM_TANIMOTO || method == RSD_SIM_DICE) {
            b_sq = np_sum225_thread([&](int e) { return __dmul_rn(bv(e), bv(e)); });
        }
    }
    double *out = plain ? scores + (perm[r] - global_base) : nullptr;
    for (int q0 = 0; q0 < nq; q0 += RSD_SIM_QT) {
        const int nt = min(RSD_SIM_QT, nq - q0);
        __syncthreads();                                                       // the previous tile is no longer read
        for (int i = tid; i < nt * RSD_TF; i += blockDim.x) {
            const SimQuery &qq = Q[q0 + i / RSD_TF];
            s_a[i / RSD_TF][i % RSD_TF] = pearson ? qq.tfc[i % RSD_TF] : qq.tf[i % RSD_TF];
        }
        if (tid < nt) s_asq[tid] = pearson ? Q[q0 + tid].tfc_sq : Q[q0 + tid].tf_sq;
        __syncthreads();
        if (!plain) continue;
        for (int t = 0; t < nt; ++t) {
            const double *a = s_a[t];
            const double a_sq = s_asq[t];
            double v;
            if (pearson) {
                const double num = np_sum225_thread([&](int e) { return __dmul_rn(a[e], __dadd_rn(bv(e), -avg)); });
                v = __ddiv_rn(num, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
            } else if (method == RSD_SIM_EUCLIDEAN) {
                const double d = np_sum225_thread([&](int e) { const double x = __dadd_rn(a[e], -bv(e)); return __dmul_rn(x, x); });
                v = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(d)));
            } else if (method == RSD_SIM_MANHATTAN) {
                const double d = np_sum225_thread([&](int e) { return fabs(__dadd_rn(a[e], -bv(e))); });
                v = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(d)));
            } else {
                const double num = np_sum225_thread([&](int e) { return corner(e) ? __dmul_rn(a[e], bv(e)) : 0.0; });
                if (method == RSD_SIM_COSINE) v = __ddiv_rn(num, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
                else if (method == RSD_SIM_TANIMOTO) v = __ddiv_rn(num, __dadd_rn(__dadd_rn(a_sq, b_sq), -num));
                else v = __ddiv_rn(__dmul_rn(2.0, num), __dadd_rn(a_sq, b_sq));
            }
            out[(size_t)(q0 + t) * stride] = v;
        }
    }
}

// One warp per worklist record, nq queries (k_sim_tf for a batch): the record's TF matrix (centred for Pearson) and
// its own sums once in shared memory, then the per-query sums with the query vectors read from SimQuery; the final
// divisions run one query per lane.
__global__ void __launch_bounds__(128)
k_sim_tf_batch(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
               int db_bits, const int64_t *__restrict__ perm, int64_t global_base, const SimQuery *__restrict__ Q, int nq, int method,
               double *__restrict__ scores, int64_t stride, const int *__restrict__ worklist, const int *__restrict__ worklist_n) {
    __shared__ double s_v[4][RSD_TF];
    __shared__ double s_sum[4][RSD_SIM_QB];                   // per query: num, or the distance sum
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const bool pearson = method == RSD_SIM_PEARSON, dist = method == RSD_SIM_EUCLIDEAN || method == RSD_SIM_MANHATTAN;
    double *v = s_v[wib], *sum = s_sum[wib];
    // the worklist length is loaded again per record instead of being held across the division calls below (ptxas
    // would keep it on the stack)
    for (int rr = blockIdx.x * 4 + wib; rr < __ldcg(worklist_n); rr += gridDim.x * 4) {
        const int64_t r = worklist[rr];
        const int len = db_len[r];
        const int64_t st = db_start[r];
        tf_build(v, len, [&](int i) { return (int)pk_get(db_words, st, i, db_bits); });
        if (pearson) {
            const double avg = __ddiv_rn(np_sum225([&](int e) { return v[e]; }), 225.0);
            for (int e = lane; e < RSD_TF; e += 32) v[e] = __dadd_rn(v[e], -avg);
            __syncwarp();
        }
        const double b_sq = dist ? 0.0 : np_sum225([&](int e) { return __dmul_rn(v[e], v[e]); });
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
            const double *a = pearson ? Q[q].tfc : Q[q].tf;
            const double s = method == RSD_SIM_EUCLIDEAN ? np_sum225([&](int e) { const double x = __dadd_rn(a[e], -v[e]); return __dmul_rn(x, x); })
                           : method == RSD_SIM_MANHATTAN ? np_sum225([&](int e) { return fabs(__dadd_rn(a[e], -v[e])); })
                           : np_sum225([&](int e) { return __dmul_rn(a[e], v[e]); });
            if (lane == 0) sum[q] = s;
        }
        __syncwarp();
        double *out = scores + (perm[r] - global_base);
        for (int q = lane; q < nq; q += 32) {
            const double s = sum[q], a_sq = pearson ? Q[q].tfc_sq : Q[q].tf_sq;
            double o;
            if (dist) o = __ddiv_rn(1.0, __dadd_rn(1.0, __dsqrt_rn(s)));
            else if (method == RSD_SIM_COSINE || pearson) o = __ddiv_rn(s, __dsqrt_rn(__dmul_rn(a_sq, b_sq)));
            else if (method == RSD_SIM_TANIMOTO) o = __ddiv_rn(s, __dadd_rn(__dadd_rn(a_sq, b_sq), -s));
            else o = __ddiv_rn(__dmul_rn(2.0, s), __dadd_rn(a_sq, b_sq));
            out[(size_t)q * stride] = o;
        }
        __syncwarp();
    }
}

// k_sim_filter for a batch: query blockIdx.y, its scores at scores + q * stride, its candidates at [q][cap]
__global__ void k_sim_filter_batch(const double *__restrict__ scores, int64_t stride, int64_t r0, int64_t n, int64_t global_base, TopkState tk) {
    const int q = blockIdx.y;
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double s = scores[(size_t)q * stride + r0 + r];
    const long long g = global_base + r0 + r;
    const double ts = tk.tau_s[q]; const long long ti = tk.tau_i[q];
    if (s > ts || (s == ts && g <= ti)) {
        const int slot = atomicAdd(&tk.cand_n[q], 1);
        if (slot < tk.cap) { tk.cand_s[(size_t)q * tk.cap + slot] = s; tk.cand_i[(size_t)q * tk.cap + slot] = g; }
    }
}
