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
//
// idf and tf-idf vectors (search_collection with vector_type 'idf' / 'tf-idf', IR:189-225 and IR:458-465): the batch
// kernels above take the vector type VT as a template argument; the query and record matrices are then the idf vector
// (idf[p] at every distinct literal bigram p of the sequence) or the tf-idf product tf . idf, and everything after
// that -- centring, norms, the measures, the top-k -- is the 'tf' code unchanged.  idf[p] = log10(N / df[p]) comes
// from the collection's document-frequency table, built once per loaded database:
//   k_idf_inv    collection index -> stored record (inverse of db_perm)
//   k_idf_pres   literal-bigram presence sets of a chunk of records, in collection order
//   k_idf_chain  the 225 df sums over that chunk, each one serial fp64 chain in collection order
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

#define RSD_VEC_TF 0              // the 'tf' vectors; RSD_VEC_IDF / RSD_VEC_TFIDF are declared in include/rsd.h

// One warp turns the TF matrix v of a sequence (tf_build) into its idf (VT == RSD_VEC_IDF) or tf-idf vector
// (RSD_VEC_TFIDF).  IR:189-216: the idf vector is idf[p] at every distinct literal bigram p of the sequence and 0
// elsewhere.  IR:219-223: tf-idf = np.dot(tf, idf), which numpy's BLAS evaluates per element as a fused multiply-add
// chain over k = 0..14 ascending from +0.0.  w = 225 doubles and pres = 8 words of shared memory for this warp.
template <int VT, typename G>
__device__ __forceinline__ void vec_from_tf(double *v, double *w, uint32_t *pres, int len, G get, const double *__restrict__ idf) {
    const int lane = threadIdx.x & 31;
    if (lane < 8) pres[lane] = 0u;
    __syncwarp();
    for (int i = lane; i + 1 < len; i += 32) {
        const int e = get(i) * 15 + get(i + 1);
        atomicOr(&pres[e >> 5], 1u << (e & 31));
    }
    __syncwarp();
    double *iv = VT == RSD_VEC_IDF ? v : w;
    for (int e = lane; e < RSD_TF; e += 32) iv[e] = (pres[e >> 5] >> (e & 31) & 1u) ? idf[e] : 0.0;
    __syncwarp();
    if constexpr (VT == RSD_VEC_TFIDF) {
        double o[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int e = lane + 32 * t, i = e / 15, j = e % 15;
            double acc = 0.0;
            if (e < RSD_TF)
                for (int k = 0; k < 15; ++k) acc = __fma_rn(v[i * 15 + k], w[k * 15 + j], acc);
            o[t] = acc;
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 8; ++t) if (lane + 32 * t < RSD_TF) v[lane + 32 * t] = o[t];
        __syncwarp();
    }
}

// the representations of one query (one warp; v = 225 doubles of shared memory).  VT != RSD_VEC_TF: tf / tfc / tf_sq /
// tfc_sq hold the query's idf or tf-idf vector instead of its TF matrix (vec_from_tf; w, pres, idf as there).
template <int VT = RSD_VEC_TF>
__device__ __forceinline__ void sim_query_build(double *v, const uint8_t *__restrict__ q, int len, SimQuery *out,
                                                double *w = nullptr, uint32_t *pres = nullptr, const double *__restrict__ idf = nullptr) {
    const int lane = threadIdx.x;
    tf_build(v, len, [&](int i) { return (int)q[i]; });
    if constexpr (VT != RSD_VEC_TF) vec_from_tf<VT>(v, w, pres, len, [&](int i) { return (int)q[i]; }, idf);
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

// one CTA per query of a batch: query q is codes[off[q] .. off[q+1]) -> out[q]; vector type VT (idf: the table, VT != 0)
template <int VT>
__global__ void __launch_bounds__(32) k_sim_query_batch(const uint8_t *__restrict__ codes, const int64_t *__restrict__ off, SimQuery *out,
                                                        const double *__restrict__ idf) {
    __shared__ double v[RSD_TF];
    __shared__ double w[VT == RSD_VEC_TFIDF ? RSD_TF : 1];
    __shared__ uint32_t pres[8];
    const int q = blockIdx.x;
    sim_query_build<VT>(v, codes + off[q], (int)(off[q + 1] - off[q]), out + q, w, pres, idf);
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
//
// VT = RSD_VEC_IDF / RSD_VEC_TFIDF (idf = the 225-entry table): the record's idf vector is idf[p] at its literal bigrams,
// all in the corner.  Its tf-idf entry (i, j) of the corner is the fused chain sum_k tf[i][k] * idf_vec[k][j] over
// k = 0..3: the terms k >= 4 are fma(0, x, acc) with x finite and >= +0, and every acc of the chain is >= +0, so each
// leaves acc unchanged; every entry outside the corner is a chain of such terms from +0.0, so +0.  Two things of the
// 'tf' case do not carry over: np.average of the vector is a real pairwise sum (np_sum225_thread), and the query
// entries are >= +0 only while every idf entry is (a_nonneg, checked on the host when the table is built); otherwise
// num of cosine / Tanimoto / Dice is the full sum.
template <int VT>
__global__ void __launch_bounds__(128)
k_sim_tf_thread_batch(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
                      int64_t n_rec, int db_bits, const int64_t *__restrict__ perm, int64_t global_base,
                      const SimQuery *__restrict__ Q, int nq, int method, double *__restrict__ scores, int64_t stride,
                      int *__restrict__ worklist, int *__restrict__ worklist_n, const double *__restrict__ idf, int a_nonneg) {
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
    if constexpr (VT == RSD_VEC_TF) {
#pragma unroll
        for (int e = 0; e < 16; ++e) b[e] = plain ? (double)s_cnt[e][tid] : 0.0;
    } else {
        double iv[16];                                                         // the record's idf vector (corner)
#pragma unroll
        for (int e = 0; e < 16; ++e) iv[e] = plain && s_cnt[e][tid] ? __ldg(&idf[e / 4 * 15 + e % 4]) : 0.0;
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            if constexpr (VT == RSD_VEC_IDF) b[e] = iv[e];
            else {
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < 4; ++k) acc = __fma_rn((double)s_cnt[e / 4 * 4 + k][tid], iv[k * 4 + e % 4], acc);
                b[e] = plain ? acc : 0.0;
            }
        }
    }
    auto corner = [](int e) { return e / 15 < 4 && e % 15 < 4; };
    auto bv = [&](int e) -> double { return corner(e) ? b[e / 15 * 4 + e % 15] : 0.0; };
    const bool skip_zero = VT == RSD_VEC_TF || a_nonneg;                      // num: the 209 non-corner terms are +0
    double avg = 0.0, b_sq = 0.0;
    if (plain) {
        if (pearson) {
            if constexpr (VT == RSD_VEC_TF) avg = __ddiv_rn((double)(len > 0 ? len - 1 : 0), 225.0);   // the counts sum exactly (k_sim_tf_thread)
            else avg = __ddiv_rn(np_sum225_thread(bv), 225.0);
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
                const double num = np_sum225_thread([&](int e) { return corner(e) || !skip_zero ? __dmul_rn(a[e], bv(e)) : 0.0; });
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
// divisions run one query per lane.  VT != RSD_VEC_TF: the record's idf / tf-idf vector instead (vec_from_tf).
template <int VT>
__global__ void __launch_bounds__(128)
k_sim_tf_batch(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len,
               int db_bits, const int64_t *__restrict__ perm, int64_t global_base, const SimQuery *__restrict__ Q, int nq, int method,
               double *__restrict__ scores, int64_t stride, const int *__restrict__ worklist, const int *__restrict__ worklist_n,
               const double *__restrict__ idf) {
    __shared__ double s_v[4][RSD_TF];
    __shared__ double s_w[4][VT == RSD_VEC_TFIDF ? RSD_TF : 1];
    __shared__ uint32_t s_pres[4][8];
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
        if constexpr (VT != RSD_VEC_TF) vec_from_tf<VT>(v, s_w[wib], s_pres[wib], len, [&](int i) { return (int)pk_get(db_words, st, i, db_bits); }, idf);
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

// ------------------------------------------------------------------------------------------------------------------
// document-frequency table of the idf vectors (IR:189-216)
// ------------------------------------------------------------------------------------------------------------------
// compare_pair_to_seq(p, doc) (IR:225-252) depends only on the set of literal bigrams of the document: it is the
// largest product wa * wb over the expansions (a, b) of p (possibilities(p[0]) x possibilities(p[1]), IR:255-287, at
// most 8 x 8; p itself is the expansion of product 1) whose bigram a + b occurs, and 0 when none occurs.  The host
// lists every pair's expansions by product, largest first (IdfExp), so the value is the product of the first one present.
#define RSD_IDF_EXP 64
#define RSD_IDF_T 160             // records per tile of k_idf_chain (one per worker thread)

struct IdfExp {
    int n[RSD_TF];                        // expansions of pair p
    uint8_t e[RSD_TF][RSD_IDF_EXP];       // their bigrams (a * 15 + b)
    double w[RSD_TF][RSD_IDF_EXP];        // their products wa * wb, non-increasing
};

// inv[perm[r] - global_base] = r: the stored record of every collection index of the shard
__global__ void k_idf_inv(const int64_t *__restrict__ perm, int64_t global_base, int64_t n, int64_t *__restrict__ inv) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) inv[perm[r] - global_base] = r;
}

// The literal-bigram presence sets (225 bits in 8 words) of the records i0 .. i0 + n - 1 of the shard, in collection
// order: pres[8 * i + word].  One thread per record.
__global__ void __launch_bounds__(256)
k_idf_pres(const uint32_t *__restrict__ db_words, const int64_t *__restrict__ db_start, const int32_t *__restrict__ db_len, int db_bits,
           const int64_t *__restrict__ inv, int64_t i0, int64_t n, uint32_t *__restrict__ pres) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t r = inv[i0 + i];
    const int len = db_len[r];
    const int64_t st = db_start[r];
    uint32_t m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (len > 0) {
        uint32_t prev = pk_get(db_words, st, 0, db_bits);
        for (int j = 1; j < len; ++j) {
            const uint32_t cur = pk_get(db_words, st, j, db_bits);
            const uint32_t e = prev * 15u + cur;
#pragma unroll
            for (int w = 0; w < 8; ++w) m[w] |= (e >> 5 == (uint32_t)w) ? 1u << (e & 31u) : 0u;      // registers, no local array
            prev = cur;
        }
    }
    uint4 *o = reinterpret_cast<uint4 *>(pres + 8 * i);
    o[0] = make_uint4(m[0], m[1], m[2], m[3]);
    o[1] = make_uint4(m[4], m[5], m[6], m[7]);
}

// df[p] += compare_pair_to_seq(p, record i) for i = 0 .. n - 1 in that order (IR:205-212: `df = df + v` over
// collection.find({})).  Each of the 225 sums is one dependent chain of __dadd_rn -- the order decides the bits, so no
// tree or atomic reduction.  CTA = row a of the table (pairs a * 15 + j, j = 0..14), 32 + RSD_IDF_T threads: lane j of
// warp 0 runs the chain of pair j over one tile of values while the other RSD_IDF_T threads compute the next tile's
// values (one record each, all 15 pairs) into the other shared buffer.  df carries the sums from launch to launch.
__global__ void __launch_bounds__(32 + RSD_IDF_T)
k_idf_chain(const uint32_t *__restrict__ pres, int64_t n, const IdfExp *__restrict__ X, double *__restrict__ df) {
    constexpr int TP = RSD_IDF_T + 1;                         // row stride: the 15 chain lanes read 15 different banks
    __shared__ double s_val[2][15 * TP];
    __shared__ double s_w[15][RSD_IDF_EXP];
    __shared__ uint8_t s_e[15][RSD_IDF_EXP];
    __shared__ int s_n[15];
    const int a = blockIdx.x, tid = threadIdx.x;
    for (int x = tid; x < 15 * RSD_IDF_EXP; x += blockDim.x) {
        const int j = x / RSD_IDF_EXP, m = x % RSD_IDF_EXP;
        s_w[j][m] = X->w[a * 15 + j][m]; s_e[j][m] = X->e[a * 15 + j][m];
    }
    if (tid < 15) s_n[tid] = X->n[a * 15 + tid];
    double acc = tid < 15 ? df[a * 15 + tid] : 0.0;
    __syncthreads();
    const int64_t n_tiles = (n + RSD_IDF_T - 1) / RSD_IDF_T;
    for (int64_t t = 0; t <= n_tiles; ++t) {
        if (tid < 32) {
            if (t > 0 && tid < 15) {                            // the chains over tile t - 1
                const double *val = s_val[(t - 1) & 1] + tid * TP;
                const int cnt = (int)min((int64_t)RSD_IDF_T, n - (t - 1) * RSD_IDF_T);
#pragma unroll 8
                for (int x = 0; x < cnt; ++x) acc = __dadd_rn(acc, val[x]);
            }
        } else if (t < n_tiles) {                               // the values of tile t
            const int x = tid - 32;
            const int64_t i = t * RSD_IDF_T + x;
            if (i < n) {
                const uint4 p0 = reinterpret_cast<const uint4 *>(pres + 8 * i)[0], p1 = reinterpret_cast<const uint4 *>(pres + 8 * i)[1];
                double *val = s_val[t & 1] + x;
                for (int j = 0; j < 15; ++j) {
                    double v = 0.0;
                    for (int m = 0; m < s_n[j]; ++m) {
                        const int e = s_e[j][m], q = e >> 5;
                        const uint4 h = q < 4 ? p0 : p1;           // selects, so the set stays in registers
                        const uint32_t word = (q & 3) == 0 ? h.x : (q & 3) == 1 ? h.y : (q & 3) == 2 ? h.z : h.w;
                        if (word >> (e & 31) & 1u) { v = s_w[j][m]; break; }
                    }
                    val[j * TP] = v;
                }
            }
        }
        __syncthreads();
    }
    if (tid < 15) df[a * 15 + tid] = acc;
}
