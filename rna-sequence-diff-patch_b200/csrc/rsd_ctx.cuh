// rsd_ctx.cuh — the context object behind the opaque rsd_ctx handle (host side).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <unistd.h>
#include <algorithm>
#include <new>
#include <vector>

#include "k_plan.cuh"

int rsd_fail(int code, const char *fmt, ...);

#define RSD_MAX_CHUNKS 16

#define RSD_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            cudaGetLastError();                                                                     \
            return rsd_fail(e__ == cudaErrorMemoryAllocation ? RSD_ENOMEM : RSD_ECUDA, "%s: %s (%s:%d)", #call, \
                            cudaGetErrorString(e__), __FILE__, __LINE__);                          \
        }                                                                                           \
    } while (0)

#define RSD_OK_OR_RETURN(call)            \
    do {                                  \
        int rc__ = (call);                \
        if (rc__ != 0) return rc__;       \
    } while (0)

// grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap && p) return 0;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            e = cudaMalloc(&p, bytes + 256);
            want = bytes + 256;
            if (e != cudaSuccess) { cudaGetLastError(); p = nullptr; return rsd_fail(4 /*RSD_ENOMEM*/, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e)); }
        }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct SeqBufs { DevBuf words, start, len; void release() { words.release(); start.release(); len.release(); } };

struct ModeInfo {
    int mode;       // RSD_MODE_*
    int k;          // scale_log2 (int modes)
    IntCosts ic;
    F64Costs fc;
    bool dyadic, i16_ok, i32_ok;
};

// Plan arrays + hand-off scratch of one batch in flight; the chunks of a host call use one slot each so their
// kernels may overlap, everything else uses slot 0.
struct PlanSlot {
    DevBuf scratch, pair_bin, bins, groups, trace;
    bool dirty = true;           // bin counters need a memset before the next plan
    PlanView pv;
    ModeInfo mi;
    int64_t n_pairs = 0, max_n = 0;
    void release() { scratch.release(); pair_bin.release(); bins.release(); groups.release(); trace.release(); dirty = true; }
};

// Hits of a range search on the host, query by query in the order the search saw the queries: cnt[q] hits each,
// concatenated in idx / dist, every query's hits by global index ascending.
struct RangeOut {
    double max_dist = 0;
    std::vector<int64_t> cnt, idx;
    std::vector<double> dist;
};

struct rsd_ctx {
    int device = 0;
    bool inited = false;
    pid_t pid = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr, copy_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_sync = nullptr, ev_chunk[RSD_MAX_CHUNKS] = {}, ev_t0[RSD_MAX_CHUNKS] = {}, ev_t1[RSD_MAX_CHUNKS] = {}, ev_done[RSD_MAX_CHUNKS] = {};
    cudaEvent_t ev_begin = nullptr, ev_len = nullptr, ev_plans = nullptr, ev_tab = nullptr;
    double last_ms_override = 0.0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing = false, timed = false;
    int64_t launches = 0;

    bool have_costs = false;
    double ins = 0, del = 0, sub[15][15];
    IntCosts *d_ic = nullptr;
    F64Costs *d_fc = nullptr;

    SeqBufs bufA, bufB, bufX, bufQ;
    DevBuf out_f64;
    // host batch calls with a canonical layout / raw codes: block-offset tables (pinned staging + device copy),
    // raw code bytes and symbol offsets per side
    void *h_stage = nullptr; size_t h_stage_cap = 0;
    DevBuf d_stage, raw_codes[2], sym_start[2];
    PlanSlot slots[RSD_MAX_CHUNKS];
    DevBuf mat_vals, mat_mask, mat_ab;
    // script / patch
    int64_t dirs_budget_words = 0, dirs_budget_out_bytes = 0;     // chunk budget of the script path, measured once
    DevBuf dirs, s_op, s_oi, s_oj, s_nops, s_ok, s_tmp, p_out, p_len, p_err, misc;
    // long pairs (rsd_long.inl): one pool carved per batch, job tables
    DevBuf long_pool, long_jobs;
    void *long_hstage = nullptr; size_t long_hstage_cap = 0;     // pinned staging of rsd_long_pairs
    size_t long_bound_hw = 0;              // head of long_pool that has only ever held tagged boundary words
    float long_fwd_ms = 0.f;
    size_t long_budget = 0;                // memory budget of the long-pair planner (measured once, see rsd_long.inl)
    unsigned long_gen = 0;                 // generation tag of the boundary words (k_long2.cuh)
    // database shard
    SeqBufs db;
    int64_t db_n = 0, db_base = 0, db_nwords = 0, db_maxlen = 0;
    int db_bits = 0;
    uint32_t db_symmask = 0;
    int64_t db_tier_end[16] = {};          // stored records [0, db_tier_end[t]) use only the t+1 most common symbols
    uint32_t db_tier_mask[16] = {};        // ... whose set is db_tier_mask[t]
    bool db_loaded = false;
    DevBuf db_dist, db_topi, db_tops, db_aux, db_perm;
    int search_per_sm = 0, search_per_sm_nq = -1, search_per_sm_qrows = -1;      // occupancy of the search kernel, asked once per shape
    bool search_per_sm_range = false;                                             // ... and epilogue
    // range search: hit append buffer of one query batch (keys and distances, each two halves for the sort), the
    // 64-bit hit counter + per-query offsets, the sort's scratch
    DevBuf rng_keys, rng_dist, rng_n, rng_tmp;
    DevBuf sim_q, sim_scores, sim_aux, sim_codes, sim_work;
    DevBuf sim_off, sim_top;               // rsd_db_similarity_batch: query offsets, [2][Q][k] top-k lists
    // idf / tf-idf vectors: idf_dev = idf[225] then the df partial sums [225]; idf_exp = IdfExp; idf_work = one chunk of
    // presence sets, then the inverse of db_perm, while the table is built
    DevBuf idf_dev, idf_exp, idf_work;
    bool idf_ready = false;                // idf_df / idf_tab / idf_dev hold the loaded database's table
    bool idf_nonneg = true;                // every idf entry is finite and >= +0
    double idf_df[225], idf_tab[225];

    int ensure_device();
    int classify(uint32_t symmask, int64_t max_m, int64_t max_n, int bits, int force_mode, ModeInfo &mi) const;
    int upload_costs(const ModeInfo &mi, cudaStream_t st);
    int upload_seqs(SeqBufs &sb, const uint32_t *words, const int64_t *start, const int32_t *len, int64_t n,
                    int64_t n_words, cudaStream_t st);
    int make_plan(PlanSlot &sl, const int32_t *d_alen, const int32_t *d_blen, int64_t n_pairs, int C, int allow_twin, double *d_out,
                  cudaStream_t st, PlanView &pv, int64_t max_m, int64_t max_n, int band);
    int distance_plan(PlanSlot &sl, const int32_t *a_len, const int32_t *b_len, int64_t n_pairs, int64_t max_m, int64_t max_n, int bits,
                      uint32_t symmask, int force_mode, bool load_costs, double *d_out, int *mode_out, cudaStream_t st);
    int distance_launch(PlanSlot &sl, const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, const uint32_t *b_words,
                        const int64_t *b_start, const int32_t *b_len, int64_t max_m, int bits, double *d_out, cudaStream_t st,
                        cudaEvent_t t0, cudaEvent_t t1);
    int distance_dev(const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, const uint32_t *b_words,
                     const int64_t *b_start, const int32_t *b_len, int64_t n_pairs, int64_t max_m, int64_t max_n,
                     int bits, uint32_t symmask, int force_mode, double *d_out, int *mode_out, cudaStream_t st,
                     cudaEvent_t t0, cudaEvent_t t1);
    int fast_prefix(uint32_t q_symmask, int64_t max_qlen, int bits, int force_mode, ModeInfo &mi_fast, uint32_t lut[4], int64_t &n_fast) const;
    int search_dev(const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len, int64_t n_queries,
                   int64_t max_qlen, int bits, uint32_t q_symmask, int k, int force_mode, int64_t *top_idx,
                   double *top_score, double *all_scores_dev, int *mode_out, cudaStream_t st, RangeOut *ro, bool record_start);
    int64_t range_cap() const { return (int64_t)(std::min(rng_keys.cap, rng_dist.cap) / 16); }     // hits the buffer holds
    int range_reserve(int64_t hits, int qb);
    int range_collect(int nq, int qb, RangeOut &ro, bool &rerun, cudaStream_t st);
    int script_pipeline(const int32_t *a_len, const int32_t *b_len, int64_t n_pairs, int bits, uint32_t symmask,
                        int force_mode, int64_t max_ops, bool with_x, uint8_t *op, int32_t *oi, int32_t *oj,
                        int32_t *n_ops, double *dist, uint8_t *ok, int *mode_out);
    void free_all() {
        bufA.release(); bufB.release(); bufX.release(); bufQ.release(); db.release();
        for (PlanSlot &s : slots) s.release();
        DevBuf *all[] = {&out_f64, &mat_vals, &mat_mask, &mat_ab,
                         &long_pool, &long_jobs, &dirs, &s_op, &s_oi, &s_oj, &s_nops, &s_ok, &s_tmp, &p_out, &p_len, &p_err, &misc,
                         &db_dist, &db_topi, &db_tops, &db_aux, &db_perm, &rng_keys, &rng_dist, &rng_n, &rng_tmp, &sim_q, &sim_scores, &sim_aux, &sim_codes, &sim_work, &sim_off, &sim_top,
                         &idf_dev, &idf_exp, &idf_work};
        for (DevBuf *b : all) b->release();
        d_stage.release(); for (int s = 0; s < 2; ++s) { raw_codes[s].release(); sym_start[s].release(); }
        if (h_stage) { cudaFreeHost(h_stage); h_stage = nullptr; h_stage_cap = 0; }
        if (long_hstage) { cudaFreeHost(long_hstage); long_hstage = nullptr; long_hstage_cap = 0; }
    }
};
