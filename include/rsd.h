/*
 * rsd.h — C ABI of librsd.so: the B200-native (sm_100a) weighted Wagner–Fischer engine.
 *
 * This is the drop-in boundary for the hot path of plsakr/rna-sequence-diff-patch.  The reference
 * has no FFI; its boundary is the Python module surface of StringEditDistance.py / IRMethods.py
 * (SURVEY 8b).  Every entry point below names the reference interface it replaces (file:line under
 * /root/reference; SED = StringEditDistance.py, IR = IRMethods.py).  The Python mirror of those
 * modules (rna-sequence-diff-patch_b200/dropin/) binds exactly these symbols with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns an int status (RSD_OK == 0) and leaves
 *     a message for rsd_last_error() (thread-local) otherwise.
 *   - buffers are caller-owned and caller-sized.  "host" entry points take host pointers and do
 *     the H2D/D2H copies themselves (pinned memory makes them fast, pageable works);
 *     "*_dev" entry points take device pointers + a CUDA stream handle (void*) and never
 *     synchronise the device.
 *   - the CUDA context is created lazily on the first call in the calling process (the reference's
 *     callers fork: IR:411,489,512), never at load time; a handle must not cross fork().
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with RSD_ENODEV.
 *
 * Symbols and packing
 *   - symbol code = index in "AGCUYRWSKMDVHBN" (IR:13, the row/column order of costs.json);
 *     code 15 = spare symbol that only matches itself (SED:79-81 never looks such a pair up).
 *   - packed batch ("pk"): little-endian u32 words; bits==4 -> 8 symbols per word, symbol k of a
 *     sequence lives in word start[s] + k/8, bits 4*(k%8); bits==2 -> 16 per word (codes < 4 only).
 *     Every sequence starts on a word boundary; start[] is in words; the word buffer must be
 *     followed by >= 4 readable padding words (rsd_pack writes them).
 *
 * Numeric modes (SURVEY section 0 item 2): chosen per call from the active costs and the symbols
 * present.  INT modes are used only when every reachable cost times 2^k is an integer, so they are
 * bit-identical to the reference's fp64; otherwise FP64 with the reference's operation order
 * (SED:95-109: left+ins, up+del, diag+sub; min; == ties).
 */
#ifndef RSD_H
#define RSD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSD_ABI_VERSION 1

enum {
    RSD_OK = 0,
    RSD_EINVAL = 1,     /* bad argument (message says which)                         */
    RSD_ENODEV = 2,     /* no CUDA device / driver: there is no CPU fallback         */
    RSD_ECUDA = 3,      /* a CUDA call failed                                        */
    RSD_ENOMEM = 4,     /* device or host allocation failed                          */
    RSD_ECOSTS = 5,     /* costs out of contract: negative, NaN or infinite          */
    RSD_ERANGE = 6      /* sequence too long for this entry point, or output > cap   */
};

enum {                  /* numeric mode actually used, reported through *mode_out    */
    RSD_MODE_I16X2 = 1, /* scaled int16, two pairs per register (DPX VIADDMNMX.S16x2)*/
    RSD_MODE_I32 = 2,   /* scaled int32                                              */
    RSD_MODE_F64 = 3    /* IEEE fp64, reference operation order                      */
};

enum { RSD_OP_INSERT = 0, RSD_OP_DELETE = 1, RSD_OP_UPDATE = 2 };  /* candidate order SED:103 */

typedef struct rsd_ctx rsd_ctx;

/* ---- library / context ------------------------------------------------------------------- */
int rsd_abi_version(void);
const char *rsd_last_error(void);
/* number of visible CUDA devices (0 when none); never creates a context */
int rsd_device_count(void);
/* create a context bound to `device`; the CUDA context itself is created on first use */
int rsd_create(int device, rsd_ctx **out);
int rsd_destroy(rsd_ctx *ctx);
/* pinned host memory helpers for callers without another allocator */
int rsd_host_alloc(void **out, int64_t bytes);
int rsd_host_free(void *p);

/* ---- costs: replaces the module globals default_costs / user_costs (SED:6-27) ---------------
 * sub is row-major [15][15], sub[src*15+dst] = C['update'][src][dst]; the diagonal is ignored
 * (SED:79-81).  Rejects negative / NaN / inf with RSD_ECOSTS (SURVEY Appendix A, last bullet). */
int rsd_set_costs(rsd_ctx *ctx, double ins, double del, const double *sub);
/* which mode a call would use for sequences made of the symbols in `symmask` (bit c = code c
 * present) with lengths up to max_m (source) / max_n (destination); *scale_log2_out = k */
int rsd_classify(rsd_ctx *ctx, uint32_t symmask, int64_t max_m, int64_t max_n, int force_mode,
                 int *mode_out, int *scale_log2_out);

/* ---- packing (ingest; host side, not on the hot path) ------------------------------------- */
/* words needed to pack n sequences given their lengths (includes the 4 padding words) */
int64_t rsd_pack_words(const int32_t *len, int64_t n, int bits);
/* codes: 1 byte per symbol, concatenated; off[n+1] symbol offsets.  Writes words/start/len and
 * ORs the symbols seen into *symmask_inout.  bits in {2,4}; bits==2 with a code >= 4 -> RSD_EINVAL */
int rsd_pack(const uint8_t *codes, const int64_t *off, int64_t n, int bits,
             uint32_t *words, int64_t *start, int32_t *len, uint32_t *symmask_inout);

/* ---- batched distance: replaces wagnerFisher(...)[-1][-1].value (SED:133-224, IR:439) -------
 * pair p = (source sequence p of A, destination sequence p of B); out[p] = D[m][n] as fp64.
 * max_m / max_n: upper bounds of the source / destination lengths as recorded at pack time
 * (0 = let the library scan a_len / b_len; an understated bound is an error the library cannot see).
 * force_mode: 0 = classify, or one of RSD_MODE_* (tests use it to cross-check the modes; forcing
 * an INT mode on costs that are not exactly representable fails with RSD_EINVAL).
 * a_start / b_start may be NULL: the side then has rsd_pack's canonical layout (sequence p starts at word
 * sum_{q<p} nwords(len[q])) and its offsets are rebuilt on the device from the lengths — 8 bytes per sequence
 * that never cross PCIe, and no layout check on the host.
 * Large batches are copied in five growing chunks on a copy stream while earlier chunks compute; that needs the
 * sequences stored in pair order without overlap (checked in one pass over caller-supplied start[] / len[]) —
 * otherwise the whole batch is copied first.
 * A context serialises its own work: do not overlap calls on one context from several streams. */
int rsd_distance_batch(rsd_ctx *ctx,
                       const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                       const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                       int64_t n_pairs, int64_t max_m, int64_t max_n, int bits, uint32_t symmask, int force_mode,
                       double *out, int *mode_out);
/* same from RAW symbol codes (1 byte per symbol, sequences concatenated without gaps in pair order, as the
 * reference's callers hold their strings: wagnerFisher(str1, str2), SED:133): the codes are copied chunk by chunk
 * and packed on the device (k_pack_codes), so ingest overlaps the kernels instead of preceding them.
 * bits: packing to use (2 needs every code < 4; a code that does not fit fails with RSD_EINVAL after the call's
 * work); symmask: symbols present, 0 = unknown (classified as if every symbol the packing can hold occurred). */
int rsd_distance_batch_codes(rsd_ctx *ctx, const uint8_t *a_codes, const int32_t *a_len,
                             const uint8_t *b_codes, const int32_t *b_len, int64_t n_pairs,
                             int64_t max_m, int64_t max_n, int bits, uint32_t symmask, int force_mode,
                             double *out, int *mode_out);
/* rsd_distance_batch with device pointers, asynchronous on `stream` (a cudaStream_t) */
int rsd_distance_batch_dev(rsd_ctx *ctx,
                           const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len,
                           const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len,
                           int64_t n_pairs, int64_t max_m, int64_t max_n, int bits, uint32_t symmask,
                           int force_mode, double *out, int *mode_out, void *stream);

/* ---- one pair, whole matrix: replaces the dp object of wagnerFisher (SED:133-224) ------------
 * values[(m+1)*(n+1)] fp64 row-major and mask[(m+1)*(n+1)]: bit0 INS, bit1 DEL, bit2 UPD = the
 * predecessor edges the reference creates (SED:109-124,163,181).  Always FP64 mode.
 * a/b: 1 byte per symbol codes (host). */
int rsd_matrix(rsd_ctx *ctx, const uint8_t *a, int32_t m, const uint8_t *b, int32_t n,
               double *values, uint8_t *mask);

/* ---- batched canonical edit script: replaces generate_es(create_paths(dp)[0], s1, s2)
 * (SED:228-334; canonical rule SURVEY a8: min cost, fewest edges, then INS < DEL < UPD).
 * Per pair p, ops are written origin->sink into slot p of stride `max_ops` (>= max(m+n)):
 *   op[p*max_ops+k] in RSD_OP_*, oi/oj = the matrix cell (1-based) the op enters, so the
 *   reference's fields are source.index = oi-1, destination.index = oj-1 (-1 wraps, SED:302-323).
 * n_ops[p] = number of ops, dist[p] = D[m][n]. */
int rsd_script_batch(rsd_ctx *ctx,
                     const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                     const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                     int64_t n_pairs, int bits, uint32_t symmask, int force_mode, int64_t max_ops,
                     uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist, int *mode_out);

/* ---- batched patch: replaces patching(es, str1) (SED:380-457) for scripts produced by
 * rsd_script_batch (closed form, SURVEY a12).  x = the strings to patch (packed like A), one per
 * pair; out: 1 byte per symbol codes in slot p of stride max_out (>= max(len x + n_ops));
 * err[p] in {0, 1, -1} (SED:389-399); out_len[p] = patched length (0 when -1).
 * Scripts must be paths of their pair: op codes 0/1/2 whose counts end at cell (a_len, b_len), and,
 * where oi / oj are given (either may be NULL), oj[t] = the destination cell entered by an INS or
 * UPD, oi[t] = the source cell entered by a DEL or UPD.  Scripts of rsd_script_batch and their
 * reverses (generate_rev_es) are paths; anything else fails with RSD_EINVAL naming the pair and the
 * op, checked on the host before any device work.  Hand-edited scripts go through sed.patching. */
int rsd_patch_batch(rsd_ctx *ctx,
                    const uint8_t *op, const int32_t *oi, const int32_t *oj, const int32_t *n_ops, int64_t max_ops,
                    const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                    const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                    const uint32_t *x_words, const int64_t *x_start, const int32_t *x_len, int64_t x_nwords,
                    int64_t n_pairs, int bits, int64_t max_out,
                    uint8_t *out, int32_t *out_len, int32_t *err);

/* ---- fused C3 pipeline: script + patch(A) + on-device round-trip check against B -------------
 * (timing.py:196-199 intent: patching(es, seq1) == seq2).  ok[p] = 1 when patch(script_p, A_p)
 * reproduces B_p with error code 0.  Scripts are returned like rsd_script_batch when op != NULL. */
int rsd_script_patch_check_batch(rsd_ctx *ctx,
                     const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                     const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                     int64_t n_pairs, int bits, uint32_t symmask, int force_mode, int64_t max_ops,
                     uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist,
                     uint8_t *ok, int *mode_out);

/* ---- database search: replaces search_collection(query, _, collection, wf_score)
 * (IR:443-477, default costs at that call site IR:470) + the stable descending top-k of
 * performance.py:12-15.  The packed database shard stays resident on the device. */
int rsd_db_load(rsd_ctx *ctx, const uint32_t *words, const int64_t *start, const int32_t *len,
                int64_t n_records, int64_t n_words, int bits, uint32_t symmask, int64_t global_index_base);
int rsd_db_free(rsd_ctx *ctx);
/* Append n_records records (packed like rsd_db_load, same `bits` as the loaded database) to the end of the loaded
 * database: record j gets global index global_index_base + db_n + j.  The state afterwards is the one rsd_db_load
 * gives for the concatenation (old records, then new ones, in order): the same stored order (records sorted by tier,
 * length and collection index, the tiers re-derived from the symbol counts of the concatenation), tiers, maximum
 * length and word count; the symbol mask is the OR of the old mask and `symmask`.  Every search then answers as after
 * a fresh load.  The stored order is rebuilt on the device: the loaded records are not uploaded again.  A built idf
 * table is continued over the new records, not rebuilt.  Refused with RSD_EINVAL, before any device work: no database
 * loaded, `bits` other than the database's, a 2-bit database with `symmask` outside ACGU, a negative length, a record
 * outside the word buffer, NULL buffers with n_records > 0.  n_records == 0 changes nothing.  An error before the new
 * layout is complete leaves the loaded database and its idf table unchanged; if only the idf continuation fails, the
 * appended database stands (RSD_OK) and its table is rebuilt on next use. */
int rsd_db_append(rsd_ctx *ctx, const uint32_t *words, const int64_t *start, const int32_t *len,
                  int64_t n_records, int64_t n_words, int bits, uint32_t symmask);
/* Introspection (tests, tools): the stored order of the loaded database.  *n_records = db_n; perm[db_n] (may be NULL)
 * = global index of stored record r; tier_end[16], tier_mask[16] (either may be NULL): stored records
 * [0, tier_end[t]) use only the symbols tier_mask[t]. */
int rsd_db_layout(rsd_ctx *ctx, int64_t *n_records, int64_t *perm, int64_t *tier_end, uint32_t *tier_mask);
/* queries packed like a batch; for each query q: the k best records of this shard by
 * (score = 1/(1+D) descending, global index ascending): top_idx[q*k+r] (global index, -1 when the
 * shard has fewer than k records), top_score[q*k+r].  all_scores (optional, host) receives
 * n_queries * n_records fp64 scores in record order = the list search_collection returns. */
int rsd_db_search_topk(rsd_ctx *ctx, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                       int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, int k, int force_mode,
                       int64_t *top_idx, double *top_score, double *all_scores, int *mode_out);
/* device-output variant for multi-GPU callers that gather with NCCL: top_idx/top_score are device
 * pointers, asynchronous on `stream` */
int rsd_db_search_topk_dev(rsd_ctx *ctx, const uint32_t *q_words_dev, const int64_t *q_start_dev,
                           const int32_t *q_len_dev, int64_t n_queries, int64_t max_qlen, int bits,
                           uint32_t q_symmask, int k, int force_mode,
                           int64_t *top_idx_dev, double *top_score_dev, int *mode_out, void *stream);
/* Range search: replaces the wf_score scan of search_collection (IR:466-477) followed by a filter on
 * the distance.  For each query q (caller order): every record r of this shard with D(q, r) <= max_dist,
 * D being the fp64 value rsd_distance_batch returns for (source = query, destination = record); the
 * bound is inclusive and exact (integer modes compare the scaled distance with floor(max_dist * 2^k)).
 * CSR output, each query's hits by global index ascending: hit_off[n_queries + 1], hit_idx[total]
 * (global index), hit_dist[total] = D.  cap is the length of hit_idx / hit_dist: more hits than cap
 * return RSD_ERANGE with hit_off complete (the total is hit_off[n_queries]) and the hit arrays
 * unspecified.  max_dist must be >= 0 and not NaN (+inf: every record).  force_mode / mode_out as
 * in rsd_db_search_topk. */
int rsd_db_search_range(rsd_ctx *ctx, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                        int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, double max_dist,
                        int force_mode, int64_t cap, int64_t *hit_off, int64_t *hit_idx, double *hit_dist,
                        int *mode_out);
/* Set / multiset / TF-vector similarity of one query against the loaded database — the other scorers
 * of search_collection (IRMethods.py:443-477 with the measures of IRMethods.py:49-389; documents'
 * 'tf' vectors are rebuilt on the device from the sequences, what fa_import.py:49 stores).  `method`
 * is one of RSD_SIM_*; q_codes are symbol codes 0..14.  all_scores (may be NULL) receives db_n fp64
 * scores in record order; k > 0 also returns the top-k with the key (score desc, global index asc).
 * Scores equal the reference's numpy arithmetic bit for bit; its 0/0 cases come back as NaN and are
 * never ranked.  The cost tables play no role here. */
enum {
    RSD_SIM_SET_INTERSECTION = 0, RSD_SIM_SET_JACCARD = 1, RSD_SIM_SET_DICE = 2,
    RSD_SIM_MULTI_INTERSECTION = 3, RSD_SIM_MULTI_JACCARD = 4, RSD_SIM_MULTI_DICE = 5,
    RSD_SIM_COSINE = 6, RSD_SIM_PEARSON = 7, RSD_SIM_EUCLIDEAN = 8, RSD_SIM_MANHATTAN = 9,
    RSD_SIM_TANIMOTO = 10, RSD_SIM_DICE = 11
};
int rsd_db_similarity(rsd_ctx *ctx, const uint8_t *q_codes, int32_t q_len, int method, int k,
                      int64_t *top_idx, double *top_score, double *all_scores);
/* rsd_db_similarity for a batch of queries: query q is q_codes[q_off[q] .. q_off[q+1]) (codes 0..14, q_off[0] == 0,
 * non-decreasing, each length <= INT32_MAX).  top_idx / top_score [n_queries][k] (k in 0..RSD_TOPK_MAX; -1 / 0.0 past
 * the rankable records, NaN never ranked); all_scores (may be NULL) [n_queries][db_n] in record order.
 * Row q is bit for bit what rsd_db_similarity returns for query q alone.  The records are read once per query batch
 * (up to 64 queries, fewer when device memory is short or RSD_SIM_QBATCH asks for fewer), not once per query.
 * Arguments are checked on the host before any device work (RSD_EINVAL); n_queries == 0 writes nothing. */
int rsd_db_similarity_batch(rsd_ctx *ctx, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                            int method, int k, int64_t *top_idx, double *top_score, double *all_scores);
/* The idf and tf-idf vector types of search_collection (IRMethods.py:458-465; the vectors of IRMethods.py:189-225).
 * The idf vector of a sequence is idf[p] = log10(N / df[p]) (0 where df[p] == 0) at each distinct literal bigram p of
 * it, 0 elsewhere; tf-idf is the matrix product tf . idf.  df[p] is the sum over the collection, in collection order,
 * of compare_pair_to_seq(p, document) (IRMethods.py:225-252), N the number of records.  The table is built on the
 * device on first use after rsd_db_load, continued by rsd_db_append and kept until the next rsd_db_load / rsd_db_free;
 * idf is computed on the host
 * from df exactly as Python's math.log(N / df, 10).  A database loaded with global_index_base != 0 is one shard of a
 * collection whose other records it does not know: these calls refuse it (RSD_EINVAL); use rsd_multi for shards. */
enum { RSD_VEC_IDF = 1, RSD_VEC_TFIDF = 2 };
/* df[225], idf[225] (either may be NULL) of the loaded database, row-major [15][15] in table order; builds the table
 * when needed */
int rsd_db_idf_table(rsd_ctx *ctx, double *df, double *idf);
/* rsd_db_similarity_batch over the idf (RSD_VEC_IDF) or tf-idf (RSD_VEC_TFIDF) vectors of the query and the records;
 * method in RSD_SIM_COSINE..RSD_SIM_DICE (the set and multiset measures have no vector type: RSD_EINVAL).  Same
 * outputs, batching and argument checks as rsd_db_similarity_batch; the scores equal the reference's bit for bit. */
int rsd_db_vector_similarity_batch(rsd_ctx *ctx, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                                   int vector_type, int method, int k, int64_t *top_idx, double *top_score,
                                   double *all_scores);
/* merge G shards' top-k lists (each n_queries*k, shard-major) with the same key — the reduction
 * run after the gather (host side, O(G*k) per query) */
int rsd_topk_merge(const int64_t *idx, const double *score, int n_shards, int64_t n_queries, int k,
                   int64_t *out_idx, double *out_score);

/* ---- database search over several GPUs of one box, ONE process -------------------------------------------
 * Replaces the process fan-out under IRMethods.create_search_threads / search_collection (IR:443-515) on the
 * wf_score path and for the similarity measures: the database is cut into contiguous shards balanced by symbols,
 * one per device; the query batch goes to every device; each device keeps a local top-k; the lists (Q * k * 16
 * bytes per device) are gathered with ONE grouped ncclAllGather over NVLink and merged with the key (score desc, index asc) — identical to the
 * stable descending sort over the whole collection because shards are index-contiguous.  NCCL is bound at run
 * time (dlopen), only when more than one distinct device is used.  devices == NULL / n_devices == 0: all visible
 * devices.  A device may be listed several times (shards emulated on one GPU; the gather is then plain copies). */
typedef struct rsd_multi rsd_multi;
int rsd_multi_create(const int *devices, int n_devices, rsd_multi **out);
int rsd_multi_destroy(rsd_multi *m);
int rsd_multi_device_count(rsd_multi *m);
int rsd_multi_set_costs(rsd_multi *m, double ins, double del, const double *sub);
int rsd_multi_db_load(rsd_multi *m, const uint32_t *words, const int64_t *start, const int32_t *len,
                      int64_t n_records, int64_t n_words, int bits, uint32_t symmask);
int rsd_multi_db_free(rsd_multi *m);
/* rsd_db_append over the whole database: the records go to the last shard (shards stay index-contiguous, they are not
 * rebalanced: a reload does that); a built idf table is continued and the new table goes to every device */
int rsd_multi_db_append(rsd_multi *m, const uint32_t *words, const int64_t *start, const int32_t *len,
                        int64_t n_records, int64_t n_words, int bits, uint32_t symmask);
/* like rsd_db_search_topk, over the whole database; all_scores (optional) is [n_queries][n_records] */
int rsd_multi_db_search_topk(rsd_multi *m, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                             int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, int k, int force_mode,
                             int64_t *top_idx, double *top_score, double *all_scores, int *mode_out);
/* like rsd_db_similarity_batch, over the whole database: every device scores its shard, the local top-k lists go
 * through the same gather and merge as rsd_multi_db_search_topk; all_scores (optional) is [n_queries][n_records] */
int rsd_multi_db_similarity(rsd_multi *m, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                            int method, int k, int64_t *top_idx, double *top_score, double *all_scores);
/* rsd_db_idf_table over the whole database: the df sums run through the shards in order (device 0's partial sums
 * continue on device 1, ...), and every device gets the one idf table */
int rsd_multi_db_idf_table(rsd_multi *m, double *df, double *idf);
/* rsd_db_vector_similarity_batch over the whole database, scored and gathered like rsd_multi_db_similarity */
int rsd_multi_db_vector_similarity(rsd_multi *m, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                                   int vector_type, int method, int k, int64_t *top_idx, double *top_score,
                                   double *all_scores);
/* like rsd_db_search_range (which replaces the wf_score scan of search_collection, IR:466-477, followed
 * by a filter on the distance), over the whole database: each device searches its shard, and the hits of
 * a query are the shards' hits in shard order; cap / RSD_ERANGE apply to the total */
int rsd_multi_db_search_range(rsd_multi *m, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                              int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, double max_dist,
                              int force_mode, int64_t cap, int64_t *hit_off, int64_t *hit_idx, double *hit_dist,
                              int *mode_out);
int64_t rsd_multi_launch_count(rsd_multi *m);

/* ---- long pairs (>= ~10 kb): block-tiled wavefront with traceback ----------------------------
 * Replaces wagnerFisher + create_paths(dp)[0] + generate_es (StringEditDistance.py:133-334) for pairs whose
 * matrix the reference cannot hold (~500 B per cell).  a / b: 1 byte per symbol (code 0..14, table order).
 * Script output as in rsd_script_batch: op (0 insert, 1 delete, 2 update) and the matrix cell (oi, oj) each
 * op enters, origin -> sink; max_ops >= m + n.
 * rsd_long_pair: one pair.  A pair whose 2-bit direction matrix does not fit the device (or whose column
 * panels exceed the co-resident CTAs) is computed in row blocks from stored key rows (linear-space overflow
 * path: checkpoint rows top to bottom, then recomputation with directions and traceback bottom to top) —
 * same distance and script as the one-launch path. */
int rsd_long_pair(rsd_ctx *ctx, const uint8_t *a, int64_t m, const uint8_t *b, int64_t n,
                  int force_mode, int want_script, int64_t max_ops,
                  uint8_t *op, int32_t *oi, int32_t *oj, int64_t *n_ops, double *dist, int *mode_out);
/* rsd_long_pairs: a batch of long pairs (BASELINE config 4) in as few launches as memory allows; the pairs of
 * a launch share the GPU (rings of CTAs, one pair after the other per ring).  Arrays of n_pairs entries;
 * oi / oj (the arrays or single entries) may be NULL; mode_out (optional) receives one mode per pair. */
int rsd_long_pairs(rsd_ctx *ctx, int n_pairs, const uint8_t *const *a, const int64_t *m,
                   const uint8_t *const *b, const int64_t *n, int force_mode, int want_script,
                   const int64_t *max_ops, uint8_t *const *op, int32_t *const *oi, int32_t *const *oj,
                   int64_t *n_ops, double *dist, int *mode_out);
/* device time in ms of the forward (matrix fill) launches of the last rsd_long_pair(s) call (rsd_set_timing) */
double rsd_long_forward_ms(rsd_ctx *ctx);

/* ---- introspection for bench.py / tests ---------------------------------------------------- */
/* kernels launched by this context since creation (bench.py's gpu_launches) */
int64_t rsd_launch_count(rsd_ctx *ctx);
/* device time in ms of the dominant kernel of the last batch call, measured with CUDA events on
 * the stream it was launched on (0 when the call did not time it) */
double rsd_last_kernel_ms(rsd_ctx *ctx);
/* enable/disable that per-kernel timing (adds two event records per call) */
int rsd_set_timing(rsd_ctx *ctx, int on);
/* INT32 / DPX / FP64 issue-rate microbenchmark: ops per second of `which`
 * (0 IADD3, 1 VIADDMNMX.S32, 2 VIADDMNMX.S16x2 [counted as 1 op/instr/lane], 3 PRMT, 4 DADD,
 *  5 IMAD, 6 VIMNMX3, 7 mixed IMAD+ALU) */
int rsd_ubench(rsd_ctx *ctx, int which, double *ops_per_s);

#ifdef __cplusplus
}
#endif
#endif /* RSD_H */
