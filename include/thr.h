/*
 * thr.h — C-ABI of libthr.so: the B200-native triple-hybrid retrieval scoring path.
 *
 * This is the drop-in boundary below the reference's Python retriever.  Every entry
 * point replaces the arithmetic behind one reference call site (cited per function,
 * paths relative to the reference checkout).  The reference itself has no FFI: its
 * scoring lives in Postgres RPCs and an HTTP reranker, so the binding a maintainer
 * adds is the ctypes stub shown in INTEGRATION.md.
 *
 * Conventions
 *   - Plain C: pointers and sizes only, no torch / C++ types.
 *   - Every pointer is a DEVICE pointer on the handle's GPU unless the name starts
 *     with `h_`.  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - Every call returns 0 (THR_OK) or a negative THR_E* code; thr_last_error()
 *     returns a human-readable message for the most recent failure on that handle.
 *   - Calls enqueue work on `stream` and return; device-side failures (candidate
 *     buffer overflow, pipeline watchdog) are reported by thr_sync().
 *   - A handle is thread-compatible: one thread at a time per handle, no globals.
 *   - There is NO CPU fallback anywhere behind this interface.
 */
#ifndef THR_H_
#define THR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define THR_ABI_VERSION 13

enum {
  THR_OK = 0,
  THR_EINVAL = -1,       /* bad argument */
  THR_ECUDA = -2,        /* CUDA runtime / driver error */
  THR_EUNSUPPORTED = -3, /* shape outside what the sm_100a kernels are built for */
  THR_ENOINDEX = -4,     /* a *_topk call before the matching *_index_set */
  THR_EOVERFLOW = -5,    /* device candidate buffer overflowed (reported by thr_sync) */
  THR_ETIMEOUT = -6,     /* device pipeline watchdog fired (reported by thr_sync) */
  THR_ENOMEM = -7
};

/* Fusion variants: which reference arithmetic thr_fuse reproduces bit-for-bit. */
enum {
  THR_FUSE_RAG2 = 0,   /* w / (k + rank)          src/voice_agent/rag2/retrieval.py:358-376 */
  THR_FUSE_LIB = 1,    /* w * (1.0 / (k + rank))  triple-hybrid-rag/src/triple_hybrid_rag/core/fusion.py:167-185 */
  THR_FUSE_RAG1 = 2    /* 1.0 / (k + rank0 + 1)   src/voice_agent/retrieval/hybrid_search.py:460-501 */
};

/* Order of candidates whose fused fp64 scores are exactly equal. */
enum {
  THR_TIE_INSERTION = 0, /* reference behaviour: stable sort, lexical -> semantic -> graph first-seen order */
  THR_TIE_CHUNK_ID = 1   /* BASELINE.json north_star: ascending chunk id */
};

typedef struct thr_handle thr_handle;

/* ---- lifetime ------------------------------------------------------------------- */

int thr_abi_version(void);
int thr_create(int device, thr_handle** out);
int thr_destroy(thr_handle* h);
/* Message of the last failure on `h` (h == NULL: last thr_create failure). Never NULL. */
const char* thr_last_error(const thr_handle* h);
/* Synchronise `stream` and surface device-side failures recorded since the last thr_sync. */
int thr_sync(thr_handle* h, void* stream);
/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
int64_t thr_launch_count(const thr_handle* h);
/* Let kernels launched through `h` read memory of `peer_device` (cudaDeviceCanAccessPeer, then
 * cudaDeviceEnablePeerAccess in the handle's device context; a runtime setting of this process only).  Already
 * enabled, or peer_device == the handle's device: THR_OK.  THR_EUNSUPPORTED when the pair cannot peer. */
int thr_peer_enable(thr_handle* h, int peer_device);

/* Per-kernel device timing.  When enabled, every kernel launch is bracketed by CUDA events on the
 * launch stream; thr_prof_read synchronises the device, adds up the elapsed times recorded for
 * `slot` since the last thr_prof_reset and returns the number of launches.  This is how bench.py
 * measures the dominant kernel inside the timed step (roofline.achieved). */
enum {
  THR_PROF_DENSE_SCORE = 0, THR_PROF_DENSE_FINALIZE = 1, THR_PROF_BM25 = 2, THR_PROF_FUSE = 3,
  THR_PROF_MAXSIM = 4, THR_PROF_MERGE = 5, THR_PROF_SAFETY = 6, THR_PROF_BM25_PREP = 7,
  THR_PROF_DENSE_SEED = 8, /* seed pass of thr_dense_topk: prefix scoring + threshold select (two launches) */
  THR_PROF_RERANK = 9,     /* thr_rerank_rows + thr_rerank_finish around thr_maxsim */
  THR_PROF_SLOTS = 10
};
int thr_prof_enable(thr_handle* h, int on);
/* Time only the slots whose bit is set in `mask` (bit s = slot s; default: all).  An event pair costs ~3 us of
 * stream time: bench.py times the roofline kernels inside the timed region and the small ones in a pass of their own. */
int thr_prof_select(thr_handle* h, unsigned mask);
int thr_prof_reset(thr_handle* h);
int thr_prof_read(thr_handle* h, int slot, double* total_ms, int64_t* launches);

/* ---- K1: semantic channel — exact dense top-k ------------------------------------
 * Replaces RAG2Retriever._semantic_search -> RPC rag2_semantic_search
 *   src/voice_agent/rag2/retrieval.py:294-314
 *   database/migrations/20260114_rag2_schema.sql:377-410   (ORDER BY embedding <=> q LIMIT n;
 *   similarity = 1 - cosine distance; vectors are L2-normalised so ranking is by dot product).
 * Exact (brute force), not HNSW.
 *
 * X: bf16 [N, D] row-major, resident for the lifetime of the index (not copied).
 * D must be a multiple of 64, 64 <= D <= 8192.  id_base is added to every returned id
 * (the shard's first global chunk id).
 */
int thr_dense_index_set(thr_handle* h, const void* X, int64_t N, int D, int64_t id_base);

/* Q: bf16 [B, D].  For each query: the k chunks with the largest dot product, ordered by
 * (score desc, id asc).  Scores are the fp64 dot products of the bf16 inputs (tensor-core
 * fp32 scores select k + margin survivors, which are re-scored exactly before the final sort).
 *   out_ids    [B, k] int64   (id_base + row; -1 past out_count)
 *   out_scores [B, k] double
 *   out_count  [B]    int32   min(k, N live rows)
 *   out_gap    [B]    float, nullable: (exact k-th score) - (best tensor-core score that was
 *              NOT re-scored); the result is certified exact when gap > the fp32 accumulation
 *              error bound.  +inf when every chunk was re-scored.
 * 1 <= k, k + margin <= 256.  Rows marked in the deletion bitmap (thr_dense_deleted_set) are never returned.
 */
int thr_dense_topk(thr_handle* h, const void* Q, int B, int k, int margin,
                   int64_t* out_ids, double* out_scores, int32_t* out_count, float* out_gap,
                   void* stream);

/* Tag filter of the semantic channel — the `collection` predicate of rag2_semantic_search
 * (database/migrations/20260114_rag2_schema.sql:404-406) evaluated inside the scan instead of by
 * over-fetching.  tags [N] uint16 on the device (8-byte aligned, stays resident; NULL clears): one tag per
 * chunk, e.g. the collection id.  thr_dense_topk_tagged is thr_dense_topk restricted, per query, to the
 * chunks whose tag equals want[q] (want [B] int32 on the device; < 0 = no restriction; NULL = plain
 * thr_dense_topk): the exact top-k of the filtered corpus, out_count = min(k, eligible chunks).
 */
int thr_dense_tags_set(thr_handle* h, const uint16_t* tags);
int thr_dense_topk_tagged(thr_handle* h, const void* Q, int B, int k, int margin, const int32_t* want,
                          int64_t* out_ids, double* out_scores, int32_t* out_count, float* out_gap,
                          void* stream);

/* Deletion bitmap of the semantic channel: rows removed from the corpus without a rebuild.  bits
 * [ceil(N / 32)] uint32 on the device (16-byte aligned, stays resident; NULL clears): bit i % 32 of word i / 32
 * set = row i is deleted.  While it is set, every thr_dense_topk / thr_dense_topk_tagged call (every query, any
 * want) skips deleted rows inside the scan: they are never returned, thresholds are learnt from live rows only,
 * out_count = min(k, live eligible rows), and out_gap keeps its meaning over the eligible rows.  Like the tags,
 * the bitmap is dropped by the next thr_dense_index_set.
 */
int thr_dense_deleted_set(thr_handle* h, const uint32_t* bits);

/* ---- K2: lexical channel — BM25 top-k over a blocked CSR inverted index ----------
 * Replaces RAG2Retriever._lexical_search -> RPC rag2_lexical_search
 *   src/voice_agent/rag2/retrieval.py:273-292
 *   database/migrations/20260114_rag2_schema.sql:341-374
 * (interface: space-joined keywords, top-`limit` by descending score).  The scoring
 * formula is BM25 as BASELINE.json's north_star asks (Postgres ts_rank_cd is not in the
 * reference tree); it is defined in oracle/bm25.py and DESIGN.md.
 *
 * Index layout (built by triple_hybrid_rag_b200.index.BM25Index on the device): a CSR inverted
 * index with per-term range skips.
 *   postings: 8-byte records {uint32 local_doc, float impact}, term-major, doc ascending inside a
 *   term; impact = tf*(k1+1)/(tf + k1*(1-b+b*len/avgdl)); 16 bytes of padding after the last record.
 *   Documents are split into n_blk ranges of blk_docs consecutive local doc ids;
 *   skip [V*n_blk + 1] int64: postings[skip[t*n_blk + r] .. skip[t*n_blk + r + 1]) are term t's
 *   postings inside range r (so skip[t*n_blk] .. skip[(t+1)*n_blk] is term t's whole list: the
 *   usual CSR indptr is skip[::n_blk]);  idf [V] float.
 * blk_docs must be a power of two in [256, 2048] (the skip granularity: one warp of the kernel owns one range at a
 * time).  idf must be >= 0 (BM25's ln(1 + ...) always is: the kernel relies on partial sums never decreasing) and,
 * unless 0, lie in [2^-40, 2^20]; impacts must be BM25's (0 <= impact < k1 + 1; anything below 2^15 is safe): the
 * kernel accumulates sums scaled by 2^-40 (exactly: a power of two) to keep two bits of every slot for a generation tag.
 * Arrays stay resident (not copied).
 */
int thr_bm25_index_set(thr_handle* h, const int64_t* skip, const void* postings,
                       const float* idf, int64_t n_docs, int32_t n_blk, int32_t blk_docs,
                       int32_t V, int64_t id_base);

/* q_terms [q_off[B]] int32 term ids (OR semantics; a term id outside [0,V) is ignored),
 * q_off [B+1] int32.  score(d) = sum over the query's terms IN ORDER of idf[t]*impact(t,d),
 * accumulated in fp32 (round-to-nearest, no FMA contraction) — the order is part of the
 * definition, so results are bit-reproducible.  Only docs with score > 0 are eligible;
 * order is (score desc, id asc).
 *   out_ids [B,k] int64 (-1 past count), out_scores [B,k] float, out_count [B] int32.
 * 1 <= k <= 256, at most 32 terms per query.  Docs marked in the deletion bitmap (thr_bm25_deleted_set) are never
 * returned.
 */
int thr_bm25_topk(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                  int64_t* out_ids, float* out_scores, int32_t* out_count, void* stream);

/* Tag filter of the lexical channel (the `collection` predicate of rag2_lexical_search, :368-370): same
 * contract as thr_dense_tags_set / thr_dense_topk_tagged; tags [n_docs] uint16 on the device, 8-byte aligned. */
int thr_bm25_tags_set(thr_handle* h, const uint16_t* tags);
int thr_bm25_topk_tagged(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                         const int32_t* want, int64_t* out_ids, float* out_scores, int32_t* out_count,
                         void* stream);

/* Deletion bitmap of the lexical channel: same contract as thr_dense_deleted_set, over local doc ids; bits
 * [ceil(n_docs / 32)] uint32 on the device, 16-byte aligned.  Applies to every thr_bm25_topk* call (OR and AND,
 * any want); dropped by the next thr_bm25_index_set.  idf is the caller's: recompute it from the live docs and
 * write it into the resident idf array when the live set changes.  The planner's cost estimates keep counting
 * the postings of deleted docs. */
int thr_bm25_deleted_set(thr_handle* h, const uint32_t* bits);

/* AND semantics — the `tsv @@ plainto_tsquery(...)` predicate of rag2_lexical_search
 * (database/migrations/20260114_rag2_schema.sql:369: every lexeme of the query must match).  thr_bm25_topk_ex is
 * thr_bm25_topk_tagged (want may be NULL) with flags: THR_BM25_REQUIRE_ALL keeps only docs that contain EVERY
 * distinct term of the query (a repeated term counts and scores once; a term id outside [0,V) or without
 * postings means no doc matches); scores and order are as above, restricted to those docs. */
enum { THR_BM25_REQUIRE_ALL = 1 };
int thr_bm25_topk_ex(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                     const int32_t* want, int flags, int64_t* out_ids, float* out_scores, int32_t* out_count,
                     void* stream);

/* ---- K3: weighted RRF fusion + safety threshold + conformal denoise ---------------
 * Replaces, bit-exactly in fp64:
 *   THR_FUSE_RAG2: RAG2Retriever._retrieve_candidates merge + _fuse_rrf
 *                  src/voice_agent/rag2/retrieval.py:203-271, :358-376
 *   THR_FUSE_LIB : RRFFusion.fuse incl. _apply_safety_threshold, _apply_conformal_denoising
 *                  triple-hybrid-rag/src/triple_hybrid_rag/core/fusion.py:52-247
 *   THR_FUSE_RAG1: HybridSearcher._rrf_fusion  src/voice_agent/retrieval/hybrid_search.py:460-501
 *
 * Three ranked id lists per query in CSR form (ids int64, off int32 [B+1]); rank = 1 + position.
 * Negative ids are padding and ignored, so a fixed-width [B,k] top-k result (-1 past its count) can
 * be passed as is with off[q] = q*k.  A NULL ids pointer means the channel is absent for every query.  *_sc are the channels' raw
 * scores (double, nullable; only THR_FUSE_LIB reads them).  weights [B,3] double in the order
 * lexical, semantic, graph.  Each list may be at most 256 long.
 *
 * THR_FUSE_LIB applies, after the sort: keep rows whose max raw channel score >= safety_thr
 * (skipped when safety_thr <= 0), then if denoise != 0 and >= 3 rows remain keep rrf >=
 * numpy.percentile(rrf, (1 - alpha) * 100) (linear interpolation), then truncate to top_k
 * (top_k <= 0: no truncation).  The other variants only sort and truncate.
 *
 * Outputs, row-major with row stride max_out (>= the largest possible union, or >= top_k):
 *   out_ids [B,max_out] int64, out_rrf [B,max_out] double,
 *   out_ranks [B,max_out,3] int32 (0 = absent from that channel),
 *   out_raw [B,max_out,3] double, nullable (merged raw scores, THR_FUSE_LIB),
 *   out_count [B] int32.
 */
int thr_fuse(thr_handle* h, int variant, int tie_mode, int B,
             const int64_t* lex_ids, const int32_t* lex_off, const double* lex_sc,
             const int64_t* sem_ids, const int32_t* sem_off, const double* sem_sc,
             const int64_t* gr_ids, const int32_t* gr_off, const double* gr_sc,
             const double* weights, int rrf_k, double safety_thr, double alpha, int denoise,
             int top_k, int max_out,
             int64_t* out_ids, double* out_rrf, int32_t* out_ranks, double* out_raw,
             int32_t* out_count, void* stream);

/* RAG2Retriever._fuse_rrf   src/voice_agent/rag2/retrieval.py:358-376
 * The reference's own signature: candidates that already carry their 1-based channel ranks.
 * Per query q with candidates [off[q], off[q+1]) (at most 1024): ranks [n,3] int32 in the order
 * lexical, semantic, graph; 0 = absent (Python truthiness of `c.lexical_rank`).  weights [B,3].
 *   out_rrf   [n] double : rrf_score of candidate i, bit-identical to the Python floats
 *   out_order [n] int32  : for each query, candidate indices (relative to off[q]) in the order of
 *                          sorted(candidates, key=rrf_score, reverse=True) — stable, ties keep input order.
 */
int thr_fuse_ranked(thr_handle* h, int B, const int32_t* off, const int32_t* ranks,
                    const double* weights, int rrf_k, double* out_rrf, int32_t* out_order,
                    void* stream);

/* RAG2Retriever._apply_safety   src/voice_agent/rag2/retrieval.py:461-495
 * Per query q with candidates [off[q], off[q+1]) in their current (post-rerank) order:
 *   s_i = has_rerank[i] && rerank[i] != 0 ? rerank[i] : rrf[i]      (`rerank_score or rrf_score`)
 *   max_score = max s_i; refused = max_score < threshold  (empty list: refused, max 0)
 *   keep[i] = !refused && s_i >= alpha*max_score && (#kept before i) < top_k
 * has_rerank nullable (= all zero).  Outputs keep [n] uint8, refused [B] uint8, max_score [B] double.
 */
int thr_safety(thr_handle* h, int B, const int32_t* off, const double* rerank,
               const uint8_t* has_rerank, const double* rrf, double threshold, double alpha,
               int top_k, uint8_t* keep, uint8_t* refused, double* max_score, void* stream);

/* ---- K4: late-interaction MaxSim rerank -----------------------------------------
 * Stands where RAG2Retriever._rerank calls Qwen3VLReranker._rerank_batch_native(query,
 * documents) -> List[float]   src/voice_agent/rag2/retrieval.py:405-459,
 * src/voice_agent/retrieval/reranker.py:287-354  (one score per candidate, input order).
 * score(q, c) = sum_i max_j <Qtok[q,i,:], Dtok[c,j,:]>  over i < q_len[q], j < d_len[c].
 *
 * Qtok bf16 [B, Tq, d]; Dtok bf16 [n_docs, Td, d] token store; cand [B, C] int64 rows of
 * the store (< 0: slot skipped, score -inf); q_len [B] / d_len [n_docs] int32 nullable
 * (= full).  out [B, C] float.  d == 128, Td in {64,128}, 1 <= Tq <= 128.
 */
int thr_maxsim(thr_handle* h, const void* Qtok, const int32_t* q_len, int B, int Tq, int d,
               const void* Dtok, const int32_t* d_len, int64_t n_docs, int Td,
               const int64_t* cand, int C, float* out, void* stream);

/* thr_maxsim on a residual-compressed token store (the ColBERTv2 / PLAID layout, 2-bit codes): 36 B per token
 * instead of 256 B.  Every array is on the device; d == 128, Td in {64, 128}:
 *   centroids bf16 [n_centroids, 128]  the codebook (16-byte aligned; read through L2)
 *   weights   fp32 [128, 4]            weights[k, c] = reconstruction value of code c in dimension k (16-byte aligned)
 *   cids      int32 [n_rows, Td]       centroid of each token, in [0, n_centroids)
 *   codes     uint32 [n_rows, Td, 8]   2-bit code of dimension k = bits 2*(k % 16), 2*(k % 16) + 1 of word k / 16
 *   d_len     int32 [n_rows], nullable tokens per row, as in thr_maxsim
 * Token j of row r decodes to x[k] = bf16_rn(fp32(centroids[cids[r, j], k]) + weights[k, code]) (one fp32 add,
 * round to nearest, no FMA; no renormalisation), and the score is thr_maxsim's on the decoded store: for the same
 * inputs the outputs are bit-identical to thr_maxsim(Qtok, decode(store), ...).  Constraints are thr_maxsim's
 * except that n_rows * Td may exceed 2^31.  A candidate < 0 or >= n_rows scores -inf.  The caller guarantees cids in
 * range (a cid outside the table is clamped, never dereferenced).  Timed in the THR_PROF_MAXSIM slot.
 */
int thr_maxsim_packed(thr_handle* h, const void* Qtok, const int32_t* q_len, int B, int Tq, int d,
                      const uint32_t* codes, const int32_t* cids, const void* centroids, int64_t n_centroids,
                      const float* weights, const int32_t* d_len, int64_t n_rows, int Td,
                      const int64_t* cand, int C, float* out, void* stream);

/* The batched rerank stage around thr_maxsim — RAG2Retriever.retrieve steps 4-6, src/voice_agent/rag2/retrieval.py:175-191,
 * for B queries at once (the reference runs them one query at a time in Python).
 *
 * thr_rerank_rows: the first C candidates of each fused list -> rows of THIS rank's token store.
 *   ids [B, stride] int64 fused ids (-1 padded), count [B]; a candidate whose id lies in [id_lo, id_hi) (the chunk-id
 *   range this rank owns) maps to row (id - id_lo + row_off), taken modulo `period` when period > 0 (a synthetic store
 *   that repeats: row_off = id_lo % period makes the row a function of the GLOBAL id, whatever the sharding); every other
 *   slot maps to -1, which thr_maxsim scores -inf.  rows [B, C] int64.
 * With a sharded corpus the ranks then exchange the [B, C] float scores with one all-reduce(MAX) (exactly one rank owns
 * a candidate); single GPU: no exchange.
 *
 * thr_rerank_finish: `_rerank`'s ordering and `_apply_safety` (retrieval.py:455, :461-495) on the merged scores.
 *   raw [B, C] float: MaxSim sums, -inf where the candidate was not scored.  Per query, over its first
 *   n = min(count, C) candidates:  rerank_score = min(1, max(0, 0.5 * (raw / Tq + 1))) in fp64 (none if raw == -inf);
 *   order = sorted(key = rerank_score or 0, reverse = True), stable;  s_i = rerank_score or rrf_score;
 *   max_score = max s_i; refused = max_score < threshold (n == 0: refused, 0.0);
 *   keep_i = !refused && s_i >= alpha * max_score && fewer than top_k kept before i.
 *   Outputs in the reranked order, [B, C]: out_ids (-1 padded), out_rerank (-1 where none), out_rrf, out_keep;
 *   out_n [B], refused [B] uint8, max_score [B].  1 <= C <= 256.
 */
int thr_rerank_rows(thr_handle* h, const int64_t* ids, const int32_t* count, int B, int C, int stride,
                    int64_t id_lo, int64_t id_hi, int64_t period, int64_t row_off, int64_t* rows, void* stream);
int thr_rerank_finish(thr_handle* h, int B, int C, int stride, const int64_t* ids, const double* rrf,
                      const int32_t* count, const float* raw, int Tq, double threshold, double alpha, int top_k,
                      int64_t* out_ids, double* out_rerank, double* out_rrf, uint8_t* out_keep, int32_t* out_n,
                      uint8_t* refused, double* max_score, void* stream);

/* ---- K5: merge of per-shard top-k lists (consumes the all-gather buffer) ----------
 * scores [G,B,k_in] double, ids [G,B,k_in] int64, counts [G,B] int32 (valid prefix per list).
 * Per query the k_out best by (score desc, id asc).  G*k_in <= 2048, k_out <= 256.
 */
int thr_merge_topk(thr_handle* h, const double* scores, const int64_t* ids,
                   const int32_t* counts, int G, int B, int k_in, int k_out,
                   double* out_scores, int64_t* out_ids, int32_t* out_count, void* stream);

/* ---- K5 around the product's exchange step (one all-gather per batch) -------------
 * A rank's message is [scores f64 2*B*k | ids i64 2*B*k | counts i32 2*B] bytes, k = max(k_sem, k_lex):
 * row block 0 = the rank's semantic lists (thr_dense_topk output), block 1 = its lexical lists
 * (thr_bm25_topk output), padded with (-inf, -1).  thr_exchange_pack writes it in one launch;
 * thr_exchange_merge consumes the all-gathered buffer [G][msg bytes] and writes both channels' merged
 * lists in the formats thr_dense_topk / thr_bm25_topk use, so thr_fuse runs on them unchanged.
 * New with sharding (SURVEY.md 8e); same ordering as thr_merge_topk: (score desc, id asc).  Every rank's lists must
 * arrive in that order (thr_dense_topk and thr_bm25_topk write them so): the merge places an entry at its position
 * in its own list plus the number of entries that precede it in the other ranks' lists (binary searches), it does
 * not sort.  G <= 64.
 */
int64_t thr_exchange_msg_bytes(int B, int k_sem, int k_lex);
int thr_exchange_pack(thr_handle* h, const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                      const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt, int B, int k_sem,
                      int k_lex, void* msg, void* stream);
int thr_exchange_merge(thr_handle* h, const void* gathered, int G, int B, int k_sem, int k_lex,
                       int64_t* d_ids, double* d_sc, int32_t* d_cnt, int64_t* l_ids, float* l_sc,
                       int32_t* l_cnt, void* stream);

/* The same exchange over peer memory, without a collective call: thr_exchange_push packs this rank's message
 * and stores it straight into slot `rank` of EVERY rank's gathered buffer (peer_bufs [G] device array of the
 * ranks' buffer bases in this process' address space, e.g. torch symmetric memory; + buf_off bytes), then raises
 * this rank's entry of every rank's signal array (peer_signals [G] bases + sig_off bytes, uint64 [G], zero
 * before the first step) to `seq` with release semantics at system scope.  done_counter: a zero-initialised
 * uint32 on the device, owned by the caller.  thr_exchange_merge_pushed is thr_exchange_merge that first waits
 * (acquire, bounded by a 60 s watchdog -> THR_ETIMEOUT) until signals[g] >= seq for every g.  seq grows by one
 * per step; alternate two buffer halves (buf_off) between consecutive steps so that a fast rank's next push
 * cannot overwrite a message a slow rank is still merging.
 */
int thr_exchange_push(thr_handle* h, const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                      const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt, int B, int k_sem,
                      int k_lex, void* const* peer_bufs, int64_t buf_off, uint64_t* const* peer_signals,
                      int64_t sig_off, int rank, int G, uint64_t seq, uint32_t* done_counter, void* stream);
int thr_exchange_merge_pushed(thr_handle* h, const void* gathered, const uint64_t* signals, uint64_t seq,
                              int G, int B, int k_sem, int k_lex, int64_t* d_ids, double* d_sc,
                              int32_t* d_cnt, int64_t* l_ids, float* l_sc, int32_t* l_cnt, void* stream);

/* ---- in-process sharding: one index over several handles (ShardedSearcher) -------------
 * thr_shard_merge: the merge step of a sharded search in ONE process, without a message: the home handle reads every
 * shard's K1 / K2 outputs where they are (peer memory, or local copies) through device arrays of pointers:
 *   semantic sources s < S_sem: d_ids_src[s] [B, k_sem] int64, d_sc_src[s] [B, k_sem] double, d_cnt_src[s] [B] int32,
 *     d_gap_src[s] [B] float (nullable table when d_gap is NULL) — thr_dense_topk outputs;
 *   lexical sources s < S_lex: l_ids_src[s] [B, k_lex] int64, l_sc_src[s] [B, k_lex] float, l_cnt_src[s] [B] int32 —
 *     thr_bm25_topk outputs (a shard with a lexical delta segment contributes two sources).
 * Outputs, on the handle's GPU, are both channels' merged lists in exactly the formats thr_dense_topk /
 * thr_bm25_topk write (thr_fuse runs on them unchanged), ordered by (score desc, id asc), placed by rank as
 * thr_exchange_merge does; d_gap [B] (nullable) = min over the semantic sources' gaps, the certificate of the merged
 * list (the global top-k is a subset of the union of exact per-shard top-k lists).  One launch for both channels;
 * each row's lists are staged in shared memory with coalesced loads before any search.
 * 1 <= S_sem, S_lex <= 64, 1 <= k <= 256; THR_EUNSUPPORTED when S * k of a channel exceeds 12288.  Timed in the
 * THR_PROF_MERGE slot.
 *
 * thr_rerank_finish_shards: thr_rerank_finish on the element-wise max of S raw [B, C] float arrays (raws: device
 * array of S pointers; exactly one shard scores a candidate, the others report -inf).  S == 1 is bit-identical to
 * thr_rerank_finish.  Replaces the all-reduce(MAX) of the multi-process stage.  Timed in THR_PROF_RERANK.
 */
int thr_shard_merge(thr_handle* h, int B, int k_sem, int k_lex, int S_sem, const int64_t* const* d_ids_src,
                    const double* const* d_sc_src, const int32_t* const* d_cnt_src, const float* const* d_gap_src,
                    int S_lex, const int64_t* const* l_ids_src, const float* const* l_sc_src,
                    const int32_t* const* l_cnt_src, int64_t* d_ids, double* d_sc, int32_t* d_cnt, float* d_gap,
                    int64_t* l_ids, float* l_sc, int32_t* l_cnt, void* stream);
int thr_rerank_finish_shards(thr_handle* h, int B, int C, int stride, const int64_t* ids, const double* rrf,
                             const int32_t* count, const float* const* raws, int S, int Tq, double threshold,
                             double alpha, int top_k, int64_t* out_ids, double* out_rerank, double* out_rrf,
                             uint8_t* out_keep, int32_t* out_n, uint8_t* refused, double* max_score, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* THR_H_ */
