// bm25.cu — K2: BM25 top-k over a CSR inverted index with per-term range skips (lexical channel).
//
// Stands where RAG2Retriever._lexical_search calls the rag2_lexical_search RPC
//   (src/voice_agent/rag2/retrieval.py:273-292, database/migrations/20260114_rag2_schema.sql:341-374):
//   same interface (keyword list in, top-`limit` by descending score out); the scoring formula is
//   BM25 as BASELINE.json's north_star asks.  Definition (oracle/bm25.py restates it on the CPU):
//     score(d) = fp32 sum, over the query's terms in order, of  idf[t] * impact(t, d)
//   with fp32 round-to-nearest multiply and add and no FMA contraction, so the result does not
//   depend on scheduling; docs with score > 0 are ranked by (score desc, id asc).
//
// Index (include/thr.h): postings {u32 doc, f32 impact} in term-major CSR order (doc ascending inside
// a term) and skip[t * n_blk + r] = first posting of term t whose doc lies in range r (blk_docs docs).
//
// Launch sequence of thr_bm25_topk: bm25_plan_kernel (cost per query, cut queries into units = doc-range slices of
// about equal cost, order them heaviest first) -> bm25_range_kernel (one unit at a time per CTA, fetched
// dynamically; writes each unit's sorted top-k) -> bm25_merge_kernel (per query, merge its units' lists).
//
// bm25_range_kernel (round 2; DESIGN.md §4/§8 has the measurements that led here).  The round-1 kernel let a
// CTA own a 30720-doc accumulator and sent every consumer warp through every chunk of postings: ~970 M warp
// instructions per 10M-doc batch, most of them barrier/poll/scan overhead.  Here a WARP owns one skip range
// (blk_docs docs, one fp32 slot per doc in shared memory) at a time and nothing is shared between warps on
// the hot path:
//   * lane t <-> query term t loads the range's two skip entries; a term's postings inside the range are one
//     contiguous piece, read straight from global memory (coalesced 8-byte loads, kDepth chunks of 32 in
//     flight per warp, L2 prefetch two ranges ahead) — no staging ring, no mbarriers, no producer warp;
//   * terms are added in query order by the owning warp (docs of one term are distinct: no atomics; only
//     __syncwarp between chunks), so the fp32 sum is the definition's;
//   * there is no scan of the accumulator: an add that takes a slot across the running threshold tau
//     (old <= tau < new; contributions are >= 0, so exactly one add per qualifying doc does) remembers the doc in
//     a register, the final scores of those docs are read back after the last term, and the range is cleared
//     with 16-byte stores.  A lane that crosses twice in one range, or tau == 0, falls back to scanning the
//     warp's own slots (the warm-up of a unit, and queries with fewer than k hits);
//   * candidates go to a per-warp list in global memory (appends are rare once tau has converged); tau is
//     shared per CTA and tracked by a 256-bin histogram of candidate scores (a warp walks it after it
//     appended: the k-th best candidate's bin edge is a lower bound of the final k-th score), exact
//     warp-level sort-select only when a list stays long after filtering (massive ties); units of one query on
//     different CTAs exchange tau through one global word.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kMaxTerms = 32;                    // lanes of a warp: one per query term
constexpr int kMaxBlkDocs = 2048;                // largest skip range
constexpr int kMaxSelB = 256;                    // largest k

struct Posting { uint32_t doc; float imp; };

// A work unit: one query restricted to the doc ranges [r0, r1).
struct Unit { int q; int r0; int r1; unsigned cost; };
constexpr int kMaxUnitsPerQuery = 64;    // small batches: one query can still spread over many SMs

struct Bm25Args {
  const int64_t* skip;    // [V * n_blk + 1]
  const Posting* post;
  const float* idf;
  int64_t n_docs;
  int n_blk, blk_docs, blk_shift, V;
  const int32_t* q_terms;
  const int32_t* q_off;
  const int32_t* order;   // work units, heaviest first
  const Unit* units;
  const int* total_units;
  int* work_counter;
  int B, k;
  uint64_t* part_keys;    // [max_units][k] sorted descending
  int32_t* part_cnt;      // [max_units]
  const uint16_t* tags;   // [n_docs] nullable: per-doc tag (collection id) for filtered queries
  const int32_t* want;    // [B] nullable: tag a query's docs must carry, < 0 = any
  const uint32_t* deleted;  // [ceil(n_docs / 32)] nullable: bit d % 32 of word d / 32 set = doc d is deleted
  uint64_t* wlists;       // [grid][warps][kListCap] per-warp candidate lists
  unsigned* tau_q;        // [B] running threshold per query (fp32 bits of a score >= 0), shared by its units
  int require_all;        // AND semantics: a doc must contain every (distinct, known) query term
  thr_dev_status* status;
};

// ------------------------------------------------------------------------------------------------
constexpr int kListCap = 1024;       // entries of a warp's candidate list (global memory)
constexpr int kListHigh = 512;       // compaction watermark after a range in crossing mode
constexpr int kListRoom = 384;       // a compaction leaves at most this many entries (>= kMaxSelB)
constexpr int kDepth = 4;            // posting chunks (32 postings each) in flight per warp
#ifndef THR_BM25_DESC_CAP
#define THR_BM25_DESC_CAP 64
#endif
#ifndef THR_BM25_GRAB
#define THR_BM25_GRAB 4
#endif
constexpr int kDescCap = THR_BM25_DESC_CAP;   // piece descriptors per warp (16 B each): >= kMaxTerms + kDepth - 1
constexpr int kGrab = THR_BM25_GRAB;          // consecutive ranges a warp takes from its unit at a time
static_assert(kDescCap >= kMaxTerms + kDepth - 1 && (kDescCap & (kDescCap - 1)) == 0,
              "the descriptor ring holds at least a range of a 32-term query and is a power of two");
// Generation tags: a slot holds {2-bit generation tag, 30-bit fp32 pattern of the SCALED partial sum}.  All scores of
// a range are accumulated multiplied by 2^-40 (idf is scaled once per unit; a power-of-two factor commutes with every
// fp32 rounding as long as nothing under- or overflows, so the final score times 2^40 is bit-identical to the unscaled
// sum): scaled sums stay below 2.0, so bits 31 and 30 of their patterns are free.  A range stamps the slots it writes
// with its generation (range count of this warp modulo 4); a slot whose tag is another generation reads as 0, so the
// 8 KB of a warp's accumulator are cleared once per FOUR ranges instead of after every range — clearing was 64 of the
// ~155 shared-memory wavefronts per range, on the pipe that limits this kernel (DESIGN.md §8).
// Requirements (checked when the index is set): idf == 0 or 2^-40 <= idf <= 2^20; impacts are BM25's (< k1 + 1).
constexpr float kAccScale = 9.094947017729282e-13f;   // 2^-40
constexpr float kAccUnscale = 1099511627776.f;         // 2^40
constexpr uint32_t kAccMask = 0x3fffffffu;
constexpr int kHistBins = 256;
constexpr int kHistShift = 19;                 // 16 bins per octave
constexpr uint32_t kHistBase = 121u << 4;      // bin 0 starts at 2^-6 (everything smaller lands there too)
static_assert(kListRoom >= kMaxSelB && kListCap - kListRoom >= 128 + 32, "list head-room");

struct RangeShared {
  uint32_t hist[kHistBins];    // candidate scores of the current unit
  uint32_t hist2[256];         // radix-select scratch of the unit's final merge
  unsigned tau_bits;           // the unit's running threshold (bits of a float >= 0)
  int next_range;
  int unit;
  int lock;                    // guards `scratch` during a warp's exact sort-select
  int n_total;                 // unit end: candidates that survive the final threshold
  int n_out;
  int want_sel;
  unsigned long long prefix;
};

__device__ __forceinline__ int tau_bin(uint32_t score_bits) {
  const int b = (int)(score_bits >> kHistShift) - (int)kHistBase;
  return min(max(b, 0), kHistBins - 1);
}
__device__ __forceinline__ uint32_t key_bits(uint64_t key) { return (uint32_t)(key >> 32) & 0x7fffffffu; }

// Lower bound of the k-th best candidate score seen by the CTA so far, from the histogram: the lower edge of
// the bin that holds the k-th best, minus one ulp (so that ties with the edge survive the strict filter).
// 0 when the histogram holds fewer than k candidates or the k-th lies in the catch-all bin 0.  Warp-collective.
__device__ __forceinline__ uint32_t hist_tau(const uint32_t* hist, int k, int lane) {
  int d = 0, above = 0;
  const bool mine = radix_find_digit(hist, k, lane, &d, &above);
  uint32_t t = 0;
  if (mine && d >= 1) t = ((uint32_t)(d + (int)kHistBase) << kHistShift) - 1u;
  return __reduce_max_sync(0xffffffffu, t);
}

// Keep the entries whose score is > tau, in place and in order.  Warp-collective; returns the new length.
__device__ int list_filter(uint64_t* list, int n, uint32_t tau_bits, int lane) {
  int out = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    const uint64_t key = i < n ? __ldcg(list + i) : 0ull;
    const bool keep = i < n && key_bits(key) > tau_bits;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) __stcg(list + out + __popc(m & ((1u << lane) - 1u)), key);
    out += __popc(m);
  }
  __syncwarp();
  return out;
}

// Exact: sort the list (descending keys = score desc, id asc) in the CTA's scratch and keep the k best.
// Returns the new length; *tau_out = one ulp below the k-th best score (0 if the list is shorter than k).
__device__ int list_select(uint64_t* list, int n, int k, uint64_t* scratch, int* lock, int lane, uint32_t* tau_out) {
  if (lane == 0) {
    while (atomicCAS(lock, 0, 1) != 0) __nanosleep(200);
  }
  __syncwarp();
  int P = 32, lg = 5;
  while (P < n) { P <<= 1; ++lg; }
  for (int i = lane; i < P; i += 32) scratch[i] = i < n ? __ldcg(list + i) : 0ull;
  __syncwarp();
  for (int ls = 1; ls <= lg; ++ls) {          // size = 1 << ls
    for (int lt = ls - 1; lt >= 0; --lt) {    // stride = 1 << lt
      const int stride = 1 << lt;
      for (int i = lane; i < (P >> 1); i += 32) {
        const int lo = ((i >> lt) << (lt + 1)) | (i & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo >> ls) & 1) == 0;
        const uint64_t x = scratch[lo], y = scratch[hi];
        if (desc ? (y > x) : (x > y)) { scratch[lo] = y; scratch[hi] = x; }
      }
      __syncwarp();
    }
  }
  const int m = min(n, k);
  for (int i = lane; i < m; i += 32) __stcg(list + i, scratch[i]);
  *tau_out = n >= k ? key_bits(scratch[k - 1]) - 1u : 0u;
  __syncwarp();
  if (lane == 0) { __threadfence_block(); atomicExch(lock, 0); }
  __syncwarp();
  return m;
}

// kAnd: AND semantics (thr_bm25_topk_ex with THR_BM25_REQUIRE_ALL) — a second per-doc array counts the terms that
// hit the doc; only docs hit by every distinct known term of the query are candidates.
template <int kBlk, bool kAnd>
__global__ void __launch_bounds__(kBlk == 2048 ? 768 : 1024, 1) bm25_range_kernel(const Bm25Args a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 127u) & ~127u;
  uint8_t* sm0 = smem_raw + (base - smem_u32(smem_raw));
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  float* acc_all = (float*)sm0;                                        // [nw][kBlk]
  uint8_t* hit_all = (uint8_t*)(acc_all + (size_t)nw * kBlk);          // [nw][kBlk] matched-term counts (kAnd)
  uint64_t* scratch = (uint64_t*)(hit_all + (kAnd ? (size_t)nw * kBlk : 0));   // [kListCap]
  uint8_t* desc_all = (uint8_t*)(scratch + kListCap);                  // [nw][kDescCap] 16-byte piece descriptors
  RangeShared* sh = (RangeShared*)(desc_all + (size_t)nw * kDescCap * 16);
  volatile RangeShared* vsh = sh;

  for (int i = tid; i < nw * kBlk; i += blockDim.x) acc_all[i] = 0.f;
  if (kAnd)
    for (int i = tid; i < nw * kBlk / 4; i += blockDim.x) ((uint32_t*)hit_all)[i] = 0u;
  for (int i = tid; i < kHistBins; i += blockDim.x) sh->hist[i] = 0u;
  if (tid == 0) { sh->lock = 0; sh->n_total = 0; sh->n_out = 0; }
  // Shared-window addresses used on the hot path, made opaque so that the compiler keeps them in registers instead
  // of re-deriving them from the window base at every use (measured: 34 instructions per range).
  uint32_t acc_u = smem_u32(acc_all + (size_t)warp * kBlk);            // this warp's accumulator
  uint32_t hit_u = smem_u32(hit_all + (kAnd ? (size_t)warp * kBlk : 0));
  uint32_t tau_u = smem_u32(&sh->tau_bits);
  asm volatile("" : "+r"(acc_u), "+r"(hit_u), "+r"(tau_u));
  uint64_t* const list = a.wlists + ((size_t)blockIdx.x * nw + warp) * kListCap;
  uint32_t gen = 0;     // generation of the range this warp works on (all slots are 0 = generation 0, value 0 at start)
  const unsigned lt_mask = (1u << lane) - 1u;
  constexpr int kShift = kBlk == 2048 ? 11 : kBlk == 1024 ? 10 : kBlk == 512 ? 9 : 8;
  static_assert((1 << kShift) == kBlk, "kBlk must be 256, 512, 1024 or 2048");

  for (;;) {
    __syncthreads();
    if (tid == 0) {
      const int w = atomicAdd(a.work_counter, 1);
      const int u = w < *a.total_units ? a.order[w] : -1;
      sh->unit = u;
      if (u >= 0) {
        sh->next_range = a.units[u].r0;
        sh->tau_bits = *(volatile unsigned*)&a.tau_q[a.units[u].q];
      }
    }
    __syncthreads();
    const int unit = vsh->unit;
    if (unit < 0) break;
    const int q = a.units[unit].q, r0 = a.units[unit].r0, r1 = a.units[unit].r1;
    const int qlo = a.q_off[q];
    const int nt = min(a.q_off[q + 1] - qlo, kMaxTerms);   // longer queries are reported by bm25_cost_kernel
    int term = -1;
    float wgt = 0.f;
    if (lane < nt) {
      term = a.q_terms[qlo + lane];
      if (term < 0 || term >= a.V) term = -1; else wgt = a.idf[term] * kAccScale;   // exact: a power of two
    }
    int need = 0;      // AND semantics: distinct known terms of the query; an unknown term -> no doc can match
    bool and_dead = false;
    if (kAnd) {
      bool dup = false;
      for (int u = 0; u < nt; ++u) {
        const int tu = __shfl_sync(0xffffffffu, term, u);
        if (u < lane && tu == term) dup = true;
      }
      need = __popc(__ballot_sync(0xffffffffu, term >= 0 && !dup));
      and_dead = __any_sync(0xffffffffu, lane < nt && term < 0) || need == 0;
      if (dup) term = -1;       // a repeated keyword counts once (plainto_tsquery builds a set of lexemes)
    }
    const int want = (a.tags && a.want) ? a.want[q] : -1;
    const bool any_term = __any_sync(0xffffffffu, term >= 0) && !and_dead;
    const int64_t* row = a.skip + (size_t)(term < 0 ? 0 : term) * a.n_blk;
    int n_list = 0;

    // Walk the histogram, raise the CTA's threshold, tell the query's other units.
    auto raise_tau = [&]() {
      const uint32_t tb = hist_tau(sh->hist, a.k, lane);
      if (lane == 0 && tb > vsh->tau_bits) {
        atomicMax(&sh->tau_bits, tb);
        atomicMax(&a.tau_q[q], tb);
      }
      __syncwarp();
    };
    // Make room in this warp's list: drop what the threshold has overtaken; if the list is still long (ties,
    // or a threshold that cannot rise because the query has few hits) select its k best exactly.
    auto compact = [&]() {
      raise_tau();
      n_list = list_filter(list, n_list, vsh->tau_bits, lane);
      if (n_list > kListRoom) {
        uint32_t tw = 0;
        n_list = list_select(list, n_list, a.k, scratch, &sh->lock, lane, &tw);
        if (lane == 0 && tw > vsh->tau_bits) {
          atomicMax(&sh->tau_bits, tw);
          atomicMax(&a.tau_q[q], tw);
        }
        __syncwarp();
      }
    };
    // Append the lanes' candidates (has) to the list; room for 32 entries is the caller's invariant.  Every candidate
    // passes here, so the tag filter acts on all of them.  The deletion bitmap is tested by the two callers (a test
    // here costs the AND instantiations spills: the slow scan reads one word for a lane's four docs); either way a
    // deleted doc never enters a list, and the threshold (the histogram of appended scores) is learnt from live docs.
    auto append = [&](bool has, float score, uint32_t doc) {
      if (has && want >= 0) has = (int)__ldg(a.tags + doc) == want;
      const unsigned m = __ballot_sync(0xffffffffu, has);
      if (m) {
        if (has) {
          __stcg(list + n_list + __popc(m & lt_mask), pack_key(score, doc));
          atomicAdd(&sh->hist[tau_bin(__float_as_uint(score))], 1u);
        }
        n_list += __popc(m);
      }
    };

    // ---- the unit's posting stream ------------------------------------------------------------------------
    // Two levels.  refill(): lane t <-> query term t turns the next grab of ranges into piece descriptors in a per-warp
    // RING in shared memory — one per (range, term with postings there), in range then query order:
    // {pointer to the piece's first posting, postings | first-of-range flag + range, idf} — all terms of a range at
    // once (ballot + popc give the slots).  A range is padded with empty descriptors to a multiple of kDepth chunks,
    // so its first chunk always lands in buffer 0 of the pipeline below.  The ring is refilled at range boundaries
    // whenever a whole grab fits, so the loader normally never runs out of descriptors and the register pipeline
    // does not drain between grabs (round 2's first descriptor version rebuilt a LIST when the previous one was used
    // up: 34 % of the samples sat on the first add after every rebuild).
    // Stream: kDepth chunks of <= 32 postings are in flight in registers; buffer j holds bn[j] postings of one
    // piece (lane < bn[j] has one), weight bw[j]; an empty chunk (bn <= 0) is a no-op for the adds.
    // descriptor word z: postings of the piece (bits 0-12, <= 2048); on a range's first piece also kNewRange | range << 14
    constexpr int kNewRange = 1 << 13;
    constexpr int kRangeShift = 14;
    const uint32_t tb_lo = term >= 0 ? (uint32_t)__ldg(row) : 0u;          // low word of the term's first posting index
    const Posting* const tp = a.post + (term >= 0 ? __ldg(row) : 0);       // the term's first posting
    uint32_t desc_u = smem_u32(desc_all + (size_t)warp * kDescCap * 16);
    asm volatile("" : "+r"(desc_u));
    const int per_range = __popc(__ballot_sync(0xffffffffu, term >= 0)) + kDepth - 1;   // most descriptors a range takes
    // a grab: gsz consecutive ranges, handed out by the unit's atomic counter; a grab always fits half the ring
    const int gsz = max(1, min(min(kGrab, (kDescCap / 2) / per_range), max(1, (r1 - r0) / (nw * 8))));
    const int grab_max = gsz * per_range;
    int np = 0, pi = 0;              // descriptors appended / fetched so far (ring positions are these modulo kDescCap)
    auto reserve = [&]() -> int {    // the next grab's first range (>= r1: the unit's ranges are used up)
      int lo_ = 0;
      if (lane == 0) lo_ = atomicAdd(&sh->next_range, gsz);
      lo_ = __shfl_sync(0xffffffffu, lo_, 0);
      if (term >= 0 && lo_ < r1) {   // its skip entries -> L2 (two sectors hold a term's gsz + 1 entries)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(row + lo_));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(row + min(lo_ + gsz, a.n_blk)));
      }
      return lo_;
    };
    int next_lo = any_term ? reserve() : r1;
    auto refill = [&]() {            // descriptors of the grab at next_lo -> ring; reserves the grab after it
      const int lo_ = next_lo;
      uint32_t e[kGrab + 1];         // skip entries of [lo_, lo_ + kGrab] relative to the term's first posting
#pragma unroll
      for (int i = 0; i <= kGrab; ++i)
        e[i] = term >= 0 ? __ldg((const uint32_t*)(row + min(lo_ + i, a.n_blk))) - tb_lo : 0u;
      next_lo = reserve();
      if (lane == 0) {
        const unsigned gt = *(volatile unsigned*)&a.tau_q[q];   // what the query's other units have learnt
        if (gt > vsh->tau_bits) atomicMax(&sh->tau_bits, gt);
      }
#pragma unroll
      for (int i = 0; i < kGrab; ++i) {
        const int r = lo_ + i;
        if (i < gsz && r < r1) {
          const int cnt = (int)(e[i + 1] - e[i]);
          unsigned live = __ballot_sync(0xffffffffu, cnt > 0);
          if (kAnd && __popc(live) < need) live = 0;   // a term without postings here: no doc of the range matches
          if (live) {
            const int nch = cnt > 0 ? (cnt + 31) >> 5 : 0;
            const int tot = __reduce_add_sync(0xffffffffu, nch);
            if (cnt > 0) {
              const Posting* pp = tp + e[i];
              const bool first = (live & lt_mask) == 0u;
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};"
                           ::"r"(desc_u + (uint32_t)((np + __popc(live & lt_mask)) & (kDescCap - 1)) * 16u),
                           "r"((uint32_t)(uintptr_t)pp), "r"((uint32_t)((uintptr_t)pp >> 32)),
                           "r"((uint32_t)cnt | (first ? ((uint32_t)kNewRange | ((uint32_t)r << kRangeShift)) : 0u)),
                           "r"(__float_as_uint(wgt))
                           : "memory");
            }
            np += __popc(live);
            const int pad = (-tot) & (kDepth - 1);
            if (lane < pad)
              asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(desc_u + (uint32_t)((np + lane) & (kDescCap - 1)) * 16u), "r"(0u)
                           : "memory");
            np += pad;
          }
        }
      }
      __syncwarp();
    };

    int lrem = 0, flag0 = 0;
    const Posting* lbase = a.post;   // the piece being streamed, the lane's next posting in it, postings left (<= 0: none)
    uint32_t loff = 0;
    float lw = 0.f;
    uint32_t bd[kDepth], bi[kDepth];
    float bw[kDepth];
    int bn[kDepth];
    // Buffer j's next chunk: the next 32 postings of the current piece, or of the next descriptor's piece.  Branch-free
    // apart from the descriptor fetch: with no piece left the chunk is empty (bn <= 0, no lane loads).
#define THR_ISSUE(j)                                                                                     \
  {                                                                                                      \
    if ((j) == 0) flag0 = 0;                                                                             \
    if (lrem <= 0 && pi < np) {                                                                          \
      uint32_t x_, y_, z_, w_;                                                                           \
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"                                            \
                   : "=r"(x_), "=r"(y_), "=r"(z_), "=r"(w_)                                              \
                   : "r"(desc_u + (uint32_t)(pi & (kDescCap - 1)) * 16u));                               \
      ++pi;                                                                                              \
      lbase = (const Posting*)(((unsigned long long)y_ << 32) | x_);                                     \
      loff = (uint32_t)lane;                                                                             \
      lrem = (int)(z_ & (uint32_t)(kNewRange - 1));                                                      \
      if ((j) == 0) flag0 = (int)(z_ >> 13);     /* != 0 on a range's first piece: flag | range << 1 */   \
      lw = __uint_as_float(w_);                                                                          \
    }                                                                                                    \
    bn[j] = lrem;                                                                                        \
    bw[j] = lw;                                                                                          \
    asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.s32 p, %2, %3;\n\t"                                      \
                 "@p ld.global.nc.v2.u32 {%0, %1}, [%4];\n\t}"                                           \
                 : "+r"(bd[j]), "+r"(bi[j])                                                              \
                 : "r"(lane), "r"(lrem), "l"(lbase + loff));                                             \
    loff += 32u;                                                                                         \
    lrem -= 32;                                                                                          \
  }

    // Adds of one chunk: predicated straight-line code (an empty chunk, bn = 0, is a no-op).  ncross / cross_doc:
    // the lane's threshold crossings.  The slot of doc d of the range starting at doc0 is acc0 + 4 d with
    // acc0 = &acc[0] - 4 doc0 (mod 2^32).
#define THR_ADD(j)                                                                                       \
  {                                                                                                      \
    asm volatile(                                                                                        \
        "{\n\t.reg .pred p, c, g;\n\t.reg .f32 o, n, x;\n\t.reg .u32 ad, v, t;\n\t"                      \
        "setp.lt.s32 p, %2, %3;\n\t"                                                                     \
        "mad.lo.u32 ad, %4, 4, %5;\n\t"                                                                  \
        "mov.u32 v, 0;\n\t"                                                                              \
        "@p ld.shared.u32 v, [ad];\n\t"                                                                  \
        "and.b32 t, v, 0xc0000000;\n\t"            /* the slot's generation tag */                       \
        "setp.eq.u32 g, t, %9;\n\t"                                                                      \
        "and.b32 v, v, 0x3fffffff;\n\t"                                                                  \
        "selp.u32 v, v, 0, g;\n\t"                 /* another generation's value reads as 0 */           \
        "mov.b32 o, v;\n\t"                                                                              \
        "mul.rn.f32 x, %6, %7;\n\t"                                                                      \
        "add.rn.f32 n, o, x;\n\t"                                                                        \
        "mov.b32 v, n;\n\t"                                                                              \
        "or.b32 v, v, %9;\n\t"                                                                           \
        "@p st.shared.u32 [ad], v;\n\t"                                                                  \
        "setp.gt.and.f32 c, n, %8, p;\n\t"                                                               \
        "setp.le.and.f32 c, o, %8, c;\n\t"                                                               \
        "@c add.s32 %0, %0, 1;\n\t"                                                                      \
        "@c mov.u32 %1, %4;\n\t}"                                                                        \
        : "+r"(ncross), "+r"(cross_doc)                                                                  \
        : "r"(lane), "r"(bn[j]), "r"(bd[j]), "r"(acc0), "f"(bw[j]), "f"(__uint_as_float(bi[j])), "f"(tau_s),        \
          "r"(gtag)                                                                                      \
        : "memory");                                                                                     \
    if (kAnd) {                                                                                          \
      asm volatile(                                                                                      \
          "{\n\t.reg .pred p;\n\t.reg .u32 h, ad;\n\t"                                                   \
          "setp.lt.s32 p, %0, %1;\n\t"                                                                   \
          "add.u32 ad, %2, %3;\n\t"                                                                      \
          "@p ld.shared.u8 h, [ad];\n\t"                                                                 \
          "@p add.u32 h, h, 1;\n\t"                                                                      \
          "@p st.shared.u8 [ad], h;\n\t}"                                                                \
          :                                                                                              \
          : "r"(lane), "r"(bn[j]), "r"(bd[j]), "r"(hit0)                                                 \
          : "memory");                                                                                   \
    }                                                                                                    \
  }

    static_assert(kDepth == 4, "the pipeline below is unrolled by hand for four buffers");
#pragma unroll
    for (int j = 0; j < kDepth; ++j) { bd[j] = 0u; bi[j] = 0u; bn[j] = 0; bw[j] = 0.f; }
    for (;;) {   // one range per iteration, its first chunk in buffer 0
      // keep the ring ahead of the loader: append grabs while a whole one fits (usually none or one per iteration)
      while (next_lo < r1 && (np - pi) + grab_max <= kDescCap) refill();
      if (bn[0] <= 0) {                 // the pipeline is empty: the unit's start, or its ranges are used up
        if (pi >= np) break;
        THR_ISSUE(0) THR_ISSUE(1) THR_ISSUE(2) THR_ISSUE(3)
      }
      const uint32_t doc0 = (uint32_t)(flag0 >> 1) << kShift;     // flag0 = 1 | range << 1 on a range's first chunk
      const uint32_t acc0 = acc_u - doc0 * 4u, hit0 = hit_u - doc0;
      float tau;
      asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(tau) : "r"(tau_u));
      const float tau_s = tau * kAccScale;                         // the threshold in the accumulator's scale (exact)
      const uint32_t gtag = gen << 30;                             // this range's generation tag
      int ncross = 0;
      uint32_t cross_doc = 0xffffffffu;
      do {
        THR_ADD(0) THR_ISSUE(0)
        THR_ADD(1) THR_ISSUE(1)
        THR_ADD(2) THR_ISSUE(2)
        THR_ADD(3) THR_ISSUE(3)
      } while (bn[0] > 0 && !flag0);   // until buffer 0 starts another range (or is empty: no descriptor was left)
      __syncwarp();
      // ---- the range is complete: collect its candidates, clear its slots ----
      const bool scan = tau <= 0.f || __any_sync(0xffffffffu, ncross > 1);
      int appended = 0;
      if (!scan) {
        const unsigned cm = __ballot_sync(0xffffffffu, cross_doc != 0xffffffffu);
        if (cm) {
          float v = 0.f;
          uint32_t hc = (uint32_t)need;
          if (cross_doc != 0xffffffffu) {
            uint32_t vb;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(vb) : "r"(acc0 + cross_doc * 4u));
            v = __uint_as_float(vb & kAccMask) * kAccUnscale;      // written in this range: the tag is gtag
            if (kAnd) asm volatile("ld.shared.u8 %0, [%1];" : "=r"(hc) : "r"(hit0 + cross_doc));
          }
          const int before = n_list;
          append(cross_doc != 0xffffffffu && v > tau && (!kAnd || hc == (uint32_t)need) &&
                     !(a.deleted && ((__ldg(a.deleted + (cross_doc >> 5)) >> (cross_doc & 31u)) & 1u)),
                 v, cross_doc);
          appended = n_list - before;
        }
      } else {
        // Slow path (a unit's warm-up; queries with fewer than k hits): test every slot of the range.
        const int before = n_list;
        for (int j = 0; j < kBlk / 128; ++j) {
          if (n_list > kListCap - 128 - 32) compact();
          const float tcur = __uint_as_float(vsh->tau_bits);
          uint32_t v[4];
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                       : "r"(acc_u + (uint32_t)(j * 32 + lane) * 16u));
#pragma unroll
          for (int c = 0; c < 4; ++c) v[c] = (v[c] & ~kAccMask) == gtag ? (v[c] & kAccMask) : 0u;
          const uint32_t m = max(max(v[0], v[1]), max(v[2], v[3]));
          uint32_t hc4 = 0u;
          if (kAnd) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(hc4) : "r"(hit_u + (uint32_t)(j * 32 + lane) * 4u));
          if (__any_sync(0xffffffffu, m != 0u)) {
            // the lane's four docs share a bitmap word; docs past n_docs (the last range's tail) have none
            const uint32_t doc4 = doc0 + (uint32_t)(j * 32 + lane) * 4u;
            const uint32_t dead4 = a.deleted && doc4 < a.n_docs ? __ldg(a.deleted + (doc4 >> 5)) >> (doc4 & 31u) : 0u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float x = __uint_as_float(v[c]) * kAccUnscale;
              const bool all = !kAnd || ((hc4 >> (8 * c)) & 255u) == (uint32_t)need;
              append(x > tcur && x > 0.f && all && !((dead4 >> c) & 1u), x, doc4 + c);
            }
          }
        }
        appended = n_list - before;
      }
      __syncwarp();
      gen = (gen + 1u) & 3u;
      if (gen == 0u) {      // the tags wrap: clear the accumulator (once per four ranges)
#pragma unroll
        for (int j = 0; j < kBlk / 128; ++j)
          asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(acc_u + (uint32_t)(j * 32 + lane) * 16u), "r"(0u)
                       : "memory");
      }
      if (kAnd) {
#pragma unroll
        for (int j = 0; j < kBlk / 128; ++j)
          asm volatile("st.shared.b32 [%0], %1;" ::"r"(hit_u + (uint32_t)(j * 32 + lane) * 4u), "r"(0u) : "memory");
      }
      __syncwarp();
      if (appended) {
        if (n_list > kListHigh) compact();
        else raise_tau();
      }
    }
#undef THR_ISSUE
#undef THR_ADD

    // ================= unit end: the CTA's k best =================
    __syncthreads();
    {
      const uint32_t tb = vsh->tau_bits;
      n_list = list_filter(list, n_list, tb, lane);
      if (lane == 0 && n_list) atomicAdd(&sh->n_total, n_list);
    }
    __syncthreads();
    const int n_total = vsh->n_total;
    int n_fin;
    if (n_total <= kMaxSelB) {
      int pos = 0;
      if (lane == 0 && n_list) pos = atomicAdd(&sh->n_out, n_list);
      pos = __shfl_sync(0xffffffffu, pos, 0);
      for (int i = lane; i < n_list; i += 32) scratch[pos + i] = __ldcg(list + i);
      n_fin = n_total;
    } else {
      // radix select of the k-th largest key over the warps' lists (keys are distinct: they carry the doc id)
      if (tid == 0) { sh->prefix = 0ull; sh->want_sel = a.k; }
      for (int pass = 0; pass < 8; ++pass) {
        const int shift = 56 - 8 * pass;
        for (int i = tid; i < 256; i += blockDim.x) sh->hist2[i] = 0u;
        __syncthreads();
        const uint64_t prefix = sh->prefix;
        for (int i = lane; i < n_list; i += 32) {
          const uint64_t key = __ldcg(list + i);
          if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8)))
            atomicAdd(&sh->hist2[(uint32_t)(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {
          const int wsel = sh->want_sel;
          int d, above;
          if (radix_find_digit(sh->hist2, wsel, tid, &d, &above)) {
            sh->want_sel = wsel - above;
            sh->prefix = prefix | ((unsigned long long)d << shift);
          }
        }
        __syncthreads();
      }
      const uint64_t T = sh->prefix;
      for (int i = lane; i < n_list; i += 32) {
        const uint64_t key = __ldcg(list + i);
        if (key >= T) {
          const int pos = atomicAdd(&sh->n_out, 1);
          if (pos < kMaxSelB) scratch[pos] = key;
        }
      }
      n_fin = min(n_total, a.k);
    }
    __syncthreads();
    n_fin = min(n_fin, min(vsh->n_out, kMaxSelB));
    for (int i = n_fin + tid; i < kMaxSelB; i += blockDim.x) scratch[i] = 0ull;
    __syncthreads();
    for (int size = 2; size <= kMaxSelB; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        if (tid < kMaxSelB / 2) {
          const int lo = ((tid / stride) * (stride << 1)) + (tid % stride);
          const int hi = lo + stride;
          const bool desc_block = ((lo & size) == 0);
          const uint64_t x = scratch[lo], y = scratch[hi];
          const bool swap = desc_block ? (y > x) : (x > y);
          if (swap) { scratch[lo] = y; scratch[hi] = x; }
        }
        __syncthreads();
      }
    }
    const int n_keep = min(n_fin, a.k);
    if (tid == 0) a.part_cnt[unit] = n_keep;
    for (int i = tid; i < n_keep; i += blockDim.x) a.part_keys[(size_t)unit * a.k + i] = scratch[i];
    for (int i = tid; i < kHistBins; i += blockDim.x) sh->hist[i] = 0u;
    if (tid == 0) { sh->n_total = 0; sh->n_out = 0; }
  }
}

// df per term; also checks idf >= 0: the kernel relies on a doc's partial sums never decreasing.
__global__ void bm25_df_kernel(const int64_t* skip, const float* idf, int n_blk, int V, int64_t* df,
                               thr_dev_status* status) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= V) return;
  df[t] = skip[(size_t)(t + 1) * n_blk] - skip[(size_t)t * n_blk];
  // idf >= 0 (partial sums never decrease) and, unless 0, within [2^-40, 2^20] (the accumulator's scaled range)
  if (!(idf[t] >= 0.f) || (idf[t] > 0.f && (idf[t] < 9.094947017729282e-13f || idf[t] > 1048576.f)))
    dev_report(status, THR_EINVAL, 461, t);
}

// Single block: cut queries into units of roughly equal cost.  A range costs its postings plus a fixed
// per-range overhead (range_cost postings' worth of work: skip loads, clearing the slots), so light queries are
// split as well.
constexpr unsigned long long kRangeCostDefault = 150;  // list building, clearing and bookkeeping of a range, in postings (~200 instructions at ~1.3 per posting)
constexpr long long kTermCostDefault = 15;             // per (term, range) piece on top of its postings (descriptor + a partly filled chunk)
constexpr int kUnitsPerCtaDefault = 1;   // measured at 10M / 1.25M docs, batch 256: 1 -> 1.13 / 0.22 ms, 2 -> 1.21 / 0.26, 4 -> 1.23 / 0.33
// One launch prepares a batch (round 2: cost, plan and order used to be three launches; at 8 GPUs the fixed
// per-step kernels are what separates the scaling curve from linear): per-query cost -> units -> heaviest first.
constexpr int kPlanStage = 4096;
__global__ void __launch_bounds__(1024) bm25_plan_kernel(const int32_t* q_terms, const int32_t* q_off, const int64_t* df,
                                                          int V, long long term_cost, unsigned long long* keys,
                                                          unsigned* tau_q, thr_dev_status* status, int B, int n_blk,
                                                          int num_slots, unsigned long long kRangeCost,
                                                          Unit* units, int* unit_base,
                                                          int* total_units, int* work_counter, int32_t* order) {
  __shared__ unsigned long long s_tot;
  __shared__ int s_carry;
  __shared__ int s_scan[1024];
  __shared__ unsigned s_cost[kPlanStage];
  const int tid = threadIdx.x;
  if (tid == 0) { s_tot = 0; s_carry = 0; *work_counter = 0; }
  // cost[q] = total postings of the query's terms + term_cost per (term with postings, range): the kernel's time
  // follows the number of (term, range) pieces as well as the number of postings.  Also resets the query's threshold.
  for (int q = tid; q < B; q += 1024) {
    tau_q[q] = 0u;
    // more terms than a warp has lanes for: reported by thr_sync, never silently truncated
    if (q_off[q + 1] - q_off[q] > kMaxTerms) dev_report(status, THR_EINVAL, 460, q);
    long long c = 0;
    const int i_end = q_off[q + 1];
    for (int i0 = q_off[q]; i0 < i_end; i0 += 8) {   // eight terms a time: their loads do not wait for each other
      int t[8];
      long long d[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) t[u] = i0 + u < i_end ? q_terms[i0 + u] : -1;
#pragma unroll
      for (int u = 0; u < 8; ++u) d[u] = (t[u] >= 0 && t[u] < V) ? df[t[u]] : 0;
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (d[u] > 0) c += d[u] + term_cost * n_blk;
    }
    if (c > 0xffffffffll) c = 0xffffffffll;
    keys[q] = ((unsigned long long)c << 32) | (unsigned)(0xffffffffu - (unsigned)q);
  }
  __syncthreads();
  unsigned long long part = 0;
  for (int q = tid; q < B; q += 1024) part += (keys[q] >> 32) + kRangeCost * (unsigned long long)n_blk;
  for (int sh = 16; sh > 0; sh >>= 1) part += __shfl_xor_sync(0xffffffffu, part, sh);
  if ((tid & 31) == 0 && part) atomicAdd(&s_tot, part);   // one shared-memory atomic per warp, not per thread
  __syncthreads();
  unsigned long long target = s_tot / (unsigned long long)num_slots + 1;
  if (target < 16384ull) target = 16384ull;
  for (int q0 = 0; q0 < B; q0 += 1024) {
    const int q = q0 + tid;
    int nu = 0;
    unsigned long long c = 0;
    if (q < B) {
      c = (keys[q] >> 32) + kRangeCost * (unsigned long long)n_blk;
      nu = (int)((c + target - 1) / target);
      if (nu < 1) nu = 1;
      if (nu > kMaxUnitsPerQuery) nu = kMaxUnitsPerQuery;
      if (nu > n_blk) nu = n_blk;
    }
    s_scan[tid] = nu;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {  // inclusive Hillis-Steele scan
      int v = tid >= off ? s_scan[tid - off] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    const int base = s_carry + s_scan[tid] - nu;
    if (q < B) {
      unit_base[q] = base;
      for (int u = 0; u < nu; ++u) {
        Unit x;
        x.q = q;
        x.r0 = (int)((long long)n_blk * u / nu);
        x.r1 = (int)((long long)n_blk * (u + 1) / nu);
        x.cost = (unsigned)min(c / (unsigned long long)nu, 0xffffffffull);
        units[base + u] = x;
      }
    }
    __syncthreads();
    if (tid == 1023) s_carry += s_scan[1023];
    __syncthreads();
  }
  if (tid == 0) { unit_base[B] = s_carry; *total_units = s_carry; }
  __syncthreads();
  // rank sort of the units by cost, heaviest first (a few hundred units; at most B * kMaxUnitsPerQuery)
  const int n = s_carry;
  const bool staged = n <= kPlanStage;   // the costs of a few hundred units: compared out of shared memory
  if (staged) {
    for (int u = tid; u < n; u += 1024) s_cost[u] = units[u].cost;
    __syncthreads();
  }
  for (int u = tid; u < n; u += 1024) {
    const unsigned cu = staged ? s_cost[u] : units[u].cost;
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const unsigned cj = staged ? s_cost[j] : units[j].cost;
      rank += (cj > cu || (cj == cu && j < u)) ? 1 : 0;
    }
    order[rank] = u;
  }
}

// Per query: merge the sorted partial lists of its units -> final top-k.
__global__ void __launch_bounds__(256) bm25_merge_kernel(const uint64_t* part_keys, const int32_t* part_cnt,
                                                         const int* unit_base, int k, int64_t id_base,
                                                         int64_t* out_ids, float* out_scores, int32_t* out_count) {
  extern __shared__ uint64_t keys[];   // next power of two >= kMaxUnitsPerQuery * k
  const int q = blockIdx.x, tid = threadIdx.x;
  const int u0 = unit_base[q], u1 = unit_base[q + 1];
  const int slots = (u1 - u0) * k;
  int P = 32;
  while (P < slots) P <<= 1;
  for (int i = tid; i < P; i += 256) {
    uint64_t key = 0ull;
    if (i < slots) {
      const int u = u0 + i / k, j = i % k;
      if (j < part_cnt[u]) key = part_keys[(size_t)u * k + j];
    }
    keys[i] = key;
  }
  __syncthreads();
  if (u1 - u0 > 1) {   // a single unit's list is already sorted
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < (P >> 1); i += 256) {
          int lo = ((i / stride) * (stride << 1)) + (i % stride);
          int hi = lo + stride;
          bool desc_block = ((lo & size) == 0);
          uint64_t x = keys[lo], y = keys[hi];
          bool swap = desc_block ? (y > x) : (x > y);
          if (swap) { keys[lo] = y; keys[hi] = x; }
        }
        bitonic_stage_sync(size, stride, P, 32);
      }
    }
  }
  int n = 0;
  for (int u = u0; u < u1; ++u) n += part_cnt[u];
  if (n > k) n = k;
  if (tid == 0) out_count[q] = n;
  for (int i = tid; i < k; i += 256) {
    size_t o = (size_t)q * k + i;
    if (i < n) {
      out_ids[o] = id_base + (int64_t)key_index(keys[i]);
      out_scores[o] = key_score(keys[i]);
    } else {
      out_ids[o] = -1;
      out_scores[o] = 0.f;
    }
  }
}

}  // namespace

struct thr_bm25_state {
  const int64_t* skip;
  const void* post;
  const float* idf;
  int64_t n_docs;
  int n_blk, blk_docs, blk_shift, V;
  int64_t id_base;
  int64_t* df;  // [V] device
  const uint16_t* tags;  // [n_docs] device, nullable
  const uint32_t* deleted;  // [ceil(n_docs / 32)] device, nullable
  // planner tuning (per handle; THR_BM25_* environment variables are read once, when the index is set)
  int units_per_cta;
  long long range_cost, term_cost;
  int warps;    // warps per CTA of bm25_range_kernel (0: as many as shared memory holds)
};

void thr_bm25_state_free(thr_handle* h) {
  if (h->bm25) {
    if (h->bm25->df) cudaFree(h->bm25->df);
    free(h->bm25);
    h->bm25 = nullptr;
  }
}

static int bm25_topk_impl(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                          const int32_t* want, int require_all, int64_t* out_ids, float* out_scores,
                          int32_t* out_count, void* stream);

extern "C" {

int thr_bm25_index_set(thr_handle* h, const int64_t* skip, const void* postings, const float* idf,
                       int64_t n_docs, int32_t n_blk, int32_t blk_docs, int32_t V, int64_t id_base) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, skip && postings && idf, "thr_bm25_index_set: NULL argument");
  THR_REQUIRE(h, n_docs >= 1 && V >= 1 && n_blk >= 1, "thr_bm25_index_set: empty index");
  int shift = 0;
  while ((1 << shift) < blk_docs) ++shift;
  if ((1 << shift) != blk_docs || blk_docs < 256 || blk_docs > kMaxBlkDocs)
    return thr_fail(h, THR_EUNSUPPORTED, "thr_bm25_index_set: blk_docs = %d must be a power of two in [256, %d]",
                    blk_docs, kMaxBlkDocs);
  THR_REQUIRE(h, (int64_t)n_blk * blk_docs >= n_docs && (int64_t)(n_blk - 1) * blk_docs < n_docs,
              "thr_bm25_index_set: n_blk does not match n_docs / blk_docs");
  THR_REQUIRE(h, n_docs < ((int64_t)1 << 32), "thr_bm25_index_set: more than 2^32 docs per shard");
  THR_REQUIRE(h, ((uintptr_t)postings & 15u) == 0, "thr_bm25_index_set: postings must be 16-byte aligned");
  THR_REQUIRE(h, ((uintptr_t)skip & 7u) == 0, "thr_bm25_index_set: skip must be 8-byte aligned");
  thr_bm25_state_free(h);
  thr_bm25_state* st = (thr_bm25_state*)calloc(1, sizeof(thr_bm25_state));
  if (!st) return thr_fail(h, THR_ENOMEM, "out of host memory");
  st->skip = skip; st->post = postings; st->idf = idf; st->n_docs = n_docs; st->n_blk = n_blk;
  st->blk_docs = blk_docs; st->blk_shift = shift; st->V = V; st->id_base = id_base;
  const char* e1 = getenv("THR_BM25_TERM_COST");
  st->term_cost = e1 ? atoll(e1) : kTermCostDefault;
  e1 = getenv("THR_BM25_UNITS_PER_SM");
  st->units_per_cta = e1 ? atoi(e1) : kUnitsPerCtaDefault;
  if (st->units_per_cta < 1) st->units_per_cta = 1;
  e1 = getenv("THR_BM25_RANGE_COST");
  st->range_cost = e1 ? atoll(e1) : (long long)kRangeCostDefault;
  e1 = getenv("THR_BM25_WARPS");
  st->warps = e1 ? atoi(e1) : 0;
  cudaError_t e = cudaMalloc((void**)&st->df, (size_t)V * sizeof(int64_t));
  if (e != cudaSuccess) { free(st); return thr_fail(h, THR_ENOMEM, "cudaMalloc(df): %s", cudaGetErrorString(e)); }
  bm25_df_kernel<<<(V + 255) / 256, 256>>>(skip, idf, n_blk, V, st->df, h->d_status);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    cudaFree(st->df); free(st);
    return thr_fail(h, THR_ECUDA, "bm25_df_kernel: %s", cudaGetErrorString(e));
  }
  if (h->h_status->code == THR_EINVAL && h->h_status->where == 461) {
    const long long t = h->h_status->aux;
    h->h_status->code = 0;
    cudaFree(st->df); free(st);
    return thr_fail(h, THR_EINVAL, "thr_bm25_index_set: idf[%lld] is negative, NaN or outside {0} U [2^-40, 2^20] (idf must be >= 0)", t);
  }
  h->launches++;
  h->bm25 = st;
  return THR_OK;
}

int thr_bm25_tags_set(thr_handle* h, const uint16_t* tags) {
  if (!h) return THR_EINVAL;
  if (!h->bm25) return thr_fail(h, THR_ENOINDEX, "thr_bm25_tags_set: call thr_bm25_index_set first");
  THR_REQUIRE(h, ((uintptr_t)tags & 7u) == 0, "thr_bm25_tags_set: tags must be 8-byte aligned");
  h->bm25->tags = tags;
  return THR_OK;
}

int thr_bm25_deleted_set(thr_handle* h, const uint32_t* bits) {
  if (!h) return THR_EINVAL;
  if (!h->bm25) return thr_fail(h, THR_ENOINDEX, "thr_bm25_deleted_set: call thr_bm25_index_set first");
  THR_REQUIRE(h, ((uintptr_t)bits & 15u) == 0, "thr_bm25_deleted_set: bits must be 16-byte aligned");
  h->bm25->deleted = bits;
  return THR_OK;
}

int thr_bm25_topk(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                  int64_t* out_ids, float* out_scores, int32_t* out_count, void* stream) {
  return bm25_topk_impl(h, q_terms, q_off, B, k, nullptr, 0, out_ids, out_scores, out_count, stream);
}

int thr_bm25_topk_tagged(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                         const int32_t* want, int64_t* out_ids, float* out_scores, int32_t* out_count,
                         void* stream) {
  return bm25_topk_impl(h, q_terms, q_off, B, k, want, 0, out_ids, out_scores, out_count, stream);
}

int thr_bm25_topk_ex(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                     const int32_t* want, int flags, int64_t* out_ids, float* out_scores,
                     int32_t* out_count, void* stream) {
  if (h && (flags & ~THR_BM25_REQUIRE_ALL)) return thr_fail(h, THR_EINVAL, "thr_bm25_topk_ex: unknown flag bits 0x%x", flags);
  return bm25_topk_impl(h, q_terms, q_off, B, k, want, (flags & THR_BM25_REQUIRE_ALL) ? 1 : 0, out_ids, out_scores,
                        out_count, stream);
}

}  // extern "C"

template <int kBlk, bool kAnd>
static cudaError_t launch_range2(const Bm25Args& a, int grid, int warps, size_t smem, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(bm25_range_kernel<kBlk, kAnd>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(bm25_range_kernel<kBlk, kAnd>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  if (e != cudaSuccess) return e;
  bm25_range_kernel<kBlk, kAnd><<<grid, warps * 32, smem, s>>>(a);
  return cudaSuccess;
}
template <int kBlk>
static cudaError_t launch_range(const Bm25Args& a, int grid, int warps, size_t smem, cudaStream_t s) {
  return a.require_all ? launch_range2<kBlk, true>(a, grid, warps, smem, s) : launch_range2<kBlk, false>(a, grid, warps, smem, s);
}

static int bm25_topk_impl(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, int k,
                          const int32_t* want, int require_all, int64_t* out_ids, float* out_scores,
                          int32_t* out_count, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  thr_bm25_state* st = h->bm25;
  if (!st) return thr_fail(h, THR_ENOINDEX, "thr_bm25_topk: call thr_bm25_index_set first");
  THR_REQUIRE(h, want == nullptr || st->tags != nullptr, "thr_bm25_topk_tagged: call thr_bm25_tags_set first");
  THR_REQUIRE(h, B >= 0 && k >= 1 && k <= kMaxSelB, "thr_bm25_topk: need 1 <= k <= %d", kMaxSelB);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, q_terms && q_off && out_ids && out_scores && out_count, "thr_bm25_topk: NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = h->num_sms;
  // warps per CTA: one accumulator (blk_docs fp32 slots) each, as many as shared memory holds (at most 32)
  const size_t fixed = (size_t)kListCap * 8 + sizeof(RangeShared) + 256;
  const size_t per_warp = (size_t)st->blk_docs * (require_all ? 5 : 4) + kDescCap * 16;   // fp32 slots (+ u8 hit counts) + descriptor ring
  int warps = (int)((232448 - fixed) / per_warp);
  if (warps > 32) warps = 32;
  if (st->warps > 0 && st->warps < warps) warps = st->warps;
  const size_t smem = (size_t)warps * per_warp + fixed;
  // scratch: cost keys | units | order | unit_base | counters | partial lists | tau per query | per-warp lists
  const size_t max_units = (size_t)B * kMaxUnitsPerQuery;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t o_keys = 0;
  const size_t o_units = o_keys + up((size_t)B * 8);
  const size_t o_order = o_units + up(max_units * sizeof(Unit));
  const size_t o_base = o_order + up(max_units * 4);
  const size_t o_cnt = o_base + up((size_t)(B + 1) * 4);
  const size_t o_pcnt = o_cnt + 256;
  const size_t o_pkeys = o_pcnt + up(max_units * 4);
  const size_t o_tau = o_pkeys + up(max_units * (size_t)k * 8);
  const size_t o_wl = o_tau + up((size_t)B * 4);
  const size_t need = o_wl + up((size_t)grid * warps * kListCap * 8);
  uint8_t* ws = (uint8_t*)thr_scratch(h, 1, need);
  if (!ws) return THR_ENOMEM;
  unsigned long long* keys = (unsigned long long*)(ws + o_keys);
  Unit* units = (Unit*)(ws + o_units);
  int32_t* order = (int32_t*)(ws + o_order);
  int* unit_base = (int*)(ws + o_base);
  int* counter = (int*)(ws + o_cnt);
  int* total_units = counter + 1;
  int32_t* part_cnt = (int32_t*)(ws + o_pcnt);
  uint64_t* part_keys = (uint64_t*)(ws + o_pkeys);

  int tok = thr_prof_begin(h, THR_PROF_BM25_PREP, s);
  // Work is cut into about `grid * units_per_cta` units of equal cost (heaviest first, fetched dynamically).
  bm25_plan_kernel<<<1, 1024, 0, s>>>(q_terms, q_off, st->df, st->V, st->term_cost, keys, (unsigned*)(ws + o_tau),
                                      h->d_status, B, st->n_blk, grid * st->units_per_cta,
                                      (unsigned long long)st->range_cost, units, unit_base, total_units, counter, order);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "bm25_plan_kernel");

  Bm25Args a;
  a.skip = st->skip; a.post = (const Posting*)st->post; a.idf = st->idf; a.n_docs = st->n_docs;
  a.n_blk = st->n_blk; a.blk_docs = st->blk_docs; a.blk_shift = st->blk_shift; a.V = st->V;
  a.q_terms = q_terms; a.q_off = q_off; a.order = order; a.units = units; a.total_units = total_units;
  a.work_counter = counter; a.B = B; a.k = k; a.part_keys = part_keys; a.part_cnt = part_cnt;
  a.tags = want ? st->tags : nullptr; a.want = want; a.deleted = st->deleted;
  a.wlists = (uint64_t*)(ws + o_wl); a.tau_q = (unsigned*)(ws + o_tau); a.require_all = require_all;
  a.status = h->d_status;
  tok = thr_prof_begin(h, THR_PROF_BM25, s);
  cudaError_t le;
  switch (st->blk_docs) {
    case 2048: le = launch_range<2048>(a, grid, warps, smem, s); break;
    case 1024: le = launch_range<1024>(a, grid, warps, smem, s); break;
    case 512: le = launch_range<512>(a, grid, warps, smem, s); break;
    default: le = launch_range<256>(a, grid, warps, smem, s); break;
  }
  thr_prof_end(h, tok, s);
  if (le != cudaSuccess) return thr_fail(h, THR_ECUDA, "bm25_range_kernel attributes: %s", cudaGetErrorString(le));
  THR_CHECK_LAUNCH(h, "bm25_range_kernel");
  tok = thr_prof_begin(h, THR_PROF_BM25_PREP, s);
  size_t merge_slots = 32;
  while (merge_slots < (size_t)kMaxUnitsPerQuery * k) merge_slots <<= 1;
  THR_CUDA(h, cudaFuncSetAttribute(bm25_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(merge_slots * 8)));
  bm25_merge_kernel<<<B, 256, merge_slots * 8, s>>>(part_keys, part_cnt, unit_base, k, st->id_base, out_ids, out_scores,
                                                    out_count);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "bm25_merge_kernel");
  return THR_OK;
}
