// scope.cu — document-scoped search: the exact semantic and lexical top-k of each query over its own list of rows,
// scored on those rows instead of a corpus scan (thr_dense_topk_rows, thr_bm25_topk_rows in include/thr.h).
//
// A query's scope is rows[off[q] .. off[q+1]) (global ids).  Two launches per channel:
//   scope_*_rows_kernel   a fixed grid of n_cta CTAs cuts the concatenated scopes [off[0], off[B]) into equal slices
//                         (at least kMinSlice* positions each, so a small scope stays on few CTAs); a CTA walks the
//                         queries its slice touches, scores each held, live, tag-matching row exactly and keeps that
//                         query's top k in a running buffer in shared memory, then writes one sorted list per
//                         (CTA, query) it touched: "segment" b + q, unique because the (b, q) pairs of non-empty
//                         segments form a staircase.
//   scope_reduce_kernel   one CTA per query: the same running top-k over the query's segments, then the outputs in
//                         thr_dense_topk's / thr_bm25_topk's format.
// Scratch (the channel's arena): (n_cta + B) segments of k (u64 key, u32 index) pairs plus one count each, about
// 12 (n_cta + B) k bytes: 1.7 MB at B = 256, k = 256 on 148 SMs.  Nothing depends on the scope sizes, so the host never
// reads them and a scope may hold anything from no row to every row of the handle.
//
// Keys: (orderable fp64 score, ~local row) — a larger key is better, so the order is (score desc, id asc).  BM25's fp32
// scores widen to fp64 exactly.  The dense score is rescore_rows', the function K1's finalize and thr_dense_rescore
// use; the BM25 score is K2's definition: the fp32 sum over the query's terms in query order of fp32(idf * impact), each
// impact found by a binary search of the row's skip range of the term.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kThreads = 512;
constexpr int kBuf = 1024;         // running top-k buffer (entries)
constexpr int kRound = 512;        // most entries one round may add: the buffer is compacted when fewer are free
constexpr int kMaxK = 256;
constexpr int kMaxTerms = 32;      // as K2
constexpr int kMinSliceDense = 64;
constexpr int kMinSliceBm25 = 512;
constexpr int kDenseGroups = kRound / (kThreads / 32 * kInFlight);   // kInFlight-row groups per warp and round
static_assert(kBuf - kRound >= kMaxK, "a compaction keeps k entries and leaves room for a round");

__device__ __forceinline__ uint64_t f64_orderable(double d) {
  const uint64_t u = (uint64_t)__double_as_longlong(d + 0.0);   // -0.0 -> +0.0: equal scores get equal keys
  return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_from_orderable(uint64_t u) {
  return __longlong_as_double((long long)((u & 0x8000000000000000ull) ? (u & 0x7fffffffffffffffull) : ~u));
}

// The running top-k of one query, in shared memory.  Entries above the threshold (the k-th best key once the buffer
// has been compacted) are appended by any thread; topk_round_end() compacts to the best k when a round might not fit.
struct TopK {
  uint64_t hi[kBuf];
  uint32_t lo[kBuf];
  uint64_t tau_hi;
  uint32_t tau_lo;
  int cnt;
};

__device__ __forceinline__ void topk_reset(TopK& t) {
  if (threadIdx.x == 0) { t.cnt = 0; t.tau_hi = 0; t.tau_lo = 0; }
}

__device__ __forceinline__ void topk_offer(TopK& t, uint64_t hi, uint32_t lo) {
  if (hi > t.tau_hi || (hi == t.tau_hi && lo > t.tau_lo)) {
    const int s = atomicAdd(&t.cnt, 1);
    t.hi[s] = hi;
    t.lo[s] = lo;
  }
}

// Sort the first n entries descending (bitonic over the next power of two; padding keys are 0).  CTA-wide.
__device__ void topk_sort(TopK& t, int n) {
  int n2 = 2;
  while (n2 < n) n2 <<= 1;
  for (int i = n + (int)threadIdx.x; i < n2; i += kThreads) { t.hi[i] = 0; t.lo[i] = 0; }
  __syncthreads();
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const int i = threadIdx.x;
      if (i < (n2 >> 1)) {
        const int a = ((i / stride) * (stride << 1)) + (i % stride), b = a + stride;
        const uint64_t xh = t.hi[a], yh = t.hi[b];
        const uint32_t xl = t.lo[a], yl = t.lo[b];
        const bool y_gt = yh > xh || (yh == xh && yl > xl);
        const bool x_gt = xh > yh || (xh == yh && xl > yl);
        if ((a & size) == 0 ? y_gt : x_gt) { t.hi[a] = yh; t.hi[b] = xh; t.lo[a] = yl; t.lo[b] = xl; }
      }
      __syncthreads();
    }
  }
}

// End of a round: every thread has offered; keep the best k when the next round might not fit.  CTA-wide.
__device__ void topk_round_end(TopK& t, int k) {
  __syncthreads();
  const int n = t.cnt;
  if (n > kBuf - kRound) {
    topk_sort(t, n);
    if (threadIdx.x == 0) { t.cnt = k; t.tau_hi = t.hi[k - 1]; t.tau_lo = t.lo[k - 1]; }
  }
  __syncthreads();
}

struct Slices {
  int64_t p0, total, chunk;
};
// The CTAs' slices of the concatenated scopes: CTA b scores positions [p0 + min(total, b chunk), p0 + min(total,
// (b + 1) chunk)).  Both kernels compute it the same way from off[0], off[B].
__device__ __forceinline__ Slices slices_of(const int64_t* off, int B, int n_cta, int min_slice) {
  Slices s;
  s.p0 = off[0];
  s.total = max(off[B] - s.p0, (int64_t)0);
  s.chunk = max((s.total + n_cta - 1) / n_cta, (int64_t)min_slice);
  return s;
}

struct ScopeArgs {
  int B, k, n_cta, min_slice;
  const int64_t* rows;
  const int64_t* off;
  const int32_t* want;      // nullable; with it, tags is set
  const uint16_t* tags;
  const uint32_t* deleted;  // nullable
  int64_t N, id_base;       // rows held: [id_base, id_base + N)
  // dense
  const __nv_bfloat16* Q;
  const __nv_bfloat16* X;
  int D;
  // BM25
  const int32_t* q_terms;
  const int32_t* q_off;
  const int64_t* skip;
  const uint2* post;        // {u32 doc, f32 impact}
  const float* idf;
  int n_blk, blk_shift, V, require_all;
  thr_dev_status* status;
  // segments [n_cta + B]
  uint64_t* seg_hi;
  uint32_t* seg_lo;
  int32_t* seg_cnt;
};

__device__ __forceinline__ bool row_eligible(const ScopeArgs& a, int64_t id, int want, uint32_t* r_out) {
  const int64_t r = id - a.id_base;
  if (id < 0 || r < 0 || r >= a.N) return false;
  if (want >= 0 && (int)a.tags[r] != want) return false;
  if (a.deleted && ((a.deleted[r >> 5] >> (r & 31)) & 1u)) return false;
  *r_out = (uint32_t)r;
  return true;
}

// The sorted best k of the buffer -> segment `seg`.  CTA-wide; resets the buffer.
__device__ void flush_segment(const ScopeArgs& a, TopK& t, int seg) {
  __syncthreads();
  const int n = t.cnt;
  topk_sort(t, n);
  const int m = min(n, a.k);
  for (int i = threadIdx.x; i < m; i += kThreads) {
    a.seg_hi[(size_t)seg * a.k + i] = t.hi[i];
    a.seg_lo[(size_t)seg * a.k + i] = t.lo[i];
  }
  if (threadIdx.x == 0) a.seg_cnt[seg] = m;
  __syncthreads();
  topk_reset(t);
  __syncthreads();
}

// Walks the queries CTA blockIdx.x's slice touches; body(q, lo, hi) scores positions [lo, hi) of query q into t.
template <typename Body>
__device__ __forceinline__ void for_each_segment(const ScopeArgs& a, TopK& t, Body body) {
  __shared__ int s_q;
  const Slices sl = slices_of(a.off, a.B, a.n_cta, a.min_slice);
  const int64_t s_lo = sl.p0 + min(sl.total, (int64_t)blockIdx.x * sl.chunk);
  const int64_t s_hi = sl.p0 + min(sl.total, (int64_t)(blockIdx.x + 1) * sl.chunk);
  if (s_lo >= s_hi) return;   // CTA-uniform
  if (threadIdx.x == 0) {     // the last q with off[q] <= s_lo (off is non-decreasing)
    int lo = 0, hi = a.B;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (a.off[mid] <= s_lo) lo = mid; else hi = mid - 1;
    }
    s_q = min(lo, a.B - 1);
  }
  topk_reset(t);
  __syncthreads();
  for (int q = s_q; q < a.B; ++q) {
    const int64_t q_lo = a.off[q], q_hi = a.off[q + 1];
    if (q_lo >= s_hi) break;
    const int64_t lo = max(s_lo, q_lo), hi = min(s_hi, q_hi);
    if (lo >= hi) continue;
    body(q, lo, hi);
    flush_segment(a, t, blockIdx.x + q);
  }
}

// ------------------------------------------------------------------------------------------------
// Semantic: a warp re-scores kInFlight rows at a time with rescore_rows (K1's bits); a round is kRound positions.
__global__ void __launch_bounds__(kThreads, 2) scope_dense_rows_kernel(const ScopeArgs a) {
  extern __shared__ uint8_t dsm[];
  __nv_bfloat16* qrow = (__nv_bfloat16*)dsm;
  __shared__ TopK t;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for_each_segment(a, t, [&](int q, int64_t lo, int64_t hi) {
    for (int i = threadIdx.x; i < a.D; i += kThreads) qrow[i] = a.Q[(size_t)q * a.D + i];
    const int want = a.want ? a.want[q] : -1;
    __syncthreads();
    for (int64_t p0 = lo; p0 < hi; p0 += kRound) {
      for (int g = 0; g < kDenseGroups; ++g) {
        const int64_t pg = p0 + ((int64_t)g * (kThreads / 32) + warp) * kInFlight;
        if (pg >= hi) break;   // warp-uniform
        uint32_t idx[kInFlight];
        bool ok[kInFlight], any = false;
#pragma unroll
        for (int u = 0; u < kInFlight; ++u) {
          idx[u] = 0;
          ok[u] = pg + u < hi && row_eligible(a, a.rows[pg + u], want, &idx[u]);
          any |= ok[u];
        }
        if (!any) continue;    // warp-uniform: every lane read the same rows
        double acc[kInFlight];
        rescore_rows(a.X, a.D, a.D, idx, qrow, lane, acc);
        if (lane == 0) {
#pragma unroll
          for (int u = 0; u < kInFlight; ++u)
            if (ok[u]) topk_offer(t, f64_orderable(acc[u]), ~idx[u]);
        }
      }
      topk_round_end(t, a.k);
    }
  });
}

// ------------------------------------------------------------------------------------------------
// Lexical: one thread per (query, row); the query's terms (K2's treatment of repeats and unknown ids) in shared memory.
__global__ void __launch_bounds__(kThreads) scope_bm25_rows_kernel(const ScopeArgs a) {
  __shared__ TopK t;
  __shared__ int s_term[kMaxTerms];
  __shared__ float s_w[kMaxTerms];
  __shared__ int s_nt, s_need, s_dead;
  for_each_segment(a, t, [&](int q, int64_t lo, int64_t hi) {
    if (threadIdx.x < 32) {
      const int lane = threadIdx.x;
      const int qlo = a.q_off[q], n_all = a.q_off[q + 1] - qlo;
      if (lane == 0 && n_all > kMaxTerms) dev_report(a.status, THR_EINVAL, 460, q);   // K2 reports it the same way
      const int nt = min(n_all, kMaxTerms);
      int term = lane < nt ? a.q_terms[qlo + lane] : -1;
      const bool known = term >= 0 && term < a.V;
      const bool unknown = lane < nt && !known;
      if (!known) term = -1;
      // AND: a repeated term counts and scores once; an unknown term means no row matches
      bool dup = false;
      for (int u = 0; u < nt; ++u) {
        const int tu = __shfl_sync(0xffffffffu, term, u);
        if (u < lane && tu == term) dup = true;
      }
      const int need = __popc(__ballot_sync(0xffffffffu, term >= 0 && !dup));
      const bool dead = __any_sync(0xffffffffu, unknown) || need == 0;
      if (a.require_all && dup) term = -1;
      if (lane < kMaxTerms) {
        s_term[lane] = term;
        s_w[lane] = term >= 0 ? a.idf[term] : 0.f;
      }
      if (lane == 0) { s_nt = nt; s_need = need; s_dead = a.require_all ? (int)dead : 0; }
    }
    __syncthreads();
    const int want = a.want ? a.want[q] : -1;
    const int nt = s_nt;
    for (int64_t p0 = lo; p0 < hi; p0 += kRound) {
      const int64_t p = p0 + threadIdx.x;
      uint32_t r = 0;
      if (p < hi && !s_dead && row_eligible(a, a.rows[p], want, &r)) {
        const int blk = (int)(r >> a.blk_shift);
        float s = 0.f;
        int hits = 0;
        for (int j = 0; j < nt; ++j) {
          const int tj = s_term[j];
          if (tj < 0) continue;
          const int64_t* sk = a.skip + (size_t)tj * a.n_blk + blk;
          int64_t b0 = sk[0], b1 = sk[1];   // the term's postings in the row's range, docs ascending
          while (b0 < b1) {
            const int64_t mid = (b0 + b1) >> 1;
            if (a.post[mid].x < r) b0 = mid + 1; else b1 = mid;
          }
          if (b0 < sk[1]) {
            const uint2 e = a.post[b0];
            if (e.x == r) {
              s = __fadd_rn(s, __fmul_rn(s_w[j], __uint_as_float(e.y)));
              ++hits;
            }
          }
        }
        if (s > 0.f && (!a.require_all || hits == s_need)) topk_offer(t, f64_orderable((double)s), ~r);
      }
      topk_round_end(t, a.k);
    }
  });
}

// ------------------------------------------------------------------------------------------------
// One CTA per query: the running top-k over its segments, then the channel's output format.
struct ReduceArgs {
  int B, k, n_cta, min_slice;
  const int64_t* off;
  int64_t id_base;
  const uint64_t* seg_hi;
  const uint32_t* seg_lo;
  const int32_t* seg_cnt;
  int64_t* out_ids;
  double* out_scores_f64;   // semantic (-inf padded), or
  float* out_scores_f32;    // lexical (0 padded)
  int32_t* out_count;
  float* out_gap;           // nullable: +inf
};

__global__ void __launch_bounds__(kThreads) scope_reduce_kernel(const ReduceArgs a) {
  __shared__ TopK t;
  const int q = blockIdx.x;
  const Slices sl = slices_of(a.off, a.B, a.n_cta, a.min_slice);
  const int64_t q_lo = a.off[q], q_hi = a.off[q + 1];
  topk_reset(t);
  __syncthreads();
  if (q_lo < q_hi) {   // CTA-uniform
    const int b_lo = (int)((q_lo - sl.p0) / sl.chunk), b_hi = (int)((q_hi - 1 - sl.p0) / sl.chunk);
    for (int b = b_lo; b <= b_hi; ++b) {
      const int64_t s_lo = sl.p0 + min(sl.total, (int64_t)b * sl.chunk);
      const int64_t s_hi = sl.p0 + min(sl.total, (int64_t)(b + 1) * sl.chunk);
      if (max(s_lo, q_lo) >= min(s_hi, q_hi)) continue;
      const int seg = b + q;
      const int n = a.seg_cnt[seg];
      if ((int)threadIdx.x < n)
        topk_offer(t, a.seg_hi[(size_t)seg * a.k + threadIdx.x], a.seg_lo[(size_t)seg * a.k + threadIdx.x]);
      topk_round_end(t, a.k);
    }
  }
  const int n = t.cnt;
  topk_sort(t, n);
  const int m = min(n, a.k);
  for (int i = threadIdx.x; i < a.k; i += kThreads) {
    const size_t o = (size_t)q * a.k + i;
    const bool has = i < m;
    a.out_ids[o] = has ? a.id_base + (int64_t)(~t.lo[i]) : -1;
    const double sc = has ? f64_from_orderable(t.hi[i]) : -CUDART_INF;
    if (a.out_scores_f64) a.out_scores_f64[o] = sc;
    else a.out_scores_f32[o] = has ? (float)sc : 0.f;
  }
  if (threadIdx.x == 0) {
    a.out_count[q] = m;
    if (a.out_gap) a.out_gap[q] = CUDART_INF_F;
  }
}

// Scratch and launches shared by both channels.
int scope_run(thr_handle* h, int arena, int prof_slot, ScopeArgs& a, ReduceArgs& r, bool dense, size_t dyn_smem,
              cudaStream_t s) {
  a.n_cta = 2 * h->num_sms;
  const size_t n_seg = (size_t)a.n_cta + a.B;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t o_lo = up(n_seg * a.k * 8), o_cnt = o_lo + up(n_seg * a.k * 4);
  uint8_t* ws = (uint8_t*)thr_scratch(h, arena, o_cnt + n_seg * 4);
  if (!ws) return THR_ENOMEM;
  a.seg_hi = (uint64_t*)ws; a.seg_lo = (uint32_t*)(ws + o_lo); a.seg_cnt = (int32_t*)(ws + o_cnt);
  a.status = h->d_status;
  r.B = a.B; r.k = a.k; r.n_cta = a.n_cta; r.min_slice = a.min_slice; r.off = a.off; r.id_base = a.id_base;
  r.seg_hi = a.seg_hi; r.seg_lo = a.seg_lo; r.seg_cnt = a.seg_cnt;
  int tok = thr_prof_begin(h, prof_slot, s);
  if (dense) {
    THR_CUDA(h, cudaFuncSetAttribute(scope_dense_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn_smem));
    scope_dense_rows_kernel<<<a.n_cta, kThreads, dyn_smem, s>>>(a);
  } else {
    scope_bm25_rows_kernel<<<a.n_cta, kThreads, 0, s>>>(a);
  }
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, dense ? "scope_dense_rows_kernel" : "scope_bm25_rows_kernel");
  tok = thr_prof_begin(h, prof_slot, s);
  scope_reduce_kernel<<<a.B, kThreads, 0, s>>>(r);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "scope_reduce_kernel");
  return THR_OK;
}

}  // namespace

extern "C" {

int thr_dense_topk_rows(thr_handle* h, const void* Q, int B, const int64_t* rows, const int64_t* off, int k,
                        const int32_t* want, int64_t* out_ids, double* out_scores, int32_t* out_count, float* out_gap,
                        void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  thr_dense_view v;
  if (thr_dense_view_get(h, &v) != THR_OK) return thr_fail(h, THR_ENOINDEX, "thr_dense_topk_rows: call thr_dense_index_set first");
  THR_REQUIRE(h, want == nullptr || v.tags != nullptr, "thr_dense_topk_rows: call thr_dense_tags_set first");
  THR_REQUIRE(h, B >= 0 && k >= 1 && k <= kMaxK, "thr_dense_topk_rows: need B >= 0 and 1 <= k <= %d", kMaxK);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, Q && rows && off && out_ids && out_scores && out_count, "thr_dense_topk_rows: NULL argument");
  ScopeArgs a = {};
  a.B = B; a.k = k; a.min_slice = kMinSliceDense; a.rows = rows; a.off = off; a.want = want;
  a.tags = want ? v.tags : nullptr; a.deleted = v.deleted; a.N = v.N; a.id_base = v.id_base;
  a.Q = (const __nv_bfloat16*)Q; a.X = (const __nv_bfloat16*)v.X; a.D = v.D;
  ReduceArgs r = {};
  r.out_ids = out_ids; r.out_scores_f64 = out_scores; r.out_count = out_count; r.out_gap = out_gap;
  return scope_run(h, 0, THR_PROF_DENSE_SCORE, a, r, true, (size_t)v.D * 2, (cudaStream_t)stream);
}

int thr_bm25_topk_rows(thr_handle* h, const int32_t* q_terms, const int32_t* q_off, int B, const int64_t* rows,
                       const int64_t* off, int k, const int32_t* want, int flags, int64_t* out_ids, float* out_scores,
                       int32_t* out_count, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  if (flags & ~THR_BM25_REQUIRE_ALL) return thr_fail(h, THR_EINVAL, "thr_bm25_topk_rows: unknown flag bits 0x%x", flags);
  thr_bm25_view v;
  if (thr_bm25_view_get(h, &v) != THR_OK) return thr_fail(h, THR_ENOINDEX, "thr_bm25_topk_rows: call thr_bm25_index_set first");
  THR_REQUIRE(h, want == nullptr || v.tags != nullptr, "thr_bm25_topk_rows: call thr_bm25_tags_set first");
  THR_REQUIRE(h, B >= 0 && k >= 1 && k <= kMaxK, "thr_bm25_topk_rows: need B >= 0 and 1 <= k <= %d", kMaxK);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, q_terms && q_off && rows && off && out_ids && out_scores && out_count,
              "thr_bm25_topk_rows: NULL argument");
  ScopeArgs a = {};
  a.B = B; a.k = k; a.min_slice = kMinSliceBm25; a.rows = rows; a.off = off; a.want = want;
  a.tags = want ? v.tags : nullptr; a.deleted = v.deleted; a.N = v.n_docs; a.id_base = v.id_base;
  a.q_terms = q_terms; a.q_off = q_off; a.skip = v.skip; a.post = (const uint2*)v.post; a.idf = v.idf;
  a.n_blk = v.n_blk; a.blk_shift = v.blk_shift; a.V = v.V; a.require_all = (flags & THR_BM25_REQUIRE_ALL) ? 1 : 0;
  ReduceArgs r = {};
  r.out_ids = out_ids; r.out_scores_f32 = out_scores; r.out_count = out_count;
  return scope_run(h, 1, THR_PROF_BM25, a, r, false, 0, (cudaStream_t)stream);
}

}  // extern "C"
