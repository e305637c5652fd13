// fuse.cu — K3: weighted RRF fusion + safety threshold + conformal denoise, K5: shard merge,
// and the RAG 2.0 safety/denoise filter.  All arithmetic that the reference does in Python
// floats is done here in fp64 with explicit round-to-nearest intrinsics (no FMA contraction),
// in the reference's operation order, so results are bit-identical.
//
// Reference semantics restated (paths relative to the reference checkout):
//   merge + ranks : src/voice_agent/rag2/retrieval.py:203-271
//   RRF (RAG2)    : src/voice_agent/rag2/retrieval.py:358-376          w / (k + rank)
//   RRF (library) : triple-hybrid-rag/src/triple_hybrid_rag/core/fusion.py:52-185   w * (1.0 / (k + rank))
//   RRF (RAG1)    : src/voice_agent/retrieval/hybrid_search.py:460-501 1.0 / (k + rank0 + 1)
//   safety (lib)  : fusion.py:187-216, denoise: fusion.py:218-247 (numpy.percentile, linear)
//   safety (RAG2) : src/voice_agent/rag2/retrieval.py:461-495
#include "common.cuh"

namespace {

constexpr int kMaxList = 256;            // longest single channel list
constexpr int kMaxEntries = 3 * kMaxList;
constexpr int kSortPad = 1024;
constexpr int kFuseThreads = 256;

struct FuseArgs {
  const int64_t* ids[3];
  const int32_t* off[3];
  const double* sc[3];
  const double* weights;  // [B,3]
  int rrf_k;
  double safety_thr;
  double alpha;
  int denoise;
  int top_k;
  int max_out;
  int tie_mode;
  int64_t* out_ids;
  double* out_rrf;
  int32_t* out_ranks;
  double* out_raw;
  int32_t* out_count;
  thr_dev_status* status;
};

// numpy.percentile(a, q) with method="linear" (numpy 2.x, lib/_function_base_impl.py:
// _QuantileMethods['linear'], _get_indexes, _get_gamma, _lerp) on an ascending array that is
// given as the reverse of `desc` (a[i] = desc[n-1-i]).
__device__ double percentile_linear_desc(const double* desc_vals, const uint16_t* order, int n,
                                         double q) {
  double quant = __ddiv_rn(q, 100.0);
  double vi = __dmul_rn((double)(n - 1), quant);
  long long lo, hi;
  if (vi >= (double)(n - 1)) {
    lo = hi = n - 1;
  } else if (vi < 0.0) {
    lo = hi = 0;
  } else {
    lo = (long long)floor(vi);
    hi = lo + 1;
  }
  // gamma uses the (possibly clamped) previous index exactly as numpy does; when lo == hi the
  // interpolation collapses to a[lo] for finite inputs.
  double prev_for_gamma = (vi >= (double)(n - 1)) ? -1.0 : ((vi < 0.0) ? 0.0 : (double)lo);
  double t = __dsub_rn(vi, prev_for_gamma);
  double a = desc_vals[order[n - 1 - lo]];
  double b = desc_vals[order[n - 1 - hi]];
  double diff = __dsub_rn(b, a);
  double r = __dadd_rn(a, __dmul_rn(diff, t));
  if (t >= 0.5) r = __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, t)));
  return r;
}

template <int kVariant>
__global__ void __launch_bounds__(kFuseThreads) fuse_kernel(FuseArgs a) {
  __shared__ int64_t e_id[kMaxEntries];
  __shared__ double e_rrf[kMaxEntries];
  __shared__ double e_raw[3][kMaxEntries];
  __shared__ uint16_t e_rank[3][kMaxEntries];
  __shared__ uint16_t e_pos[kMaxEntries];
  __shared__ uint8_t e_chan[kMaxEntries];
  __shared__ uint16_t perm[kSortPad];
  __shared__ uint16_t grp[kSortPad];   // entry indices sorted by (id, entry index)
  __shared__ uint8_t keep[kMaxEntries];
  __shared__ int s_n[4];      // entries per channel + total
  __shared__ int s_unique;
  __shared__ double s_thr;
  __shared__ int s_out;

  const int q = blockIdx.x;
  const int tid = threadIdx.x;

  if (tid == 0) {
    int tot = 0;
    for (int c = 0; c < 3; ++c) {
      int n = 0;
      if (a.ids[c] != nullptr) n = a.off[c][q + 1] - a.off[c][q];
      if (n > kMaxList) {
        dev_report(a.status, THR_EOVERFLOW, 300 + c, n);
        n = kMaxList;
      }
      s_n[c] = n;
      tot += n;
    }
    s_n[3] = tot;
    s_unique = 0;
  }
  __syncthreads();
  const int n0 = s_n[0], n1 = s_n[1], n = s_n[3];

  // 1. concatenate lexical -> semantic -> graph (the reference's dict insertion order)
  for (int e = tid; e < n; e += kFuseThreads) {
    int c = e < n0 ? 0 : (e < n0 + n1 ? 1 : 2);
    int p = e - (c == 0 ? 0 : (c == 1 ? n0 : n0 + n1));
    int64_t src = (int64_t)a.off[c][q] + p;
    e_id[e] = a.ids[c][src];
    e_chan[e] = (uint8_t)c;
    e_pos[e] = (uint16_t)p;
    e_raw[c][e] = (kVariant != THR_FUSE_RAG2 && a.sc[c] != nullptr) ? a.sc[c][src] : 0.0;
  }
  for (int i = tid; i < kSortPad; i += kFuseThreads) perm[i] = 0xffff;
  __syncthreads();

  // 2. one candidate per distinct id, owned by its first occurrence.  Entries are sorted by (id, entry
  //    index) with a bitonic network, so every id's occurrences form a run in entry order; the thread at
  //    the head of a run walks it (almost always 1-3 entries) — O(n log^2 n) instead of O(n^2) scans.
  const double w[3] = {a.weights[q * 3 + 0], a.weights[q * 3 + 1], a.weights[q * 3 + 2]};
  {
    int P2 = 32;
    while (P2 < n) P2 <<= 1;
    for (int i = tid; i < P2; i += kFuseThreads) grp[i] = i < n ? (uint16_t)i : 0xffff;
    __syncthreads();
    auto id_before = [&](uint16_t x, uint16_t y) -> bool {  // x strictly before y; padding (id < 0) last
      if (x == 0xffff) return false;
      if (y == 0xffff) return true;
      const int64_t ix = e_id[x], iy = e_id[y];
      const bool px = ix < 0, py = iy < 0;
      if (px != py) return py;
      if (ix != iy) return ix < iy;
      return x < y;
    };
    for (int size = 2; size <= P2; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int i = tid; i < (P2 >> 1); i += kFuseThreads) {
          int lo = ((i / stride) * (stride << 1)) + (i % stride);
          int hi = lo + stride;
          bool ascending = ((lo & size) == 0);
          uint16_t x = grp[lo], y = grp[hi];
          bool swap = ascending ? id_before(y, x) : id_before(x, y);
          if (swap) { grp[lo] = y; grp[hi] = x; }
        }
        bitonic_stage_sync(size, stride, P2, 32);
      }
    }
  }
  for (int i = tid; i < n; i += kFuseThreads) {
    const int e = grp[i];
    const int64_t id = e_id[e];
    if (id < 0) continue;  // padding of a fixed-width [B,k] result (-1 past the channel's count)
    if (i > 0 && e_id[grp[i - 1]] == id) continue;  // not the head of its run

    int rank0 = 0, rank1 = 0, rank2 = 0;  // 1-based rank of the LAST occurrence per channel
    int occ0 = 0, occ1 = 0, occ2 = 0;
    double raw0 = 0.0, raw1 = 0.0, raw2 = 0.0;
    double rrf = 0.0;
    for (int t = i; t < n; ++t) {
      const int j = grp[t];
      if (e_id[j] != id) break;
      const int c = e_chan[j];
      const int r = (int)e_pos[j] + 1;
      const double rv = e_raw[c][j];
      if (c == 0) { rank0 = r; occ0 += 1; raw0 = kVariant == THR_FUSE_RAG1 ? fmax(raw0, rv) : rv; }
      else if (c == 1) { rank1 = r; occ1 += 1; raw1 = kVariant == THR_FUSE_RAG1 ? fmax(raw1, rv) : rv; }
      else { rank2 = r; occ2 += 1; raw2 = kVariant == THR_FUSE_RAG1 ? fmax(raw2, rv) : rv; }
      if (kVariant == THR_FUSE_RAG1) rrf = __dadd_rn(rrf, __ddiv_rn(1.0, (double)(a.rrf_k + r)));  // r = rank0 + 1
    }
    const int last_rank[3] = {rank0, rank1, rank2};
    const int occ[3] = {occ0, occ1, occ2};
    if (kVariant == THR_FUSE_RAG2) {
#pragma unroll
      for (int c = 0; c < 3; ++c)
        if (last_rank[c]) rrf = __dadd_rn(rrf, __ddiv_rn(w[c], (double)(a.rrf_k + last_rank[c])));
    } else if (kVariant == THR_FUSE_LIB) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (!occ[c]) continue;
        double sc = __dmul_rn(w[c], __ddiv_rn(1.0, (double)(a.rrf_k + last_rank[c])));
        for (int k = 0; k < occ[c]; ++k) rrf = __dadd_rn(rrf, sc);  // the merge loop adds once per occurrence
      }
    }
    e_rrf[e] = rrf;
    e_rank[0][e] = (uint16_t)rank0; e_rank[1][e] = (uint16_t)rank1; e_rank[2][e] = (uint16_t)rank2;
    e_raw[0][e] = raw0; e_raw[1][e] = raw1; e_raw[2][e] = raw2;
    int slot = atomicAdd(&s_unique, 1);
    perm[slot] = (uint16_t)e;
  }
  __syncthreads();
  const int m = s_unique;

  // 3. sort by (rrf desc, tie asc); tie = first-seen index (stable sort) or chunk id
  int P = 32;
  while (P < m) P <<= 1;
  auto before = [&](uint16_t x, uint16_t y) -> bool {  // x strictly before y
    if (x == 0xffff) return false;
    if (y == 0xffff) return true;
    double rx = e_rrf[x], ry = e_rrf[y];
    if (rx != ry) return rx > ry;
    if (a.tie_mode == THR_TIE_CHUNK_ID) {
      int64_t ix = e_id[x], iy = e_id[y];
      if (ix != iy) return ix < iy;
    }
    return x < y;
  };
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (P >> 1); i += kFuseThreads) {
        int lo = ((i / stride) * (stride << 1)) + (i % stride);
        int hi = lo + stride;
        bool ascending = ((lo & size) == 0);
        uint16_t x = perm[lo], y = perm[hi];
        bool swap = ascending ? before(y, x) : before(x, y);
        if (swap) { perm[lo] = y; perm[hi] = x; }
      }
      bitonic_stage_sync(size, stride, P, 32);
    }
  }

  // 4. filters (library variant), then truncation
  for (int i = tid; i < m; i += kFuseThreads) {
    bool k = true;
    if (kVariant == THR_FUSE_LIB && a.safety_thr > 0.0) {
      int e = perm[i];
      // max(semantic or 0.0, lexical or 0.0, graph or 0.0): Python's max keeps the first of equals
      double mx = e_raw[1][e];
      if (e_raw[0][e] > mx) mx = e_raw[0][e];
      if (e_raw[2][e] > mx) mx = e_raw[2][e];
      k = mx >= a.safety_thr;
    }
    keep[i] = k;
  }
  __syncthreads();

  if (tid < 32) {
    // compact `keep` in order (warp 0), reusing perm in place (write index <= read index)
    int base = 0;
    for (int i0 = 0; i0 < m; i0 += 32) {
      int i = i0 + tid;
      bool k = i < m && keep[i];
      uint16_t v = i < m ? perm[i] : 0xffff;
      unsigned bal = __ballot_sync(0xffffffffu, k);
      __syncwarp();
      if (k) perm[base + __popc(bal & ((1u << tid) - 1))] = v;
      base += __popc(bal);
      __syncwarp();
    }
    int nA = base;
    if (kVariant == THR_FUSE_LIB && a.denoise && nA >= 3) {
      if (tid == 0) {
        double qpct = __dmul_rn(__dsub_rn(1.0, a.alpha), 100.0);
        s_thr = percentile_linear_desc(e_rrf, perm, nA, qpct);
      }
      __syncwarp();
      double thr = s_thr;
      int base2 = 0;
      for (int i0 = 0; i0 < nA; i0 += 32) {
        int i = i0 + tid;
        uint16_t v = i < nA ? perm[i] : 0xffff;
        bool k = i < nA && e_rrf[v] >= thr;
        unsigned bal = __ballot_sync(0xffffffffu, k);
        __syncwarp();
        if (k) perm[base2 + __popc(bal & ((1u << tid) - 1))] = v;
        base2 += __popc(bal);
        __syncwarp();
      }
      nA = base2;
    }
    if (a.top_k > 0 && nA > a.top_k) nA = a.top_k;
    if (nA > a.max_out) {
      if (tid == 0) dev_report(a.status, THR_EOVERFLOW, 310, nA);
      nA = a.max_out;
    }
    if (tid == 0) s_out = nA;
  }
  __syncthreads();

  // 5. outputs
  const int nout = s_out;
  if (tid == 0) a.out_count[q] = nout;
  for (int i = tid; i < a.max_out; i += kFuseThreads) {
    size_t o = (size_t)q * a.max_out + i;
    if (i < nout) {
      int e = perm[i];
      a.out_ids[o] = e_id[e];
      a.out_rrf[o] = e_rrf[e];
      for (int c = 0; c < 3; ++c) {
        a.out_ranks[o * 3 + c] = e_rank[c][e];
        if (a.out_raw) a.out_raw[o * 3 + c] = e_raw[c][e];
      }
    } else {
      a.out_ids[o] = -1;
      a.out_rrf[o] = 0.0;
      for (int c = 0; c < 3; ++c) {
        a.out_ranks[o * 3 + c] = 0;
        if (a.out_raw) a.out_raw[o * 3 + c] = 0.0;
      }
    }
  }
}

// RAG2Retriever._fuse_rrf on candidates that already carry their channel ranks
// (src/voice_agent/rag2/retrieval.py:358-376): score = 0.0 (+ w_lex/(k+r_lex)) (+ w_sem/(k+r_sem))
// (+ w_graph/(k+r_graph)), a channel contributing when its rank is truthy (non-zero); then Python's
// stable sorted(..., reverse=True): descending score, equal scores keep their input order.
__global__ void __launch_bounds__(kFuseThreads) fuse_ranked_kernel(const int32_t* off, const int32_t* ranks,
                                                                   const double* weights, int rrf_k,
                                                                   double* out_rrf, int32_t* out_order,
                                                                   thr_dev_status* status) {
  __shared__ double s_rrf[kSortPad];
  __shared__ uint16_t perm[kSortPad];
  const int q = blockIdx.x, tid = threadIdx.x;
  const int lo = off[q];
  int n = off[q + 1] - lo;
  if (n > kSortPad) {
    if (tid == 0) dev_report(status, THR_EOVERFLOW, 320, n);
    n = kSortPad;
  }
  const double w[3] = {weights[q * 3 + 0], weights[q * 3 + 1], weights[q * 3 + 2]};
  for (int i = tid; i < kSortPad; i += kFuseThreads) {
    double rrf = 0.0;
    if (i < n) {
      for (int c = 0; c < 3; ++c) {
        const int r = ranks[(size_t)(lo + i) * 3 + c];
        if (r != 0) rrf = __dadd_rn(rrf, __ddiv_rn(w[c], (double)(rrf_k + r)));
      }
      out_rrf[lo + i] = rrf;
    }
    s_rrf[i] = rrf;
    perm[i] = i < n ? (uint16_t)i : 0xffff;
  }
  __syncthreads();
  int P = 32;
  while (P < n) P <<= 1;
  auto before = [&](uint16_t x, uint16_t y) -> bool {
    if (x == 0xffff) return false;
    if (y == 0xffff) return true;
    const double rx = s_rrf[x], ry = s_rrf[y];
    if (rx != ry) return rx > ry;
    return x < y;
  };
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (P >> 1); i += kFuseThreads) {
        int a = ((i / stride) * (stride << 1)) + (i % stride);
        int b = a + stride;
        bool ascending = ((a & size) == 0);
        uint16_t x = perm[a], y = perm[b];
        bool swap = ascending ? before(y, x) : before(x, y);
        if (swap) { perm[a] = y; perm[b] = x; }
      }
      bitonic_stage_sync(size, stride, P, 32);
    }
  }
  for (int i = tid; i < n; i += kFuseThreads) out_order[lo + i] = perm[i];
}

// RAG2Retriever._apply_safety — one warp per query.
__global__ void __launch_bounds__(128) safety_kernel(int B, const int32_t* off, const double* rerank,
                                                     const uint8_t* has_rerank, const double* rrf,
                                                     double threshold, double alpha, int top_k,
                                                     uint8_t* keep, uint8_t* refused,
                                                     double* max_score) {
  int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (q >= B) return;
  int lo = off[q], hi = off[q + 1];
  auto score = [&](int i) -> double {
    // `c.rerank_score or c.rrf_score`: None and 0.0 are both falsy
    if (has_rerank && has_rerank[i] && rerank[i] != 0.0) return rerank[i];
    return rrf[i];
  };
  if (hi <= lo) {
    if (lane == 0) { refused[q] = 1; max_score[q] = 0.0; }
    return;
  }
  double mx = -INFINITY;
  for (int i = lo + lane; i < hi; i += 32) mx = fmax(mx, score(i));
  for (int s = 16; s > 0; s >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  bool ref = mx < threshold;
  if (lane == 0) { refused[q] = ref ? 1 : 0; max_score[q] = mx; }
  double min_score = __dmul_rn(alpha, mx);
  int kept = 0;
  for (int i0 = lo; i0 < hi; i0 += 32) {
    int i = i0 + lane;
    bool k = !ref && i < hi && score(i) >= min_score;
    unsigned bal = __ballot_sync(0xffffffffu, k);
    int before = kept + __popc(bal & ((1u << lane) - 1));
    if (i < hi) keep[i] = (k && before < top_k) ? 1 : 0;
    kept += __popc(bal);
  }
}

// K5: per query merge of G lists of (score, id) -> k_out best by (score desc, id asc).
constexpr int kMergeMax = 2048;
__global__ void __launch_bounds__(256) merge_kernel(const double* scores, const int64_t* ids,
                                                    const int32_t* counts, int G, int B, int k_in,
                                                    int k_out, double* out_scores, int64_t* out_ids,
                                                    int32_t* out_count) {
  __shared__ double s_sc[kMergeMax];
  __shared__ int64_t s_id[kMergeMax];
  __shared__ int s_total;
  const int q = blockIdx.x, tid = threadIdx.x;
  const int n = G * k_in;
  int P = 32;
  while (P < n) P <<= 1;
  if (tid == 0) s_total = 0;
  __syncthreads();
  int local = 0;
  for (int i = tid; i < P; i += 256) {
    double s = -INFINITY;
    int64_t id = INT64_MAX;
    if (i < n) {
      int g = i / k_in, j = i % k_in;
      int cnt = counts ? counts[g * B + q] : k_in;
      if (j < cnt) {
        size_t src = ((size_t)g * B + q) * k_in + j;
        s = scores[src];
        id = ids[src];
        ++local;
      }
    }
    s_sc[i] = s;
    s_id[i] = id;
  }
  if (local) atomicAdd(&s_total, local);
  __syncthreads();
  auto before = [&](int x, int y) -> bool {
    int64_t ix = s_id[x], iy = s_id[y];
    bool vx = ix != INT64_MAX, vy = iy != INT64_MAX;
    if (vx != vy) return vx;
    double sx = s_sc[x], sy = s_sc[y];
    if (sx != sy) return sx > sy;
    return ix < iy;
  };
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (P >> 1); i += 256) {
        int lo = ((i / stride) * (stride << 1)) + (i % stride);
        int hi = lo + stride;
        bool ascending = ((lo & size) == 0);
        bool swap = ascending ? before(hi, lo) : before(lo, hi);
        if (swap) {
          double ts = s_sc[lo]; s_sc[lo] = s_sc[hi]; s_sc[hi] = ts;
          int64_t ti = s_id[lo]; s_id[lo] = s_id[hi]; s_id[hi] = ti;
        }
      }
      bitonic_stage_sync(size, stride, P, 32);
    }
  }
  int nout = min(s_total, k_out);
  if (tid == 0) out_count[q] = nout;
  for (int i = tid; i < k_out; i += 256) {
    size_t o = (size_t)q * k_out + i;
    out_scores[o] = i < nout ? s_sc[i] : -INFINITY;
    out_ids[o] = i < nout ? s_id[i] : -1;
  }
}


// ---- K5 for the product's exchange step, two launches around the one all-gather -----------------
// Message of one rank (bytes): [scores f64 2*B*k | ids i64 2*B*k | counts i32 2*B]; row block 0 holds the semantic
// lists, block 1 the lexical ones, k = max(k_sem, k_lex), lists padded with (-inf, -1).
__global__ void __launch_bounds__(256) exchange_pack_kernel(const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                                                            const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt,
                                                            int B, int k_sem, int k_lex, int k, uint8_t* msg) {
  const size_t n = (size_t)2 * B * k;
  double* sc = (double*)msg;
  int64_t* ids = (int64_t*)(msg + n * 8);
  int32_t* cnt = (int32_t*)(msg + 2 * n * 8);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % k);
    const int row = (int)(i / k);
    double s = -INFINITY;
    int64_t id = -1;
    if (row < B) {
      if (j < k_sem) { s = d_sc[(size_t)row * k_sem + j]; id = d_ids[(size_t)row * k_sem + j]; }
    } else if (j < k_lex) {
      s = (double)l_sc[(size_t)(row - B) * k_lex + j];
      id = l_ids[(size_t)(row - B) * k_lex + j];
    }
    sc[i] = s;
    ids[i] = id;
    if (j == 0) cnt[row] = row < B ? d_cnt[row] : l_cnt[row - B];
  }
}

// The same message, but PUSHED: every element is stored straight into slot `rank` of every rank's gathered buffer
// (peer stores over NVLink into symmetric memory; the own buffer is one of the G destinations), and the last CTA
// to finish raises this rank's sequence number in every rank's signal array.  Pack, transfer and notification are
// one kernel; no collective call, no copy engine.  `done` is a zero-initialised device counter.
__global__ void __launch_bounds__(256) exchange_push_kernel(const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                                                            const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt,
                                                            int B, int k_sem, int k_lex, int k,
                                                            uint8_t* const* peer_bufs, size_t slot_off,
                                                            unsigned long long* const* peer_sig, size_t sig_off, int rank,
                                                            int G, unsigned long long seq, unsigned int* done) {
  const size_t n = (size_t)2 * B * k;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % k);
    const int row = (int)(i / k);
    double s = -INFINITY;
    int64_t id = -1;
    if (row < B) {
      if (j < k_sem) { s = d_sc[(size_t)row * k_sem + j]; id = d_ids[(size_t)row * k_sem + j]; }
    } else if (j < k_lex) {
      s = (double)l_sc[(size_t)(row - B) * k_lex + j];
      id = l_ids[(size_t)(row - B) * k_lex + j];
    }
    const int32_t c = j == 0 ? (row < B ? d_cnt[row] : l_cnt[row - B]) : 0;
    for (int g = 0; g < G; ++g) {
      uint8_t* msg = peer_bufs[g] + slot_off;
      ((double*)msg)[i] = s;
      ((int64_t*)(msg + n * 8))[i] = id;
      if (j == 0) ((int32_t*)(msg + 2 * n * 8))[row] = c;
    }
  }
  __threadfence_system();   // this thread's peer stores are performed before the CTA counts itself done
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(done, 1u);
    if (prev == gridDim.x - 1) {   // last CTA: every CTA's stores are visible system-wide (fence cumulativity)
      *done = 0u;
      __threadfence_system();
      for (int g = 0; g < G; ++g) {
        unsigned long long* p = (unsigned long long*)((uint8_t*)peer_sig[g] + sig_off) + rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(seq) : "memory");
      }
    }
  }
}

// The merge step of K5's exchange and of thr_shard_merge: one CTA holds one (channel, query) row's G lists in shared
// memory (list g at s_sc + g * k / s_id + g * k, its first s_cnt[g] <= k entries valid), each sorted by (score desc, id
// asc), and writes the channel's merged list in the channel's own output format (semantic: f64 scores, -inf padding;
// lexical: f32 scores, 0 padding as thr_bm25_topk writes them).  Rows [0, B) are semantic, [B, 2B) lexical.
// Every list is sorted already: merge by RANK instead of sorting — an entry's place in the merged list is its place in
// its own list plus, for every other list, the number of entries that precede it there (a binary search).  No
// exchange network, no barrier between the staging and the output.
__device__ __forceinline__ void merge_staged_write(const double* s_sc, const int64_t* s_id, const int* s_cnt, int G,
                                                  int k, int row, int B, int k_sem, int k_lex, int64_t* d_ids,
                                                  double* d_sc, int32_t* d_cnt, int64_t* l_ids, float* l_sc,
                                                  int32_t* l_cnt) {
  const int n = G * k;
  int total = 0;
  for (int g = 0; g < G; ++g) total += s_cnt[g];
  const int k_out = row < B ? k_sem : k_lex;
  const int nout = min(total, k_out);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int g = i / k, j = i - g * k;
    if (j >= s_cnt[g] || j >= nout) continue;   // an entry's merged place is at least its place in its own list
    const double s = s_sc[i];
    const int64_t id = s_id[i];
    int rank = j;
    for (int g2 = 0; g2 < G && rank < nout; ++g2) {
      if (g2 == g) continue;
      // entries of list g2 that precede (s, id); equal (score, id) pairs cannot come from two lists of a sharded
      // corpus — if they ever do, the lower list goes first, so the merged places stay a permutation
      int lo = 0, hi = s_cnt[g2];
      const double* sc2 = s_sc + g2 * k;
      const int64_t* id2 = s_id + g2 * k;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const double sm = sc2[mid];
        const int64_t im = id2[mid];
        const bool before = sm > s || (sm == s && (im < id || (im == id && g2 < g)));
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < nout) {
      if (row < B) {
        d_sc[(size_t)row * k_sem + rank] = s;
        d_ids[(size_t)row * k_sem + rank] = id;
      } else {
        const int q = row - B;
        l_sc[(size_t)q * k_lex + rank] = (float)s;
        l_ids[(size_t)q * k_lex + rank] = id;
      }
    }
  }
  if (row < B) {
    if (threadIdx.x == 0) d_cnt[row] = nout;
    for (int i = nout + threadIdx.x; i < k_sem; i += blockDim.x) {
      d_sc[(size_t)row * k_sem + i] = -INFINITY;
      d_ids[(size_t)row * k_sem + i] = -1;
    }
  } else {
    const int q = row - B;
    if (threadIdx.x == 0) l_cnt[q] = nout;
    for (int i = nout + threadIdx.x; i < k_lex; i += blockDim.x) {
      l_sc[(size_t)q * k_lex + i] = 0.f;
      l_ids[(size_t)q * k_lex + i] = -1;
    }
  }
}

// One CTA per (channel, query): merge the G lists out of the gathered messages, write the channel's final list in
// the channel's own output format (semantic: f64 scores, -inf padding; lexical: f32 scores, 0 padding as
// thr_bm25_topk writes them).
// sig != nullptr (pushed messages): sig[g] >= seq says rank g's message of this step has landed in `gathered`.
// The wait is for another PROCESS (its host may be late by a page fault, an allocation, a slow first step), so its
// bound is far longer than the on-chip pipelines' 2 s: a dead peer still surfaces as THR_ETIMEOUT, a slow one does not.
constexpr unsigned long long kPeerWatchdogNs = 60ull * 1000000000ull;
__global__ void __launch_bounds__(256) exchange_merge_kernel(const uint8_t* gathered, size_t msg_bytes, int G, int B,
                                                             int k_sem, int k_lex, int k, int64_t* d_ids, double* d_sc,
                                                             int32_t* d_cnt, int64_t* l_ids, float* l_sc,
                                                             int32_t* l_cnt, const unsigned long long* sig,
                                                             unsigned long long seq, thr_dev_status* status) {
  __shared__ double s_sc[kMergeMax];
  __shared__ int64_t s_id[kMergeMax];
  const int row = blockIdx.x, tid = threadIdx.x;
  if (sig) {
    if (tid < G) {   // bounded wait: a rank that never arrives surfaces as THR_ETIMEOUT, not as a hung GPU
      uint64_t t0 = 0;
      for (uint32_t spin = 1;; ++spin) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(sig + tid) : "memory");
        if (v >= seq) break;
        if ((spin & 1023u) == 0) {
          const uint64_t now = global_timer_ns();
          if (t0 == 0) t0 = now;
          if (now - t0 > kPeerWatchdogNs) { dev_report(status, THR_ETIMEOUT, 520, (long long)tid); __trap(); }
        }
      }
    }
    __syncthreads();
  }
  // Every rank's list is sorted already (score desc, id asc): merge by RANK instead of sorting — an entry's place in
  // the merged list is its place in its own list plus, for every other list, the number of entries that precede it
  // there (a binary search).  No exchange network, no barrier between the staging and the output.
  const int n = G * k;
  const size_t nrow = (size_t)2 * B * k;
  __shared__ int s_cnt[64];
  if (tid < G) {
    const uint8_t* m = gathered + (size_t)tid * msg_bytes;
    s_cnt[tid] = min(max(__ldcg((const int32_t*)(m + 2 * nrow * 8) + row), 0), k);   // L2 is the point of coherence for peer stores
  }
  __syncthreads();
  for (int i = tid; i < n; i += 256) {
    const int g = i / k, j = i - g * k;
    if (j < s_cnt[g]) {
      const uint8_t* m = gathered + (size_t)g * msg_bytes;
      s_sc[i] = __ldcg((const double*)m + (size_t)row * k + j);
      s_id[i] = (int64_t)__ldcg((const long long*)(m + nrow * 8) + (size_t)row * k + j);
    }
  }
  __syncthreads();
  merge_staged_write(s_sc, s_id, s_cnt, G, k, row, B, k_sem, k_lex, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt);
}

// thr_shard_merge: one CTA per (channel, query) row.  The sources are other handles' K1 / K2 outputs, possibly on other
// GPUs (every load a peer round trip), so the row's S lists are first staged into shared memory with coalesced loads
// (one pass over counts, one over entries, lexical f32 scores widened to f64 exactly); the binary searches of the
// rank merge then run on shared memory only.  Dynamic shared memory: S_max * k * 16 bytes.
constexpr int kShardMergeMax = 12288;   // entries staged per row: 192 KB of shared memory
struct ShardSources {
  const int64_t* const* d_ids; const double* const* d_sc; const int32_t* const* d_cnt; const float* const* d_gap;
  const int64_t* const* l_ids; const float* const* l_sc; const int32_t* const* l_cnt;
  int S_sem, S_lex;
};

__global__ void __launch_bounds__(256) shard_merge_kernel(const ShardSources src, int B, int k_sem, int k_lex,
                                                          int64_t* d_ids, double* d_sc, int32_t* d_cnt, float* d_gap,
                                                          int64_t* l_ids, float* l_sc, int32_t* l_cnt) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ int s_cnt[64];
  const int row = blockIdx.x, tid = threadIdx.x;
  const bool sem = row < B;
  const int q = sem ? row : row - B;
  const int S = sem ? src.S_sem : src.S_lex;
  const int k = sem ? k_sem : k_lex;
  double* s_sc = (double*)smem;
  int64_t* s_id = (int64_t*)(smem + (size_t)S * k * sizeof(double));
  __shared__ float s_gap[64];
  if (tid < S) {
    s_cnt[tid] = min(max(sem ? src.d_cnt[tid][q] : src.l_cnt[tid][q], 0), k);
    if (sem && d_gap) s_gap[tid] = src.d_gap[tid][q];
  }
  __syncthreads();
  if (sem && d_gap && tid == 0) {   // certificate of the merged list: if every source's top-k is exact, so is theirs
    float g = INFINITY;
    for (int s = 0; s < S; ++s) g = fminf(g, s_gap[s]);
    d_gap[q] = g;
  }
  const int n = S * k;
  for (int i = tid; i < n; i += blockDim.x) {
    const int g = i / k, j = i - g * k;
    if (j < s_cnt[g]) {
      const size_t o = (size_t)q * k + j;
      s_sc[i] = sem ? src.d_sc[g][o] : (double)src.l_sc[g][o];
      s_id[i] = sem ? src.d_ids[g][o] : src.l_ids[g][o];
    }
  }
  __syncthreads();
  merge_staged_write(s_sc, s_id, s_cnt, S, k, row, B, k_sem, k_lex, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt);
}
}  // namespace

extern "C" {

int thr_fuse(thr_handle* h, int variant, int tie_mode, int B, const int64_t* lex_ids,
             const int32_t* lex_off, const double* lex_sc, const int64_t* sem_ids,
             const int32_t* sem_off, const double* sem_sc, const int64_t* gr_ids,
             const int32_t* gr_off, const double* gr_sc, const double* weights, int rrf_k,
             double safety_thr, double alpha, int denoise, int top_k, int max_out,
             int64_t* out_ids, double* out_rrf, int32_t* out_ranks, double* out_raw,
             int32_t* out_count, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0, "thr_fuse: B < 0");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, variant >= THR_FUSE_RAG2 && variant <= THR_FUSE_RAG1, "thr_fuse: unknown variant %d", variant);
  THR_REQUIRE(h, tie_mode == THR_TIE_INSERTION || tie_mode == THR_TIE_CHUNK_ID, "thr_fuse: unknown tie_mode %d", tie_mode);
  THR_REQUIRE(h, weights && out_ids && out_rrf && out_ranks && out_count, "thr_fuse: NULL weights/output");
  THR_REQUIRE(h, (lex_ids == nullptr || lex_off) && (sem_ids == nullptr || sem_off) && (gr_ids == nullptr || gr_off),
              "thr_fuse: ids without offsets");
  THR_REQUIRE(h, max_out >= 1, "thr_fuse: max_out < 1");
  THR_REQUIRE(h, rrf_k >= 0, "thr_fuse: rrf_k < 0");
  FuseArgs a;
  a.ids[0] = lex_ids; a.off[0] = lex_off; a.sc[0] = lex_sc;
  a.ids[1] = sem_ids; a.off[1] = sem_off; a.sc[1] = sem_sc;
  a.ids[2] = gr_ids;  a.off[2] = gr_off;  a.sc[2] = gr_sc;
  a.weights = weights; a.rrf_k = rrf_k; a.safety_thr = safety_thr; a.alpha = alpha;
  a.denoise = denoise; a.top_k = top_k; a.max_out = max_out; a.tie_mode = tie_mode;
  a.out_ids = out_ids; a.out_rrf = out_rrf; a.out_ranks = out_ranks; a.out_raw = out_raw;
  a.out_count = out_count; a.status = h->d_status;
  cudaStream_t s = (cudaStream_t)stream;
  const int tok = thr_prof_begin(h, THR_PROF_FUSE, s);
  if (variant == THR_FUSE_RAG2) fuse_kernel<THR_FUSE_RAG2><<<B, kFuseThreads, 0, s>>>(a);
  else if (variant == THR_FUSE_LIB) fuse_kernel<THR_FUSE_LIB><<<B, kFuseThreads, 0, s>>>(a);
  else fuse_kernel<THR_FUSE_RAG1><<<B, kFuseThreads, 0, s>>>(a);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "fuse_kernel");
  return THR_OK;
}

int thr_fuse_ranked(thr_handle* h, int B, const int32_t* off, const int32_t* ranks, const double* weights,
                    int rrf_k, double* out_rrf, int32_t* out_order, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && rrf_k >= 0, "thr_fuse_ranked: bad B / rrf_k");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, off && ranks && weights && out_rrf && out_order, "thr_fuse_ranked: NULL argument");
  const int tok = thr_prof_begin(h, THR_PROF_FUSE, (cudaStream_t)stream);
  fuse_ranked_kernel<<<B, kFuseThreads, 0, (cudaStream_t)stream>>>(off, ranks, weights, rrf_k, out_rrf, out_order,
                                                                   h->d_status);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "fuse_ranked_kernel");
  return THR_OK;
}

int thr_safety(thr_handle* h, int B, const int32_t* off, const double* rerank,
               const uint8_t* has_rerank, const double* rrf, double threshold, double alpha,
               int top_k, uint8_t* keep, uint8_t* refused, double* max_score, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0, "thr_safety: B < 0");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, off && rrf && keep && refused && max_score, "thr_safety: NULL argument");
  THR_REQUIRE(h, has_rerank == nullptr || rerank != nullptr, "thr_safety: has_rerank without rerank");
  const int tok = thr_prof_begin(h, THR_PROF_SAFETY, (cudaStream_t)stream);
  safety_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(B, off, rerank, has_rerank, rrf, threshold,
                                                               alpha, top_k, keep, refused, max_score);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "safety_kernel");
  return THR_OK;
}

int thr_merge_topk(thr_handle* h, const double* scores, const int64_t* ids, const int32_t* counts,
                   int G, int B, int k_in, int k_out, double* out_scores, int64_t* out_ids,
                   int32_t* out_count, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, G >= 1 && B >= 0 && k_in >= 1 && k_out >= 1, "thr_merge_topk: bad sizes");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, (int64_t)G * k_in <= kMergeMax, "thr_merge_topk: G*k_in = %lld exceeds %d",
              (long long)G * k_in, kMergeMax);
  THR_REQUIRE(h, k_out <= 256, "thr_merge_topk: k_out > 256");
  THR_REQUIRE(h, scores && ids && out_scores && out_ids && out_count, "thr_merge_topk: NULL argument");
  const int tok = thr_prof_begin(h, THR_PROF_MERGE, (cudaStream_t)stream);
  merge_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(scores, ids, counts, G, B, k_in, k_out, out_scores,
                                                    out_ids, out_count);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "merge_kernel");
  return THR_OK;
}

int64_t thr_exchange_msg_bytes(int B, int k_sem, int k_lex) {
  const int64_t k = k_sem > k_lex ? k_sem : k_lex;
  return 2 * (2 * (int64_t)B * k * 8) + 2 * (int64_t)B * 4;
}

int thr_exchange_pack(thr_handle* h, const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                      const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt, int B, int k_sem, int k_lex,
                      void* msg, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && k_sem >= 1 && k_lex >= 1, "thr_exchange_pack: bad sizes");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, d_ids && d_sc && d_cnt && l_ids && l_sc && l_cnt && msg, "thr_exchange_pack: NULL argument");
  THR_REQUIRE(h, ((uintptr_t)msg & 7u) == 0, "thr_exchange_pack: msg must be 8-byte aligned");
  const int k = k_sem > k_lex ? k_sem : k_lex;
  const size_t n = (size_t)2 * B * k;
  const int blocks = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
  const int tok = thr_prof_begin(h, THR_PROF_MERGE, (cudaStream_t)stream);
  exchange_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, B, k_sem, k_lex,
                                                                 k, (uint8_t*)msg);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "exchange_pack_kernel");
  return THR_OK;
}

int thr_exchange_merge_pushed(thr_handle* h, const void* gathered, const uint64_t* signals, uint64_t seq, int G, int B,
                              int k_sem, int k_lex, int64_t* d_ids, double* d_sc, int32_t* d_cnt, int64_t* l_ids,
                              float* l_sc, int32_t* l_cnt, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, G >= 1 && B >= 0 && k_sem >= 1 && k_lex >= 1, "thr_exchange_merge: bad sizes");
  THR_REQUIRE(h, G <= 256, "thr_exchange_merge: more than 256 ranks");
  if (B == 0) return THR_OK;
  const int k = k_sem > k_lex ? k_sem : k_lex;
  THR_REQUIRE(h, (int64_t)G * k <= kMergeMax, "thr_exchange_merge: G*k = %lld exceeds %d", (long long)G * k, kMergeMax);
  THR_REQUIRE(h, G <= 64, "thr_exchange_merge: %d ranks exceed 64", G);
  THR_REQUIRE(h, k_sem <= 256 && k_lex <= 256, "thr_exchange_merge: k > 256");
  THR_REQUIRE(h, gathered && d_ids && d_sc && d_cnt && l_ids && l_sc && l_cnt, "thr_exchange_merge: NULL argument");
  THR_REQUIRE(h, ((uintptr_t)gathered & 7u) == 0, "thr_exchange_merge: buffer must be 8-byte aligned");
  const int tok = thr_prof_begin(h, THR_PROF_MERGE, (cudaStream_t)stream);
  exchange_merge_kernel<<<2 * B, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)gathered,
                                                                 (size_t)thr_exchange_msg_bytes(B, k_sem, k_lex), G, B, k_sem,
                                                                 k_lex, k, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt,
                                                                 (const unsigned long long*)signals, (unsigned long long)seq,
                                                                 h->d_status);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "exchange_merge_kernel");
  return THR_OK;
}

int thr_exchange_merge(thr_handle* h, const void* gathered, int G, int B, int k_sem, int k_lex, int64_t* d_ids,
                       double* d_sc, int32_t* d_cnt, int64_t* l_ids, float* l_sc, int32_t* l_cnt, void* stream) {
  return thr_exchange_merge_pushed(h, gathered, nullptr, 0, G, B, k_sem, k_lex, d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt,
                                   stream);
}

int thr_exchange_push(thr_handle* h, const int64_t* d_ids, const double* d_sc, const int32_t* d_cnt,
                      const int64_t* l_ids, const float* l_sc, const int32_t* l_cnt, int B, int k_sem, int k_lex,
                      void* const* peer_bufs, int64_t buf_off, uint64_t* const* peer_signals, int64_t sig_off, int rank,
                      int G, uint64_t seq, uint32_t* done_counter, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && k_sem >= 1 && k_lex >= 1 && G >= 1 && rank >= 0 && rank < G, "thr_exchange_push: bad sizes");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, d_ids && d_sc && d_cnt && l_ids && l_sc && l_cnt && peer_bufs && peer_signals && done_counter,
              "thr_exchange_push: NULL argument");
  THR_REQUIRE(h, buf_off >= 0 && (buf_off & 7) == 0 && sig_off >= 0 && (sig_off & 7) == 0,
              "thr_exchange_push: offsets must be non-negative multiples of 8");
  const int k = k_sem > k_lex ? k_sem : k_lex;
  const size_t n = (size_t)2 * B * k;
  const int blocks = (int)((n + 255) / 256 < 592 ? (n + 255) / 256 : 592);
  const size_t slot_off = (size_t)buf_off + (size_t)rank * (size_t)thr_exchange_msg_bytes(B, k_sem, k_lex);
  const int tok = thr_prof_begin(h, THR_PROF_MERGE, (cudaStream_t)stream);
  exchange_push_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      d_ids, d_sc, d_cnt, l_ids, l_sc, l_cnt, B, k_sem, k_lex, k, (uint8_t* const*)peer_bufs, slot_off,
      (unsigned long long* const*)peer_signals, (size_t)sig_off, rank, G, (unsigned long long)seq, done_counter);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "exchange_push_kernel");
  return THR_OK;
}


int thr_shard_merge(thr_handle* h, int B, int k_sem, int k_lex, int S_sem, const int64_t* const* d_ids_src,
                    const double* const* d_sc_src, const int32_t* const* d_cnt_src, const float* const* d_gap_src,
                    int S_lex, const int64_t* const* l_ids_src, const float* const* l_sc_src,
                    const int32_t* const* l_cnt_src, int64_t* d_ids, double* d_sc, int32_t* d_cnt, float* d_gap,
                    int64_t* l_ids, float* l_sc, int32_t* l_cnt, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && k_sem >= 1 && k_lex >= 1 && k_sem <= 256 && k_lex <= 256,
              "thr_shard_merge: need 1 <= k_sem, k_lex <= 256");
  THR_REQUIRE(h, S_sem >= 1 && S_sem <= 64 && S_lex >= 1 && S_lex <= 64, "thr_shard_merge: need 1 <= S <= 64 per channel");
  if (B == 0) return THR_OK;
  const int64_t n_max = (int64_t)S_sem * k_sem > (int64_t)S_lex * k_lex ? (int64_t)S_sem * k_sem : (int64_t)S_lex * k_lex;
  if (n_max > kShardMergeMax)
    return thr_fail(h, THR_EUNSUPPORTED, "thr_shard_merge: S * k = %lld exceeds %d", (long long)n_max, kShardMergeMax);
  THR_REQUIRE(h, d_ids_src && d_sc_src && d_cnt_src && l_ids_src && l_sc_src && l_cnt_src && d_ids && d_sc && d_cnt &&
                     l_ids && l_sc && l_cnt && (d_gap == nullptr || d_gap_src != nullptr),
              "thr_shard_merge: NULL argument");
  const size_t smem = (size_t)n_max * 16;
  THR_CUDA(h, cudaFuncSetAttribute(shard_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ShardSources src;
  src.d_ids = d_ids_src; src.d_sc = d_sc_src; src.d_cnt = d_cnt_src; src.d_gap = d_gap_src;
  src.l_ids = l_ids_src; src.l_sc = l_sc_src; src.l_cnt = l_cnt_src; src.S_sem = S_sem; src.S_lex = S_lex;
  const int tok = thr_prof_begin(h, THR_PROF_MERGE, (cudaStream_t)stream);
  shard_merge_kernel<<<2 * B, 256, smem, (cudaStream_t)stream>>>(src, B, k_sem, k_lex, d_ids, d_sc, d_cnt, d_gap, l_ids,
                                                                 l_sc, l_cnt);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "shard_merge_kernel");
  return THR_OK;
}

}  // extern "C"
