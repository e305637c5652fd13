// rerank.cu — the batched rerank stage around K4: candidate ids -> token-store rows before thr_maxsim, and
// `_rerank`'s ordering plus `_apply_safety` after it.
//
// Reference: RAG2Retriever.retrieve steps 4-6 (src/voice_agent/rag2/retrieval.py:175-191): the fused list is cut
// to rag2_rerank_top_k, every candidate gets a rerank_score, the list is re-ordered by
// `sorted(candidates, key=lambda x: x.rerank_score or 0, reverse=True)` (stable; :455) and _apply_safety (:461-495)
// keeps what clears the threshold.  The reference does this one query at a time in Python; here one CTA per query.
// With a sharded corpus each rank scores the candidates whose chunks it owns (rerank_rows_kernel maps the others to
// -1, which thr_maxsim scores -inf), the ranks exchange the [B, C] score matrix with ONE all-reduce(MAX), and this
// kernel runs replicated on the merged scores.  In one process (thr_rerank_finish_shards) the kernel takes the element-
// wise max of the shards' [B, C] arrays itself, read through peer memory.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kRerankMaxC = 256;

__global__ void rerank_rows_kernel(const int64_t* ids, const int32_t* count, int B, int C, int stride,
                                   int64_t id_lo, int64_t id_hi, int64_t period, int64_t row_off, int64_t* rows) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int q = i / C, j = i % C;
  int64_t r = -1;
  if (j < count[q]) {
    const int64_t id = ids[(size_t)q * stride + j];
    if (id >= id_lo && id < id_hi) r = period > 0 ? (id - id_lo + row_off) % period : id - id_lo + row_off;
  }
  rows[i] = r;
}

struct FinishArgs {
  int B, C, stride, Tq, top_k;
  const int64_t* ids;      // [B, stride] fused ids (-1 padded)
  const double* rrf;       // [B, stride]
  const int32_t* count;    // [B]
  const float* raw;        // [B, C] MaxSim sums; -inf = nobody scored the candidate
  const float* const* raws;  // or (raw == nullptr) n_raw such arrays, one per shard: their element-wise max
  int n_raw;
  double threshold, alpha;
  int64_t* out_ids;        // [B, C] in the reranked order, -1 padded
  double* out_rerank;      // [B, C] rerank_score in [0, 1] (-1 where the candidate has none)
  double* out_rrf;         // [B, C]
  uint8_t* out_keep;       // [B, C] survives _apply_safety
  int32_t* out_n;          // [B] candidates considered (min(count, C))
  uint8_t* refused;        // [B]
  double* max_score;       // [B]
};

__global__ void __launch_bounds__(kRerankMaxC) rerank_finish_kernel(const FinishArgs a) {
  __shared__ double s_key[kRerankMaxC];
  __shared__ int s_pos[kRerankMaxC];
  __shared__ double s_red[kRerankMaxC / 32];
  __shared__ int s_cnt[kRerankMaxC / 32];
  __shared__ float s_raw[kRerankMaxC];
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(min(a.count[q], a.C), kRerankMaxC);
  // the candidate's raw score, read once (coalesced; the shards' arrays may be in peer memory)
  if (tid < n) {
    const size_t o = (size_t)q * a.C + tid;
    float r;
    if (a.raw) {
      r = a.raw[o];
    } else {
      r = a.raws[0][o];
      for (int s = 1; s < a.n_raw; ++s) r = fmaxf(r, a.raws[s][o]);
    }
    s_raw[tid] = r;
  }
  // rerank_score = min(1, max(0, 0.5 * (s / Tq + 1))) in fp64, one rounded operation at a time (the Python of
  // GpuMaxSimReranker.score_rows); a candidate nobody scored has none.
  double score = -1.0;
  bool has = false;
  if (tid < n) {
    const float r = s_raw[tid];
    if (r > -CUDART_INF_F) {
      has = true;
      double x = __dmul_rn(0.5, __dadd_rn(__ddiv_rn((double)r, (double)a.Tq), 1.0));
      score = fmin(1.0, fmax(0.0, x));
    }
  }
  // sorted(..., key=rerank_score or 0, reverse=True): descending key, equal keys keep their order
  s_key[tid] = tid < n ? (has ? score : 0.0) : -CUDART_INF;
  s_pos[tid] = tid;
  __syncthreads();
  for (int size = 2; size <= kRerankMaxC; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const int i = tid;
      const int j = i ^ stride;
      if (j > i) {
        const bool desc = (i & size) == 0;
        const double ki = s_key[i], kj = s_key[j];
        const int pi = s_pos[i], pj = s_pos[j];
        const bool i_first = ki > kj || (ki == kj && pi < pj);   // i belongs before j in the final order
        if (desc ? !i_first : i_first) { s_key[i] = kj; s_key[j] = ki; s_pos[i] = pj; s_pos[j] = pi; }
      }
      bitonic_stage_sync(size, stride, kRerankMaxC, 16);
    }
  }
  const int src = s_pos[tid];                       // the candidate that lands at position tid
  // every thread needs (score, has) of candidate `src`: recompute it from the inputs
  double sc = -1.0, rr = 0.0;
  bool hs = false;
  int64_t id = -1;
  if (tid < n) {
    const float r = s_raw[src];
    if (r > -CUDART_INF_F) {
      hs = true;
      sc = fmin(1.0, fmax(0.0, __dmul_rn(0.5, __dadd_rn(__ddiv_rn((double)r, (double)a.Tq), 1.0))));
    }
    rr = a.rrf[(size_t)q * a.stride + src];
    id = a.ids[(size_t)q * a.stride + src];
  }
  // _apply_safety on the reordered list: s_i = rerank_score or rrf_score (None and 0.0 are falsy)
  const double eff = tid < n ? ((hs && sc != 0.0) ? sc : rr) : -CUDART_INF;
  double mx = eff;
  for (int s = 16; s > 0; s >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = s_red[0];
  for (int w = 1; w < kRerankMaxC / 32; ++w) mx = fmax(mx, s_red[w]);
  const bool ref = n == 0 || mx < a.threshold;
  const double floor_ = __dmul_rn(a.alpha, mx);
  const bool pass = !ref && tid < n && eff >= floor_;
  const unsigned bal = __ballot_sync(0xffffffffu, pass);
  if (lane == 0) s_cnt[warp] = __popc(bal);
  __syncthreads();
  int before = __popc(bal & ((1u << lane) - 1u));
  for (int w = 0; w < warp; ++w) before += s_cnt[w];
  if (tid < a.C) {
    const size_t o = (size_t)q * a.C + tid;
    a.out_ids[o] = tid < n ? id : -1;
    a.out_rerank[o] = tid < n ? sc : -1.0;
    a.out_rrf[o] = tid < n ? rr : 0.0;
    a.out_keep[o] = (pass && before < a.top_k) ? 1 : 0;
  }
  if (tid == 0) {
    a.out_n[q] = n;
    a.refused[q] = ref ? 1 : 0;
    a.max_score[q] = n == 0 ? 0.0 : mx;
  }
}

}  // namespace

extern "C" {

int thr_rerank_rows(thr_handle* h, const int64_t* ids, const int32_t* count, int B, int C, int stride,
                    int64_t id_lo, int64_t id_hi, int64_t period, int64_t row_off, int64_t* rows, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && C >= 1 && stride >= C, "thr_rerank_rows: need C >= 1 and stride >= C");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, ids && count && rows && row_off >= 0, "thr_rerank_rows: NULL argument or negative row_off");
  const int tok = thr_prof_begin(h, THR_PROF_RERANK, (cudaStream_t)stream);
  rerank_rows_kernel<<<(B * C + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ids, count, B, C, stride, id_lo, id_hi, period, row_off, rows);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "rerank_rows_kernel");
  return THR_OK;
}

static int rerank_finish_launch(thr_handle* h, const char* name, int B, int C, int stride, const int64_t* ids,
                                const double* rrf, const int32_t* count, const float* raw, const float* const* raws,
                                int n_raw, int Tq, double threshold, double alpha, int top_k, int64_t* out_ids,
                                double* out_rerank, double* out_rrf, uint8_t* out_keep, int32_t* out_n, uint8_t* refused,
                                double* max_score, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && C >= 1 && C <= kRerankMaxC && stride >= C && Tq >= 1, "%s: need 1 <= C <= %d, stride >= C, Tq >= 1", name, kRerankMaxC);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, ids && rrf && count && (raw || raws) && out_ids && out_rerank && out_rrf && out_keep && out_n && refused && max_score,
              "%s: NULL argument", name);
  FinishArgs a;
  a.B = B; a.C = C; a.stride = stride; a.Tq = Tq; a.top_k = top_k; a.ids = ids; a.rrf = rrf; a.count = count; a.raw = raw;
  a.raws = raws; a.n_raw = n_raw;
  a.threshold = threshold; a.alpha = alpha; a.out_ids = out_ids; a.out_rerank = out_rerank; a.out_rrf = out_rrf;
  a.out_keep = out_keep; a.out_n = out_n; a.refused = refused; a.max_score = max_score;
  const int tok = thr_prof_begin(h, THR_PROF_RERANK, (cudaStream_t)stream);
  rerank_finish_kernel<<<B, kRerankMaxC, 0, (cudaStream_t)stream>>>(a);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, "rerank_finish_kernel");
  return THR_OK;
}

int thr_rerank_finish(thr_handle* h, int B, int C, int stride, const int64_t* ids, const double* rrf,
                      const int32_t* count, const float* raw, int Tq, double threshold, double alpha, int top_k,
                      int64_t* out_ids, double* out_rerank, double* out_rrf, uint8_t* out_keep, int32_t* out_n,
                      uint8_t* refused, double* max_score, void* stream) {
  return rerank_finish_launch(h, "thr_rerank_finish", B, C, stride, ids, rrf, count, raw, nullptr, 0, Tq, threshold, alpha,
                              top_k, out_ids, out_rerank, out_rrf, out_keep, out_n, refused, max_score, stream);
}

int thr_rerank_finish_shards(thr_handle* h, int B, int C, int stride, const int64_t* ids, const double* rrf,
                             const int32_t* count, const float* const* raws, int S, int Tq, double threshold,
                             double alpha, int top_k, int64_t* out_ids, double* out_rerank, double* out_rrf,
                             uint8_t* out_keep, int32_t* out_n, uint8_t* refused, double* max_score, void* stream) {
  if (h && S < 1) return thr_fail(h, THR_EINVAL, "thr_rerank_finish_shards: S < 1");
  return rerank_finish_launch(h, "thr_rerank_finish_shards", B, C, stride, ids, rrf, count, nullptr, raws, S, Tq, threshold,
                              alpha, top_k, out_ids, out_rerank, out_rrf, out_keep, out_n, refused, max_score, stream);
}

}  // extern "C"
