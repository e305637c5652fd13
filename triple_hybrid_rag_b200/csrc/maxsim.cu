// maxsim.cu — K4: late-interaction MaxSim rerank.
//
// Stands where RAG2Retriever._rerank calls Qwen3VLReranker._rerank_batch_native(query, documents)
//   (src/voice_agent/rag2/retrieval.py:405-459, src/voice_agent/retrieval/reranker.py:287-354):
//   one relevance score per candidate, in input order.  The reference scores with an HTTP
//   cross-encoder; BASELINE.json's north_star replaces that with
//     score(q, c) = sum_{i < q_len} max_{j < d_len} <Qtok[q,i,:], Dtok[c,j,:]>      (d = 128).
//
// One CTA handles a (query, slice of its candidates) unit: the query's token tile (A operand,
// 128 rows, rows >= q_len are ignored by the epilogue) stays in shared memory, candidates stream
// through a TMA ring (one candidate = Td x 128 bf16 = one stage), one tcgen05.mma chain of 8 K-steps
// per candidate into one of 4 TMEM accumulators (128 lanes x Td columns), and the epilogue does the
// row max (over TMEM columns, in registers) and the sum over query tokens.  For Tq <= 32 (<= 64) the
// query tile is stacked 4 (2) times in the 128 MMA rows: every epilogue warp then owns valid TMEM lanes and
// scans only a quarter (half) of the doc-token columns; partial maxima meet in shared memory.
// The scores matrix [Tq x Td] never leaves the SM.  At Tq = 32 the kernel is HBM-bound
// (2*Tq = 64 FLOP per byte of candidate tokens).
//
// maxsim_kernel<true> scores a residual-compressed store (thr_maxsim_packed, format in include/thr.h): the query
// tile still arrives by TMA, but eight decoder warps replace the candidates' TMA loads.  They rebuild each candidate's
// bf16 tokens (centroid row through L2 + 2-bit residual code, fp32 add, round to bf16) into the same swizzled stage
// layout TMA writes, so the MMA and epilogue below are shared and the packed score is bit-identical to thr_maxsim on
// the decoded store.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kD = 128;             // token embedding width
constexpr int kStagesM = 5;
constexpr int kAccM = 4;            // TMEM accumulators, 128 columns apart
constexpr int kThreadsM = 192;      // warps 0-3 epilogue, 4 producer, 5 MMA
constexpr int kDecGroupThreads = 128;                     // packed: one decoder group = 4 warps, fills every other stage
constexpr int kDecGroups = 2;
constexpr int kThreadsPacked = kThreadsM + kDecGroups * kDecGroupThreads;   // warps 6-13 decode
constexpr int kATileBytes = 128 * kD * 2;                 // 32 KB (two 64-wide halves)
constexpr int kMaxStageBytes = 128 * kD * 2;              // Td <= 128
constexpr int kSmemM = kATileBytes + kStagesM * kMaxStageBytes + 1024 + 512;

struct MaxSimArgs {
  int B, Tq, Td, C;
  int64_t n_docs;
  const int32_t* q_len;
  const int32_t* d_len;
  const int64_t* cand;
  float* out;
  int slices;       // candidate slices per query
  int per_slice;    // candidates per slice
  int reps;         // copies of the query tile stacked in the 128 MMA rows (4 for Tq <= 32, 2 for Tq <= 64, else 1)
  thr_dev_status* status;
  // packed store (maxsim_kernel<true> only); n_docs is its row count
  const uint32_t* codes;      // [n_docs, Td, 8]
  const int32_t* cids;        // [n_docs, Td]
  const uint4* centroids;     // [n_centroids, 128] bf16, 16 rows of 16 B per centroid
  const float* weights;       // [128, 4]
  int64_t n_centroids;
};

// Decoder group `grp` of maxsim_kernel<true>: rebuilds the candidates of stage iterations it = grp (mod kDecGroups)
// into their ring stage, exactly as TMA would have written the decoded bf16 store (SWIZZLE_128B, K-major: 16-byte
// chunk c of token j in chunk slot c ^ (j & 7) of the token's 128-byte row in each 64-column half).  Thread t owns
// the 8 dimensions of 16-byte chunk q = t % 16 for every token it touches, so its 32 reconstruction values stay in
// registers.
__device__ __forceinline__ void maxsim_decode_stages(const MaxSimArgs& a, int grp, int t, uint32_t stage_base,
                                                     uint32_t stage_stride, uint32_t bar_full0, uint32_t bar_empty0,
                                                     int units) {
  const int q = t & 15;               // chunk: dims 8q .. 8q+7, code word q / 2, bits 16 * (q & 1) + 2e
  const int tok0 = t >> 4;            // tokens tok0, tok0 + 8, ...
  float w0[8], w1[8], w2[8], w3[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float4 v = reinterpret_cast<const float4*>(a.weights)[8 * q + e];
    w0[e] = v.x; w1[e] = v.y; w2[e] = v.z; w3[e] = v.w;
  }
  const uint32_t half_bytes = (uint32_t)a.Td * 128u;
  const uint32_t dst_q = (uint32_t)(q >> 3) * half_bytes;
  const uint32_t cmax = (uint32_t)(a.n_centroids - 1);
  uint32_t it = 0;
  for (int u = blockIdx.x; u < units; u += gridDim.x) {
    const int b = u / a.slices, sl = u % a.slices;
    const int c_lo = sl * a.per_slice, c_hi = min(a.C, c_lo + a.per_slice);
    for (int c = c_lo; c < c_hi; ++c, ++it) {
      if ((int)(it % kDecGroups) != grp) continue;
      const int s = it % kStagesM;
      const uint32_t ph = (it / kStagesM) & 1u;
      int64_t doc = a.cand[(size_t)b * a.C + c];
      if (doc < 0 || doc >= a.n_docs) doc = 0;  // slot is skipped by the epilogue
      const int64_t tok_base = doc * a.Td;      // 64-bit: the packed store has no 2^31-token limit
      const uint32_t dst = stage_base + (uint32_t)s * stage_stride + dst_q;
      mbar_wait_relaxed(bar_empty0 + 8u * s, ph ^ 1u, a.status, 530);
      for (int j0 = 0; j0 < a.Td; j0 += 64) {
        uint32_t cid[8], word[8];
        uint4 cen[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int64_t tok = tok_base + j0 + tok0 + 8 * i;
          cid[i] = min((uint32_t)__ldcs(a.cids + tok), cmax);   // never dereference a cid outside the table
          word[i] = __ldcs(a.codes + tok * 8 + (q >> 1)) >> (16 * (q & 1));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) cen[i] = __ldg(a.centroids + (int64_t)cid[i] * 16 + q);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t in[4] = {cen[i].x, cen[i].y, cen[i].z, cen[i].w};
          uint32_t outw[4];
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            float x[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int e = 2 * p + h;
              const uint32_t code = (word[i] >> (2 * e)) & 3u;
              const float wv = (code & 2u) ? ((code & 1u) ? w3[e] : w2[e]) : ((code & 1u) ? w1[e] : w0[e]);
              const float cv = __uint_as_float(h ? (in[p] & 0xffff0000u) : (in[p] << 16));
              x[h] = __fadd_rn(cv, wv);
            }
            const __nv_bfloat162 r2 = __floats2bfloat162_rn(x[0], x[1]);
            outw[p] = *reinterpret_cast<const uint32_t*>(&r2);
          }
          const int j = j0 + tok0 + 8 * i;
          const uint32_t addr = dst + (uint32_t)j * 128u + ((uint32_t)((q & 7) ^ (j & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(outw[0]), "r"(outw[1]),
                       "r"(outw[2]), "r"(outw[3])
                       : "memory");
        }
      }
      fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core's async proxy
      mbar_arrive(bar_full0 + 8u * s);
    }
  }
}

// kPacked = false: candidates arrive by TMA from a bf16 store (map_d); true: decoder warps build them from the packed
// store in `a` (map_d unused).  Everything else is one code path.
template <bool kPacked>
__global__ void __launch_bounds__(kPacked ? kThreadsPacked : kThreadsM, 1)
maxsim_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_d,
              const MaxSimArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_smem = smem_base;                       // [2 halves][128 rows][64] bf16
  const uint32_t half_bytes_b = (uint32_t)a.Td * 64 * 2;   // one K-half of a candidate
  const uint32_t stage_bytes = 2 * half_bytes_b;
  auto b_smem = [&](int s) { return smem_base + kATileBytes + (uint32_t)s * kMaxStageBytes; };
  const uint32_t bar_base = smem_base + kATileBytes + kStagesM * kMaxStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStagesM + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStagesM + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStagesM + kAccM + s); };
  const uint32_t qfull_bar = bar_base + 8u * (2 * kStagesM + 2 * kAccM);
  const uint32_t qempty_bar = qfull_bar + 8u;
  const uint32_t tmem_slot = qempty_bar + 8u;
  __shared__ float pmax[kAccM][128];   // [accumulator][replica * rows_per_rep + token]: partial row maxima

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    // a packed stage is full once every thread of its decoder group has arrived
    for (int s = 0; s < kStagesM; ++s) { mbar_init(full_bar(s), kPacked ? kDecGroupThreads : 1); mbar_init(empty_bar(s), 1); }
    for (int s = 0; s < kAccM; ++s) { mbar_init(tfull_bar(s), 1); mbar_init(tempty_bar(s), 1); }
    mbar_init(qfull_bar, 1);
    mbar_init(qempty_bar, 1);
    fence_mbar_init_cluster();
  }
  if (warp == 4 && lane == 0) { tma_prefetch_desc(&map_q); if (!kPacked) tma_prefetch_desc(&map_d); }
  if (warp == 5) { tmem_alloc<1>(tmem_slot, 512); tmem_relinquish<1>(); }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  const int units = a.B * a.slices;

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0, ucount = 0;
      for (int u = blockIdx.x; u < units; u += gridDim.x, ++ucount) {
        const int b = u / a.slices, sl = u % a.slices;
        const int c_lo = sl * a.per_slice, c_hi = min(a.C, c_lo + a.per_slice);
        // query tile: wait until the MMAs of the previous unit no longer read it
        mbar_wait(qempty_bar, (ucount & 1u) ^ 1u, a.status, 500);
        mbar_arrive_expect_tx(qfull_bar, kATileBytes);
        // the query tile is stacked `reps` times in the 128 rows so that every epilogue warp owns valid rows
        const int rows_per_rep = 128 / a.reps;
        for (int rp = 0; rp < a.reps; ++rp) {
          const uint32_t dst = a_smem + (uint32_t)(rp * rows_per_rep) * 128u;
          tma_load_2d(dst, &map_q, qfull_bar, 0, b * a.Tq, THR_L2_EVICT_LAST);
          tma_load_2d(dst + 128 * 64 * 2, &map_q, qfull_bar, 64, b * a.Tq, THR_L2_EVICT_LAST);
        }
        if constexpr (!kPacked) {   // packed: the decoder warps fill the candidate stages
          for (int c = c_lo; c < c_hi; ++c, ++it) {
            const int s = it % kStagesM;
            const uint32_t ph = (it / kStagesM) & 1u;
            int64_t doc = a.cand[(size_t)b * a.C + c];
            if (doc < 0 || doc >= a.n_docs) doc = 0;  // slot is skipped by the epilogue
            mbar_wait(empty_bar(s), ph ^ 1u, a.status, 501);
            mbar_arrive_expect_tx(full_bar(s), stage_bytes);
            const int32_t row = (int32_t)(doc * a.Td);
            tma_load_2d(b_smem(s), &map_d, full_bar(s), 0, row, THR_L2_EVICT_FIRST);
            tma_load_2d(b_smem(s) + half_bytes_b, &map_d, full_bar(s), 64, row, THR_L2_EVICT_FIRST);
          }
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_f32(128, (uint32_t)a.Td);
      uint32_t it = 0, ucount = 0;
      for (int u = blockIdx.x; u < units; u += gridDim.x, ++ucount) {
        const int sl = u % a.slices;
        const int c_lo = sl * a.per_slice, c_hi = min(a.C, c_lo + a.per_slice);
        mbar_wait(qfull_bar, ucount & 1u, a.status, 510);
        tc_fence_after_sync();
        for (int c = c_lo; c < c_hi; ++c, ++it) {
          const int s = it % kStagesM;
          const uint32_t ph = (it / kStagesM) & 1u;
          const int acc = it % kAccM;
          const uint32_t aph = (it / kAccM) & 1u;
          mbar_wait(tempty_bar(acc), aph ^ 1u, a.status, 511);
          mbar_wait(full_bar(s), ph, a.status, 512);
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 128);
#pragma unroll
          for (int k = 0; k < kD / 16; ++k) {
            const int half = k >> 2, kk = k & 3;
            const uint64_t adesc = umma_desc_sw128(a_smem + half * (128 * 64 * 2)) + (uint64_t)(kk * 2);
            const uint64_t bdesc = umma_desc_sw128(b_smem(s) + half * half_bytes_b) + (uint64_t)(kk * 2);
            umma_bf16<1>(d_tmem, adesc, bdesc, idesc, k != 0 ? 1u : 0u);
          }
          umma_commit_1cta(empty_bar(s));
          umma_commit_1cta(tfull_bar(acc));
        }
        umma_commit_1cta(qempty_bar);  // query tile reusable once this unit's MMAs are done
      }
    }
  } else if (warp >= 6) {
    // ===================== decoders (packed store only) =====================
    if constexpr (kPacked) {
      const int t = (int)threadIdx.x - kThreadsM;
      maxsim_decode_stages(a, t / kDecGroupThreads, t % kDecGroupThreads, b_smem(0), kMaxStageBytes, full_bar(0),
                           empty_bar(0), units);
    }
  } else {
    // ===================== epilogue: row max over doc tokens, sum over query tokens =====================
    // TMEM lane quarter w belongs to warp w.  With the query tile stacked `reps` times, replica r (rows
    // r*rows_per_rep ..) only scans doc-token columns [r*Td/reps, (r+1)*Td/reps): the four warps split the
    // columns instead of three of them idling; partial maxima meet in shared memory, warp 0 sums.
    const uint32_t lane_base = warp * 32;
    const int rows_per_rep = 128 / a.reps;
    const int my_row = (int)(lane_base + lane);
    const int rep = my_row / rows_per_rep;
    const int cols_per_rep = a.Td / a.reps;
    uint32_t it = 0;
    for (int u = blockIdx.x; u < units; u += gridDim.x) {
      const int b = u / a.slices, sl = u % a.slices;
      const int c_lo = sl * a.per_slice, c_hi = min(a.C, c_lo + a.per_slice);
      int ql = a.q_len ? a.q_len[b] : a.Tq;
      ql = max(0, min(ql, a.Tq));
      for (int c = c_lo; c < c_hi; ++c, ++it) {
        const int acc = it % kAccM;
        const uint32_t aph = (it / kAccM) & 1u;
        const int64_t doc = a.cand[(size_t)b * a.C + c];
        const bool doc_ok = doc >= 0 && doc < a.n_docs;
        int dl = a.Td;
        if (doc_ok && a.d_len) dl = max(0, min(a.d_len[doc], a.Td));
        mbar_wait(tfull_bar(acc), aph, a.status, 520);
        tc_fence_after_sync();
        float m = -CUDART_INF_F;
        const int col_lo = rep * cols_per_rep, col_hi = min(dl, col_lo + cols_per_rep);
        if (doc_ok && (int)(lane_base % rows_per_rep) < ql) {   // warp-uniform: some row of this warp is a live token
          for (int c0 = col_lo; c0 < col_hi; c0 += 32) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + (lane_base << 16) + (uint32_t)(acc * 128 + c0), r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < col_hi) m = fmaxf(m, __uint_as_float(r[j]));
          }
        }
        pmax[acc][my_row] = m;
        tc_fence_before_sync();
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (warp == 0) {
          float v = 0.f;
          for (int t = (int)lane; t < rows_per_rep; t += 32) {
            float mm = pmax[acc][t];
            for (int rp = 1; rp < a.reps; ++rp) mm = fmaxf(mm, pmax[acc][rp * rows_per_rep + t]);
            if (t < ql && dl > 0 && doc_ok) v += mm;
          }
#pragma unroll
          for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
          if (lane == 0) {
            a.out[(size_t)b * a.C + c] = doc_ok ? v : -CUDART_INF_F;
            mbar_arrive(tempty_bar(acc));  // every epilogue warp has passed the barrier above
          }
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 5) {
    __syncwarp();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

// Work split and launch shared by both entry points (the candidates of a query are cut into slices so that every SM
// has units).
template <bool kPacked>
int maxsim_launch(thr_handle* h, const CUtensorMap& map_q, const CUtensorMap& map_d, MaxSimArgs& a, int B, int C,
                  void* stream) {
  a.status = h->d_status;
  a.reps = a.Tq <= 32 ? 4 : (a.Tq <= 64 ? 2 : 1);
  int slices = (4 * h->num_sms + B - 1) / B;
  if (slices < 1) slices = 1;
  if (slices > C) slices = C;
  a.per_slice = (C + slices - 1) / slices;
  a.slices = (C + a.per_slice - 1) / a.per_slice;
  const int units = B * a.slices;
  constexpr int threads = kPacked ? kThreadsPacked : kThreadsM;
  THR_CUDA(h, cudaFuncSetAttribute(maxsim_kernel<kPacked>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemM));
  int grid = units < h->num_sms ? units : h->num_sms;
  const int tok = thr_prof_begin(h, THR_PROF_MAXSIM, (cudaStream_t)stream);
  maxsim_kernel<kPacked><<<grid, threads, kSmemM, (cudaStream_t)stream>>>(map_q, map_d, a);
  thr_prof_end(h, tok, (cudaStream_t)stream);
  THR_CHECK_LAUNCH(h, kPacked ? "maxsim_kernel<packed>" : "maxsim_kernel");
  return THR_OK;
}

}  // namespace

extern "C" {

int thr_maxsim(thr_handle* h, const void* Qtok, const int32_t* q_len, int B, int Tq, int d,
               const void* Dtok, const int32_t* d_len, int64_t n_docs, int Td, const int64_t* cand,
               int C, float* out, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && C >= 0, "thr_maxsim: negative sizes");
  if (B == 0 || C == 0) return THR_OK;
  THR_REQUIRE(h, Qtok && Dtok && cand && out, "thr_maxsim: NULL argument");
  if (d != kD) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim: d = %d, kernels are built for d = %d", d, kD);
  if (Td != 64 && Td != 128) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim: Td = %d must be 64 or 128", Td);
  if (Tq < 1 || Tq > 128) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim: Tq = %d must be in [1, 128]", Tq);
  THR_REQUIRE(h, n_docs >= 1 && n_docs * Td < ((int64_t)1 << 31), "thr_maxsim: token store too large for TMA row index");
  CUtensorMap map_q, map_d;
  const uint32_t q_box_rows = Tq <= 32 ? 32u : (Tq <= 64 ? 64u : 128u);   // one replica of the query tile per load
  int rc = thr_encode_tma_2d_bf16(h, &map_q, Qtok, (uint64_t)B * Tq, kD, q_box_rows, 64);
  if (rc != THR_OK) return rc;
  rc = thr_encode_tma_2d_bf16(h, &map_d, Dtok, (uint64_t)n_docs * Td, kD, (uint32_t)Td, 64);
  if (rc != THR_OK) return rc;
  MaxSimArgs a = {};
  a.B = B; a.Tq = Tq; a.Td = Td; a.C = C; a.n_docs = n_docs; a.q_len = q_len; a.d_len = d_len;
  a.cand = cand; a.out = out;
  return maxsim_launch<false>(h, map_q, map_d, a, B, C, stream);
}

int thr_maxsim_packed(thr_handle* h, const void* Qtok, const int32_t* q_len, int B, int Tq, int d,
                      const uint32_t* codes, const int32_t* cids, const void* centroids, int64_t n_centroids,
                      const float* weights, const int32_t* d_len, int64_t n_rows, int Td, const int64_t* cand,
                      int C, float* out, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && C >= 0, "thr_maxsim_packed: negative sizes");
  if (B == 0 || C == 0) return THR_OK;
  THR_REQUIRE(h, Qtok && codes && cids && centroids && weights && cand && out, "thr_maxsim_packed: NULL argument");
  if (d != kD) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim_packed: d = %d, kernels are built for d = %d", d, kD);
  if (Td != 64 && Td != 128) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim_packed: Td = %d must be 64 or 128", Td);
  if (Tq < 1 || Tq > 128) return thr_fail(h, THR_EUNSUPPORTED, "thr_maxsim_packed: Tq = %d must be in [1, 128]", Tq);
  THR_REQUIRE(h, n_rows >= 1 && n_centroids >= 1 && n_centroids <= ((int64_t)1 << 31),
              "thr_maxsim_packed: need n_rows >= 1 and 1 <= n_centroids <= 2^31");
  THR_REQUIRE(h, ((uintptr_t)centroids & 15) == 0 && ((uintptr_t)weights & 15) == 0 && ((uintptr_t)codes & 3) == 0 &&
                     ((uintptr_t)cids & 3) == 0,
              "thr_maxsim_packed: centroids and weights must be 16-byte aligned, codes and cids 4-byte aligned");
  CUtensorMap map_q, map_unused;
  memset(&map_unused, 0, sizeof(map_unused));
  const uint32_t q_box_rows = Tq <= 32 ? 32u : (Tq <= 64 ? 64u : 128u);
  int rc = thr_encode_tma_2d_bf16(h, &map_q, Qtok, (uint64_t)B * Tq, kD, q_box_rows, 64);
  if (rc != THR_OK) return rc;
  MaxSimArgs a = {};
  a.B = B; a.Tq = Tq; a.Td = Td; a.C = C; a.n_docs = n_rows; a.q_len = q_len; a.d_len = d_len;
  a.cand = cand; a.out = out;
  a.codes = codes; a.cids = cids; a.centroids = (const uint4*)centroids; a.weights = weights;
  a.n_centroids = n_centroids;
  return maxsim_launch<true>(h, map_q, map_unused, a, B, C, stream);
}

}  // extern "C"
