// dense_topk.cu — K1: exact dense top-k (semantic channel).
//
// Replaces RAG2Retriever._semantic_search -> rag2_semantic_search
//   (src/voice_agent/rag2/retrieval.py:294-314, database/migrations/20260114_rag2_schema.sql:377-410):
//   ORDER BY embedding <=> q LIMIT n on L2-normalised vectors == top-n by dot product.
//
// Two kernels:
//   dense_score_kernel   persistent, warp-specialised tcgen05 GEMM  S = Q . X^T  (bf16 -> fp32 in
//                        TMEM) whose epilogue never writes S: each TMEM lane (= one query) filters its
//                        256 fresh scores against a running per-query threshold and appends survivors
//                        to a small per-(cluster, query) candidate list; lists are compacted to the
//                        best K' = k + margin by a warp-cooperative radix descent when they fill up.
//   dense_finalize_kernel one CTA per query: radix-select the global best K' of the cluster lists,
//                        re-score them exactly (fp64 dot of the bf16 inputs), sort by
//                        (score desc, id asc), emit top-k and the exactness certificate gap.
// Both take the scored width D apart from the row pitch, so thr_dense_topk_prefix runs them over the leading d_scan
// columns of the same rows (the prefix funnel); dense_rescore_kernel re-scores a pool at full width with the
// finalize's own re-score, and dense_funnel_finish_kernel orders it.
//
// Layout per cluster step ("tile"): 128*kCtaGroup queries x 256 chunks x D.
//   kCtaGroup = 2 : CTA pair, tcgen05.mma.cta_group::2 M=256 N=256, each CTA loads 128 query rows and
//                   128 chunk rows per 64-wide k-block (32 KB / stage / CTA, 6 stages).
//   kCtaGroup = 1 : single CTA, M=128 N=256 (48 KB / stage, 4 stages) — fallback and bring-up path.
// Warp roles (192 threads): warps 0-3 epilogue (TMEM lane quarter = warp id), warp 4 TMA producer,
// warp 5 TMEM allocator + MMA issuer.
#include <math_constants.h>

#include "common.cuh"

namespace {

constexpr int kBlockM = 128;       // query rows per CTA
constexpr int kTileN = 256;        // chunks per tile (UMMA N)
constexpr int kBlockK = 64;        // bf16 elements per k-block = one 128-byte swizzle row
constexpr int kAccStages = 2;      // 2 x 256 TMEM columns
constexpr int kTmemCols = 512;
constexpr int kCap = 1024;         // candidate slots per (cluster, query); raw keys {~idx, score bits}
constexpr int kMaxSel = 256;       // largest K' = k + margin
constexpr int kScoreThreads = 192;
constexpr int kFinalThreads = 512;
constexpr int kMaxClusters = 160;    // finalize / seed select: clusters of one launch (<= SMs / cta_group), a multiple of 32
constexpr int kSeedTiles = 3;      // tiles per cluster in the seed pass (default for large shards)
constexpr int kSeedTilesMax = kCap / kTileN;   // 4 x 256 candidates fill a list exactly; the lists stay uncompacted

template <int G> struct ScoreCfg {
  // measured at 10M x 1536, B = 256: 4 stages 6.54 ms, 5 stages 6.17 ms, 7 stages 6.26 ms
  static constexpr int kStages = (G == 2) ? 7 : 4;
  static constexpr int kABytes = kBlockM * kBlockK * 2;                 // 16 KB
  static constexpr int kBBytes = (G == 2 ? 128 : 256) * kBlockK * 2;    // 16 / 32 KB
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTxBytes = kStageBytes * G;                      // per full barrier phase
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
};

struct ScoreArgs {
  int B;            // queries
  int64_t N;        // chunks
  int D;
  int ksel;         // K' = k + margin
  int n_clusters;
  int Bpad;         // row stride of cand/cnt
  uint64_t* cand;   // [n_clusters][Bpad][kCap]
  int32_t* cnt;     // [n_clusters][Bpad]
  const float* tau_init;  // [Bpad] nullable: per-query lower bound of the K'-th best score (seed pass)
  int seed_mode;          // seed pass: leave the lists uncompacted (<= kSeedTilesMax * kTileN entries each)
  const uint16_t* tags;   // [N] nullable: per-chunk tag (collection id) for filtered queries
  const int32_t* want;    // [B] nullable: tag a query's chunks must carry, < 0 = any
  const uint32_t* deleted;  // [ceil(N / 32)] nullable: bit i % 32 of word i / 32 set = row i is deleted
  thr_dev_status* status;
};

// Candidate lists hold RAW keys (fp32 score bits << 32 | ~chunk_index): the epilogue appends them with
// three predicated instructions per score; the order-preserving transform is applied when a list is
// read (here and in the finalize kernel).
__device__ __forceinline__ uint64_t raw_to_orderable(uint64_t raw) {
  return ((uint64_t)f32_orderable(__uint_as_float((uint32_t)(raw >> 32))) << 32) | (raw & 0xffffffffull);
}

// Warp-cooperative: keep the `ksel` largest of the n (<= kCap) distinct keys in row[0..n), in place.
// Returns the ksel-th largest key in ORDERABLE form (valid in every lane).  Requires n > ksel.
__device__ uint64_t warp_compact_topk(uint64_t* row, int n, int ksel, uint32_t lane) {
  constexpr int kPer = kCap / 32;
  uint32_t hi[kPer], lo[kPer];
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    int i = lane + 32 * j;
    uint64_t key = i < n ? row[i] : 0ull;   // raw: score bits << 32 | ~idx
    hi[j] = i < n ? f32_orderable(__uint_as_float((uint32_t)(key >> 32))) : 0u;
    lo[j] = (uint32_t)key;
  }
  // radix descent over the 64 key bits: T = largest value with count(keys >= T) >= ksel
  uint32_t t_hi = 0, t_lo = 0;
  bool exact = false;
  for (int bit = 31; bit >= 0 && !exact; --bit) {
    uint32_t c_hi = t_hi | (1u << bit);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) c += (hi[j] >= c_hi) ? 1 : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if (c >= ksel) t_hi = c_hi;
    exact = (c == ksel);
  }
  for (int bit = 31; bit >= 0 && !exact; --bit) {
    uint32_t c_lo = t_lo | (1u << bit);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) c += (hi[j] > t_hi || (hi[j] == t_hi && lo[j] >= c_lo)) ? 1 : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if (c >= ksel) t_lo = c_lo;
    exact = (c == ksel);
  }
  // compact survivors to the front (order is irrelevant) and find the smallest survivor
  __syncwarp();
  int base = 0;
  uint32_t m_hi = 0xffffffffu, m_lo = 0xffffffffu;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    bool keep = hi[j] > t_hi || (hi[j] == t_hi && lo[j] >= t_lo);
    keep = keep && (int)(lane + 32 * j) < n;
    unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      row[base + __popc(bal & ((1u << lane) - 1))] =
          ((uint64_t)__float_as_uint(f32_from_orderable(hi[j])) << 32) | lo[j];
      if (hi[j] < m_hi || (hi[j] == m_hi && lo[j] < m_lo)) { m_hi = hi[j]; m_lo = lo[j]; }
    }
    base += __popc(bal);
  }
  uint64_t mn = ((uint64_t)m_hi << 32) | m_lo;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    uint64_t o = __shfl_xor_sync(0xffffffffu, mn, s);
    mn = o < mn ? o : mn;
  }
  __syncwarp();
  return mn;
}

// kSeed: the seed pass (a.seed_mode): thresholds stay at -inf, lists stay uncompacted, and without a tag filter or a
// deletion bitmap every score of a tile is stored — with 32-byte stores, four entries a time (the generic append path stores 8 bytes per lane
// per instruction into 32 different rows: at one wavefront per row that path alone was ~2/3 of the seed pass).
template <int G, bool kSeed>
__global__ void __launch_bounds__(kScoreThreads, 1)
dense_score_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x,
                   const ScoreArgs a) {
  using Cfg = ScoreCfg<G>;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: SWIZZLE_128B atoms and UMMA descriptors with base_offset = 0
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + Cfg::kStages * Cfg::kStageBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + kAccStages + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::kStages + 2 * kAccStages);
  auto a_smem = [&](int s) { return smem_base + s * Cfg::kStageBytes; };
  auto b_smem = [&](int s) { return smem_base + s * Cfg::kStageBytes + Cfg::kABytes; };

  const uint32_t warp = threadIdx.x >> 5;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t rank = (G == 2) ? cluster_ctarank() : 0u;
  const int cluster_id = (G == 2) ? (blockIdx.x >> 1) : blockIdx.x;
  const bool leader = rank == 0;

  const int kblocks = a.D / kBlockK;
  const int64_t tiles_total = (a.N + kTileN - 1) / kTileN;
  const int64_t tile_lo = tiles_total * cluster_id / a.n_clusters;
  const int64_t tile_hi = tiles_total * (cluster_id + 1) / a.n_clusters;
  const int qrows = kBlockM * G;
  const int qblocks = (a.B + qrows - 1) / qrows;

  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), 4 * G);
    }
    fence_mbar_init_cluster();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_x);
  }
  if (warp == 5) {
    tmem_alloc<G>(tmem_slot, kTmemCols);
    tmem_relinquish<G>();
  }
  tc_fence_before_sync();
  __syncthreads();
  if (G == 2) cluster_sync_all();
  tc_fence_after_sync();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 4) {
    // ===================== TMA producer (one lane, both CTAs of a pair) =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int qb = 0; qb < qblocks; ++qb) {
        const int q_row = qb * qrows + (int)rank * kBlockM;
        for (int64_t t = tile_lo; t < tile_hi; ++t) {
          const int32_t x_row = (int32_t)(t * kTileN + (G == 2 ? (int64_t)rank * 128 : 0));
          for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, a.status, 100);
            const uint32_t fb = (G == 2) ? mapa_u32(full_bar(stage), 0) : full_bar(stage);
            if (leader) mbar_arrive_expect_tx(full_bar(stage), Cfg::kTxBytes);
            if (G == 2) {
              tma_load_2d_pair(a_smem(stage), &map_q, fb, kb * kBlockK, q_row, THR_L2_EVICT_LAST);
              tma_load_2d_pair(b_smem(stage), &map_x, fb, kb * kBlockK, x_row, THR_L2_EVICT_FIRST);
            } else {
              tma_load_2d(a_smem(stage), &map_q, fb, kb * kBlockK, q_row, THR_L2_EVICT_LAST);
              tma_load_2d(b_smem(stage), &map_x, fb, kb * kBlockK, x_row, THR_L2_EVICT_FIRST);
              tma_load_2d(b_smem(stage) + 128 * kBlockK * 2, &map_x, fb, kb * kBlockK, x_row + 128,
                          THR_L2_EVICT_FIRST);
            }
            if (++stage == (uint32_t)Cfg::kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer (leader CTA) =====================
    // The whole warp runs the loop converged (uniform branches, uniform registers); one elected
    // lane issues the tcgen05 instructions.  Descriptors are precomputed: stage s adds
    // s * (stage bytes >> 4) to the 14-bit start-address field, K-step k adds 2 (32 bytes).
    if (leader) {
      const bool issuer = elect_one();  // one lane issues; elect.sync lets the compiler emit plain uniform code
      constexpr uint32_t idesc = umma_idesc_bf16_f32(kBlockM * G, kTileN);
      constexpr uint32_t kStageDescStep = (uint32_t)Cfg::kStageBytes >> 4;
      const uint64_t adesc0 = umma_desc_sw128(a_smem(0));
      const uint64_t bdesc0 = umma_desc_sw128(b_smem(0));
      uint32_t stage = 0, phase = 0, tcount = 0;
      for (int qb = 0; qb < qblocks; ++qb) {
        for (int64_t t = tile_lo; t < tile_hi; ++t, ++tcount) {
          const uint32_t acc = tcount & 1u;
          const uint32_t aph = (tcount >> 1) & 1u;
          mbar_wait(tempty_bar(acc), aph ^ 1u, a.status, 200);
          tc_fence_after_sync();
          const uint32_t d_tmem = tmem_base + acc * (uint32_t)kTileN;
          for (int kb = 0; kb < kblocks; ++kb) {
            mbar_wait(full_bar(stage), phase, a.status, 201);
            tc_fence_after_sync();
            if (issuer) {
              const uint64_t adesc = adesc0 + (uint64_t)(stage * kStageDescStep);
              const uint64_t bdesc = bdesc0 + (uint64_t)(stage * kStageDescStep);
              // four K = 16 steps per 64-wide k-block: +2 in the descriptor's start-address field = 32 bytes
              umma_bf16<G>(d_tmem, adesc, bdesc, idesc, kb != 0 ? 1u : 0u);
              umma_bf16<G>(d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
              umma_bf16<G>(d_tmem, adesc + 4, bdesc + 4, idesc, 1u);
              umma_bf16<G>(d_tmem, adesc + 6, bdesc + 6, idesc, 1u);
              if (G == 2) umma_commit_pair_mcast(empty_bar(stage), 0x3);
              else umma_commit_1cta(empty_bar(stage));
            }
            __syncwarp();
            if (++stage == (uint32_t)Cfg::kStages) { stage = 0; phase ^= 1u; }
          }
          if (issuer) {
            if (G == 2) umma_commit_pair_mcast(tfull_bar(acc), 0x3);
            else umma_commit_1cta(tfull_bar(acc));
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ===================== epilogue: fused per-query top-K' filter =====================
    const uint32_t lane_base = warp * 32;  // TMEM lane quarter of this warp
    uint32_t tcount = 0;
    bool ok = true;
    for (int qb = 0; qb < qblocks && ok; ++qb) {
      const int row = qb * qrows + (int)rank * kBlockM + (int)lane_base + (int)lane;  // query index
      const bool row_valid = row < a.B;
      uint64_t* rowbuf = a.cand + ((size_t)cluster_id * a.Bpad + (row_valid ? row : 0)) * kCap;
      // padding rows of the query block never pass; a seeded threshold is a valid lower bound of the
      // global K'-th best score, so nothing that could reach the final top-k is filtered
      float tau = row_valid ? (a.tau_init ? a.tau_init[row] : -CUDART_INF_F) : CUDART_INF_F;
      // tag filter: a chunk outside the query's tag is never appended, so every threshold (seed pass included) is
      // learnt from eligible chunks only and the result is the exact top-k of the filtered corpus
      const int want = (row_valid && a.tags && a.want) ? a.want[row] : -1;
      // deleted rows are dropped at the same place: thresholds, seed bound included, come from live rows only (the
      // seed pass takes the filtered path below when a bitmap is set, so a deleted row never reaches its select)
      int cnt = 0;
      for (int64_t t = tile_lo; t < tile_hi && ok; ++t, ++tcount) {
        const int acc = tcount & 1;
        const uint32_t aph = (tcount >> 1) & 1u;
        // make room: a tile can add up to kTileN survivors per query
        unsigned need = __ballot_sync(0xffffffffu, row_valid && cnt > kCap - kTileN);
        while (need) {
          const int src = __ffs(need) - 1;
          need &= need - 1;
          const int n_src = __shfl_sync(0xffffffffu, cnt, src);
          uint64_t* buf_src = (uint64_t*)__shfl_sync(0xffffffffu, (unsigned long long)rowbuf, src);
          __syncwarp();
          const uint64_t kth = warp_compact_topk(buf_src, n_src, a.ksel, lane);
          if ((int)lane == src) { cnt = a.ksel; tau = key_score(kth); }
        }
        // warp-uniform outcome: the loop below uses full-mask warp collectives
        if (!__all_sync(0xffffffffu, mbar_wait(tfull_bar(acc), aph, a.status, 300))) { ok = false; break; }
        tc_fence_after_sync();
        const int64_t col0 = t * kTileN;
        const int ncols = (int)min((int64_t)kTileN, a.N - col0);
        uint64_t* wptr = rowbuf + cnt;
        if (kSeed && a.tags == nullptr && a.deleted == nullptr && ncols == kTileN) {
          // seed pass, full tile, no tag filter: all kTileN scores of the row, in column order
#pragma unroll 1
          for (int c = 0; c < kTileN / 32; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + (lane_base << 16) + (uint32_t)(acc * kTileN + c * 32), r);
            tmem_ld_wait();
            if (row_valid) {
              const uint32_t inv0 = ~(uint32_t)(col0 + c * 32);
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const uint64_t e0 = ((uint64_t)r[j] << 32) | (uint64_t)(inv0 - (uint32_t)j);
                const uint64_t e1 = ((uint64_t)r[j + 1] << 32) | (uint64_t)(inv0 - (uint32_t)(j + 1));
                const uint64_t e2 = ((uint64_t)r[j + 2] << 32) | (uint64_t)(inv0 - (uint32_t)(j + 2));
                const uint64_t e3 = ((uint64_t)r[j + 3] << 32) | (uint64_t)(inv0 - (uint32_t)(j + 3));
                asm volatile("st.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(wptr + j), "l"(e0), "l"(e1), "l"(e2),
                             "l"(e3) : "memory");
              }
              wptr += 32;
            }
          }
        } else if (ncols == kTileN) {
          // full tile
#pragma unroll 1
          for (int c = 0; c < kTileN / 32; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + (lane_base << 16) + (uint32_t)(acc * kTileN + c * 32), r);
            tmem_ld_wait();
            {  // all 32 lanes take part in the votes; lanes without a query row never pass (tau = +inf)
              const uint32_t inv0 = ~(uint32_t)(col0 + c * 32);  // ~(col0 + c*32 + j) == inv0 - j
// Four columns at a time: max + one compare + one warp vote; the (predicated) appends run only when
// some lane of the warp passes — after warm-up that is ~ 128*K'/seen of the groups.
#define P1(j, tg)                                                                                  \
  if (__uint_as_float(r[j]) > tau && (want < 0 || (int)(tg) == want) && !((dw >> (j)) & 1u))       \
    *wptr++ = ((uint64_t)r[j] << 32) | (uint64_t)(inv0 - (uint32_t)(j));
#define P(j)                                                                                       \
  {                                                                                                \
    const float m4 = fmaxf(fmaxf(__uint_as_float(r[j]), __uint_as_float(r[j + 1])),                \
                           fmaxf(__uint_as_float(r[j + 2]), __uint_as_float(r[j + 3])));           \
    if (__any_sync(0xffffffffu, m4 > tau)) {                                                       \
      asm volatile("" ::: "memory"); /* keep this a real (warp-uniform) branch */                  \
      ushort4 tg = make_ushort4(0, 0, 0, 0);                                                       \
      if (a.tags) tg = __ldg((const ushort4*)(a.tags + col0 + c * 32 + (j))); /* 8-byte aligned */ \
      const uint32_t dw = a.deleted ? __ldg(a.deleted + ((col0 >> 5) + c)) : 0u; /* the c block's word */ \
      P1(j, tg.x) P1(j + 1, tg.y) P1(j + 2, tg.z) P1(j + 3, tg.w)                                  \
    }                                                                                              \
  }
              P(0); P(4); P(8); P(12); P(16); P(20); P(24); P(28);
#undef P1
#undef P
            }
          }
        } else if (ncols < kTileN) {
          // last, partial tile of the corpus (zero-filled rows past N are skipped)
#pragma unroll 1
          for (int c = 0; c < kTileN / 32; ++c) {
            uint32_t r[32];
            tmem_ld_32x32(tmem_base + (lane_base << 16) + (uint32_t)(acc * kTileN + c * 32), r);
            tmem_ld_wait();
            if (row_valid) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int col = c * 32 + j;
                if (__uint_as_float(r[j]) > tau && col < ncols && (want < 0 || (int)a.tags[col0 + col] == want) &&
                    !(a.deleted && ((a.deleted[(col0 + col) >> 5] >> ((col0 + col) & 31)) & 1u)))
                  *wptr++ = ((uint64_t)r[j] << 32) | (uint64_t)(~(uint32_t)(col0 + col));
              }
            }
          }
        }
        cnt = (int)(wptr - rowbuf);
        if (cnt > kCap) {  // cannot happen given the pre-tile compaction; keep the invariant loud
          dev_report(a.status, THR_EOVERFLOW, 301, cnt);
          cnt = kCap;
        }
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) {
          if (G == 2) mbar_arrive_cluster(mapa_u32(tempty_bar(acc), 0));
          else mbar_arrive(tempty_bar(acc));
        }
      }
      // final compaction of this query block: every list ends with <= K' entries
      unsigned need = __ballot_sync(0xffffffffu, row_valid && cnt > a.ksel && !kSeed);
      while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int n_src = __shfl_sync(0xffffffffu, cnt, src);
        uint64_t* buf_src = (uint64_t*)__shfl_sync(0xffffffffu, (unsigned long long)rowbuf, src);
        __syncwarp();
        (void)warp_compact_topk(buf_src, n_src, a.ksel, lane);
        if ((int)lane == src) cnt = a.ksel;
      }
      if (row_valid) a.cnt[(size_t)cluster_id * a.Bpad + row] = ok ? cnt : 0;
    }
  }

  // ---- teardown: nobody may exit (or free TMEM) while the peer can still signal us ----
  tc_fence_before_sync();
  __syncthreads();
  if (G == 2) cluster_sync_all();
  if (warp == 5) {
    __syncwarp();
    tmem_dealloc<G>(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// Finalize: global select + exact re-score + sort.
// ------------------------------------------------------------------------------------------------
struct FinalArgs {
  const __nv_bfloat16* Q;
  const __nv_bfloat16* X;
  int B, D;         // D: the columns scored (the prefix width); ld: the row pitch of Q and X
  int64_t ld;
  int64_t N, id_base;
  int k, ksel, n_clusters, Bpad;
  const uint64_t* cand;
  const int32_t* cnt;
  int64_t* out_ids;
  double* out_scores;
  int32_t* out_count;
  float* out_gap;
};

// Order n <= kMaxSel (score, id) pairs by (score desc, id asc) without barriers: element e = tid / P is counted by P
// adjacent threads (P = kFinalThreads / the next power of two >= max(n, 32)), each over every P-th other element.  The
// pairs are distinct, so the ranks are a permutation.  Every thread of the CTA must call it; it returns the rank of
// element *e (valid in the thread with part == 0, and only when *e < n).
template <typename Id>
__device__ __forceinline__ int rank_by_score_id(const double* sc, const Id* id, int n, int* e, int* part) {
  const int tid = threadIdx.x;
  int n2 = 32;
  while (n2 < n) n2 <<= 1;
  const int P = kFinalThreads / n2;   // 2 .. 16 threads per element, adjacent lanes
  *e = tid / P;
  *part = tid - *e * P;
  int rank = 0;
  if (*e < n) {
    const double se = sc[*e];
    const Id ie = id[*e];
    for (int j = *part; j < n; j += P) {
      const double sj = sc[j];
      const Id ij = id[j];
      rank += (sj > se || (sj == se && ij < ie)) ? 1 : 0;
    }
  }
  for (int sh = 1; sh < P; sh <<= 1) rank += __shfl_xor_sync(0xffffffffu, rank, sh);
  return rank;
}

__global__ void __launch_bounds__(kFinalThreads, 2) dense_finalize_kernel(const FinalArgs a) {
  extern __shared__ uint8_t fsm[];
  // layout: keys [n_clusters*ksel] u64 | qrow [D] bf16
  uint64_t* keys = (uint64_t*)fsm;
  __nv_bfloat16* qrow = (__nv_bfloat16*)(keys + (size_t)a.n_clusters * a.ksel);
  __shared__ uint32_t hist[256];
  __shared__ int s_n[kMaxClusters], s_off[kMaxClusters];
  __shared__ uint64_t s_prefix;
  __shared__ unsigned long long s_minkey;
  __shared__ int s_want, s_m, s_nsel, s_done;
  __shared__ uint64_t sel_key[kMaxSel];
  __shared__ double sel_score[kMaxSel];
  __shared__ uint32_t sel_idx[kMaxSel];

  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_nsel = 0; s_minkey = ~0ull; }
  for (int i = tid; i < a.D; i += kFinalThreads) qrow[i] = a.Q[(size_t)q * a.ld + i];
  // 1. gather the per-cluster lists of this query: list lengths first (one load per cluster, all in flight), an
  //    exclusive scan over the clusters by the first warp, then one flat copy whose loads do not depend on each other
  for (int c = tid; c < kMaxClusters; c += kFinalThreads)
    s_n[c] = c < a.n_clusters ? min(a.cnt[(size_t)c * a.Bpad + q], a.ksel) : 0;
  __syncthreads();
  if (warp == 0) {
    constexpr int kPer = kMaxClusters / 32;
    int n[kPer], sum = 0;
#pragma unroll
    for (int i = 0; i < kPer; ++i) { n[i] = s_n[lane * kPer + i]; sum += n[i]; }
    int incl = sum;
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, s);
      if (lane >= s) incl += v;
    }
    int off = incl - sum;
#pragma unroll
    for (int i = 0; i < kPer; ++i) { s_off[lane * kPer + i] = off; off += n[i]; }
    if (lane == 31) s_m = incl;
  }
  __syncthreads();
  {
    const int total = a.n_clusters * a.ksel;
#pragma unroll 4
    for (int j = tid; j < total; j += kFinalThreads) {
      const int c = j / a.ksel, i = j - c * a.ksel;
      if (i < s_n[c]) keys[s_off[c] + i] = raw_to_orderable(a.cand[((size_t)c * a.Bpad + q) * kCap + i]);
    }
  }
  __syncthreads();
  const int m = s_m;
  const int nsel = min(m, a.ksel);

  // 2. K'-th largest key by MSD radix select (8 bits per pass); keys are distinct.  The walk stops as soon as the
  //    bin it descends into holds exactly the keys still wanted (normally after three or four passes): every key of
  //    that bin is selected, so the threshold is the bin's lower edge.
  uint64_t T = 0;
  if (m > a.ksel) {
    if (tid == 0) { s_prefix = 0; s_want = a.ksel; s_done = 0; }
    for (int pass = 0; pass < 8; ++pass) {
      const int shift = 56 - 8 * pass;
      if (tid < 256) hist[tid] = 0;
      __syncthreads();
      if (s_done) break;   // uniform: written before the barrier that ended the previous pass
      const uint64_t prefix = s_prefix;
      for (int i = tid; i < m; i += kFinalThreads) {
        const uint64_t key = keys[i];
        const bool match = pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8));
        if (match) atomicAdd(&hist[(uint32_t)(key >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (tid < 32) {
        const int want = s_want;
        int d, above;
        if (radix_find_digit(hist, want, tid, &d, &above)) {
          s_want = want - above;
          s_prefix = prefix | ((uint64_t)d << shift);
          if ((int)hist[d] == want - above) s_done = 1;
        }
      }
      __syncthreads();
    }
    T = s_prefix;
  }
  // 3. collect survivors; the smallest of them is the K'-th best key (the certificate's reference score).  Their
  //    rows are asked into L2 right away: the re-scoring below then waits on L2, not on HBM.
  for (int i = tid; i < m; i += kFinalThreads) {
    const uint64_t key = keys[i];
    if (key >= T) {
      int slot = atomicAdd(&s_nsel, 1);
      if (slot < kMaxSel) sel_key[slot] = key;
      atomicMin(&s_minkey, (unsigned long long)key);
    }
  }
  __syncthreads();
  {
    const int lines = (a.D * 2 + 127) / 128;
    for (int j = tid; j < nsel * lines; j += kFinalThreads) {
      const int r = j / lines, l = j - r * lines;
      const char* p = (const char*)(a.X + (size_t)key_index(sel_key[r]) * a.ld) + (size_t)l * 128;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    }
  }

  // 4. exact re-score: fp64 dot of the bf16 inputs, one warp per kInFlight survivors, fixed summation order
  constexpr int kWarpsF = kFinalThreads / 32;
  for (int i0 = warp * kInFlight; i0 < nsel; i0 += kWarpsF * kInFlight) {
    uint32_t idx[kInFlight];
    double acc[kInFlight];
#pragma unroll
    for (int u = 0; u < kInFlight; ++u) idx[u] = i0 + u < nsel ? key_index(sel_key[i0 + u]) : 0u;
    rescore_rows(a.X, a.ld, a.D, idx, qrow, lane, acc);
#pragma unroll
    for (int u = 0; u < kInFlight; ++u)
      if (lane == 0 && i0 + u < nsel) { sel_score[i0 + u] = acc[u]; sel_idx[i0 + u] = idx[u]; }
  }
  __syncthreads();

  // 5. order by (score desc, idx asc) without barriers; every survivor writes its own output row
  const int nout = min(nsel, a.k);
  int e, part;
  const int rank = rank_by_score_id(sel_score, sel_idx, nsel, &e, &part);
  if (e < nsel && part == 0 && rank < nout) {
    const double se = sel_score[e];
    const size_t o = (size_t)q * a.k + rank;
    a.out_ids[o] = a.id_base + (int64_t)sel_idx[e];
    a.out_scores[o] = se;
    if (rank == nout - 1 && a.out_gap) {
      // every chunk that was not re-scored has a tensor-core score <= the K'-th best key's
      a.out_gap[q] = m > a.ksel ? (float)(se - (double)key_score((uint64_t)s_minkey)) : CUDART_INF_F;
    }
  }

  // 6. padding, count
  if (tid == 0) {
    a.out_count[q] = nout;
    if (a.out_gap && nout == 0) a.out_gap[q] = CUDART_INF_F;
  }
  for (int i = nout + tid; i < a.k; i += kFinalThreads) {
    const size_t o = (size_t)q * a.k + i;
    a.out_ids[o] = -1;
    a.out_scores[o] = -CUDART_INF;
  }
}

// ------------------------------------------------------------------------------------------------
// Seed select: a lower bound of each query's corpus-wide K'-th best score from the (uncompacted) lists of
// the seed pass: tau = the K'-th best score of the sample, one ulp lower so that the filter's strict ">"
// keeps ties.  At least K' sample chunks score above tau, so the corpus-wide K'-th best does too.
//
// The lists are read ONCE (they are ~100 MB per batch and do not stay in L2): a strided subsample (the first
// few entries of every list) gives a rough cut r under which about 4 K' of the sample's scores are expected;
// the one pass over all entries keeps those >= r (a few hundred) in shared memory, and the K'-th best of the
// kept ones is exact.  When the cut turns out useless (fewer than K' kept: an unrepresentative subsample; or more
// than the buffer holds: massive ties) the kernel falls back to a two-level histogram over all entries (12 + 8
// bits, two more passes), whose bound is the lower edge of a 20-bit bin — looser, still a valid lower bound.
// ------------------------------------------------------------------------------------------------
constexpr int kSelThreads = 512;
constexpr int kSelBuf = 4096;   // subsample, then the kept scores (orderable u32)

// want-th largest (1-based, want <= n) of v[0..n) in shared memory, by the whole CTA: MSD radix select, 8 bits a pass.
__device__ uint32_t cta_kth_largest_u32(const uint32_t* v, int n, int want, uint32_t* hist, uint32_t* s_pref,
                                        int* s_want) {
  const int tid = threadIdx.x;
  if (tid == 0) { *s_pref = 0; *s_want = want; }
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    const uint32_t prefix = *s_pref;
    for (int i = tid; i < n; i += kSelThreads) {
      const uint32_t key = v[i];
      const bool match = ((uint64_t)key >> (shift + 8)) == ((uint64_t)prefix >> (shift + 8));
      if (match) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid < 32) {
      const int w = *s_want;
      int d, above;
      if (radix_find_digit(hist, w, tid, &d, &above)) {
        *s_want = w - above;
        *s_pref = prefix | ((uint32_t)d << shift);
      }
    }
    __syncthreads();
  }
  return *s_pref;
}

__global__ void __launch_bounds__(kSelThreads) dense_seed_select_kernel(const uint64_t* cand, const int32_t* cnt,
                                                                        int n_clusters, int Bpad, int ksel,
                                                                        float* tau_out) {
  __shared__ uint32_t buf[kSelBuf];
  __shared__ uint32_t hist[4096];
  __shared__ uint32_t part[256];
  __shared__ int s_n[kMaxClusters];
  __shared__ uint32_t s_pref, s_bin, s_above;
  __shared__ int s_want, s_total, s_nsub, s_keep;
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_total = 0; s_nsub = 0; s_keep = 0; }
  __syncthreads();
  const int per = kSelBuf / n_clusters;   // subsample: the first `per` entries of every list
  for (int c = tid; c < n_clusters; c += kSelThreads) {
    const int n = min(cnt[(size_t)c * Bpad + q], kCap);
    s_n[c] = n;
    atomicAdd(&s_total, n);
    atomicAdd(&s_nsub, min(n, per));
  }
  __syncthreads();
  const int total = s_total, nsub = s_nsub;
  float tau = -CUDART_INF_F;
  if (total >= ksel) {   // else: fewer than K' candidates in the whole sample, no bound
    // scores of list c, entry i (the high word of the raw 8-byte key)
    auto score_bits = [&](int c, int i) -> uint32_t {
      return f32_orderable(__uint_as_float((uint32_t)(cand[((size_t)c * Bpad + q) * kCap + i] >> 32)));
    };
    // 1. the rough cut: the R-th best of the subsample, R such that ~4 K' of all entries are expected above it
    uint32_t r = 0;
    if (total > kSelBuf / 2) {
      for (int j = tid; j < n_clusters * per; j += kSelThreads) {
        const int c = j / per, i = j - c * per;
        buf[j] = i < s_n[c] ? score_bits(c, i) : 0u;   // holes: the smallest key
      }
      __syncthreads();
      long long R = (4ll * ksel * nsub + total - 1) / total;
      if (R < 1) R = 1;
      if (R > nsub) R = nsub;
      r = cta_kth_largest_u32(buf, n_clusters * per, (int)R, hist, &s_pref, &s_want);
      __syncthreads();
    }
    // 2. one pass over every entry: keep the scores >= r.  A warp per list, eight loads per lane in flight.
    for (int c = warp; c < n_clusters; c += kSelThreads / 32) {
      const int n = s_n[c];
      for (int i0 = lane; i0 < n; i0 += 256) {
        uint32_t o[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) o[u] = i0 + 32 * u < n ? score_bits(c, i0 + 32 * u) : 0u;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (i0 + 32 * u < n && o[u] >= r) {
            const int slot = atomicAdd(&s_keep, 1);
            if (slot < kSelBuf) buf[slot] = o[u];
          }
        }
      }
    }
    __syncthreads();
    const int kept = s_keep;
    if (kept >= ksel && kept <= kSelBuf) {
      // 3. exact: the K'-th best of the kept scores is the K'-th best of the sample
      const uint32_t v = cta_kth_largest_u32(buf, kept, ksel, hist, &s_pref, &s_want);
      tau = f32_from_orderable(v > 0 ? v - 1u : 0u);
    } else {
      // fallback: two-level histogram over all entries
      uint32_t prefix = 0, above = 0;
      bool enough = true;
      for (int level = 0; level < 2 && enough; ++level) {
        const int nb = level == 0 ? 4096 : 256;
        for (int i = tid; i < nb; i += kSelThreads) hist[i] = 0;
        __syncthreads();
        for (int c = warp; c < n_clusters; c += kSelThreads / 32) {
          const int n = s_n[c];
          for (int i = lane; i < n; i += 32) {
            const uint32_t o = score_bits(c, i);
            if (level == 0) atomicAdd(&hist[o >> 20], 1u);
            else if ((o >> 20) == prefix) atomicAdd(&hist[(o >> 12) & 255u], 1u);
          }
        }
        __syncthreads();
        // suffix sums: thread t < 256 owns bins [t*per_t, (t+1)*per_t); find the bin where the count from the top
        // reaches ksel
        const int per_t = nb / 256;
        if (tid < 256) {
          uint32_t mine = 0;
          for (int j = 0; j < per_t; ++j) mine += hist[tid * per_t + j];
          part[tid] = mine;
        }
        __syncthreads();
        if (tid == 0) {
          uint32_t cum = above;
          int t = 255;
          for (; t >= 0; --t) {
            if (cum + part[t] >= (uint32_t)ksel) break;
            cum += part[t];
          }
          if (t < 0) { s_bin = 0xffffffffu; s_above = cum; }
          else {
            int b = t * per_t + per_t - 1;
            for (; b > t * per_t; --b) {
              if (cum + hist[b] >= (uint32_t)ksel) break;
              cum += hist[b];
            }
            s_bin = (uint32_t)b;
            s_above = cum;
          }
        }
        __syncthreads();
        if (s_bin == 0xffffffffu) enough = false;
        else if (level == 0) prefix = s_bin;
        else prefix = (prefix << 8) | s_bin;
        above = s_above;
        __syncthreads();
      }
      if (enough) {
        const uint32_t edge = prefix << 12;  // 20 significant bits of the orderable score
        tau = f32_from_orderable(edge > 0 ? edge - 1u : 0u);
      }
    }
  }
  if (tid == 0) tau_out[q] = tau;
}

// ------------------------------------------------------------------------------------------------
// Prefix funnel: full-width re-score of a candidate pool, and the final order over the shards' scores.
// ------------------------------------------------------------------------------------------------
struct RescoreArgs {
  const __nv_bfloat16* Q;   // [B, D]
  const __nv_bfloat16* X;   // [N, D]
  int D, P;
  int64_t N, id_base;
  const int64_t* ids;       // [B, P] global ids, -1 padded
  const int32_t* count;     // [B]
  double* out;              // [B, P]
};
constexpr int kRescoreRows = kFinalThreads / 32 * kInFlight;   // pool entries per CTA

// grid (B, ceil(P / kRescoreRows)): a CTA re-scores kRescoreRows entries of one query's pool, kInFlight per warp
__global__ void __launch_bounds__(kFinalThreads) dense_rescore_kernel(const RescoreArgs a) {
  extern __shared__ uint8_t rsm[];
  __nv_bfloat16* qrow = (__nv_bfloat16*)rsm;
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < a.D; i += kFinalThreads) qrow[i] = a.Q[(size_t)q * a.D + i];
  __syncthreads();
  const int n = min(max(a.count[q], 0), a.P);
  const int i0 = blockIdx.y * kRescoreRows + warp * kInFlight;
  if (i0 >= a.P) return;   // warp-uniform
  uint32_t idx[kInFlight];
  bool mine[kInFlight], any = false;
#pragma unroll
  for (int u = 0; u < kInFlight; ++u) {
    const int64_t id = i0 + u < n ? a.ids[(size_t)q * a.P + i0 + u] : -1;
    mine[u] = id >= a.id_base && id < a.id_base + a.N;   // a row of this handle (padding never is)
    idx[u] = mine[u] ? (uint32_t)(id - a.id_base) : 0u;
    any |= mine[u];
  }
  double acc[kInFlight] = {};
  if (any) rescore_rows(a.X, a.D, a.D, idx, qrow, lane, acc);
  if (lane == 0) {
#pragma unroll
    for (int u = 0; u < kInFlight; ++u)
      if (i0 + u < a.P) a.out[(size_t)q * a.P + i0 + u] = mine[u] ? acc[u] : -CUDART_INF;
  }
}

struct FunnelFinishArgs {
  int P, k, S;
  const int64_t* ids;            // [B, P]
  const int32_t* count;          // [B]
  const double* const* scores;   // [S] -> [B, P]
  int64_t* out_ids;
  double* out_scores;
  int32_t* out_count;
};

// one CTA per query: the element-wise max over the S score arrays, then the first min(k, count) by (score desc, id asc)
__global__ void __launch_bounds__(kFinalThreads) dense_funnel_finish_kernel(const FunnelFinishArgs a) {
  __shared__ double s_sc[kMaxSel];
  __shared__ int64_t s_id[kMaxSel];
  const int q = blockIdx.x, tid = threadIdx.x;
  const int n = min(max(a.count[q], 0), a.P);
  for (int j = tid; j < n; j += kFinalThreads) {
    const size_t o = (size_t)q * a.P + j;
    double v = -CUDART_INF;
    for (int s = 0; s < a.S; ++s) v = fmax(v, a.scores[s][o]);
    s_sc[j] = v;
    s_id[j] = a.ids[o];
  }
  __syncthreads();
  const int nout = min(n, a.k);
  int e, part;
  const int rank = rank_by_score_id(s_sc, s_id, n, &e, &part);
  if (e < n && part == 0 && rank < nout) {
    const size_t o = (size_t)q * a.k + rank;
    a.out_ids[o] = s_id[e];
    a.out_scores[o] = s_sc[e];
  }
  if (tid == 0) a.out_count[q] = nout;
  for (int i = nout + tid; i < a.k; i += kFinalThreads) {
    const size_t o = (size_t)q * a.k + i;
    a.out_ids[o] = -1;
    a.out_scores[o] = -CUDART_INF;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------
struct thr_dense_state {
  const void* X;
  int64_t N;
  int D;
  int64_t id_base;
  CUtensorMap map_x;   // the leading map_d columns of X (row pitch D): D when the index is set, then the last d_scan
  int map_d;
  int cta_group;  // 2 (pair) or 1; THR_DENSE_CTA_GROUP overrides for bring-up
  const uint16_t* tags;  // [N] device, nullable
  const uint32_t* deleted;  // [ceil(N / 32)] device, nullable
  // tuning knobs, read from the environment ONCE, when the index is set (THR_DENSE_SEED_TILES, THR_DENSE_NO_SEED)
  int seed_tiles;  // 0: the default for the shard size
  int no_seed;
};

void thr_dense_state_free(thr_handle* h) {
  if (h->dense) { free(h->dense); h->dense = nullptr; }
}

int thr_dense_view_get(thr_handle* h, thr_dense_view* v) {
  const thr_dense_state* st = h->dense;
  if (!st) return thr_fail(h, THR_ENOINDEX, "call thr_dense_index_set first");
  v->X = st->X; v->N = st->N; v->id_base = st->id_base; v->D = st->D; v->tags = st->tags; v->deleted = st->deleted;
  return THR_OK;
}

template <int G>
static int launch_score(thr_handle* h, const CUtensorMap& mq, const CUtensorMap& mx, const ScoreArgs& a,
                        cudaStream_t stream, int prof_slot = THR_PROF_DENSE_SCORE) {
  using Cfg = ScoreCfg<G>;
  auto kernel = a.seed_mode ? dense_score_kernel<G, true> : dense_score_kernel<G, false>;
  THR_CUDA(h, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(a.n_clusters * G);
  cfg.blockDim = dim3(kScoreThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = G;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const int tok = thr_prof_begin(h, prof_slot, stream);
  THR_CUDA(h, cudaLaunchKernelEx(&cfg, kernel, mq, mx, a));
  thr_prof_end(h, tok, stream);
  h->launches++;
  return THR_OK;
}

extern "C" {

int thr_dense_index_set(thr_handle* h, const void* X, int64_t N, int D, int64_t id_base) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, X != nullptr && N >= 1, "thr_dense_index_set: empty index");
  THR_REQUIRE(h, N < (int64_t)1 << 31, "thr_dense_index_set: N = %lld exceeds 2^31 rows per shard", (long long)N);
  if (D % kBlockK != 0 || D < kBlockK || D > 8192)
    return thr_fail(h, THR_EUNSUPPORTED, "thr_dense_index_set: D = %d must be a multiple of 64 in [64, 8192]", D);
  thr_dense_state_free(h);
  thr_dense_state* st = (thr_dense_state*)calloc(1, sizeof(thr_dense_state));
  if (!st) return thr_fail(h, THR_ENOMEM, "out of host memory");
  st->X = X; st->N = N; st->D = D; st->id_base = id_base;
  int rc = thr_encode_tma_2d_bf16(h, &st->map_x, X, (uint64_t)N, (uint64_t)D, 128, kBlockK);
  if (rc != THR_OK) { free(st); return rc; }
  st->map_d = D;
  st->cta_group = 2;
  const char* env = getenv("THR_DENSE_CTA_GROUP");
  if (env && env[0] == '1') st->cta_group = 1;
  env = getenv("THR_DENSE_SEED_TILES");
  st->seed_tiles = env ? atoi(env) : 0;
  if (st->seed_tiles > kSeedTilesMax) st->seed_tiles = kSeedTilesMax;
  env = getenv("THR_DENSE_NO_SEED");
  st->no_seed = env && env[0] == '1';
  h->dense = st;
  return THR_OK;
}

int thr_dense_tags_set(thr_handle* h, const uint16_t* tags) {
  if (!h) return THR_EINVAL;
  if (!h->dense) return thr_fail(h, THR_ENOINDEX, "thr_dense_tags_set: call thr_dense_index_set first");
  THR_REQUIRE(h, ((uintptr_t)tags & 7u) == 0, "thr_dense_tags_set: tags must be 8-byte aligned");
  h->dense->tags = tags;
  return THR_OK;
}

int thr_dense_deleted_set(thr_handle* h, const uint32_t* bits) {
  if (!h) return THR_EINVAL;
  if (!h->dense) return thr_fail(h, THR_ENOINDEX, "thr_dense_deleted_set: call thr_dense_index_set first");
  THR_REQUIRE(h, ((uintptr_t)bits & 15u) == 0, "thr_dense_deleted_set: bits must be 16-byte aligned");
  h->dense->deleted = bits;
  return THR_OK;
}

int thr_dense_topk(thr_handle* h, const void* Q, int B, int k, int margin, int64_t* out_ids,
                   double* out_scores, int32_t* out_count, float* out_gap, void* stream) {
  return thr_dense_topk_tagged(h, Q, B, k, margin, nullptr, out_ids, out_scores, out_count, out_gap, stream);
}

int thr_dense_topk_tagged(thr_handle* h, const void* Q, int B, int k, int margin, const int32_t* want,
                          int64_t* out_ids, double* out_scores, int32_t* out_count, float* out_gap,
                          void* stream) {
  if (!h) return THR_EINVAL;
  if (!h->dense) return thr_fail(h, THR_ENOINDEX, "thr_dense_topk: call thr_dense_index_set first");
  return thr_dense_topk_prefix(h, Q, B, k, margin, want, h->dense->D, out_ids, out_scores, out_count, out_gap,
                               stream);
}

int thr_dense_topk_prefix(thr_handle* h, const void* Q, int B, int k, int margin, const int32_t* want, int d_scan,
                          int64_t* out_ids, double* out_scores, int32_t* out_count, float* out_gap, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  thr_dense_state* st = h->dense;
  if (!st) return thr_fail(h, THR_ENOINDEX, "thr_dense_topk: call thr_dense_index_set first");
  THR_REQUIRE(h, want == nullptr || st->tags != nullptr, "thr_dense_topk_tagged: call thr_dense_tags_set first");
  THR_REQUIRE(h, B >= 0 && k >= 1 && margin >= 0, "thr_dense_topk: bad B/k/margin");
  THR_REQUIRE(h, d_scan % kBlockK == 0 && d_scan >= kBlockK && d_scan <= st->D,
              "thr_dense_topk_prefix: d_scan = %d must be a multiple of 64 in [64, D = %d]", d_scan, st->D);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, k + margin <= kMaxSel, "thr_dense_topk: k + margin = %d exceeds %d", k + margin, kMaxSel);
  THR_REQUIRE(h, Q && out_ids && out_scores && out_count, "thr_dense_topk: NULL argument");
  cudaStream_t s = (cudaStream_t)stream;
  int rc;
  if (st->map_d != d_scan) {   // the same rows, fewer columns: the map's width changes, its row pitch stays D
    st->map_d = 0;
    rc = thr_encode_tma_2d_bf16(h, &st->map_x, st->X, (uint64_t)st->N, (uint64_t)d_scan, 128, kBlockK,
                                (uint64_t)st->D);
    if (rc != THR_OK) return rc;
    st->map_d = d_scan;
  }
  // up to 128 queries fit one CTA's M = 128 tile: the single-CTA kernel then does half the MMA work per
  // chunk tile and the scan is HBM-bound (batch-1 latency); larger batches use the CTA pair (M = 256)
  // (only while the finalize kernel's shared memory — one K' list per CTA — still fits)
  const bool small_ok = (size_t)h->num_sms * (k + margin) * 8 + (size_t)d_scan * 2 <= 200 * 1024;
  const int G = (B <= kBlockM && small_ok) ? 1 : st->cta_group;
  const int64_t tiles = (st->N + kTileN - 1) / kTileN;
  int n_clusters = h->num_sms / G;
  if ((int64_t)n_clusters > tiles) n_clusters = (int)tiles;
  THR_REQUIRE(h, n_clusters <= kMaxClusters, "thr_dense_topk: %d clusters exceed %d", n_clusters, kMaxClusters);
  const int Bpad = (B + 255) & ~255;
  const size_t cand_bytes = (size_t)n_clusters * Bpad * kCap * sizeof(uint64_t);
  const size_t cnt_bytes = (size_t)n_clusters * Bpad * sizeof(int32_t);
  uint8_t* ws = (uint8_t*)thr_scratch(h, 0, cand_bytes + cnt_bytes + (size_t)Bpad * sizeof(float));
  if (!ws) return THR_ENOMEM;

  CUtensorMap map_q;
  rc = thr_encode_tma_2d_bf16(h, &map_q, Q, (uint64_t)B, (uint64_t)d_scan, 128, kBlockK, (uint64_t)st->D);
  if (rc != THR_OK) return rc;

  ScoreArgs a;
  a.B = B; a.N = st->N; a.D = d_scan; a.ksel = k + margin; a.n_clusters = n_clusters; a.Bpad = Bpad;
  a.cand = (uint64_t*)ws; a.cnt = (int32_t*)(ws + cand_bytes); a.status = h->d_status;
  a.tau_init = nullptr;
  a.seed_mode = 0;
  a.tags = want ? st->tags : nullptr;
  a.want = want;
  a.deleted = st->deleted;
  float* tau_seed = (float*)(ws + cand_bytes + cnt_bytes);

  FinalArgs f;
  f.Q = (const __nv_bfloat16*)Q; f.X = (const __nv_bfloat16*)st->X; f.B = B; f.D = d_scan; f.ld = st->D; f.N = st->N;
  f.id_base = st->id_base; f.k = k; f.ksel = k + margin; f.n_clusters = n_clusters; f.Bpad = Bpad;
  f.cand = a.cand; f.cnt = a.cnt; f.out_ids = out_ids; f.out_scores = out_scores;
  f.out_count = out_count; f.out_gap = out_gap;
  const size_t fsmem = (size_t)n_clusters * f.ksel * sizeof(uint64_t) + (size_t)d_scan * 2;
  THR_CUDA(h, cudaFuncSetAttribute(dense_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));

  // Seed pass: score a small prefix of the corpus first and start the full pass from its K'-th best
  // score.  Every cluster then filters with a threshold learnt from ~130k chunks from its first tile on
  // (instead of from -inf), which cuts the epilogue's append work and list compactions several-fold.
  // tiles per cluster in the seed pass (<= kSeedTilesMax: the uncompacted lists must fit): a longer prefix gives a
  // tighter threshold but costs its own scoring and a select over n_clusters * tiles * 256 scores per query
  const int seed_tiles_env = st->seed_tiles;   // THR_DENSE_SEED_TILES, read when the index was set
  // measured at D = 1536, B = 256 (score + seed, ms): 1.25M rows 0.897 / 0.854 / 0.915 for 1 / 2 / 3 tiles,
  // 2.5M rows 1.84 / 1.76 / 1.73
  const int seed_tiles = seed_tiles_env > 0 ? seed_tiles_env : (st->N >= 2000000 ? kSeedTiles : 2);
  const int64_t seed_rows = (int64_t)n_clusters * seed_tiles * kTileN;
  if (st->N >= 16 * seed_rows && !st->no_seed) {
    ScoreArgs sa = a;
    sa.N = seed_rows;
    sa.seed_mode = 1;
    rc = (G == 2) ? launch_score<2>(h, map_q, st->map_x, sa, s, THR_PROF_DENSE_SEED)
                  : launch_score<1>(h, map_q, st->map_x, sa, s, THR_PROF_DENSE_SEED);
    if (rc != THR_OK) return rc;
    const int tok0 = thr_prof_begin(h, THR_PROF_DENSE_SEED, s);
    dense_seed_select_kernel<<<B, kSelThreads, 0, s>>>(a.cand, a.cnt, n_clusters, Bpad, k + margin, tau_seed);
    thr_prof_end(h, tok0, s);
    THR_CHECK_LAUNCH(h, "dense_seed_select_kernel");
    a.tau_init = tau_seed;
  }
  // (no clearing of a.cnt between the passes: every cluster writes the count of every valid query row on its way out)
  rc = (G == 2) ? launch_score<2>(h, map_q, st->map_x, a, s) : launch_score<1>(h, map_q, st->map_x, a, s);
  if (rc != THR_OK) return rc;

  const int tok = thr_prof_begin(h, THR_PROF_DENSE_FINALIZE, s);
  dense_finalize_kernel<<<B, kFinalThreads, fsmem, s>>>(f);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "dense_finalize_kernel");
  return THR_OK;
}

int thr_dense_rescore(thr_handle* h, const void* Q, int B, const int64_t* ids, const int32_t* count, int P,
                      double* out, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  thr_dense_state* st = h->dense;
  if (!st) return thr_fail(h, THR_ENOINDEX, "thr_dense_rescore: call thr_dense_index_set first");
  THR_REQUIRE(h, B >= 0 && P >= 1, "thr_dense_rescore: bad B/P");
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, Q && ids && count && out, "thr_dense_rescore: NULL argument");
  RescoreArgs a;
  a.Q = (const __nv_bfloat16*)Q; a.X = (const __nv_bfloat16*)st->X; a.D = st->D; a.P = P; a.N = st->N;
  a.id_base = st->id_base; a.ids = ids; a.count = count; a.out = out;
  const size_t smem = (size_t)st->D * 2;
  cudaStream_t s = (cudaStream_t)stream;
  const int tok = thr_prof_begin(h, THR_PROF_DENSE_FINALIZE, s);
  dense_rescore_kernel<<<dim3(B, (P + kRescoreRows - 1) / kRescoreRows), kFinalThreads, smem, s>>>(a);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "dense_rescore_kernel");
  return THR_OK;
}

int thr_dense_funnel_finish(thr_handle* h, int B, int P, int k, const int64_t* ids, const int32_t* count,
                            const double* const* scores, int S, int64_t* out_ids, double* out_scores,
                            int32_t* out_count, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, B >= 0 && k >= 1 && k <= P && P <= kMaxSel && S >= 1 && S <= 64,
              "thr_dense_funnel_finish: need 1 <= k <= P <= %d and 1 <= S <= 64 (k = %d, P = %d, S = %d)", kMaxSel, k,
              P, S);
  if (B == 0) return THR_OK;
  THR_REQUIRE(h, ids && count && scores && out_ids && out_scores && out_count, "thr_dense_funnel_finish: NULL argument");
  FunnelFinishArgs a;
  a.P = P; a.k = k; a.S = S; a.ids = ids; a.count = count; a.scores = scores;
  a.out_ids = out_ids; a.out_scores = out_scores; a.out_count = out_count;
  cudaStream_t s = (cudaStream_t)stream;
  const int tok = thr_prof_begin(h, THR_PROF_DENSE_FINALIZE, s);
  dense_funnel_finish_kernel<<<B, kFinalThreads, 0, s>>>(a);
  thr_prof_end(h, tok, s);
  THR_CHECK_LAUNCH(h, "dense_funnel_finish_kernel");
  return THR_OK;
}

}  // extern "C"
