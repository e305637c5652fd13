// common.cuh — handle, error plumbing and the sm_100a PTX wrappers shared by the kernels.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/thr.h"

// ------------------------------------------------------------------------------------
// Handle
// ------------------------------------------------------------------------------------

struct thr_dense_state;
struct thr_bm25_state;

// Device-visible status word: kernels record failures here, thr_sync() reads it back.
struct thr_dev_status {
  int code;      // 0 or a THR_E* value (first failure wins)
  int where;     // kernel-specific location tag
  long long aux; // kernel-specific detail
};

struct thr_handle {
  int device;
  int num_sms;
  char err[512];
  int64_t launches;
  thr_dev_status* d_status;  // device alias of h_status
  thr_dev_status* h_status;  // pinned, mapped host memory: still readable after a trapped kernel
  thr_dense_state* dense;
  thr_bm25_state* bm25;
  void* scratch[2];          // device scratch, grown on demand: one arena per channel (0 dense, 1 BM25), so that the two
  size_t scratch_bytes[2];   // channels of one batch may run on different streams at the same time
  // per-kernel timing (thr_prof_*): ring of event pairs
  int prof_on;
  unsigned prof_mask;        // slots that are timed (thr_prof_select; all by default)
  int prof_n;
  cudaEvent_t* prof_ev;      // [2 * kProfMax]
  unsigned char* prof_slot;  // [kProfMax]
};
constexpr int kProfMax = 8192;
// Bracket a launch with events when profiling is on (no-ops otherwise).
int thr_prof_begin(thr_handle* h, int slot, cudaStream_t s);
void thr_prof_end(thr_handle* h, int token, cudaStream_t s);

int thr_fail(thr_handle* h, int code, const char* fmt, ...);
// Grow-only device scratch owned by the handle (arena 0: dense, 1: BM25). Returns NULL (and sets err) on failure.
void* thr_scratch(thr_handle* h, int arena, size_t bytes);
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda needed).  ld: row pitch in elements
// (0: cols), so that a map can cover the leading `cols` columns of a wider row-major matrix.
int thr_encode_tma_2d_bf16(thr_handle* h, CUtensorMap* map, const void* base, uint64_t rows,
                           uint64_t cols, uint32_t box_rows, uint32_t box_cols, uint64_t ld = 0);

// What a handle's indexes hold, for kernels outside the file that owns the index state (scope.cu).
// THR_ENOINDEX (with the message set) when the index is not set.
struct thr_dense_view {
  const void* X;              // bf16 [N, D]
  int64_t N, id_base;
  int D;
  const uint16_t* tags;       // nullable
  const uint32_t* deleted;    // nullable
};
struct thr_bm25_view {
  const int64_t* skip;        // [V * n_blk + 1]
  const void* post;           // {u32 doc, f32 impact} records
  const float* idf;
  int64_t n_docs, id_base;
  int n_blk, blk_shift, V;
  const uint16_t* tags;       // nullable
  const uint32_t* deleted;    // nullable
};
int thr_dense_view_get(thr_handle* h, thr_dense_view* v);
int thr_bm25_view_get(thr_handle* h, thr_bm25_view* v);

#define THR_CUDA(h, expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess)                                                             \
      return thr_fail((h), THR_ECUDA, "%s failed: %s (%s:%d)", #expr,                  \
                      cudaGetErrorString(_e), __FILE__, __LINE__);                     \
  } while (0)

#define THR_CHECK_LAUNCH(h, name)                                                      \
  do {                                                                                 \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess)                                                             \
      return thr_fail((h), THR_ECUDA, "launch of %s failed: %s", (name),               \
                      cudaGetErrorString(_e));                                         \
    (h)->launches++;                                                                   \
  } while (0)

#define THR_REQUIRE(h, cond, ...)                                                      \
  do {                                                                                 \
    if (!(cond)) return thr_fail((h), THR_EINVAL, __VA_ARGS__);                        \
  } while (0)

// ------------------------------------------------------------------------------------
// Device helpers
// ------------------------------------------------------------------------------------

// The status word is zero-copy host memory (no PCIe atomics assumed): first writer wins, benignly racy.
__device__ __forceinline__ void dev_report(thr_dev_status* st, int code, int where, long long aux) {
  volatile thr_dev_status* v = st;
  if (v->code == 0) {
    v->where = where;
    v->aux = aux;
    __threadfence_system();
    v->code = code;
    __threadfence_system();
  }
}

// Monotone map float -> uint32 so that unsigned order == float order (NaN-free inputs).
__device__ __forceinline__ uint32_t f32_orderable(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_from_orderable(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
// (score desc, index asc) as one descending u64 key.
__device__ __forceinline__ uint64_t pack_key(float score, uint32_t idx) {
  return ((uint64_t)f32_orderable(score) << 32) | (uint64_t)(0xffffffffu - idx);
}
__device__ __forceinline__ float key_score(uint64_t key) { return f32_from_orderable((uint32_t)(key >> 32)); }
__device__ __forceinline__ uint32_t key_index(uint64_t key) { return 0xffffffffu - (uint32_t)key; }

// One step of an MSD radix select over a 256-bin histogram in shared memory, by the first warp of the CTA
// (tid < 32, all 32 lanes): finds the digit d whose bin holds the want-th largest key, counting from bin 255 down
// (8 bins per lane + a warp scan instead of one thread walking up to 255 dependent shared-memory loads).
// Returns true in the one lane that found it, with d and the number of keys in the bins above d.
__device__ __forceinline__ bool radix_find_digit(const uint32_t* hist, int want, int lane, int* d_out, int* above_out) {
  int h[8], sum = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { h[i] = (int)hist[255 - 8 * lane - i]; sum += h[i]; }
  int incl = sum;
#pragma unroll
  for (int s = 1; s < 32; s <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, s);
    if (lane >= s) incl += v;
  }
  int cum = incl - sum;
  // the lane whose bins contain the want-th key; if the bins hold fewer than `want` keys in total, lane 31 ends
  // at digit 0 like the serial walk would
  const bool mine = cum < want && (want <= incl || lane == 31);
  if (mine) {
    int d = 255 - 8 * lane;
#pragma unroll
    for (int i = 0; i < 7; ++i)
      if (cum + h[i] < want && d == 255 - 8 * lane - i) { cum += h[i]; --d; }
    *d_out = d;
    *above_out = cum;
  }
  return mine;
}

// The barrier after one compare-exchange stage (size, stride) of a shared-memory bitonic network over P slots.
// A stage whose stride is <= `local` only moves data inside blocks of 2 * local consecutive slots, and each block
// belongs to one warp (pair layout, thread i owns pairs i, i + blockDim, ...: local = 32; slot layout, thread i owns
// slot i and its partner i ^ stride: local = 16).  Such a stage needs a warp barrier only; the CTA barrier is kept
// around the strides that couple warps (before one, after one, and after the last stage).
__device__ __forceinline__ void bitonic_stage_sync(int size, int stride, int P, int local) {
  const int next = stride > 1 ? (stride >> 1) : size;   // the first stride of the next size is `size`
  if (stride > local || next > local || (stride == 1 && size >= P)) __syncthreads();
  else __syncwarp();
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- cluster ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  cluster_arrive();
  cluster_wait();
}
// Address of `local_smem_addr` inside CTA `rank` of this cluster (shared::cluster window).
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}

// ---- mbarrier ----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init_cluster() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Arrive on a barrier that lives in another CTA of the cluster (address from mapa_u32).
// Default semantics (release at CTA scope), as CUTLASS' ClusterBarrier::arrive: the barriers this
// is used for order TMEM accesses, which the tcgen05 fences cover; a cluster-scope release would
// compile to MEMBAR.ALL.GPU and wait for every outstanding candidate store.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Same with a suspend-time hint (ns): the warp may sleep in hardware until the phase completes or the
// hint elapses, instead of burning issue slots in a spin loop.
__device__ __forceinline__ bool mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
// Acquire at cluster scope: needed when the arrive came from the peer CTA.
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a pipeline bug must surface as THR_ETIMEOUT, never as a hung GPU.  The bound is
// wall-clock (globaltimer, ns) because try_wait's own suspend slice is implementation-defined.
#ifndef THR_WATCHDOG_NS
#define THR_WATCHDOG_NS 2000000000ull
#endif
__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Returns true, or records THR_ETIMEOUT and traps: a trapped kernel fails the launch (sticky error,
// reported by thr_sync) but can never leave warps parked on a barrier that will not complete.
template <bool kClusterScope>
__device__ __forceinline__ bool mbar_wait_impl(uint32_t bar, uint32_t parity, thr_dev_status* st,
                                               int where) {
  uint64_t t0 = 0;
  for (uint32_t spin = 1;; ++spin) {
    bool ok = kClusterScope ? mbar_try_wait_cluster(bar, parity) : mbar_try_wait(bar, parity);
    if (ok) return true;
    if ((spin & 255u) == 0) {
      uint64_t now = global_timer_ns();
      if (t0 == 0) t0 = now;
      if (now - t0 > THR_WATCHDOG_NS) {
        dev_report(st, THR_ETIMEOUT, where, (long long)parity);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, thr_dev_status* st,
                                          int where) {
  return mbar_wait_impl<false>(bar, parity, st, where);
}
// For latency-tolerant roles (producers waiting for a free slot, helpers waiting for data): sleeps in
// hardware between polls so that the waiting warp leaves the issue slots to the working warps.
__device__ __forceinline__ bool mbar_wait_relaxed(uint32_t bar, uint32_t parity, thr_dev_status* st,
                                                  int where) {
  uint64_t t0 = 0;
  for (uint32_t spin = 1;; ++spin) {
    if (mbar_try_wait_hint(bar, parity, 2000u)) return true;
    if ((spin & 63u) == 0) {
      uint64_t now = global_timer_ns();
      if (t0 == 0) t0 = now;
      if (now - t0 > THR_WATCHDOG_NS) {
        dev_report(st, THR_ETIMEOUT, where, (long long)parity);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ bool mbar_wait_cluster(uint32_t bar, uint32_t parity,
                                                  thr_dev_status* st, int where) {
  return mbar_wait_impl<true>(bar, parity, st, where);
}

// ---- TMA ---------------------------------------------------------------------------------
// L2 cache-hint policies (same encodings CUTLASS passes as TMA::CacheHintSm90).
#define THR_L2_EVICT_NORMAL 0x1000000000000000ull
#define THR_L2_EVICT_FIRST 0x12F0000000000000ull
#define THR_L2_EVICT_LAST 0x14F0000000000000ull

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// 2-D tiled load into this CTA's shared memory, completion on this CTA's mbarrier.
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map,
                                            uint32_t bar, int32_t c0, int32_t c1,
                                            uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
// Same, issued by either CTA of a cta_group::2 pair: `bar` must be a shared::cluster address
// (normally the leader CTA's barrier via mapa_u32), data lands in the issuing CTA.
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const CUtensorMap* map,
                                                 uint32_t cluster_bar, int32_t c0, int32_t c1,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      ".L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(smem_dst), "l"(map), "r"(cluster_bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}

// ---- tcgen05 / TMEM ----------------------------------------------------------------------
template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
                 "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
                 "r"(ncols)
                 : "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 tile whose rows are 128 bytes (64 bf16),
// written by TMA with CU_TENSOR_MAP_SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), the
// leading-dimension offset is unused for swizzled K-major layouts, descriptor version 1 (sm_100),
// layout type 2 = SWIZZLE_128B.  Field positions: cute/arch/mma_sm100_desc.hpp SmemDescriptor.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3ffffu) >> 4);  // start address   bits [0,14)
  d |= (uint64_t)0 << 16;                        // LBO (unused)    bits [16,30)
  d |= (uint64_t)(1024u >> 4) << 32;             // SBO = 1024 B    bits [32,46)
  d |= (uint64_t)1 << 46;                        // version = 1     bits [46,48)
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B    bits [61,64)
  return d;
}

// Instruction descriptor, kind::f16: A = B = bf16 (K-major), D = fp32, dense.
// Field positions: cute/arch/mma_sm100_desc.hpp InstrDescriptor.
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(uint32_t M, uint32_t N) {
  return (1u << 4)      // c_format = F32
         | (1u << 7)    // a_format = BF16
         | (1u << 10)   // b_format = BF16
         | (0u << 15)   // a_major  = K
         | (0u << 16)   // b_major  = K
         | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; one thread issues for the CTA (or the CTA pair).
template <int kCtaGroup>
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// Make `bar` (this CTA) complete-arrive once all previously issued tcgen05.mma finished.
__device__ __forceinline__ void umma_commit_1cta(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// cta_group::2: arrive on the barrier at the same offset in every CTA of `mask`.
__device__ __forceinline__ void umma_commit_pair_mcast(uint32_t bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives lane (base + t).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- the exact dense re-score ---------------------------------------------------------------
// The exact re-score: fp64 dot of the bf16 inputs over columns [0, D) of kInFlight rows of X (row pitch ld) with the
// query row qrow (shared memory), by one warp in a fixed summation order: lane l accumulates columns l*8 .. l*8+7 of
// every 256-column block with fma, then an xor-shuffle reduction.  Every lane returns the sums.  Four rows are in
// flight so that their scattered row reads overlap.  K1's finalize, thr_dense_rescore and thr_dense_topk_rows all call
// it, so a row's score is the same bits in each.
constexpr int kInFlight = 4;
__device__ __forceinline__ void rescore_rows(const __nv_bfloat16* X, int64_t ld, int D, const uint32_t (&idx)[kInFlight],
                                             const __nv_bfloat16* qrow, int lane, double (&acc)[kInFlight]) {
#pragma unroll
  for (int u = 0; u < kInFlight; ++u) acc[u] = 0.0;
  for (int d0 = lane * 8; d0 < D; d0 += 256) {
    uint4 xv[kInFlight];
#pragma unroll
    for (int u = 0; u < kInFlight; ++u) xv[u] = *reinterpret_cast<const uint4*>(X + (size_t)idx[u] * ld + d0);
    double qd[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) qd[e] = (double)__bfloat162float(qrow[d0 + e]);
#pragma unroll
    for (int u = 0; u < kInFlight; ++u) {
      const __nv_bfloat16* xe = reinterpret_cast<const __nv_bfloat16*>(&xv[u]);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[u] = fma((double)__bfloat162float(xe[e]), qd[e], acc[u]);
    }
  }
#pragma unroll
  for (int u = 0; u < kInFlight; ++u) {
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], sh);
  }
}
