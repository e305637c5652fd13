// api.cu — handle lifetime, error reporting, scratch and TMA descriptor encoding for libthr.so.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

static char g_create_err[512] = "";

void thr_dense_state_free(thr_handle* h);
void thr_bm25_state_free(thr_handle* h);

int thr_fail(thr_handle* h, int code, const char* fmt, ...) {
  char* dst = h ? h->err : g_create_err;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(dst, 512, fmt, ap);
  va_end(ap);
  return code;
}

void* thr_scratch(thr_handle* h, int arena, size_t bytes) {
  if (bytes <= h->scratch_bytes[arena]) return h->scratch[arena];
  if (h->scratch[arena]) {
    cudaDeviceSynchronize();  // previous users may still be in flight
    cudaFree(h->scratch[arena]);
    h->scratch[arena] = nullptr;
    h->scratch_bytes[arena] = 0;
  }
  size_t want = bytes + (bytes >> 2);
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    thr_fail(h, THR_ENOMEM, "cudaMalloc(%zu) for scratch failed: %s", want, cudaGetErrorString(e));
    return nullptr;
  }
  h->scratch[arena] = p;
  h->scratch_bytes[arena] = want;
  return p;
}

int thr_prof_begin(thr_handle* h, int slot, cudaStream_t s) {
  if (!h->prof_on || h->prof_n >= kProfMax || !((h->prof_mask >> slot) & 1u)) return -1;
  int i = h->prof_n++;
  h->prof_slot[i] = (unsigned char)slot;
  cudaEventRecord(h->prof_ev[2 * i], s);
  return i;
}
void thr_prof_end(thr_handle* h, int token, cudaStream_t s) {
  if (token >= 0) cudaEventRecord(h->prof_ev[2 * token + 1], s);
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                    const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int thr_encode_tma_2d_bf16(thr_handle* h, CUtensorMap* map, const void* base, uint64_t rows,
                           uint64_t cols, uint32_t box_rows, uint32_t box_cols) {
  static encode_tiled_fn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p)
      return thr_fail(h, THR_ECUDA, "cuTensorMapEncodeTiled entry point unavailable: %s",
                      cudaGetErrorString(e));
    fn = (encode_tiled_fn)p;
  }
  if (((uintptr_t)base & 15u) != 0 || (cols * 2) % 16 != 0)
    return thr_fail(h, THR_EINVAL, "TMA source must be 16-byte aligned with a 16-byte row pitch");
  cuuint64_t dims[2] = {cols, rows};           // innermost first
  cuuint64_t strides[1] = {cols * 2};          // bytes, dims 1..rank-1
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides,
                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return thr_fail(h, THR_ECUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu)",
                    (int)r, (unsigned long long)rows, (unsigned long long)cols);
  return THR_OK;
}

extern "C" {

int thr_abi_version(void) { return THR_ABI_VERSION; }

int thr_create(int device, thr_handle** out) {
  if (!out) return thr_fail(nullptr, THR_EINVAL, "thr_create: out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return thr_fail(nullptr, THR_ECUDA, "thr_create: no CUDA device (%s); there is no CPU fallback",
                    cudaGetErrorString(e));
  if (device < 0 || device >= count)
    return thr_fail(nullptr, THR_EINVAL, "thr_create: device %d out of range [0,%d)", device, count);
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess)
    return thr_fail(nullptr, THR_ECUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10)
    return thr_fail(nullptr, THR_EUNSUPPORTED,
                    "thr_create: device %d is sm_%d%d; libthr is built for sm_100a (B200) only", device,
                    prop.major, prop.minor);
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return thr_fail(nullptr, THR_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  thr_handle* h = (thr_handle*)calloc(1, sizeof(thr_handle));
  if (!h) return thr_fail(nullptr, THR_ENOMEM, "thr_create: out of host memory");
  h->device = device;
  h->prof_mask = 0xffffffffu;
  h->num_sms = prop.multiProcessorCount;
  e = cudaHostAlloc((void**)&h->h_status, sizeof(thr_dev_status), cudaHostAllocMapped);
  if (e == cudaSuccess) {
    memset(h->h_status, 0, sizeof(thr_dev_status));
    e = cudaHostGetDevicePointer((void**)&h->d_status, h->h_status, 0);
  }
  if (e != cudaSuccess) {
    free(h);
    return thr_fail(nullptr, THR_ECUDA, "thr_create: status word: %s", cudaGetErrorString(e));
  }
  h->err[0] = 0;
  *out = h;
  return THR_OK;
}

int thr_destroy(thr_handle* h) {
  if (!h) return THR_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  thr_dense_state_free(h);
  thr_bm25_state_free(h);
  for (int i = 0; i < 2; ++i)
    if (h->scratch[i]) cudaFree(h->scratch[i]);
  if (h->prof_ev) {
    for (int i = 0; i < 2 * kProfMax; ++i) cudaEventDestroy(h->prof_ev[i]);
    free(h->prof_ev);
    free(h->prof_slot);
  }
  if (h->h_status) cudaFreeHost(h->h_status);
  free(h);
  return THR_OK;
}

int thr_prof_enable(thr_handle* h, int on) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  if (on && !h->prof_ev) {
    h->prof_ev = (cudaEvent_t*)calloc(2 * kProfMax, sizeof(cudaEvent_t));
    h->prof_slot = (unsigned char*)calloc(kProfMax, 1);
    if (!h->prof_ev || !h->prof_slot) return thr_fail(h, THR_ENOMEM, "out of host memory");
    for (int i = 0; i < 2 * kProfMax; ++i) THR_CUDA(h, cudaEventCreate(&h->prof_ev[i]));
  }
  h->prof_on = on ? 1 : 0;
  return THR_OK;
}

int thr_prof_select(thr_handle* h, unsigned mask) {
  if (!h) return THR_EINVAL;
  h->prof_mask = mask;
  return THR_OK;
}

int thr_prof_reset(thr_handle* h) {
  if (!h) return THR_EINVAL;
  h->prof_n = 0;
  return THR_OK;
}

int thr_prof_read(thr_handle* h, int slot, double* total_ms, int64_t* launches) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  THR_REQUIRE(h, slot >= 0 && slot < THR_PROF_SLOTS && total_ms && launches, "thr_prof_read: bad argument");
  THR_CUDA(h, cudaDeviceSynchronize());
  double tot = 0.0;
  int64_t n = 0;
  for (int i = 0; i < h->prof_n; ++i) {
    if (h->prof_slot[i] != slot) continue;
    float ms = 0.f;
    THR_CUDA(h, cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
    tot += ms;
    ++n;
  }
  *total_ms = tot;
  *launches = n;
  return THR_OK;
}

const char* thr_last_error(const thr_handle* h) { return h ? h->err : g_create_err; }

int64_t thr_launch_count(const thr_handle* h) { return h ? h->launches : 0; }

int thr_peer_enable(thr_handle* h, int peer_device) {
  if (!h) return THR_EINVAL;
  THR_CUDA(h, cudaSetDevice(h->device));
  int count = 0;
  THR_CUDA(h, cudaGetDeviceCount(&count));
  THR_REQUIRE(h, peer_device >= 0 && peer_device < count, "thr_peer_enable: device %d out of range [0,%d)", peer_device, count);
  if (peer_device == h->device) return THR_OK;
  int can = 0;
  THR_CUDA(h, cudaDeviceCanAccessPeer(&can, h->device, peer_device));
  if (!can)
    return thr_fail(h, THR_EUNSUPPORTED, "thr_peer_enable: device %d cannot access device %d", h->device, peer_device);
  const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();   // clear the sticky-free "already enabled" status: it is success here
    return THR_OK;
  }
  if (e != cudaSuccess)
    return thr_fail(h, THR_ECUDA, "cudaDeviceEnablePeerAccess(%d) on device %d: %s", peer_device, h->device,
                    cudaGetErrorString(e));
  return THR_OK;
}

int thr_sync(thr_handle* h, void* stream) {
  if (!h) return THR_EINVAL;
  cudaSetDevice(h->device);
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  volatile thr_dev_status* st = h->h_status;
  if (st->code != 0) {
    int code = st->code, where = st->where;
    long long aux = st->aux;
    st->code = 0;
    const char* what = code == THR_EOVERFLOW  ? "candidate buffer overflow"
                       : code == THR_ETIMEOUT ? "pipeline watchdog timeout (kernel trapped)"
                       : code == THR_EINVAL   ? "invalid input detected on the device (tag 460: a BM25 query has more than 32 terms)"
                                              : "device-side failure";
    return thr_fail(h, code, "%s (kernel tag %d, detail %lld)%s%s", what, where, aux,
                    e != cudaSuccess ? "; CUDA: " : "", e != cudaSuccess ? cudaGetErrorString(e) : "");
  }
  if (e != cudaSuccess)
    return thr_fail(h, THR_ECUDA, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
  return THR_OK;
}

}  // extern "C"
