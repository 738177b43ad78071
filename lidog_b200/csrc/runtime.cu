// Per-device runtime of liblidog_b200: SM count, the device error word the bounded mbarrier waits report into,
// the self-resetting schedule / ticket counters, TMA descriptor encoding, and the library-owned scratch ARENA.
//
// Arena (SURVEY.md 8b "ownership"): every fused layer entry point (lg_conv_layer_*, lg_bn_layer_*, lg_coords_pyramid)
// needs scratch that only lives for the duration of the call -- split-K partials, block partials of the BN
// reductions, scan workspaces, exchange staging.  It comes from one cudaMalloc'ed block per (device, stream) that
// grows monotonically and is reused by every call: stream order makes the reuse safe, the block is outside torch's
// caching allocator (so the reference loop's per-step torch.cuda.empty_cache(), trainer_lighting_2d.py:147-148,
// never turns scratch into cudaMalloc calls) and the host issues no allocation per layer.
#include <mutex>
#include <string.h>

#include "common.cuh"
#include "runtime.cuh"

namespace lg {

namespace {
constexpr int kMaxDevices = 64;
constexpr int kMaxArenas = 16;  // (device, stream) pairs in use at once; LiDOG uses one stream per process
struct Arena {
  cudaStream_t stream = nullptr;
  bool used = false;
  char* base = nullptr;
  size_t cap = 0, off = 0;
};
struct DeviceRt {
  bool ready = false;
  int sm_count = 0;
  int* err_word = nullptr;
  int* counters = nullptr;  // kCounterSlots slots of 8 ints, zero at rest (every kernel leaves its slot zeroed)
  unsigned seq = 0;
  Arena arenas[kMaxArenas];
};
DeviceRt g_rt[kMaxDevices];
std::mutex g_mu;
constexpr int kCounterSlots = 64;

int device_rt(DeviceRt** out) {
  int dev = 0;
  LG_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) {
    set_error("device index %d out of range", dev);
    return LG_ERR_INVALID;
  }
  DeviceRt& r = g_rt[dev];
  if (!r.ready) {
    LG_CUDA_OK(cudaDeviceGetAttribute(&r.sm_count, cudaDevAttrMultiProcessorCount, dev));
    LG_CUDA_OK(cudaMalloc(&r.err_word, sizeof(int)));
    LG_CUDA_OK(cudaMemset(r.err_word, 0, sizeof(int)));
    LG_CUDA_OK(cudaMalloc(&r.counters, kCounterSlots * 8 * sizeof(int)));
    LG_CUDA_OK(cudaMemset(r.counters, 0, kCounterSlots * 8 * sizeof(int)));
    r.ready = true;
  }
  *out = &r;
  return LG_OK;
}
}  // namespace

int tc_runtime(int* sm_count, int** err_word) {
  std::lock_guard<std::mutex> lock(g_mu);
  DeviceRt* r;
  int rc = device_rt(&r);
  if (rc) return rc;
  *sm_count = r->sm_count;
  *err_word = r->err_word;
  return LG_OK;
}

// Counter slots are handed out round-robin so launches in flight on different streams never share one.
int counter_slot(int** out) {
  std::lock_guard<std::mutex> lock(g_mu);
  DeviceRt* r;
  int rc = device_rt(&r);
  if (rc) return rc;
  *out = r->counters + 8 * (r->seq++ % kCounterSlots);
  return LG_OK;
}

int arena_begin(cudaStream_t stream, size_t bytes, ArenaCursor* cur) {
  std::lock_guard<std::mutex> lock(g_mu);
  DeviceRt* r;
  int rc = device_rt(&r);
  if (rc) return rc;
  Arena* a = nullptr;
  for (int i = 0; i < kMaxArenas && !a; ++i)
    if (r->arenas[i].used && r->arenas[i].stream == stream) a = &r->arenas[i];
  for (int i = 0; i < kMaxArenas && !a; ++i)
    if (!r->arenas[i].used) {
      a = &r->arenas[i];
      a->used = true;
      a->stream = stream;
    }
  if (!a) {
    set_error("arena: more than %d streams use the library on one device", kMaxArenas);
    return LG_ERR_INVALID;
  }
  bytes = (bytes + 1023) & ~(size_t)1023;
  if (bytes > a->cap) {
    // grow: cudaFree waits for the work in flight, so nothing still reads the old block
    if (a->base) LG_CUDA_OK(cudaFree(a->base));
    a->base = nullptr;
    a->cap = 0;
    size_t want = bytes + bytes / 4;
    if (want < (size_t)8 << 20) want = (size_t)8 << 20;
    LG_CUDA_OK(cudaMalloc(&a->base, want));
    a->cap = want;
  }
  cur->base = a->base;
  cur->cap = a->cap;
  cur->off = 0;
  return LG_OK;
}

void* arena_take(ArenaCursor* cur, size_t bytes) {
  const size_t off = cur->off;
  cur->off = off + ((bytes + 255) & ~(size_t)255);
  return cur->off <= cur->cap ? cur->base + off : nullptr;
}

size_t arena_total_bytes() {
  std::lock_guard<std::mutex> lock(g_mu);
  size_t t = 0;
  for (auto& r : g_rt)
    for (auto& a : r.arenas) t += a.cap;
  return t;
}

int arena_release_all() {
  std::lock_guard<std::mutex> lock(g_mu);
  int dev0 = 0;
  LG_CUDA_OK(cudaGetDevice(&dev0));
  for (int d = 0; d < kMaxDevices; ++d)
    for (auto& a : g_rt[d].arenas)
      if (a.base) {
        LG_CUDA_OK(cudaSetDevice(d));
        LG_CUDA_OK(cudaFree(a.base));
        a = Arena();
      }
  LG_CUDA_OK(cudaSetDevice(dev0));
  return LG_OK;
}

// ------------------------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2D row-major 16-bit matrix [rows][cols]; box = box_rows x 32 columns, SWIZZLE_64B
int tc_make_tmap(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return LG_ERR_CUDA;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)(rows > 0 ? rows : 1)};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld box_rows=%d", (int)r, (long long)rows,
              (long long)cols, box_rows);
    return LG_ERR_CUDA;
  }
  return LG_OK;
}

}  // namespace lg

using namespace lg;

extern "C" size_t lg_arena_bytes(void) { return arena_total_bytes(); }
extern "C" int lg_arena_release(void) { return arena_release_all(); }
