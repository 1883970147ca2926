#include "common.h"

#include <unordered_map>

#include <mutex>

namespace abcgpt {

char* last_error_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}

// The caller decides (abcgpt_set_pdl): on for the chain of small kernels of a decoded token (+11 % tokens/s), off for the
// training step, where every kernel fills the GPU for 25-400 us and the early-resident CTAs cost more than the hidden launch
// latency (measured -1.8 %).
static bool g_pdl = false;
void set_pdl(bool on) { g_pdl = on; }
bool pdl_enabled() { return g_pdl; }

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static CUtensorMapDataType dtype_of(int elem_bytes) {
  return elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
}

static int encode_tmap_2d_uncached(CUtensorMap* tm, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer,
                                   uint64_t row_bytes, uint32_t box_inner, uint32_t box_outer, int swizzle_bytes);

// ---- descriptor cache ------------------------------------------------------------------------------------------------
// A tensor map is a pure function of (pointer, element size, dims, pitch, box, swizzle) and costs a few microseconds of
// driver time to encode.  The training step re-uses ~400 of them every iteration and the decode loop ~100 per generated
// token (there the host-side launch cost IS the step time), so encoded maps are kept in a small per-thread table.
namespace {
struct TmapKey {
  const void* ptr;
  uint64_t inner, outer, row_bytes;
  uint32_t box_inner, box_outer;
  int elem_bytes, swizzle;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && inner == o.inner && outer == o.outer && row_bytes == o.row_bytes && box_inner == o.box_inner &&
           box_outer == o.box_outer && elem_bytes == o.elem_bytes && swizzle == o.swizzle;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
    h ^= (k.inner + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (k.outer * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
    h ^= (k.row_bytes + (static_cast<uint64_t>(k.box_inner) << 40) + (static_cast<uint64_t>(k.box_outer) << 20) +
          (static_cast<uint64_t>(k.elem_bytes) << 4) + static_cast<uint64_t>(k.swizzle) + (h << 6) + (h >> 2));
    return static_cast<size_t>(h);
  }
};
std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash>& tmap_cache() {
  thread_local std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  return cache;
}
constexpr size_t kTmapCacheMax = 16384;
}  // namespace

int encode_tmap_2d(CUtensorMap* tm, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer,
                   uint64_t row_bytes, uint32_t box_inner, uint32_t box_outer, bool swizzle128) {
  return encode_tmap_2d_sw(tm, ptr, elem_bytes, inner, outer, row_bytes, box_inner, box_outer, swizzle128 ? 128 : 0);
}

int encode_tmap_2d_sw(CUtensorMap* tm, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer,
                      uint64_t row_bytes, uint32_t box_inner, uint32_t box_outer, int swizzle_bytes) {
  const TmapKey key{ptr, inner, outer, row_bytes, box_inner, box_outer, elem_bytes, swizzle_bytes};
  auto& cache = tmap_cache();
  if (auto it = cache.find(key); it != cache.end()) {
    *tm = it->second;
    return 0;
  }
  const int rc = encode_tmap_2d_uncached(tm, ptr, elem_bytes, inner, outer, row_bytes, box_inner, box_outer, swizzle_bytes);
  if (rc == 0) {
    if (cache.size() >= kTmapCacheMax) cache.clear();
    cache.emplace(key, *tm);
  }
  return rc;
}

static int encode_tmap_2d_uncached(CUtensorMap* tm, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer,
                                   uint64_t row_bytes, uint32_t box_inner, uint32_t box_outer, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(-2, "cuTensorMapEncodeTiled entry point unavailable");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) return fail(-1, "TMA base pointer must be 16-byte aligned");
  if ((row_bytes & 15) != 0) return fail(-1, "TMA row pitch must be a multiple of 16 bytes (got %llu)",
                                         (unsigned long long)row_bytes);
  if (swizzle_bytes != 0 && swizzle_bytes != 64 && swizzle_bytes != 128) return fail(-1, "TMA swizzle must be 0, 64 or 128 bytes");
  if (swizzle_bytes != 0 && box_inner * elem_bytes != static_cast<uint32_t>(swizzle_bytes))
    return fail(-1, "a %d-byte swizzle needs a %d-byte inner box", swizzle_bytes, swizzle_bytes);
  if (box_inner > 256 || box_outer > 256) return fail(-1, "TMA box dims must be <= 256");
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, dtype_of(elem_bytes), 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(1000 + static_cast<int>(r), "cuTensorMapEncodeTiled(2d) failed with CUresult %d (inner=%llu outer=%llu "
                "pitch=%llu box=%ux%u)", (int)r, (unsigned long long)inner, (unsigned long long)outer,
                (unsigned long long)row_bytes, box_inner, box_outer);
  return 0;
}

int encode_tmap_3d(CUtensorMap* tm, const void* ptr, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                   uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1, uint32_t box2,
                   bool swizzle128) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(-2, "cuTensorMapEncodeTiled entry point unavailable");
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) return fail(-1, "TMA base pointer must be 16-byte aligned");
  if ((stride1_bytes & 15) != 0 || (stride2_bytes & 15) != 0) return fail(-1, "TMA strides must be multiples of 16 B");
  if (swizzle128 && box0 * elem_bytes != 128) return fail(-1, "swizzle128 needs a 128-byte inner box");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, dtype_of(elem_bytes), 3, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(1000 + static_cast<int>(r), "cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
  return 0;
}

}  // namespace abcgpt
