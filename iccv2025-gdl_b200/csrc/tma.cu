// tma.cu — host side of the Tensor Memory Accelerator plumbing declared in tma.cuh: CUtensorMap creation through the
// driver entry point fetched from the runtime (the library does not link libcuda), with a small cache keyed by
// (pointer, geometry, box) so that a CUDA-graph-captured step never re-encodes a descriptor.
#include <mutex>
#include <unordered_map>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "tma.cuh"

namespace gdl {
using namespace tc05;

// ------------------------------------------------------------------------------------------
// tensor-map cache
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

struct TmapKey {
  uint64_t v[6];
  bool operator==(const TmapKey& o) const { return memcmp(v, o.v, sizeof(v)) == 0; }
};
struct TmapHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : k.v) h = (h ^ x) * 1099511628211ull;
    return (size_t)h;
  }
};
static std::mutex g_tmap_mu;
static std::unordered_map<TmapKey, CUtensorMap*, TmapHash> g_tmaps;

static const CUtensorMap* cached_tmap(const TmapKey& key, cuuint32_t rank, void* ptr, const cuuint64_t* dims,
                                      const cuuint64_t* strides, const cuuint32_t* box,
                                      CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  std::lock_guard<std::mutex> lk(g_tmap_mu);
  auto it = g_tmaps.find(key);
  if (it != g_tmaps.end()) return it->second;
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_last_error("cuTensorMapEncodeTiled entry point not available");
    return nullptr;
  }
  CUtensorMap* m = nullptr;
  if (posix_memalign(reinterpret_cast<void**>(&m), 64, sizeof(CUtensorMap)) != 0) return nullptr;
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, ptr, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    set_last_error(buf);
    free(m);
    return nullptr;
  }
  g_tmaps.emplace(key, m);
  return m;
}

const CUtensorMap* tmap_nhwc(const void* ptr, int N, int H, int W, int C, int box_w, int box_h) {
  TmapKey key{{(uint64_t)ptr, ((uint64_t)N << 32) | (uint32_t)H, ((uint64_t)W << 32) | (uint32_t)C,
               ((uint64_t)box_w << 32) | (uint32_t)box_h, 4, 0}};
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  return cached_tmap(key, 4, const_cast<void*>(ptr), dims, strides, box);
}

const CUtensorMap* tmap_rows(const void* ptr, int64_t rows, int64_t K, int box_rows) {
  TmapKey key{{(uint64_t)ptr, (uint64_t)rows, (uint64_t)K, (uint64_t)box_rows, 2, 0}};
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  return cached_tmap(key, 2, const_cast<void*>(ptr), dims, strides, box);
}

// Strided 4-D view {C, W, H, N} of a bf16 tensor (element strides sW, sH, sN; channels contiguous),
// box {64, box_w, box_h, box_n}: whole padded pixel rows / row bands / images per TMA operation
// (conv_flat.cu, conv_wgrad_flat.cu).  box_w may exceed W: the surplus pixels are out-of-bounds zero fill.
const CUtensorMap* tmap_view4(const void* ptr, int C, int W, int H, int N, int64_t sW, int64_t sH, int64_t sN,
                              int box_w, int box_h, int box_n) {
  TmapKey key{{(uint64_t)ptr, ((uint64_t)N << 32) | (uint32_t)H, ((uint64_t)W << 32) | (uint32_t)C,
               ((uint64_t)box_w << 32) | ((uint64_t)box_h << 16) | (uint64_t)box_n | 0x80000000ull,
               (uint64_t)sW ^ ((uint64_t)sH << 24), (uint64_t)sN}};
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sW * 2, (cuuint64_t)sH * 2, (cuuint64_t)sN * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_n};
  return cached_tmap(key, 4, const_cast<void*>(ptr), dims, strides, box);
}

// 16-channel (32-byte rows, 32-byte swizzle) variants used by the space-to-depth stems.
const CUtensorMap* tmap_nhwc16(const void* ptr, int N, int H, int W, int box_w, int box_h) {
  TmapKey key{{(uint64_t)ptr, ((uint64_t)N << 32) | (uint32_t)H, ((uint64_t)W << 32) | 16u,
               ((uint64_t)box_w << 32) | (uint32_t)box_h, 4, 32}};
  cuuint64_t dims[4] = {16, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {32, (cuuint64_t)W * 32, (cuuint64_t)H * W * 32};
  cuuint32_t box[4] = {16, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  return cached_tmap(key, 4, const_cast<void*>(ptr), dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}
const CUtensorMap* tmap_rows16(const void* ptr, int64_t rows, int64_t K, int box_rows) {
  TmapKey key{{(uint64_t)ptr, (uint64_t)rows, (uint64_t)K, (uint64_t)box_rows, 2, 32}};
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {16, (cuuint32_t)box_rows};
  return cached_tmap(key, 2, const_cast<void*>(ptr), dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

}  // namespace gdl
