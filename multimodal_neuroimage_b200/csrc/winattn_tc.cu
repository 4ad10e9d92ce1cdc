// winattn_tc.cu -- translation unit of the tcgen05 / TMEM / TMA window-attention kernels: their host entry points
// (winattn_tc.h) are defined in winattn_tc_fwd.cuh, winattn_tc_qkv_fwd.cuh and winattn_tc_bwd.cuh.
#include "winattn_tc.h"

#include "winattn_tc_bwd.cuh"
#include "winattn_tc_qkv_fwd.cuh"

namespace mmn { namespace tc {

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  });
  return fn;
}

// Encoding a tensor map costs ~1.5 us of host time and a launch needs 32 (forward) to 56 (backward) of them, which made
// eager launches host-bound below ~100 us of kernel time.  Training loops present the same (pointer, geometry) pairs step
// after step (caching allocator), so the eight maps of a tensor are kept in a small direct-mapped cache.
namespace {
struct MapKey {
  const void* ptr; long long row_stride; int batch, channels, grid[3], win[3];
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && row_stride == o.row_stride && batch == o.batch && channels == o.channels && grid[0] == o.grid[0] &&
           grid[1] == o.grid[1] && grid[2] == o.grid[2] && win[0] == o.win[0] && win[1] == o.win[1] && win[2] == o.win[2];
  }
};
struct MapEntry { bool valid = false; MapKey key; CUtensorMap maps[8]; };
constexpr int kMapCacheSize = 256;
std::mutex g_map_mu;
MapEntry g_map_cache[kMapCacheSize];
}  // namespace

bool make_window_maps(CUtensorMap* out, const void* ptr, long long row_stride, int batch, int channels, const WinShape& g) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return false;
  if (reinterpret_cast<uintptr_t>(ptr) % 16) return false;
  MapKey key{ptr, row_stride, batch, channels, {g.grid[0], g.grid[1], g.grid[2]}, {g.win[0], g.win[1], g.win[2]}};
  const size_t hsh = (reinterpret_cast<uintptr_t>(ptr) >> 4) * 0x9E3779B97F4A7C15ull ^ (size_t)row_stride * 1315423911u ^
                     (size_t)batch * 2654435761u ^ (size_t)(g.win[0] * 31 + g.win[1] * 7 + g.win[2]);
  MapEntry& slot = g_map_cache[(hsh >> 17) % kMapCacheSize];
  std::lock_guard<std::mutex> lock(g_map_mu);
  if (slot.valid && slot.key == key) {
    for (int c = 0; c < 8; ++c) out[c] = slot.maps[c];
    return true;
  }
  cuuint64_t dims[5] = {(cuuint64_t)channels, (cuuint64_t)g.grid[2], (cuuint64_t)g.grid[1], (cuuint64_t)g.grid[0], (cuuint64_t)batch};
  cuuint64_t rs = (cuuint64_t)row_stride * 2;
  cuuint64_t strides[4] = {rs, rs * g.grid[2], rs * g.grid[2] * g.grid[1], rs * g.grid[2] * g.grid[1] * g.grid[0]};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  for (int cls = 0; cls < 8; ++cls) {
    cuuint32_t box[5] = {kD, (cuuint32_t)(cls & 4 ? g.win[2] / 2 : g.win[2]), (cuuint32_t)(cls & 2 ? g.win[1] / 2 : g.win[1]),
                         (cuuint32_t)(cls & 1 ? g.win[0] / 2 : g.win[0]), 1};
    for (int i = 1; i < 4; ++i) if (box[i] < 1) box[i] = 1;      // class unused for this geometry (unit extent)
    CUresult r = enc(&out[cls], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
  }
  slot.key = key;
  for (int c = 0; c < 8; ++c) slot.maps[c] = out[c];
  slot.valid = true;
  return true;
}

}}  // namespace mmn::tc
