// Host-side TMA descriptor construction.  cuTensorMapEncodeTiled is fetched through the runtime's driver entry
// point lookup so that libltxcuda.so has no link-time dependency on libcuda.so (it must build on a GPU-less box).
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <set>

#include "ltx_internal.h"

namespace ltx {

bool pdl_enabled(int cls) {
  static const bool on = [] { const char* e = getenv("LTX_PDL"); return e ? atoi(e) != 0 : true; }();
  static const int mask = [] { const char* e = getenv("LTX_PDL_MASK"); return e ? atoi(e) : 0xFF; }();
  return on && ((mask >> cls) & 1);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  LTX_CHECK(fn != nullptr, 3, "cuTensorMapEncodeTiled not available (no CUDA driver / no sm_100a device)");
  return fn;
}

CUtensorMap make_tmap_2d(const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                         uint32_t box_cols) {
  LTX_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, 2, "TMA base must be 16-byte aligned");
  LTX_CHECK((ld * 2) % 16 == 0, 2, "TMA row pitch must be a multiple of 16 bytes");
  LTX_CHECK(box_rows <= 256 && box_cols * 2 == 128, 2, "TMA box: <=256 rows, 128-byte inner extent");
  CUtensorMap m;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTX_CHECK(r == CUDA_SUCCESS, 3, "cuTensorMapEncodeTiled(2d) failed: " + std::to_string(static_cast<int>(r)));
  return m;
}

CUtensorMap make_tmap_thwc(const void* base, uint64_t T, uint64_t H, uint64_t W, uint64_t C, uint32_t bt, uint32_t bh,
                           uint32_t bw) {
  LTX_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, 2, "TMA base must be 16-byte aligned");
  LTX_CHECK(C % 8 == 0, 2, "channels must be a multiple of 8");
  LTX_CHECK(bt * bh * bw <= 256 && bw <= 256 && bh <= 256, 2, "TMA conv box too large");
  CUtensorMap m;
  cuuint64_t dims[4] = {C, W, H, T};
  cuuint64_t strides[3] = {C * 2, W * C * 2, H * W * C * 2};
  cuuint32_t box[4] = {64, bw, bh, bt};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTX_CHECK(r == CUDA_SUCCESS, 3, "cuTensorMapEncodeTiled(4d) failed: " + std::to_string(static_cast<int>(r)));
  return m;
}

CUtensorMap make_tmap_3d(const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1, uint64_t stride2,
                         uint32_t box0, uint32_t box1) {
  // bf16 tensor, dims (d0 fastest, d1, d2), strides in ELEMENTS for d1 / d2; box = [box0, box1, 1], 128B swizzle.
  LTX_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, 2, "TMA base must be 16-byte aligned");
  LTX_CHECK((stride1 * 2) % 16 == 0 && (stride2 * 2) % 16 == 0, 2, "TMA strides must be multiples of 16 bytes");
  LTX_CHECK(box0 * 2 == 128 && box1 <= 256, 2, "TMA box: 128-byte inner extent, <= 256 rows");
  CUtensorMap m;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1 * 2, stride2 * 2};
  cuuint32_t box[3] = {box0, box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTX_CHECK(r == CUDA_SUCCESS, 3, "cuTensorMapEncodeTiled(3d) failed: " + std::to_string(static_cast<int>(r)));
  return m;
}

CUtensorMap make_tmap_u8(const void* base, uint64_t rows, uint64_t row_bytes, uint32_t box_rows, uint32_t box_bytes) {
  LTX_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && row_bytes % 16 == 0, 2, "TMA u8: 16-byte alignment");
  LTX_CHECK(box_rows <= 256 && box_bytes % 16 == 0 && box_bytes <= 256, 2, "TMA u8 box");
  CUtensorMap m;
  cuuint64_t dims[2] = {row_bytes, rows};
  cuuint64_t strides[1] = {row_bytes};
  cuuint32_t box[2] = {box_bytes, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTX_CHECK(r == CUDA_SUCCESS, 3, "cuTensorMapEncodeTiled(u8) failed: " + std::to_string(static_cast<int>(r)));
  return m;
}

CUtensorMap make_tmap_u8_sw128(const void* base, uint64_t rows, uint64_t cols, uint64_t row_bytes, uint32_t box_rows) {
  LTX_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && row_bytes % 16 == 0 && cols % 16 == 0, 2, "TMA u8: 16-byte alignment");
  LTX_CHECK(box_rows <= 256, 2, "TMA u8 box: <= 256 rows");
  CUtensorMap m;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {row_bytes};
  cuuint32_t box[2] = {128, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  LTX_CHECK(r == CUDA_SUCCESS, 3, "cuTensorMapEncodeTiled(u8, sw128) failed: " + std::to_string(static_cast<int>(r)));
  return m;
}

// Per-device caches (one process may hold contexts on several GPUs, each driven by its own host thread): the SM count and the
// set of kernels that already opted in to more than 48 KB of dynamic shared memory -- cudaFuncSetAttribute is per device.
namespace {
constexpr int kMaxDevices = 64;
std::mutex g_attr_mutex;
std::set<const void*> g_smem_done[kMaxDevices];
std::atomic<int> g_sm_count[kMaxDevices];
int current_device() {
  int dev = 0;
  LTX_CUDA(cudaGetDevice(&dev));
  LTX_CHECK(dev >= 0 && dev < kMaxDevices, 3, "device index out of range");
  return dev;
}
}  // namespace

int device_sm_count() {
  const int dev = current_device();
  int n = g_sm_count[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    LTX_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    g_sm_count[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

void ensure_dyn_smem(const void* kernel, size_t bytes) {
  const int dev = current_device();
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  if (g_smem_done[dev].count(kernel)) return;
  LTX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes)));
  g_smem_done[dev].insert(kernel);
}

}  // namespace ltx
