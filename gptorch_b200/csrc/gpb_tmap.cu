// gpb_tmap.cu -- host-side TMA tensor-map encoding (driver entry point fetched at run time, no -lcuda).
#include "gpb_common.cuh"
#include <cudaTypedefs.h>
#include <mutex>
#include <atomic>
#include <cstdio>
#include <cstring>

namespace gpb {

static thread_local char g_last_error[512] = "";

void set_last_error(cudaError_t e, const char* file, int line) {
  snprintf(g_last_error, sizeof(g_last_error), "CUDA error %d (%s) at %s:%d", static_cast<int>(e),
           cudaGetErrorString(e), file, line);
}
void set_last_error_msg(const char* msg) { snprintf(g_last_error, sizeof(g_last_error), "%s", msg); }
const char* last_error() { return g_last_error; }

static std::atomic<long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
long launch_count() { return g_launches.load(std::memory_order_relaxed); }
void reset_launch_count() { g_launches.store(0, std::memory_order_relaxed); }

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  });
  return fn;
}

int make_tmap_f64(CUtensorMap* out, const double* base, long rows, long cols, long ld, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) { set_last_error_msg("cuTensorMapEncodeTiled entry point unavailable"); return GPB_ERR_DRIVER; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld & 1) || rows <= 0 || cols <= 0 || ld < cols) {
    set_last_error_msg("tensor map: base must be 16-byte aligned, ld even and >= cols");
    return GPB_ERR_ALIGN;
  }
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * sizeof(double)};
  cuuint32_t box[2] = {16u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_last_error, sizeof(g_last_error), "cuTensorMapEncodeTiled failed with CUresult %d (rows=%ld cols=%ld ld=%ld box=%d)",
             static_cast<int>(r), rows, cols, ld, box_rows);
    return GPB_ERR_DRIVER;
  }
  return GPB_OK;
}

int make_tmap_i8_slices(CUtensorMap* out, const int8_t* base, long rows, int k, int slices, int box_k, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) { set_last_error_msg("cuTensorMapEncodeTiled entry point unavailable"); return GPB_ERR_DRIVER; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (k & 15) || rows <= 0 || k <= 0 || slices <= 0) {
    set_last_error_msg("int8 slice tensor map: base must be 16-byte aligned and k a multiple of 16");
    return GPB_ERR_ALIGN;
  }
  cuuint64_t gdim[3] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(slices), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[2] = {static_cast<cuuint64_t>(k), static_cast<cuuint64_t>(k) * slices};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(box_k), 1u, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  const CUtensorMapSwizzle swz = box_k == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : box_k == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    snprintf(g_last_error, sizeof(g_last_error), "cuTensorMapEncodeTiled (int8) failed with CUresult %d (rows=%ld k=%d S=%d)",
             static_cast<int>(r), rows, k, slices);
    return GPB_ERR_DRIVER;
  }
  return GPB_OK;
}

}  // namespace gpb
