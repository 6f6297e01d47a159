// gpb_common.cuh -- shared device helpers for the gptorch-b200 CUDA library (sm_100a only).
//
// Everything in this library is IEEE fp64 (the reference fixes torch.double, gptorch/util.py:11-12).
// The FP64 tensor path on sm_100a is the warp-level DMMA.8x8x4 (tcgen05 has no f64 kind); operand
// tiles are staged in shared memory by TMA (cp.async.bulk.tensor + mbarrier) with the 128-byte swizzle.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>
#include <atomic>

#define GPB_OK 0
#define GPB_ERR_BADARG (-1)
#define GPB_ERR_ALIGN (-2)
#define GPB_ERR_CUDA (-3)
#define GPB_ERR_DRIVER (-4)
#define GPB_ERR_UNSUPPORTED (-5)

#define GPB_CUDA_CHECK(expr)                                   \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) { gpb::set_last_error(_e, __FILE__, __LINE__); return GPB_ERR_CUDA; } \
  } while (0)

namespace gpb {

void set_last_error(cudaError_t e, const char* file, int line);
// Every kernel launch of this library is counted (bench.py reports it as gpu_launches).
void count_launch(int n = 1);
long launch_count();
void reset_launch_count();

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remember the largest size set for each device.
// `state` is a per-kernel static array of GPB_MAX_DEVICES ints, zero-initialised.
constexpr int GPB_MAX_DEVICES = 64;
// (atomics: the library may be entered from several host threads; setting the attribute twice is harmless.)
template <typename KernelT>
inline int ensure_dynamic_smem(KernelT kernel, int bytes, std::atomic<int>* state) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= GPB_MAX_DEVICES) return GPB_ERR_CUDA;
  if (bytes > state[dev].load(std::memory_order_relaxed)) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { set_last_error(e, __FILE__, __LINE__); return GPB_ERR_CUDA; }
    state[dev].store(bytes, std::memory_order_relaxed);
  }
  return GPB_OK;
}

// Block size every blocked algorithm in this library is built on (diagonal blocks, Dinv workspace).
constexpr int NB = 128;

// ----------------------------------------------------------------------------------------------
// PTX wrappers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}

// TMA 2-D tiled load global -> shared; completion is signalled on `bar` as transaction bytes.
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// Thread-block clusters: this CTA's rank in its cluster, and a barrier over every thread of the cluster that also orders
// shared-memory writes (mbarrier initialisation included) before the peers' reads.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// D(8x8) += A(8x4,row) * B(4x8,col), fp64.  Lane l holds A[l>>2][l&3], B[l&3][l>>2], C[l>>2][2*(l&3)+{0,1}].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}
// Same instruction, but ordered with respect to the other volatile asm statements of the kernel (shared-memory
// fragment loads, mbarrier arrives).  The TMA-ring GEMM must not let the compiler sink the MMAs that consume the
// last fragments of a stage below the "stage empty" arrive: an MMA issues only once its operand loads have
// returned, so MMA-before-arrive is what guarantees that no LDS of the stage is still in flight when the
// producer is allowed to overwrite it.
__device__ __forceinline__ void dmma884_ordered(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double ld_shared_f64(uint32_t addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
  return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic block-wide sum (fixed tree); result valid in thread 0.  `scratch` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  if (w == 0) {
    double t = lane < nw ? scratch[lane] : 0.0;
    t = warp_sum(t);
    v = t;
  }
  return v;
}

// ----------------------------------------------------------------------------------------------
// Host helpers (gpb_tmap.cu)
// ----------------------------------------------------------------------------------------------
// Encode a 2-D fp64 row-major tensor map: `rows` x `cols` view at `base` with leading dimension `ld`
// (elements), box = box_rows x 16 columns (128 bytes, SWIZZLE_128B), out-of-bounds elements read as 0.
int make_tmap_f64(CUtensorMap* out, const double* base, long rows, long cols, long ld, int box_rows);
// Encode the int8 slice buffer of the sliced GEMM (`rows` rows of `slices` x k bytes, slice-major inside a row) as a 3-D
// map (k, slice, row); box = box_rows rows x box_k bytes of ONE slice, swizzled by box_k (32, 64 or 128 bytes), k beyond
// the slice and rows beyond `rows` read as 0.
int make_tmap_i8_slices(CUtensorMap* out, const int8_t* base, long rows, int k, int slices, int box_k, int box_rows);

}  // namespace gpb
