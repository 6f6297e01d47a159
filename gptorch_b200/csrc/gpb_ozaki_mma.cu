// gpb_ozaki_mma.cu -- the int8-sliced FP64-equivalent product C = beta C + alpha A B^T (DESIGN.md section 8) as ONE
// tcgen05 kernel: all weight-class sums of a 128 x BN output tile accumulate in tensor memory, and the epilogue
// recombines them in fp64.  Operands are the slice buffers of oz_split_kernel / oz_split_t_kernel (gpb_ozaki.cu), both
// in the forward layout (slice s of a row at byte offset s k), with one power-of-two scale per row.
//
// Class u = s + t collects the products Q^A_s (Q^B_t)^T.  The B slices of one k-chunk lie in shared memory one after the
// other (slice-major, BN rows each), so A_s times B slices t0 .. t0 + nt - 1 is a single MMA of N = BN nt whose output
// columns are exactly the accumulators of the classes s + t0 .. s + t0 + nt - 1 (class u at TMEM columns BN u ..
// BN u + BN - 1).  Classes u >= S are never formed.  The S classes of a 64-column tile fill the 512 TMEM columns at S = 8,
// so S <= 8 uses BN = 64 and S = 9 (the blocked inverse's products, gpb_chol.cu) BN = 48.  For S = 8 one k-step of 32
// bytes is 12 MMAs (N <= 256) instead of 36 of N = 64, and reads A once per MMA: 120 KB of shared memory per 9.4 M MAC,
// inside the 128 B/clk an SM can deliver.  For S = 9 it is 13 MMAs (N <= 240): 120 KB per 8.8 M MAC.
//
// A narrow tile reloads the same 128 A rows for every BN output columns, and A is most of the operand bytes (S = 9:
// 36.9 KB of A and 13.8 KB of B per 32-byte k-step).  So CTAs run in clusters of two that take neighbouring tiles of one
// tile row: each loads its own B slices and half of the A slices, the latter multicast into both CTAs' shared memory,
// which halves the A traffic out of L2.  Both CTAs of a pair run the same k loop over the union of their two k-ranges
// (a 48-column pair can straddle two 128-blocks; the split wrote zeros in the triangular operands' zero blocks, so the
// extra k-steps add zero to the exact sums).
//
// The int32 class sums are exact ((u + 1) k 4096 < 2^31, checked by the driver), and the epilogue runs the operation
// sequence of oz_recombine_kernel (Horner from class S-1 down, then (alpha sa_i 2^-14) sb_j t, then beta C + val), so the
// result is bitwise the one of the unfused library engine.
//
// Roles (192 threads): warp 0 issues the TMA loads into a ring of stages, warp 1 allocates TMEM and one lane issues the
// MMAs (tcgen05.commit releases each stage in both CTAs of the pair and finally signals the epilogue), warps 2-5 read the
// class planes with tcgen05.ld (warp w owns TMEM lanes 32 (w % 4) ..) and write C.
#include "gpb_common.cuh"
#include "gpb_ozaki.cuh"
#include <algorithm>

namespace gpb {

namespace {

constexpr int I8_BM = 128;
constexpr int I8_CH = 64;                          // k bytes per stage and slice (SWIZZLE_64B rows)
constexpr int I8_RING_BYTES = 198 * 1024;          // shared memory given to the stage ring (two stages at S = 9)
constexpr int I8_THREADS = 192;

struct I8Params {
  int m, n, k;
  double alpha, beta;
  const double* sa;
  const double* sb;
  double* C;
  long ldc;
  int lower, gi0;
  double* Cdiag;
  int a_trans, a_tri, a_row0, a_col0;
  int b_trans, b_tri, b_row0, b_col0;
  int tiles_m, tiles_n, pairs_n;
};

// tile width: the S class accumulators of BN columns each must fit the 512 TMEM columns (S = 9: 432 of them)
constexpr int i8_bn(int S) { return S <= 8 ? 64 : 48; }

template <int S, int BN>
struct I8Cfg {
  static_assert(S * BN <= 512, "the class accumulators exceed tensor memory");
  static constexpr int A_BYTES = S * I8_BM * I8_CH;
  static constexpr int B_BYTES = S * BN * I8_CH;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = std::min(8, I8_RING_BYTES / STAGE_BYTES);
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256;
  static_assert(STAGES >= 2 && SMEM_BYTES <= 227 * 1024, "the stage ring needs two stages in shared memory");
  static constexpr int TMEM_COLS = S * BN <= 256 ? 256 : 512;
  static constexpr int MAX_NT = 256 / BN;         // B slices per MMA (N <= 256)
  // tile rows visited together, pair column by pair column: the ~74 resident pairs share GROUP A blocks of 128 rows
  // and 74 / GROUP B blocks of 2 BN rows, streamed through L2.
  static constexpr int GROUP = BN == 64 ? 16 : 4;
};

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
      "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
      : "memory");
}

// The same box written to the same shared-memory offset in both CTAs of the pair; each CTA's barrier at `bar`'s offset
// receives the bytes.
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
      " [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(dst),
      "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
      : "memory");
}

// K-major operand tile with 64-byte rows and the 64-byte swizzle: 8-row groups 512 bytes apart (SBO), LBO unused.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>(1) << 16) |
         (static_cast<uint64_t>((8 * I8_CH) >> 4) << 32) | (static_cast<uint64_t>(1) << 46) | (static_cast<uint64_t>(4) << 61);
}

// kind::i8 instruction descriptor: s32 accumulator, signed A and B, both K-major, M = 128.
__host__ __device__ constexpr uint32_t i8_idesc(int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(I8_BM >> 4) << 24);
}

__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc));
}

__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Arrives on the barrier at `bar`'s offset in both CTAs of the pair once this CTA's MMAs so far have completed.
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)), "h"(static_cast<uint16_t>(3))
               : "memory");
}

__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}

template <int S, int BN = i8_bn(S)>
__global__ void __launch_bounds__(I8_THREADS, 1)
oz_mma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const I8Params p) {
  using Cfg = I8Cfg<S, BN>;
  constexpr int STAGES = Cfg::STAGES;

  // ---- tile: cluster c is tile row tm and pair column pc, CTA rank r takes tile column 2 pc + r.  Pairs go in groups
  // of Cfg::GROUP tile rows, pair column by pair column inside a group ----------------------------------------------
  const uint32_t rank = cluster_ctarank();
  int tm, pc;
  {
    const int c = blockIdx.x >> 1;
    const int per_group = Cfg::GROUP * p.pairs_n;
    const int g = c / per_group;
    const int first = g * Cfg::GROUP;
    const int rows = min(Cfg::GROUP, p.tiles_m - first);
    const int l = c - g * per_group;
    tm = first + l % rows;
    pc = l / rows;
  }
  const int tn = 2 * pc + static_cast<int>(rank);
  const bool phantom = tn >= p.tiles_n;                        // odd tiles_n: the last pair's second tile stores nothing
  const int m0 = tm * I8_BM, n0 = tn * BN;
  const int m_last = min(m0 + I8_BM, p.m) - 1;
  // the pair's columns: the k range and the early return below are the pair's, so that both CTAs take them alike
  const int pn0 = 2 * pc * BN, pn_last = min(pn0 + 2 * BN, p.n) - 1;
  if (p.lower && (pn0 >> 7) > ((p.gi0 + m_last) >> 7)) return;        // every column right of every row's diagonal block

  // ---- k range: the triangular-by-blocks operands are zero outside it (the split wrote zeros there) -------------
  int k_lo = 0, k_hi = p.k;
  if (p.a_tri) {
    if (p.a_trans) k_hi = min(k_hi, ((p.a_col0 + m_last) / NB + 1) * NB - p.a_row0);
    else k_lo = max(k_lo, ((p.a_row0 + m0) / NB) * NB - p.a_col0);
  }
  if (p.b_tri) {
    if (p.b_trans) k_hi = min(k_hi, ((p.b_col0 + pn_last) / NB + 1) * NB - p.b_row0);
    else k_lo = max(k_lo, ((p.b_row0 + pn0) / NB) * NB - p.b_col0);
  }
  k_lo &= ~(I8_CH - 1);
  const int nk = k_hi > k_lo ? (k_hi - k_lo + I8_CH - 1) / I8_CH : 0;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_al + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* acc_bar = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 2);                            // released by the MMAs of both CTAs
    }
    mbar_init(acc_bar, 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(Cfg::TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync();                                              // the peer's barriers are initialised before any load
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // =============================== TMA producer ==============================================
    if (lane == 0) {
      tma_prefetch_desc(&mapA);
      tma_prefetch_desc(&mapB);
      // a stage is refilled once both CTAs' MMAs have released it: this CTA writes A into the peer's copy too
      for (int it = 0; it < nk; ++it) {
        const int s = it % STAGES;
        mbar_wait(&empty_bar[s], ((it / STAGES) & 1) ^ 1u);
        mbar_expect_tx(&full_bar[s], phantom ? Cfg::A_BYTES : Cfg::STAGE_BYTES);
        const uint32_t a_dst = smem_base + s * Cfg::STAGE_BYTES, b_dst = a_dst + Cfg::A_BYTES;
        const int kx = k_lo + it * I8_CH;
#pragma unroll
        for (int q = static_cast<int>(rank); q < S; q += 2)
          tma_load_3d_pair(a_dst + q * (I8_BM * I8_CH), &mapA, kx, q, m0, &full_bar[s]);
        if (!phantom) {
#pragma unroll
          for (int q = 0; q < S; ++q) tma_load_3d(b_dst + q * (BN * I8_CH), &mapB, kx, q, n0, &full_bar[s]);
        }
      }
      // wait for the last releases of every stage: after this no arrival from the peer is still in flight to this CTA
      for (int it = nk; it < nk + STAGES; ++it) mbar_wait(&empty_bar[it % STAGES], ((it / STAGES) & 1) ^ 1u);
    }
  } else if (warp == 1) {
    // =============================== MMA issue ================================================
    if (lane == 0 && nk > 0) {
      for (int it = 0; it < nk; ++it) {
        const int s = it % STAGES;
        mbar_wait(&full_bar[s], (it / STAGES) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t a_base = smem_base + s * Cfg::STAGE_BYTES, b_base = a_base + Cfg::A_BYTES;
#pragma unroll
        for (int kk = 0; kk < I8_CH / 32; ++kk) {
#pragma unroll
          for (int sa = 0; sa < S; ++sa) {
#pragma unroll
            for (int t0 = 0; t0 < S - sa; t0 += Cfg::MAX_NT) {
              const int nt = min(Cfg::MAX_NT, S - sa - t0);
              const uint64_t ad = smem_desc(a_base + sa * (I8_BM * I8_CH) + kk * 32);
              const uint64_t bd = smem_desc(b_base + t0 * (BN * I8_CH) + kk * 32);
              const uint32_t acc = (it > 0 || kk > 0 || sa > 0) ? 1u : 0u;   // sa = 0 covers every class first
              mma_i8(tmem + static_cast<uint32_t>((sa + t0) * BN), ad, bd, i8_idesc(nt * BN), acc);
            }
          }
        }
        mma_commit_pair(&empty_bar[s]);
      }
      mma_commit(acc_bar);
    }
  } else {
    // =============================== epilogue =================================================
    const int quarter = warp & 3;
    const int i = m0 + 32 * quarter + lane;
    const bool row_ok = i < p.m;
    const uint32_t t_row = tmem + (static_cast<uint32_t>(32 * quarter) << 16);
    const int gi = p.gi0 + i;
    // where the 8 columns from n0 + c0 go (nullptr: not stored).  They lie in one 128-block: gpb_potri_lower's diagonal
    // blocks go to Cdiag ([row][NB]), the blocks right of the diagonal nowhere.
    auto dest = [&](int c0) -> double* {
      const int j = n0 + c0;
      if (!row_ok || j >= p.n || (p.lower && (j >> 7) > (gi >> 7))) return nullptr;
      if (p.Cdiag != nullptr && (j >> 7) == (gi >> 7)) return p.Cdiag + static_cast<long>(gi) * NB + (j & (NB - 1));
      return p.C + static_cast<long>(i) * p.ldc + j;
    };
    if (nk > 0) {
      mbar_wait(acc_bar, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    const double down = 1.0 / static_cast<double>(1 << 7);
    const double si = row_ok ? p.alpha * p.sa[i] * (down * down) : 0.0;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 8) {
      uint32_t v[S][8];
      __syncwarp();
      if (nk > 0) {
#pragma unroll
        for (int u = 0; u < S; ++u) tmem_ld_x8(t_row + static_cast<uint32_t>(u * BN + c0), v[u]);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      } else {
#pragma unroll
        for (int u = 0; u < S; ++u)
#pragma unroll
          for (int q = 0; q < 8; ++q) v[u][q] = 0u;
      }
      const int j = n0 + c0;
      if (double* c = dest(c0)) {
        double t[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) t[q] = 0.0;
#pragma unroll
        for (int u = S - 1; u >= 0; --u)                              // Horner from the smallest weight class up
#pragma unroll
          for (int q = 0; q < 8; ++q) t[q] = t[q] * down + static_cast<double>(static_cast<int32_t>(v[u][q]));
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (j + q < p.n) {
            const double val = (si * p.sb[j + q]) * t[q];
            c[q] = p.beta == 0.0 ? val : p.beta * c[q] + val;
          }
        }
      }
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  cluster_sync();                                              // no CTA leaves while its peer may still signal it
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(Cfg::TMEM_COLS));
  }
}

template <int S>
int launch_s(const CUtensorMap& mapA, const CUtensorMap& mapB, const I8Params& p, cudaStream_t stream) {
  using Cfg = I8Cfg<S, i8_bn(S)>;
  static std::atomic<int> smem_state[GPB_MAX_DEVICES];
  if (int rc = ensure_dynamic_smem(oz_mma_kernel<S>, Cfg::SMEM_BYTES, smem_state)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(2L * p.tiles_m * p.pairs_n));
  cfg.blockDim = dim3(I8_THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  GPB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, oz_mma_kernel<S>, mapA, mapB, p));
  count_launch();
  GPB_CUDA_CHECK(cudaGetLastError());
  return GPB_OK;
}

}  // namespace

int ozaki_mma_launch(const OzEx& x, const int8_t* a8, const int8_t* b8, const double* sa, const double* sb) {
  const int S = x.slices;
  if (S < 2 || S > OZ_MMA_MAX_TILE_SLICES) return GPB_ERR_UNSUPPORTED;
  const int bn = i8_bn(S);
  CUtensorMap mapA, mapB;
  int rc = make_tmap_i8_slices(&mapA, a8, x.m, x.k, S, I8_CH, I8_BM);
  if (rc) return rc;
  rc = make_tmap_i8_slices(&mapB, b8, x.n, x.k, S, I8_CH, bn);
  if (rc) return rc;
  I8Params p;
  p.m = x.m; p.n = x.n; p.k = x.k;
  p.alpha = x.alpha; p.beta = x.beta;
  p.sa = sa; p.sb = sb;
  p.C = x.C; p.ldc = x.ldc;
  p.lower = x.lower; p.gi0 = x.gi0; p.Cdiag = x.Cdiag;
  p.a_trans = x.a_trans; p.a_tri = x.a_tri; p.a_row0 = x.a_row0; p.a_col0 = x.a_col0;
  p.b_trans = x.b_trans; p.b_tri = x.b_tri; p.b_row0 = x.b_row0; p.b_col0 = x.b_col0;
  p.tiles_m = (x.m + I8_BM - 1) / I8_BM;
  p.tiles_n = (x.n + bn - 1) / bn;
  p.pairs_n = (p.tiles_n + 1) / 2;
  switch (S) {
    case 2: return launch_s<2>(mapA, mapB, p, x.stream);
    case 3: return launch_s<3>(mapA, mapB, p, x.stream);
    case 4: return launch_s<4>(mapA, mapB, p, x.stream);
    case 5: return launch_s<5>(mapA, mapB, p, x.stream);
    case 6: return launch_s<6>(mapA, mapB, p, x.stream);
    case 7: return launch_s<7>(mapA, mapB, p, x.stream);
    case 8: return launch_s<8>(mapA, mapB, p, x.stream);
    case 9: return launch_s<9>(mapA, mapB, p, x.stream);
  }
  return GPB_ERR_UNSUPPORTED;
}

}  // namespace gpb
