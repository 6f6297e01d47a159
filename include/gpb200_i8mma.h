/* gpb200_i8mma.h -- switch of libgpb200.so's fused int8-sliced product engine (DESIGN.md section 8).
 *
 * A companion of gpb200.h with the same conventions.  The large trailing updates of gpb_potrf_lower run by default as
 * FP64-equivalent products on the INT8 tensor path: every row is cut into `slices` signed 7-bit digits relative to its
 * own power-of-two scale and one tcgen05 kernel forms every digit product and recombines it in fp64.  While the engine
 * is on, the large products of gpb_potri_lower and gpb_trtri_upper run on it too, at a fixed 9 slices (orders that are
 * a multiple of 16).  gpb_gemm_ozaki_nt reaches the same kernel with 2..8 slices.  While gpb_ozaki_config (gpb200.h) is
 * above 0 the library engine takes precedence.  Available from gpb_version() >= 103; the sliced inverse from 104.
 */
#ifndef GPB200_I8MMA_H_
#define GPB200_I8MMA_H_

#include "gpb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Number of slices of the fused engine: 2..8, or 0 for the FP64 DMMA engine; 1 and values above 8 select the default,
 * 8 slices.  The initial value comes from the environment variable GPB_I8MMA (default 8).  0 also returns the blocked
 * inverse to the FP64 DMMA engine.  slices < 0 only queries.  Returns the previous value.  Setting 0 returns the
 * engine's device workspaces. */
int gpb_i8mma_config(int slices);

#ifdef __cplusplus
}
#endif
#endif /* GPB200_I8MMA_H_ */
