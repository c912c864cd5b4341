// Shared device helpers: unfused IEEE arithmetic, bulk asynchronous copies, warp/block reductions.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/glimpse_b200.h"

#define GB_MAX_OBS 8
#define GB_XCH 36 /* doubles per slot of a block reduction (28 moment sums at most) */
// histogram bins the 110 / 224 KB launch choice of large templates assumes (uint8 frames of up to 4 bands: 1021 bins)
#define GB_MAX_BINS 1024
// bands of a frame, and the grey levels of a uint8 frame with that many (its band sums 0 .. 255 * bands)
#define GB_MAX_BANDS 8
#define GB_MAX_U8_BINS (255 * GB_MAX_BANDS + 1)
// Templates up to this many pixels keep their high-passed copy and CDF tables in shared memory next to the search window;
// larger ones (GB_PLAN_LARGE_TEMPLATES, up to GB_MAX_TEMPLATE_SIDE a side) are read from global memory.
#define GB_SMEM_TEMPLATE 1024
#define GB_MAX_TEMPLATE_SIDE 128

// particle flag bits, in the order the reference would raise (tracker.py:106-119, observer.py:201,
// raster.py:961-973)
#define GB_F_VIEW_OOB 1u
#define GB_F_NOT_VISIBLE 2u
#define GB_F_NAN 4u
#define GB_F_SAMPLE_OUTSIDE 8u
#define GB_F_DEM_OOB 16u
#define GB_F_WINDOW 32u
#define GB_F_TEMPLATE 64u
#define GB_F_EVOLVE_OOB 128u /* a tangent model sampled its DEM out of bounds while evolving (before the particle tests) */

namespace gb {

// NumPy evaluates element-wise expressions one rounded operation at a time; these keep nvcc from
// contracting a*b+c into an FMA where bit-faithfulness to the reference is cheap to keep.
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double quo(double a, double b) { return __ddiv_rn(a, b); }

__device__ __forceinline__ double shfl_down(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
__device__ __forceinline__ double shfl_up(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
__device__ __forceinline__ double shfl_xor(double v, int d) { return __shfl_xor_sync(0xffffffffu, v, d); }

// ---------------------------------------------------------------------------------------------
// Bulk asynchronous copies global -> shared (the TMA engine's 1-D mode: `cp.async.bulk`, SASS UBLKCP)
// completing on an mbarrier.  Sizes are multiples of 16 bytes, both addresses 16-byte aligned.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_global, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(__cvta_generic_to_global(src_global)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 2-D tile of a tensor described by a CUtensorMap (the TMA engine's tiled mode: `cp.async.bulk.tensor.2d`, SASS UTMALDG):
// the box of the map whose first element is (x, y) lands densely in shared memory (128-byte aligned), out-of-range elements
// as zeros, and completes on the mbarrier with the box's full byte count.
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const void* tmap, int x, int y, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// Message passing between CTAs without the sequentially consistent fence of __threadfence() (which also
// invalidates the SM's L1): the producer's atomic carries release semantics at GPU scope, the consumer reads
// the published data with GPU-scope loads (served by L2).
__device__ __forceinline__ int atomic_add_release_gpu(int* p, int v) {
  int old;
  asm volatile("atom.add.release.gpu.global.s32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ double load_relaxed_gpu(const double* p) {
  double v;
  asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += shfl_xor(v, d);
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmin(v, shfl_xor(v, d));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmax(v, shfl_xor(v, d));
  return v;
}

// Work area of the block reductions of k_init / k_moments (dynamic shared memory).
struct SmemHeader {
  double red[32][GB_XCH];  // per-warp partials of a block reduction
  double bcast[GB_XCH];    // block-wide broadcast values
  int iflags[4];
};

// Bitwise OR of one word per thread across the CTA (__syncthreads_or only tells whether any is non-zero).
// `slot` is one shared-memory word owned by the caller.
__device__ __forceinline__ unsigned block_or(unsigned v, unsigned* slot) {
  if (threadIdx.x == 0) *slot = 0u;
  __syncthreads();
  v = __reduce_or_sync(0xffffffffu, v);
  if ((threadIdx.x & 31) == 0 && v) atomicOr(slot, v);
  __syncthreads();
  const unsigned out = *slot;
  __syncthreads();
  return out;
}

// Block reduction of K per-thread doubles (OP 0: sum, 1: min); the result is left in
// hdr->bcast[0..K), visible to all threads on return.  Maxima are reduced as minima of negatives.
// Stage 1: shuffles inside each warp; stage 2: warp k combines the per-warp partials of value k.
template <int K, int OP>
__device__ __forceinline__ void block_reduce(double (&v)[K], SmemHeader* hdr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const double x = OP == 0 ? warp_sum(v[k]) : warp_min(v[k]);
    if (lane == 0) hdr->red[warp][k] = x;
  }
  __syncthreads();
  for (int k = warp; k < K; k += nwarp) {
    double x = lane < nwarp ? hdr->red[lane][k] : (OP == 0 ? 0.0 : CUDART_INF);
    x = OP == 0 ? warp_sum(x) : warp_min(x);
    if (lane == 0) hdr->bcast[k] = x;
  }
  __syncthreads();
}

}  // namespace gb
