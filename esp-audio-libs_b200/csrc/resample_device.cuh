// Device-side helpers shared by the resampler kernels (resample_kernel.cu, resample_ni_kernel.cu): mbarrier /
// TMA / cp.async wrappers, the packed-FP32 multiply-add, tile constants.  Internal.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.hpp"
#include "kernels.hpp"

namespace espb {
namespace {

constexpr int NB = kOutputsPerBlock;  // 8
constexpr int SGN = kSeriesPerRow;    // 128
constexpr uint32_t kPassDone = 1u << 9;  // rtab flag next to r0 (bits 0-3), r1 (4-7)
constexpr int RG = 4;  // rows per skip group / inner unroll

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(a),
      "r"(parity)
      : "memory");
}
// TMA bulk copy global -> shared, completion counted on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void cp_async_16(void *dst_smem, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// Shared-memory tile of `rows` x 128 series for the layout stages (caller layout <-> time-major).  The 16-byte units
// of a row are XOR-permuted by a function of the row: the time-major side moves whole units (one conflict-free
// LDS.128 / STS.128 per lane: consecutive lanes, consecutive units of one row), the stream-major side — consecutive
// frames of one stream, i.e. consecutive rows of one column — spreads over the banks because rows 4m + i map m and i
// into different bits of the permutation.  8 shared-memory wavefronts per 512 bytes moved instead of the 24 of the
// padded scalar tile (pitch 129: two-way conflicts on the scalar stores, four scalar loads per 128-bit store).
struct SwzTile {
  float *p;
  __device__ __forceinline__ static int unit(int row, int u) { return u ^ (((row >> 2) ^ ((row & 3) << 3)) & 31); }
  __device__ __forceinline__ float &at(int row, int col) const {
    return p[row * kSeriesPerRow + (unit(row, col >> 2) << 2) + (col & 3)];
  }
  __device__ __forceinline__ float4 &vec(int row, int u) const {
    return *reinterpret_cast<float4 *>(p + row * kSeriesPerRow + (unit(row, u) << 2));
  }
};

// ---- staging overlap (DESIGN.md §4.5): the resampler is launched as a programmatic dependent of the transposing
// kernel and starts while that kernel is still filling xt; a CTA waits for the row tiles it reads on per-tile
// counters the transposing CTAs bump (release) after their stores.
__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// generic-proxy writes (made visible by the acquire above) -> async-proxy reads (the TMA bulk copies of xt)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;\n" ::: "memory"); }
// primary side: dependants may be scheduled as soon as every CTA of this grid has got here
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }

// L2 eviction-priority policies (createpolicy) and accesses that carry one
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;\n" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ld_global_hint(const float4 *p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;\n"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ void st_global_hint(float4 *p, float4 v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;\n" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w), "l"(pol)
               : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s_hint(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar,
                                                  uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;\n" ::"r"(
          smem_u32(dst_smem)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
      : "memory");
}

// Counting arrival on a shared-memory word.  Relaxed is enough: every shared-memory load of the stage
// has already returned its value (the FMAs consumed them) when the warp gets here, so nothing of this
// warp can still observe the refill; the refill itself is published by the mbarrier arrive (release).
__device__ __forceinline__ int smem_arrive(int *counter) {
  int old;
  asm volatile("atom.relaxed.cta.shared::cta.add.s32 %0, [%1], 1;\n" : "=r"(old) : "r"(smem_u32(counter)) : "memory");
  return old;
}

// Packed FP32 pairs (Blackwell FFMA2): two independent IEEE FMAs per lane per instruction — the same
// results as two scalar FFMAs, half the issue slots.  A pair is (filter 0, filter 1) of one output, whose
// coefficients are adjacent in G.
// Fast mode only: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (unlike the scalar forms, whose
// explicit .rn is honoured), so exact mode keeps scalar FMUL + FADD.
__device__ __forceinline__ float2 fma2(float2 g, float x, float2 acc) {
  return __ffma2_rn(g, make_float2(x, x), acc);  // SASS: FFMA2 acc, g.F32x2, x.F32 (scalar broadcast), acc
}

template <bool EXACT>
__device__ __forceinline__ float mac(float g, float x, float acc) {
  if (EXACT)
    return __fadd_rn(acc, __fmul_rn(g, x));  // dsps_dotprod_f32_ansi.c:20 — separate multiply and add
  return __fmaf_rn(g, x, acc);
}

}  // namespace
}  // namespace espb
