// art_biquad on the device: Direct-Form-I sections, sequential in time, one thread per series
// (stream x channel), thousands of series in flight.
//
// Reference: src/resample/art_biquad.cpp:73-93 (biquad_apply_buffer) — the sum
//   x*a0 + in_d1*a1 + in_d2*a2 - b1*out_d1 - b2*out_d2
// is evaluated left to right with every product and sum rounded (no FMA): contraction moves the
// result by up to 1.8e-6 (SURVEY.md §8a R8), so only __fmul_rn/__fadd_rn/__fsub_rn are used.
// Cascaded sections are applied per sample instead of as separate buffer passes; the arithmetic
// per section is unchanged, so the result is bit-identical.
//
// Data movement.  The recurrence is latency-bound (~12 cycles per section per sample) and cannot
// be parallelised in time without changing the arithmetic, so everything else must stay off its
// critical path.  The kernel works on the time-major layout  buf[group][row][128 series]  (the
// resampler's own staging layout): a CTA of 128 threads owns a group, 32-row chunks (16 KB,
// contiguous) are streamed through a 4-stage shared-memory ring by TMA bulk loads, filtered in
// place by the thread that owns the column, and written back by TMA bulk stores — HBM sees only
// full 16 KB transfers, the threads only conflict-free LDS/STS.
//
// Long single streams (few series, many rows) run in time blocks (blockIdx.y): block k filters rows
// [k*L, (k+1)*L) after re-running the recurrence over the W rows before it from a zero state ("warm-up"),
// out of place.  Once the two trajectories (true state vs zero start) have rounded to the same two
// consecutive outputs they stay bit-identical; measured on the CPU oracle this happens within 64 rows for
// pole radius 0.49, 256 for 0.77, 4096 for 0.92, and never for 0.98.  That merge is an empirical event, so it
// is VERIFIED, not assumed: every block records the state it reached at its first row (after the warm-up)
// and at its end; espb_biquad_verify_kernel then walks the blocks of each series in order and compares, bit
// for bit, block k's start state with block k-1's end state.  Equal state + equal input = equal continuation,
// so an unbroken chain of equalities from block 0 (which starts from the true saved state) proves that the
// output is the sequential one.  Where the states differ the series' block is filtered again from the true
// state (sequentially, by the thread that owns the series) and the chain continues from its corrected end.
// The result is therefore the reference's (art_biquad.cpp:73-93) by construction; a failed merge only costs
// time.  The verify kernel also commits the final state (the block kernel never writes the saved state, so
// no block can read a state that another block of the same launch has already replaced).
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.hpp"
#include "kernels.hpp"
#include "pcm_device.cuh"

namespace espb {

namespace {

constexpr int SGN = kSeriesPerRow;  // 128
constexpr int RB = 32;              // rows per chunk
constexpr int BSTAGES = 4;

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store(void *dst, const void *src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}

struct Section {
  float in_d1, in_d2, out_d1, out_d2;
};

template <bool FIRST_ORDER>
__device__ __forceinline__ float section_step(Section &s, float x, const BiquadParams &c) {
  float sum = __fadd_rn(__fmul_rn(x, c.a0), __fmul_rn(s.in_d1, c.a1));
  if (!FIRST_ORDER)
    sum = __fadd_rn(sum, __fmul_rn(s.in_d2, c.a2));
  sum = __fsub_rn(sum, __fmul_rn(c.b1, s.out_d1));
  if (!FIRST_ORDER)
    sum = __fsub_rn(sum, __fmul_rn(c.b2, s.out_d2));
  s.out_d2 = s.out_d1;
  s.out_d1 = sum;
  s.in_d2 = s.in_d1;
  s.in_d1 = x;
  return sum;
}

// src/dst: first group of the launch (may be the same buffer when there is one time block); rows
// [row_first, row_first + n_rows) of every group are filtered.  blk_first + blockIdx.y = time block of block_rows rows
// (0 = all rows in one block) preceded by warm_rows rows of warm-up; n_blocks = time blocks of the whole call.
template <int NSEC, bool FIRST_ORDER>
__global__ void __launch_bounds__(SGN)
    espb_biquad_tm_kernel(const float *src, float *dst, int64_t rows_cap, int row_first, int n_rows, BiquadParams c,
                          float *__restrict__ state, int n_series, int block_rows, int warm_rows,
                          float4 *__restrict__ blk_state, int blk_first, int n_blocks) {
  extern __shared__ __align__(128) unsigned char bq_smem[];
  float (*ring)[RB][SGN] = reinterpret_cast<float (*)[RB][SGN]>(bq_smem);  // [BSTAGES][RB][SGN]
  uint64_t *full = reinterpret_cast<uint64_t *>(bq_smem + sizeof(float) * BSTAGES * RB * SGN);
  const int tid = threadIdx.x;
  const int q = blockIdx.x * SGN + tid;
  // this CTA's time block: rows [blk_lo, blk_hi), started warm_rows earlier (block 0 starts from the saved state)
  const int blk = blk_first + blockIdx.y;
  const int blk_lo = block_rows > 0 ? blk * block_rows : 0;
  const int blk_hi = (block_rows > 0 && blk_lo + block_rows < n_rows) ? blk_lo + block_rows : n_rows;
  const int run_lo = (blk == 0 || blk_lo < warm_rows) ? 0 : blk_lo - warm_rows;
  const bool from_saved_state = (run_lo == 0);
  const bool last_block = (blk_hi == n_rows);
  const float *gsrc = src + ((int64_t) blockIdx.x * rows_cap + row_first + run_lo) * SGN;
  float *gdst = dst + ((int64_t) blockIdx.x * rows_cap + row_first + run_lo) * SGN;
  const int run_rows = blk_hi - run_lo;
  const int n_chunks = (run_rows + RB - 1) / RB;
  const int first_store_chunk = (blk_lo - run_lo) / RB;  // warm-up chunks are filtered but not written

  Section sec[NSEC];
  if (q < n_series && from_saved_state) {
#pragma unroll
    for (int k = 0; k < NSEC; ++k) {
      const float4 v = *reinterpret_cast<const float4 *>(state + ((int64_t) q * NSEC + k) * 4);
      sec[k].in_d1 = v.x;
      sec[k].in_d2 = v.y;
      sec[k].out_d1 = v.z;
      sec[k].out_d2 = v.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < NSEC; ++k)
      sec[k].in_d1 = sec[k].in_d2 = sec[k].out_d1 = sec[k].out_d2 = 0.0f;
  }

  auto chunk_rows = [&](int k) { return (k + 1) * RB <= run_rows ? RB : run_rows - k * RB; };
  auto load_chunk = [&](int k) {
    const int st = k % BSTAGES;
    const uint32_t bytes = (uint32_t) chunk_rows(k) * SGN * sizeof(float);
    mbar_expect_tx(&full[st], bytes);
    tma_load(&ring[st][0][0], gsrc + (int64_t) k * RB * SGN, bytes, &full[st]);
  };

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < BSTAGES; ++s)
      mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    for (int k = 0; k < BSTAGES - 1 && k < n_chunks; ++k)
      load_chunk(k);
  }
  __syncthreads();

  // time-block mode: (start, end) state of block `blk` of this thread's series, for the verify kernel (indexed by the
  // call's block count: a launch may cover only a slice of the blocks)
  float4 *rec = blk_state ? blk_state + (((size_t) blockIdx.x * n_blocks + blk) * NSEC * 2) * SGN + tid : nullptr;
  for (int k = 0; k < n_chunks; ++k) {
    const int st = k % BSTAGES;
    const int rows = chunk_rows(k);
    if (rec && k == first_store_chunk) {
#pragma unroll
      for (int s = 0; s < NSEC; ++s)
        rec[(s * 2) * SGN] = make_float4(sec[s].in_d1, sec[s].in_d2, sec[s].out_d1, sec[s].out_d2);
    }
    mbar_wait(&full[st], (uint32_t) ((k / BSTAGES) & 1));
    float *col = &ring[st][0][tid];
    if (rows == RB) {
#pragma unroll 8
      for (int r = 0; r < RB; ++r) {
        float v = col[r * SGN];
#pragma unroll
        for (int s = 0; s < NSEC; ++s)
          v = section_step<FIRST_ORDER>(sec[s], v, c);
        col[r * SGN] = v;
      }
    } else {
      for (int r = 0; r < rows; ++r) {
        float v = col[r * SGN];
#pragma unroll
        for (int s = 0; s < NSEC; ++s)
          v = section_step<FIRST_ORDER>(sec[s], v, c);
        col[r * SGN] = v;
      }
    }
    // generic-proxy writes -> visible to the async proxy, then one thread stores the chunk and refills
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      if (k >= first_store_chunk)
        tma_store(gdst + (int64_t) k * RB * SGN, &ring[st][0][0], (uint32_t) rows * SGN * sizeof(float));
      asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");  // (possibly empty) group keeps the count uniform
      if (k + BSTAGES - 1 < n_chunks) {
        // stage (k-1) % BSTAGES is reused: its store (issued last iteration) must have read shared memory
        asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");
        load_chunk(k + BSTAGES - 1);
      }
    }
  }
  if (tid == 0)
    asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");

  if (rec) {
#pragma unroll
    for (int s = 0; s < NSEC; ++s)
      rec[(s * 2 + 1) * SGN] = make_float4(sec[s].in_d1, sec[s].in_d2, sec[s].out_d1, sec[s].out_d2);
  } else if (q < n_series && last_block) {
#pragma unroll
    for (int k = 0; k < NSEC; ++k)
      *reinterpret_cast<float4 *>(state + ((int64_t) q * NSEC + k) * 4) =
          make_float4(sec[k].in_d1, sec[k].in_d2, sec[k].out_d1, sec[k].out_d2);
  }
}

// ---------------------------------------------------------------------------------
// Post-filter + float_to_quantized in ONE pass for mono streams (Resampler::resample's tail, resampler.cpp:142-153:
// biquad_apply_buffer, then float_to_quantized).  For a mono stream the 32 rows of a chunk are 32 consecutive samples
// of the series' own output row, so the chunk can leave as packed PCM straight from the ring: one read of 4 bytes
// and one write of NBYTES bytes per sample instead of 4 + 4 (filter in place) + 4 + NBYTES (quantising layout stage).
// The recurrence is latency-bound with one warp per scheduler, so the quantisation must not sit in its instruction
// stream (a first version in which the filtering thread quantised its own results ran 1.95 ms for the two stages'
// 2.14): the CTA is warp-specialised — warps 0-3 filter in place exactly like espb_biquad_tm_kernel, warps 4-11 take
// each filtered chunk from shared memory, quantise (quantization_utils.cpp:50-94, branch-free), pack 16 samples per
// thread and store them with 128-bit stores, then hand the stage back for the next TMA load.  Hand-overs are named
// barriers (filter: bar.arrive, packer: bar.sync).  Full 32-row chunks only; the rows of the last partial chunk are
// written back as filtered floats for the generic tail path.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;\n" ::"r"(id), "r"(count) : "memory");
}

constexpr int BQP_THREADS = 3 * SGN;  // 4 filter warps + 8 packer warps (16 rows of a series per packer thread)
template <int NSEC, bool FIRST_ORDER, int NBYTES, bool BITS32>
__global__ void __launch_bounds__(BQP_THREADS)
    espb_biquad_tm_pcm_kernel(float *buf, int64_t rows_cap, int row_first, int n_rows, BiquadParams c,
                              float *__restrict__ state, int n_series, uint8_t *__restrict__ out, int64_t out_row_bytes,
                              F2QConst qc, uint32_t *__restrict__ clipped_per_stream) {
  extern __shared__ __align__(128) unsigned char bq_smem[];
  float (*ring)[RB][SGN] = reinterpret_cast<float (*)[RB][SGN]>(bq_smem);  // [BSTAGES][RB][SGN]
  uint64_t *full = reinterpret_cast<uint64_t *>(bq_smem + sizeof(float) * BSTAGES * RB * SGN);
  const bool packer = threadIdx.x >= SGN;
  const int tid = threadIdx.x & (SGN - 1);
  const int q = blockIdx.x * SGN + tid;  // series = stream (mono)
  float *gbuf = buf + ((int64_t) blockIdx.x * rows_cap + row_first) * SGN;
  const int n_chunks = (n_rows + RB - 1) / RB;
  auto chunk_rows = [&](int k) { return (k + 1) * RB <= n_rows ? RB : n_rows - k * RB; };
  auto load_chunk = [&](int k) {
    const int st = k % BSTAGES;
    const uint32_t bytes = (uint32_t) chunk_rows(k) * SGN * sizeof(float);
    mbar_expect_tx(&full[st], bytes);
    tma_load(&ring[st][0][0], gbuf + (int64_t) k * RB * SGN, bytes, &full[st]);
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < BSTAGES; ++s)
      mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    for (int k = 0; k < BSTAGES && k < n_chunks; ++k)
      load_chunk(k);
  }
  __syncthreads();

  if (!packer) {
    // ---- filter warps: espb_biquad_tm_kernel's loop, in place in the ring
    Section sec[NSEC];
#pragma unroll
    for (int k = 0; k < NSEC; ++k) {
      float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (q < n_series)
        v = *reinterpret_cast<const float4 *>(state + ((int64_t) q * NSEC + k) * 4);
      sec[k].in_d1 = v.x, sec[k].in_d2 = v.y, sec[k].out_d1 = v.z, sec[k].out_d2 = v.w;
    }
    for (int k = 0; k < n_chunks; ++k) {
      const int st = k % BSTAGES;
      const int rows = chunk_rows(k);
      mbar_wait(&full[st], (uint32_t) ((k / BSTAGES) & 1));
      float *col = &ring[st][0][tid];
      if (rows == RB) {
#pragma unroll 8
        for (int r = 0; r < RB; ++r) {
          float v = col[r * SGN];
#pragma unroll
          for (int s = 0; s < NSEC; ++s)
            v = section_step<FIRST_ORDER>(sec[s], v, c);
          col[r * SGN] = v;
        }
        // (the stage is overwritten by a TMA load after the packers are done: order these generic-proxy writes
        //  before it, as espb_biquad_tm_kernel does before its TMA store)
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        named_bar_arrive(1 + st, BQP_THREADS);  // the chunk is filtered: over to the packers
      } else {  // the last, partial chunk: filtered floats back to the rows they came from
        for (int r = 0; r < rows; ++r) {
          float v = col[r * SGN];
#pragma unroll
          for (int s = 0; s < NSEC; ++s)
            v = section_step<FIRST_ORDER>(sec[s], v, c);
          gbuf[((int64_t) k * RB + r) * SGN + tid] = v;
        }
      }
    }
    if (q < n_series) {
#pragma unroll
      for (int k = 0; k < NSEC; ++k)
        *reinterpret_cast<float4 *>(state + ((int64_t) q * NSEC + k) * 4) =
            make_float4(sec[k].in_d1, sec[k].in_d2, sec[k].out_d1, sec[k].out_d2);
    }
  } else {
    // ---- packer warps: quantise + pack + store each filtered chunk, then refill its stage.  Two threads per series
    // (16 rows each): a chunk must be packed in less time than it takes to filter the next one, or the ring fills
    // with filtered chunks and the filter warps starve (one packer thread per series: 18 % of the samples in the
    // filter's wait for TMA data, 1.82 ms per C3 step).
    constexpr int HR = RB / 2;
    const int half = (threadIdx.x - SGN) >> 7;  // 0 / 1: rows [0, 16) / [16, 32) of the chunk
    uint32_t clipped = 0;
    uint8_t *orow = out + (int64_t) q * out_row_bytes + (int64_t) half * HR * NBYTES;
    const int n_full = n_rows / RB;
    for (int k = 0; k < n_full; ++k) {
      const int st = k % BSTAGES;
      named_bar_sync(1 + st, BQP_THREADS);
      const float *col = &ring[st][half * HR][tid];
      uint32_t w[HR / 4 * NBYTES];  // 16 samples, packed
#pragma unroll
      for (int g = 0; g < HR / 4; ++g) {
        int32_t s4[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          s4[i] = quantise_one_nb<BITS32>(col[(g * 4 + i) * SGN], qc, clipped);
        encode_words<NBYTES>(s4, w + g * NBYTES);
      }
      named_bar_sync(1 + BSTAGES, 2 * SGN);  // every packer has read the stage
      if (threadIdx.x == SGN && k + BSTAGES < n_chunks)
        load_chunk(k + BSTAGES);
      if (q < n_series) {
        uint4 *dst = reinterpret_cast<uint4 *>(orow + (int64_t) k * RB * NBYTES);
#pragma unroll
        for (int i = 0; i < HR / 16 * NBYTES; ++i)
          dst[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
      }
    }
    if (q < n_series && clipped && clipped_per_stream)
      atomicAdd(clipped_per_stream + q, clipped);
  }
}

__device__ __forceinline__ bool same_bits(const float4 &a, const float4 &b) {
  return __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y) &&
         __float_as_uint(a.z) == __float_as_uint(b.z) && __float_as_uint(a.w) == __float_as_uint(b.w);
}

// Time blocks of ONE group with few series (a single stereo or 8-channel stream: C4).  The kernel above would run one
// CTA per block with 8 of its 128 threads holding a series and move whole 512-byte rows through its ring, 15/16 of
// them padding.  Here a thread is a (block, series) pair — 128 / lanes blocks per CTA — that reads only its own
// column (the lanes of a block share one 32-byte sector per row, 16 rows of loads in flight ahead of the recurrence)
// and writes only its own results.  Same recurrence, same warm-up, same state record (so the chain check, the
// verify kernel and the repairs are shared); since nothing is staged the blocks can be shorter, which is where the
// parallelism for a single stream comes from.
template <int NSEC, bool FIRST_ORDER>
__global__ void __launch_bounds__(SGN)
    espb_biquad_tm_few_kernel(const float *__restrict__ src, float *__restrict__ dst, int row_first, int n_rows,
                              BiquadParams c, const float *__restrict__ state, int n_series, int lanes, int block_rows,
                              int warm_rows, int n_blocks, float4 *__restrict__ blk_state) {
  const int gid = blockIdx.x * SGN + threadIdx.x;
  const int blk = gid / lanes, q = gid - blk * lanes;
  if (blk >= n_blocks || q >= n_series)
    return;
  const int blk_lo = blk * block_rows;
  const int blk_hi = blk_lo + block_rows < n_rows ? blk_lo + block_rows : n_rows;
  const int run_lo = (blk == 0 || blk_lo < warm_rows) ? 0 : blk_lo - warm_rows;
  Section sec[NSEC];
#pragma unroll
  for (int k = 0; k < NSEC; ++k) {
    float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (run_lo == 0)
      v = *reinterpret_cast<const float4 *>(state + ((int64_t) q * NSEC + k) * 4);
    sec[k].in_d1 = v.x, sec[k].in_d2 = v.y, sec[k].out_d1 = v.z, sec[k].out_d2 = v.w;
  }
  const float *ps = src + (int64_t) (row_first + run_lo) * SGN + q;
  float *pd = dst + (int64_t) (row_first + run_lo) * SGN + q;
  float4 *rec = blk_state + ((size_t) blk * NSEC * 2) * SGN + q;  // (group 0)
  const int n = blk_hi - run_lo, store_from = blk_lo - run_lo;
  // batches of U rows, the next batch's loads in flight while this one runs through the recurrence (a batch of loads
  // costs ~1 us of latency, the recurrence ~24 ns per row: without the prefetch the loads were 3/4 of the time)
  constexpr int U = 32;
  float xn[U];
#pragma unroll
  for (int i = 0; i < U; ++i)
    xn[i] = i < n ? __ldg(ps + (int64_t) i * SGN) : 0.0f;
  for (int r0 = 0; r0 < n; r0 += U) {
    float x[U];
#pragma unroll
    for (int i = 0; i < U; ++i)
      x[i] = xn[i];
#pragma unroll
    for (int i = 0; i < U; ++i)
      xn[i] = r0 + U + i < n ? __ldg(ps + (int64_t) (r0 + U + i) * SGN) : 0.0f;
#pragma unroll
    for (int i = 0; i < U; ++i) {
      const int r = r0 + i;
      if (r < n) {
        if (r == store_from) {  // the state this block's own rows start from, for the chain check
#pragma unroll
          for (int s2 = 0; s2 < NSEC; ++s2)
            rec[(s2 * 2) * SGN] = make_float4(sec[s2].in_d1, sec[s2].in_d2, sec[s2].out_d1, sec[s2].out_d2);
        }
        float v = x[i];
#pragma unroll
        for (int s2 = 0; s2 < NSEC; ++s2)
          v = section_step<FIRST_ORDER>(sec[s2], v, c);
        if (r >= store_from)
          pd[(int64_t) r * SGN] = v;
      }
    }
  }
#pragma unroll
  for (int s2 = 0; s2 < NSEC; ++s2)
    rec[(s2 * 2 + 1) * SGN] = make_float4(sec[s2].in_d1, sec[s2].in_d2, sec[s2].out_d1, sec[s2].out_d2);
}

// The comparisons of the chain check do not depend on each other — only a repair does — so they run first, one
// thread per (series, block), and leave one flag per group: unbroken chains (the normal case) then cost the verify
// kernel one load per series instead of a sequential walk over all blocks (C4, 352 blocks: 378 us -> a few us).
template <int NSEC>
__global__ void __launch_bounds__(SGN)
    espb_biquad_chain_check_kernel(const float4 *__restrict__ blk_state, int n_blocks, int n_series,
                                   unsigned int *__restrict__ group_broken, int k_first) {
  const int tid = threadIdx.x, k = k_first + blockIdx.y;  // hand-over from block k - 1 to block k
  if (blockIdx.x * SGN + tid >= n_series)
    return;
  const float4 *rec = blk_state + ((size_t) blockIdx.x * n_blocks * NSEC * 2) * SGN + tid;
  const float4 *rk = rec + (size_t) k * NSEC * 2 * SGN, *rp = rec + (size_t) (k - 1) * NSEC * 2 * SGN;
  bool same = true;
#pragma unroll
  for (int s = 0; s < NSEC; ++s) {
    const float4 a = rk[(s * 2) * SGN], b = rp[(s * 2 + 1) * SGN];
    same = same && __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y) &&
           __float_as_uint(a.z) == __float_as_uint(b.z) && __float_as_uint(a.w) == __float_as_uint(b.w);
  }
  if (!same)
    atomicOr(group_broken + blockIdx.x, 1u);
}

// Chain check of the time blocks (see the header): one thread per series walks its blocks in order.  A block whose
// recorded start state is not bit-identical to the true end state of its predecessor is filtered again from that
// state.  `mismatches` counts such blocks (diagnostics; the launcher widens the warm-up when it sees any).
template <int NSEC, bool FIRST_ORDER>
__global__ void __launch_bounds__(SGN)
    espb_biquad_verify_kernel(const float *src, float *dst, int64_t rows_cap, int row_first, int n_rows, BiquadParams c,
                              float *__restrict__ state, int n_series, int block_rows, int n_blocks,
                              const float4 *__restrict__ blk_state, unsigned int *mismatches,
                              const unsigned int *__restrict__ group_broken) {
  const int tid = threadIdx.x;
  const int q = blockIdx.x * SGN + tid;
  if (q >= n_series)
    return;
  const float4 *rec = blk_state + ((size_t) blockIdx.x * n_blocks * NSEC * 2) * SGN + tid;
  if (group_broken && group_broken[blockIdx.x] == 0) {
    // every hand-over of every series of this group was found bit-identical (espb_biquad_chain_check_kernel): the
    // output is the sequential one as it stands; commit the state the last block ended in
#pragma unroll
    for (int s = 0; s < NSEC; ++s)
      *reinterpret_cast<float4 *>(state + ((int64_t) q * NSEC + s) * 4) =
          rec[((size_t) (n_blocks - 1) * NSEC * 2 + s * 2 + 1) * SGN];
    return;
  }
  float4 truth[NSEC];  // the true state at the end of the previous block
#pragma unroll
  for (int s = 0; s < NSEC; ++s)
    truth[s] = rec[(s * 2 + 1) * SGN];  // block 0 started from the saved state
  unsigned int bad = 0;
  for (int k = 1; k < n_blocks; ++k) {
    const float4 *rk = rec + (size_t) k * NSEC * 2 * SGN;
    bool same = true;
#pragma unroll
    for (int s = 0; s < NSEC; ++s)
      same = same && same_bits(rk[(s * 2) * SGN], truth[s]);
    if (same) {
#pragma unroll
      for (int s = 0; s < NSEC; ++s)
        truth[s] = rk[(s * 2 + 1) * SGN];
      continue;
    }
    ++bad;
    Section sec[NSEC];
#pragma unroll
    for (int s = 0; s < NSEC; ++s) {
      sec[s].in_d1 = truth[s].x;
      sec[s].in_d2 = truth[s].y;
      sec[s].out_d1 = truth[s].z;
      sec[s].out_d2 = truth[s].w;
    }
    const int lo = k * block_rows, hi = lo + block_rows < n_rows ? lo + block_rows : n_rows;
    const float *ps = src + ((int64_t) blockIdx.x * rows_cap + row_first + lo) * SGN + tid;
    float *pd = dst + ((int64_t) blockIdx.x * rows_cap + row_first + lo) * SGN + tid;
    for (int r = 0; r < hi - lo; ++r) {
      float v = ps[(int64_t) r * SGN];
#pragma unroll
      for (int s = 0; s < NSEC; ++s)
        v = section_step<FIRST_ORDER>(sec[s], v, c);
      pd[(int64_t) r * SGN] = v;
    }
#pragma unroll
    for (int s = 0; s < NSEC; ++s)
      truth[s] = make_float4(sec[s].in_d1, sec[s].in_d2, sec[s].out_d1, sec[s].out_d2);
  }
#pragma unroll
  for (int s = 0; s < NSEC; ++s)
    *reinterpret_cast<float4 *>(state + ((int64_t) q * NSEC + s) * 4) = truth[s];
  if (bad && mismatches)
    atomicAdd(mismatches, bad);
}

// ---------------------------------------------------------------------------------
// One pass on the CALLER'S layout (the stand-alone biquad_apply_buffer): no trip through time-major scratch.
// A CTA owns 128 series.  Chunks of 64 frames come in by 16-byte cp.async in the caller's memory order — a "unit" is
// what is contiguous there: the 64 x channels floats of a stream when interleaved, 64 frames of a plane when planar —
// and stay in that order in the shared-memory tile (unit pitch + 4 floats); the thread that owns a series walks its
// column of the tile (stride = series per unit, a compile-time constant), and the filtered tile goes back by 128-bit
// stores.  CL_STAGES chunks are in flight per CTA.  8 algorithmic bytes per sample, in place.  The recurrence is the
// floor: ~40 cycles per frame (two sections) for every series, however many there are.  Unaligned rows and the last
// partial chunk take 4-byte copies into a series-major tile of pitch 65.
// ---------------------------------------------------------------------------------
constexpr int CL_ROWS = 64, CL_LOG_ROWS = 6, CL_STAGES = 3;  // 64-frame chunks: half the barriers per frame of 32
__host__ __device__ constexpr int cl_pitch(bool vec) { return vec ? CL_ROWS + 4 : CL_ROWS + 1; }

// LUT >= 0: log2(series per unit) known at compile time (the 16-byte form: the column stride of the filter loop must
// be a constant, or the compiler cannot move a row's load above the previous row's store and the recurrence waits
// for shared memory every row — measured 1.7x slower); LUT < 0: the 4-byte form, taken from the argument.
template <int NSEC, bool FIRST_ORDER, int LUT>
__global__ void __launch_bounds__(2 * SGN)
    espb_biquad_cl_kernel(float *buf, int64_t ss, int64_t cs, int64_t fs, int channels, int lu_arg, int n_series,
                          int n_frames, BiquadParams c, float *__restrict__ state) {
  constexpr bool VEC = LUT >= 0;
  const int lu = VEC ? LUT : lu_arg;
  constexpr int CL_PITCH = cl_pitch(VEC);
  extern __shared__ __align__(16) unsigned char cl_smem[];
  float (*tile)[SGN * CL_PITCH] = reinterpret_cast<float (*)[SGN * CL_PITCH]>(cl_smem);  // [CL_STAGES][128 x pitch]
  int64_t *base_tab = reinterpret_cast<int64_t *>(cl_smem + sizeof(float) * CL_STAGES * SGN * CL_PITCH);  // [128]
  // Warp-specialised: threads [0, 128) own a series each and only run the recurrence; threads [128, 256) only move
  // data (cp.async in, 128-bit stores out).  With one CTA per SM the recurrence used to stand still during every
  // copy phase of its own threads (78 cycles per frame for two sections instead of ~45); hand-overs are named
  // barriers: LOADED[stage] (copiers arrive, filters wait), FILTERED[stage] (the reverse), COPY (copiers only).
  const bool copier = threadIdx.x >= SGN;
  const int tid = threadIdx.x & (SGN - 1);
  const int q0 = blockIdx.x * SGN;
  const int q = q0 + tid;
  const int n_chunks = (n_frames + CL_ROWS - 1) / CL_ROWS;
  constexpr int BAR_LOADED = 1, BAR_FILTERED = 1 + CL_STAGES, BAR_COPY = 1 + 2 * CL_STAGES;
  // where frame 0 of every series of this CTA lies (-1: no such series); frame j is j * fs further
  if (!copier) {
    const int st = q / channels, ch = q - st * channels;
    base_tab[tid] = q < n_series ? (int64_t) st * ss + (int64_t) ch * cs : (int64_t) -1;
  }
  __syncthreads();
  // Memory-order enumeration of a chunk: a unit (a stream when interleaved, a plane when planar) holds 2^lu series;
  // element e of a unit's run of 32 << lu floats is frame e >> lu of its series e & (2^lu - 1).  Consecutive threads
  // touch consecutive addresses; everything is shifts.
  const int run_mask = (CL_ROWS << lu) - 1, unit_mask = (1 << lu) - 1, run_shift = CL_LOG_ROWS + lu;
  const int unit_pitch = (CL_ROWS << lu) + 4;  // VEC tile: [unit][frame][series of the unit] + 4 floats of padding
  auto load_chunk = [&](int k) {
    float *t = tile[k % CL_STAGES];
    const int j0 = k * CL_ROWS;
    if (VEC && j0 + CL_ROWS <= n_frames) {
      // 16-byte copies: a unit's 32 << lu floats of this chunk are contiguous and aligned in memory and stay in
      // memory order in the tile (unit pitch (32 << lu) + 4)
#pragma unroll
      for (int i = tid; i < SGN * (CL_ROWS / 4); i += SGN) {
        const int u = i >> (CL_LOG_ROWS - 2 + lu), v4 = (i & (((CL_ROWS / 4) << lu) - 1)) * 4;
        const int64_t base = base_tab[u << lu];
        if (base >= 0)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(t + u * unit_pitch + v4)),
                       "l"(buf + base + (int64_t) j0 * fs + v4)
                       : "memory");
      }
    } else {
#pragma unroll 4
      for (int i = tid; i < SGN * CL_ROWS; i += SGN) {
        const int e = i & run_mask;
        const int jj = e >> lu, sl = ((i >> run_shift) << lu) + (e & unit_mask);
        const int64_t base = base_tab[sl];
        if (base >= 0 && j0 + jj < n_frames)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(smem_u32(t + sl * CL_PITCH + jj)),
                       "l"(buf + base + (int64_t) (j0 + jj) * fs)
                       : "memory");
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };
  auto store_chunk = [&](int k) {
    float *t = tile[k % CL_STAGES];
    const int j0 = k * CL_ROWS;
    if (VEC && j0 + CL_ROWS <= n_frames) {
#pragma unroll
      for (int i = tid; i < SGN * (CL_ROWS / 4); i += SGN) {
        const int u = i >> (CL_LOG_ROWS - 2 + lu), v4 = (i & (((CL_ROWS / 4) << lu) - 1)) * 4;
        const int64_t base = base_tab[u << lu];
        if (base >= 0)
          *reinterpret_cast<float4 *>(buf + base + (int64_t) j0 * fs + v4) =
              *reinterpret_cast<const float4 *>(t + u * unit_pitch + v4);
      }
    } else {
#pragma unroll 4
      for (int i = tid; i < SGN * CL_ROWS; i += SGN) {
        const int e = i & run_mask;
        const int jj = e >> lu, sl = ((i >> run_shift) << lu) + (e & unit_mask);
        const int64_t base = base_tab[sl];
        if (base >= 0 && j0 + jj < n_frames)
          buf[base + (int64_t) (j0 + jj) * fs] = t[sl * CL_PITCH + jj];
      }
    }
  };
  if (copier) {
    for (int k = 0; k < CL_STAGES - 1; ++k) {
      if (k < n_chunks)
        load_chunk(k);
      else
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    }
    for (int k = 0; k < n_chunks; ++k) {
      asm volatile("cp.async.wait_group %0;\n" ::"n"(CL_STAGES - 2) : "memory");  // chunk k has landed (this thread's part)
      named_bar_arrive(BAR_LOADED + k % CL_STAGES, 2 * SGN);
      if (k >= 1) {
        named_bar_sync(BAR_FILTERED + (k - 1) % CL_STAGES, 2 * SGN);
        store_chunk(k - 1);
        named_bar_sync(BAR_COPY, SGN);  // every copier has read that stage: it may be refilled
      }
      if (k + CL_STAGES - 1 < n_chunks)
        load_chunk(k + CL_STAGES - 1);  // into the stage of chunk k - 1
      else
        asm volatile("cp.async.commit_group;\n" ::: "memory");
    }
    named_bar_sync(BAR_FILTERED + (n_chunks - 1) % CL_STAGES, 2 * SGN);
    store_chunk(n_chunks - 1);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    return;
  }
  Section sec[NSEC];
  if (q < n_series) {
#pragma unroll
    for (int k = 0; k < NSEC; ++k) {
      const float4 v = *reinterpret_cast<const float4 *>(state + ((int64_t) q * NSEC + k) * 4);
      sec[k].in_d1 = v.x, sec[k].in_d2 = v.y, sec[k].out_d1 = v.z, sec[k].out_d2 = v.w;
    }
  } else {
#pragma unroll
    for (int k = 0; k < NSEC; ++k)
      sec[k].in_d1 = sec[k].in_d2 = sec[k].out_d1 = sec[k].out_d2 = 0.0f;
  }
  for (int k = 0; k < n_chunks; ++k) {
    named_bar_sync(BAR_LOADED + k % CL_STAGES, 2 * SGN);
    float *t = tile[k % CL_STAGES];
    const int j0 = k * CL_ROWS;
    const int rows = j0 + CL_ROWS <= n_frames ? CL_ROWS : n_frames - j0;
    // this thread's series: column tid of the series-major tile, or (unit tid >> lu, series tid & mask) of the VEC tile
    if (rows == CL_ROWS) {
      constexpr int rstep = VEC ? (1 << (LUT < 0 ? 0 : LUT)) : 1;
      float *mine = VEC ? t + (tid >> lu) * unit_pitch + (tid & unit_mask) : t + tid * CL_PITCH;
#pragma unroll 8
      for (int r = 0; r < CL_ROWS; ++r) {
        float v = mine[r * rstep];
#pragma unroll
        for (int s2 = 0; s2 < NSEC; ++s2)
          v = section_step<FIRST_ORDER>(sec[s2], v, c);
        mine[r * rstep] = v;
      }
    } else {
      float *mine = t + tid * CL_PITCH;
      for (int r = 0; r < rows; ++r) {
        float v = mine[r];
#pragma unroll
        for (int s2 = 0; s2 < NSEC; ++s2)
          v = section_step<FIRST_ORDER>(sec[s2], v, c);
        mine[r] = v;
      }
    }
    named_bar_arrive(BAR_FILTERED + k % CL_STAGES, 2 * SGN);
  }
  if (q < n_series) {
#pragma unroll
    for (int k = 0; k < NSEC; ++k)
      *reinterpret_cast<float4 *>(state + ((int64_t) q * NSEC + k) * 4) =
          make_float4(sec[k].in_d1, sec[k].in_d2, sec[k].out_d1, sec[k].out_d2);
  }
}

template <int NSEC, int LUT>
cudaError_t launch_cl(float *buf, int64_t ss, int64_t cs, int64_t fs, int channels, int lu, int n_series,
                      int n_frames, const BiquadParams &c, float *state, cudaStream_t stream) {
  const int grid = (n_series + SGN - 1) / SGN;
  const size_t smem = sizeof(float) * CL_STAGES * SGN * cl_pitch(LUT >= 0) + SGN * sizeof(int64_t);
  static PerDeviceOnce once;
  if (once.first()) {
    cudaError_t e = cudaSuccess;
    const void *fns[2] = {reinterpret_cast<const void *>(espb_biquad_cl_kernel<NSEC, true, LUT>),
                          reinterpret_cast<const void *>(espb_biquad_cl_kernel<NSEC, false, LUT>)};
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
      e = cudaFuncSetAttribute(fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(fns[i], cudaFuncAttributePreferredSharedMemoryCarveout,
                                 (int) cudaSharedmemCarveoutMaxShared);
    }
    if (e != cudaSuccess)
      return e;
  }
  if (c.first_order)
    espb_biquad_cl_kernel<NSEC, true, LUT><<<grid, 2 * SGN, smem, stream>>>(buf, ss, cs, fs, channels, lu, n_series,
                                                                         n_frames, c, state);
  else
    espb_biquad_cl_kernel<NSEC, false, LUT><<<grid, 2 * SGN, smem, stream>>>(buf, ss, cs, fs, channels, lu, n_series,
                                                                          n_frames, c, state);
  count_launch();
  return cudaGetLastError();
}

template <int NSEC>
cudaError_t launch_cl_any(bool vec, float *buf, int64_t ss, int64_t cs, int64_t fs, int channels, int lu, int n_series,
                          int n_frames, const BiquadParams &c, float *state, cudaStream_t stream) {
  if (!vec)
    return launch_cl<NSEC, -1>(buf, ss, cs, fs, channels, lu, n_series, n_frames, c, state, stream);
  switch (lu) {
    case 0:
      return launch_cl<NSEC, 0>(buf, ss, cs, fs, channels, lu, n_series, n_frames, c, state, stream);
    case 1:
      return launch_cl<NSEC, 1>(buf, ss, cs, fs, channels, lu, n_series, n_frames, c, state, stream);
    case 2:
      return launch_cl<NSEC, 2>(buf, ss, cs, fs, channels, lu, n_series, n_frames, c, state, stream);
    default:
      return launch_cl<NSEC, 3>(buf, ss, cs, fs, channels, lu, n_series, n_frames, c, state, stream);
  }
}

template <int NSEC>
cudaError_t launch_tm(const float *src, float *dst, int64_t rows_cap, int row_first, int n_rows, int n_series,
                      const BiquadParams &c, float *state, int block_rows, int warm_rows, float *blk_state,
                      unsigned int *mismatches, cudaStream_t stream, unsigned int *chain_broken) {
  const int n_blocks = block_rows > 0 ? (n_rows + block_rows - 1) / block_rows : 1;
  float4 *rec = block_rows > 0 ? reinterpret_cast<float4 *>(blk_state) : nullptr;
  const dim3 grid((n_series + SGN - 1) / SGN);  // groups (time blocks: y, in slices)
  const size_t smem = sizeof(float) * BSTAGES * RB * SGN + BSTAGES * sizeof(uint64_t);
  static PerDeviceOnce once;
  if (once.first()) {
    cudaError_t e = cudaFuncSetAttribute(espb_biquad_tm_kernel<NSEC, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(espb_biquad_tm_kernel<NSEC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               (int) smem);
    if (e != cudaSuccess)
      return e;
  }
  if (rec && n_series <= kBiquadFewSeries) {  // one group, few series: threads are (block, series) pairs
    int lanes = 4;
    while (lanes < n_series)
      lanes *= 2;
    const int ctas = (n_blocks * lanes + SGN - 1) / SGN;
    if (c.first_order)
      espb_biquad_tm_few_kernel<NSEC, true><<<ctas, SGN, 0, stream>>>(src, dst, row_first, n_rows, c, state, n_series,
                                                                     lanes, block_rows, warm_rows, n_blocks, rec);
    else
      espb_biquad_tm_few_kernel<NSEC, false><<<ctas, SGN, 0, stream>>>(src, dst, row_first, n_rows, c, state, n_series,
                                                                      lanes, block_rows, warm_rows, n_blocks, rec);
    count_launch();
  } else {  // time blocks ride on y
    cudaError_t e = for_each_y_slice(n_blocks, [&](int b0, int nb) {
      const dim3 grid_b(grid.x, nb);
      if (c.first_order)
        espb_biquad_tm_kernel<NSEC, true><<<grid_b, SGN, smem, stream>>>(src, dst, rows_cap, row_first, n_rows, c,
                                                                         state, n_series, block_rows, warm_rows, rec,
                                                                         b0, n_blocks);
      else
        espb_biquad_tm_kernel<NSEC, false><<<grid_b, SGN, smem, stream>>>(src, dst, rows_cap, row_first, n_rows, c,
                                                                          state, n_series, block_rows, warm_rows, rec,
                                                                          b0, n_blocks);
      count_launch();
      return cudaGetLastError();
    });
    if (e != cudaSuccess)
      return e;
  }
  if (rec) {  // prove (or repair) the block hand-overs and commit the final state
    unsigned int *broken = chain_broken;  // one word per group of this launch; NULL: always walk the chain
    if (broken) {
      cudaError_t e = cudaMemsetAsync(broken, 0, grid.x * sizeof(unsigned int), stream);
      if (e != cudaSuccess)
        return e;
    }
    if (broken && n_blocks > 1) {  // the n_blocks - 1 hand-overs ride on y
      cudaError_t e = for_each_y_slice(n_blocks - 1, [&](int k0, int nk) {
        espb_biquad_chain_check_kernel<NSEC><<<dim3(grid.x, nk), SGN, 0, stream>>>(rec, n_blocks, n_series, broken,
                                                                                   k0 + 1);
        count_launch();
        return cudaGetLastError();
      });
      if (e != cudaSuccess)
        return e;
    }
    if (c.first_order)
      espb_biquad_verify_kernel<NSEC, true><<<grid.x, SGN, 0, stream>>>(src, dst, rows_cap, row_first, n_rows, c, state,
                                                                       n_series, block_rows, n_blocks, rec, mismatches,
                                                                       broken);
    else
      espb_biquad_verify_kernel<NSEC, false><<<grid.x, SGN, 0, stream>>>(src, dst, rows_cap, row_first, n_rows, c,
                                                                        state, n_series, block_rows, n_blocks, rec,
                                                                        mismatches, broken);
    count_launch();
  }
  return cudaGetLastError();
}

}  // namespace

// One-pass filter on the caller's layout.  Returns cudaErrorNotSupported when the layout is neither interleaved with
// a channel count that divides 128 nor frame-contiguous (the caller then takes the time-major route).
cudaError_t launch_biquad_cl(float *buf, int64_t ss, int64_t cs, int64_t fs, int channels, int n_series, int n_frames,
                             int n_sections, BiquadParams c, float *state, cudaStream_t stream) {
  if (n_series <= 0 || n_frames <= 0)
    return cudaSuccess;
  int unit_series = -1;  // log2 of the series per contiguous run
  if (fs == 1)
    unit_series = 0;  // planar (or mono): a plane's frames are contiguous
  else if (cs == 1 && fs == channels && (channels == 2 || channels == 4 || channels == 8))
    unit_series = channels == 2 ? 1 : (channels == 4 ? 2 : 3);  // interleaved: frames x channels of a stream are
  else
    return cudaErrorNotSupported;
  // 16-byte copies: every unit's frame 0 on a 16-byte boundary (a unit is a stream when interleaved, a plane else)
  const bool vec = (uintptr_t) buf % 16 == 0 && ss % 4 == 0 &&
                   (unit_series > 0 || cs % 4 == 0 || channels == 1);
  switch (n_sections) {
    case 1:
      return launch_cl_any<1>(vec, buf, ss, cs, fs, channels, unit_series, n_series, n_frames, c, state, stream);
    case 2:
      return launch_cl_any<2>(vec, buf, ss, cs, fs, channels, unit_series, n_series, n_frames, c, state, stream);
    case 3:
      return launch_cl_any<3>(vec, buf, ss, cs, fs, channels, unit_series, n_series, n_frames, c, state, stream);
    case 4:
      return launch_cl_any<4>(vec, buf, ss, cs, fs, channels, unit_series, n_series, n_frames, c, state, stream);
    default:
      return cudaErrorInvalidValue;
  }
}

size_t biquad_block_state_floats(int n_series, int n_sections, int n_rows, int block_rows) {
  if (block_rows <= 0 || block_rows >= n_rows)
    return 0;
  const size_t n_blocks = ((size_t) n_rows + block_rows - 1) / block_rows;
  const size_t n_groups = (size_t) ((n_series + SGN - 1) / SGN);
  return n_groups * n_blocks * n_sections * 2 * SGN * 4;
}

namespace {
template <int NSEC, int NBYTES>
cudaError_t launch_tm_pcm(float *buf, int64_t rows_cap, int row_first, int n_rows, int n_series, BiquadParams c,
                          float *state, uint8_t *out, int64_t out_row_bytes, const F2QConst &qc, uint32_t *clipped,
                          cudaStream_t stream) {
  const size_t smem = sizeof(float) * BSTAGES * RB * SGN + BSTAGES * sizeof(uint64_t);
  constexpr bool B32 = NBYTES == 4;  // (bits == 32 is the only 4-byte depth with its own clipping rule)
  const bool bits32 = B32 && qc.bits == 32;
  static PerDeviceOnce once;
  if (once.first()) {
    cudaError_t e = cudaFuncSetAttribute(espb_biquad_tm_pcm_kernel<NSEC, true, NBYTES, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(espb_biquad_tm_pcm_kernel<NSEC, false, NBYTES, false>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess && B32)
      e = cudaFuncSetAttribute(espb_biquad_tm_pcm_kernel<NSEC, true, NBYTES, B32>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess && B32)
      e = cudaFuncSetAttribute(espb_biquad_tm_pcm_kernel<NSEC, false, NBYTES, B32>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess)
      return e;
  }
  const int grid = (n_series + SGN - 1) / SGN;
#define ESPB_BQP(FO_, B_)                                                                                          \
  espb_biquad_tm_pcm_kernel<NSEC, FO_, NBYTES, B_><<<grid, BQP_THREADS, smem, stream>>>(buf, rows_cap, row_first, n_rows, c, \
                                                                                    state, n_series, out,          \
                                                                                    out_row_bytes, qc, clipped)
  if (c.first_order) {
    if (bits32)
      ESPB_BQP(true, B32);
    else
      ESPB_BQP(true, false);
  } else {
    if (bits32)
      ESPB_BQP(false, B32);
    else
      ESPB_BQP(false, false);
  }
#undef ESPB_BQP
  count_launch();
  return cudaGetLastError();
}
template <int NSEC>
cudaError_t launch_tm_pcm_bytes(int nbytes, float *buf, int64_t rows_cap, int row_first, int n_rows, int n_series,
                                BiquadParams c, float *state, uint8_t *out, int64_t out_row_bytes, const F2QConst &qc,
                                uint32_t *clipped, cudaStream_t stream) {
  switch (nbytes) {
    case 1:
      return launch_tm_pcm<NSEC, 1>(buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped, stream);
    case 2:
      return launch_tm_pcm<NSEC, 2>(buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped, stream);
    case 3:
      return launch_tm_pcm<NSEC, 3>(buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped, stream);
    default:
      return launch_tm_pcm<NSEC, 4>(buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped, stream);
  }
}
}  // namespace

// Mono streams: filter rows [row_first, row_first + n_rows) of buf (time-major) and write them as packed PCM to
// out[stream] — frames [0, returned) — in one pass; the filtered floats of the remaining rows (the last partial
// 32-row chunk) are written back to buf for the caller's generic tail path.  Returns 0 (nothing enqueued) when the
// output rows are not 16-byte aligned or there is no full chunk.
int launch_biquad_tm_pcm(float *buf, int64_t rows_cap, int row_first, int n_rows, int n_series, int n_sections,
                         BiquadParams c, float *state, uint8_t *out, int64_t out_row_bytes, int bits,
                         uint32_t *clipped_per_stream, cudaStream_t stream, cudaError_t *err) {
  *err = cudaSuccess;
  if (n_series <= 0 || n_rows < RB || bits < 1 || bits > 32 || ((uintptr_t) out % 16) || (out_row_bytes % 16))
    return 0;
  const int nbytes = (bits + 7) / 8;
  const F2QConst qc = make_f2q_const(bits);
  switch (n_sections) {
    case 1:
      *err = launch_tm_pcm_bytes<1>(nbytes, buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped_per_stream, stream);
      break;
    case 2:
      *err = launch_tm_pcm_bytes<2>(nbytes, buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped_per_stream, stream);
      break;
    case 3:
      *err = launch_tm_pcm_bytes<3>(nbytes, buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped_per_stream, stream);
      break;
    case 4:
      *err = launch_tm_pcm_bytes<4>(nbytes, buf, rows_cap, row_first, n_rows, n_series, c, state, out, out_row_bytes, qc, clipped_per_stream, stream);
      break;
    default:
      return 0;
  }
  return (n_rows / RB) * RB;
}

cudaError_t launch_biquad_tm(const float *src, float *dst, int64_t rows_cap, int row_first, int n_rows, int n_series,
                             int n_sections, BiquadParams c, float *state, int block_rows, int warm_rows,
                             cudaStream_t stream, float *blk_state, unsigned int *mismatches,
                             unsigned int *chain_broken) {
  if (n_series <= 0 || n_rows <= 0)
    return cudaSuccess;
  if (block_rows >= n_rows)
    block_rows = 0;
  if (block_rows > 0 && (block_rows % RB || warm_rows % RB || src == dst || !blk_state))
    return cudaErrorInvalidValue;  // time blocks: multiples of the 32-row chunk, out of place, with a state record
  switch (n_sections) {
    case 1:
      return launch_tm<1>(src, dst, rows_cap, row_first, n_rows, n_series, c, state, block_rows, warm_rows,
                          blk_state, mismatches, stream, chain_broken);
    case 2:
      return launch_tm<2>(src, dst, rows_cap, row_first, n_rows, n_series, c, state, block_rows, warm_rows,
                          blk_state, mismatches, stream, chain_broken);
    case 3:
      return launch_tm<3>(src, dst, rows_cap, row_first, n_rows, n_series, c, state, block_rows, warm_rows,
                          blk_state, mismatches, stream, chain_broken);
    case 4:
      return launch_tm<4>(src, dst, rows_cap, row_first, n_rows, n_series, c, state, block_rows, warm_rows,
                          blk_state, mismatches, stream, chain_broken);
    default:
      return cudaErrorInvalidValue;
  }
}

}  // namespace espb
