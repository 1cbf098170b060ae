// ART polyphase resampler — sm_100a kernels.
//
// What is computed (reference art_resampler.cpp:432-451 + dsps_dotprod_f32_ansi.c:17-25):
//   out[series][n] = blend_n( sum_k H[phase_n][k]   * x[series][ws_n + k],
//                             sum_k H[phase_n+1][k] * x[series][ws_n + k] )
// with each sum evaluated strictly in tap order by ONE accumulator (FFMA chain in fast
// mode, FMUL+FADD in exact mode) — splitting a sum across lanes or accumulators moves the
// result by up to 1.8e-6 against the reference (SURVEY.md §8a R5) and is not allowed.
//
// Data layout in HBM (ours, built per call):
//   xt[group g][row r][128 series]   time-major input staging: row r holds input frame
//        j = r - numTaps of the 128 series (stream x channel) of group g; rows [0, numTaps)
//        are the frames carried over from the previous call (the reference keeps them at
//        the front of its ring, art_resampler.cpp:216-222), rows past the input are zero.
//        Written by espb_transpose_kernel from the caller's stream-major buffers.
//   G[chunk][row][block-in-pass b][n in block][f]  =  H[phase_n + f][j - ws_n]  (0 outside the
//        window): the two coefficient columns of every output, pre-skewed to input rows.
//        The schedule (ws_n, phase_n, w_n) is identical for all streams, so G is expanded
//        once per call (espb_expand_kernel) and shared by every CTA.
// With these, one chunk (32 input rows) of either operand is ONE contiguous 16 KB block.
//
// Kernel.  A CTA (4 warps, four CTAs per SM) owns one group (128 series) and sweeps "passes" of 4
// consecutive output blocks (8 outputs each, one block per warp) over the union of their windows in chunks of 32
// rows, streamed through a 2-stage shared-memory ring with two TMA bulk copies per
// chunk (cp.async.bulk -> mbarrier complete_tx; SASS UBLKCP).  There is no producer warp (a fifth warp would not fit
// four times per SM next to 128-register consumers): the last warp to finish reading a stage re-arms its mbarrier
// and issues the refill.  At set-up the CTA builds a table of what each warp does in each chunk (first / last
// 4-row group inside its window, end-of-pass flag), so the main loop has no window arithmetic and no global loads.
// The warps wait on the stage's "full" mbarrier, and per input row do the rank-1 update
//     acc[series e][n][f] += G[row][n][f] * x[row][series e]
// of a 4-series x 8-output x 2-filter register tile: x is one per-lane 128-bit LDS, G four warp-uniform 128-bit LDS
// (broadcast) -> 32 packed FFMA2 (64 FMUL+FADD in exact mode) per 5 LDS, 8 shared-memory wavefronts per row, every
// accumulator visiting its taps in order.  No block-wide barrier in the main loop; warps whose window does not reach
// a chunk (or a group of 4 rows) skip it.  At the end of a pass the block's 8 schedule entries are already in shared
// memory (cp.async issued at the top of the last chunk); blend, then 128-bit stores in the caller's layout.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.hpp"
#include "kernels.hpp"
#include "resample_device.cuh"

namespace espb {


// Segmented schedule -> finalized entries: every output finds its arithmetic-progression run (plan.cpp:
// build_schedule_segments) by binary search, rebuilds its offset exactly (all terms are multiples of one ulp of the
// run's binade, so the double-precision product and sum are exact and the conversion back does not round) and
// finishes it like plan.cpp:finalize_entries (the same IEEE operations, so the same bits).  The host uploads a few
// hundred bytes per ring cycle instead of 16 bytes per output.
__global__ void __launch_bounds__(256)
    espb_expand_schedule_kernel(const SchedSegment *__restrict__ segs, int n_segs, OutEntry *__restrict__ outs, int n,
                                float n_filters, int lowpass, int interp) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n)
    return;
  int lo = 0, hi = n_segs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&segs[mid].n0) <= k)
      lo = mid;
    else
      hi = mid - 1;
  }
  const SchedSegment sg = segs[lo];
  const float off = (float) ((double) sg.off0 + (double) (k - sg.n0) * (double) sg.inc);
  const float fl = (float) (int) off;
  float frac = __fsub_rn(off, fl);
  OutEntry e;
  e.ws = sg.ws_base + (int32_t) fl;
  e.phase = 0;
  e.w = 0.0f;
  if (frac == 0.0f && !lowpass) {
    e.kind = kKindPass;
  } else if (!interp) {
    e.kind = kKindSingle;
    e.phase = (int) __fadd_rn(__fmul_rn(frac, n_filters), 0.5f);
  } else {
    frac = __fmul_rn(frac, n_filters);
    const int i = (int) frac;
    frac = __fsub_rn(frac, (float) i);
    e.phase = i;
    e.w = frac;
    e.kind = (frac == 0.0f && !lowpass) ? kKindSingle : kKindBlend;
  }
  outs[k] = e;
}

// ---------------------------------------------------------------------------------
// G expansion.  CTAs stride over the chunks; within a chunk a warp takes 32 consecutive rows of one float4
// (two outputs x two filters), so its reads of a filter row are one coalesced 128-byte line and the two schedule
// entries are warp-uniform; the tile goes through (padded) shared memory and leaves as contiguous 16-byte stores.
// ---------------------------------------------------------------------------------
constexpr int kExpandThreads = 256;
// rows x (float4 per row + 1 pad); a row of either G form is 16 float4: 4 blocks x 16 floats, or 8 blocks x 8
constexpr int kExpandTileFloat4 = kResampleChunkRows * (kResampleWarps * kGRowFloats / 4 + 1);

__global__ void __launch_bounds__(kExpandThreads)
    espb_expand_kernel(const float *__restrict__ bank, const OutEntry *__restrict__ outs,
                       const ChunkEntry *__restrict__ chunks, float *__restrict__ G, int chunk_first, int n_chunks,
                       int n_out, int taps, int bpp, int grf) {
  constexpr int CJ = kResampleChunkRows;
  __shared__ float4 tile[kExpandTileFloat4];
  const int quads_per_row = bpp * (grf / 4);
  const bool ni = grf == kGRowFloatsNI;
  const int pitch = quads_per_row + 1;
  const int total = CJ * quads_per_row;
  for (int cc = blockIdx.x; cc < n_chunks; cc += gridDim.x) {
    const ChunkEntry ce = chunks[chunk_first + cc];
    for (int i = threadIdx.x; i < total; i += kExpandThreads) {
      const int quad = i / CJ, jj = i - quad * CJ;  // rows fastest: a warp reads one filter row contiguously
      // block in pass; the quad holds outputs (2 pair, 2 pair + 1) x (filter 0, 1), or four outputs x one filter
      const int b = ni ? quad >> 1 : quad >> 2, pair = ni ? (quad & 1) * 2 : quad & 3;
      const int j = ce.j_start + jj;
      float v[4];
      if (ni) {
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          const int o = (ce.pass * bpp + b) * NB + pair * 2 + h;
          float c0 = 0.0f;
          if (o < n_out) {
            const OutEntry e = outs[o];
            const int k = j - e.ws;
            if (k >= 0 && k < taps && e.kind >= kKindSingle)
              c0 = __ldg(bank + (size_t) e.phase * taps + k);
          }
          v[h] = c0;
        }
      } else
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int o = (ce.pass * bpp + b) * NB + pair * 2 + h;
        float c0 = 0.0f, c1 = 0.0f;
        if (o < n_out) {
          const OutEntry e = outs[o];
          const int k = j - e.ws;
          if (k >= 0 && k < taps && e.kind >= kKindSingle) {
            c0 = __ldg(bank + (size_t) e.phase * taps + k);
            if (e.kind == kKindBlend)
              c1 = __ldg(bank + (size_t) (e.phase + 1) * taps + k);
          }
        }
        v[2 * h] = c0;
        v[2 * h + 1] = c1;
      }
      tile[jj * pitch + quad] = make_float4(v[0], v[1], v[2], v[3]);
    }
    __syncthreads();
    float4 *dst = reinterpret_cast<float4 *>(G + (size_t) cc * CJ * bpp * grf);
    for (int i = threadIdx.x; i < total; i += kExpandThreads) {
      const int jj = i / quads_per_row, quad = i - jj * quads_per_row;
      dst[i] = tile[jj * pitch + quad];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------
// Transposing stage: caller layout (stream-major, any strides) -> xt[group][row][128].
// A CTA moves a 128-series x R-row tile through shared memory so that both the HBM reads
// (along time within a stream) and the HBM writes (along series) are coalesced.  Frames
// [j_begin, n_in) go to rows row_first + j; `pad_rows` rows after the input are zeroed
// (chunks may read up to 31 rows past the last window).
// ---------------------------------------------------------------------------------
constexpr int TR_ROWS = 32;   // generic kernel
constexpr int TF_ROWS = 64;   // fast kernel
constexpr int TF_THREADS = 256;

// Fast path: interleaved input (channel stride 1, frame stride CH) with CH in {1,2,4,8}, or planar
// input (frame stride 1; CH = 1 and one "stream" per series), 16-byte aligned rows, full tiles only.
// VEC-float loads along time (4, 2 or 1 as the alignment of the rows allows), index arithmetic by shifts only.
// One tile: ROWS frames x 128 series of group g starting at frame j0, through `tile` (ROWS x (SGN + 1) floats).
template <int CH, bool PLANAR, int VEC, int ROWS>
__device__ __forceinline__ void transpose_fast_tile(const SwzTile tile, int g, int j0, const float *__restrict__ in,
                                                    int64_t in_ss, int64_t in_cs, int channels, int n_series,
                                                    float *__restrict__ xt, int64_t rows_cap, int row_first) {
  const int tid = threadIdx.x;
  constexpr int UNITS = SGN / CH;              // contiguous runs per group (streams, or series when planar)
  constexpr int V_PER_UNIT = ROWS * CH / VEC;  // vectors per run
  // 16-byte units of a row that hold series of this group (all 32 but in the last group), and the runs they span:
  // a group with few series — one stereo or 8-channel stream per context — neither fills nor stores the rest of
  // the tile (those units of xt were zeroed when the staging buffers were allocated; nobody reads them as data)
  const int units = (n_series - g * SGN + 3) / 4 < SGN / 4 ? (n_series - g * SGN + 3) / 4 : SGN / 4;
  const int runs_here = (units * 4 + CH - 1) / CH < UNITS ? (units * 4 + CH - 1) / CH : UNITS;
#pragma unroll 4
  for (int v = tid; v < runs_here * V_PER_UNIT; v += TF_THREADS) {
    const int unit = v / V_PER_UNIT, off4 = v % V_PER_UNIT;  // powers of two: shifts
    const int q0 = g * SGN + unit * CH;                       // first series of the run
    float xv[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k)
      xv[k] = 0.0f;
    if (q0 < n_series) {
      const float *src;
      if (PLANAR) {
        const int st = q0 / channels, ch = q0 - st * channels;
        src = in + (int64_t) st * in_ss + (int64_t) ch * in_cs + j0;
      } else {
        src = in + (int64_t) (q0 / CH) * in_ss + (int64_t) j0 * CH;
      }
      if constexpr (VEC == 4) {
        const float4 x = __ldg(reinterpret_cast<const float4 *>(src) + off4);
        xv[0] = x.x, xv[1] = x.y, xv[2] = x.z, xv[3] = x.w;
      } else if constexpr (VEC == 2) {
        const float2 x = __ldg(reinterpret_cast<const float2 *>(src) + off4);
        xv[0] = x.x, xv[1] = x.y;
      } else {
        xv[0] = __ldg(src + off4);
      }
    }
    const int e0 = off4 * VEC;
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      const int e = e0 + k;
      tile.at(e / CH, unit * CH + (e % CH)) = xv[k];
    }
  }
  __syncthreads();
  float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + row_first + j0) * SGN);
#pragma unroll 4
  for (int i = tid; i < ROWS * (SGN / 4); i += TF_THREADS) {
    const int t = i / (SGN / 4), c4 = i % (SGN / 4);
    if (c4 < units)
      dst[i] = tile.vec(t, c4);
  }
}

template <int CH, bool PLANAR, int VEC>
__global__ void __launch_bounds__(TF_THREADS)
    espb_transpose_fast_kernel(const float *__restrict__ in, int64_t in_ss, int64_t in_cs, int channels,
                               int n_series, float *__restrict__ xt, int64_t rows_cap, int row_first) {
  __shared__ __align__(16) float tile_s[TF_ROWS * SGN];
  const SwzTile tile{tile_s};
  transpose_fast_tile<CH, PLANAR, VEC, TF_ROWS>(tile, blockIdx.x, blockIdx.y * TF_ROWS, in, in_ss, in_cs, channels,
                                                n_series, xt, rows_cap, row_first);
}

// The same tiles (32 rows each) from a resident grid that signals its progress: CTAs stride over the tiles in time
// order (all groups of row tile 0, then of row tile 1, ...) and bump ready[row tile] once a tile's stores are out.
// The resampler kernel is launched behind it as a programmatic dependent (griddepcontrol.launch_dependents at the
// top: it may start as soon as every CTA of this grid is running) and its CTAs wait on those counters for the rows
// they read, so the FMA-bound kernel starts a few row tiles after this one and hides part of it (DESIGN.md §4.5).
// This grid never waits for anything and is fully resident (two CTAs per SM): the dependants cannot starve it.
// POLICY: the caller's frames are read once — loads carry an L2 evict-first policy.
// Deliberately NOT software-pipelined: a 512-thread version with the next tile's loads in flight during the stores
// finishes in half the time but slows the resampler next to it by more than it saves (measured, §4.5) — what the
// resampler pays for is the memory traffic beside its own latency-critical TMA loads, not the occupied slot.
template <int CH, bool PLANAR, bool POLICY>
__global__ void __launch_bounds__(TF_THREADS)
    espb_transpose_flags_kernel(const float *__restrict__ in, int64_t in_ss, int64_t in_cs, int channels, int n_series,
                                float *__restrict__ xt, int64_t rows_cap, int row_first, int n_groups, int n_tiles,
                                int *__restrict__ ready) {
  constexpr int ROWS = kReadyTileRows;
  __shared__ __align__(16) float tile_s[ROWS * SGN];
  const SwzTile tile{tile_s};
  grid_launch_dependents();
  const int tid = threadIdx.x;
  constexpr int UNITS = SGN / CH;            // contiguous runs per group (streams, or series when planar)
  constexpr int V_PER_UNIT = ROWS * CH / 4;  // float4 per run
  uint64_t pol = 0;
  if (POLICY)
    pol = l2_policy_evict_first();
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int y = t / n_groups, g = t - y * n_groups, j0 = y * ROWS;
#pragma unroll 4
    for (int v = tid; v < UNITS * V_PER_UNIT; v += TF_THREADS) {
      const int unit = v / V_PER_UNIT, off4 = v % V_PER_UNIT;  // powers of two: shifts
      const int q0 = g * SGN + unit * CH;                       // first series of the run
      float4 x = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (q0 < n_series) {
        const float *src;
        if (PLANAR) {
          const int st = q0 / channels, ch = q0 - st * channels;
          src = in + (int64_t) st * in_ss + (int64_t) ch * in_cs + j0;
        } else {
          src = in + (int64_t) (q0 / CH) * in_ss + (int64_t) j0 * CH;
        }
        x = POLICY ? ld_global_hint(reinterpret_cast<const float4 *>(src) + off4, pol)
                   : __ldg(reinterpret_cast<const float4 *>(src) + off4);
      }
      const float xv[4] = {x.x, x.y, x.z, x.w};
      const int e0 = off4 * 4;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        tile.at((e0 + k) / CH, unit * CH + ((e0 + k) % CH)) = xv[k];
    }
    __syncthreads();
    float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + row_first + j0) * SGN);
#pragma unroll 4
    for (int i = tid; i < ROWS * (SGN / 4); i += TF_THREADS) {
      const int row = i / (SGN / 4), c4 = i % (SGN / 4);
      dst[i] = tile.vec(row, c4);
    }
    __syncthreads();  // every thread's stores are issued (and the tile may be overwritten)
    if (tid == 0) {
      __threadfence();  // ... and visible device-wide before the count
      atomicAdd(ready + y, 1);
    }
  }
}

// Generic path: any strides / channel count / alignment, partial tiles and the zero padding.
__global__ void __launch_bounds__(256)
    espb_transpose_kernel(const float *__restrict__ in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                          int n_series, int n_in, float *__restrict__ xt, int64_t rows_cap, int row_first,
                          int j_begin, int pad_rows) {
  __shared__ float tile[TR_ROWS][SGN + 1];
  const int g = blockIdx.x;
  const int j0 = j_begin + blockIdx.y * TR_ROWS;  // first input frame of this tile
  const int tid = threadIdx.x;
  const int total_rows = n_in + pad_rows;
  // 0: frames contiguous (planar)  1: interleaved and the group covers whole streams  2: generic
  const int mapping = (in_fs == 1) ? 0 : ((in_cs == 1 && in_fs == channels && SGN % channels == 0) ? 1 : 2);
  for (int i = tid; i < SGN * TR_ROWS; i += 256) {
    int sl, t;
    if (mapping == 0) {
      sl = i / TR_ROWS;
      t = i - sl * TR_ROWS;
    } else if (mapping == 1) {
      const int per = TR_ROWS * channels;
      const int stl = i / per, r = i - stl * per;
      t = r / channels;
      sl = stl * channels + (r - t * channels);
    } else {
      t = i / SGN;
      sl = i - t * SGN;
    }
    const int q = g * SGN + sl, j = j0 + t;
    float v = 0.0f;
    if (q < n_series && j < n_in) {
      const int st = q / channels, ch = q - st * channels;
      v = __ldg(in + (int64_t) st * in_ss + (int64_t) ch * in_cs + (int64_t) j * in_fs);
    }
    tile[t][sl] = v;
  }
  __syncthreads();
  float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + row_first + j0) * SGN);
  for (int i = tid; i < TR_ROWS * (SGN / 4); i += 256) {
    const int t = i / (SGN / 4), c4 = i - t * (SGN / 4);
    if (j0 + t < total_rows)
      dst[i] = make_float4(tile[t][c4 * 4], tile[t][c4 * 4 + 1], tile[t][c4 * 4 + 2], tile[t][c4 * 4 + 3]);
  }
}

// Small calls (real-time chunks): the carried frames, the new input and the zero padding of a call in ONE launch
// instead of a strided device copy plus two transposition kernels.  blockIdx.y < hist_tiles copies history rows
// (time-major to time-major), the other tiles are the generic transposing tiles.
__global__ void __launch_bounds__(256)
    espb_stage_small_kernel(const float *__restrict__ old_xt, int carry_row, int taps, int hist_tiles,
                            const float *__restrict__ in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                            int n_series, int n_in, float *__restrict__ xt, int64_t rows_cap, int pad_rows) {
  __shared__ float tile[TR_ROWS][SGN + 1];
  const int g = blockIdx.x;
  const int tid = threadIdx.x;
  if ((int) blockIdx.y < hist_tiles) {
    const int r0 = blockIdx.y * TR_ROWS;
    const float4 *src = reinterpret_cast<const float4 *>(old_xt + ((int64_t) g * rows_cap + carry_row + r0) * SGN);
    float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + r0) * SGN);
    for (int i = tid; i < TR_ROWS * (SGN / 4); i += 256)
      if (r0 + i / (SGN / 4) < taps)
        dst[i] = __ldg(src + i);
    return;
  }
  const int j0 = ((int) blockIdx.y - hist_tiles) * TR_ROWS;
  const int total_rows = n_in + pad_rows;
  const int mapping = (in_fs == 1) ? 0 : ((in_cs == 1 && in_fs == channels && SGN % channels == 0) ? 1 : 2);
  for (int i = tid; i < SGN * TR_ROWS; i += 256) {
    int sl, t;
    if (mapping == 0) {
      sl = i / TR_ROWS;
      t = i - sl * TR_ROWS;
    } else if (mapping == 1) {
      const int per = TR_ROWS * channels;
      const int stl = i / per, r = i - stl * per;
      t = r / channels;
      sl = stl * channels + (r - t * channels);
    } else {
      t = i / SGN;
      sl = i - t * SGN;
    }
    const int q = g * SGN + sl, j = j0 + t;
    float v = 0.0f;
    if (q < n_series && j < n_in) {
      const int st = q / channels, ch = q - st * channels;
      v = __ldg(in + (int64_t) st * in_ss + (int64_t) ch * in_cs + (int64_t) j * in_fs);
    }
    tile[t][sl] = v;
  }
  __syncthreads();
  float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + taps + j0) * SGN);
  for (int i = tid; i < TR_ROWS * (SGN / 4); i += 256) {
    const int t = i / (SGN / 4), c4 = i - t * (SGN / 4);
    if (j0 + t < total_rows)
      dst[i] = make_float4(tile[t][c4 * 4], tile[t][c4 * 4 + 1], tile[t][c4 * 4 + 2], tile[t][c4 * 4 + 3]);
  }
}

// Planar input given as one pointer per (stream, channel) plane — the reference's resampleProcess signature
// (`const float *const *inputs`, include/art_resampler.h:36-37): separately allocated channel buffers.  Same tiling
// as the generic kernel (frames contiguous per plane: a warp reads 32 consecutive frames of one plane).
__global__ void __launch_bounds__(256)
    espb_transpose_ptr_kernel(const float *const *__restrict__ planes, int n_series, int n_in,
                              float *__restrict__ xt, int64_t rows_cap, int row_first, int j_begin, int pad_rows) {
  __shared__ float tile[TR_ROWS][SGN + 1];
  const int g = blockIdx.x;
  const int j0 = j_begin + blockIdx.y * TR_ROWS;
  const int tid = threadIdx.x;
  const int total_rows = n_in + pad_rows;
  for (int i = tid; i < SGN * TR_ROWS; i += 256) {
    const int sl = i / TR_ROWS, t = i - sl * TR_ROWS;
    const int q = g * SGN + sl, j = j0 + t;
    float v = 0.0f;
    if (q < n_series && j < n_in)
      v = __ldg(planes[q] + j);
    tile[t][sl] = v;
  }
  __syncthreads();
  float4 *dst = reinterpret_cast<float4 *>(xt + ((int64_t) g * rows_cap + row_first + j0) * SGN);
  for (int i = tid; i < TR_ROWS * (SGN / 4); i += 256) {
    const int t = i / (SGN / 4), c4 = i - t * (SGN / 4);
    if (j0 + t < total_rows)
      dst[i] = make_float4(tile[t][c4 * 4], tile[t][c4 * 4 + 1], tile[t][c4 * 4 + 2], tile[t][c4 * 4 + 3]);
  }
}

__global__ void __launch_bounds__(256)
    espb_untranspose_ptr_kernel(const float *__restrict__ tm, int64_t rows_cap, int row_first, int j_begin,
                                int n_rows, float *const *__restrict__ planes, int n_series) {
  __shared__ float tile[TR_ROWS][SGN + 1];
  const int g = blockIdx.x;
  const int j0 = j_begin + blockIdx.y * TR_ROWS;
  const int tid = threadIdx.x;
  const float *src = tm + ((int64_t) g * rows_cap + row_first + j0) * SGN;
  for (int i = tid; i < TR_ROWS * SGN; i += 256) {
    const int t = i / SGN, sl = i - t * SGN;
    tile[t][sl] = (j0 + t < n_rows) ? __ldg(src + i) : 0.0f;
  }
  __syncthreads();
  for (int i = tid; i < SGN * TR_ROWS; i += 256) {
    const int sl = i / TR_ROWS, t = i - sl * TR_ROWS;
    const int q = g * SGN + sl, j = j0 + t;
    if (q < n_series && j < n_rows)
      planes[q][j] = tile[t][sl];
  }
}

// ---------------------------------------------------------------------------------
// Inverse stage: time-major tm[group][row][128] -> caller layout.  Same tiling as the transposing
// stage: 128-bit loads along series, 128-bit stores along time.
// ---------------------------------------------------------------------------------
template <int CH, bool PLANAR>
__global__ void __launch_bounds__(TF_THREADS)
    espb_untranspose_fast_kernel(const float *__restrict__ tm, int64_t rows_cap, int row_first, float *__restrict__ out,
                                 int64_t out_ss, int64_t out_cs, int channels, int n_series) {
  __shared__ __align__(16) float tile_s[TF_ROWS * SGN];
  const SwzTile tile{tile_s};
  const int g = blockIdx.x;
  const int j0 = blockIdx.y * TF_ROWS;
  const int tid = threadIdx.x;
  const float4 *src = reinterpret_cast<const float4 *>(tm + ((int64_t) g * rows_cap + row_first + j0) * SGN);
  constexpr int UNITS = SGN / CH;
  constexpr int V_PER_UNIT = TF_ROWS * CH / 4;
  // (a group with few series reads and lays out only the 16-byte units that hold series: transpose_fast_tile)
  const int units = (n_series - g * SGN + 3) / 4 < SGN / 4 ? (n_series - g * SGN + 3) / 4 : SGN / 4;
  const int runs_here = (units * 4 + CH - 1) / CH < UNITS ? (units * 4 + CH - 1) / CH : UNITS;
#pragma unroll 4
  for (int i = tid; i < TF_ROWS * (SGN / 4); i += TF_THREADS) {
    const int t = i / (SGN / 4), c4 = i % (SGN / 4);
    if (c4 < units)
      tile.vec(t, c4) = __ldg(src + i);
  }
  __syncthreads();
#pragma unroll 4
  for (int v = tid; v < runs_here * V_PER_UNIT; v += TF_THREADS) {
    const int unit = v / V_PER_UNIT, off4 = v % V_PER_UNIT;
    const int q0 = g * SGN + unit * CH;
    if (q0 >= n_series)
      continue;
    float *dst;
    if (PLANAR) {
      const int st = q0 / channels, ch = q0 - st * channels;
      dst = out + (int64_t) st * out_ss + (int64_t) ch * out_cs + j0;
    } else {
      dst = out + (int64_t) (q0 / CH) * out_ss + (int64_t) j0 * CH;
    }
    const int e0 = off4 * 4;
    float x[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int e = e0 + k;
      x[k] = tile.at(e / CH, unit * CH + (e % CH));
    }
    reinterpret_cast<float4 *>(dst)[off4] = make_float4(x[0], x[1], x[2], x[3]);
  }
}

__global__ void __launch_bounds__(256)
    espb_untranspose_kernel(const float *__restrict__ tm, int64_t rows_cap, int row_first, int j_begin, int n_rows,
                            float *__restrict__ out, int64_t out_ss, int64_t out_cs, int64_t out_fs, int channels,
                            int n_series) {
  __shared__ float tile[TR_ROWS][SGN + 1];
  const int g = blockIdx.x;
  const int j0 = j_begin + blockIdx.y * TR_ROWS;
  const int tid = threadIdx.x;
  const float *src = tm + ((int64_t) g * rows_cap + row_first + j0) * SGN;
  for (int i = tid; i < TR_ROWS * SGN; i += 256) {
    const int t = i / SGN, sl = i - t * SGN;
    tile[t][sl] = (j0 + t < n_rows) ? __ldg(src + i) : 0.0f;
  }
  __syncthreads();
  const int mapping = (out_fs == 1) ? 0 : ((out_cs == 1 && out_fs == channels && SGN % channels == 0) ? 1 : 2);
  for (int i = tid; i < SGN * TR_ROWS; i += 256) {
    int sl, t;
    if (mapping == 0) {
      sl = i / TR_ROWS;
      t = i - sl * TR_ROWS;
    } else if (mapping == 1) {
      const int per = TR_ROWS * channels;
      const int stl = i / per, r = i - stl * per;
      t = r / channels;
      sl = stl * channels + (r - t * channels);
    } else {
      t = i / SGN;
      sl = i - t * SGN;
    }
    const int q = g * SGN + sl, j = j0 + t;
    if (q < n_series && j < n_rows) {
      const int st = q / channels, ch = q - st * channels;
      out[(int64_t) st * out_ss + (int64_t) ch * out_cs + (int64_t) j * out_fs] = tile[t][sl];
    }
  }
}

// ---------------------------------------------------------------------------------
// Resampler
// ---------------------------------------------------------------------------------
// BPP: output blocks (= warps) per pass; NST: ring stages; CJ: rows per chunk.  Four 4-warp CTAs per SM: measured 5 %
// faster than two 8-warp CTAs at C2 (shorter passes: less idle time at the pass edges, twice the x traffic from L2).
// (Results in the caller's layout are written once and never read back, but streaming / evict-first stores are not
// the answer: __stcs and st.global.L2::cache_hint(evict_first) were both measured 5 % slower — 7.39 against 7.02 ms —
// a lane's 64 contiguous bytes leave as four 16-byte stores and the hinted forms give up their merging in L2.)
__device__ __forceinline__ void out_store4(float4 *p, float4 v) { *p = v; }

template <bool EXACT, bool TMCAP>
__global__ void __launch_bounds__(kResampleWarps * 32, 16 / kResampleWarps) espb_resample_kernel(const ResampleParams p) {
  constexpr int BPP = kResampleWarps, NST = kResampleStages, CJ = kResampleChunkRows;
  constexpr int NTHREADS = BPP * 32;
  constexpr int STAGES = NST;
  constexpr int MAXC = kMaxChunksPerCta;
  static_assert(kMaxPassesPerCta * BPP * sizeof(int2) <= (size_t) NST * CJ * SGN * sizeof(float), "set-up table");
  constexpr int XS_STAGE = CJ * SGN;                // floats
  constexpr int GS_STAGE = CJ * BPP * kGRowFloats;  // floats
  constexpr uint32_t X_BYTES = XS_STAGE * sizeof(float), G_BYTES = GS_STAGE * sizeof(float);

  extern __shared__ __align__(128) unsigned char smem_raw[];
  float *gs = reinterpret_cast<float *>(smem_raw);                        // [STAGES][CJ][BPP][16]
  float *xs = gs + STAGES * GS_STAGE;                                     // [STAGES][CJ][128]
  uint64_t *full = reinterpret_cast<uint64_t *>(xs + STAGES * XS_STAGE);  // [STAGES] TMA landed
  int *done = reinterpret_cast<int *>(full + STAGES);                     // [2*STAGES] warps done with a stage
  int32_t *jtab = reinterpret_cast<int32_t *>(done + 2 * STAGES);         // [MAXC] first input row of each chunk
  // [MAXC][BPP] what warp w does in chunk c: row groups [r0, r1), end-of-pass flag
  uint16_t *rtab = reinterpret_cast<uint16_t *>(jtab + MAXC);
  // [BPP][NB] schedule entries of the block each warp is finishing, fetched by cp.async during the pass's last chunk
  OutEntry *etab = reinterpret_cast<OutEntry *>(rtab + MAXC * BPP);
  int32_t *hdr = reinterpret_cast<int32_t *>(etab + BPP * NB);  // [4] CTA constants for the refilling lane
  int2 *wtab = reinterpret_cast<int2 *>(smem_raw);  // set-up only (the ring is not in use yet): [MAXP][BPP] windows

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int group = blockIdx.x;
  const int T = p.taps;

  // ---- which passes / chunks this CTA sweeps
  const int pass_first = p.pass_first + blockIdx.y * p.passes_per_cta;
  int pass_last = pass_first + p.passes_per_cta;
  if (pass_last > p.pass_end)
    pass_last = p.pass_end;
  const int chunk_first = p.pass_chunk_begin[pass_first], chunk_last = p.pass_chunk_begin[pass_last];
  const int n_chunks = __shfl_sync(0xffffffffu, chunk_last - chunk_first, 0);  // warp-uniform by construction

  // ---- build the signal-independent tables this CTA needs (no global loads, no index arithmetic in the main loop)
  for (int i = tid; i < (pass_last - pass_first) * BPP; i += NTHREADS) {  // window [lo, hi) of (pass, warp)
    const int o0 = ((pass_first + i / BPP) * BPP + (i % BPP)) * NB;
    int2 w = make_int2(0, 0);
    if (o0 < p.n_out) {
      const int o1 = (o0 + NB <= p.n_out ? o0 + NB : p.n_out) - 1;
      w.x = p.outs[o0].ws;
      w.y = p.outs[o1].ws + T;
    }
    wtab[i] = w;
  }
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    hdr[0] = chunk_first - p.g_chunk_base;
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  for (int i = tid; i < n_chunks; i += NTHREADS) {
    const ChunkEntry ce = p.chunks[chunk_first + i];
    const bool last_of_pass = (i + 1 == n_chunks) || (p.chunks[chunk_first + i + 1].pass != ce.pass);
    jtab[i] = ce.j_start;
    // rows of this chunk inside each warp's window, in groups of RG (rows outside it only multiply zeros)
#pragma unroll
    for (int w = 0; w < BPP; ++w) {
      const int2 win = wtab[(ce.pass - pass_first) * BPP + w];
      int r0 = win.x - ce.j_start, r1 = win.y - ce.j_start;
      r0 = r0 < 0 ? 0 : (r0 / RG);
      r1 = r1 > CJ ? CJ / RG : ((r1 + RG - 1) / RG);
      if (r0 > CJ / RG)
        r0 = CJ / RG;
      if (r1 < r0)
        r1 = r0;
      rtab[i * BPP + w] = (uint16_t) (r0 | (r1 << 4) | (last_of_pass ? kPassDone : 0));
    }
  }
  __syncthreads();

  // Fill stage c % STAGES with chunk c: two TMA bulk copies (16 KB of G, 16 KB of x) on one mbarrier.
  // (Addresses are rebuilt from the parameters here — one lane runs this once per chunk — rather than held in
  // registers across the FMA loop.)
  auto issue_chunk = [&](int c) {
    const int st = c % STAGES;
    const float *xt_group = p.xt + (int64_t) blockIdx.x * p.xt_rows * SGN;
    mbar_expect_tx(&full[st], X_BYTES + G_BYTES);
    tma_bulk_g2s(gs + st * GS_STAGE, p.G + (size_t) (hdr[0] + c) * GS_STAGE, G_BYTES, &full[st]);
    tma_bulk_g2s(xs + st * XS_STAGE, xt_group + (int64_t) (jtab[c] + T) * SGN, X_BYTES, &full[st]);
  };
  // Staging overlap: this grid may have started while the transposing kernel is still writing xt.  Wait for the
  // row tiles this CTA reads (one poller per tile; the writers never wait for anything and are all resident, so
  // this always ends — the trap only turns a protocol error into a loud failure instead of a hung device).
  if (p.ready != nullptr && n_chunks > 0) {
    const int j_hi = jtab[n_chunks - 1] + CJ - 1;
    if (j_hi >= 0) {
      const int j_lo = jtab[0];
      const int y_lo = j_lo > 0 ? j_lo / kReadyTileRows : 0;
      int y_hi = j_hi / kReadyTileRows;
      y_hi = y_hi < p.ready_tiles ? y_hi : p.ready_tiles - 1;
      for (int y = y_lo + tid; y <= y_hi; y += NTHREADS) {
        const long long t0 = clock64();
        while (ld_acquire_gpu(p.ready + y) < p.ready_target) {
          __nanosleep(200);
          if (clock64() - t0 > (4ll << 31))  // ~4 s
            __trap();
        }
      }
    }
    __syncthreads();
    fence_proxy_async();
  }
  if (tid == 0)
    for (int c = 0; c < STAGES && c < n_chunks; ++c)
      issue_chunk(c);

  // accumulators [series e][output n] x (filter 0, filter 1): packed pairs in fast mode, scalars in exact mode
  float2 acc2[EXACT ? 1 : 4][EXACT ? 1 : NB];
  float acc1[EXACT ? 4 : 1][EXACT ? NB : 1][2];
  auto clear_acc = [&]() {
    if constexpr (EXACT) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int n = 0; n < NB; ++n)
          acc1[e][n][0] = acc1[e][n][1] = 0.0f;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int n = 0; n < NB; ++n)
          acc2[e][n] = make_float2(0.0f, 0.0f);
    }
  };
  clear_acc();

  int cur_pass = pass_first;
  uint32_t role_next = rtab[warp];
  for (int c = 0; c < n_chunks; ++c) {
    const int st = c % STAGES;
    const uint32_t role = role_next;
    const bool pass_done = (role & kPassDone) != 0;
    const int r0 = role & 15, r1 = (role >> 4) & 15;
    if (pass_done && lane < NB) {  // the epilogue's schedule entries: global -> shared, no register held meanwhile
      int o = (cur_pass * BPP + warp) * NB + lane;
      o = o < p.n_out ? o : p.n_out - 1;
      cp_async_16(&etab[warp * NB + lane], &p.outs[o]);
    }
    mbar_wait(&full[st], (uint32_t) ((c / STAGES) & 1));
    {
      const float *xrow = xs + st * XS_STAGE + lane * 4;
      const float *grow = gs + st * GS_STAGE + warp * kGRowFloats;
      for (int jb = r0; jb < r1; ++jb) {
        const float *xb = xrow + jb * RG * SGN;
        const float *gb = grow + jb * RG * BPP * kGRowFloats;
#pragma unroll
        for (int jj = 0; jj < RG; ++jj) {
          const float4 xv = *reinterpret_cast<const float4 *>(xb + jj * SGN);
          if constexpr (EXACT) {
            const float4 *gp = reinterpret_cast<const float4 *>(gb + jj * BPP * kGRowFloats);
            const float4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];
            const float x4[4] = {xv.x, xv.y, xv.z, xv.w};
            const float g16[16] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w,
                                   g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z, g3.w};
#pragma unroll
            for (int n = 0; n < NB; ++n)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                acc1[e][n][0] = mac<true>(g16[2 * n], x4[e], acc1[e][n][0]);
                acc1[e][n][1] = mac<true>(g16[2 * n + 1], x4[e], acc1[e][n][1]);
              }
          } else {
            const float4 *gp = reinterpret_cast<const float4 *>(gb + jj * BPP * kGRowFloats);
            const float4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];
            const float x4[4] = {xv.x, xv.y, xv.z, xv.w};
            const float2 gg[NB] = {make_float2(g0.x, g0.y), make_float2(g0.z, g0.w), make_float2(g1.x, g1.y),
                                   make_float2(g1.z, g1.w), make_float2(g2.x, g2.y), make_float2(g2.z, g2.w),
                                   make_float2(g3.x, g3.y), make_float2(g3.z, g3.w)};  // (filter 0, filter 1) pairs
#pragma unroll
            for (int n = 0; n < NB; ++n)
#pragma unroll
              for (int e = 0; e < 4; ++e)
                acc2[e][n] = fma2(gg[n], x4[e], acc2[e][n]);
          }
        }
      }
    }

    // Release the stage.  The last of the BPP warps to get here re-arms it and issues the refill
    // (chunk c + STAGES); nobody waits for anybody.  (A designated refilling warp that waits for the others on an
    // "empty" mbarrier was measured 17 % slower: it cannot run ahead while it waits.)
    role_next = rtab[(c + 1) * BPP + warp];  // (one entry past the CTA's last chunk is still inside the table)
    __syncwarp();
    if (lane == 0) {
      if (smem_arrive(&done[st]) == BPP - 1) {
        done[st] = 0;  // published to the other warps by the release of the mbarrier arrive below
        if (c + STAGES < n_chunks)
          issue_chunk(c + STAGES);
      }
    }

    // ---- end of pass: blend, store, clear
    if (pass_done) {
      cp_async_wait_all();
      __syncwarp();
      const int o0 = (cur_pass * BPP + warp) * NB;
      const OutEntry *et = etab + warp * NB;
      float v[4][NB];
#pragma unroll
      for (int n = 0; n < NB; ++n) {
        const OutEntry en = et[n];  // one broadcast LDS.128
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float sum1, sum2;
          if constexpr (EXACT) {
            sum1 = acc1[e][n][0];
            sum2 = acc1[e][n][1];
          } else {
            sum1 = acc2[e][n].x;
            sum2 = acc2[e][n].y;
          }
          if (en.kind == kKindBlend) {  // art_resampler.cpp:450, un-fused
            v[e][n] = __fadd_rn(__fmul_rn(sum2, en.w), __fmul_rn(sum1, __fsub_rn(1.0f, en.w)));
          } else if (en.kind == kKindSingle) {
            v[e][n] = sum1;
          } else {  // pass-through: *source (art_resampler.cpp:426,440) = tap numTaps/2-1 of the window
            v[e][n] = p.xt[((int64_t) group * p.xt_rows + (en.ws + T / 2 - 1 + T)) * SGN + lane * 4 + e];
          }
        }
      }
      const int series0 = group * SGN + lane * 4;
      if (TMCAP && p.out_vec == kOutVecTimeMajor) {  // scratch for a following in-library stage: one 16-byte store per lane
        float *dst = p.out_tm + ((int64_t) group * p.out_tm_rows + o0) * SGN + lane * 4;
#pragma unroll
        for (int n = 0; n < NB; ++n)
          if (o0 + n < p.n_out)
            *reinterpret_cast<float4 *>(dst + n * SGN) = make_float4(v[0][n], v[1][n], v[2][n], v[3][n]);
      } else if (p.out_vec == kOutVecStereo && o0 + NB <= p.n_out) {
        // interleaved stereo: a lane owns two streams x 8 frames x 2 channels = 2 x 64 contiguous bytes
        float *dst = p.out + (int64_t) (series0 >> 1) * p.out_ss + (int64_t) o0 * 2;
        if (series0 < p.n_series) {
#pragma unroll
          for (int k = 0; k < NB / 2; ++k)
            out_store4(reinterpret_cast<float4 *>(dst) + k, make_float4(v[0][2 * k], v[1][2 * k], v[0][2 * k + 1], v[1][2 * k + 1]));
        }
        if (series0 + 2 < p.n_series) {
          dst += p.out_ss;
#pragma unroll
          for (int k = 0; k < NB / 2; ++k)
            out_store4(reinterpret_cast<float4 *>(dst) + k, make_float4(v[2][2 * k], v[3][2 * k], v[2][2 * k + 1], v[3][2 * k + 1]));
        }
      } else if (p.out_vec == kOutVecFrame4 && o0 + NB <= p.n_out) {
        // interleaved, channel count a multiple of 4: the lane's 4 series are 16 contiguous bytes of every frame
        if (series0 < p.n_series) {
          const int sidx = series0 / p.channels, ch = series0 - sidx * p.channels;
          float *dst = p.out + (int64_t) sidx * p.out_ss + ch + (int64_t) o0 * p.channels;
#pragma unroll
          for (int n = 0; n < NB; ++n)
            out_store4(reinterpret_cast<float4 *>(dst + n * p.channels), make_float4(v[0][n], v[1][n], v[2][n], v[3][n]));
        }
      } else if (p.out_vec == kOutVecPlanar && o0 + NB <= p.n_out) {
        // frames contiguous per series (planar, or interleaved mono): 8 frames = 32 contiguous bytes per series
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int series = series0 + e;
          if (series < p.n_series) {
            const int sidx = series / p.channels, ch = series - sidx * p.channels;
            float4 *dst = reinterpret_cast<float4 *>(p.out + (int64_t) sidx * p.out_ss + (int64_t) ch * p.out_cs + o0);
            out_store4(dst, make_float4(v[e][0], v[e][1], v[e][2], v[e][3]));
            out_store4(dst + 1, make_float4(v[e][4], v[e][5], v[e][6], v[e][7]));
          }
        }
      } else {  // any layout, partial blocks
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int series = series0 + e;
          if (series < p.n_series) {
            const int sidx = series / p.channels, ch = series - sidx * p.channels;
            float *dst = p.out + (int64_t) sidx * p.out_ss + (int64_t) ch * p.out_cs + (int64_t) o0 * p.out_fs;
#pragma unroll
            for (int n = 0; n < NB; ++n)
              if (o0 + n < p.n_out)
                dst[(int64_t) n * p.out_fs] = v[e][n];
          }
        }
      }
      clear_acc();
      ++cur_pass;
    }
  }
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
size_t resample_smem_bytes(int bpp, int grf) {
  constexpr int stages = kResampleStages, CJ = kResampleChunkRows;
  return (size_t) stages * (CJ * bpp * grf + CJ * SGN) * sizeof(float) + stages * sizeof(uint64_t) +
         stages * sizeof(uint64_t) + kMaxChunksPerCta * (sizeof(int32_t) + bpp * sizeof(uint16_t)) +
         (size_t) bpp * NB * sizeof(OutEntry) + 4 * sizeof(int32_t);
}

size_t g_chunk_floats(int bpp, int grf) { return (size_t) kResampleChunkRows * bpp * grf; }

cudaError_t launch_expand_schedule(const SchedSegment *segs, int n_segs, OutEntry *outs, int n, int n_filters,
                                   bool lowpass, bool interp, cudaStream_t stream) {
  if (n <= 0 || n_segs <= 0)
    return cudaSuccess;
  espb_expand_schedule_kernel<<<(n + 255) / 256, 256, 0, stream>>>(segs, n_segs, outs, n, (float) n_filters, lowpass,
                                                                   interp);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_expand(const float *bank, const OutEntry *outs, const ChunkEntry *chunks, float *G,
                          int chunk_first, int n_chunks, int n_out, int taps, int bpp, cudaStream_t stream,
                          int grf) {
  if (n_chunks <= 0)
    return cudaSuccess;
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess)
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  static const int per_sm = getenv("ESPB_EXPAND_CTAS") ? atoi(getenv("ESPB_EXPAND_CTAS")) : 64;
  const int grid = n_chunks < sms * per_sm ? n_chunks : sms * per_sm;  // (a few chunks per CTA at most)
  espb_expand_kernel<<<grid, kExpandThreads, 0, stream>>>(bank, outs, chunks, G, chunk_first, n_chunks, n_out, taps,
                                                          bpp, grf);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_transpose(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels, int n_series,
                             int n_in, float *xt, int64_t rows_cap, int row_first, int pad_rows,
                             cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  if (n_groups <= 0 || n_in + pad_rows <= 0)
    return cudaSuccess;
  // full 64-row tiles through the fast kernel when the layout allows it, with the widest loads the alignment allows
  int fast_rows = 0;
  const bool interleaved = (in_cs == 1 && in_fs == channels);
  const bool planar = (in_fs == 1);
  // rows start at in + stream * in_ss (+ channel * in_cs when planar) + a multiple of 64 frames
  const bool cs_ok4 = interleaved || in_cs % 4 == 0, cs_ok2 = interleaved || in_cs % 2 == 0;
  int vec = 1;
  if ((uintptr_t) in % 16 == 0 && in_ss % 4 == 0 && cs_ok4)
    vec = 4;
  else if ((uintptr_t) in % 8 == 0 && in_ss % 2 == 0 && cs_ok2)
    vec = 2;
  const bool fast_layout = (interleaved && (channels == 1 || channels == 2 || channels == 4 || channels == 8)) || planar;
  if (n_in >= TF_ROWS && fast_layout) {
    // a slice starting at tile y0 reads from frame y0 * TF_ROWS on (in_fs = channels or 1 here) and writes the rows
    // from row_first + y0 * TF_ROWS on
    cudaError_t e = for_each_y_slice(n_in / TF_ROWS, [&](int y0, int ny) {
      const dim3 grid(n_groups, ny);
      const float *in_y = in + (int64_t) y0 * TF_ROWS * in_fs;
      const int row_y = row_first + y0 * TF_ROWS;
#define ESPB_TR(CH_, PL_)                                                                                             \
  (vec == 4 ? espb_transpose_fast_kernel<CH_, PL_, 4><<<grid, TF_THREADS, 0, stream>>>(in_y, in_ss, in_cs, channels,   \
                                                                                      n_series, xt, rows_cap, row_y)   \
   : vec == 2                                                                                                         \
       ? espb_transpose_fast_kernel<CH_, PL_, 2><<<grid, TF_THREADS, 0, stream>>>(in_y, in_ss, in_cs, channels,        \
                                                                                 n_series, xt, rows_cap, row_y)        \
       : espb_transpose_fast_kernel<CH_, PL_, 1><<<grid, TF_THREADS, 0, stream>>>(in_y, in_ss, in_cs, channels,        \
                                                                                 n_series, xt, rows_cap, row_y))
      if (interleaved && channels == 1)
        ESPB_TR(1, false);
      else if (interleaved && channels == 2)
        ESPB_TR(2, false);
      else if (interleaved && channels == 4)
        ESPB_TR(4, false);
      else if (interleaved && channels == 8)
        ESPB_TR(8, false);
      else
        ESPB_TR(1, true);
#undef ESPB_TR
      count_launch();
      return cudaGetLastError();
    });
    if (e != cudaSuccess)
      return e;
    fast_rows = (n_in / TF_ROWS) * TF_ROWS;
  }
  cudaError_t e = launch_transpose_from(in, in_ss, in_cs, in_fs, channels, n_series, n_in, xt, rows_cap, row_first,
                                        fast_rows, pad_rows, stream);
  return e != cudaSuccess ? e : cudaGetLastError();
}

// The staging of a long call arranged for overlap with the resampler (see espb_transpose_flags_kernel): everything
// the flagged kernel does not cover (frames past the last full 32-row tile, the zero padding) goes first, then the
// counters are cleared, then the flagged kernel — which must be the last thing enqueued before the resampler.
// *n_tiles = row tiles it will signal; 0 = layout not covered, nothing was enqueued (use launch_transpose).
cudaError_t launch_transpose_flags(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                                   int n_series, int n_in, float *xt, int64_t rows_cap, int row_first, int pad_rows,
                                   int *ready, int ctas_per_sm, cudaStream_t stream, int *n_tiles) {
  *n_tiles = 0;
  const int n_groups = (n_series + SGN - 1) / SGN;
  const bool interleaved = (in_cs == 1 && in_fs == channels);
  const bool planar = (in_fs == 1);
  const bool cs_ok4 = interleaved || in_cs % 4 == 0;
  const bool covered = (interleaved && (channels == 1 || channels == 2 || channels == 4 || channels == 8)) || planar;
  if (n_groups <= 0 || n_in < kReadyTileRows || !covered || (uintptr_t) in % 16 != 0 || in_ss % 4 != 0 || !cs_ok4)
    return cudaSuccess;
  const int tiles_y = n_in / kReadyTileRows, fast_rows = tiles_y * kReadyTileRows;
  cudaError_t e = launch_transpose_from(in, in_ss, in_cs, in_fs, channels, n_series, n_in, xt, rows_cap, row_first,
                                        fast_rows, pad_rows, stream);
  if (e != cudaSuccess)
    return e;
  e = cudaMemsetAsync(ready, 0, (size_t) tiles_y * sizeof(int), stream);
  if (e != cudaSuccess)
    return e;
  int sms = 148, dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess)
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long total = (long) tiles_y * n_groups;
  // ctas_per_sm > 0: that many per SM (at most 4); < 0: -ctas_per_sm CTAs in all (never more than one wave)
  long resident = ctas_per_sm < 0 ? -ctas_per_sm : (long) sms * (ctas_per_sm < 1 ? 1 : (ctas_per_sm > 4 ? 4 : ctas_per_sm));
  if (resident > (long) sms * 4)
    resident = (long) sms * 4;
  static const bool evict_first = getenv("ESPB_STAGE_POLICY") == nullptr || atoi(getenv("ESPB_STAGE_POLICY")) != 0;
  const int grid = (int) (total < resident ? total : resident);
  // The resampler's CTAs can only join an SM that is already configured for their shared-memory carve-out (an SM
  // re-partitions L1 / shared memory only when idle): run this kernel under the same, maximal, carve-out.
#define ESPB_TRF1(CH_, PL_, POL_)                                                                               \
  do {                                                                                                          \
    static PerDeviceOnce once;                                                                                  \
    if (once.first())                                                                                           \
      cudaFuncSetAttribute(espb_transpose_flags_kernel<CH_, PL_, POL_>,                                         \
                           cudaFuncAttributePreferredSharedMemoryCarveout, (int) cudaSharedmemCarveoutMaxShared); \
    espb_transpose_flags_kernel<CH_, PL_, POL_><<<grid, TF_THREADS, 0, stream>>>(in, in_ss, in_cs, channels,    \
                                                                                 n_series, xt, rows_cap,        \
                                                                                 row_first, n_groups,           \
                                                                                 (int) total, ready);           \
  } while (0)
#define ESPB_TRF(CH_, PL_)        \
  do {                            \
    if (evict_first)              \
      ESPB_TRF1(CH_, PL_, true);  \
    else                          \
      ESPB_TRF1(CH_, PL_, false); \
  } while (0)
  if (interleaved && channels == 1)
    ESPB_TRF(1, false);
  else if (interleaved && channels == 2)
    ESPB_TRF(2, false);
  else if (interleaved && channels == 4)
    ESPB_TRF(4, false);
  else if (interleaved && channels == 8)
    ESPB_TRF(8, false);
  else
    ESPB_TRF(1, true);
#undef ESPB_TRF1
#undef ESPB_TRF
  count_launch();
  *n_tiles = tiles_y;
  return cudaGetLastError();
}

cudaError_t launch_stage_small(const float *old_xt, int carry_row, int taps, const float *in, int64_t in_ss,
                               int64_t in_cs, int64_t in_fs, int channels, int n_series, int n_in, float *xt,
                               int64_t rows_cap, int pad_rows, cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  if (n_groups <= 0)
    return cudaSuccess;
  const int hist_tiles = (taps + TR_ROWS - 1) / TR_ROWS;
  dim3 grid(n_groups, hist_tiles + (n_in + pad_rows + TR_ROWS - 1) / TR_ROWS);
  espb_stage_small_kernel<<<grid, 256, 0, stream>>>(old_xt, carry_row, taps, hist_tiles, in, in_ss, in_cs, in_fs,
                                                    channels, n_series, n_in, xt, rows_cap, pad_rows);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_transpose_ptrs(const float *const *planes_dev, int n_series, int n_in, float *xt, int64_t rows_cap,
                                  int row_first, int pad_rows, cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  if (n_groups <= 0 || n_in + pad_rows <= 0)
    return cudaSuccess;
  return for_each_y_slice((n_in + pad_rows + TR_ROWS - 1) / TR_ROWS, [&](int y0, int ny) {
    espb_transpose_ptr_kernel<<<dim3(n_groups, ny), 256, 0, stream>>>(planes_dev, n_series, n_in, xt, rows_cap,
                                                                      row_first, y0 * TR_ROWS, pad_rows);
    count_launch();
    return cudaGetLastError();
  });
}

cudaError_t launch_untranspose_ptrs(const float *tm, int64_t rows_cap, int row_first, int n_rows,
                                    float *const *planes_dev, int n_series, cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  if (n_groups <= 0 || n_rows <= 0)
    return cudaSuccess;
  return for_each_y_slice((n_rows + TR_ROWS - 1) / TR_ROWS, [&](int y0, int ny) {
    espb_untranspose_ptr_kernel<<<dim3(n_groups, ny), 256, 0, stream>>>(tm, rows_cap, row_first, y0 * TR_ROWS, n_rows,
                                                                        planes_dev, n_series);
    count_launch();
    return cudaGetLastError();
  });
}

// generic kernels only, starting at frame j_begin (used for the tails after the fused PCM tiles)
cudaError_t launch_transpose_from(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                                  int n_series, int n_in, float *xt, int64_t rows_cap, int row_first, int j_begin,
                                  int pad_rows, cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  const int rest = n_in + pad_rows - j_begin;
  if (n_groups <= 0 || rest <= 0)
    return cudaSuccess;
  return for_each_y_slice((rest + TR_ROWS - 1) / TR_ROWS, [&](int y0, int ny) {
    espb_transpose_kernel<<<dim3(n_groups, ny), 256, 0, stream>>>(in, in_ss, in_cs, in_fs, channels, n_series, n_in, xt,
                                                                  rows_cap, row_first, j_begin + y0 * TR_ROWS,
                                                                  pad_rows);
    count_launch();
    return cudaGetLastError();
  });
}

cudaError_t launch_untranspose_from(const float *tm, int64_t rows_cap, int row_first, int j_begin, int n_rows,
                                    float *out, int64_t out_ss, int64_t out_cs, int64_t out_fs, int channels,
                                    int n_series, cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  const int rest = n_rows - j_begin;
  if (n_groups <= 0 || rest <= 0)
    return cudaSuccess;
  return for_each_y_slice((rest + TR_ROWS - 1) / TR_ROWS, [&](int y0, int ny) {
    espb_untranspose_kernel<<<dim3(n_groups, ny), 256, 0, stream>>>(tm, rows_cap, row_first, j_begin + y0 * TR_ROWS,
                                                                    n_rows, out, out_ss, out_cs, out_fs, channels,
                                                                    n_series);
    count_launch();
    return cudaGetLastError();
  });
}

cudaError_t launch_untranspose(const float *tm, int64_t rows_cap, int row_first, int n_rows, float *out,
                               int64_t out_ss, int64_t out_cs, int64_t out_fs, int channels, int n_series,
                               cudaStream_t stream) {
  const int n_groups = (n_series + SGN - 1) / SGN;
  if (n_groups <= 0 || n_rows <= 0)
    return cudaSuccess;
  int fast_rows = 0;
  const bool aligned = ((uintptr_t) out % 16 == 0) && (out_ss % 4 == 0);
  const bool interleaved = (out_cs == 1 && out_fs == channels);
  const bool planar = (out_fs == 1) && (out_cs % 4 == 0);
  const bool fast_layout = (interleaved && (channels == 1 || channels == 2 || channels == 4 || channels == 8)) || planar;
  if (aligned && n_rows >= TF_ROWS && fast_layout) {
    // a slice starting at tile y0 reads the rows from row_first + y0 * TF_ROWS on and writes from frame y0 * TF_ROWS
    // on (out_fs = channels or 1 here)
    cudaError_t e = for_each_y_slice(n_rows / TF_ROWS, [&](int y0, int ny) {
      const dim3 grid(n_groups, ny);
      const int row_y = row_first + y0 * TF_ROWS;
      float *out_y = out + (int64_t) y0 * TF_ROWS * out_fs;
      if (interleaved && channels == 1)
        espb_untranspose_fast_kernel<1, false><<<grid, TF_THREADS, 0, stream>>>(tm, rows_cap, row_y, out_y, out_ss,
                                                                                out_cs, channels, n_series);
      else if (interleaved && channels == 2)
        espb_untranspose_fast_kernel<2, false><<<grid, TF_THREADS, 0, stream>>>(tm, rows_cap, row_y, out_y, out_ss,
                                                                                out_cs, channels, n_series);
      else if (interleaved && channels == 4)
        espb_untranspose_fast_kernel<4, false><<<grid, TF_THREADS, 0, stream>>>(tm, rows_cap, row_y, out_y, out_ss,
                                                                                out_cs, channels, n_series);
      else if (interleaved && channels == 8)
        espb_untranspose_fast_kernel<8, false><<<grid, TF_THREADS, 0, stream>>>(tm, rows_cap, row_y, out_y, out_ss,
                                                                                out_cs, channels, n_series);
      else
        espb_untranspose_fast_kernel<1, true><<<grid, TF_THREADS, 0, stream>>>(tm, rows_cap, row_y, out_y, out_ss,
                                                                               out_cs, channels, n_series);
      count_launch();
      return cudaGetLastError();
    });
    if (e != cudaSuccess)
      return e;
    fast_rows = (n_rows / TF_ROWS) * TF_ROWS;
  }
  cudaError_t e = launch_untranspose_from(tm, rows_cap, row_first, fast_rows, n_rows, out, out_ss, out_cs, out_fs,
                                          channels, n_series, stream);
  return e != cudaSuccess ? e : cudaGetLastError();
}

template <bool EXACT, bool TMCAP>
static cudaError_t launch_resample_t(const ResampleParams &p, int n_groups, int n_ctas_y, cudaStream_t stream) {
  const size_t smem = resample_smem_bytes(kResampleWarps);
  static PerDeviceOnce once;
  if (once.first()) {
    cudaError_t e = cudaFuncSetAttribute(espb_resample_kernel<EXACT, TMCAP>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess)
      return e;
    // four CTAs per SM need the full 228 KB carve-out (the default heuristic sizes it for one)
    e = cudaFuncSetAttribute(espb_resample_kernel<EXACT, TMCAP>, cudaFuncAttributePreferredSharedMemoryCarveout,
                             (int) cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess)
      return e;
    if (getenv("ESPB_DEBUG")) {
      int nb = 0;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, espb_resample_kernel<EXACT, TMCAP>, kResampleWarps * 32, smem);
      cudaFuncAttributes fa;
      cudaFuncGetAttributes(&fa, espb_resample_kernel<EXACT, TMCAP>);
      fprintf(stderr, "[espb] resample<%d,%d>: smem %zu B, %d regs, occupancy %d CTA/SM\n", (int) EXACT, (int) TMCAP,
              smem, fa.numRegs, nb);
    }
  }
  dim3 grid(n_groups, n_ctas_y);
  if (p.ready != nullptr) {
    // programmatic dependent of the kernel launched just before on this stream (espb_transpose_flags_kernel): the
    // CTAs start while it runs and synchronise with it through p.ready, not through the stream
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kResampleWarps * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, espb_resample_kernel<EXACT, TMCAP>, p);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
  }
  espb_resample_kernel<EXACT, TMCAP><<<grid, kResampleWarps * 32, smem, stream>>>(p);
  count_launch();
  return cudaGetLastError();
}

// one launch of the resampler over n_ctas_y CTA rows of passes from q.pass_first on
static cudaError_t launch_resample_slice(const ResampleParams &q, int n_groups, int n_ctas_y, bool exact, bool tm,
                                         cudaStream_t stream, bool non_interpolating) {
  if (non_interpolating)  // one filter per output: resample_ni_kernel.cu
    return launch_resample_ni(q, n_groups, n_ctas_y, exact, tm, stream);
  // TMCAP: the variant that can also write time-major scratch (kept apart: folding that branch into the
  // caller-layout variant costs it 1.4 % through register allocation)
  if (exact)
    return tm ? launch_resample_t<true, true>(q, n_groups, n_ctas_y, stream)
              : launch_resample_t<true, false>(q, n_groups, n_ctas_y, stream);
  return tm ? launch_resample_t<false, true>(q, n_groups, n_ctas_y, stream)
            : launch_resample_t<false, false>(q, n_groups, n_ctas_y, stream);
}

cudaError_t launch_resample(const ResampleParams &p, bool exact, cudaStream_t stream, bool non_interpolating) {
  const int n_groups = (p.n_series + SGN - 1) / SGN;
  const int n_passes = p.pass_end - p.pass_first;
  if (n_groups <= 0 || n_passes <= 0)
    return cudaSuccess;
  const int n_ctas_y_total = (n_passes + p.passes_per_cta - 1) / p.passes_per_cta;
  const bool tm = p.out_tm != nullptr;
  ResampleParams q = p;
  q.out_vec = tm ? kOutVecTimeMajor : kOutVecNone;
  // 128-bit stores when the caller's layout keeps a lane's results contiguous and aligned
  if (!tm && (uintptr_t) p.out % 16 == 0 && p.out_ss % 4 == 0) {
    if (p.out_fs == 1 && (p.out_cs % 4 == 0 || p.channels == 1))  // planar, or mono (no second channel plane)
      q.out_vec = kOutVecPlanar;
    else if (p.out_cs == 1 && p.out_fs == p.channels && p.channels == 2)
      q.out_vec = kOutVecStereo;
    else if (p.out_cs == 1 && p.out_fs == p.channels && p.channels % 4 == 0)
      q.out_vec = kOutVecFrame4;
  }
  // CTAs over passes ride on y: a slice starting at CTA row y0 starts at pass pass_first + y0 * passes_per_cta
  return for_each_y_slice(n_ctas_y_total, [&](int y0, int n_ctas_y) {
    ResampleParams qy = q;
    qy.pass_first = p.pass_first + y0 * p.passes_per_cta;
    return launch_resample_slice(qy, n_groups, n_ctas_y, exact, tm, stream, non_interpolating);
  });
}

}  // namespace espb
