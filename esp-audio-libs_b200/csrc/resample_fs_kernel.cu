// ART polyphase resampler — the few-series form ("lanes over time").
//
// The standard kernel (resample_kernel.cu) maps lanes to series: a warp owns 128 series and 8 outputs, and the
// coefficients of those outputs are a warp-uniform broadcast.  With a handful of series — the reference's own use,
// one stereo stream per context (include/resampler.h:64, art_resampler.cpp:208-243), or one 8-channel stream —
// 2..8 of its 128 series slots carry data.  This kernel turns the mapping around: a lane owns OUTPUTS.
//
//   lane  = (output n, chunk of SV series)            SV = 2, 4 or 8 series held per lane, B outputs per lane
//   CTA   = 128 lanes = (128 / Q) x B consecutive outputs of all Q x SV series slots
//   loop  = taps k = 0 .. T-1 in order (tap-synchronous): acc[n][s] += (H[phase_n][k], H[phase_n+1][k]) * x[ws_n+k][s]
//
// — one accumulator per dot product, taps in order, FFMA chain (fast) or FMUL+FADD (exact), exactly like the
// standard kernel and the reference (dsps_dotprod_f32_ansi.c:17-25), but with no padded rows at all.
//
// Operands.  Nothing here is warp-uniform (every lane has its own phase and its own window), so both operands come
// from shared memory as per-lane loads:
//   * the input window of the CTA's outputs: rows [ws_first, ws_last + T) of the time-major staging buffer, copied
//     once per CTA into a compact tile [row][Q x SV] (cp.async);
//   * the filter bank, which does not fit shared memory (263 KB at T = F = 256, 4.2 MB at 1024 x 1024), streamed as
//     TAP-RANGE SLICES: slice t holds taps [t KT, (t+1) KT) of ALL F+1 phases (<= 21 KB), one TMA bulk copy from a
//     slice-major copy of the bank built at init (`bank_tr`), through a 3-stage ring; the last warp to finish a
//     slice re-arms its mbarrier and issues the refill (same protocol as the standard kernel).  The slice row pitch
//     is KT+1 floats, so lanes reading the same tap of different phases hit different banks.
// Per tap a lane issues 2 LDS.32 (coefficients of phase and phase+1) + one LDS of SV floats (x) for SV FFMA2: the
// loop is bound by shared-memory wavefronts, not by the FMA pipe (2+SV/... wavefronts per 2 SV FMA cycles: about 25 %
// of the FMA peak for one stereo stream, 40 % for 8 series) — every x value and every coefficient pair is used by
// exactly SV or one FFMA2, and no tiling can raise that for a single series (DESIGN.md §4.2).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.hpp"
#include "kernels.hpp"
#include "resample_device.cuh"

namespace espb {

namespace {

constexpr int FS_THREADS = 128;
constexpr int FS_WARPS = FS_THREADS / 32;
constexpr int FS_MAX_STAGES = 4;

template <int SV>
struct XVec;
template <>
struct XVec<2> {
  float v[2];
  __device__ __forceinline__ void load(const float *p) {
    const float2 t = *reinterpret_cast<const float2 *>(p);
    v[0] = t.x, v[1] = t.y;
  }
};
template <>
struct XVec<4> {
  float v[4];
  __device__ __forceinline__ void load(const float *p) {
    const float4 t = *reinterpret_cast<const float4 *>(p);
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  }
};
template <>
struct XVec<8> {
  float v[8];
  __device__ __forceinline__ void load(const float *p) {
    const float4 t = *reinterpret_cast<const float4 *>(p), u = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w, v[4] = u.x, v[5] = u.y, v[6] = u.z, v[7] = u.w;
  }
};

template <int SV, int B, bool EXACT>
__global__ void __launch_bounds__(FS_THREADS) espb_resample_fs_kernel(const FsParams pp) {
  FsParams p = pp;
  if (pp.groups) {  // fused clock groups: this CTA works on group blockIdx.y (its own schedule, rows and output)
    const FsGroupDesc gd = pp.groups[blockIdx.y];
    p.x = pp.x + gd.x_off;
    p.outs = pp.outs + gd.outs_begin;
    p.n_out = gd.n_out;
    p.out = pp.out + gd.out_off;
    const int per_cta = (FS_THREADS / pp.q_per_out) * B;
    if ((int) blockIdx.x * per_cta >= gd.n_out)
      return;
  }
  extern __shared__ __align__(128) unsigned char fs_smem[];
  const int FS_STAGES = p.stages;
  float *slices = reinterpret_cast<float *>(fs_smem);                            // [stages][slice_floats]
  float *xtile = slices + (size_t) FS_STAGES * p.slice_floats;                   // [x_rows][x_pitch]
  uint64_t *full = reinterpret_cast<uint64_t *>(xtile + (size_t) p.x_tile_floats);  // [stages]
  int *done = reinterpret_cast<int *>(full + FS_MAX_STAGES);                        // [stages]

  const int tid = threadIdx.x, lane = tid & 31;
  const int Q = p.q_per_out, NL = FS_THREADS / Q;  // series chunks per output, outputs per round of the CTA
  const int n_local = tid / Q, qc = tid - n_local * Q;
  const bool active_lane = n_local < NL;
  const int svt = Q * SV;  // series slots per input row
  // floats per x-tile row: an ODD number of 16-byte units, so that the rows of neighbouring outputs (2-3 apart when
  // down-sampling) fall into different bank groups (an even pitch folds them onto half of the banks: measured 91 %
  // LSU-wavefront utilisation at 14 % of the FMA peak for 8 series before this)
  const int xpitch = p.x_pitch;
  const int M = NL * B;    // outputs per CTA
  const int n0 = blockIdx.x * M;
  const int n_end = n0 + M < p.n_out ? n0 + M : p.n_out;
  const int T = p.taps, KT = p.kt, pitch = KT + 1, n_slices = T / KT;

  if (tid == 0) {
    for (int s = 0; s < FS_STAGES; ++s) {
      mbar_init(&full[s], 1);
      done[s] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  auto issue_slice = [&](int t) {
    const int st = t % FS_STAGES;
    const uint32_t bytes = (uint32_t) p.slice_floats * sizeof(float);
    mbar_expect_tx(&full[st], bytes);
    tma_bulk_g2s(slices + (size_t) st * p.slice_floats, p.bank_tr + (size_t) t * p.slice_floats, bytes, &full[st]);
  };
  if (tid == 0)
    for (int t = 0; t < FS_STAGES && t < n_slices; ++t)
      issue_slice(t);

  // ---- the input rows of this CTA's outputs -> compact tile
  const int j0 = p.outs[n0].ws;                 // windows advance monotonically
  const int j1 = p.outs[n_end - 1].ws + T;      // one past the last row any of them reads
  {
    const int rows = j1 - j0;
    const float *src = p.x + (int64_t) (j0 + p.x_row0) * p.x_fs;
    if (svt >= 4) {  // 16-byte units (the staging rows are 512-byte aligned, svt is a multiple of 4)
      const int upr = svt / 4;
      for (int i = tid; i < rows * upr; i += FS_THREADS) {
        const int r = i / upr, u = i - r * upr;
        cp_async_16(xtile + (size_t) r * xpitch + u * 4, src + (int64_t) r * p.x_fs + u * 4);
      }
    } else {  // SV = 2, one chunk: 8 bytes per row
      for (int i = tid; i < rows; i += FS_THREADS)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(smem_u32(xtile + (size_t) i * 2)),
                     "l"(src + (int64_t) i * p.x_fs)
                     : "memory");
    }
  }

  // ---- this lane's outputs: n0 + i * NL + n_local
  int ph_off[B];    // row offset of the phase inside a slice, floats
  int x_off[B];     // offset of the window's first sample inside the tile, floats
  float wgt[B];
  int kind[B];
#pragma unroll
  for (int i = 0; i < B; ++i) {
    const int n = n0 + i * NL + n_local;
    OutEntry e;
    e.ws = j0, e.phase = 0, e.w = 0.0f, e.kind = kKindNone;
    if (active_lane && n < n_end)
      e = p.outs[n];
    ph_off[i] = e.phase * pitch;
    x_off[i] = (e.ws - j0) * xpitch + qc * SV;
    wgt[i] = e.w;
    kind[i] = e.kind;
  }
  cp_async_wait_all();
  __syncthreads();

  float2 acc2[EXACT ? 1 : B][EXACT ? 1 : SV];
  float acc1[EXACT ? B : 1][EXACT ? SV : 1][2];
#pragma unroll
  for (int i = 0; i < B; ++i)
#pragma unroll
    for (int s = 0; s < SV; ++s) {
      if constexpr (EXACT)
        acc1[i][s][0] = acc1[i][s][1] = 0.0f;
      else
        acc2[i][s] = make_float2(0.0f, 0.0f);
    }

  for (int t = 0; t < n_slices; ++t) {
    const int st = t % FS_STAGES;
    mbar_wait(&full[st], (uint32_t) ((t / FS_STAGES) & 1));
    const float *sl = slices + (size_t) st * p.slice_floats;
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const float *c0 = sl + ph_off[i];
      const float *xp = xtile + x_off[i] + (size_t) t * KT * xpitch;
      for (int kk = 0; kk < KT; kk += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float h0 = c0[kk + u], h1 = c0[pitch + kk + u];
          XVec<SV> xv;
          xv.load(xp + (size_t) (kk + u) * xpitch);
#pragma unroll
          for (int s = 0; s < SV; ++s) {
            if constexpr (EXACT) {
              acc1[i][s][0] = mac<true>(h0, xv.v[s], acc1[i][s][0]);
              acc1[i][s][1] = mac<true>(h1, xv.v[s], acc1[i][s][1]);
            } else {
              acc2[i][s] = fma2(make_float2(h0, h1), xv.v[s], acc2[i][s]);
            }
          }
        }
      }
    }
    // release the slice; the last warp to get here refills it (resample_kernel.cu has the argument)
    __syncwarp();
    if (lane == 0) {
      if (smem_arrive(&done[st]) == FS_WARPS - 1) {
        done[st] = 0;
        if (t + FS_STAGES < n_slices)
          issue_slice(t + FS_STAGES);
      }
    }
  }

  // ---- blend and store (art_resampler.cpp:421-451)
#pragma unroll
  for (int i = 0; i < B; ++i) {
    const int n = n0 + i * NL + n_local;
    if (!active_lane || n >= n_end)
      continue;
    float v[SV];
#pragma unroll
    for (int s = 0; s < SV; ++s) {
      float sum1, sum2;
      if constexpr (EXACT) {
        sum1 = acc1[i][s][0];
        sum2 = acc1[i][s][1];
      } else {
        sum1 = acc2[i][s].x;
        sum2 = acc2[i][s].y;
      }
      if (kind[i] == kKindBlend)
        v[s] = __fadd_rn(__fmul_rn(sum2, wgt[i]), __fmul_rn(sum1, __fsub_rn(1.0f, wgt[i])));
      else if (kind[i] == kKindSingle)
        v[s] = sum1;
      else  // pass-through: *source = tap numTaps/2-1 of the window
        v[s] = xtile[x_off[i] + (size_t) (T / 2 - 1) * xpitch + s];
    }
    const int q0 = qc * SV;  // first series of this lane
    if (p.out_tm) {
      float *dst = p.out_tm + (int64_t) n * SGN + q0;
      if constexpr (SV == 2) {
        *reinterpret_cast<float2 *>(dst) = make_float2(v[0], v[1]);
      } else {
#pragma unroll
        for (int s = 0; s < SV; s += 4)
          *reinterpret_cast<float4 *>(dst + s) = make_float4(v[s], v[s + 1], v[s + 2], v[s + 3]);
      }
    } else if (p.out_vec && q0 + SV <= p.n_series) {
      // interleaved, the lane's SV series are SV contiguous channels of one frame of one stream
      const int sidx = q0 / p.channels, ch = q0 - sidx * p.channels;
      float *dst = p.out + (int64_t) sidx * p.out_ss + ch + (int64_t) n * p.out_fs;
      if constexpr (SV == 2) {
        *reinterpret_cast<float2 *>(dst) = make_float2(v[0], v[1]);
      } else {
#pragma unroll
        for (int s = 0; s < SV; s += 4)
          *reinterpret_cast<float4 *>(dst + s) = make_float4(v[s], v[s + 1], v[s + 2], v[s + 3]);
      }
    } else {
#pragma unroll
      for (int s = 0; s < SV; ++s) {
        const int q = q0 + s;
        if (q < p.n_series) {
          const int sidx = q / p.channels, ch = q - sidx * p.channels;
          p.out[(int64_t) sidx * p.out_ss + (int64_t) ch * p.out_cs + (int64_t) n * p.out_fs] = v[s];
        }
      }
    }
  }
}

template <int SV, int B, bool EXACT>
cudaError_t launch_fs_t(const FsParams &p, size_t smem, dim3 grid, cudaStream_t stream) {
  static PerDeviceOnce once;
  static size_t smem_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (once.first() || (dev >= 0 && dev < 64 && smem > smem_set[dev])) {
    cudaError_t e = cudaFuncSetAttribute(espb_resample_fs_kernel<SV, B, EXACT>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int) (200 * 1024));
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(espb_resample_fs_kernel<SV, B, EXACT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                               (int) cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess)
      return e;
    if (dev >= 0 && dev < 64)
      smem_set[dev] = 200 * 1024;
    if (getenv("ESPB_DEBUG")) {
      int nb = 0;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, espb_resample_fs_kernel<SV, B, EXACT>, FS_THREADS, smem);
      cudaFuncAttributes fa;
      cudaFuncGetAttributes(&fa, espb_resample_fs_kernel<SV, B, EXACT>);
      fprintf(stderr, "[espb] resample_fs<%d,%d,%d>: smem %zu B, %d regs, occupancy %d CTA/SM\n", SV, B, (int) EXACT,
              smem, fa.numRegs, nb);
    }
  }
  espb_resample_fs_kernel<SV, B, EXACT><<<grid, FS_THREADS, smem, stream>>>(p);
  count_launch();
  return cudaGetLastError();
}

}  // namespace

// ---------------------------------------------------------------------------------
// Fused clock groups: staging and schedule expansion for all groups of a set in one launch each.
// ---------------------------------------------------------------------------------
// Row r < taps of a group's new staging rows = row carry_row + r of its previous ones (the frames the reference keeps
// at the front of its ring, art_resampler.cpp:216-222); row taps + j = input frame j of the group's streams
// (interleaved caller layout), series beyond n_series are zero.
__global__ void __launch_bounds__(256)
    espb_fsg_stage_kernel(const FsGroupDesc *__restrict__ groups, const float *__restrict__ old_buf,
                          float *__restrict__ new_buf, int pitch, int taps, const float *__restrict__ in, int64_t in_ss,
                          int channels, int n_series, int rows_per_cta) {
  const FsGroupDesc gd = groups[blockIdx.y];
  const int rows = taps + gd.n_in;
  const int r0 = blockIdx.x * rows_per_cta;
  if (r0 >= rows)
    return;
  const int r1 = r0 + rows_per_cta < rows ? r0 + rows_per_cta : rows;
  float *dst = new_buf + gd.x_off;
  const float *old = old_buf + gd.x_old_off;
  const float *src = in + gd.in_off;
  for (int i = threadIdx.x; i < (r1 - r0) * pitch; i += blockDim.x) {
    const int r = r0 + i / pitch, q = i % pitch;
    float v = 0.0f;
    if (r < taps) {
      v = old[(int64_t) (gd.carry_row + r) * pitch + q];
    } else if (q < n_series) {
      const int st = q / channels, ch = q - st * channels;
      v = __ldg(src + (int64_t) st * in_ss + (int64_t) (r - taps) * channels + ch);
    }
    dst[(int64_t) r * pitch + q] = v;
  }
}

__global__ void __launch_bounds__(256)
    espb_expand_schedule_groups_kernel(const FsGroupDesc *__restrict__ groups, const SchedSegment *__restrict__ segs,
                                       OutEntry *__restrict__ outs, float n_filters, int lowpass, int interp) {
  const FsGroupDesc gd = groups[blockIdx.y];
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= gd.n_out)
    return;
  const SchedSegment *sg0 = segs + gd.seg_begin;
  int lo = 0, hi = gd.n_segs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&sg0[mid].n0) <= k)
      lo = mid;
    else
      hi = mid - 1;
  }
  const SchedSegment sg = sg0[lo];
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
  outs[gd.outs_begin + k] = e;
}

cudaError_t launch_fsg_stage(const FsGroupDesc *groups, int n_groups, const float *old_buf, float *new_buf, int pitch,
                             int taps, const float *in, int64_t in_ss, int channels, int n_series, int max_rows,
                             cudaStream_t stream) {
  if (n_groups <= 0 || max_rows <= 0)
    return cudaSuccess;
  // about 2048 elements per CTA
  int rows_per_cta = 2048 / pitch;
  rows_per_cta = rows_per_cta < 1 ? 1 : rows_per_cta;
  // groups ride on y: a slice takes the descriptors from its first group on (their offsets are absolute)
  return for_each_y_slice(n_groups, [&](int g0, int ng) {
    const dim3 grid((max_rows + rows_per_cta - 1) / rows_per_cta, ng);
    espb_fsg_stage_kernel<<<grid, 256, 0, stream>>>(groups + g0, old_buf, new_buf, pitch, taps, in, in_ss, channels,
                                                    n_series, rows_per_cta);
    count_launch();
    return cudaGetLastError();
  });
}

cudaError_t launch_expand_schedule_groups(const FsGroupDesc *groups, int n_groups, const SchedSegment *segs,
                                          OutEntry *outs, int max_n_out, int n_filters, bool lowpass, bool interp,
                                          cudaStream_t stream) {
  if (n_groups <= 0 || max_n_out <= 0)
    return cudaSuccess;
  return for_each_y_slice(n_groups, [&](int g0, int ng) {
    const dim3 grid((max_n_out + 255) / 256, ng);
    espb_expand_schedule_groups_kernel<<<grid, 256, 0, stream>>>(groups + g0, segs, outs, (float) n_filters, lowpass,
                                                                 interp);
    count_launch();
    return cudaGetLastError();
  });
}

// Tap-range width of the slices: the widest power of two (4..64) that divides `taps` and keeps one slice of all
// filters+2 rows (pitch kt+1) within 21 KB, so that three stages and the input tile leave room for two CTAs per SM.
int fs_slice_taps(int taps, int filters) {
  long budget = 21 * 1024;  // bytes per slice
  if (const char *v = getenv("ESPB_FS_SLICE_KB"))
    if (atoi(v) > 0)
      budget = atol(v) * 1024;
  int kt = 4;
  while (kt < 64 && taps % (kt * 2) == 0 && (long) ((filters + 2) * (kt * 2 + 1) * sizeof(float)) <= budget)
    kt *= 2;
  return kt;
}

size_t fs_slice_floats(int filters, int kt) { return ((size_t) (filters + 2) * (kt + 1) + 3) & ~(size_t) 3; }

// Slice-major copy of the bank: [taps / kt][filters + 2 rows][kt + 1] floats (row filters+1 and the pad column are zero).
void fs_build_bank_slices(const float *bank, int taps, int filters, int kt, float *dst) {
  const size_t sf = fs_slice_floats(filters, kt);
  const int n_slices = taps / kt, pitch = kt + 1;
  for (size_t i = 0; i < sf * n_slices; ++i)
    dst[i] = 0.0f;
  for (int t = 0; t < n_slices; ++t)
    for (int r = 0; r <= filters; ++r)
      for (int k = 0; k < kt; ++k)
        dst[t * sf + (size_t) r * pitch + k] = bank[(size_t) r * taps + t * kt + k];
}

FsGeometry fs_geometry(int n_series) {
  FsGeometry g{};
  if (n_series <= 2)
    g.sv = 2, g.b = 4, g.q = 1;
  else if (n_series <= 4)
    g.sv = 4, g.b = 4, g.q = 1;
  else
    g.sv = 8, g.b = 2, g.q = (n_series + 7) / 8;
  g.outputs_per_cta = (FS_THREADS / g.q) * g.b;
  return g;
}

int fs_x_pitch(const FsGeometry &g) {
  const int svt = g.q * g.sv;
  return (svt >= 8 && (svt / 4) % 2 == 0) ? svt + 4 : svt;
}

int fs_stages() {
  static int st = 0;
  if (!st) {
    const char *v = getenv("ESPB_FS_STAGES");
    const int n = v ? atoi(v) : 0;
    st = (n >= 2 && n <= FS_MAX_STAGES) ? n : 2;  // measured: 2 stages (more CTAs per SM) >= 3 on every shape
  }
  return st;
}

size_t fs_smem_bytes(const FsGeometry &g, size_t slice_floats, int x_rows) {
  return (fs_stages() * slice_floats + (((size_t) x_rows * fs_x_pitch(g) + 3) & ~(size_t) 3)) * sizeof(float) +
         FS_MAX_STAGES * (sizeof(uint64_t) + sizeof(int)) + 16;
}

cudaError_t launch_resample_fs(const FsParams &p_in, const FsGeometry &g, int x_rows, bool exact,
                               cudaStream_t stream, int n_groups) {
  if (p_in.n_out <= 0 || p_in.n_series <= 0)
    return cudaSuccess;
  FsParams p = p_in;
  p.q_per_out = g.q;
  p.x_pitch = fs_x_pitch(g);
  p.stages = fs_stages();
  p.x_tile_floats = (int) (((size_t) x_rows * p.x_pitch + 3) & ~(size_t) 3);
  const size_t smem = fs_smem_bytes(g, (size_t) p.slice_floats, x_rows);
  if (smem > 200 * 1024)
    return cudaErrorInvalidValue;
  // vector stores: interleaved caller layout whose channel count keeps a lane's series inside one frame
  p.out_vec = (!p.out_tm && p.out_cs == 1 && p.channels % g.sv == 0 && (uintptr_t) p.out % 16 == 0 &&
               p.out_ss % 4 == 0 && p.out_fs % g.sv == 0)
                  ? 1
                  : 0;
  // (fused groups: n_out is the largest group's count; CTAs past a group's own count leave at once)
  // (fused groups ride on y: a slice takes the descriptors from its first group on)
  return for_each_y_slice(p.groups ? n_groups : 1, [&](int g0, int ng) {
    FsParams pg = p;
    if (p.groups)
      pg.groups = p.groups + g0;
    const dim3 grid((p.n_out + g.outputs_per_cta - 1) / g.outputs_per_cta, ng);
#define ESPB_FS(SV_, B_) \
  (exact ? launch_fs_t<SV_, B_, true>(pg, smem, grid, stream) : launch_fs_t<SV_, B_, false>(pg, smem, grid, stream))
    if (g.sv == 2 && g.b == 4)
      return ESPB_FS(2, 4);
    if (g.sv == 4 && g.b == 4)
      return ESPB_FS(4, 4);
    if (g.sv == 8 && g.b == 2)
      return ESPB_FS(8, 2);
#undef ESPB_FS
    return cudaErrorInvalidValue;
  });
}

}  // namespace espb
