// ART polyphase resampler — the non-interpolating form (flags without SUBSAMPLE_INTERPOLATE: one dot product with
// the nearest filter phase per output, art_resampler.cpp:421-430) of the sm_100a kernel.  Same ring, roles and
// epilogue as resample_kernel.cu.  G carries one coefficient per (row, output) — 8 floats per row and block — and a
// warp owns TWO adjacent output blocks of a pass (the pass plan is built with 8 blocks per pass for 4 warps), so its
// tile is 4 series x 16 outputs: per row one per-lane LDS.128 of x and four warp-uniform LDS.128 of G feed 32 packed
// FFMA2 — two neighbouring outputs per instruction, their coefficients are adjacent in G — exactly the instruction
// mix of the interpolating kernel (8 shared-memory wavefronts per 32 FFMA2; the 4 x 8 tile of round 1 paid 6
// wavefronts per 16).  2T flop per sample on a path that executes 2T, not 4T.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.hpp"
#include "kernels.hpp"
#include "resample_device.cuh"

namespace espb {

template <int BPP, int NST, int CJ, bool EXACT, bool TMCAP>
__global__ void __launch_bounds__(BPP * 32, 16 / BPP) espb_resample_ni_kernel(const ResampleParams p) {
  constexpr int GRF = kGRowFloatsNI;  // one coefficient per output and row
  constexpr int WB = kNiBlocksPerWarp;  // output blocks per warp
  constexpr int PB = BPP * WB;          // blocks per pass of the plan
  constexpr int NO = NB * WB;           // outputs per warp
  constexpr int NTHREADS = BPP * 32;
  constexpr int STAGES = NST;
  constexpr int MAXC = kMaxChunksPerCta;
  static_assert(kMaxPassesPerCta * BPP * sizeof(int2) <= (size_t) NST * CJ * SGN * sizeof(float), "set-up table");
  constexpr int XS_STAGE = CJ * SGN;       // floats
  constexpr int GS_STAGE = CJ * PB * GRF;  // floats
  constexpr uint32_t X_BYTES = XS_STAGE * sizeof(float), G_BYTES = GS_STAGE * sizeof(float);

  extern __shared__ __align__(128) unsigned char smem_raw[];
  float *gs = reinterpret_cast<float *>(smem_raw);                        // [STAGES][CJ][PB][8]
  float *xs = gs + STAGES * GS_STAGE;                                     // [STAGES][CJ][128]
  uint64_t *full = reinterpret_cast<uint64_t *>(xs + STAGES * XS_STAGE);  // [STAGES] TMA landed
  int *done = reinterpret_cast<int *>(full + STAGES);                     // [2*STAGES] warps done with a stage
  int32_t *jtab = reinterpret_cast<int32_t *>(done + 2 * STAGES);         // [MAXC] first input row of each chunk
  // [MAXC][BPP] what warp w does in chunk c: row groups [r0, r1), end-of-pass flag
  uint16_t *rtab = reinterpret_cast<uint16_t *>(jtab + MAXC);
  // [BPP][NO] schedule entries of the blocks each warp is finishing, fetched by cp.async during the pass's last chunk
  OutEntry *etab = reinterpret_cast<OutEntry *>(rtab + MAXC * BPP);
  int32_t *hdr = reinterpret_cast<int32_t *>(etab + BPP * NO);  // [4] CTA constants for the refilling lane
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
    const int o0 = ((pass_first + i / BPP) * PB + (i % BPP) * WB) * NB;
    int2 w = make_int2(0, 0);
    if (o0 < p.n_out) {
      const int o1 = (o0 + NO <= p.n_out ? o0 + NO : p.n_out) - 1;
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
  // staging overlap (resample_kernel.cu has the protocol): wait for the row tiles this CTA reads
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

  // accumulators [series e][output n]: one dot product per output (art_resampler.cpp:421-430)
  // (fast mode: two neighbouring outputs share one packed FFMA2 — their coefficients are adjacent in G)
  float acc[EXACT ? 4 : 1][EXACT ? NO : 1];
  float2 accp[EXACT ? 1 : 4][EXACT ? 1 : NO / 2];
  auto clear_acc = [&]() {
    if constexpr (EXACT) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int n = 0; n < NO; ++n)
          acc[e][n] = 0.0f;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int m = 0; m < NO / 2; ++m)
          accp[e][m] = make_float2(0.0f, 0.0f);
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
    if (pass_done && lane < NO) {  // the epilogue's schedule entries: global -> shared, no register held meanwhile
      int o = (cur_pass * PB + warp * WB) * NB + lane;
      o = o < p.n_out ? o : p.n_out - 1;
      cp_async_16(&etab[warp * NO + lane], &p.outs[o]);
    }
    mbar_wait(&full[st], (uint32_t) ((c / STAGES) & 1));
    {
      const float *xrow = xs + st * XS_STAGE + lane * 4;
      const float *grow = gs + st * GS_STAGE + warp * WB * GRF;
      for (int jb = r0; jb < r1; ++jb) {
        const float *xb = xrow + jb * RG * SGN;
        const float *gb = grow + jb * RG * PB * GRF;
#pragma unroll
        for (int jj = 0; jj < RG; ++jj) {
          const float4 xv = *reinterpret_cast<const float4 *>(xb + jj * SGN);
          const float4 *gp = reinterpret_cast<const float4 *>(gb + jj * PB * GRF);
          const float4 g0 = gp[0], g1 = gp[1], g2 = gp[2], g3 = gp[3];  // 16 outputs: blocks 2 warp, 2 warp + 1
          const float x4[4] = {xv.x, xv.y, xv.z, xv.w};
          if constexpr (EXACT) {
            const float g16[NO] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w,
                                   g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z, g3.w};
#pragma unroll
            for (int n = 0; n < NO; ++n)
#pragma unroll
              for (int e = 0; e < 4; ++e)
                acc[e][n] = mac<true>(g16[n], x4[e], acc[e][n]);
          } else {
            const float2 gg[NO / 2] = {make_float2(g0.x, g0.y), make_float2(g0.z, g0.w), make_float2(g1.x, g1.y),
                                       make_float2(g1.z, g1.w), make_float2(g2.x, g2.y), make_float2(g2.z, g2.w),
                                       make_float2(g3.x, g3.y), make_float2(g3.z, g3.w)};  // (output 2m, output 2m + 1)
#pragma unroll
            for (int m = 0; m < NO / 2; ++m)
#pragma unroll
              for (int e = 0; e < 4; ++e)
                accp[e][m] = fma2(gg[m], x4[e], accp[e][m]);
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

    // ---- end of pass: store, clear (the warp's two blocks one after the other)
    if (pass_done) {
      cp_async_wait_all();
      __syncwarp();
      const int series0 = group * SGN + lane * 4;
#pragma unroll
      for (int h = 0; h < WB; ++h) {
        const int o0 = (cur_pass * PB + warp * WB + h) * NB;
        const OutEntry *et = etab + warp * NO + h * NB;
        float v[4][NB];
#pragma unroll
        for (int n = 0; n < NB; ++n) {
          const OutEntry en = et[n];  // one broadcast LDS.128
          const int nn = h * NB + n;  // index in the warp's 16 outputs
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (en.kind >= kKindSingle) {  // (no blend without SUBSAMPLE_INTERPOLATE)
              v[e][n] = EXACT ? acc[EXACT ? e : 0][EXACT ? nn : 0]
                              : ((nn & 1) ? accp[EXACT ? 0 : e][EXACT ? 0 : nn / 2].y
                                          : accp[EXACT ? 0 : e][EXACT ? 0 : nn / 2].x);
            } else {  // pass-through: *source (art_resampler.cpp:426,440) = tap numTaps/2-1 of the window
              v[e][n] = p.xt[((int64_t) group * p.xt_rows + (en.ws + T / 2 - 1 + T)) * SGN + lane * 4 + e];
            }
          }
        }
        if (TMCAP && p.out_vec == kOutVecTimeMajor) {  // scratch for a following in-library stage
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
              reinterpret_cast<float4 *>(dst)[k] = make_float4(v[0][2 * k], v[1][2 * k], v[0][2 * k + 1], v[1][2 * k + 1]);
          }
          if (series0 + 2 < p.n_series) {
            dst += p.out_ss;
#pragma unroll
            for (int k = 0; k < NB / 2; ++k)
              reinterpret_cast<float4 *>(dst)[k] = make_float4(v[2][2 * k], v[3][2 * k], v[2][2 * k + 1], v[3][2 * k + 1]);
          }
        } else if (p.out_vec == kOutVecFrame4 && o0 + NB <= p.n_out) {
          // interleaved, channel count a multiple of 4: the lane's 4 series are 16 contiguous bytes of every frame
          if (series0 < p.n_series) {
            const int sidx = series0 / p.channels, ch = series0 - sidx * p.channels;
            float *dst = p.out + (int64_t) sidx * p.out_ss + ch + (int64_t) o0 * p.channels;
#pragma unroll
            for (int n = 0; n < NB; ++n)
              *reinterpret_cast<float4 *>(dst + n * p.channels) = make_float4(v[0][n], v[1][n], v[2][n], v[3][n]);
          }
        } else if (p.out_vec == kOutVecPlanar && o0 + NB <= p.n_out) {
          // frames contiguous per series (planar, or interleaved mono): 8 frames = 32 contiguous bytes per series
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int series = series0 + e;
            if (series < p.n_series) {
              const int sidx = series / p.channels, ch = series - sidx * p.channels;
              float4 *dst = reinterpret_cast<float4 *>(p.out + (int64_t) sidx * p.out_ss + (int64_t) ch * p.out_cs + o0);
              dst[0] = make_float4(v[e][0], v[e][1], v[e][2], v[e][3]);
              dst[1] = make_float4(v[e][4], v[e][5], v[e][6], v[e][7]);
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
      }
      clear_acc();
      ++cur_pass;
    }
  }
}

// Shared memory of one CTA: the ring (G stage: 32 rows x 8 blocks x 8 coefficients; x stage: 32 rows x 128 series),
// barriers, the chunk tables and the schedule entries of 4 warps x 16 outputs.
size_t resample_ni_smem_bytes(int warps, int CJ, int stages) {
  return (size_t) stages * ((size_t) CJ * warps * kNiBlocksPerWarp * kGRowFloatsNI + (size_t) CJ * SGN) * sizeof(float) +
         2 * stages * sizeof(uint64_t) + kMaxChunksPerCta * (sizeof(int32_t) + warps * sizeof(uint16_t)) +
         (size_t) warps * kNiBlocksPerWarp * NB * sizeof(OutEntry) + 4 * sizeof(int32_t);
}

template <int BPP, int NST, int CJ, bool EXACT, bool TMCAP>
static cudaError_t launch_ni_t(const ResampleParams &p, int n_groups, int n_ctas_y, cudaStream_t stream) {
  const size_t smem = resample_ni_smem_bytes(BPP, CJ, NST);
  static PerDeviceOnce once;
  if (once.first()) {
    cudaError_t e = cudaFuncSetAttribute(espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP>,
                               cudaFuncAttributePreferredSharedMemoryCarveout, (int) cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess)
      return e;
    if (getenv("ESPB_DEBUG")) {
      int nb = 0;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP>, BPP * 32,
                                                    smem);
      cudaFuncAttributes fa;
      cudaFuncGetAttributes(&fa, espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP>);
      fprintf(stderr, "[espb] resample_ni<%d,%d,%d,%d,%d>: smem %zu B, %d regs, occupancy %d CTA/SM\n", BPP, NST, CJ,
              (int) EXACT, (int) TMCAP, smem, fa.numRegs, nb);
    }
  }
  dim3 grid(n_groups, n_ctas_y);
  if (p.ready != nullptr) {  // programmatic dependent of the staging kernel launched just before (resample_kernel.cu)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(BPP * 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP>, p);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
  }
  espb_resample_ni_kernel<BPP, NST, CJ, EXACT, TMCAP><<<grid, BPP * 32, smem, stream>>>(p);
  count_launch();
  return cudaGetLastError();
}

// q.out_vec is already set by launch_resample
cudaError_t launch_resample_ni(const ResampleParams &q, int n_groups, int n_ctas_y, bool exact, bool tm,
                               cudaStream_t stream) {
  constexpr int W = kResampleWarps, NST = kResampleStages, CJ = kResampleChunkRows;
  if (exact)
    return tm ? launch_ni_t<W, NST, CJ, true, true>(q, n_groups, n_ctas_y, stream)
              : launch_ni_t<W, NST, CJ, true, false>(q, n_groups, n_ctas_y, stream);
  return tm ? launch_ni_t<W, NST, CJ, false, true>(q, n_groups, n_ctas_y, stream)
            : launch_ni_t<W, NST, CJ, false, false>(q, n_groups, n_ctas_y, stream);
}

}  // namespace espb
