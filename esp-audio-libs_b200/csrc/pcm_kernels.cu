// quantization_utils on the device: packed little-endian PCM <-> float.
//
// Reference: src/quantization_utils.cpp:6-48 (quantized_to_float) and :50-94
// (float_to_quantized).  Integer/byte work, HBM-bound: each thread converts four
// samples per step with 32-bit word loads/stores (4*nbytes bytes of PCM, one 128-bit
// float access); a scalar byte path covers unaligned buffers and row tails.
// Bit-exact with the reference for finite inputs (float->int32 of out-of-range values
// is undefined behaviour in the reference; here it saturates).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "common.hpp"
#include "kernels.hpp"
#include "pcm_device.cuh"
#include "resample_device.cuh"

namespace espb {

namespace {

// ---- decode: little-endian bytes -> the reference's int32 `value` -----------------
template <int NBYTES>
__device__ __forceinline__ int32_t decode_bytes(const uint8_t *p) {
  if (NBYTES == 1)
    return (int32_t) p[0] - 128;  // :14
  if (NBYTES == 2)
    return (int32_t) (int16_t) ((uint32_t) p[0] | ((uint32_t) p[1] << 8));  // :21-23
  if (NBYTES == 3)
    return (int32_t) ((uint32_t) p[0] | ((uint32_t) p[1] << 8)) + (int32_t) (int8_t) p[2] * 65536;  // :30-33
  // :40-44 — byte 2 is sign-extended as well as byte 3 (reference quirk, reproduced)
  uint32_t v = (uint32_t) p[0] | ((uint32_t) p[1] << 8);
  v += (uint32_t) ((int32_t) (int8_t) p[2] * 65536);
  v += (uint32_t) p[3] << 24;
  return (int32_t) v;
}

// four samples from NBYTES 32-bit words
template <int NBYTES>
__device__ __forceinline__ void decode_words(const uint32_t *w, int32_t v[4]) {
  if (NBYTES == 1) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      v[i] = (int32_t) ((w[0] >> (8 * i)) & 0xffu) - 128;
  } else if (NBYTES == 2) {
    v[0] = (int32_t) (int16_t) (w[0] & 0xffffu);
    v[1] = (int32_t) (int16_t) (w[0] >> 16);
    v[2] = (int32_t) (int16_t) (w[1] & 0xffffu);
    v[3] = (int32_t) (int16_t) (w[1] >> 16);
  } else if (NBYTES == 3) {
    const uint32_t s0 = w[0] & 0xffffffu;
    const uint32_t s1 = (w[0] >> 24) | ((w[1] & 0xffffu) << 8);
    const uint32_t s2 = (w[1] >> 16) | ((w[2] & 0xffu) << 16);
    const uint32_t s3 = w[2] >> 8;
    v[0] = (int32_t) (s0 << 8) >> 8;
    v[1] = (int32_t) (s1 << 8) >> 8;
    v[2] = (int32_t) (s2 << 8) >> 8;
    v[3] = (int32_t) (s3 << 8) >> 8;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)  // sign-extending byte 2 subtracts 2^24 when it is >= 0x80
      v[i] = (int32_t) (w[i] - ((w[i] & 0x00800000u) << 1));
  }
}

template <int NBYTES>
__global__ void __launch_bounds__(256)
    espb_q2f_kernel(const uint8_t *__restrict__ in, int64_t in_row_bytes, float *__restrict__ out,
                    int64_t out_row_floats, uint32_t n, float k, int vec_ok) {
  const uint8_t *irow = in + (int64_t) blockIdx.y * in_row_bytes;
  float *orow = out + (int64_t) blockIdx.y * out_row_floats;
  const uint32_t groups = vec_ok ? n / 4 : 0;
  const uint32_t stride = gridDim.x * blockDim.x;
  // (consecutive lanes take consecutive 4-sample groups, so the 128-bit stores of a warp are one contiguous 512 bytes;
  //  a 16-samples-per-thread form with 128-bit loads was measured slower here — its stores are 64 bytes apart — while
  //  it is the faster one for the encoder below, whose wide side is the load)
#pragma unroll 4
  for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(irow) + (size_t) g * NBYTES;
    uint32_t w[NBYTES];
    if (NBYTES == 2 && vec_ok == 2) {  // (16-byte aligned rows: a group's 8 bytes are one 64-bit load)
      const uint2 t = __ldg(reinterpret_cast<const uint2 *>(wp));
      w[0] = t.x, w[NBYTES > 1 ? 1 : 0] = t.y;
    } else if (NBYTES == 4 && vec_ok == 2) {
      const uint4 t = __ldg(reinterpret_cast<const uint4 *>(wp));
      w[0] = t.x, w[NBYTES > 1 ? 1 : 0] = t.y, w[NBYTES > 2 ? 2 : 0] = t.z, w[NBYTES > 3 ? 3 : 0] = t.w;
    } else {
#pragma unroll
      for (int i = 0; i < NBYTES; ++i)
        w[i] = __ldg(wp + i);
    }
    int32_t v[4];
    decode_words<NBYTES>(w, v);
    float4 f;
    f.x = __fmul_rn(__int2float_rn(v[0]), k);
    f.y = __fmul_rn(__int2float_rn(v[1]), k);
    f.z = __fmul_rn(__int2float_rn(v[2]), k);
    f.w = __fmul_rn(__int2float_rn(v[3]), k);
    reinterpret_cast<float4 *>(orow)[g] = f;
  }
  for (uint32_t i = groups * 4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    orow[i] = __fmul_rn(__int2float_rn(decode_bytes<NBYTES>(irow + (size_t) i * NBYTES)), k);
}

// (F2QConst, quantise_one, encode_words: pcm_device.cuh — shared with the fused filter + quantise kernel)

template <int NBYTES>
__global__ void __launch_bounds__(256)
    espb_f2q_kernel(const float *__restrict__ in, int64_t in_row_floats, uint8_t *__restrict__ out,
                    int64_t out_row_bytes, uint32_t n, F2QConst c, uint32_t *__restrict__ clipped_out,
                    int clipped_per_row, int vec_ok) {
  const float *irow = in + (int64_t) blockIdx.y * in_row_floats;
  uint8_t *orow = out + (int64_t) blockIdx.y * out_row_bytes;
  const uint32_t groups = vec_ok ? n / 4 : 0;
  const uint32_t stride = gridDim.x * blockDim.x;
  uint32_t clipped = 0;
  // 16 samples per thread and iteration, 128-bit accesses only: four loads, NBYTES stores (vec_ok == 2)
  const uint32_t wide = (vec_ok == 2) ? n / 16 : 0;
  for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < wide; g += stride) {
    uint32_t w[4 * NBYTES];
    float4 f[4];
#pragma unroll
    for (int h = 0; h < 4; ++h)
      f[h] = __ldg(reinterpret_cast<const float4 *>(irow) + (size_t) g * 4 + h);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      int32_t v[4];
      v[0] = quantise_one(f[h].x, c, clipped);
      v[1] = quantise_one(f[h].y, c, clipped);
      v[2] = quantise_one(f[h].z, c, clipped);
      v[3] = quantise_one(f[h].w, c, clipped);
      encode_words<NBYTES>(v, w + h * NBYTES);
    }
    uint4 *wp = reinterpret_cast<uint4 *>(orow) + (size_t) g * NBYTES;
#pragma unroll
    for (int i = 0; i < NBYTES; ++i)
      wp[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
  }
  for (uint32_t g = wide * 4 + blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
    const float4 f = __ldg(reinterpret_cast<const float4 *>(irow) + g);
    int32_t v[4];
    v[0] = quantise_one(f.x, c, clipped);
    v[1] = quantise_one(f.y, c, clipped);
    v[2] = quantise_one(f.z, c, clipped);
    v[3] = quantise_one(f.w, c, clipped);
    uint32_t w[NBYTES];
    encode_words<NBYTES>(v, w);
    uint32_t *wp = reinterpret_cast<uint32_t *>(orow) + (size_t) g * NBYTES;
#pragma unroll
    for (int i = 0; i < NBYTES; ++i)
      wp[i] = w[i];
  }
  for (uint32_t i = groups * 4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int32_t v = quantise_one(irow[i], c, clipped);
    uint8_t *bp = orow + (size_t) i * NBYTES;
#pragma unroll
    for (int b = 0; b < NBYTES; ++b)
      bp[b] = (uint8_t) ((uint32_t) v >> (8 * b));  // :80-90
  }
  // clip count: warp shuffle reduction, one atomic per warp
#pragma unroll
  for (int d = 16; d > 0; d >>= 1)
    clipped += __shfl_xor_sync(0xffffffffu, clipped, d);
  if ((threadIdx.x & 31) == 0 && clipped && clipped_out)
    atomicAdd(clipped_out + (clipped_per_row ? blockIdx.y : 0), clipped);
}

// ---- fused with the layout stages of the resampler ------------------------------------
// PCM rows (stream-major, channels interleaved) <-> time-major float tm[group][row][128 series]: the
// conversion rides on the transposing pass, so the wrapper path never materialises a stream-major float
// copy.  Tiles of 128 series x 64 frames through shared memory; 32-bit word accesses on the PCM side
// (4 samples = NBYTES words), 128-bit on the float side.  CH in {1,2,4,8}; full tiles only.
// (SGN = kSeriesPerRow = 128: resample_device.cuh)
constexpr int PT_ROWS = 64;
constexpr int PT_THREADS = 256;

template <int NBYTES, int CH>
__global__ void __launch_bounds__(PT_THREADS)
    espb_pcm_to_tm_kernel(const uint8_t *__restrict__ in, int64_t in_row_bytes, float *__restrict__ tm,
                          int64_t rows_cap, int row_first, int n_series, float k) {
  __shared__ __align__(16) float tile_s[PT_ROWS * SGN];
  const SwzTile tile{tile_s};
  const int g = blockIdx.x, j0 = blockIdx.y * PT_ROWS, tid = threadIdx.x;
  constexpr int UNITS = SGN / CH;            // streams per group
  constexpr int GROUPS = PT_ROWS * CH / 4;   // 4-sample groups per stream per tile
  // 16-byte units of a row that hold series of this group (all 32 but in the last group), and the streams they span:
  // a group with few series neither fills nor stores the rest of the tile
  const int units = (n_series - g * SGN + 3) / 4 < SGN / 4 ? (n_series - g * SGN + 3) / 4 : SGN / 4;
  const int streams_here = (units * 4 + CH - 1) / CH < UNITS ? (units * 4 + CH - 1) / CH : UNITS;
#pragma unroll 2
  for (int v = tid; v < streams_here * GROUPS; v += PT_THREADS) {
    const int unit = v / GROUPS, grp = v % GROUPS;
    const int q0 = g * SGN + unit * CH;
    int32_t s[4] = {0, 0, 0, 0};
    if (q0 < n_series) {
      const uint32_t *wp = reinterpret_cast<const uint32_t *>(in + (int64_t) (q0 / CH) * in_row_bytes +
                                                              ((int64_t) j0 * CH + grp * 4) * NBYTES);
      uint32_t w[NBYTES];
#pragma unroll
      for (int i = 0; i < NBYTES; ++i)
        w[i] = __ldg(wp + i);
      decode_words<NBYTES>(w, s);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = grp * 4 + i;
      tile.at(e / CH, unit * CH + (e % CH)) = (q0 < n_series) ? __fmul_rn(__int2float_rn(s[i]), k) : 0.0f;
    }
  }
  __syncthreads();
  float4 *dst = reinterpret_cast<float4 *>(tm + ((int64_t) g * rows_cap + row_first + j0) * SGN);
#pragma unroll 4
  for (int i = tid; i < PT_ROWS * (SGN / 4); i += PT_THREADS) {
    const int t = i / (SGN / 4), c4 = i % (SGN / 4);
    if (c4 < units)
      dst[i] = tile.vec(t, c4);
  }
}

template <int NBYTES, int CH>
__global__ void __launch_bounds__(PT_THREADS)
    espb_tm_to_pcm_kernel(const float *__restrict__ tm, int64_t rows_cap, int row_first, uint8_t *__restrict__ out,
                          int64_t out_row_bytes, int n_series, F2QConst c, uint32_t *__restrict__ clipped_per_stream) {
  __shared__ __align__(16) float tile_s[PT_ROWS * SGN];
  const SwzTile tile{tile_s};
  const int g = blockIdx.x, j0 = blockIdx.y * PT_ROWS, tid = threadIdx.x;
  const float4 *src = reinterpret_cast<const float4 *>(tm + ((int64_t) g * rows_cap + row_first + j0) * SGN);
  constexpr int UNITS = SGN / CH;
  constexpr int GROUPS = PT_ROWS * CH / 4;
  // (a group with few series reads and converts only the 16-byte units that hold series: espb_pcm_to_tm_kernel)
  const int units = (n_series - g * SGN + 3) / 4 < SGN / 4 ? (n_series - g * SGN + 3) / 4 : SGN / 4;
  const int streams_here = (units * 4 + CH - 1) / CH < UNITS ? (units * 4 + CH - 1) / CH : UNITS;
#pragma unroll 4
  for (int i = tid; i < PT_ROWS * (SGN / 4); i += PT_THREADS) {
    const int t = i / (SGN / 4), c4 = i % (SGN / 4);
    if (c4 < units)
      tile.vec(t, c4) = __ldg(src + i);
  }
  __syncthreads();
#pragma unroll 2
  for (int v = tid; v < streams_here * GROUPS; v += PT_THREADS) {
    const int unit = v / GROUPS, grp = v % GROUPS;
    const int q0 = g * SGN + unit * CH;
    if (q0 >= n_series)
      continue;
    const int stream = q0 / CH;
    uint32_t clipped = 0;
    int32_t s[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int e = grp * 4 + i;
      s[i] = quantise_one(tile.at(e / CH, unit * CH + (e % CH)), c, clipped);
    }
    uint32_t w[NBYTES];
    encode_words<NBYTES>(s, w);
    uint32_t *wp = reinterpret_cast<uint32_t *>(out + (int64_t) stream * out_row_bytes +
                                                ((int64_t) j0 * CH + grp * 4) * NBYTES);
#pragma unroll
    for (int i = 0; i < NBYTES; ++i)
      wp[i] = w[i];
    if (clipped && clipped_per_stream)
      atomicAdd(clipped_per_stream + stream, clipped);  // clipping is rare: no reduction needed
  }
}

template <int NBYTES>
bool launch_pcm_to_tm_ch(int ch, dim3 grid, cudaStream_t s, const uint8_t *in, int64_t in_row_bytes, float *tm,
                         int64_t rows_cap, int row_first, int n_series, float k) {
  switch (ch) {
    case 1:
      espb_pcm_to_tm_kernel<NBYTES, 1><<<grid, PT_THREADS, 0, s>>>(in, in_row_bytes, tm, rows_cap, row_first, n_series, k);
      return true;
    case 2:
      espb_pcm_to_tm_kernel<NBYTES, 2><<<grid, PT_THREADS, 0, s>>>(in, in_row_bytes, tm, rows_cap, row_first, n_series, k);
      return true;
    case 4:
      espb_pcm_to_tm_kernel<NBYTES, 4><<<grid, PT_THREADS, 0, s>>>(in, in_row_bytes, tm, rows_cap, row_first, n_series, k);
      return true;
    case 8:
      espb_pcm_to_tm_kernel<NBYTES, 8><<<grid, PT_THREADS, 0, s>>>(in, in_row_bytes, tm, rows_cap, row_first, n_series, k);
      return true;
    default:
      return false;
  }
}

template <int NBYTES>
bool launch_tm_to_pcm_ch(int ch, dim3 grid, cudaStream_t s, const float *tm, int64_t rows_cap, int row_first,
                         uint8_t *out, int64_t out_row_bytes, int n_series, const F2QConst &c, uint32_t *clipped) {
  switch (ch) {
    case 1:
      espb_tm_to_pcm_kernel<NBYTES, 1><<<grid, PT_THREADS, 0, s>>>(tm, rows_cap, row_first, out, out_row_bytes, n_series, c, clipped);
      return true;
    case 2:
      espb_tm_to_pcm_kernel<NBYTES, 2><<<grid, PT_THREADS, 0, s>>>(tm, rows_cap, row_first, out, out_row_bytes, n_series, c, clipped);
      return true;
    case 4:
      espb_tm_to_pcm_kernel<NBYTES, 4><<<grid, PT_THREADS, 0, s>>>(tm, rows_cap, row_first, out, out_row_bytes, n_series, c, clipped);
      return true;
    case 8:
      espb_tm_to_pcm_kernel<NBYTES, 8><<<grid, PT_THREADS, 0, s>>>(tm, rows_cap, row_first, out, out_row_bytes, n_series, c, clipped);
      return true;
    default:
      return false;
  }
}


inline unsigned grid_x_for(uint32_t n, int rows) {
  // enough CTAs to cover the row once at 4 samples/thread, capped so rows*grid stays sane
  uint64_t want = ((uint64_t) n / 4 + 255) / 256;
  if (want < 1)
    want = 1;
  // (grid-stride loops over FEW resident CTAs were the reason these kernels sat at 0.81-0.88 of the copy peak: with
  //  16 CTAs per SM every thread walks ~55 iterations and the whole grid touches one narrow moving window of the
  //  buffers; 512 per SM — a few iterations per thread — measured 0.95-1.08 for all six conversions)
  static const int per_sm = getenv("ESPB_PCM_CTAS") ? atoi(getenv("ESPB_PCM_CTAS")) : 512;
  const uint64_t cap = rows >= 148 * 8 ? 4 : (148 * per_sm + rows - 1) / rows;
  if (want > cap)
    want = cap;
  return (unsigned) want;
}

}  // namespace

cudaError_t launch_q2f(const uint8_t *in, int64_t in_row_bytes, float *out, int64_t out_row_floats, int rows,
                       uint32_t row_samples, int bits, float gain_factor, cudaStream_t stream) {
  if (rows <= 0 || row_samples == 0)
    return cudaSuccess;
  if (rows > grid_y_max())  // rows ride on gridDim.y: larger batches go in slices
    return for_each_y_slice(rows, [&](int r0, int nr) {
      return launch_q2f(in + (int64_t) r0 * in_row_bytes, in_row_bytes, out + (int64_t) r0 * out_row_floats,
                        out_row_floats, nr, row_samples, bits, gain_factor, stream);
    });
  const int nbytes = (bits + 7) / 8;
  int vec_ok = ((uintptr_t) in % 4 == 0) && (in_row_bytes % 4 == 0 || rows == 1) &&
               ((uintptr_t) out % 16 == 0) && (out_row_floats % 4 == 0 || rows == 1);
  if (vec_ok && (uintptr_t) in % 16 == 0 && (in_row_bytes % 16 == 0 || rows == 1))
    vec_ok = 2;  // 128-bit loads on the PCM side too
  dim3 grid(grid_x_for(row_samples, rows), rows);
  switch (nbytes) {
    case 1:
      espb_q2f_kernel<1><<<grid, 256, 0, stream>>>(in, in_row_bytes, out, out_row_floats, row_samples, gain_factor,
                                                  vec_ok);
      break;
    case 2:
      espb_q2f_kernel<2><<<grid, 256, 0, stream>>>(in, in_row_bytes, out, out_row_floats, row_samples, gain_factor,
                                                  vec_ok);
      break;
    case 3:
      espb_q2f_kernel<3><<<grid, 256, 0, stream>>>(in, in_row_bytes, out, out_row_floats, row_samples, gain_factor,
                                                  vec_ok);
      break;
    case 4:
      espb_q2f_kernel<4><<<grid, 256, 0, stream>>>(in, in_row_bytes, out, out_row_floats, row_samples, gain_factor,
                                                  vec_ok);
      break;
    default:
      return cudaErrorInvalidValue;
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_f2q(const float *in, int64_t in_row_floats, uint8_t *out, int64_t out_row_bytes, int rows,
                       uint32_t row_samples, int bits, uint32_t *clipped, bool clipped_per_row, cudaStream_t stream) {
  if (rows <= 0 || row_samples == 0)
    return cudaSuccess;
  if (rows > grid_y_max())  // rows ride on gridDim.y: larger batches go in slices
    return for_each_y_slice(rows, [&](int r0, int nr) {
      return launch_f2q(in + (int64_t) r0 * in_row_floats, in_row_floats, out + (int64_t) r0 * out_row_bytes,
                        out_row_bytes, nr, row_samples, bits, (clipped && clipped_per_row) ? clipped + r0 : clipped,
                        clipped_per_row, stream);
    });
  const int nbytes = (bits + 7) / 8;
  const F2QConst c = make_f2q_const(bits);
  int vec_ok = ((uintptr_t) out % 4 == 0) && (out_row_bytes % 4 == 0 || rows == 1) &&
               ((uintptr_t) in % 16 == 0) && (in_row_floats % 4 == 0 || rows == 1);
  if (vec_ok && (uintptr_t) out % 16 == 0 && (out_row_bytes % 16 == 0 || rows == 1))
    vec_ok = 2;  // 128-bit stores on the PCM side too
  dim3 grid(grid_x_for(row_samples, rows), rows);
  switch (nbytes) {
    case 1:
      espb_f2q_kernel<1><<<grid, 256, 0, stream>>>(in, in_row_floats, out, out_row_bytes, row_samples, c, clipped,
                                                  clipped_per_row, vec_ok);
      break;
    case 2:
      espb_f2q_kernel<2><<<grid, 256, 0, stream>>>(in, in_row_floats, out, out_row_bytes, row_samples, c, clipped,
                                                  clipped_per_row, vec_ok);
      break;
    case 3:
      espb_f2q_kernel<3><<<grid, 256, 0, stream>>>(in, in_row_floats, out, out_row_bytes, row_samples, c, clipped,
                                                  clipped_per_row, vec_ok);
      break;
    case 4:
      espb_f2q_kernel<4><<<grid, 256, 0, stream>>>(in, in_row_floats, out, out_row_bytes, row_samples, c, clipped,
                                                  clipped_per_row, vec_ok);
      break;
    default:
      return cudaErrorInvalidValue;
  }
  count_launch();
  return cudaGetLastError();
}

// Frames [0, n_frames) (n_frames a multiple of 64) of every stream -> rows row_first.. of tm.  Returns the
// number of frames handled: 0 when the layout does not qualify (caller falls back to q2f + transpose).
int launch_pcm_to_tm(const uint8_t *in, int64_t in_row_bytes, int bits, float gain_factor, int channels, int n_series,
                     int n_frames, float *tm, int64_t rows_cap, int row_first, cudaStream_t stream, cudaError_t *err) {
  *err = cudaSuccess;
  const int fast = (n_frames / PT_ROWS) * PT_ROWS;
  if (fast <= 0 || ((uintptr_t) in % 4) || (in_row_bytes % 4) || n_series <= 0)
    return 0;
  const int nbytes = (bits + 7) / 8;
  if (nbytes < 1 || nbytes > 4 || !(channels == 1 || channels == 2 || channels == 4 || channels == 8))
    return 0;
  // tiles of frames ride on y: a slice starting at tile y0 reads from frame y0 * PT_ROWS on
  *err = for_each_y_slice(fast / PT_ROWS, [&](int y0, int ny) {
    const dim3 grid((n_series + SGN - 1) / SGN, ny);
    const uint8_t *in_y = in + (int64_t) y0 * PT_ROWS * channels * nbytes;
    const int row_y = row_first + y0 * PT_ROWS;
    switch (nbytes) {
      case 1:
        launch_pcm_to_tm_ch<1>(channels, grid, stream, in_y, in_row_bytes, tm, rows_cap, row_y, n_series, gain_factor);
        break;
      case 2:
        launch_pcm_to_tm_ch<2>(channels, grid, stream, in_y, in_row_bytes, tm, rows_cap, row_y, n_series, gain_factor);
        break;
      case 3:
        launch_pcm_to_tm_ch<3>(channels, grid, stream, in_y, in_row_bytes, tm, rows_cap, row_y, n_series, gain_factor);
        break;
      default:
        launch_pcm_to_tm_ch<4>(channels, grid, stream, in_y, in_row_bytes, tm, rows_cap, row_y, n_series, gain_factor);
        break;
    }
    count_launch();
    return cudaGetLastError();
  });
  return fast;
}

// Rows [row_first, row_first + n_frames) of tm -> frames [0, n_frames) of every stream's PCM row.
int launch_tm_to_pcm(const float *tm, int64_t rows_cap, int row_first, int n_frames, uint8_t *out,
                     int64_t out_row_bytes, int bits, int channels, int n_series, uint32_t *clipped_per_stream,
                     cudaStream_t stream, cudaError_t *err) {
  *err = cudaSuccess;
  const int fast = (n_frames / PT_ROWS) * PT_ROWS;
  if (fast <= 0 || ((uintptr_t) out % 4) || (out_row_bytes % 4) || n_series <= 0)
    return 0;
  const int nbytes = (bits + 7) / 8;
  if (nbytes < 1 || nbytes > 4 || !(channels == 1 || channels == 2 || channels == 4 || channels == 8))
    return 0;
  const F2QConst c = make_f2q_const(bits);
  // tiles of frames ride on y: a slice starting at tile y0 writes from frame y0 * PT_ROWS on
  *err = for_each_y_slice(fast / PT_ROWS, [&](int y0, int ny) {
    const dim3 grid((n_series + SGN - 1) / SGN, ny);
    const int row_y = row_first + y0 * PT_ROWS;
    uint8_t *out_y = out + (int64_t) y0 * PT_ROWS * channels * nbytes;
    switch (nbytes) {
      case 1:
        launch_tm_to_pcm_ch<1>(channels, grid, stream, tm, rows_cap, row_y, out_y, out_row_bytes, n_series, c, clipped_per_stream);
        break;
      case 2:
        launch_tm_to_pcm_ch<2>(channels, grid, stream, tm, rows_cap, row_y, out_y, out_row_bytes, n_series, c, clipped_per_stream);
        break;
      case 3:
        launch_tm_to_pcm_ch<3>(channels, grid, stream, tm, rows_cap, row_y, out_y, out_row_bytes, n_series, c, clipped_per_stream);
        break;
      default:
        launch_tm_to_pcm_ch<4>(channels, grid, stream, tm, rows_cap, row_y, out_y, out_row_bytes, n_series, c, clipped_per_stream);
        break;
    }
    count_launch();
    return cudaGetLastError();
  });
  return fast;
}

}  // namespace espb
