// Launch wrappers for the sm_100a kernels (internal; the public boundary is include/esp_audio_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "common.hpp"

namespace espb {

void count_launch();  // bumps the process-wide kernel-launch counter (api.cu)

// CUDA refuses a launch whose gridDim.y exceeds 65,535 (every compute capability).  Launchers that put frames,
// outputs, time blocks, passes or groups on y enqueue one launch per slice of at most grid_y_max() along y; each
// kernel takes the slice's first index through an offset it already has (a starting frame or pass, advanced pointers).
constexpr int kMaxGridY = 65535;
int grid_y_max();  // kMaxGridY; ESPB_GRID_Y_MAX (read once, clamped to [1, kMaxGridY]) lowers it to test the slicing
// launch(first, count) for consecutive slices [first, first + count) of [0, total); stops at the first error
template <class F>
cudaError_t for_each_y_slice(int64_t total, F &&launch) {
  const int64_t step = grid_y_max();
  for (int64_t y0 = 0; y0 < total; y0 += step) {
    const cudaError_t e = launch((int) y0, (int) (total - y0 < step ? total - y0 : step));
    if (e != cudaSuccess)
      return e;
  }
  return cudaSuccess;
}

// Function attributes (dynamic shared-memory size, carve-out) are per device: one flag per device and kernel.
struct PerDeviceOnce {
  bool done[64] = {};
  // true the first time it is asked on the current device
  bool first() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
      return true;
    const bool was = done[dev];
    done[dev] = true;
    return !was;
  }
};

struct ResampleParams {
  const float *xt;  // time-major input staging of the first group of this launch: [group][xt_rows][128]
  int64_t xt_rows;  // rows per group (row r = input frame r - taps)
  float *out;
  int64_t out_ss, out_cs, out_fs;  // stream / channel / frame strides of the caller's output, floats
  float *out_tm;                   // if not NULL: write time-major yt[group][out_tm_rows][128] instead of `out`
  int64_t out_tm_rows;
  const float *G;                  // expanded coefficients, chunk-major, starting at chunk g_chunk_base
  const ChunkEntry *chunks;
  const int32_t *pass_chunk_begin;
  const OutEntry *outs;
  int n_series, channels, n_out, taps;
  int pass_first, pass_end, passes_per_cta, g_chunk_base;
  int out_vec;  // OutVec: set by launch_resample from the output layout
  // staging overlap: if not NULL, input frames [t * 32, t * 32 + 32) of every group are in xt once ready[t] has
  // reached ready_target (t < ready_tiles; rows past the last tile were staged before the launch) — the kernel was
  // launched as a programmatic dependent of the transposing kernel and waits per CTA for the tiles it reads
  const int *ready;
  int ready_tiles, ready_target;
};
constexpr int kReadyTileRows = 32;
enum OutVec : int { kOutVecNone = 0, kOutVecPlanar = 1, kOutVecStereo = 2, kOutVecFrame4 = 3, kOutVecTimeMajor = 4 };

size_t resample_smem_bytes(int bpp, int g_row_floats = kGRowFloats);
size_t g_chunk_floats(int bpp, int g_row_floats = kGRowFloats);
cudaError_t launch_expand_schedule(const SchedSegment *segs, int n_segs, OutEntry *outs, int n, int n_filters,
                                   bool lowpass, bool interp, cudaStream_t stream);
cudaError_t launch_expand(const float *bank, const OutEntry *outs, const ChunkEntry *chunks, float *G,
                          int chunk_first, int n_chunks, int n_out, int taps, int bpp, cudaStream_t stream,
                          int g_row_floats = kGRowFloats);
cudaError_t launch_resample(const ResampleParams &p, bool exact, cudaStream_t stream, bool non_interpolating = false);
// non-interpolating form (resample_ni_kernel.cu): G rows of kGRowFloatsNI floats
cudaError_t launch_resample_ni(const ResampleParams &q, int n_groups, int n_ctas_y, bool exact, bool tm,
                               cudaStream_t stream);
cudaError_t launch_transpose(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels, int n_series,
                             int n_in, float *xt, int64_t rows_cap, int row_first, int pad_rows,
                             cudaStream_t stream);
// staging arranged for overlap with the resampler launch that must follow immediately (ResampleParams::ready)
cudaError_t launch_transpose_flags(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                                   int n_series, int n_in, float *xt, int64_t rows_cap, int row_first, int pad_rows,
                                   int *ready, int ctas_per_sm, cudaStream_t stream, int *n_tiles);

// Fused clock groups (groups.cu): one launch serves every group of a set; blockIdx.y selects the group.  Offsets are
// in floats / entries relative to the pointers in FsParams.
struct FsGroupDesc {
  int64_t x_off;      // this group's staging rows inside the current staging buffer
  int64_t x_old_off;  // ... inside the previous one (the carried frames)
  int64_t out_off;    // first stream of the group in the caller's output
  int64_t in_off;     // ... in the caller's input
  int64_t outs_begin;           // first entry of the group in the concatenated schedule
  int32_t n_in, n_out;
  int32_t seg_begin, n_segs;    // its runs in the concatenated segment table
  int32_t carry_row;            // row of the previous staging buffer where the carried frames start
};
// small calls: carried frames (rows [carry_row, carry_row + taps) of old_xt) + new input + zero padding in one launch
cudaError_t launch_stage_small(const float *old_xt, int carry_row, int taps, const float *in, int64_t in_ss,
                               int64_t in_cs, int64_t in_fs, int channels, int n_series, int n_in, float *xt,
                               int64_t rows_cap, int pad_rows, cudaStream_t stream);
// planar buffers given as one device pointer per (stream, channel) plane (the table itself in device memory)
cudaError_t launch_transpose_ptrs(const float *const *planes_dev, int n_series, int n_in, float *xt, int64_t rows_cap,
                                  int row_first, int pad_rows, cudaStream_t stream);
cudaError_t launch_untranspose_ptrs(const float *tm, int64_t rows_cap, int row_first, int n_rows,
                                    float *const *planes_dev, int n_series, cudaStream_t stream);

// Few-series form (resample_fs_kernel.cu): lanes own outputs instead of series; no expanded coefficients, no
// chunk tables — the finalized schedule, the time-major staging rows and a slice-major copy of the bank.
struct FsParams {
  const float *x;    // frame j of series q: x[(j + x_row0) * x_fs + q]
  int64_t x_fs;
  int x_row0;
  float *out;
  int64_t out_ss, out_cs, out_fs;
  float *out_tm;     // if not NULL: time-major rows of 128 floats instead of `out`
  const float *bank_tr;  // [taps / kt][slice_floats]
  const OutEntry *outs;  // finalized
  int n_series, channels, n_out, taps;
  int kt, slice_floats;
  int q_per_out, x_tile_floats, out_vec, x_pitch, stages;  // set by the launcher
  const FsGroupDesc *groups;              // fused clock groups: per-group offsets and counts (blockIdx.y), else NULL
};
struct FsGeometry {
  int sv, b, q;          // series per lane, outputs per lane, lanes per output
  int outputs_per_cta;
};
constexpr int kFsMaxSeries = 32;
int fs_slice_taps(int taps, int filters);
size_t fs_slice_floats(int filters, int kt);
void fs_build_bank_slices(const float *bank, int taps, int filters, int kt, float *dst);
FsGeometry fs_geometry(int n_series);
size_t fs_smem_bytes(const FsGeometry &g, size_t slice_floats, int x_rows);
cudaError_t launch_resample_fs(const FsParams &p, const FsGeometry &g, int x_rows, bool exact, cudaStream_t stream,
                               int n_groups = 1);
// fused clock groups: carried frames + new input of every group -> compact time-major staging rows [row][pitch]
cudaError_t launch_fsg_stage(const FsGroupDesc *groups, int n_groups, const float *old_buf, float *new_buf, int pitch,
                             int taps, const float *in, int64_t in_ss, int channels, int n_series, int max_rows,
                             cudaStream_t stream);
// ... and the per-output schedule entries of every group from the concatenated segment table
cudaError_t launch_expand_schedule_groups(const FsGroupDesc *groups, int n_groups, const SchedSegment *segs,
                                          OutEntry *outs, int max_n_out, int n_filters, bool lowpass, bool interp,
                                          cudaStream_t stream);

// quantization_utils
cudaError_t launch_q2f(const uint8_t *in, int64_t in_row_bytes, float *out, int64_t out_row_floats, int rows,
                       uint32_t row_samples, int bits, float gain_factor, cudaStream_t stream);
cudaError_t launch_f2q(const float *in, int64_t in_row_floats, uint8_t *out, int64_t out_row_bytes, int rows,
                       uint32_t row_samples, int bits, uint32_t *clipped, bool clipped_per_row, cudaStream_t stream);

// PCM <-> time-major float, fused conversion + layout change (full 64-frame tiles, channels in {1,2,4,8},
// 4-byte aligned PCM rows).  Return the number of frames handled (0: not applicable, use the separate stages).
int launch_pcm_to_tm(const uint8_t *in, int64_t in_row_bytes, int bits, float gain_factor, int channels, int n_series,
                     int n_frames, float *tm, int64_t rows_cap, int row_first, cudaStream_t stream, cudaError_t *err);
int launch_tm_to_pcm(const float *tm, int64_t rows_cap, int row_first, int n_frames, uint8_t *out,
                     int64_t out_row_bytes, int bits, int channels, int n_series, uint32_t *clipped_per_stream,
                     cudaStream_t stream, cudaError_t *err);
// the stage-by-stage twins with a starting frame (tails after the fused tiles, other layouts)
cudaError_t launch_transpose_from(const float *in, int64_t in_ss, int64_t in_cs, int64_t in_fs, int channels,
                                  int n_series, int n_in, float *xt, int64_t rows_cap, int row_first, int j_begin,
                                  int pad_rows, cudaStream_t stream);
cudaError_t launch_untranspose_from(const float *tm, int64_t rows_cap, int row_first, int j_begin, int n_rows,
                                    float *out, int64_t out_ss, int64_t out_cs, int64_t out_fs, int channels,
                                    int n_series, cudaStream_t stream);

// art_biquad
struct BiquadParams {
  float a0, a1, a2, b1, b2;
  int first_order;
};
// time-major filter of rows [row_first, row_first + n_rows) of src[group][rows_cap][128] into dst (same
// geometry; may be src itself when block_rows == 0).  block_rows > 0: time blocks with warm_rows of warm-up.
// Time blocks need `blk_state` (biquad_block_state_floats() floats: the state every block reached at its first row and
// at its end, which espb_biquad_verify_kernel compares — and repairs where they differ — before committing the final
// state) and may be given a counter of repaired blocks.
size_t biquad_block_state_floats(int n_series, int n_sections, int n_rows, int block_rows);
// banks of at most this many series (one group) run their time blocks as (block, series) threads: shorter blocks pay
constexpr int kBiquadFewSeries = 32;
// the same filter in ONE pass on the caller's layout (interleaved or frame-contiguous; cudaErrorNotSupported else)
cudaError_t launch_biquad_cl(float *buf, int64_t ss, int64_t cs, int64_t fs, int channels, int n_series, int n_frames,
                             int n_sections, BiquadParams c, float *state, cudaStream_t stream);
cudaError_t launch_biquad_tm(const float *src, float *dst, int64_t rows_cap, int row_first, int n_rows, int n_series,
                             int n_sections, BiquadParams c, float *state /* [series][section][4] */,
                             int block_rows, int warm_rows, cudaStream_t stream, float *blk_state = nullptr,
                             unsigned int *mismatches = nullptr, unsigned int *chain_broken = nullptr);
// (chain_broken: one scratch word per group of the launch; with it the hand-overs are compared in parallel first and
//  the sequential walk is taken only by groups in which one differs)
// mono streams: post-filter + float_to_quantized in one pass (biquad_kernel.cu); returns the frames written as PCM
int launch_biquad_tm_pcm(float *buf, int64_t rows_cap, int row_first, int n_rows, int n_series, int n_sections,
                         BiquadParams c, float *state, uint8_t *out, int64_t out_row_bytes, int bits,
                         uint32_t *clipped_per_stream, cudaStream_t stream, cudaError_t *err);
// time-major -> caller layout (inverse of launch_transpose): rows [row_first, row_first + n_rows)
cudaError_t launch_untranspose(const float *tm, int64_t rows_cap, int row_first, int n_rows, float *out,
                               int64_t out_ss, int64_t out_cs, int64_t out_fs, int channels, int n_series,
                               cudaStream_t stream);

// dsp.h Q15 helpers (element strides; any of the buffers may alias as in the reference)
cudaError_t launch_add_s16(const int16_t *a, const int16_t *b, int16_t *out, uint64_t n, int64_t s1, int64_t s2,
                           int64_t so, int shift, cudaStream_t stream);
cudaError_t launch_mulc_s16(const int16_t *a, int16_t *out, uint64_t n, int16_t c, int64_t si, int64_t so,
                            cudaStream_t stream);

// utilities
cudaError_t launch_checksum(const uint32_t *words, uint64_t n, unsigned long long *sum_dev, cudaStream_t stream);
cudaError_t run_tile_probe(double *tflops);
cudaError_t run_fma_probe(double *tflops, double *clock_mhz, double *tflops_scalar, double *tflops_packed);

}  // namespace espb
