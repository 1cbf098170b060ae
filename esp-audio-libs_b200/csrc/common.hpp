// Shared host/device definitions for the B200 ART resampler path.
#pragma once
#include <stdint.h>

namespace espb {

// Tile geometry of the resampler kernel (see DESIGN.md "Resampler kernel").
constexpr int kOutputsPerBlock = 8;   // NB: outputs accumulated per thread
constexpr int kChunkRows = 40;        // zero rows staged after the input (a chunk reads up to 31 rows past a window)
constexpr int kSeriesPerRow = 128;    // series (stream x channel) per warp row: 32 lanes x 4
constexpr int kGRowFloats = 2 * kOutputsPerBlock;  // 16 coefficients per (row, output block)
constexpr int kGRowFloatsNI = kOutputsPerBlock;    // 8 in the non-interpolating form (one filter per output)
constexpr int kNiBlocksPerWarp = 2;  // ... whose warps own two adjacent blocks each: its pass plan has 8 blocks per pass
// The resampler kernels' geometry: 4 warps per CTA (one output block each per pass), four CTAs per SM, input rows
// streamed in 32-row chunks through a 2-stage shared-memory ring.
constexpr int kResampleWarps = 4;
constexpr int kResampleStages = 2;
constexpr int kResampleChunkRows = 32;
constexpr int kMaxChunksPerCta = 320;  // chunk-table entries a CTA caches in shared memory
constexpr int kMaxPassesPerCta = 64;

// What the reference does for one output sample (art_resampler.cpp:421-451).
enum OutKind : int32_t {
  kKindNone = 0,    // padding past the last output of the call
  kKindPass = 1,    // fractional offset == 0 and no low-pass: *source        (:425, :439)
  kKindSingle = 2,  // one dot product (non-interpolating, or blend weight 0) (:428, :445)
  kKindBlend = 3,   // sum2*w + sum1*(1-w)                                    (:450)
};

// One entry of the position schedule: everything about output n that does not depend
// on the signal.  `ws` is the index (relative to the first input frame of this call;
// negative = carried history) of the first of the numTaps window samples.
struct OutEntry {
  int32_t ws;
  int32_t phase;   // filter row of sum1 (row phase+1 is sum2)
  float w;         // blend weight
  int32_t kind;    // OutKind
};

// A run of consecutive outputs whose offsets form an exact arithmetic progression (plan.cpp:build_schedule_segments):
// output n0 + j has offset off0 + j * inc (exact: all terms are multiples of one ulp) and window start
// ws_base + floor(offset).  The host emits a few of these per ring cycle; the device expands them into OutEntry.
struct SchedSegment {
  int32_t n0, count;
  int32_t ws_base;
  float off0, inc;
};

// One pipeline chunk: kChunkRows consecutive input frames starting at j_start that
// belong to pass `pass` (a pass = blocks_per_pass output blocks sharing one sweep).
struct ChunkEntry {
  int32_t j_start;
  int32_t pass;
};

}  // namespace espb
