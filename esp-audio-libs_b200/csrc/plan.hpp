// Host-side planning for the B200 ART resampler path: everything that is
// signal-independent is computed here once per call and shared by all streams.
#pragma once
#include <stdlib.h>

#include <vector>

#include "common.hpp"

namespace espb {

constexpr int kFlagInterpolate = 0x1, kFlagBlackmanHarris = 0x2, kFlagLowpass = 0x4;

// Position state of a context (include/art_resampler.h:25-29: outputOffset, inputIndex).
struct ArtState {
  float offset;
  int index;
};

struct ArtGeometry {
  int taps, filters, flags;
};

// resampleInit's parameter normalisation (art_resampler.cpp:82-97).  Returns false (after
// printing the reference's stderr line) for invalid taps / filters.
bool normalise_init(int taps, int filters, float *lowpass, int *flags);

// The (filters+1) x taps windowed-sinc bank, bit-identical to init_filter
// (art_resampler.cpp:379-419); needs the same libm (glibc sinf/cosf) as the reference.
void build_filter_bank(const ArtGeometry &g, float lowpass, std::vector<float> &bank);

ArtState initial_state(int taps);  // art_resampler.cpp:135-136

// Growable array of plain structs without value-initialisation (the schedule tables are written once,
// front to back, right after sizing).
// The owner may hook the (rare) moments the storage moves — the CUDA layer page-locks the tables so that their
// uploads are asynchronous DMA copies instead of staged ones; this header itself stays free of CUDA.
template <typename T>
struct PodBuffer {
  T *ptr = nullptr;
  size_t count = 0, cap = 0;
  void (*on_release)(void *p) = nullptr;               // called before the storage is moved or freed
  void (*on_acquire)(void *p, size_t bytes) = nullptr;  // called after new storage has been obtained
  PodBuffer() = default;
  PodBuffer(const PodBuffer &) = delete;
  PodBuffer &operator=(const PodBuffer &) = delete;
  ~PodBuffer() {
    if (ptr && on_release)
      on_release(ptr);
    free(ptr);
  }
  void reserve(size_t n) {
    if (n > cap) {
      n += n / 8 + 64;  // head-room: table sizes wander from call to call, and moving a page-locked table is costly
      if (ptr && on_release)
        on_release(ptr);
      ptr = static_cast<T *>(realloc(ptr, n * sizeof(T)));
      cap = n;
      if (ptr && on_acquire)
        on_acquire(ptr, cap * sizeof(T));
    }
  }
  void clear() { count = 0; }
  void swap_storage(PodBuffer &o) {  // (both sides are expected to carry the same hooks)
    T *p = ptr;
    ptr = o.ptr;
    o.ptr = p;
    size_t t = count;
    count = o.count;
    o.count = t;
    t = cap;
    cap = o.cap;
    o.cap = t;
  }
  void push_back(const T &v) {
    if (count == cap)
      reserve(cap ? cap * 2 : 1024);
    ptr[count++] = v;
  }
  T *data() { return ptr; }
  const T *data() const { return ptr; }
  size_t size() const { return count; }
  T &operator[](size_t i) { return ptr[i]; }
  const T &operator[](size_t i) const { return ptr[i]; }
};

struct Schedule {
  PodBuffer<OutEntry> outs;       // per-output entries (sequential form; empty in the segmented form)
  PodBuffer<SchedSegment> segs;   // segmented form: arithmetic-progression runs, expanded on the device
  bool segmented = false;
  unsigned used = 0, generated = 0;
  ArtState end{};
};

// Data-free run of the resampleProcess state machine (art_resampler.cpp:172-199 /
// :213-240) that records, per output, the window start / phase / weight / kind.
void build_schedule(const ArtGeometry &g, ArtState start, int n_in, int n_out, float ratio, Schedule &s);
// The same schedule in closed form.  The offset is a sequential FP32 accumulator (art_resampler.cpp:195,236), but
// inside one binade every addition of the same step rounds the same way, so the offsets of consecutive outputs are an
// exact arithmetic progression until the offset crosses a power of two or the ring is rebased (:175-181).  The host
// walks those pieces (a handful per ring cycle of 15 x taps input frames: O(frames / taps) work instead of
// O(frames)), using real float additions at every piece boundary and the sequential machine wherever the closed form
// does not apply (tie roundings, the end of the input); the per-output entries are expanded on the device
// (espb_expand_schedule_kernel).  Bit-identical to build_schedule by construction and by test (test_host_plan.py).
void build_schedule_segments(const ArtGeometry &g, ArtState start, int n_in, int n_out, float ratio, Schedule &s);
// window start of output k of either form (segment lookup through *cursor, which callers walk monotonically)
int32_t schedule_ws(const Schedule &s, int k, int *cursor);
// host expansion of the segmented form into finalized entries (host API, tests)
void expand_segments(const ArtGeometry &g, const Schedule &s, OutEntry *out);
// Second pass of the schedule (host version; espb_expand_schedule_kernel has the device twin).
void finalize_entries(const ArtGeometry &g, OutEntry *entries, size_t n);

unsigned required_samples(const ArtGeometry &g, ArtState st, int n_out, float ratio);  // :257-279
unsigned expected_output(const ArtGeometry &g, ArtState st, int n_in, float ratio);    // :281-306
float position_of(const ArtGeometry &g, ArtState st);                                   // :348

// Pass / chunk tables for the kernel: pass p covers outputs [p*opp, (p+1)*opp) and
// sweeps input rows [ws(first), ws(last)+taps) in chunks of chunk_rows (<= kChunkRows).
struct PassPlan {
  int outputs_per_pass = 0;
  PodBuffer<ChunkEntry> chunks;
  PodBuffer<int32_t> pass_chunk_begin;  // n_passes + 1 prefix
  int n_passes() const { return (int) pass_chunk_begin.size() - 1; }
};
void build_pass_plan(const Schedule &s, int taps, int blocks_per_pass, int chunk_rows, PassPlan &p);

// art_biquad.cpp:16-38 (design in double, stored as float).
struct BiquadCoeffs {
  float a0, a1, a2, b1, b2;
};
void design_lowpass(BiquadCoeffs *c, double frequency);
void design_highpass(BiquadCoeffs *c, double frequency);

// Resampler::initialize policy (resampler.cpp:38-94).
struct WrapperPolicy {
  bool resampling = false, pre = false, post = false;
  float sample_ratio = 1.0f, lowpass_ratio = 1.0f, art_lowpass = 1.0f;
  int art_flags = 0;
  BiquadCoeffs coeffs{};
};
void decide_policy(float src_rate, float dst_rate, int taps, bool use_filter, bool interpolate, WrapperPolicy *p);

// quantization_utils.cpp:8,11,18,27,37 — the per-call scale factor (host powf).
float q2f_gain_factor(int bits, float gain_db);

}  // namespace espb
