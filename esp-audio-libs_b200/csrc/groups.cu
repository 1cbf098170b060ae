// Ratio groups: per-stream / time-varying resampling ratios (ASRC; SURVEY.md §8f N1).
//
// In the reference every stream owns a context and `ratio` is an argument of every resampleProcess call
// (art_resampler.cpp:57-62, :167, :208), so two streams may run at different, drifting ratios.  The batched
// kernel shares the position schedule and the expanded coefficients among the streams of a context, which
// needs them in lock-step.  Streams that follow the same clock (same ratio trajectory, same chunking) form a
// *group*; a group set holds one batch context per group and runs the groups of a call concurrently on
// internal CUDA streams forked from / joined to the caller's stream.  Every group keeps its own persistent
// device-side state (history, position), so calls may be chunked freely and each group's ratio may change
// from call to call.
//
// Two forms.  Groups of any size: one batch context per group, run concurrently on internal CUDA streams (the generic
// form; each group is a launch sequence of its own, so it suits a few large groups).  MANY SMALL groups — every group
// the same number of streams and at most 32 series, the "one clock per stream" case — are FUSED: the set owns one
// compact staging buffer, one schedule table and one copy of the filter bank, the host only plans (closed-form
// schedule, about a microsecond per group) and fills one descriptor per group, and a call is four operations
// whatever the number of groups: one upload (descriptors + schedule runs), one staging kernel (carried frames and
// new input of every group), one schedule-expansion kernel, one launch of the few-series resampler kernel with
// blockIdx.y = group.  Per-group position state lives in state-only contexts (espb_resampleGroupsContext), so
// advance / position / required / expected work per group exactly as on a context of the reference.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/esp_audio_b200.h"
#include "internal.hpp"
#include "kernels.hpp"
#include "plan.hpp"

using namespace espb;

namespace {

// The fused form (see the header of this file).
struct FusedSet {
  int n_groups = 0, streams_per_group = 0, channels = 0, n_series = 0, pitch = 0;
  ArtGeometry geo{};
  FsGeometry fg{};
  int kt = 0;
  size_t slice_floats = 0;
  float *bank_tr = nullptr;
  float *buf[2] = {nullptr, nullptr};  // [group][rows_cap][pitch] staging rows; the two alternate from call to call
  int cur = 0;
  int64_t rows_cap = 0;
  std::vector<int> carry_row;          // per group: where its carried frames start in buf[cur]
  OutEntry *d_outs = nullptr;
  size_t outs_cap = 0;
  // per-call blob: [n_groups] FsGroupDesc, then the schedule runs of all groups; two pinned copies alternate
  unsigned char *h_blob[2] = {nullptr, nullptr};
  size_t h_cap[2] = {0, 0};
  cudaEvent_t h_done[2] = {nullptr, nullptr};
  bool h_pending[2] = {false, false};
  int h_cur = 0;
  unsigned char *d_blob = nullptr;
  size_t d_cap = 0;
  Schedule sched;  // scratch of the planner
};

}  // namespace

struct EspbResampleGroups {
  int channels = 0;
  int device = 0;
  std::vector<EspbResampleBatch *> ctx;
  std::vector<int> first_stream, n_streams;
  std::vector<cudaStream_t> streams;
  std::vector<cudaEvent_t> joined;
  cudaEvent_t fork = nullptr;
  FusedSet *fused = nullptr;
};

namespace {

void fused_free(FusedSet *f) {
  if (!f)
    return;
  cudaFree(f->bank_tr);
  cudaFree(f->buf[0]);
  cudaFree(f->buf[1]);
  cudaFree(f->d_outs);
  cudaFree(f->d_blob);
  for (int i = 0; i < 2; ++i) {
    if (f->h_done[i]) {
      cudaEventSynchronize(f->h_done[i]);
      cudaEventDestroy(f->h_done[i]);
    }
    if (f->h_blob[i])
      cudaFreeHost(f->h_blob[i]);
  }
  delete f;
}

// Both staging buffers hold at least `rows` rows per group; the carried frames move along.
int fused_ensure_rows(FusedSet *f, int64_t rows) {
  if (rows <= f->rows_cap)
    return ESPB_OK;
  rows = rows + rows / 4 + 64;
  const size_t bytes = (size_t) f->n_groups * rows * f->pitch * sizeof(float);
  float *nb[2] = {nullptr, nullptr};
  cudaError_t e = f->rows_cap > 0 ? cudaDeviceSynchronize() : cudaSuccess;  // earlier calls may still use the old rows
  if (e == cudaSuccess)
    e = cudaMalloc(&nb[0], bytes);
  if (e == cudaSuccess)
    e = cudaMalloc(&nb[1], bytes);
  if (e == cudaSuccess)
    e = cudaMemset(nb[0], 0, bytes);
  if (e == cudaSuccess)
    e = cudaMemset(nb[1], 0, bytes);
  const size_t row_bytes = (size_t) f->pitch * sizeof(float);
  for (int g = 0; g < f->n_groups && e == cudaSuccess && f->rows_cap > 0; ++g)  // carried frames -> rows [0, taps)
    e = cudaMemcpy(nb[0] + (size_t) g * rows * f->pitch,
                   f->buf[f->cur] + ((size_t) g * f->rows_cap + f->carry_row[g]) * f->pitch, f->geo.taps * row_bytes,
                   cudaMemcpyDeviceToDevice);
  if (e != cudaSuccess) {
    cudaFree(nb[0]);
    cudaFree(nb[1]);
    return api_fail(ESPB_ERR_CUDA, "clock groups: staging buffers", cudaGetErrorString(e));
  }
  cudaFree(f->buf[0]);
  cudaFree(f->buf[1]);
  f->buf[0] = nb[0];
  f->buf[1] = nb[1];
  f->cur = 0;
  f->rows_cap = rows;
  for (int &c : f->carry_row)
    c = 0;
  return ESPB_OK;
}

FusedSet *fused_create(int n_groups, int streams_per_group, int channels, const ArtGeometry &geo,
                       const std::vector<float> &bank) {
  FusedSet *f = new (std::nothrow) FusedSet();
  if (!f)
    return nullptr;
  f->n_groups = n_groups;
  f->streams_per_group = streams_per_group;
  f->channels = channels;
  f->n_series = streams_per_group * channels;
  f->geo = geo;
  f->fg = fs_geometry(f->n_series);
  f->pitch = f->fg.q * f->fg.sv;
  f->kt = fs_slice_taps(geo.taps, geo.filters);
  f->slice_floats = fs_slice_floats(geo.filters, f->kt);
  f->carry_row.assign(n_groups, 0);
  std::vector<float> tr(f->slice_floats * (geo.taps / f->kt));
  fs_build_bank_slices(bank.data(), geo.taps, geo.filters, f->kt, tr.data());
  cudaError_t e = cudaMalloc(&f->bank_tr, tr.size() * sizeof(float));
  if (e == cudaSuccess)
    e = cudaMemcpy(f->bank_tr, tr.data(), tr.size() * sizeof(float), cudaMemcpyHostToDevice);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i)
    e = cudaEventCreateWithFlags(&f->h_done[i], cudaEventDisableTiming);
  if (e != cudaSuccess || fused_ensure_rows(f, geo.taps + 64) != ESPB_OK) {
    fused_free(f);
    return nullptr;
  }
  return f;
}

int fused_process(EspbResampleGroups *g, const float *in, int64_t in_ss, const int *n_in, float *out, int64_t out_ss,
                  const int *n_out, const float *ratios, EspbResampleResult *results, cudaStream_t stream) {
  FusedSet *f = g->fused;
  const int G = f->n_groups, T = f->geo.taps;
  {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != g->device)
      return api_fail(ESPB_ERR_STATE, "clock groups: created on another CUDA device (espb_set_device before the call)");
  }
  int max_in = 0;
  for (int k = 0; k < G; ++k) {
    if (!(ratios[k] > 0.0f) || !(ratios[k] <= 3.0e38f))
      return api_fail(ESPB_ERR_ARG, "clock groups: every ratio must be a positive finite number");
    const int n = n_in[k] > 0 ? n_in[k] : 0;
    max_in = n > max_in ? n : max_in;
  }
  if (int rc = fused_ensure_rows(f, (int64_t) T + max_in))
    return rc;
  // ---- plan: one closed-form schedule per group, into the pinned blob of this call
  const int hb = f->h_cur;
  f->h_cur = 1 - f->h_cur;
  if (f->h_pending[hb]) {  // (the upload of the call before the previous one: long finished in a stream of calls)
    cudaEventSynchronize(f->h_done[hb]);
    f->h_pending[hb] = false;
  }
  std::vector<FsGroupDesc> desc(G);
  std::vector<SchedSegment> segs;
  segs.reserve((size_t) G * 8);
  std::vector<ArtState> end_state(G);
  size_t total_out = 0;
  int max_out = 0, max_rows = 0, x_rows = T;
  const int m = f->fg.outputs_per_cta;
  for (int k = 0; k < G; ++k) {
    const int ni = n_in[k] > 0 ? n_in[k] : 0;
    build_schedule_segments(f->geo, context_state(g->ctx[k]), ni, n_out[k], ratios[k], f->sched);
    const int gen = (int) f->sched.generated;
    results[k].input_used = f->sched.used;
    results[k].output_generated = f->sched.generated;
    end_state[k] = f->sched.end;
    FsGroupDesc &d = desc[k];
    d.x_off = (int64_t) k * f->rows_cap * f->pitch;
    d.x_old_off = d.x_off;
    d.out_off = (int64_t) g->first_stream[k] * out_ss;
    d.in_off = (int64_t) g->first_stream[k] * in_ss;
    d.n_in = ni;
    d.n_out = gen;
    d.outs_begin = (int64_t) total_out;
    d.seg_begin = (int32_t) segs.size();
    d.n_segs = (int32_t) f->sched.segs.size();
    d.carry_row = f->carry_row[k];
    for (size_t i = 0; i < f->sched.segs.size(); ++i)
      segs.push_back(f->sched.segs[i]);
    int cursor = 0;
    for (int first = 0; first < gen; first += m) {  // widest input tile of a CTA (its first window .. last window + taps)
      const int last = (first + m < gen ? first + m : gen) - 1;
      const int w0 = schedule_ws(f->sched, first, &cursor);
      const int span = schedule_ws(f->sched, last, &cursor) - w0 + T;
      x_rows = span > x_rows ? span : x_rows;
    }
    total_out += (size_t) gen;
    max_out = gen > max_out ? gen : max_out;
    max_rows = T + ni > max_rows ? T + ni : max_rows;
  }
  if (total_out > 0 && fs_smem_bytes(f->fg, f->slice_floats, x_rows) > (size_t) 200 * 1024)
    return api_fail(ESPB_ERR_ARG, "clock groups: ratio too small for the fused form (input tile exceeds shared memory)");
  const size_t blob_bytes = (size_t) G * sizeof(FsGroupDesc) + segs.size() * sizeof(SchedSegment);
  if (blob_bytes > f->h_cap[hb]) {
    if (f->h_blob[hb])
      cudaFreeHost(f->h_blob[hb]);
    f->h_blob[hb] = nullptr;
    f->h_cap[hb] = 0;
    if (cudaMallocHost(&f->h_blob[hb], blob_bytes * 2) != cudaSuccess)
      return api_fail(ESPB_ERR_NOMEM, "clock groups: pinned tables");
    f->h_cap[hb] = blob_bytes * 2;
  }
  if (blob_bytes > f->d_cap) {
    cudaFree(f->d_blob);  // (waits for earlier work that may still read it)
    f->d_blob = nullptr;
    f->d_cap = 0;
    if (cudaMalloc(&f->d_blob, blob_bytes * 2) != cudaSuccess)
      return api_fail(ESPB_ERR_NOMEM, "clock groups: device tables");
    f->d_cap = blob_bytes * 2;
  }
  if (total_out > f->outs_cap) {
    cudaFree(f->d_outs);
    f->d_outs = nullptr;
    f->outs_cap = 0;
    if (cudaMalloc(&f->d_outs, (total_out + total_out / 4) * sizeof(OutEntry)) != cudaSuccess)
      return api_fail(ESPB_ERR_NOMEM, "clock groups: schedule entries");
    f->outs_cap = total_out + total_out / 4;
  }
  memcpy(f->h_blob[hb], desc.data(), (size_t) G * sizeof(FsGroupDesc));
  if (!segs.empty())
    memcpy(f->h_blob[hb] + (size_t) G * sizeof(FsGroupDesc), segs.data(), segs.size() * sizeof(SchedSegment));
#define GR_TRY(expr, what)                                                          \
  do {                                                                              \
    cudaError_t e__ = (expr);                                                       \
    if (e__ != cudaSuccess)                                                         \
      return api_fail(ESPB_ERR_CUDA, "clock groups: " what, cudaGetErrorString(e__)); \
  } while (0)
  GR_TRY(cudaMemcpyAsync(f->d_blob, f->h_blob[hb], blob_bytes, cudaMemcpyHostToDevice, stream), "upload");
  GR_TRY(cudaEventRecord(f->h_done[hb], stream), "event");
  f->h_pending[hb] = true;
  const FsGroupDesc *d_desc = reinterpret_cast<const FsGroupDesc *>(f->d_blob);
  const SchedSegment *d_segs = reinterpret_cast<const SchedSegment *>(f->d_blob + (size_t) G * sizeof(FsGroupDesc));
  float *x_new = f->buf[1 - f->cur];
  // carried frames + new input of every group -> the other staging buffer
  GR_TRY(launch_fsg_stage(d_desc, G, f->buf[f->cur], x_new, f->pitch, T, in, in_ss, f->channels, f->n_series, max_rows,
                          stream),
         "staging kernel");
  if (total_out > 0) {
    GR_TRY(launch_expand_schedule_groups(d_desc, G, d_segs, f->d_outs, max_out, f->geo.filters,
                                         (f->geo.flags & kFlagLowpass) != 0, (f->geo.flags & kFlagInterpolate) != 0,
                                         stream),
           "schedule kernel");
    FsParams fp{};
    fp.x = x_new;
    fp.x_fs = f->pitch;
    fp.x_row0 = T;
    fp.out = out;
    fp.out_ss = out_ss;
    fp.out_cs = 1;
    fp.out_fs = f->channels;
    fp.out_tm = nullptr;
    fp.bank_tr = f->bank_tr;
    fp.outs = f->d_outs;
    fp.n_series = f->n_series;
    fp.channels = f->channels;
    fp.n_out = max_out;
    fp.taps = T;
    fp.kt = f->kt;
    fp.slice_floats = (int) f->slice_floats;
    fp.groups = d_desc;
    GR_TRY(launch_resample_fs(fp, f->fg, x_rows, context_mode(g->ctx[0]) == ESPB_MODE_EXACT, stream, G),
           "few-series resample kernel");
  }
#undef GR_TRY
  // ---- the call is enqueued: commit the per-group state (art_resampler.cpp keeps it in the context)
  f->cur = 1 - f->cur;
  for (int k = 0; k < G; ++k) {
    f->carry_row[k] = (int) results[k].input_used;  // frames [used - taps, used) are rows [used, used + taps)
    set_context_state(g->ctx[k], end_state[k]);
  }
  api_ok();
  return ESPB_OK;
}

}  // namespace

extern "C" {

void espb_resampleGroupsFree(EspbResampleGroups *g) {
  if (!g)
    return;
  for (EspbResampleBatch *c : g->ctx)
    espb_resampleFree(c);
  for (cudaStream_t s : g->streams)
    cudaStreamDestroy(s);
  for (cudaEvent_t e : g->joined)
    cudaEventDestroy(e);
  if (g->fork)
    cudaEventDestroy(g->fork);
  fused_free(g->fused);
  delete g;
}

EspbResampleGroups *espb_resampleGroupsInit(int num_groups, const int *streams_per_group, int numChannels, int numTaps,
                                            int numFilters, float lowpassRatio, int flags) {
  if (num_groups <= 0 || !streams_per_group) {
    fprintf(stderr, "resampleGroupsInit: needs at least one group\n");
    return nullptr;
  }
  EspbResampleGroups *g = new (std::nothrow) EspbResampleGroups();
  if (!g)
    return nullptr;
  g->channels = numChannels;
  cudaGetDevice(&g->device);
  // many small equal groups: the fused form (ESPB_GROUPS_FUSED=0 keeps one context per group)
  bool uniform = num_groups >= 2 && numChannels > 0 && streams_per_group[0] > 0 &&
                 (long long) streams_per_group[0] * numChannels <= kFsMaxSeries;
  for (int k = 1; k < num_groups && uniform; ++k)
    uniform = streams_per_group[k] == streams_per_group[0];
  {
    const char *v = getenv("ESPB_GROUPS_FUSED");
    if (v && *v == '0')
      uniform = false;
  }
  if (uniform) {
    float lp = lowpassRatio;
    int fl = flags;
    if (!normalise_init(numTaps, numFilters, &lp, &fl) || espb_device_count() <= 0) {
      api_fail(ESPB_ERR_ARG, "resampleGroupsInit: invalid taps/filters, or no CUDA device");
      delete g;
      return nullptr;
    }
    const ArtGeometry geo{numTaps, numFilters, fl};
    std::vector<float> bank;
    build_filter_bank(geo, lp, bank);
    g->fused = fused_create(num_groups, streams_per_group[0], numChannels, geo, bank);
    if (!g->fused) {
      api_fail(ESPB_ERR_CUDA, "resampleGroupsInit: device allocation");
      delete g;
      return nullptr;
    }
    int first = 0;
    for (int k = 0; k < num_groups; ++k) {
      g->ctx.push_back(new_state_only_context(streams_per_group[k], numChannels, geo, lp));
      g->first_stream.push_back(first);
      g->n_streams.push_back(streams_per_group[k]);
      first += streams_per_group[k];
    }
    return g;
  }
  int first = 0;
  for (int k = 0; k < num_groups; ++k) {
    EspbResampleBatch *c = espb_resampleInit(streams_per_group[k], numChannels, numTaps, numFilters, lowpassRatio, flags);
    cudaStream_t s = nullptr;
    cudaEvent_t e = nullptr;
    if (!c || cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
      if (c)
        espb_resampleFree(c);
      if (s)
        cudaStreamDestroy(s);
      espb_resampleGroupsFree(g);
      return nullptr;
    }
    g->ctx.push_back(c);
    g->streams.push_back(s);
    g->joined.push_back(e);
    g->first_stream.push_back(first);
    g->n_streams.push_back(streams_per_group[k]);
    first += streams_per_group[k];
  }
  if (cudaEventCreateWithFlags(&g->fork, cudaEventDisableTiming) != cudaSuccess) {
    espb_resampleGroupsFree(g);
    return nullptr;
  }
  return g;
}

int espb_resampleGroupsCount(const EspbResampleGroups *g) { return g ? (int) g->ctx.size() : 0; }
int espb_resampleGroupsIsFused(const EspbResampleGroups *g) { return (g && g->fused) ? 1 : 0; }

EspbResampleBatch *espb_resampleGroupsContext(EspbResampleGroups *g, int group) {
  return (g && group >= 0 && group < (int) g->ctx.size()) ? g->ctx[group] : nullptr;
}

int espb_resampleGroupsFirstStream(const EspbResampleGroups *g, int group) {
  return (g && group >= 0 && group < (int) g->ctx.size()) ? g->first_stream[group] : -1;
}

int espb_resampleGroupsSetMode(EspbResampleGroups *g, int mode) {
  if (!g)
    return ESPB_ERR_ARG;
  for (EspbResampleBatch *c : g->ctx) {
    if (g->fused) {
      if (mode != ESPB_MODE_FAST && mode != ESPB_MODE_EXACT)
        return api_fail(ESPB_ERR_ARG, "resampleGroupsSetMode: bad mode");
      set_context_mode(c, mode);
      continue;
    }
    const int rc = espb_resampleSetMode(c, mode);
    if (rc != ESPB_OK)
      return rc;
  }
  return ESPB_OK;
}

// resampleReset (art_resampler.cpp:144-152) for one group: silent history, initial position.
int espb_resampleGroupsReset(EspbResampleGroups *g, int group, void *stream) {
  if (!g || group < 0 || group >= (int) g->ctx.size())
    return api_fail(ESPB_ERR_ARG, "resampleGroupsReset: bad group");
  if (!g->fused)
    return espb_resampleReset(g->ctx[group], stream);
  FusedSet *f = g->fused;
  cudaError_t e = cudaMemsetAsync(f->buf[f->cur] + ((size_t) group * f->rows_cap + f->carry_row[group]) * f->pitch, 0,
                                  (size_t) f->geo.taps * f->pitch * sizeof(float),
                                  reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess)
    return api_fail(ESPB_ERR_CUDA, "resampleGroupsReset", cudaGetErrorString(e));
  set_context_state(g->ctx[group], initial_state(f->geo.taps));
  return ESPB_OK;
}

int espb_resampleGroupsProcessInterleaved(EspbResampleGroups *g, const float *in, int64_t in_stream_stride,
                                          const int *numInputFrames, float *out, int64_t out_stream_stride,
                                          const int *numOutputFrames, const float *ratios, EspbResampleResult *results,
                                          void *stream) {
  if (!g || !numInputFrames || !numOutputFrames || !ratios || !results)
    return ESPB_ERR_ARG;
  cudaStream_t caller = reinterpret_cast<cudaStream_t>(stream);
  if (g->fused)
    return fused_process(g, in, in_stream_stride, numInputFrames, out, out_stream_stride, numOutputFrames, ratios,
                         results, caller);
  if (cudaEventRecord(g->fork, caller) != cudaSuccess)
    return ESPB_ERR_CUDA;
  int rc = ESPB_OK;
  for (size_t k = 0; k < g->ctx.size(); ++k) {
    cudaStream_t s = g->streams[k];
    if (cudaStreamWaitEvent(s, g->fork, 0) != cudaSuccess)
      return ESPB_ERR_CUDA;
    const int64_t first = g->first_stream[k];
    results[k] = espb_resampleProcessInterleaved(g->ctx[k], in + first * in_stream_stride, in_stream_stride,
                                                 numInputFrames[k], out + first * out_stream_stride, out_stream_stride,
                                                 numOutputFrames[k], ratios[k], s);
    if (espb_last_status() != ESPB_OK)
      rc = espb_last_status();
    if (cudaEventRecord(g->joined[k], s) != cudaSuccess || cudaStreamWaitEvent(caller, g->joined[k], 0) != cudaSuccess)
      return ESPB_ERR_CUDA;
  }
  return rc;
}

}  // extern "C"
