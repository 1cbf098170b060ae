// C-ABI layer of the B200 ART resampler path (include/esp_audio_b200.h).
//
// Host logic only: parameter validation with the reference's conventions (NULL / false
// on failure, the same stderr lines), planning (plan.cpp), device-buffer management and
// kernel launches.  No CPU compute path exists: without a usable CUDA device every
// computing entry point fails with ESPB_ERR_CUDA.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/esp_audio_b200.h"
#include "internal.hpp"
#include "kernels.hpp"
#include "plan.hpp"

using namespace espb;

// ------------------------------------------------------------------------------------
// errors, counters
// ------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static thread_local int g_last_status = 0;  // ESPB_OK or the code of the calling thread's last failed call
static std::atomic<uint64_t> g_launches{0};

namespace espb {
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int grid_y_max() {
  static const int v = [] {
    const char *s = getenv("ESPB_GRID_Y_MAX");
    const long n = s ? atol(s) : kMaxGridY;
    return (int) (n < 1 ? 1 : (n > kMaxGridY ? kMaxGridY : n));
  }();
  return v;
}
}  // namespace espb

static int fail(int code, const char *what, const char *detail = nullptr) {
  g_last_status = code;
  g_last_error = what;
  if (detail) {
    g_last_error += ": ";
    g_last_error += detail;
  }
  return code;
}
static int cuda_fail(cudaError_t e, const char *what) { return fail(ESPB_ERR_CUDA, what, cudaGetErrorString(e)); }

#define CU_TRY(expr, what)        \
  do {                            \
    cudaError_t e__ = (expr);     \
    if (e__ != cudaSuccess)       \
      return cuda_fail(e__, what); \
  } while (0)

static inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

static long env_long(const char *name, long dflt) {
  const char *v = getenv(name);
  return (v && *v) ? strtol(v, nullptr, 10) : dflt;
}

extern "C" {

const char *espb_last_error(void) { return g_last_error.c_str(); }
int espb_last_status(void) { return g_last_status; }
int espb_abi_version(void) { return ESPB_ABI_VERSION; }
uint64_t espb_launch_count(void) { return g_launches.load(); }

// ------------------------------------------------------------------------------------
// device + buffers
// ------------------------------------------------------------------------------------
int espb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}
int espb_set_device(int device) {
  CU_TRY(cudaSetDevice(device), "cudaSetDevice");
  return ESPB_OK;
}
int espb_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem, char *name, int name_len) {
  int dev = 0;
  CU_TRY(cudaGetDevice(&dev), "cudaGetDevice");
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, dev), "cudaGetDeviceProperties");
  if (sm_count)
    *sm_count = prop.multiProcessorCount;
  if (cc_major)
    *cc_major = prop.major;
  if (cc_minor)
    *cc_minor = prop.minor;
  if (total_mem)
    *total_mem = prop.totalGlobalMem;
  if (name && name_len > 0) {
    strncpy(name, prop.name, name_len - 1);
    name[name_len - 1] = 0;
  }
  return ESPB_OK;
}
void *espb_malloc(size_t bytes) {
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    cuda_fail(e, "cudaMalloc");
    return nullptr;
  }
  return p;
}
void espb_free(void *dptr) {
  if (dptr)
    cudaFree(dptr);
}
void *espb_malloc_host(size_t bytes) {
  void *p = nullptr;
  cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
  if (e != cudaSuccess) {
    cuda_fail(e, "cudaMallocHost");
    return nullptr;
  }
  return p;
}
void espb_free_host(void *hptr) {
  if (hptr)
    cudaFreeHost(hptr);
}
int espb_memcpy_h2d(void *dst, const void *src, size_t bytes, void *stream) {
  CU_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, as_stream(stream)), "cudaMemcpyAsync h2d");
  return ESPB_OK;
}
int espb_memcpy_d2h(void *dst, const void *src, size_t bytes, void *stream) {
  CU_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, as_stream(stream)), "cudaMemcpyAsync d2h");
  return ESPB_OK;
}
int espb_memset(void *dst, int value, size_t bytes, void *stream) {
  CU_TRY(cudaMemsetAsync(dst, value, bytes, as_stream(stream)), "cudaMemsetAsync");
  return ESPB_OK;
}
void *espb_stream_create(void) {
  cudaStream_t s = nullptr;
  cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    cuda_fail(e, "cudaStreamCreate");
    return nullptr;
  }
  return s;
}
void espb_stream_destroy(void *stream) {
  if (stream)
    cudaStreamDestroy(as_stream(stream));
}
int espb_stream_sync(void *stream) {
  CU_TRY(cudaStreamSynchronize(as_stream(stream)), "cudaStreamSynchronize");
  return ESPB_OK;
}
int espb_device_sync(void) {
  CU_TRY(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
  return ESPB_OK;
}
void *espb_event_create(void) {
  cudaEvent_t ev = nullptr;
  cudaError_t e = cudaEventCreate(&ev);
  if (e != cudaSuccess) {
    cuda_fail(e, "cudaEventCreate");
    return nullptr;
  }
  return ev;
}
void espb_event_destroy(void *ev) {
  if (ev)
    cudaEventDestroy(reinterpret_cast<cudaEvent_t>(ev));
}
int espb_event_record(void *ev, void *stream) {
  CU_TRY(cudaEventRecord(reinterpret_cast<cudaEvent_t>(ev), as_stream(stream)), "cudaEventRecord");
  return ESPB_OK;
}
int espb_event_elapsed_ms(void *start, void *stop, float *ms) {
  CU_TRY(cudaEventSynchronize(reinterpret_cast<cudaEvent_t>(stop)), "cudaEventSynchronize");
  CU_TRY(cudaEventElapsedTime(ms, reinterpret_cast<cudaEvent_t>(start), reinterpret_cast<cudaEvent_t>(stop)),
         "cudaEventElapsedTime");
  return ESPB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// small RAII-free device buffer helper
// ------------------------------------------------------------------------------------
namespace {

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  // Grows with head-room: in a stream of calls the sizes wander by a few entries (frame counts alternate between n
  // and n + 1), and every re-allocation is a cudaFree — a device-wide synchronisation in the middle of the stream.
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap)
      return cudaSuccess;
    if (p)
      cudaFree(p);
    p = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 16 + 4096;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {  // no room for the slack: the exact size
      cudaGetLastError();
      e = cudaMalloc(&p, bytes);
      if (e == cudaSuccess)
        cap = bytes;
      return e;
    }
    cap = want;
    return e;
  }
  void release() {
    if (p)
      cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T *as() const {
    return static_cast<T *>(p);
  }
};

// Row-wise async copy; one flat copy when the rows are contiguous on both sides.
inline cudaError_t copy_rows_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width,
                                   size_t height, cudaMemcpyKind kind, cudaStream_t stream) {
  if (width == 0 || height == 0)
    return cudaSuccess;
  if (dpitch == width && spitch == width)
    return cudaMemcpyAsync(dst, src, width * height, kind, stream);
  return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, kind, stream);
}

struct ScheduleKey {
  uint32_t offset_bits = 0, ratio_bits = 0;
  int index = -1, n_in = -1, n_out = -1, split = 0;
  bool operator==(const ScheduleKey &o) const {
    return offset_bits == o.offset_bits && ratio_bits == o.ratio_bits && index == o.index && n_in == o.n_in &&
           n_out == o.n_out && split == o.split;
  }
};

inline uint32_t f2u(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}

}  // namespace

// ------------------------------------------------------------------------------------
// host pipelining helper shared by the ART batch and the wrapper
// ------------------------------------------------------------------------------------
namespace {

struct HostPipe {
  static const int kStreams = 3;
  // error exit of a host-buffer call: copies into the caller's buffers may still be in flight on these streams
  void drain() {
    for (int i = 0; i < kStreams; ++i)
      if (s[i])
        cudaStreamSynchronize(s[i]);
  }
  cudaStream_t s[kStreams] = {nullptr, nullptr, nullptr};
  cudaEvent_t ready = nullptr;
  bool ok = false;
  cudaError_t init() {
    if (ok)
      return cudaSuccess;
    for (int i = 0; i < kStreams; ++i) {
      cudaError_t e = cudaStreamCreateWithFlags(&s[i], cudaStreamNonBlocking);
      if (e != cudaSuccess)
        return e;
    }
    cudaError_t e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming);
    if (e != cudaSuccess)
      return e;
    ok = true;
    return cudaSuccess;
  }
  void destroy() {
    for (int i = 0; i < kStreams; ++i)
      if (s[i])
        cudaStreamDestroy(s[i]);
    if (ready)
      cudaEventDestroy(ready);
    ok = false;
  }
};

// Streams per slab of the host pipeline: about 32 slabs, each starting on a 128-series group boundary.
int pick_slab_streams(int num_streams, int channels) {
  long forced = env_long("ESPB_HOST_SLABS", 0);
  long slabs = forced > 0 ? forced : 32;  // measured: 8 slabs 40.3 ms, 32 slabs 33.2 ms per C2 step (PCIe floor ~32)
  if (slabs > num_streams)
    slabs = num_streams;
  long per = (num_streams + slabs - 1) / slabs;
  int a = kSeriesPerRow, b = channels;
  while (b) {
    int t = a % b;
    a = b;
    b = t;
  }
  const long unit = kSeriesPerRow / a;  // smallest stream count whose series fill whole groups
  per = (per + unit - 1) / unit * unit;
  return (int) per;
}

}  // namespace

// ------------------------------------------------------------------------------------
// ART resampler batch
// ------------------------------------------------------------------------------------
struct EspbResampleBatch {
  bool state_only = false;  // position state and geometry only (internal.hpp): the fused clock groups own the data
  int device = -1;  // the CUDA device that was current at creation: all of the context's memory lives there
  int num_streams = 0, channels = 0;
  ArtGeometry geo{};
  float lowpass = 1.0f;
  ArtState state{};
  int mode = ESPB_MODE_FAST;
  int bpp = 8;  // output blocks (warps) per pass
  int chunk_rows = 32;  // input rows per pipeline stage (kernel variants: 32 default; 16, 24, 36 selectable)
  std::vector<float> bank_host;
  DevBuf bank;
  // time-major input staging xt[group][row][128]: rows [0, taps) = frames carried over from the
  // previous call, rows [taps, taps + n_in) = this call's input, then zero padding.  Two buffers
  // alternate; the carry of the next call is rows [carry_row, carry_row + taps) of xt[xt_cur].
  DevBuf xt[2];
  int xt_cur = 0;
  int64_t xt_rows = 0;  // rows per group in both buffers
  int carry_row = 0;
  DevBuf yt, yt2;  // time-major output scratch [group][yt_rows][128] when a library stage follows the resampler
  int64_t yt_rows = 0, yt2_rows = 0;
  int n_groups() const { return (n_series() + kSeriesPerRow - 1) / kSeriesPerRow; }
  // per-call plan, cached by (state, n_in, n_out, ratio)
  Schedule sched;
  PassPlan plan;
  ScheduleKey key;
  bool plan_on_device = false;  // tables uploaded
  int g_resident_first = -1, g_resident_end = -1;  // chunk range currently expanded in G
  DevBuf d_outs, d_chunks, d_pcb, d_G;
  size_t g_budget_bytes = (size_t) 1 << 30;
  // device staging + CUDA streams of the host-buffer entry point
  DevBuf stage_in, stage_out;
  HostPipe pipe;
  // direct input (interleaved stereo float, see espb_resample_kernel<..., DIRECT>): decided per call
  // without SUBSAMPLE_INTERPOLATE an output is one dot product: its own kernel and half-size G rows (default geometry)
  bool non_interp = false;
  int g_row_floats() const { return non_interp ? kGRowFloatsNI : kGRowFloats; }
  // output blocks per pass of the plan and of G (the non-interpolating kernel's 4 warps own two blocks each)
  int plan_bpp() const { return non_interp ? bpp * kNiBlocksPerWarp : bpp; }
  bool direct_ok = false;    // ESPB_DIRECT=1 switches it on
  // few-series form (resample_fs_kernel.cu): lanes own outputs; chosen per context when n_series <= kFsMaxSeries
  int fs_policy = -1;        // ESPB_FS: 0 never, 1 / unset whenever the geometry allows it
  DevBuf bank_tr;            // slice-major copy of the bank
  int fs_kt = 0;
  size_t fs_slice = 0;       // floats per slice
  bool fs_call = false;      // this call runs through the few-series kernel (no pass plan, no G)
  int fs_x_rows = 0;         // rows of the widest input tile of a CTA of this call
  bool direct_call = false;  // this call's plan is split at input frame 0 and its input is read through TMA
  // options
  bool plan_cache = true;   // reuse schedule / tables / G when a call repeats (state, n_in, n_out, ratio)
  bool kernel_timing = false;
  std::vector<cudaEvent_t> ev_pool;  // pairs: [2k] before, [2k+1] after each resample-kernel launch
  size_t ev_used = 0;
  // the last asynchronous state change (reset) — processing on any other stream waits for it
  cudaEvent_t state_event = nullptr;
  bool state_event_pending = false;
  // the page-locked host tables are read by asynchronous copies: they may be rebuilt only after the last upload
  cudaEvent_t tables_uploaded = nullptr;
  bool tables_upload_pending = false;
  // ... so two sets of table storage alternate: a rebuild waits for the upload of the call before the previous one,
  // which in a stream of calls has long finished (no host/device serialisation from call to call)
  PodBuffer<OutEntry> spare_outs;
  PodBuffer<SchedSegment> spare_segs;
  DevBuf d_ptrs;  // device copy of the plane-pointer tables of espb_resampleProcessPlanes: [2][n_series]
  DevBuf d_segs;
  // small calls: runs, chunks and pass prefix travel as ONE pageable blob (one upload instead of three); the pointers
  // below are where the kernels find the tables of the current plan, whichever way they arrived
  // coefficient expansion on a side stream, next to the (HBM-bound) input staging of the same call
  cudaStream_t aux = nullptr;
  cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
  bool aux_join_pending = false;
  DevBuf d_tables;
  std::vector<unsigned char> h_tables;
  const SchedSegment *p_segs = nullptr;
  const ChunkEntry *p_chunks = nullptr;
  const int32_t *p_pcb = nullptr;
  bool sched_segments = true;  // closed-form schedule expanded on the device (ESPB_SCHED=seq: per-output host schedule)
  PodBuffer<ChunkEntry> spare_chunks;
  PodBuffer<int32_t> spare_pcb;
  cudaEvent_t spare_uploaded = nullptr;
  bool spare_upload_pending = false;
  // staging overlap (DESIGN.md §4.5): the resampler starts while the transposing kernel is still running and waits
  // per CTA on per-row-tile counters; device-buffer calls of the standard kernel only.  ESPB_OVERLAP=0 switches it off
  int overlap_staging = 1;
  int stage_ctas_per_sm = 2;  // (negative: that many CTAs in all)
  DevBuf d_ready;  // [row tiles] counters of the current call
  int n_series() const { return num_streams * channels; }
};

namespace {

int ensure_xt(EspbResampleBatch *c, int64_t rows);

// PodBuffer hooks: best effort (a table that cannot be page-locked is simply uploaded through a staging copy)
// Not the small ones: for the few KB of a real-time chunk a pageable source is faster — the driver embeds it in the
// command stream (measured 136 against 157 us per 10 ms call of 4096 stereo streams).  Beyond that a pageable source
// makes cudaMemcpyAsync stage the copy synchronously behind the stream's earlier work, which ties the host to the
// device call by call (C3: 0.77 MB of schedule per 1 s call), so everything from 64 KB on is page-locked.
constexpr size_t kPinTablesFrom = (size_t) 64 << 10;
void pin_host_range(void *p, size_t bytes) {
  if (bytes < kPinTablesFrom)  // (the same threshold decides in prepare_call whether an upload must be awaited)
    return;
  if (cudaHostRegister(p, bytes, cudaHostRegisterDefault) != cudaSuccess)
    cudaGetLastError();
}
void unpin_host_range(void *p) {
  if (cudaHostUnregister(p) != cudaSuccess)
    cudaGetLastError();
}

// Build (or reuse) the schedule + pass plan for this call and upload the tables.
int prepare_call(EspbResampleBatch *c, int n_in, int n_out, float ratio, cudaStream_t stream,
                 bool want_direct = false) {
  {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev != c->device)
      return fail(ESPB_ERR_STATE, "this context was created on another CUDA device (espb_set_device before the call)");
  }
  if (c->state_only)
    return fail(ESPB_ERR_STATE, "this context belongs to a fused clock-group set: process through espb_resampleGroups*");
  if (!(ratio > 0.0f) || !(ratio <= 3.0e38f))  // NaN, <= 0, Inf: the reference would loop for ever or index wildly
    return fail(ESPB_ERR_ARG, "resampleProcess: ratio must be a positive finite number");
  if (c->state_event_pending) {  // order this call after an asynchronous reset issued on another stream
    CU_TRY(cudaStreamWaitEvent(stream, c->state_event, 0), "cudaStreamWaitEvent");
    c->state_event_pending = false;
  }
  // direct input needs the default kernel geometry and a carry that lies inside this call's input
  want_direct = want_direct && c->direct_ok && !c->non_interp && c->bpp == 4 && c->chunk_rows == 32 &&
                n_in >= c->geo.taps;
  ScheduleKey k;
  k.offset_bits = f2u(c->state.offset);
  k.ratio_bits = f2u(ratio);
  k.index = c->state.index;
  k.n_in = n_in;
  k.n_out = n_out;
  k.split = want_direct ? 1 : 0;
  if (c->plan_cache && c->plan_on_device && k == c->key && c->direct_call == want_direct) {
    int rc = ensure_xt(c, (int64_t) c->geo.taps + (c->direct_call ? 0 : n_in) + kChunkRows);
    return rc;
  }
  c->plan_on_device = false;
  c->g_resident_first = c->g_resident_end = -1;
  {  // rebuild into the storage of the call before the previous one
    c->sched.outs.swap_storage(c->spare_outs);
    c->sched.segs.swap_storage(c->spare_segs);
    c->plan.chunks.swap_storage(c->spare_chunks);
    c->plan.pass_chunk_begin.swap_storage(c->spare_pcb);
    cudaEvent_t ev = c->tables_uploaded;
    c->tables_uploaded = c->spare_uploaded;
    c->spare_uploaded = ev;
    const bool pend = c->tables_upload_pending;
    c->tables_upload_pending = c->spare_upload_pending;
    c->spare_upload_pending = pend;
  }
  if (c->tables_upload_pending) {
    CU_TRY(cudaEventSynchronize(c->tables_uploaded), "cudaEventSynchronize");
    c->tables_upload_pending = false;
  }
  if (c->sched_segments) {  // a few runs per ring cycle; the per-output entries are expanded on the device
    build_schedule_segments(c->geo, c->state, n_in, n_out, ratio, c->sched);
  } else {
    c->sched.segmented = false;
    c->sched.segs.clear();
    build_schedule(c->geo, c->state, n_in, n_out, ratio, c->sched, /*finalize=*/false);  // pass 2 runs on the device
  }
  c->fs_call = false;
  if (c->bank_tr.p && c->fs_policy != 0 && c->sched.generated > 0) {
    // few-series form: the widest input tile (rows first window .. last window + taps of one CTA's outputs) must fit
    const FsGeometry fg = fs_geometry(c->n_series());
    const int n = (int) c->sched.generated, m = fg.outputs_per_cta;
    int span = 0, cursor = 0;
    for (int first = 0; first < n; first += m) {
      const int last = (first + m < n ? first + m : n) - 1;
      const int ws_first = schedule_ws(c->sched, first, &cursor);
      const int d = schedule_ws(c->sched, last, &cursor) - ws_first;
      span = d > span ? d : span;
    }
    c->fs_x_rows = span + c->geo.taps;
    c->fs_call = fs_smem_bytes(fg, c->fs_slice, c->fs_x_rows) <= (size_t) 200 * 1024;
  }
  if (c->fs_call)
    want_direct = false;
  c->direct_call = want_direct && (int) c->sched.used >= c->geo.taps;
  k.split = c->direct_call ? 1 : 0;
  {
    int rc = ensure_xt(c, (int64_t) c->geo.taps + (c->direct_call ? 0 : n_in) + kChunkRows);
    if (rc != ESPB_OK)
      return rc;
  }
  if (c->fs_call) {  // no passes, no chunks, no expanded coefficients
    c->plan.chunks.clear();
    c->plan.pass_chunk_begin.clear();
    c->plan.pass_chunk_begin.push_back(0);
  } else {
    build_pass_plan(c->sched, c->geo.taps, c->plan_bpp(), c->chunk_rows, c->plan, c->direct_call);
    // the kernel keeps the chunk table of its passes in shared memory: one pass must fit it.  (32 outputs at a
    // ratio below ~0.004 span more than 320 chunks of input — far outside audio use; refused, not truncated.)
    const int limit = max_chunks_per_cta(c->bpp, c->chunk_rows);
    for (int ps = 0; ps < c->plan.n_passes(); ++ps)
      if (c->plan.pass_chunk_begin[ps + 1] - c->plan.pass_chunk_begin[ps] > limit) {
        c->key = ScheduleKey{};
        return fail(ESPB_ERR_ARG, "resampleProcess: ratio too small for the kernel's per-pass chunk table");
      }
  }
  c->key = k;
  if (c->sched.generated == 0) {
    c->plan_on_device = true;
    return ESPB_OK;
  }
  CU_TRY(c->d_outs.reserve((size_t) c->sched.generated * sizeof(OutEntry)), "cudaMalloc schedule");
  const size_t seg_bytes = c->sched.segmented ? c->sched.segs.size() * sizeof(SchedSegment) : 0;
  const size_t chunk_bytes = c->fs_call ? 0 : c->plan.chunks.size() * sizeof(ChunkEntry);
  const size_t pcb_bytes = c->fs_call ? 0 : c->plan.pass_chunk_begin.size() * sizeof(int32_t);
  auto up16 = [](size_t v) { return (v + 15) & ~(size_t) 15; };
  const size_t blob_bytes = up16(seg_bytes) + up16(chunk_bytes) + up16(pcb_bytes);
  if (c->sched.segmented && blob_bytes <= ((size_t) 48 << 10)) {
    // one upload: the driver copies a pageable source of this size out before cudaMemcpyAsync returns
    CU_TRY(c->d_tables.reserve(blob_bytes + sizeof(ChunkEntry)), "cudaMalloc tables");
    c->h_tables.resize(blob_bytes);
    unsigned char *h = c->h_tables.data(), *d = c->d_tables.as<unsigned char>();
    memcpy(h, c->sched.segs.data(), seg_bytes);
    if (chunk_bytes)
      memcpy(h + up16(seg_bytes), c->plan.chunks.data(), chunk_bytes);
    if (pcb_bytes)
      memcpy(h + up16(seg_bytes) + up16(chunk_bytes), c->plan.pass_chunk_begin.data(), pcb_bytes);
    CU_TRY(cudaMemcpyAsync(d, h, blob_bytes, cudaMemcpyHostToDevice, stream), "upload tables");
    c->p_segs = reinterpret_cast<const SchedSegment *>(d);
    c->p_chunks = reinterpret_cast<const ChunkEntry *>(d + up16(seg_bytes));
    c->p_pcb = reinterpret_cast<const int32_t *>(d + up16(seg_bytes) + up16(chunk_bytes));
  } else {
    CU_TRY(c->d_chunks.reserve((c->plan.chunks.size() + 1) * sizeof(ChunkEntry)), "cudaMalloc chunks");
    CU_TRY(c->d_pcb.reserve(c->plan.pass_chunk_begin.size() * sizeof(int32_t)), "cudaMalloc passes");
    if (c->sched.segmented) {
      CU_TRY(c->d_segs.reserve(seg_bytes), "cudaMalloc schedule");
      CU_TRY(cudaMemcpyAsync(c->d_segs.p, c->sched.segs.data(), seg_bytes, cudaMemcpyHostToDevice, stream),
             "upload schedule");
    }
    if (!c->fs_call) {
      CU_TRY(cudaMemcpyAsync(c->d_chunks.p, c->plan.chunks.data(), chunk_bytes, cudaMemcpyHostToDevice, stream),
             "upload chunks");
      CU_TRY(cudaMemcpyAsync(c->d_pcb.p, c->plan.pass_chunk_begin.data(), pcb_bytes, cudaMemcpyHostToDevice, stream),
             "upload passes");
    }
    c->p_segs = c->d_segs.as<SchedSegment>();
    c->p_chunks = c->d_chunks.as<ChunkEntry>();
    c->p_pcb = c->d_pcb.as<int32_t>();
  }
  if (c->sched.segmented) {
    CU_TRY(launch_expand_schedule(c->p_segs, (int) c->sched.segs.size(), c->d_outs.as<OutEntry>(),
                                  (int) c->sched.generated, c->geo.filters, (c->geo.flags & kFlagLowpass) != 0,
                                  (c->geo.flags & kFlagInterpolate) != 0, stream),
           "schedule kernel");
  } else {
    CU_TRY(cudaMemcpyAsync(c->d_outs.p, c->sched.outs.data(), c->sched.outs.size() * sizeof(OutEntry),
                           cudaMemcpyHostToDevice, stream),
           "upload schedule");
    CU_TRY(launch_finalize(c->d_outs.as<OutEntry>(), (int) c->sched.outs.size(), c->geo.filters,
                           (c->geo.flags & kFlagLowpass) != 0, (c->geo.flags & kFlagInterpolate) != 0, stream),
           "finalize kernel");
  }
  if (!c->tables_uploaded)
    CU_TRY(cudaEventCreateWithFlags(&c->tables_uploaded, cudaEventDisableTiming), "cudaEventCreate");
  // (pageable tables were copied to a staging area before cudaMemcpyAsync returned: nothing to wait for)
  const size_t pin_from = kPinTablesFrom;
  if (c->sched.outs.cap * sizeof(OutEntry) >= pin_from || c->sched.segs.cap * sizeof(SchedSegment) >= pin_from ||
      c->plan.chunks.cap * sizeof(ChunkEntry) >= pin_from ||
      c->plan.pass_chunk_begin.cap * sizeof(int32_t) >= pin_from) {
    CU_TRY(cudaEventRecord(c->tables_uploaded, stream), "cudaEventRecord");
    c->tables_upload_pending = true;
  }
  c->plan_on_device = true;
  return ESPB_OK;
}

// Number of passes per time slab so that the expanded coefficients fit the G budget.
int passes_per_slab(const EspbResampleBatch *c) {
  const int n_passes = c->plan.n_passes();
  const size_t chunk_bytes = g_chunk_floats(c->plan_bpp(), c->chunk_rows, c->g_row_floats()) * sizeof(float);
  const size_t total = c->plan.chunks.size() * chunk_bytes;
  if (total <= c->g_budget_bytes || n_passes <= 1)
    return n_passes;
  const double avg = (double) total / n_passes;
  int pps = (int) ((double) c->g_budget_bytes / avg);
  return pps < 1 ? 1 : pps;
}

// Make chunks [first, end) resident in G.
int ensure_g(EspbResampleBatch *c, int chunk_first, int chunk_end, cudaStream_t stream) {
  if (c->g_resident_first == chunk_first && c->g_resident_end == chunk_end)
    return ESPB_OK;
  const size_t chunk_floats = g_chunk_floats(c->plan_bpp(), c->chunk_rows, c->g_row_floats());
  CU_TRY(c->d_G.reserve((size_t) (chunk_end - chunk_first) * chunk_floats * sizeof(float)), "cudaMalloc G");
  CU_TRY(launch_expand(c->bank.as<float>(), c->d_outs.as<OutEntry>(), c->p_chunks,
                       c->d_G.as<float>(), chunk_first, chunk_end - chunk_first, (int) c->sched.generated,
                       c->geo.taps, c->plan_bpp(), c->chunk_rows, c->direct_call, stream, c->g_row_floats()),
         "expand kernel");
  c->g_resident_first = chunk_first;
  c->g_resident_end = chunk_end;
  return ESPB_OK;
}

int pick_passes_per_cta(const EspbResampleBatch *c, int n_series, int pass_first, int pass_end) {
  const int n_passes = pass_end - pass_first;
  int sms = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess)
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const long groups = (n_series + kSeriesPerRow - 1) / kSeriesPerRow;
  const long slots = (long) sms * (16 / c->bpp);  // resident CTAs
  // aim for >= 32 waves of CTAs so the tail stays small (measured: 8 waves cost 2.5 %), >= 1 pass per CTA
  long ppc = env_long("ESPB_PPC", 0);
  if (ppc <= 0)
    ppc = (groups * n_passes) / (slots * 32);
  if (ppc < 1)
    ppc = 1;
  if (ppc > kMaxPassesPerCta)
    ppc = kMaxPassesPerCta;
  // the CTA caches its chunk table in shared memory: keep the longest run of ppc passes within it
  int max_chunks = 1;
  for (int ps = pass_first; ps < pass_end; ++ps) {
    const int n = c->plan.pass_chunk_begin[ps + 1] - c->plan.pass_chunk_begin[ps];
    if (n > max_chunks)
      max_chunks = n;
  }
  if (ppc * max_chunks > max_chunks_per_cta(c->bpp, c->chunk_rows))
    ppc = max_chunks_per_cta(c->bpp, c->chunk_rows) / max_chunks;
  if (ppc < 1)
    ppc = 1;  // (prepare_call has refused calls in which a single pass is longer than the table)
  return (int) ppc;
}

// Make both staging buffers hold at least `rows` rows per group, keeping the carried frames.
int ensure_xt(EspbResampleBatch *c, int64_t rows) {
  if (rows <= c->xt_rows)
    return ESPB_OK;
  if (c->xt_rows > 0)
    rows += rows / 64 + 64;  // (head-room: see DevBuf::reserve)
  const int taps = c->geo.taps;
  const size_t row_bytes = kSeriesPerRow * sizeof(float);
  const size_t bytes = (size_t) c->n_groups() * rows * row_bytes;
  DevBuf nb[2];
  // Growth is rare and synchronous (legacy-stream memset / copy below): wait for whatever earlier calls enqueued on
  // non-blocking streams, which may still be writing the rows that are about to be carried over.
  cudaError_t e = c->xt_rows > 0 ? cudaDeviceSynchronize() : cudaSuccess;
  if (e == cudaSuccess)
    e = nb[0].reserve(bytes);
  if (e == cudaSuccess)
    e = nb[1].reserve(bytes);
  if (e == cudaSuccess)  // rows nobody has written yet must still be finite (they meet zero coefficients)
    e = cudaMemset(nb[0].p, 0, bytes);
  if (e == cudaSuccess)
    e = cudaMemset(nb[1].p, 0, bytes);
  if (e == cudaSuccess && c->xt_rows > 0)  // carry rows -> rows [0, taps) of the new current buffer
    e = cudaMemcpy2D(nb[0].p, rows * row_bytes, c->xt[c->xt_cur].as<float>() + (size_t) c->carry_row * kSeriesPerRow,
                     c->xt_rows * row_bytes, taps * row_bytes, c->n_groups(), cudaMemcpyDeviceToDevice);
  else if (e == cudaSuccess)
    e = cudaMemset2D(nb[0].p, rows * row_bytes, 0, taps * row_bytes, c->n_groups());
  if (e != cudaSuccess) {
    nb[0].release();
    nb[1].release();
    return cuda_fail(e, "staging buffers");
  }
  c->xt[0].release();  // cudaFree waits for work that may still read the old buffers
  c->xt[1].release();
  c->xt[0] = nb[0];
  c->xt[1] = nb[1];
  c->xt_cur = 0;
  c->carry_row = 0;
  c->xt_rows = rows;
  return ESPB_OK;
}

// Packed-PCM endpoints of a wrapper call (Resampler::resample converts with quantization_utils on both
// sides): when given, the conversion is fused into the layout stages instead of running as separate passes.
struct PcmIn {
  const uint8_t *data = nullptr;  // row of the first stream of the range
  int64_t row_bytes = 0;
  int bits = 0;
  float gain_factor = 1.0f;
  float *scratch = nullptr;  // stream-major float rows for what the fused kernel does not cover
  int64_t scratch_row = 0;
};
struct PcmOut {
  uint8_t *data = nullptr;
  int64_t row_bytes = 0;
  int bits = 0;
  uint32_t *clipped = nullptr;  // per stream
  float *scratch = nullptr;
  int64_t scratch_row = 0;
};

// Planar buffers as pointer tables (resampleProcess, include/art_resampler.h:36-37): device copies of the tables.
struct PtrIO {
  const float *const *in = nullptr;  // [n_series] device pointers, plane q = stream q / channels, channel q % channels
  float *const *out = nullptr;
};

// Optional in-library neighbours of the resampler (Resampler::resample's pre / post low-pass).
struct StageFilter {
  const BiquadParams *params = nullptr;  // NULL: no filter
  float *state = nullptr;                // [series][sections][4] of the first series of the range
  int sections = 0;
  int block_rows = 0, warm_rows = 0;     // time-block mode of the biquad kernel (0 = sequential)
  float *blk_state = nullptr;            // per-block state record of the first group of the range (time-block mode)
  unsigned int *mismatches = nullptr;    // counter of repaired blocks
  unsigned int *chain_broken = nullptr;  // one scratch word per group of the range (parallel hand-over check)
};

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda, so it still
// loads on a machine without a driver — where nothing can be computed anyway).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qr) == cudaSuccess &&
        qr == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// Can `in` (interleaved float) be read by the resampler kernel directly?  Stereo, 16-byte aligned rows.
bool direct_input_layout(const EspbResampleBatch *c, const float *in, const EspbLayout &il) {
  return c->channels == 2 && il.channel_stride == 1 && il.frame_stride == 2 && ((uintptr_t) in % 16) == 0 &&
         il.stream_stride % 4 == 0 && il.stream_stride > 0 && encode_tiled_fn() != nullptr;
}

// dim0 = frame x channel floats of a stream, dim1 = stream; box = 16 stereo frames (128 bytes) x 64 streams with the
// 128-byte swizzle; coordinates outside [0, 2 n_in) x [0, n_streams) read as zero.
int make_input_map(CUtensorMap *map, const float *in, int64_t stream_stride, int n_in, int n_streams) {
  const cuuint64_t dims[2] = {(cuuint64_t) n_in * 2, (cuuint64_t) n_streams};
  const cuuint64_t strides[1] = {(cuuint64_t) stream_stride * sizeof(float)};
  const cuuint32_t box[2] = {32, (cuuint32_t) (kSeriesPerRow / 2)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = encode_tiled_fn()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(in), dims, strides,
                                       box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(ESPB_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  return ESPB_OK;
}

constexpr int kSmallCallFrames = 4096;  // calls up to this many input frames are staged by one fused kernel

// Stage + resample series [series_first, series_first + n_series) of the batch (series_first is a
// multiple of 128).  The carried frames and the new input go to the spare staging buffer.  `pre`
// filters the staged input in place (time-major); with `post` the resampler writes time-major
// scratch, which is filtered and then laid out as the caller wants.
int run_series_range(EspbResampleBatch *c, int series_first, int n_series, const float *in, const EspbLayout &il,
                     float *out, const EspbLayout &ol, int n_in, cudaStream_t stream, bool g_preexpanded,
                     const StageFilter *pre = nullptr, const StageFilter *post = nullptr,
                     const PcmIn *pcm_in = nullptr, const PcmOut *pcm_out = nullptr, const PtrIO *ptrs = nullptr,
                     bool overlap_ok = false) {
  const int taps = c->geo.taps;
  const int g0 = series_first / kSeriesPerRow, ng = (n_series + kSeriesPerRow - 1) / kSeriesPerRow;
  const int64_t rows = c->xt_rows;
  const size_t row_bytes = kSeriesPerRow * sizeof(float);
  const float *x_old = c->xt[c->xt_cur].as<float>() + (size_t) g0 * rows * kSeriesPerRow;
  float *x_new = c->xt[1 - c->xt_cur].as<float>() + (size_t) g0 * rows * kSeriesPerRow;
  // direct input: nothing is staged — the kernel reads the carried frames where they lie and the new frames from
  // the caller's buffer; afterwards the frames [used - taps, used) become rows [0, taps) of the other buffer
  const bool direct = c->direct_call && !pre && !post && !pcm_in && !pcm_out && !ptrs;
  if (c->direct_call && !direct)
    return fail(ESPB_ERR_STATE, "direct-input plan with library stages around the resampler");
  // real-time chunks of float input: carried frames, transposition and padding in one launch (the three separate
  // operations cost more in launch gaps than in work)
  const bool pre_on_ = pre && pre->params && n_in > 0;
  const bool small_stage = !direct && !pcm_in && !ptrs && n_in <= kSmallCallFrames &&
                           !(pre_on_ && pre->block_rows > 0 && n_in > pre->block_rows);
  if (small_stage)
    CU_TRY(launch_stage_small(x_old, c->carry_row, taps, in, il.stream_stride, il.channel_stride, il.frame_stride,
                              c->channels, n_series, n_in, x_new, rows, kChunkRows, stream),
           "staging kernel");
  else if (!direct)
    CU_TRY(cudaMemcpy2DAsync(x_new, rows * row_bytes, x_old + (size_t) c->carry_row * kSeriesPerRow, rows * row_bytes,
                             taps * row_bytes, ng, cudaMemcpyDeviceToDevice, stream),
           "carry copy");
  // caller's frames -> rows [taps, taps + n_in) of `dst` (+ `pad` zero rows): float layouts through the
  // transposing stage; packed PCM through the fused conversion, with the stage-by-stage path for the tail
  auto stage_input = [&](float *dst, int pad) -> int {
    if (ptrs) {
      CU_TRY(launch_transpose_ptrs(ptrs->in + series_first, n_series, n_in, dst, rows, taps, pad, stream),
             "transpose kernel");
      return ESPB_OK;
    }
    if (pcm_in) {
      cudaError_t e = cudaSuccess;
      const int n_streams = n_series / c->channels;
      const int fast = launch_pcm_to_tm(pcm_in->data, pcm_in->row_bytes, pcm_in->bits, pcm_in->gain_factor,
                                        c->channels, n_series, n_in, dst, rows, taps, stream, &e);
      CU_TRY(e, "pcm_to_tm kernel");
      if (fast < n_in) {
        const int nbytes = (pcm_in->bits + 7) / 8;
        CU_TRY(launch_q2f(pcm_in->data + (size_t) fast * c->channels * nbytes, pcm_in->row_bytes,
                          pcm_in->scratch + (size_t) fast * c->channels, pcm_in->scratch_row, n_streams,
                          (uint32_t) ((n_in - fast) * c->channels), pcm_in->bits, pcm_in->gain_factor, stream),
               "q2f kernel");
      }
      if (fast > 0)
        CU_TRY(launch_transpose_from(pcm_in->scratch, pcm_in->scratch_row, 1, c->channels, c->channels, n_series,
                                     n_in, dst, rows, taps, fast, pad, stream),
               "transpose kernel");
      else  // layout not covered by the fused kernel: the two separate stages
        CU_TRY(launch_transpose(pcm_in->scratch, pcm_in->scratch_row, 1, c->channels, c->channels, n_series, n_in,
                                dst, rows, taps, pad, stream),
               "transpose kernel");
      return ESPB_OK;
    }
    CU_TRY(launch_transpose(in, il.stream_stride, il.channel_stride, il.frame_stride, c->channels, n_series, n_in,
                            dst, rows, taps, pad, stream),
           "transpose kernel");
    return ESPB_OK;
  };
  const bool pre_on = pre && pre->params && n_in > 0;
  int ready_tiles = 0;  // > 0: the staging kernel just enqueued signals this many row tiles (overlap with the resampler)
  const bool pre_blocks = pre_on && pre->block_rows > 0 && n_in > pre->block_rows;
  if (direct) {
    // (no staging)
  } else if (pre_blocks) {
    // time-block pre-filter is out of place: the raw frames go to the other staging buffer (its carry rows
    // were copied above, the rest is free), the filter writes the rows the resampler reads
    float *x_raw = c->xt[c->xt_cur].as<float>() + (size_t) g0 * rows * kSeriesPerRow;
    if (int rc = stage_input(x_raw, 0))
      return rc;
    CU_TRY(cudaMemset2DAsync(x_new + (size_t) (taps + n_in) * kSeriesPerRow, rows * row_bytes, 0,
                             kChunkRows * row_bytes, ng, stream),
           "pad rows");
    CU_TRY(launch_biquad_tm(x_raw, x_new, rows, taps, n_in, n_series, pre->sections, *pre->params, pre->state,
                            pre->block_rows, pre->warm_rows, stream, pre->blk_state, pre->mismatches,
                            pre->chain_broken),
           "biquad kernel");
  } else {
    // Long float calls of the standard kernel: the transposition signals its progress per row tile and the resampler
    // is launched right behind it as a programmatic dependent (nothing may be enqueued between the two), so the
    // HBM-bound staging hides behind the FMA-bound kernel instead of preceding it.
    if (overlap_ok && c->overlap_staging && !small_stage && !pcm_in && !ptrs && !pre_on && !c->fs_call &&
        !c->kernel_timing && c->sched.generated > 0 &&
        passes_per_slab(c) >= c->plan.n_passes() && n_in >= 8 * kReadyTileRows) {
      CU_TRY(c->d_ready.reserve((size_t) (n_in / kReadyTileRows + 1) * sizeof(int)), "cudaMalloc ready counters");
      if (c->aux_join_pending) {  // the coefficients were expanded on the side stream
        CU_TRY(cudaStreamWaitEvent(stream, c->aux_join, 0), "cudaStreamWaitEvent");
        c->aux_join_pending = false;
      } else if (!g_preexpanded) {  // (a no-op when the cached plan's coefficients are still resident)
        if (int rc = ensure_g(c, 0, (int) c->plan.chunks.size(), stream))
          return rc;
      }
      CU_TRY(launch_transpose_flags(in, il.stream_stride, il.channel_stride, il.frame_stride, c->channels, n_series,
                                    n_in, x_new, rows, taps, kChunkRows, c->d_ready.as<int>(), c->stage_ctas_per_sm,
                                    stream, &ready_tiles),
             "transpose kernel");
    }
    if (!small_stage && ready_tiles == 0)
      if (int rc = stage_input(x_new, kChunkRows))
        return rc;
    if (pre_on)  // resampler.cpp:126-133, on the staged rows [taps, taps + n_in)
      CU_TRY(launch_biquad_tm(x_new, x_new, rows, taps, n_in, n_series, pre->sections, *pre->params, pre->state, 0,
                              0, stream),
             "biquad kernel");
  }
  const bool post_on = post && post->params && c->sched.generated > 0;
  const bool tm_out = (post_on || pcm_out || ptrs) && c->sched.generated > 0;  // a library stage follows the resampler
  float *y_tm = nullptr;
  if (tm_out)
    y_tm = c->yt.as<float>() + (size_t) g0 * c->yt_rows * kSeriesPerRow;
  if (c->sched.generated > 0 && c->fs_call) {
    FsParams fp{};
    fp.x = x_new;
    fp.x_fs = kSeriesPerRow;
    fp.x_row0 = taps;
    fp.out = out;
    fp.out_ss = ol.stream_stride;
    fp.out_cs = ol.channel_stride;
    fp.out_fs = ol.frame_stride;
    fp.out_tm = y_tm;
    fp.bank_tr = c->bank_tr.as<float>();
    fp.outs = c->d_outs.as<OutEntry>();
    fp.n_series = n_series;
    fp.channels = c->channels;
    fp.n_out = (int) c->sched.generated;
    fp.taps = taps;
    fp.kt = c->fs_kt;
    fp.slice_floats = (int) c->fs_slice;
    cudaEvent_t ev_after = nullptr;
    if (c->kernel_timing) {
      while (c->ev_pool.size() < c->ev_used + 2) {
        cudaEvent_t ev;
        CU_TRY(cudaEventCreate(&ev), "cudaEventCreate");
        c->ev_pool.push_back(ev);
      }
      CU_TRY(cudaEventRecord(c->ev_pool[c->ev_used], stream), "cudaEventRecord");
      ev_after = c->ev_pool[c->ev_used + 1];
      c->ev_used += 2;
    }
    CU_TRY(launch_resample_fs(fp, fs_geometry(c->n_series()), c->fs_x_rows, c->mode == ESPB_MODE_EXACT, stream),
           "few-series resample kernel");
    if (ev_after)
      CU_TRY(cudaEventRecord(ev_after, stream), "cudaEventRecord");
  } else if (c->sched.generated > 0) {
    ResampleParams p{};
    p.out_tm = y_tm;
    p.out_tm_rows = c->yt_rows;
    p.xt = direct ? x_old + (size_t) c->carry_row * kSeriesPerRow : x_new;
    p.xt_rows = rows;
    DirectInput din{};
    if (direct) {
      din.in = in;
      din.in_ss = il.stream_stride;
      if (int rc = make_input_map(&din.map, in, il.stream_stride, n_in, n_series / c->channels))
        return rc;
    }
    p.out = out;
    p.out_ss = ol.stream_stride;
    p.out_cs = ol.channel_stride;
    p.out_fs = ol.frame_stride;
    p.chunks = c->p_chunks;
    p.pass_chunk_begin = c->p_pcb;
    p.outs = c->d_outs.as<OutEntry>();
    p.n_series = n_series;
    p.channels = c->channels;
    p.n_out = (int) c->sched.generated;
    p.taps = taps;
    if (ready_tiles > 0) {
      p.ready = c->d_ready.as<int>();
      p.ready_tiles = ready_tiles;
      p.ready_target = ng;
    }
    const int n_passes = c->plan.n_passes();
    const int pps = passes_per_slab(c);
    if (c->aux_join_pending) {  // the coefficients were expanded on the side stream
      CU_TRY(cudaStreamWaitEvent(stream, c->aux_join, 0), "cudaStreamWaitEvent");
      c->aux_join_pending = false;
    }
    for (int pf = 0; pf < n_passes; pf += pps) {
      const int pe = pf + pps < n_passes ? pf + pps : n_passes;
      const int cf = c->plan.pass_chunk_begin[pf], ce = c->plan.pass_chunk_begin[pe];
      if (!g_preexpanded || pps < n_passes) {
        int rc = ensure_g(c, cf, ce, stream);
        if (rc != ESPB_OK)
          return rc;
      }
      p.G = c->d_G.as<float>();
      p.g_chunk_base = cf;
      p.pass_first = pf;
      p.pass_end = pe;
      p.passes_per_cta = pick_passes_per_cta(c, n_series, pf, pe);
      cudaEvent_t ev_after = nullptr;
      if (c->kernel_timing) {
        while (c->ev_pool.size() < c->ev_used + 2) {
          cudaEvent_t ev;
          CU_TRY(cudaEventCreate(&ev), "cudaEventCreate");
          c->ev_pool.push_back(ev);
        }
        CU_TRY(cudaEventRecord(c->ev_pool[c->ev_used], stream), "cudaEventRecord");
        ev_after = c->ev_pool[c->ev_used + 1];
        c->ev_used += 2;
      }
      CU_TRY(launch_resample(p, c->bpp, c->chunk_rows, c->mode == ESPB_MODE_EXACT, stream, direct ? &din : nullptr,
                             c->non_interp),
             "resample kernel");
      if (ev_after)
        CU_TRY(cudaEventRecord(ev_after, stream), "cudaEventRecord");
    }
  }
  if (direct) {  // the next call's carry: frames [used - taps, used), time-major, rows [0, taps) of the other buffer
    const int used = (int) c->sched.used;
    CU_TRY(launch_transpose(in + (int64_t) (used - taps) * il.frame_stride, il.stream_stride, il.channel_stride,
                            il.frame_stride, c->channels, n_series, taps, x_new, rows, 0, 0, stream),
           "carry transpose");
  }
  bool tail_done = false;
  // (worth it for many groups only: the fused kernel's filter warps share their schedulers with the packers and run
  //  1.7 ms for 48005 rows where the plain filter runs 1.15, whatever the number of groups, while the separate
  //  quantising stage costs ~8 us per group — slabs of the host pipeline, 4 groups each, stay with two passes)
  if (tm_out && post_on && pcm_out && c->channels == 1 && ng >= env_long("ESPB_FUSE_POST_GROUPS", 96) &&
      env_long("ESPB_FUSE_POST", 1) != 0 &&
      !(post->block_rows > 0 && (int) c->sched.generated > post->block_rows && c->yt2_rows >= c->yt_rows)) {
    // mono PCM output behind a post-filter (resampler.cpp:142-153): the filter's thread quantises and packs its own
    // results — one pass over the resampler's time-major output instead of two
    const int gen = (int) c->sched.generated;
    cudaError_t e = cudaSuccess;
    const int fast = launch_biquad_tm_pcm(y_tm, c->yt_rows, 0, gen, n_series, post->sections, *post->params,
                                          post->state, pcm_out->data, pcm_out->row_bytes, pcm_out->bits,
                                          pcm_out->clipped, stream, &e);
    CU_TRY(e, "biquad + quantiser kernel");
    if (fast > 0) {
      tail_done = true;
      if (fast < gen) {  // the last partial chunk came back as filtered floats: generic layout stage + quantiser
        const int nbytes = (pcm_out->bits + 7) / 8;
        CU_TRY(launch_untranspose_from(y_tm, c->yt_rows, 0, fast, gen, pcm_out->scratch, pcm_out->scratch_row, 1,
                                       c->channels, c->channels, n_series, stream),
               "untranspose kernel");
        CU_TRY(launch_f2q(pcm_out->scratch + (size_t) fast * c->channels, pcm_out->scratch_row,
                          pcm_out->data + (size_t) fast * c->channels * nbytes, pcm_out->row_bytes, n_series,
                          (uint32_t) ((gen - fast) * c->channels), pcm_out->bits, pcm_out->clipped, true, stream),
               "f2q kernel");
      }
    }
  }
  if (tm_out && !tail_done) {
    const int gen = (int) c->sched.generated;
    float *y_f = y_tm;
    if (post_on) {  // resampler.cpp:142-149
      int blocks = 0;
      if (post->block_rows > 0 && gen > post->block_rows && c->yt2_rows >= c->yt_rows) {
        y_f = c->yt2.as<float>() + (size_t) g0 * c->yt_rows * kSeriesPerRow;
        blocks = post->block_rows;
      }
      CU_TRY(launch_biquad_tm(y_tm, y_f, c->yt_rows, 0, gen, n_series, post->sections, *post->params, post->state,
                              blocks, post->warm_rows, stream, post->blk_state, post->mismatches,
                              post->chain_broken),
             "biquad kernel");
    }
    if (pcm_out) {  // resampler.cpp:152-153: float_to_quantized, fused with the way back to the caller's layout
      cudaError_t e = cudaSuccess;
      const int n_streams = n_series / c->channels;
      const int fast = launch_tm_to_pcm(y_f, c->yt_rows, 0, gen, pcm_out->data, pcm_out->row_bytes, pcm_out->bits,
                                        c->channels, n_series, pcm_out->clipped, stream, &e);
      CU_TRY(e, "tm_to_pcm kernel");
      if (fast < gen) {
        const int nbytes = (pcm_out->bits + 7) / 8;
        if (fast > 0)
          CU_TRY(launch_untranspose_from(y_f, c->yt_rows, 0, fast, gen, pcm_out->scratch, pcm_out->scratch_row, 1,
                                         c->channels, c->channels, n_series, stream),
                 "untranspose kernel");
        else
          CU_TRY(launch_untranspose(y_f, c->yt_rows, 0, gen, pcm_out->scratch, pcm_out->scratch_row, 1, c->channels,
                                    c->channels, n_series, stream),
                 "untranspose kernel");
        CU_TRY(launch_f2q(pcm_out->scratch + (size_t) fast * c->channels, pcm_out->scratch_row,
                          pcm_out->data + (size_t) fast * c->channels * nbytes, pcm_out->row_bytes, n_streams,
                          (uint32_t) ((gen - fast) * c->channels), pcm_out->bits, pcm_out->clipped, true, stream),
               "f2q kernel");
      }
    } else if (ptrs) {
      CU_TRY(launch_untranspose_ptrs(y_f, c->yt_rows, 0, gen, ptrs->out + series_first, n_series, stream),
             "untranspose kernel");
    } else {
      CU_TRY(launch_untranspose(y_f, c->yt_rows, 0, gen, out, ol.stream_stride, ol.channel_stride, ol.frame_stride,
                                c->channels, n_series, stream),
             "untranspose kernel");
    }
  }
  return ESPB_OK;
}

// Scratch for time-major resampler output (post-filter path): at least `rows` rows per group.
int ensure_yt(EspbResampleBatch *c, int64_t rows, bool second) {
  if (rows > c->yt_rows) {
    rows += rows / 64 + 64;  // (head-room: see DevBuf::reserve)
    CU_TRY(c->yt.reserve((size_t) c->n_groups() * rows * kSeriesPerRow * sizeof(float)), "output scratch");
    c->yt_rows = rows;
    c->yt2_rows = 0;
  }
  if (second && c->yt2_rows < c->yt_rows) {
    CU_TRY(c->yt2.reserve((size_t) c->n_groups() * c->yt_rows * kSeriesPerRow * sizeof(float)), "output scratch");
    c->yt2_rows = c->yt_rows;
  }
  return ESPB_OK;
}

void finish_call(EspbResampleBatch *c) {
  // the frames [used - taps, used) of this call are the next call's carry: rows [used, used + taps)
  c->xt_cur = 1 - c->xt_cur;
  c->carry_row = c->direct_call ? 0 : (int) c->sched.used;  // (direct input: the carry was written to rows [0, taps))
  c->state = c->sched.end;
}

}  // namespace

extern "C" {

EspbResampleBatch *espb_resampleInit(int num_streams, int numChannels, int numTaps, int numFilters,
                                     float lowpassRatio, int flags) {
  if (!normalise_init(numTaps, numFilters, &lowpassRatio, &flags)) {
    fail(ESPB_ERR_ARG, "resampleInit: invalid taps/filters");
    return nullptr;
  }
  if (num_streams <= 0 || numChannels <= 0) {
    fail(ESPB_ERR_ARG, "resampleInit: num_streams and numChannels must be positive");
    return nullptr;
  }
  if (espb_device_count() <= 0) {
    fail(ESPB_ERR_CUDA, "resampleInit: no CUDA device (this library has no CPU path)");
    return nullptr;
  }
  EspbResampleBatch *c = new EspbResampleBatch();
  // page-lock the per-call tables where they are built: their uploads become asynchronous DMA copies
  c->sched.outs.on_acquire = c->plan.chunks.on_acquire = c->plan.pass_chunk_begin.on_acquire = pin_host_range;
  c->sched.outs.on_release = c->plan.chunks.on_release = c->plan.pass_chunk_begin.on_release = unpin_host_range;
  c->spare_outs.on_acquire = c->spare_chunks.on_acquire = c->spare_pcb.on_acquire = pin_host_range;
  c->spare_outs.on_release = c->spare_chunks.on_release = c->spare_pcb.on_release = unpin_host_range;
  c->sched.segs.on_acquire = c->spare_segs.on_acquire = pin_host_range;
  c->sched.segs.on_release = c->spare_segs.on_release = unpin_host_range;
  {
    const char *sm = getenv("ESPB_SCHED");
    c->sched_segments = !(sm && strcmp(sm, "seq") == 0);
  }
  cudaGetDevice(&c->device);
  c->num_streams = num_streams;
  c->channels = numChannels;
  c->geo = ArtGeometry{numTaps, numFilters, flags};
  c->lowpass = lowpassRatio;
  c->state = initial_state(numTaps);
  // 4 output blocks (warps) per pass, four CTAs per SM: measured 5 % faster than 8 x 2 at C2 (shorter passes
  // leave less idle time at the pass edges); ESPB_BPP=8 selects the other variant
  c->bpp = env_long("ESPB_BPP", 4) == 8 ? 8 : 4;
  {
    // direct input (no staging pass for interleaved stereo float) is opt-in: measured equal per step at C2 (the kernel
    // is 8 % slower, the 0.58 ms transposition disappears), it only saves the staging memory
    c->direct_ok = env_long("ESPB_DIRECT", 0) != 0;
    const long cr = env_long("ESPB_CHUNK_ROWS", 32);
    c->chunk_rows = (cr == 16 || ((cr == 24 || cr == 36) && c->bpp == 4)) ? (int) cr : 32;
  }
  c->non_interp = (flags & kFlagInterpolate) == 0 && c->bpp == 4 && c->chunk_rows == 32 && env_long("ESPB_NI", 1) != 0;
  long gb = env_long("ESPB_G_MBYTES", 0);
  if (gb > 0)
    c->g_budget_bytes = (size_t) gb << 20;
  build_filter_bank(c->geo, lowpassRatio, c->bank_host);
  const size_t bank_bytes = c->bank_host.size() * sizeof(float);
  cudaError_t e = c->bank.reserve(bank_bytes);
  if (e == cudaSuccess)
    e = cudaMemcpy(c->bank.p, c->bank_host.data(), bank_bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    cuda_fail(e, "resampleInit: device allocation");
    espb_resampleFree(c);
    return nullptr;
  }
  c->fs_policy = (int) env_long("ESPB_FS", -1);
  c->overlap_staging = (int) env_long("ESPB_OVERLAP", 1);
  c->stage_ctas_per_sm = (int) env_long("ESPB_STAGE_CTAS", 2);
  if (e == cudaSuccess && c->n_series() <= kFsMaxSeries && c->fs_policy != 0) {  // few-series form: slice-major bank
    c->fs_kt = fs_slice_taps(numTaps, numFilters);
    c->fs_slice = fs_slice_floats(numFilters, c->fs_kt);
    std::vector<float> tr(c->fs_slice * (numTaps / c->fs_kt));
    fs_build_bank_slices(c->bank_host.data(), numTaps, numFilters, c->fs_kt, tr.data());
    e = c->bank_tr.reserve(tr.size() * sizeof(float));
    if (e == cudaSuccess)
      e = cudaMemcpy(c->bank_tr.p, tr.data(), tr.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cuda_fail(e, "resampleInit: device allocation");
      espb_resampleFree(c);
      return nullptr;
    }
  }
  if (ensure_xt(c, (int64_t) numTaps + kChunkRows) != ESPB_OK) {  // silent history (art_resampler.cpp:125-133)
    espb_resampleFree(c);
    return nullptr;
  }
  return c;
}

void espb_resampleFree(EspbResampleBatch *c) {
  if (!c)
    return;
  c->bank.release();
  c->bank_tr.release();
  c->xt[0].release();
  c->xt[1].release();
  c->yt.release();
  c->yt2.release();
  c->d_outs.release();
  c->d_segs.release();
  c->d_ready.release();
  c->d_tables.release();
  if (c->aux)
    cudaStreamDestroy(c->aux);
  for (cudaEvent_t ev : {c->aux_fork, c->aux_join})
    if (ev)
      cudaEventDestroy(ev);
  c->d_ptrs.release();
  c->d_chunks.release();
  c->d_pcb.release();
  c->d_G.release();
  c->stage_in.release();
  c->stage_out.release();
  c->pipe.destroy();
  for (cudaEvent_t ev : c->ev_pool)
    cudaEventDestroy(ev);
  if (c->state_event)
    cudaEventDestroy(c->state_event);
  for (cudaEvent_t ev : {c->tables_uploaded, c->spare_uploaded})
    if (ev) {
      cudaEventSynchronize(ev);  // the tables are freed (and un-pinned) with the context
      cudaEventDestroy(ev);
    }
  delete c;
}

int espb_resampleReset(EspbResampleBatch *c, void *stream) {
  if (!c)
    return fail(ESPB_ERR_ARG, "resampleReset: NULL context");
  if (c->state_only)
    return fail(ESPB_ERR_STATE, "resampleReset: group of a fused clock-group set (use espb_resampleGroupsReset)");
  const size_t row_bytes = kSeriesPerRow * sizeof(float);
  CU_TRY(cudaMemset2DAsync(c->xt[c->xt_cur].as<float>() + (size_t) c->carry_row * kSeriesPerRow,
                           c->xt_rows * row_bytes, 0, c->geo.taps * row_bytes, c->n_groups(), as_stream(stream)),
         "resampleReset");
  if (!c->state_event)
    CU_TRY(cudaEventCreateWithFlags(&c->state_event, cudaEventDisableTiming), "cudaEventCreate");
  CU_TRY(cudaEventRecord(c->state_event, as_stream(stream)), "cudaEventRecord");
  c->state_event_pending = true;
  c->state = initial_state(c->geo.taps);
  return ESPB_OK;
}

void espb_resampleAdvancePosition(EspbResampleBatch *c, float delta) {
  if (delta < 0.0f)
    fprintf(stderr, "resampleAdvancePosition() can only advance forward!\n");
  else
    c->state.offset += delta;
}

float espb_resampleGetPosition(EspbResampleBatch *c) { return position_of(c->geo, c->state); }

unsigned int espb_resampleGetRequiredSamples(EspbResampleBatch *c, int numOutputFrames, float ratio) {
  return required_samples(c->geo, c->state, numOutputFrames, ratio);
}
unsigned int espb_resampleGetExpectedOutput(EspbResampleBatch *c, int numInputFrames, float ratio) {
  return expected_output(c->geo, c->state, numInputFrames, ratio);
}

int espb_resampleSetMode(EspbResampleBatch *c, int mode) {
  if (!c || (mode != ESPB_MODE_FAST && mode != ESPB_MODE_EXACT))
    return fail(ESPB_ERR_ARG, "resampleSetMode: bad mode");
  c->mode = mode;
  return ESPB_OK;
}

int espb_resampleSetOption(EspbResampleBatch *c, int option, int value) {
  if (!c)
    return fail(ESPB_ERR_ARG, "resampleSetOption: NULL");
  switch (option) {
    case ESPB_OPT_PLAN_CACHE:
      c->plan_cache = value != 0;
      c->plan_on_device = false;
      return ESPB_OK;
    case ESPB_OPT_KERNEL_TIMING:
      c->kernel_timing = value != 0;
      c->ev_used = 0;
      return ESPB_OK;
    case ESPB_OPT_OVERLAP_STAGING:
      c->overlap_staging = value != 0;
      return ESPB_OK;
    default:
      return fail(ESPB_ERR_ARG, "resampleSetOption: unknown option");
  }
}

int espb_resampleGetKernelTime(EspbResampleBatch *c, float *total_ms, int *launches) {
  if (!c || !total_ms)
    return fail(ESPB_ERR_ARG, "resampleGetKernelTime: NULL");
  float sum = 0.0f;
  for (size_t i = 0; i + 1 < c->ev_used; i += 2) {
    CU_TRY(cudaEventSynchronize(c->ev_pool[i + 1]), "cudaEventSynchronize");
    float ms = 0.0f;
    CU_TRY(cudaEventElapsedTime(&ms, c->ev_pool[i], c->ev_pool[i + 1]), "cudaEventElapsedTime");
    sum += ms;
  }
  *total_ms = sum;
  if (launches)
    *launches = (int) (c->ev_used / 2);
  c->ev_used = 0;
  return ESPB_OK;
}

int espb_resampleGetFlags(EspbResampleBatch *c) { return c->geo.flags; }
void espb_resampleGetState(EspbResampleBatch *c, float *outputOffset, int *inputIndex) {
  *outputOffset = c->state.offset;
  *inputIndex = c->state.index;
}
int espb_resampleCopyFilters(EspbResampleBatch *c, float *host_dst) {
  if (c->state_only) {
    memcpy(host_dst, c->bank_host.data(), c->bank_host.size() * sizeof(float));
    return ESPB_OK;
  }
  // read back from the device copy: what the kernels actually use
  CU_TRY(cudaMemcpy(host_dst, c->bank.p, c->bank_host.size() * sizeof(float), cudaMemcpyDeviceToHost),
         "resampleCopyFilters");
  return ESPB_OK;
}

EspbResampleResult espb_resampleProcessLayout(EspbResampleBatch *c, const float *in, const EspbLayout *il,
                                              int numInputFrames, float *out, const EspbLayout *ol,
                                              int numOutputFrames, float ratio, void *stream) {
  EspbResampleResult res = {0, 0};
  if (!c || !il || !ol) {
    fail(ESPB_ERR_ARG, "resampleProcess: NULL argument");
    return res;
  }
  if (numInputFrames < 0)
    numInputFrames = 0;
  if (prepare_call(c, numInputFrames, numOutputFrames, ratio, as_stream(stream), direct_input_layout(c, in, *il)) !=
      ESPB_OK)
    return res;
  // Long calls: expand the coefficients on a side stream while this stream stages the input (two bandwidth-bound
  // kernels that do not depend on each other); the resampler launch waits for both.
  bool pre = false;
  if (!c->fs_call && c->sched.generated > 4096 && passes_per_slab(c) >= c->plan.n_passes() &&
      !(c->g_resident_first == 0 && c->g_resident_end == (int) c->plan.chunks.size())) {
    cudaError_t e = cudaSuccess;
    if (!c->aux) {
      e = cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking);
      if (e == cudaSuccess)
        e = cudaEventCreateWithFlags(&c->aux_fork, cudaEventDisableTiming);
      if (e == cudaSuccess)
        e = cudaEventCreateWithFlags(&c->aux_join, cudaEventDisableTiming);
    }
    if (e == cudaSuccess)
      e = cudaEventRecord(c->aux_fork, as_stream(stream));
    if (e == cudaSuccess)
      e = cudaStreamWaitEvent(c->aux, c->aux_fork, 0);
    if (e != cudaSuccess) {
      cuda_fail(e, "side stream");
      return res;
    }
    if (ensure_g(c, 0, (int) c->plan.chunks.size(), c->aux) != ESPB_OK)
      return res;
    if (cudaEventRecord(c->aux_join, c->aux) != cudaSuccess) {
      fail(ESPB_ERR_CUDA, "side stream event");
      return res;
    }
    c->aux_join_pending = true;
    pre = true;
  }
  if (run_series_range(c, 0, c->n_series(), in, *il, out, *ol, numInputFrames, as_stream(stream), pre, nullptr, nullptr,
                       nullptr, nullptr, nullptr, /*overlap_ok=*/true) != ESPB_OK)
    return res;
  res.input_used = c->sched.used;
  res.output_generated = c->sched.generated;
  finish_call(c);
  g_last_error.clear(), g_last_status = ESPB_OK;
  return res;
}

EspbResampleResult espb_resampleProcessInterleaved(EspbResampleBatch *c, const float *in, int64_t in_stream_stride,
                                                   int numInputFrames, float *out, int64_t out_stream_stride,
                                                   int numOutputFrames, float ratio, void *stream) {
  if (!c) {
    fail(ESPB_ERR_ARG, "resampleProcessInterleaved: NULL context");
    return EspbResampleResult{0, 0};
  }
  EspbLayout il = {in_stream_stride, 1, c->channels}, ol = {out_stream_stride, 1, c->channels};
  return espb_resampleProcessLayout(c, in, &il, numInputFrames, out, &ol, numOutputFrames, ratio, stream);
}

EspbResampleResult espb_resampleProcess(EspbResampleBatch *c, const float *in, int64_t in_stream_stride,
                                        int64_t in_channel_stride, int numInputFrames, float *out,
                                        int64_t out_stream_stride, int64_t out_channel_stride, int numOutputFrames,
                                        float ratio, void *stream) {
  EspbLayout il = {in_stream_stride, in_channel_stride, 1}, ol = {out_stream_stride, out_channel_stride, 1};
  return espb_resampleProcessLayout(c, in, &il, numInputFrames, out, &ol, numOutputFrames, ratio, stream);
}

// resampleProcess with the reference's own argument form (include/art_resampler.h:36-37): one pointer per plane.
// `inputs` / `outputs` are HOST arrays of num_streams * numChannels DEVICE pointers (plane q = stream q / channels,
// channel q % channels), each plane a separately allocated buffer of numInputFrames / numOutputFrames floats.
EspbResampleResult espb_resampleProcessPlanes(EspbResampleBatch *c, const float *const *inputs, int numInputFrames,
                                              float *const *outputs, int numOutputFrames, float ratio, void *stream) {
  EspbResampleResult res = {0, 0};
  if (!c || !inputs || !outputs) {
    fail(ESPB_ERR_ARG, "resampleProcessPlanes: NULL argument");
    return res;
  }
  if (numInputFrames < 0)
    numInputFrames = 0;
  cudaStream_t s = as_stream(stream);
  if (prepare_call(c, numInputFrames, numOutputFrames, ratio, s, false) != ESPB_OK)
    return res;
  const size_t n = (size_t) c->n_series();
  // the tables are small (8 bytes per plane) and pageable: the driver copies them out before the call returns
  if (c->d_ptrs.reserve(2 * n * sizeof(void *)) != cudaSuccess ||
      cudaMemcpyAsync(c->d_ptrs.p, inputs, n * sizeof(void *), cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(c->d_ptrs.as<void *>() + n, outputs, n * sizeof(void *), cudaMemcpyHostToDevice, s) !=
          cudaSuccess) {
    fail(ESPB_ERR_CUDA, "resampleProcessPlanes: pointer tables");
    return res;
  }
  if (ensure_yt(c, (int64_t) c->sched.generated, false) != ESPB_OK)
    return res;
  PtrIO io;
  io.in = reinterpret_cast<const float *const *>(c->d_ptrs.p);
  io.out = reinterpret_cast<float *const *>(c->d_ptrs.as<void *>() + n);
  const EspbLayout none = {0, 0, 1};
  if (run_series_range(c, 0, c->n_series(), nullptr, none, nullptr, none, numInputFrames, s, false, nullptr, nullptr,
                       nullptr, nullptr, &io) != ESPB_OK)
    return res;
  res.input_used = c->sched.used;
  res.output_generated = c->sched.generated;
  finish_call(c);
  g_last_error.clear(), g_last_status = ESPB_OK;
  return res;
}

// Host-buffer variant: rows of `in`/`out` are host memory (pinned for full PCIe speed).
// Streams are cut into slabs; slab i copies in, resamples and copies out on CUDA stream
// i % 3 so that H2D, compute and D2H of neighbouring slabs overlap.  Synchronous.
EspbResampleResult espb_resampleProcessInterleavedHost(EspbResampleBatch *c, const float *in,
                                                       int64_t in_stream_stride, int numInputFrames, float *out,
                                                       int64_t out_stream_stride, int numOutputFrames, float ratio);

}  // extern "C"

extern "C" {

EspbResampleResult espb_resampleProcessInterleavedHost(EspbResampleBatch *c, const float *in,
                                                       int64_t in_stream_stride, int numInputFrames, float *out,
                                                       int64_t out_stream_stride, int numOutputFrames, float ratio) {
  EspbResampleResult res = {0, 0};
  if (!c) {
    fail(ESPB_ERR_ARG, "resampleProcessInterleavedHost: NULL context");
    return res;
  }
  if (numInputFrames < 0)
    numInputFrames = 0;
  EspbResampleBatch *hs = c;
  cudaError_t e = hs->pipe.init();
  if (e != cudaSuccess) {
    cuda_fail(e, "host pipeline streams");
    return res;
  }
  const int ch = c->channels;
  const size_t in_row = (size_t) numInputFrames * ch, out_cap_row = (size_t) (numOutputFrames > 0 ? numOutputFrames : 0) * ch;
  if (hs->stage_in.reserve((in_row ? in_row : 1) * c->num_streams * sizeof(float)) != cudaSuccess ||
      hs->stage_out.reserve((out_cap_row ? out_cap_row : 1) * c->num_streams * sizeof(float)) != cudaSuccess) {
    fail(ESPB_ERR_NOMEM, "host stage device buffers");
    return res;
  }
  cudaStream_t s0 = hs->pipe.s[0];
  const int per = pick_slab_streams(c->num_streams, c->channels);
  if (in_row) {  // the first slab's copy needs no plan: it runs while the host builds the schedule
    const int ns0 = per <= c->num_streams ? per : c->num_streams;
    e = copy_rows_async(hs->stage_in.as<float>(), in_row * sizeof(float), in, (size_t) in_stream_stride * sizeof(float),
                        in_row * sizeof(float), ns0, cudaMemcpyHostToDevice, s0);
    if (e != cudaSuccess) {
      cuda_fail(e, "h2d");
      return res;
    }
  }
  {
    const EspbLayout stage_layout = {(int64_t) in_row, 1, ch};
    if (prepare_call(c, numInputFrames, numOutputFrames, ratio, s0,
                     direct_input_layout(c, hs->stage_in.as<float>(), stage_layout)) != ESPB_OK)
      return res;
  }
  const size_t out_row = (size_t) c->sched.generated * ch;
  const bool single_slab_g = passes_per_slab(c) >= c->plan.n_passes();
  if (c->sched.generated > 0 && single_slab_g && !c->fs_call) {
    if (ensure_g(c, 0, (int) c->plan.chunks.size(), s0) != ESPB_OK)
      return res;
  }
  cudaEventRecord(hs->pipe.ready, s0);
  EspbLayout il = {(int64_t) in_row, 1, ch}, ol = {(int64_t) out_cap_row, 1, ch};
  int slab = 0;
  for (int st0 = 0; st0 < c->num_streams; st0 += per, ++slab) {
    const int ns = st0 + per <= c->num_streams ? per : c->num_streams - st0;
    cudaStream_t s = single_slab_g ? hs->pipe.s[slab % HostPipe::kStreams] : s0;
    cudaStreamWaitEvent(s, hs->pipe.ready, 0);
    float *din = hs->stage_in.as<float>() + (size_t) st0 * in_row;
    float *dout = hs->stage_out.as<float>() + (size_t) st0 * out_cap_row;
    if (in_row && slab > 0) {  // (slab 0 was copied before the planning)
      e = copy_rows_async(din, in_row * sizeof(float), in + (size_t) st0 * in_stream_stride,
                          (size_t) in_stream_stride * sizeof(float), in_row * sizeof(float), ns,
                          cudaMemcpyHostToDevice, s);
      if (e != cudaSuccess) {
        cuda_fail(e, "h2d");
        hs->pipe.drain();
        return res;
      }
    }
    if (run_series_range(c, st0 * ch, ns * ch, din, il, dout, ol, numInputFrames, s, single_slab_g) != ESPB_OK) {
      hs->pipe.drain();
      return res;
    }
    if (out_row) {
      e = copy_rows_async(out + (size_t) st0 * out_stream_stride, (size_t) out_stream_stride * sizeof(float), dout,
                          out_cap_row * sizeof(float), out_row * sizeof(float), ns, cudaMemcpyDeviceToHost, s);
      if (e != cudaSuccess) {
        cuda_fail(e, "d2h");
        hs->pipe.drain();
        return res;
      }
    }
  }
  for (int i = 0; i < HostPipe::kStreams; ++i) {
    e = cudaStreamSynchronize(hs->pipe.s[i]);
    if (e != cudaSuccess) {
      cuda_fail(e, "host pipeline sync");
      return res;
    }
  }
  res.input_used = c->sched.used;
  res.output_generated = c->sched.generated;
  finish_call(c);
  g_last_error.clear(), g_last_status = ESPB_OK;
  return res;
}

// ------------------------------------------------------------------------------------
// art_biquad
// ------------------------------------------------------------------------------------
void espb_biquad_lowpass(EspbBiquadCoefficients *f, double frequency) {
  design_lowpass(reinterpret_cast<BiquadCoeffs *>(f), frequency);
}
void espb_biquad_highpass(EspbBiquadCoefficients *f, double frequency) {
  design_highpass(reinterpret_cast<BiquadCoeffs *>(f), frequency);
}

}  // extern "C"

struct EspbBiquadBatch {
  int num_series = 0, num_sections = 0;
  BiquadParams params{};
  DevBuf state;
  DevBuf tm, tm2;  // time-major scratch [group][tm_rows][128] (tm2: output side of the time-block mode)
  int64_t tm_rows = 0, tm2_rows = 0;
  // Time blocks (biquad_kernel.cu): -1 = automatic (few series and a long call: blocks of kAutoBlockRows rows),
  // 0 = one sequential run per series, > 0 = blocks of that many rows.  Exact either way: the hand-over between
  // blocks is verified bit for bit on the device and repaired where the warm-up did not converge.
  int block_rows = -1, warm_rows = 1024;
  bool one_pass = true;  // ESPB_BIQUAD_ONEPASS=0: always through time-major scratch (three passes)
  DevBuf blk_state;                      // (start, end) state of every block, for the verify kernel
  DevBuf chain_broken;                   // [groups] scratch flags of the parallel hand-over check
  DevBuf mismatch_dev;                   // [1] blocks repaired so far in the call being enqueued
  unsigned int *mismatch_host = nullptr; // pinned copy of the previous call's count
  cudaEvent_t mismatch_ready = nullptr;
  bool mismatch_pending = false;
  uint64_t repaired_total = 0;
  static constexpr int kAutoBlockRows = 8192, kAutoMaxGroups = 32, kMaxWarmRows = 1 << 16;
  static constexpr int kAutoBlockRowsFew = 2048;  // (espb_biquad_tm_few_kernel: nothing is staged, short blocks pay)
  int n_groups() const { return (num_series + kSeriesPerRow - 1) / kSeriesPerRow; }
  // rows per block for a call over n_rows rows (0: sequential)
  int blocks_for(int n_rows) const {
    if (block_rows > 0)
      return n_rows > block_rows ? block_rows : 0;
    if (block_rows < 0 && n_groups() <= kAutoMaxGroups && n_rows >= 2 * kAutoBlockRows)
      return num_series <= kBiquadFewSeries ? kAutoBlockRowsFew : kAutoBlockRows;
    return 0;
  }
};

namespace {

// Before a time-block launch: size the state record, harvest the previous call's repair count (widening the warm-up
// when the trajectories did not merge), clear the counter.  No synchronisation.
int biquad_prepare_blocks(EspbBiquadBatch *f, int n_rows, int block_rows, cudaStream_t stream) {
  const size_t floats = biquad_block_state_floats(f->num_series, f->num_sections, n_rows, block_rows);
  CU_TRY(f->blk_state.reserve(floats * sizeof(float)), "biquad block states");
  CU_TRY(f->chain_broken.reserve((size_t) ((f->num_series + kSeriesPerRow - 1) / kSeriesPerRow) * sizeof(unsigned int)),
         "biquad chain flags");
  if (!f->mismatch_dev.p) {
    CU_TRY(f->mismatch_dev.reserve(sizeof(unsigned int)), "biquad counter");
    CU_TRY(cudaMallocHost(&f->mismatch_host, sizeof(unsigned int)), "biquad counter");
    *f->mismatch_host = 0;
    CU_TRY(cudaEventCreateWithFlags(&f->mismatch_ready, cudaEventDisableTiming), "cudaEventCreate");
  }
  if (f->mismatch_pending && cudaEventQuery(f->mismatch_ready) == cudaSuccess) {
    f->mismatch_pending = false;
    if (*f->mismatch_host > 0) {
      f->repaired_total += *f->mismatch_host;
      if (f->warm_rows < EspbBiquadBatch::kMaxWarmRows)
        f->warm_rows *= 2;
    }
  }
  cudaGetLastError();  // (cudaErrorNotReady from the query is not an error)
  CU_TRY(cudaMemsetAsync(f->mismatch_dev.p, 0, sizeof(unsigned int), stream), "biquad counter");
  return ESPB_OK;
}

// After the launches of a call: bring the repair count to the host without waiting for it.
int biquad_finish_blocks(EspbBiquadBatch *f, cudaStream_t stream) {
  if (f->mismatch_pending)  // an earlier count has not been read yet: keep it (it is added up on the device side)
    return ESPB_OK;
  CU_TRY(cudaMemcpyAsync(f->mismatch_host, f->mismatch_dev.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, stream),
         "biquad counter");
  CU_TRY(cudaEventRecord(f->mismatch_ready, stream), "cudaEventRecord");
  f->mismatch_pending = true;
  return ESPB_OK;
}

}  // namespace

extern "C" {

EspbBiquadBatch *espb_biquad_init(int num_series, int num_sections, const EspbBiquadCoefficients *coeffs,
                                  float gain) {
  if (num_series <= 0 || num_sections < 1 || num_sections > 4 || !coeffs) {
    fail(ESPB_ERR_ARG, "biquad_init: bad arguments (1..4 sections)");
    return nullptr;
  }
  if (espb_device_count() <= 0) {
    fail(ESPB_ERR_CUDA, "biquad_init: no CUDA device (this library has no CPU path)");
    return nullptr;
  }
  EspbBiquadBatch *f = new EspbBiquadBatch();
  f->num_series = num_series;
  f->num_sections = num_sections;
  // art_biquad.cpp:43-51
  f->params.a0 = coeffs->a0 * gain;
  f->params.a1 = coeffs->a1 * gain;
  f->params.a2 = coeffs->a2 * gain;
  f->params.b1 = coeffs->b1;
  f->params.b2 = coeffs->b2;
  f->params.first_order = (coeffs->a2 == 0.0f && coeffs->b2 == 0.0f);
  f->one_pass = env_long("ESPB_BIQUAD_ONEPASS", 1) != 0;
  const size_t bytes = (size_t) num_series * num_sections * 4 * sizeof(float);
  cudaError_t e = f->state.reserve(bytes);
  if (e == cudaSuccess)
    e = cudaMemset(f->state.p, 0, bytes);
  if (e != cudaSuccess) {
    cuda_fail(e, "biquad_init: device allocation");
    f->state.release();
    delete f;
    return nullptr;
  }
  return f;
}

void espb_biquad_free(EspbBiquadBatch *f) {
  if (!f)
    return;
  f->tm.release();
  f->tm2.release();
  f->state.release();
  f->blk_state.release();
  f->chain_broken.release();
  f->mismatch_dev.release();
  if (f->mismatch_host)
    cudaFreeHost(f->mismatch_host);
  if (f->mismatch_ready)
    cudaEventDestroy(f->mismatch_ready);
  delete f;
}

int espb_biquad_reset(EspbBiquadBatch *f, void *stream) {
  if (!f)
    return fail(ESPB_ERR_ARG, "biquad_reset: NULL");
  CU_TRY(cudaMemsetAsync(f->state.p, 0, (size_t) f->num_series * f->num_sections * 4 * sizeof(float),
                         as_stream(stream)),
         "biquad_reset");
  return ESPB_OK;
}

int espb_biquad_apply_buffer(EspbBiquadBatch *f, float *buf, const EspbLayout *layout, int channels, int num_samples,
                             void *stream) {
  if (!f || !layout || channels <= 0)
    return fail(ESPB_ERR_ARG, "biquad_apply_buffer: bad arguments");
  if (num_samples <= 0)
    return ESPB_OK;
  const int blocks = f->blocks_for(num_samples);
  if (blocks == 0 && f->one_pass) {
    // many series (or a short call): ONE pass on the caller's layout — 8 bytes of traffic per sample
    cudaError_t e = launch_biquad_cl(buf, layout->stream_stride, layout->channel_stride, layout->frame_stride, channels,
                                     f->num_series, num_samples, f->num_sections, f->params, f->state.as<float>(),
                                     as_stream(stream));
    if (e == cudaSuccess)
      return ESPB_OK;
    if (e != cudaErrorNotSupported)
      return cuda_fail(e, "biquad kernel");
    cudaGetLastError();
  }
  // few series and a long call (time blocks), or a layout the one-pass kernel does not take:
  // caller layout -> time-major scratch -> filter -> back
  const int n_groups = (f->num_series + kSeriesPerRow - 1) / kSeriesPerRow;
  if (num_samples > f->tm_rows) {
    CU_TRY(f->tm.reserve((size_t) n_groups * num_samples * kSeriesPerRow * sizeof(float)), "biquad scratch");
    f->tm_rows = num_samples;
  }
  cudaStream_t s = as_stream(stream);
  CU_TRY(launch_transpose(buf, layout->stream_stride, layout->channel_stride, layout->frame_stride, channels,
                          f->num_series, num_samples, f->tm.as<float>(), f->tm_rows, 0, 0, s),
         "transpose kernel");
  float *filtered = f->tm.as<float>();
  if (blocks > 0) {
    if (f->tm_rows > f->tm2_rows) {
      CU_TRY(f->tm2.reserve((size_t) n_groups * f->tm_rows * kSeriesPerRow * sizeof(float)), "biquad scratch");
      f->tm2_rows = f->tm_rows;
    }
    filtered = f->tm2.as<float>();
    if (int rc = biquad_prepare_blocks(f, num_samples, blocks, s))
      return rc;
  }
  CU_TRY(launch_biquad_tm(f->tm.as<float>(), filtered, f->tm_rows, 0, num_samples, f->num_series, f->num_sections,
                          f->params, f->state.as<float>(), blocks, f->warm_rows, s, f->blk_state.as<float>(),
                          f->mismatch_dev.as<unsigned int>(), blocks > 0 ? f->chain_broken.as<unsigned int>() : nullptr),
         "biquad kernel");
  if (blocks > 0)
    if (int rc = biquad_finish_blocks(f, s))
      return rc;
  CU_TRY(launch_untranspose(filtered, f->tm_rows, 0, num_samples, buf, layout->stream_stride,
                            layout->channel_stride, layout->frame_stride, channels, f->num_series, s),
         "untranspose kernel");
  return ESPB_OK;
}

// biquad_apply_sample (art_biquad.cpp:55-69) for every series at once: samples[q] is filtered in place through
// series q's sections, the delays advance by one sample.
int espb_biquad_apply_samples(EspbBiquadBatch *f, float *samples, void *stream) {
  const EspbLayout one_per_series = {1, 1, 1};
  return espb_biquad_apply_buffer(f, samples, &one_per_series, 1, 1, stream);
}

int espb_biquad_set_time_blocks(EspbBiquadBatch *f, int block_rows, int warmup_rows) {
  if (!f || block_rows < -1 || warmup_rows < 0 || (block_rows > 0 && block_rows % 32) || warmup_rows % 32)
    return fail(ESPB_ERR_ARG, "biquad_set_time_blocks: rows must be non-negative multiples of 32 (-1: automatic)");
  f->block_rows = block_rows;
  if (warmup_rows > 0 || block_rows > 0)
    f->warm_rows = warmup_rows;
  return ESPB_OK;
}

// Diagnostics of the time-block mode: blocks whose hand-over had to be repaired so far (0 when every warm-up merged)
// and the current warm-up length.  Synchronises with the last call.
int espb_biquad_block_stats(EspbBiquadBatch *f, uint64_t *repaired_blocks, int *warmup_rows) {
  if (!f)
    return fail(ESPB_ERR_ARG, "biquad_block_stats: NULL");
  if (f->mismatch_pending) {
    CU_TRY(cudaEventSynchronize(f->mismatch_ready), "cudaEventSynchronize");
    f->mismatch_pending = false;
    f->repaired_total += *f->mismatch_host;
    if (*f->mismatch_host > 0 && f->warm_rows < EspbBiquadBatch::kMaxWarmRows)
      f->warm_rows *= 2;
  }
  if (repaired_blocks)
    *repaired_blocks = f->repaired_total;
  if (warmup_rows)
    *warmup_rows = f->warm_rows;
  return ESPB_OK;
}

int espb_biquad_get_state(EspbBiquadBatch *f, float *host_dst) {
  CU_TRY(cudaMemcpy(host_dst, f->state.p, (size_t) f->num_series * f->num_sections * 4 * sizeof(float),
                    cudaMemcpyDeviceToHost),
         "biquad_get_state");
  return ESPB_OK;
}

// ------------------------------------------------------------------------------------
// quantization_utils
// ------------------------------------------------------------------------------------
static int check_bits(uint8_t bits, const char *who) {
  if (bits < 1 || bits > 32)
    return fail(ESPB_ERR_ARG, who, "bits must be 1..32");
  return ESPB_OK;
}

int espb_quantized_to_float_rows(const uint8_t *in, int64_t in_row_stride_bytes, float *out,
                                 int64_t out_row_stride_floats, int rows, uint32_t row_samples, uint8_t input_bits,
                                 float gain_db, void *stream) {
  if (check_bits(input_bits, "quantized_to_float") != ESPB_OK)
    return ESPB_ERR_ARG;
  CU_TRY(launch_q2f(in, in_row_stride_bytes, out, out_row_stride_floats, rows, row_samples, input_bits,
                    q2f_gain_factor(input_bits, gain_db), as_stream(stream)),
         "q2f kernel");
  return ESPB_OK;
}

int espb_float_to_quantized_rows(const float *in, int64_t in_row_stride_floats, uint8_t *out,
                                 int64_t out_row_stride_bytes, int rows, uint32_t row_samples, uint8_t output_bits,
                                 uint32_t *clipped_per_row_dev, void *stream) {
  if (check_bits(output_bits, "float_to_quantized") != ESPB_OK)
    return ESPB_ERR_ARG;
  CU_TRY(launch_f2q(in, in_row_stride_floats, out, out_row_stride_bytes, rows, row_samples, output_bits,
                    clipped_per_row_dev, true, as_stream(stream)),
         "f2q kernel");
  return ESPB_OK;
}

// A flat buffer is cut into rows of 2^22 samples so that 32-bit indexing inside the kernel is safe.
static const uint64_t kFlatRow = (uint64_t) 1 << 22;

int espb_quantized_to_float(const uint8_t *in, float *out, uint64_t num_samples, uint8_t input_bits, float gain_db,
                            void *stream) {
  if (check_bits(input_bits, "quantized_to_float") != ESPB_OK)
    return ESPB_ERR_ARG;
  const int nbytes = (input_bits + 7) / 8;
  const float k = q2f_gain_factor(input_bits, gain_db);
  const uint64_t full = num_samples / kFlatRow, rem = num_samples % kFlatRow;
  for (uint64_t r0 = 0; r0 < full; r0 += 32768) {
    const int rows = (int) (full - r0 < 32768 ? full - r0 : 32768);
    CU_TRY(launch_q2f(in + r0 * kFlatRow * nbytes, (int64_t) kFlatRow * nbytes, out + r0 * kFlatRow,
                      (int64_t) kFlatRow, rows, (uint32_t) kFlatRow, input_bits, k, as_stream(stream)),
           "q2f kernel");
  }
  if (rem)
    CU_TRY(launch_q2f(in + full * kFlatRow * nbytes, 0, out + full * kFlatRow, 0, 1, (uint32_t) rem, input_bits, k,
                      as_stream(stream)),
           "q2f kernel");
  return ESPB_OK;
}

int espb_float_to_quantized(const float *in, uint8_t *out, uint64_t num_samples, uint8_t output_bits,
                            uint32_t *clipped_dev, void *stream) {
  if (check_bits(output_bits, "float_to_quantized") != ESPB_OK)
    return ESPB_ERR_ARG;
  const int nbytes = (output_bits + 7) / 8;
  const uint64_t full = num_samples / kFlatRow, rem = num_samples % kFlatRow;
  for (uint64_t r0 = 0; r0 < full; r0 += 32768) {
    const int rows = (int) (full - r0 < 32768 ? full - r0 : 32768);
    CU_TRY(launch_f2q(in + r0 * kFlatRow, (int64_t) kFlatRow, out + r0 * kFlatRow * nbytes,
                      (int64_t) kFlatRow * nbytes, rows, (uint32_t) kFlatRow, output_bits, clipped_dev, false,
                      as_stream(stream)),
           "f2q kernel");
  }
  if (rem)
    CU_TRY(launch_f2q(in + full * kFlatRow, 0, out + full * kFlatRow * nbytes, 0, 1, (uint32_t) rem, output_bits,
                      clipped_dev, false, as_stream(stream)),
           "f2q kernel");
  return ESPB_OK;
}

uint32_t espb_float_to_quantized_sync(const float *in, uint8_t *out, uint64_t num_samples, uint8_t output_bits,
                                      void *stream) {
  uint32_t *d = nullptr, h = 0;
  if (cudaMalloc(&d, sizeof(uint32_t)) != cudaSuccess) {
    fail(ESPB_ERR_NOMEM, "float_to_quantized: counter");
    return 0;
  }
  cudaMemsetAsync(d, 0, sizeof(uint32_t), as_stream(stream));
  if (espb_float_to_quantized(in, out, num_samples, output_bits, d, stream) == ESPB_OK) {
    cudaMemcpyAsync(&h, d, sizeof(uint32_t), cudaMemcpyDeviceToHost, as_stream(stream));
    cudaError_t e = cudaStreamSynchronize(as_stream(stream));
    if (e != cudaSuccess)
      cuda_fail(e, "float_to_quantized sync");
  }
  cudaFree(d);
  return h;
}

// ------------------------------------------------------------------------------------
// host-side planning (no device)
// ------------------------------------------------------------------------------------
int espb_plan_filter_bank(int numTaps, int numFilters, float lowpassRatio, int flags, float *host_dst,
                          int *effective_flags) {
  if (!normalise_init(numTaps, numFilters, &lowpassRatio, &flags))
    return fail(ESPB_ERR_ARG, "plan_filter_bank: invalid taps/filters");
  std::vector<float> bank;
  build_filter_bank(ArtGeometry{numTaps, numFilters, flags}, lowpassRatio, bank);
  if (host_dst)
    memcpy(host_dst, bank.data(), bank.size() * sizeof(float));
  if (effective_flags)
    *effective_flags = flags;
  return ESPB_OK;
}

int espb_plan_schedule(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex,
                       int numInputFrames, int numOutputFrames, float ratio, unsigned int *input_used,
                       unsigned int *output_generated, float *end_outputOffset, int *end_inputIndex,
                       int32_t *window_start, int32_t *phase, float *weight, int32_t *kind) {
  if ((numTaps & 3) || numTaps <= 0 || numTaps > 1024 || numFilters < 2 || numFilters > 1024)
    return fail(ESPB_ERR_ARG, "plan_schedule: invalid taps/filters");
  Schedule s;
  build_schedule(ArtGeometry{numTaps, numFilters, flags}, ArtState{outputOffset, inputIndex}, numInputFrames,
                 numOutputFrames, ratio, s);
  if (input_used)
    *input_used = s.used;
  if (output_generated)
    *output_generated = s.generated;
  if (end_outputOffset)
    *end_outputOffset = s.end.offset;
  if (end_inputIndex)
    *end_inputIndex = s.end.index;
  for (size_t i = 0; i < s.outs.size(); ++i) {
    if (window_start)
      window_start[i] = s.outs[i].ws;
    if (phase)
      phase[i] = s.outs[i].phase;
    if (weight)
      weight[i] = s.outs[i].w;
    if (kind)
      kind[i] = s.outs[i].kind;
  }
  return ESPB_OK;
}

// The same entries through the closed-form (segmented) schedule and its host expansion: what the device path
// computes.  Returns the number of segments (< 0 on error); outputs as in espb_plan_schedule.
int espb_plan_schedule_segments(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex,
                                int numInputFrames, int numOutputFrames, float ratio, unsigned int *input_used,
                                unsigned int *output_generated, float *end_outputOffset, int *end_inputIndex,
                                int32_t *window_start, int32_t *phase, float *weight, int32_t *kind) {
  if ((numTaps & 3) || numTaps <= 0 || numTaps > 1024 || numFilters < 2 || numFilters > 1024)
    return fail(ESPB_ERR_ARG, "plan_schedule_segments: invalid taps/filters");
  const ArtGeometry geo{numTaps, numFilters, flags};
  Schedule s;
  build_schedule_segments(geo, ArtState{outputOffset, inputIndex}, numInputFrames, numOutputFrames, ratio, s);
  if (input_used)
    *input_used = s.used;
  if (output_generated)
    *output_generated = s.generated;
  if (end_outputOffset)
    *end_outputOffset = s.end.offset;
  if (end_inputIndex)
    *end_inputIndex = s.end.index;
  if (window_start || phase || weight || kind) {
    std::vector<OutEntry> e(s.generated ? s.generated : 1);
    expand_segments(geo, s, e.data());
    int cursor = 0;
    for (size_t i = 0; i < s.generated; ++i) {
      if (window_start)
        window_start[i] = e[i].ws;
      if (phase)
        phase[i] = e[i].phase;
      if (weight)
        weight[i] = e[i].w;
      if (kind)
        kind[i] = e[i].kind;
      if (schedule_ws(s, (int) i, &cursor) != e[i].ws)
        return fail(ESPB_ERR_STATE, "plan_schedule_segments: schedule_ws disagrees with the expansion");
    }
  }
  return (int) s.segs.size();
}

int espb_plan_passes(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex, int numInputFrames,
                     int numOutputFrames, float ratio, int blocks_per_pass, int chunk_rows, int split_at_zero,
                     int32_t *chunk_start, int32_t *chunk_pass, int max_chunks, int32_t *pass_chunk_begin,
                     int max_passes) {
  if ((numTaps & 3) || numTaps <= 0 || numTaps > 1024 || numFilters < 2 || numFilters > 1024 || blocks_per_pass <= 0 ||
      chunk_rows <= 0 || chunk_rows > kChunkRows)
    return fail(ESPB_ERR_ARG, "plan_passes: invalid argument");
  Schedule s;
  build_schedule(ArtGeometry{numTaps, numFilters, flags}, ArtState{outputOffset, inputIndex}, numInputFrames,
                 numOutputFrames, ratio, s);
  PassPlan plan;
  build_pass_plan(s, numTaps, blocks_per_pass, chunk_rows, plan, split_at_zero != 0);
  const int n_chunks = (int) plan.chunks.size(), n_passes = plan.n_passes();
  for (int i = 0; i < n_chunks && i < max_chunks; ++i) {
    if (chunk_start)
      chunk_start[i] = plan.chunks[i].j_start;
    if (chunk_pass)
      chunk_pass[i] = plan.chunks[i].pass;
  }
  for (int i = 0; i <= n_passes && i < max_passes; ++i)
    if (pass_chunk_begin)
      pass_chunk_begin[i] = plan.pass_chunk_begin[i];
  return n_chunks;
}

int espb_plan_policy(const EspbResamplerConfiguration *config, EspbBiquadCoefficients *coeffs, float *sample_ratio,
                     float *art_lowpass, int *art_flags) {
  if (!config)
    return fail(ESPB_ERR_ARG, "plan_policy: NULL");
  WrapperPolicy p;
  decide_policy(config->source_sample_rate, config->target_sample_rate, config->number_of_taps,
                config->use_pre_or_post_filter != 0, config->subsample_interpolate != 0, &p);
  if (coeffs)
    memcpy(coeffs, &p.coeffs, sizeof(EspbBiquadCoefficients));
  if (sample_ratio)
    *sample_ratio = p.sample_ratio;
  if (art_lowpass)
    *art_lowpass = p.art_lowpass;
  if (art_flags) {  // resampleInit would normalise the flags the same way
    float lp = p.art_lowpass;
    int fl = p.art_flags;
    if (lp > 0.0f && lp < 1.0f)
      fl |= kFlagLowpass;
    else
      fl &= ~kFlagLowpass;
    *art_flags = p.resampling ? fl : 0;
  }
  return p.pre ? 1 : (p.post ? 2 : 0);
}

// ------------------------------------------------------------------------------------
// utilities
// ------------------------------------------------------------------------------------
int espb_checksum_u32(const void *buf, uint64_t num_words, uint64_t *sum_dev, void *stream) {
  CU_TRY(launch_checksum(static_cast<const uint32_t *>(buf), num_words,
                         reinterpret_cast<unsigned long long *>(sum_dev), as_stream(stream)),
         "checksum kernel");
  return ESPB_OK;
}

// dsps_add_s16_ansi.c:10-27 / dsps_mulc_s16_ansi.c:18-31 on device buffers.  The reference returns ESP_FAIL for a
// NULL buffer and ESP_OK otherwise (len <= 0 is a no-op there: the loop does not run).
int espb_dsps_add_s16(const int16_t *input1, const int16_t *input2, int16_t *output, int64_t len, int step1,
                      int step2, int step_out, int shift, void *stream) {
  if (!input1 || !input2 || !output)
    return fail(ESPB_ERR_ARG, "dsps_add_s16: NULL buffer (ESP_FAIL in the reference)");
  if (shift < 0 || shift > 31)
    return fail(ESPB_ERR_ARG, "dsps_add_s16: shift must be 0..31 (undefined in the reference otherwise)");
  if (len <= 0)
    return ESPB_OK;
  CU_TRY(launch_add_s16(input1, input2, output, (uint64_t) len, step1, step2, step_out, shift, as_stream(stream)),
         "add_s16 kernel");
  return ESPB_OK;
}

int espb_dsps_mulc_s16(const int16_t *input, int16_t *output, int64_t len, int16_t C, int step_in, int step_out,
                       void *stream) {
  if (!input || !output)
    return fail(ESPB_ERR_ARG, "dsps_mulc_s16: NULL buffer (ESP_FAIL in the reference)");
  if (len <= 0)
    return ESPB_OK;
  CU_TRY(launch_mulc_s16(input, output, (uint64_t) len, C, step_in, step_out, as_stream(stream)), "mulc_s16 kernel");
  return ESPB_OK;
}

int espb_measure_fp32_fma_peak(double *tflops, double *sm_clock_mhz_estimate) {
  if (!tflops)
    return fail(ESPB_ERR_ARG, "measure_fp32_fma_peak: NULL");
  CU_TRY(run_fma_probe(tflops, sm_clock_mhz_estimate, nullptr, nullptr), "fma probe");
  return ESPB_OK;
}

int espb_measure_fp32_tile_pattern(double *tflops) {
  if (!tflops)
    return fail(ESPB_ERR_ARG, "measure_fp32_tile_pattern: NULL");
  CU_TRY(run_tile_probe(tflops), "tile probe");
  return ESPB_OK;
}

int espb_measure_fp32_fma_peak2(double *tflops_scalar_ffma, double *tflops_packed_ffma2) {
  double top = 0.0;
  CU_TRY(run_fma_probe(&top, nullptr, tflops_scalar_ffma, tflops_packed_ffma2), "fma probe");
  return ESPB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// resampler::Resampler, batched
// ------------------------------------------------------------------------------------
struct EspbResampler {
  int num_streams = 0;
  size_t in_samples = 0, out_samples = 0;  // per-stream float scratch sizes (reference ctor arguments)
  EspbResamplerConfiguration cfg{};
  WrapperPolicy policy;
  EspbResampleBatch *art = nullptr;
  EspbBiquadBatch *lowpass = nullptr;
  DevBuf fin, fout, clipped, pcm_in, pcm_out;
  uint32_t *clipped_host = nullptr;  // pinned
  HostPipe pipe;
};

namespace {

struct WrapperCall {
  size_t todo = 0, used = 0, generated = 0;
};

// Steps of Resampler::resample (resampler.cpp:100-160) for stream rows [s0, s0+ns).
int wrapper_run_range(EspbResampler *r, int s0, int ns, const uint8_t *d_in, int64_t in_stride_bytes, uint8_t *d_out,
                      int64_t out_stride_bytes, const WrapperCall &wc, size_t out_free, float gain_db,
                      cudaStream_t stream, bool g_preexpanded) {
  const int ch = r->cfg.channels;
  float *fin = r->fin.as<float>() + (size_t) s0 * r->in_samples;
  float *fout = r->fout.as<float>() + (size_t) s0 * r->out_samples;
  uint32_t *clip = r->clipped.as<uint32_t>() + s0;
  const uint8_t *in = d_in + (size_t) s0 * in_stride_bytes;
  uint8_t *out = d_out + (size_t) s0 * out_stride_bytes;
  CU_TRY(cudaMemsetAsync(clip, 0, ns * sizeof(uint32_t), stream), "clip counters");
  const bool rs = r->policy.resampling;
  if (!rs) {  // :116-119 + :152-153 — bit-depth conversion only
    CU_TRY(launch_q2f(in, in_stride_bytes, fout, (int64_t) r->out_samples, ns, (uint32_t) (wc.todo * ch),
                      r->cfg.source_bits_per_sample, q2f_gain_factor(r->cfg.source_bits_per_sample, gain_db), stream),
           "q2f kernel");
    CU_TRY(launch_f2q(fout, (int64_t) r->out_samples, out, out_stride_bytes, ns, (uint32_t) (wc.generated * ch),
                      r->cfg.target_bits_per_sample, clip, true, stream),
           "f2q kernel");
    return ESPB_OK;
  }
  // :112-153 — quantized_to_float, pre-filter, resampleProcessInterleaved, post-filter, float_to_quantized:
  // the conversions ride on the layout stages of the resampler, fin/fout only hold the tails
  EspbLayout il = {(int64_t) r->in_samples, 1, ch}, ol = {(int64_t) r->out_samples, 1, ch};
  PcmIn pin;
  pin.data = in;
  pin.row_bytes = in_stride_bytes;
  pin.bits = r->cfg.source_bits_per_sample;
  pin.gain_factor = q2f_gain_factor(r->cfg.source_bits_per_sample, gain_db);
  pin.scratch = fin;
  pin.scratch_row = (int64_t) r->in_samples;
  PcmOut pout;
  pout.data = out;
  pout.row_bytes = out_stride_bytes;
  pout.bits = r->cfg.target_bits_per_sample;
  pout.clipped = clip;
  pout.scratch = fout;
  pout.scratch_row = (int64_t) r->out_samples;
  EspbBiquadBatch *lp = r->lowpass;
  StageFilter flt;
  if (lp) {
    flt.params = &lp->params;
    flt.state = lp->state.as<float>() + (size_t) s0 * ch * lp->num_sections * 4;
    flt.sections = lp->num_sections;
    const int rows = (int) (r->policy.pre ? wc.todo : wc.generated);
    flt.block_rows = lp->blocks_for(rows);
    flt.warm_rows = lp->warm_rows;
    if (flt.block_rows > 0) {  // (wrapper_plan sized the record; ranges start on group boundaries)
      const size_t n_blocks = ((size_t) rows + flt.block_rows - 1) / flt.block_rows;
      flt.blk_state = lp->blk_state.as<float>() +
                      (size_t) (s0 * ch / kSeriesPerRow) * n_blocks * lp->num_sections * 2 * kSeriesPerRow * 4;
      flt.mismatches = lp->mismatch_dev.as<unsigned int>();
      flt.chain_broken = lp->chain_broken.as<unsigned int>() + (size_t) (s0 * ch / kSeriesPerRow);
    }
  }
  (void) out_free;
  return run_series_range(r->art, s0 * ch, ns * ch, fin, il, fout, ol, (int) wc.todo, stream, g_preexpanded,
                          r->policy.pre ? &flt : nullptr, r->policy.post ? &flt : nullptr, &pin, &pout);
}

// The host-known part of the call: frames_to_process and the schedule.
int wrapper_plan(EspbResampler *r, size_t avail, size_t out_free, cudaStream_t stream, WrapperCall *wc) {
  const size_t ch = r->cfg.channels;
  if (!r->policy.resampling) {  // :108-110, :116-119 — conversion only
    const size_t todo = out_free < avail ? out_free : avail;
    if (todo * ch > r->out_samples)
      return fail(ESPB_ERR_ARG, "resample: frames exceed the float buffer size given at construction");
    wc->todo = wc->used = wc->generated = todo;
    return ESPB_OK;
  }
  // :104-107 caps the input at resampleGetRequiredSamples(output_frames_free).  Running the state machine
  // once over (all available frames, output_frames_free) stops at exactly that frame — the loop ends with
  // the last output, before it would consume another frame — so frames_to_process == frames_used and the
  // separate dry run is not needed.
  int rc = prepare_call(r->art, (int) avail, (int) out_free, r->policy.sample_ratio, stream);
  if (rc != ESPB_OK)
    return rc;
  wc->used = r->art->sched.used;
  wc->todo = wc->used;
  wc->generated = r->art->sched.generated;
  if (wc->todo * ch > r->in_samples)
    return fail(ESPB_ERR_ARG, "resample: frames exceed the float buffer size given at construction");
  if (wc->generated * ch > r->out_samples)
    return fail(ESPB_ERR_ARG, "resample: output exceeds the float buffer size given at construction");
  // the resampler writes time-major scratch; the post-filter and the PCM packing read it
  const int post_blocks = (r->policy.post && r->lowpass) ? r->lowpass->blocks_for((int) wc->generated) : 0;
  rc = ensure_yt(r->art, (int64_t) wc->generated, post_blocks > 0);
  if (rc != ESPB_OK)
    return rc;
  if (r->lowpass) {
    const int rows = (int) (r->policy.pre ? wc->todo : wc->generated);
    const int blocks = r->lowpass->blocks_for(rows);
    if (blocks > 0)
      if ((rc = biquad_prepare_blocks(r->lowpass, rows, blocks, stream)) != ESPB_OK)
        return rc;
  }
  return ESPB_OK;
}

EspbResamplerResults wrapper_finish(EspbResampler *r, const WrapperCall &wc, uint32_t *clipped_per_stream_host) {
  EspbResamplerResults res{};
  uint64_t total = 0;
  for (int s = 0; s < r->num_streams; ++s)
    total += r->clipped_host[s];
  if (clipped_per_stream_host)
    memcpy(clipped_per_stream_host, r->clipped_host, r->num_streams * sizeof(uint32_t));
  res.frames_used = wc.used;
  res.frames_generated = wc.generated;
  res.predicted_frames_used = wc.todo;
  res.clipped_samples = total;
  if (r->policy.resampling)
    finish_call(r->art);
  g_last_error.clear(), g_last_status = ESPB_OK;
  return res;
}

}  // namespace

extern "C" {

EspbResampler *espb_resampler_create(int num_streams, size_t input_buffer_samples, size_t output_buffer_samples,
                                     const EspbResamplerConfiguration *config) {
  if (!config || num_streams <= 0 || config->channels == 0) {
    fail(ESPB_ERR_ARG, "resampler_create: bad arguments");
    return nullptr;
  }
  if (espb_device_count() <= 0) {
    fail(ESPB_ERR_CUDA, "resampler_create: no CUDA device (this library has no CPU path)");
    return nullptr;
  }
  EspbResampler *r = new EspbResampler();
  r->num_streams = num_streams;
  r->cfg = *config;
  // round the per-stream scratch rows up to 4 floats so rows stay 16-byte aligned
  r->in_samples = (input_buffer_samples + 3) & ~(size_t) 3;
  r->out_samples = (output_buffer_samples + 3) & ~(size_t) 3;
  decide_policy(config->source_sample_rate, config->target_sample_rate, config->number_of_taps,
                config->use_pre_or_post_filter != 0, config->subsample_interpolate != 0, &r->policy);
  cudaError_t e = r->fin.reserve((r->in_samples ? r->in_samples : 4) * num_streams * sizeof(float));
  if (e == cudaSuccess)
    e = r->fout.reserve((r->out_samples ? r->out_samples : 4) * num_streams * sizeof(float));
  if (e == cudaSuccess)
    e = r->clipped.reserve(num_streams * sizeof(uint32_t));
  if (e == cudaSuccess)
    e = cudaMallocHost(&r->clipped_host, num_streams * sizeof(uint32_t));
  if (e != cudaSuccess) {
    cuda_fail(e, "resampler_create: device allocation");
    espb_resampler_free(r);
    return nullptr;
  }
  if (r->policy.resampling) {
    r->art = espb_resampleInit(num_streams, config->channels, config->number_of_taps, config->number_of_filters,
                               r->policy.art_lowpass, r->policy.art_flags);
    if (!r->art) {
      espb_resampler_free(r);
      return nullptr;
    }
    espb_resampleAdvancePosition(r->art, config->number_of_taps / 2.0f);  // resampler.cpp:94
    if (r->policy.pre || r->policy.post) {
      r->lowpass = espb_biquad_init(num_streams * config->channels, 2,
                                    reinterpret_cast<const EspbBiquadCoefficients *>(&r->policy.coeffs), 1.0f);
      if (!r->lowpass) {
        espb_resampler_free(r);
        return nullptr;
      }
    }
  }
  return r;
}

void espb_resampler_free(EspbResampler *r) {
  if (!r)
    return;
  if (r->art)
    espb_resampleFree(r->art);
  if (r->lowpass)
    espb_biquad_free(r->lowpass);
  r->fin.release();
  r->fout.release();
  r->clipped.release();
  r->pcm_in.release();
  r->pcm_out.release();
  if (r->clipped_host)
    cudaFreeHost(r->clipped_host);
  r->pipe.destroy();
  delete r;
}

int espb_resampler_set_mode(EspbResampler *r, int mode) {
  if (!r)
    return fail(ESPB_ERR_ARG, "resampler_set_mode: NULL");
  return r->art ? espb_resampleSetMode(r->art, mode) : ESPB_OK;
}

int espb_resampler_set_option(EspbResampler *r, int option, int value) {
  if (!r)
    return fail(ESPB_ERR_ARG, "resampler_set_option: NULL");
  return r->art ? espb_resampleSetOption(r->art, option, value) : ESPB_OK;
}

int espb_resampler_get_kernel_time(EspbResampler *r, float *total_ms, int *launches) {
  if (!r || !total_ms)
    return fail(ESPB_ERR_ARG, "resampler_get_kernel_time: NULL");
  if (!r->art) {
    *total_ms = 0.0f;
    if (launches)
      *launches = 0;
    return ESPB_OK;
  }
  return espb_resampleGetKernelTime(r->art, total_ms, launches);
}

int espb_resampler_set_biquad_time_blocks(EspbResampler *r, int block_rows, int warmup_rows) {
  if (!r)
    return fail(ESPB_ERR_ARG, "resampler_set_biquad_time_blocks: NULL");
  return r->lowpass ? espb_biquad_set_time_blocks(r->lowpass, block_rows, warmup_rows) : ESPB_OK;
}

int espb_resampler_policy(EspbResampler *r, EspbBiquadCoefficients *coeffs, float *sample_ratio, float *art_lowpass,
                          int *art_flags) {
  if (coeffs)
    memcpy(coeffs, &r->policy.coeffs, sizeof(EspbBiquadCoefficients));
  if (sample_ratio)
    *sample_ratio = r->policy.sample_ratio;
  if (art_lowpass)
    *art_lowpass = r->policy.art_lowpass;
  if (art_flags)
    *art_flags = r->art ? r->art->geo.flags : 0;
  return r->policy.pre ? 1 : (r->policy.post ? 2 : 0);
}

EspbResamplerResults espb_resampler_resample(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                             uint8_t *out, int64_t out_stride_bytes, size_t input_frames_available,
                                             size_t output_frames_free, float gain_db,
                                             uint32_t *clipped_per_stream_host, void *stream) {
  EspbResamplerResults none{};
  if (!r) {
    fail(ESPB_ERR_ARG, "resample: NULL");
    return none;
  }
  cudaStream_t s = as_stream(stream);
  WrapperCall wc;
  if (wrapper_plan(r, input_frames_available, output_frames_free, s, &wc) != ESPB_OK)
    return none;
  if (wrapper_run_range(r, 0, r->num_streams, in, in_stride_bytes, out, out_stride_bytes, wc, output_frames_free,
                        gain_db, s, false) != ESPB_OK)
    return none;
  if (r->lowpass && r->lowpass->mismatch_dev.p && biquad_finish_blocks(r->lowpass, s) != ESPB_OK)
    return none;
  cudaError_t e = cudaMemcpyAsync(r->clipped_host, r->clipped.p, r->num_streams * sizeof(uint32_t),
                                  cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess)
    e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    cuda_fail(e, "resample: sync");
    return none;
  }
  return wrapper_finish(r, wc, clipped_per_stream_host);
}

// The same call without the synchronisation: everything is enqueued on `stream` and the frame counts (known from the
// schedule) are returned at once, so the host can plan the next call while the device works on this one.  The clip
// counts of the call stay on the device (espb_resampler_clipped_dev) until the next call on this handle.
EspbResamplerResults espb_resampler_resample_async(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                                   uint8_t *out, int64_t out_stride_bytes,
                                                   size_t input_frames_available, size_t output_frames_free,
                                                   float gain_db, void *stream) {
  EspbResamplerResults none{};
  if (!r) {
    fail(ESPB_ERR_ARG, "resample_async: NULL");
    return none;
  }
  cudaStream_t s = as_stream(stream);
  WrapperCall wc;
  if (wrapper_plan(r, input_frames_available, output_frames_free, s, &wc) != ESPB_OK)
    return none;
  if (wrapper_run_range(r, 0, r->num_streams, in, in_stride_bytes, out, out_stride_bytes, wc, output_frames_free,
                        gain_db, s, false) != ESPB_OK)
    return none;
  if (r->lowpass && r->lowpass->mismatch_dev.p && biquad_finish_blocks(r->lowpass, s) != ESPB_OK)
    return none;
  memset(r->clipped_host, 0, r->num_streams * sizeof(uint32_t));
  return wrapper_finish(r, wc, nullptr);  // clipped_samples = 0: not known yet
}

int espb_resampler_biquad_block_stats(EspbResampler *r, uint64_t *repaired_blocks, int *warmup_rows) {
  if (!r)
    return fail(ESPB_ERR_ARG, "resampler_biquad_block_stats: NULL");
  if (!r->lowpass) {
    if (repaired_blocks)
      *repaired_blocks = 0;
    if (warmup_rows)
      *warmup_rows = 0;
    return ESPB_OK;
  }
  return espb_biquad_block_stats(r->lowpass, repaired_blocks, warmup_rows);
}

const uint32_t *espb_resampler_clipped_dev(EspbResampler *r) { return r ? r->clipped.as<uint32_t>() : nullptr; }

EspbResamplerResults espb_resampler_resample_host(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                                  uint8_t *out, int64_t out_stride_bytes,
                                                  size_t input_frames_available, size_t output_frames_free,
                                                  float gain_db, uint32_t *clipped_per_stream_host) {
  EspbResamplerResults none{};
  if (!r) {
    fail(ESPB_ERR_ARG, "resample_host: NULL");
    return none;
  }
  cudaError_t e = r->pipe.init();
  if (e != cudaSuccess) {
    cuda_fail(e, "host pipeline streams");
    return none;
  }
  cudaStream_t s0 = r->pipe.s[0];
  WrapperCall wc;
  if (wrapper_plan(r, input_frames_available, output_frames_free, s0, &wc) != ESPB_OK)
    return none;
  const int ch = r->cfg.channels;
  const size_t in_bytes = wc.todo * ch * ((r->cfg.source_bits_per_sample + 7) / 8);
  const size_t out_bytes = wc.generated * ch * ((r->cfg.target_bits_per_sample + 7) / 8);
  const size_t in_pitch = (in_bytes + 15) & ~(size_t) 15, out_pitch = (out_bytes + 15) & ~(size_t) 15;
  if (r->pcm_in.reserve((in_pitch ? in_pitch : 16) * r->num_streams) != cudaSuccess ||
      r->pcm_out.reserve((out_pitch ? out_pitch : 16) * r->num_streams) != cudaSuccess) {
    fail(ESPB_ERR_NOMEM, "resample_host: device staging");
    return none;
  }
  bool single_slab_g = true;
  if (r->policy.resampling && wc.generated > 0) {
    single_slab_g = passes_per_slab(r->art) >= r->art->plan.n_passes();
    if (single_slab_g && !r->art->fs_call && ensure_g(r->art, 0, (int) r->art->plan.chunks.size(), s0) != ESPB_OK)
      return none;
  }
  cudaEventRecord(r->pipe.ready, s0);
  const int per = pick_slab_streams(r->num_streams, r->cfg.channels);
  int slab = 0;
  for (int st0 = 0; st0 < r->num_streams; st0 += per, ++slab) {
    const int ns = st0 + per <= r->num_streams ? per : r->num_streams - st0;
    cudaStream_t s = single_slab_g ? r->pipe.s[slab % HostPipe::kStreams] : s0;
    cudaStreamWaitEvent(s, r->pipe.ready, 0);
    if (in_bytes) {
      e = copy_rows_async(r->pcm_in.as<uint8_t>() + (size_t) st0 * in_pitch, in_pitch,
                          in + (size_t) st0 * in_stride_bytes, (size_t) in_stride_bytes, in_bytes, ns,
                          cudaMemcpyHostToDevice, s);
      if (e != cudaSuccess) {
        cuda_fail(e, "h2d");
        r->pipe.drain();
        return none;
      }
    }
    // the range helper offsets rows by s0 itself: pass the bases
    if (wrapper_run_range(r, st0, ns, r->pcm_in.as<uint8_t>(), (int64_t) in_pitch, r->pcm_out.as<uint8_t>(),
                          (int64_t) out_pitch, wc, output_frames_free, gain_db, s, single_slab_g) != ESPB_OK) {
      r->pipe.drain();
      return none;
    }
    if (out_bytes) {
      e = copy_rows_async(out + (size_t) st0 * out_stride_bytes, (size_t) out_stride_bytes,
                          r->pcm_out.as<uint8_t>() + (size_t) st0 * out_pitch, out_pitch, out_bytes, ns,
                          cudaMemcpyDeviceToHost, s);
      if (e != cudaSuccess) {
        cuda_fail(e, "d2h");
        r->pipe.drain();
        return none;
      }
    }
    e = cudaMemcpyAsync(r->clipped_host + st0, r->clipped.as<uint32_t>() + st0, ns * sizeof(uint32_t),
                        cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) {
      cuda_fail(e, "d2h clip counts");
      r->pipe.drain();
      return none;
    }
  }
  for (int i = 0; i < HostPipe::kStreams; ++i) {
    e = cudaStreamSynchronize(r->pipe.s[i]);
    if (e != cudaSuccess) {
      cuda_fail(e, "host pipeline sync");
      return none;
    }
  }
  if (r->lowpass && r->lowpass->mismatch_dev.p && biquad_finish_blocks(r->lowpass, s0) != ESPB_OK)
    return none;
  return wrapper_finish(r, wc, clipped_per_stream_host);
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// internal.hpp
// ------------------------------------------------------------------------------------
namespace espb {

EspbResampleBatch *new_state_only_context(int num_streams, int channels, const ArtGeometry &geo, float lowpass) {
  EspbResampleBatch *c = new EspbResampleBatch();
  c->state_only = true;
  cudaGetDevice(&c->device);
  c->num_streams = num_streams;
  c->channels = channels;
  c->geo = geo;
  c->lowpass = lowpass;
  c->state = initial_state(geo.taps);
  return c;
}
ArtState context_state(const EspbResampleBatch *c) { return c->state; }
void set_context_state(EspbResampleBatch *c, ArtState st) { c->state = st; }
int context_mode(const EspbResampleBatch *c) { return c->mode; }
void set_context_mode(EspbResampleBatch *c, int mode) { c->mode = mode; }
int api_fail(int code, const char *what, const char *detail) { return fail(code, what, detail); }
void api_ok() { g_last_error.clear(), g_last_status = ESPB_OK; }

}  // namespace espb
