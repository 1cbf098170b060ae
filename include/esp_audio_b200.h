/* esp_audio_b200.h — C ABI of the B200-native ART resampler path.
 *
 * Drop-in boundary for ONE hot path of esp-audio-libs (reference paths are relative
 * to the reference tree): the ART polyphase sinc resampler, the art_biquad low-pass
 * and the quantization_utils PCM conversion, batched over independent streams and
 * executed by hand-written sm_100a kernels.  Plain pointers and sizes only; every
 * processing call takes a CUDA stream (as void*, a cudaStream_t; NULL = default
 * stream) and is asynchronous with respect to the host unless stated otherwise.
 *
 * There is no CPU fallback: every entry point that computes needs a B200-class
 * device and fails loudly (ESPB_ERR_CUDA / NULL + message in espb_last_error())
 * when none is usable.
 *
 * Batch semantics.  A batch context stands for `num_streams` independent reference
 * contexts created with identical parameters.  All streams of a batch advance in
 * lock-step (same frames in, same output capacity, same ratio per call), so the
 * position schedule — which in the reference is a signal-independent FP32
 * accumulator — is computed once per call on the host, bit-for-bit as the
 * reference's state machine does, and shared by every stream.
 *
 * Buffer addressing (device memory).  A sample of (stream s, channel c, frame n) lives
 * at   base + s*stream_stride + c*channel_stride + n*frame_stride   (units: floats).
 *   interleaved (resampleProcessInterleaved): channel_stride = 1, frame_stride = channels
 *   planar      (resampleProcess)           : channel_stride = frames per plane, frame_stride = 1
 */
#ifndef ESP_AUDIO_B200_H_
#define ESP_AUDIO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ESPB_ABI_VERSION 2

/* flags — same bits as include/art_resampler.h:21-23 */
#define ESPB_SUBSAMPLE_INTERPOLATE 0x1
#define ESPB_BLACKMAN_HARRIS 0x2
#define ESPB_INCLUDE_LOWPASS 0x4

/* error codes (the reference only has NULL / false; these add the CUDA side) */
#define ESPB_OK 0
#define ESPB_ERR_ARG (-1)
#define ESPB_ERR_CUDA (-2)
#define ESPB_ERR_NOMEM (-3)
#define ESPB_ERR_STATE (-4)

/* arithmetic mode of the resampler dot products */
#define ESPB_MODE_FAST 0  /* tap-order FFMA chain: <= 1e-6 max-abs of the reference            */
#define ESPB_MODE_EXACT 1 /* tap-order FMUL+FADD (no contraction): bit-exact with the reference */

const char *espb_last_error(void); /* thread-local message of the last failing call */
/* Status of the calling thread's last processing call: ESPB_OK, or the ESPB_ERR_* code of its failure.  The
 * processing calls keep the reference's return types ({input_used, output_generated} / ResamplerResults), in which a
 * failed call and a legitimately empty call both read {0, 0}; this tells them apart. */
int espb_last_status(void);
int espb_abi_version(void);

/* ---- device + buffers (the "device-buffer interface") ------------------------ */
int espb_device_count(void);
int espb_set_device(int device);
int espb_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem, char *name, int name_len);
void *espb_malloc(size_t bytes);           /* device memory, NULL on failure (like alloc_psram_fallback) */
void espb_free(void *dptr);
void *espb_malloc_host(size_t bytes);      /* pinned host memory */
void espb_free_host(void *hptr);
int espb_memcpy_h2d(void *dst, const void *src, size_t bytes, void *stream);
int espb_memcpy_d2h(void *dst, const void *src, size_t bytes, void *stream);
int espb_memset(void *dst, int value, size_t bytes, void *stream);
void *espb_stream_create(void);
void espb_stream_destroy(void *stream);
int espb_stream_sync(void *stream);
int espb_device_sync(void);
/* CUDA-event timing on the launching stream */
void *espb_event_create(void);
void espb_event_destroy(void *ev);
int espb_event_record(void *ev, void *stream);
int espb_event_elapsed_ms(void *start, void *stop, float *ms); /* synchronises on `stop` */
/* number of kernels this library has launched so far (process-wide) */
uint64_t espb_launch_count(void);

/* ---- ART resampler, batched: replaces include/art_resampler.h:35-45 ------------- */
typedef struct EspbResampleBatch EspbResampleBatch;

typedef struct { /* include/art_resampler.h:31-33 */
  unsigned int input_used, output_generated;
} EspbResampleResult;

typedef struct {
  int64_t stream_stride, channel_stride, frame_stride; /* in floats */
} EspbLayout;

/* resampleInit (art_resampler.cpp:78-139) for num_streams identical contexts.  Same
 * validation and the same stderr lines; NULL on invalid taps/filters or failed alloc. */
EspbResampleBatch *espb_resampleInit(int num_streams, int numChannels, int numTaps, int numFilters,
                                     float lowpassRatio, int flags);
void espb_resampleFree(EspbResampleBatch *cxt);                        /* art_resampler.cpp:353-366 */
int espb_resampleReset(EspbResampleBatch *cxt, void *stream);          /* :144-152 */
void espb_resampleAdvancePosition(EspbResampleBatch *cxt, float delta); /* :313-318 */
float espb_resampleGetPosition(EspbResampleBatch *cxt);                /* :348 */
unsigned int espb_resampleGetRequiredSamples(EspbResampleBatch *cxt, int numOutputFrames, float ratio); /* :257-279 */
unsigned int espb_resampleGetExpectedOutput(EspbResampleBatch *cxt, int numInputFrames, float ratio);   /* :281-306 */
int espb_resampleSetMode(EspbResampleBatch *cxt, int mode);            /* ESPB_MODE_FAST (default) / _EXACT */
/* options: plan cache (default on: a call that repeats the previous call's state, frame counts
 * and ratio reuses its schedule and expanded coefficients), per-launch CUDA-event timing of the
 * resampler kernel (read with espb_resampleGetKernelTime) */
#define ESPB_OPT_PLAN_CACHE 1
#define ESPB_OPT_KERNEL_TIMING 2
/* staging overlap (default on): long device-buffer calls launch the resampler kernel as a programmatic dependent of
 * the transposing stage, so the HBM-bound staging hides behind the FMA-bound kernel; results are identical either
 * way.  Kernel timing switches it off for the calls it measures (the events must bracket the kernel alone). */
#define ESPB_OPT_OVERLAP_STAGING 3
int espb_resampleSetOption(EspbResampleBatch *cxt, int option, int value);
/* sum of the resampler-kernel durations recorded since the last query, and their count */
int espb_resampleGetKernelTime(EspbResampleBatch *cxt, float *total_ms, int *launches);
/* context introspection (tests): effective flags, state, the host-built filter bank */
int espb_resampleGetFlags(EspbResampleBatch *cxt);
void espb_resampleGetState(EspbResampleBatch *cxt, float *outputOffset, int *inputIndex);
int espb_resampleCopyFilters(EspbResampleBatch *cxt, float *host_dst /* (numFilters+1)*numTaps */);

/* resampleProcessInterleaved (art_resampler.cpp:208-243): every stream consumes up to
 * numInputFrames and emits up to numOutputFrames; `in`/`out` are device pointers, rows
 * `*_stream_stride` floats apart.  The result is the same for every stream. */
EspbResampleResult espb_resampleProcessInterleaved(EspbResampleBatch *cxt, const float *in, int64_t in_stream_stride,
                                                   int numInputFrames, float *out, int64_t out_stream_stride,
                                                   int numOutputFrames, float ratio, void *stream);
/* resampleProcess (art_resampler.cpp:167-202): planar — channel planes `*_channel_stride` floats apart. */
EspbResampleResult espb_resampleProcess(EspbResampleBatch *cxt, const float *in, int64_t in_stream_stride,
                                        int64_t in_channel_stride, int numInputFrames, float *out,
                                        int64_t out_stream_stride, int64_t out_channel_stride, int numOutputFrames,
                                        float ratio, void *stream);
/* resampleProcess with the reference's own argument form (`const float *const *inputs`, `float *const *outputs`,
 * include/art_resampler.h:36-37): one pointer per plane.  `inputs` / `outputs` are HOST arrays of
 * num_streams * numChannels DEVICE pointers (plane q = stream q / numChannels, channel q % numChannels); the planes
 * may be separately allocated buffers. */
EspbResampleResult espb_resampleProcessPlanes(EspbResampleBatch *cxt, const float *const *inputs, int numInputFrames,
                                              float *const *outputs, int numOutputFrames, float ratio, void *stream);
/* general form */
EspbResampleResult espb_resampleProcessLayout(EspbResampleBatch *cxt, const float *in, const EspbLayout *in_layout,
                                              int numInputFrames, float *out, const EspbLayout *out_layout,
                                              int numOutputFrames, float ratio, void *stream);

/* resampleProcessInterleaved with HOST buffers (pinned memory gives full PCIe speed):
 * stream slabs are copied in, resampled and copied out on three internal CUDA streams so
 * that H2D, compute and D2H of neighbouring slabs overlap.  Synchronous. */
EspbResampleResult espb_resampleProcessInterleavedHost(EspbResampleBatch *cxt, const float *in,
                                                       int64_t in_stream_stride, int numInputFrames, float *out,
                                                       int64_t out_stream_stride, int numOutputFrames, float ratio);

/* ---- ratio groups: per-stream / time-varying ratios (ASRC) ------------------------------
 * The reference takes `ratio` per call and per context (art_resampler.cpp:57-62), so streams may drift apart.
 * Streams that share a clock (same ratio trajectory and chunking) form a group; a group set is one batch
 * context per group, processed concurrently on internal CUDA streams forked from and joined to the caller's
 * stream.  Group k's streams are rows [first_k, first_k + streams_per_group[k]) of the buffers, first_k being
 * the running sum.  Each group keeps its own device-side history and position between calls. */
typedef struct EspbResampleGroups EspbResampleGroups;
EspbResampleGroups *espb_resampleGroupsInit(int num_groups, const int *streams_per_group, int numChannels, int numTaps,
                                            int numFilters, float lowpassRatio, int flags);
void espb_resampleGroupsFree(EspbResampleGroups *g);
int espb_resampleGroupsCount(const EspbResampleGroups *g);
/* 1 when the set runs in the fused form: every group the same number of streams and <= 32 series ("one clock per
 * stream" and the like).  One compact staging buffer, schedule table and filter bank serve all groups, and a call is
 * four device operations whatever the number of groups (upload, staging, schedule expansion, one resampler launch with
 * a grid dimension over the groups).  espb_resampleGroupsContext then returns state-only contexts: the position calls
 * (advance / position / state / required / expected) work per group, processing goes through the set.
 * ESPB_GROUPS_FUSED=0 forces one full context per group. */
int espb_resampleGroupsIsFused(const EspbResampleGroups *g);
/* resampleReset (art_resampler.cpp:144-152) for one group */
int espb_resampleGroupsReset(EspbResampleGroups *g, int group, void *stream);
int espb_resampleGroupsFirstStream(const EspbResampleGroups *g, int group);
/* the group's batch context, for resampleAdvancePosition / Reset / GetPosition / GetRequiredSamples / ... */
EspbResampleBatch *espb_resampleGroupsContext(EspbResampleGroups *g, int group);
int espb_resampleGroupsSetMode(EspbResampleGroups *g, int mode);
/* resampleProcessInterleaved for every group with its own frame counts and ratio (arrays of num_groups
 * entries); results[k] is group k's {input_used, output_generated}.  Asynchronous on `stream`. */
int espb_resampleGroupsProcessInterleaved(EspbResampleGroups *g, const float *in, int64_t in_stream_stride,
                                          const int *numInputFrames, float *out, int64_t out_stream_stride,
                                          const int *numOutputFrames, const float *ratios, EspbResampleResult *results,
                                          void *stream);

/* ---- art_biquad: replaces include/art_biquad.h:19-36 --------------------------- */
typedef struct { /* include/art_biquad.h:19-21 */
  float a0, a1, a2, b1, b2;
} EspbBiquadCoefficients;

void espb_biquad_lowpass(EspbBiquadCoefficients *filter, double frequency);  /* art_biquad.cpp:16-25 (host) */
void espb_biquad_highpass(EspbBiquadCoefficients *filter, double frequency); /* art_biquad.cpp:29-38 (host) */

/* A bank of `num_series` Biquad states (art_biquad.h:23-28) x `num_sections` cascaded
 * sections, all sharing one coefficient set; delays live in device memory. */
typedef struct EspbBiquadBatch EspbBiquadBatch;
EspbBiquadBatch *espb_biquad_init(int num_series, int num_sections, const EspbBiquadCoefficients *coeffs,
                                  float gain);                                  /* art_biquad.cpp:43-51 */
void espb_biquad_free(EspbBiquadBatch *f);
int espb_biquad_reset(EspbBiquadBatch *f, void *stream);
/* biquad_apply_buffer (art_biquad.cpp:73-93) for every series: in place, sequential in
 * time, un-fused FP32 in the reference's order (bit-exact).  Series q of the bank is
 * (stream q / channels, channel q % channels) of the layout. */
int espb_biquad_apply_buffer(EspbBiquadBatch *f, float *buf, const EspbLayout *layout, int channels, int num_samples,
                             void *stream);
/* biquad_apply_sample (art_biquad.cpp:55-69), batched: one new sample per series (samples[q], device memory, filtered
 * in place); every series' delays advance by one step.  A latency-bound call — use apply_buffer for throughput. */
int espb_biquad_apply_samples(EspbBiquadBatch *f, float *samples, void *stream);
/* Long single streams (the north star's "block-parallel state carry"): time blocks of `block_rows` frames are
 * filtered in parallel, each after re-running the recurrence over the `warmup_rows` frames before it from a zero
 * state.  The hand-over between blocks is VERIFIED on the device — block k's state at its first frame must equal
 * block k-1's end state bit for bit (equal state + equal input = equal continuation) — and a block whose warm-up
 * did not converge is filtered again from the true state, so the output is the sequential one of
 * art_biquad.cpp:73-93 by construction; a failed merge costs time, never bits (and doubles the warm-up of later
 * calls).  block_rows: -1 = automatic (the default: blocks of 8192 frames when the bank has <= 4096 series and the
 * call is >= 16384 frames long), 0 = one sequential run per series, > 0 = that many frames (multiple of 32).
 * warmup_rows: multiple of 32 (default 1024; 0 keeps the current value in automatic mode). */
int espb_biquad_set_time_blocks(EspbBiquadBatch *f, int block_rows, int warmup_rows);
/* blocks repaired so far (0: every warm-up merged) and the current warm-up length; synchronises with the last call */
int espb_biquad_block_stats(EspbBiquadBatch *f, uint64_t *repaired_blocks, int *warmup_rows);
int espb_biquad_get_state(EspbBiquadBatch *f, float *host_dst /* num_series*num_sections*4: in_d1,in_d2,out_d1,out_d2 */);

/* ---- quantization_utils: replaces include/quantization_utils.h:15-25 ------------ */
/* quantized_to_float (quantization_utils.cpp:6-48) on device buffers. */
int espb_quantized_to_float(const uint8_t *in, float *out, uint64_t num_samples, uint8_t input_bits, float gain_db,
                            void *stream);
/* float_to_quantized (quantization_utils.cpp:50-94).  The clipped-sample count is
 * accumulated into *clipped_dev (a device uint32 the caller zeroes), so the call stays
 * asynchronous; espb_float_to_quantized_sync returns it like the reference does. */
int espb_float_to_quantized(const float *in, uint8_t *out, uint64_t num_samples, uint8_t output_bits,
                            uint32_t *clipped_dev, void *stream);
uint32_t espb_float_to_quantized_sync(const float *in, uint8_t *out, uint64_t num_samples, uint8_t output_bits,
                                      void *stream);
/* row-wise variants for batches whose rows are padded: `rows` rows of `row_samples`
 * samples, strides in bytes (input) / floats (output) and vice versa; per-row clip counts. */
int espb_quantized_to_float_rows(const uint8_t *in, int64_t in_row_stride_bytes, float *out,
                                 int64_t out_row_stride_floats, int rows, uint32_t row_samples, uint8_t input_bits,
                                 float gain_db, void *stream);
int espb_float_to_quantized_rows(const float *in, int64_t in_row_stride_floats, uint8_t *out,
                                 int64_t out_row_stride_bytes, int rows, uint32_t row_samples, uint8_t output_bits,
                                 uint32_t *clipped_per_row_dev, void *stream);

/* ---- resampler::Resampler, batched: replaces include/resampler.h:15-80 ------------ */
typedef struct { /* include/resampler.h:22-32 */
  float source_sample_rate;
  float target_sample_rate;
  uint8_t source_bits_per_sample;
  uint8_t target_bits_per_sample;
  uint8_t channels;
  uint8_t use_pre_or_post_filter; /* bool */
  uint8_t subsample_interpolate;  /* bool */
  uint16_t number_of_taps;
  uint16_t number_of_filters;
} EspbResamplerConfiguration;

typedef struct { /* include/resampler.h:15-20; clipped_samples is the batch total */
  size_t frames_used;
  size_t frames_generated;
  size_t predicted_frames_used;
  uint64_t clipped_samples;
} EspbResamplerResults;

typedef struct EspbResampler EspbResampler;
/* Resampler(input_buffer_samples, output_buffer_samples) + initialize(config)
 * (resampler.cpp:21-98), for num_streams streams.  NULL where the reference returns false.
 * Unlike the reference (lowpass_[2][2], include/resampler.h:64) any channel count works. */
EspbResampler *espb_resampler_create(int num_streams, size_t input_buffer_samples, size_t output_buffer_samples,
                                     const EspbResamplerConfiguration *config);
void espb_resampler_free(EspbResampler *r);
int espb_resampler_set_mode(EspbResampler *r, int mode);
/* time-block mode of the pre/post low-pass (see espb_biquad_set_time_blocks) */
int espb_resampler_set_biquad_time_blocks(EspbResampler *r, int block_rows, int warmup_rows);
/* ESPB_OPT_* of the wrapper's ART context; CUDA-event time of its resampler-kernel launches since the last query */
int espb_resampler_set_option(EspbResampler *r, int option, int value);
int espb_resampler_get_kernel_time(EspbResampler *r, float *total_ms, int *launches);
int espb_resampler_biquad_block_stats(EspbResampler *r, uint64_t *repaired_blocks, int *warmup_rows);
/* policy introspection: 0 none / 1 pre / 2 post; coefficients; ART low-pass and flags */
int espb_resampler_policy(EspbResampler *r, EspbBiquadCoefficients *coeffs, float *sample_ratio, float *art_lowpass,
                          int *art_flags);
/* Resampler::resample (resampler.cpp:100-160) on DEVICE buffers: row s of `in` holds
 * stream s's packed PCM (rows in_stride_bytes apart), likewise `out`.  Synchronises the
 * stream before returning (the clip count is part of the result, as in the reference).
 * clipped_per_stream_host may be NULL, else receives num_streams counts. */
EspbResamplerResults espb_resampler_resample(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                             uint8_t *out, int64_t out_stride_bytes, size_t input_frames_available,
                                             size_t output_frames_free, float gain_db,
                                             uint32_t *clipped_per_stream_host, void *stream);
/* Same call without the synchronisation (device buffers): all work is enqueued on `stream` and the frame counts —
 * known from the signal-independent schedule — are returned immediately, so a caller can prepare the next call while
 * the device runs this one.  clipped_samples is 0 in the result; the per-stream clip counts of the call are in device
 * memory (espb_resampler_clipped_dev, num_streams uint32) once `stream` has reached this point, until the next call
 * on the handle overwrites them. */
EspbResamplerResults espb_resampler_resample_async(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                                   uint8_t *out, int64_t out_stride_bytes,
                                                   size_t input_frames_available, size_t output_frames_free,
                                                   float gain_db, void *stream);
const uint32_t *espb_resampler_clipped_dev(EspbResampler *r);
/* Same call with HOST buffers: stages through pinned memory, copies host->device,
 * processes, copies device->host; stream slabs are pipelined over internal CUDA streams. */
EspbResamplerResults espb_resampler_resample_host(EspbResampler *r, const uint8_t *in, int64_t in_stride_bytes,
                                                  uint8_t *out, int64_t out_stride_bytes,
                                                  size_t input_frames_available, size_t output_frames_free,
                                                  float gain_db, uint32_t *clipped_per_stream_host);

/* ---- host-side planning (no device needed) ------------------------------------------ */
/* The signal-independent parts of the path, exposed for callers that want to size
 * buffers ahead of time and for CPU-only verification of the host logic.
 * espb_plan_filter_bank: the (numFilters+1) x numTaps bank of init_filter
 * (art_resampler.cpp:379-419) after resampleInit's flag normalisation (:82-87). */
int espb_plan_filter_bank(int numTaps, int numFilters, float lowpassRatio, int flags, float *host_dst,
                          int *effective_flags);
/* Data-free run of the resampleProcess state machine (art_resampler.cpp:172-199) from an
 * explicit (outputOffset, inputIndex): counts, end state and, when the arrays are not
 * NULL (numOutputFrames entries each), per output the window start relative to the first
 * input frame of the call, the filter phase, the blend weight and the kind
 * (1 pass-through, 2 single dot product, 3 blend). */
int espb_plan_schedule(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex,
                       int numInputFrames, int numOutputFrames, float ratio, unsigned int *input_used,
                       unsigned int *output_generated, float *end_outputOffset, int *end_inputIndex,
                       int32_t *window_start, int32_t *phase, float *weight, int32_t *kind);
/* The schedule of the same call through the closed-form ("segmented") planner the processing path uses — offsets
 * as exact arithmetic progressions per binade and ring cycle, expanded per output — for checking it against
 * espb_plan_schedule (the reference's sequential state machine).  Returns the number of segments, < 0 on error. */
int espb_plan_schedule_segments(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex,
                                int numInputFrames, int numOutputFrames, float ratio, unsigned int *input_used,
                                unsigned int *output_generated, float *end_outputOffset, int *end_inputIndex,
                                int32_t *window_start, int32_t *phase, float *weight, int32_t *kind);
/* The kernel-side work list of a call: passes of `blocks_per_pass` x 8 outputs, each swept in chunks of `chunk_rows`
 * input rows starting at chunk_start[] (relative to the call's first input frame; negative = carried frames);
 * pass p owns chunks [pass_chunk_begin[p], pass_chunk_begin[p+1]).  Returns the number of chunks
 * (arrays may be NULL or shorter: nothing is written past max_chunks / max_passes entries), < 0 on bad arguments. */
int espb_plan_passes(int numTaps, int numFilters, int flags, float outputOffset, int inputIndex, int numInputFrames,
                     int numOutputFrames, float ratio, int blocks_per_pass, int chunk_rows, int32_t *chunk_start,
                     int32_t *chunk_pass, int max_chunks, int32_t *pass_chunk_begin, int max_passes);
/* Resampler::initialize's decisions (resampler.cpp:38-94) without creating anything:
 * returns 0 none / 1 pre / 2 post filter. */
int espb_plan_policy(const EspbResamplerConfiguration *config, EspbBiquadCoefficients *coeffs, float *sample_ratio,
                     float *art_lowpass, int *art_flags);

/* ---- dsp.h Q15 helpers: replace include/dsp.h:66-93 (portable C versions) ------------- */
/* dsps_add_s16 (src/dsp/dsps_add_s16_ansi.c:10-27): out[i*step_out] = (int16)((in1[i*step1] + in2[i*step2]) >> shift),
 * the sum taken in 32 bits, the shift arithmetic, the result truncated (not saturated) — the mixer step that
 * follows float_to_quantized in ESPHome.  Device buffers; `len` may cover a whole batch (int64).  Returns ESPB_OK, or
 * ESPB_ERR_ARG where the reference returns ESP_FAIL (a NULL buffer). */
int espb_dsps_add_s16(const int16_t *input1, const int16_t *input2, int16_t *output, int64_t len, int step1,
                      int step2, int step_out, int shift, void *stream);
/* dsps_mulc_s16 (src/dsp/dsps_mulc_s16_ansi.c:18-31): out[i*step_out] = (int16)((in[i*step_in] * C) >> 15), Q15 volume. */
int espb_dsps_mulc_s16(const int16_t *input, int16_t *output, int64_t len, int16_t C, int step_in, int step_out,
                       void *stream);

/* ---- WAV header parse / emit: replaces include/wav_decoder.h:32-90 (host only) --------- */
/* WAVDecoderState (include/wav_decoder.h:34-43) and WAVDecoderResult (:45-52), same values */
#define ESPB_WAV_DECODER_BEFORE_RIFF 0
#define ESPB_WAV_DECODER_BEFORE_WAVE 1
#define ESPB_WAV_DECODER_BEFORE_FMT 2
#define ESPB_WAV_DECODER_IN_FMT 3
#define ESPB_WAV_DECODER_BEFORE_DATA 4
#define ESPB_WAV_DECODER_IN_DATA 5
#define ESPB_WAV_DECODER_SUCCESS_NEXT 0
#define ESPB_WAV_DECODER_SUCCESS_IN_DATA 1
#define ESPB_WAV_DECODER_WARNING_INCOMPLETE_DATA 2
#define ESPB_WAV_DECODER_ERROR_NO_RIFF 3
#define ESPB_WAV_DECODER_ERROR_NO_WAVE 4
#define ESPB_WAV_DECODER_ERROR_FAILED 5
typedef struct EspbWavDecoder EspbWavDecoder; /* class WAVDecoder (:54-89) */
EspbWavDecoder *espb_wav_decoder_create(void);
void espb_wav_decoder_free(EspbWavDecoder *d);
/* WAVDecoder::decode_header (src/decode/wav_decoder.cpp:8-46): parse as much of the header as `buffer` holds;
 * returns a result code; bytes_processed() says how far it got. */
int espb_wav_decoder_decode_header(EspbWavDecoder *d, const uint8_t *buffer, size_t bytes_available);
/* WAVDecoder::next (:48-149): one step — the caller skipped bytes_to_skip() and read bytes_needed() bytes */
int espb_wav_decoder_next(EspbWavDecoder *d, const uint8_t *buffer);
void espb_wav_decoder_reset(EspbWavDecoder *d); /* :151-161 (does not restore bytes_needed, like the reference) */
int espb_wav_decoder_state(const EspbWavDecoder *d);
size_t espb_wav_decoder_bytes_processed(const EspbWavDecoder *d);
size_t espb_wav_decoder_bytes_to_skip(const EspbWavDecoder *d);
size_t espb_wav_decoder_bytes_needed(const EspbWavDecoder *d);
const char *espb_wav_decoder_chunk_name(const EspbWavDecoder *d); /* 4 characters + NUL */
size_t espb_wav_decoder_chunk_bytes_left(const EspbWavDecoder *d);
uint32_t espb_wav_decoder_sample_rate(const EspbWavDecoder *d);
uint16_t espb_wav_decoder_num_channels(const EspbWavDecoder *d);
uint16_t espb_wav_decoder_bits_per_sample(const EspbWavDecoder *d);
/* canonical 44-byte PCM header (RIFF/WAVE/fmt /data) for `data_bytes` of samples; returns 44.  The reference
 * only parses; this is the matching emitter for test and bench I/O. */
size_t espb_wav_write_header(uint8_t *dst44, uint32_t sample_rate, uint16_t num_channels, uint16_t bits_per_sample,
                             uint32_t data_bytes);

/* ---- batch utilities -------------------------------------------------------------- */
/* Order-independent checksum of a float/byte buffer: wrapping 64-bit sum of the 32-bit
 * words (bytes for the u8 variant) — what each rank contributes to the NCCL gather. */
int espb_checksum_u32(const void *buf, uint64_t num_words, uint64_t *sum_dev, void *stream);
/* FFMA-only probe: achieved FP32 TFLOP/s of this device right now (roofline denominator). */
int espb_measure_fp32_fma_peak(double *tflops, double *sm_clock_mhz_estimate);
/* the two probes separately: scalar FFMA and packed FFMA2 (fma.rn.f32x2); espb_measure_fp32_fma_peak returns the
 * larger */
int espb_measure_fp32_fma_peak2(double *tflops_scalar_ffma, double *tflops_packed_ffma2);
/* the resampler's inner loop alone (register tile fed from shared memory, the kernel's occupancy, no TMA /
 * barriers / epilogue): the practical ceiling of that loop, reported next to the FMA-only peak */
int espb_measure_fp32_tile_pattern(double *tflops);

/* ---- multi-GPU: stream-sharded batches (SURVEY.md 8e) ------------------------------------------------
 * Streams are independent (the reference has no globals; a context is one stream's state), so a batch is cut into
 * contiguous stream ranges, one per GPU, with NO collective on the data path; NCCL over NVLink only gathers a few
 * 64-bit words per shard (checksum, frame and clip counts).  NCCL is resolved at run time (libnccl.so.2). */
int espb_nccl_version(void);                 /* 0: NCCL not available */
const char *espb_multi_last_error(void);
/* contiguous range [first, first + count) of shard `rank` of `world`: sizes differ by at most one stream */
void espb_shard_range(int64_t n_streams, int rank, int world, int64_t *first, int64_t *count);

/* Host-link probe: plain pinned cudaMemcpyAsync, one call per slab, on the listed devices concurrently (n_devices <= 0:
 * the current device).  out[6] = aggregate GB/s per direction {H2D alone, D2H alone, H2D while D2H runs, D2H while
 * H2D runs, both directions summed, seconds of the duplex run}: the ceiling of the host-buffer entry points. */
int espb_measure_host_link(int n_devices, const int *devices, size_t bytes, size_t slab_bytes, int reps, double *out);
/* one pattern (0: H2D alone, 1: D2H alone, 2: both at once) on the current device, GB/s per direction: lets one process
 * per GPU run the same pattern at the same time, with a barrier of the caller's between patterns */
int espb_measure_host_link_pattern(int pattern, size_t bytes, size_t slab_bytes, int reps, double *gbs);
/* prepared form: buffers page-locked once (that takes a process-dependent second), then single timed runs that the
 * caller can start on a barrier of its own — so that one process per GPU measures the link while all others copy */
typedef struct EspbLinkProbe EspbLinkProbe;
EspbLinkProbe *espb_link_probe_create(size_t bytes, size_t slab_bytes);
int espb_link_probe_run(EspbLinkProbe *p, int pattern, double *gbs, double *seconds);
void espb_link_probe_free(EspbLinkProbe *p);

/* one process drives all devices: ncclCommInitAll over `devices` (NULL: 0 .. n_devices-1; n_devices <= 0: all) */
typedef struct EspbMulti EspbMulti;
EspbMulti *espb_multi_create(int n_devices, const int *devices);
void espb_multi_free(EspbMulti *m);
int espb_multi_size(const EspbMulti *m);
int espb_multi_device(const EspbMulti *m, int rank);
/* device k contributes `words` uint64 at send_dev[k], receives world*words (rank order) at recv_dev[k]; one
 * ncclAllGather per device in one group call, on streams[k] (NULL: internal streams).  Asynchronous. */
int espb_multi_allgather_u64(EspbMulti *m, const void *const *send_dev, void *const *recv_dev, int words,
                             void *const *streams);
/* host convenience (synchronous): words_per_rank[k*words + i] -> gathered[world*words] as device 0 received them */
int espb_multi_gather_words(EspbMulti *m, const uint64_t *words_per_rank, int words, uint64_t *gathered);

/* one process per GPU: rank 0 makes the 128-byte id, the launcher's rendezvous hands it to every rank, every rank
 * joins with its current CUDA device */
typedef struct EspbDist EspbDist;
int espb_dist_unique_id(void *id128);
EspbDist *espb_dist_init(const void *id128, int rank, int world);
void espb_dist_free(EspbDist *d);
int espb_dist_rank(const EspbDist *d);
int espb_dist_world(const EspbDist *d);
int espb_dist_allgather_u64(EspbDist *d, const uint64_t *mine, int words, uint64_t *gathered /* world*words */);
int espb_dist_barrier(EspbDist *d);

#ifdef __cplusplus
}
#endif
#endif /* ESP_AUDIO_B200_H_ */
