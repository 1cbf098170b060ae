/* TEST INFRASTRUCTURE — CPU oracle for the B200 resampler path.
 *
 * Plain-C restatement of the esp-audio-libs hot path (ART polyphase sinc
 * resampler, art_biquad, quantization_utils, and the Resampler wrapper's
 * pipeline policy).  It exists ONLY as the checker for tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline leg.  The product
 * (esp-audio-libs_b200/) never includes, links or loads it.
 *
 * Parity pinning: the reference ships no tests or golden vectors for this path
 * (SURVEY.md §4), so the oracle is pinned against the UNMODIFIED reference
 * compiled here (oracle/_ref, see oracle/Makefile) — directly in
 * tests/test_oracle_vs_reference.py when oracle/_ref is present, and through
 * the committed fixtures under tests/golden/ (made by oracle/gen_golden.py from
 * oracle/_ref) everywhere else.
 *
 * Must be compiled with -ffp-contract=off (the reference arithmetic is un-fused; the one fused form,
 * orc_resample_set_fused, calls fmaf explicitly).
 */
#ifndef ART_ORACLE_H_
#define ART_ORACLE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* reference include/art_resampler.h:21-23 */
#define ORC_SUBSAMPLE_INTERPOLATE 0x1
#define ORC_BLACKMAN_HARRIS 0x2
#define ORC_INCLUDE_LOWPASS 0x4

typedef struct OrcResampler OrcResampler;

/* include/art_resampler.h:35-45 */
OrcResampler *orc_resample_init(int channels, int taps, int filters, float lowpass_ratio, int flags);
void orc_resample_free(OrcResampler *r);
void orc_resample_reset(OrcResampler *r);
void orc_resample_advance(OrcResampler *r, float delta);
float orc_resample_position(const OrcResampler *r);
unsigned orc_resample_required(const OrcResampler *r, int n_out, float ratio);
unsigned orc_resample_expected(const OrcResampler *r, int n_in, float ratio);
void orc_resample_interleaved(OrcResampler *r, const float *in, int n_in, float *out, int n_out, float ratio,
                              unsigned *used, unsigned *generated);
void orc_resample_planar(OrcResampler *r, const float *const *in, int n_in, float *const *out, int n_out,
                         float ratio, unsigned *used, unsigned *generated);
/* introspection for tests */
int orc_resample_flags(const OrcResampler *r);
void orc_resample_copy_filter(const OrcResampler *r, int idx, float *dst);
void orc_resample_state(const OrcResampler *r, float *output_offset, int *input_index);
/* Not in the reference.  Non-zero: every dot product is an fmaf chain in tap order (one rounding per multiply-add),
 * the library's fast mode (DESIGN.md §2.2); everything else is unchanged.  Per context, off by default. */
void orc_resample_set_fused(OrcResampler *r, int fused);

/* include/art_biquad.h:19-36 */
typedef struct {
  float a0, a1, a2, b1, b2;
} OrcBiquadCoeffs;
typedef struct {
  OrcBiquadCoeffs c;
  float in_d1, in_d2, out_d1, out_d2;
  int first_order;
} OrcBiquad;
void orc_biquad_lowpass(OrcBiquadCoeffs *c, double frequency);
void orc_biquad_highpass(OrcBiquadCoeffs *c, double frequency);
void orc_biquad_init(OrcBiquad *f, const OrcBiquadCoeffs *c, float gain);
void orc_biquad_apply_buffer(OrcBiquad *f, float *buf, int n, int stride);
float orc_biquad_apply_sample(OrcBiquad *f, float x);

/* include/quantization_utils.h:15-25 */
void orc_quantized_to_float(const uint8_t *in, float *out, uint32_t n, uint8_t bits, float gain_db);
uint32_t orc_float_to_quantized(const float *in, uint8_t *out, uint32_t n, uint8_t bits);

/* include/dsp.h:66-93 — Q15 helpers downstream of the path (SURVEY.md §8f N4); 0 = ESP_OK, -1 = ESP_FAIL */
int orc_add_s16(const int16_t *in1, const int16_t *in2, int16_t *out, int len, int step1, int step2, int step_out,
                int shift);
int orc_mulc_s16(const int16_t *in, int16_t *out, int len, int16_t c, int step_in, int step_out);

/* include/wav_decoder.h:32-90, src/decode/wav_decoder.cpp — WAV header state machine (SURVEY.md §8f N3).
 * States 0..5 = WAV_DECODER_BEFORE_RIFF .. IN_DATA; results 0..5 = SUCCESS_NEXT .. ERROR_FAILED. */
typedef struct {
  int state;
  size_t bytes_processed, bytes_needed, bytes_to_skip, chunk_bytes_left;
  char chunk_name[5];
  uint32_t sample_rate;
  uint16_t num_channels, bits_per_sample;
} OrcWav;
void orc_wav_init(OrcWav *w);
int orc_wav_next(OrcWav *w, const uint8_t *buffer);
int orc_wav_decode_header(OrcWav *w, const uint8_t *buffer, size_t bytes_available);
void orc_wav_reset(OrcWav *w);
/* test-binding helpers: heap handle + snapshot {state, processed, needed, skip, chunk_left, rate, channels, bits} */
void *orc_wav_create(void);
void orc_wav_free(void *w);
void orc_wav_snapshot(const void *w, uint64_t out[8], char name[5]);

/* include/resampler.h:15-80 — pipeline policy + per-chunk composition */
typedef struct OrcWrapper OrcWrapper;
OrcWrapper *orc_wrapper_create(size_t in_samples, size_t out_samples, float src_rate, float dst_rate, int src_bits,
                               int dst_bits, int channels, int use_filter, int interpolate, int taps, int filters);
void orc_wrapper_free(OrcWrapper *w);
/* results: frames_used, frames_generated, predicted_frames_used, clipped_samples */
void orc_wrapper_resample(OrcWrapper *w, const uint8_t *in, uint8_t *out, size_t in_frames, size_t out_free,
                          float gain_db, uint64_t results[4]);
/* policy introspection: pre(1)/post(2)/none(0), biquad coeffs, ART lowpass + flags */
int orc_wrapper_policy(const OrcWrapper *w, float coeffs[5], float *sample_ratio, float *art_lowpass, int *art_flags);
/* orc_resample_set_fused on the wrapper's resampler (no-op when the rates are equal) */
void orc_wrapper_set_fused(OrcWrapper *w, int fused);

/* CPU-baseline driver (bench.py cpu_baseline kind "port"): n_streams independent
 * contexts over n_threads host threads, processing time only, seconds. */
double orc_bench_resample(int n_streams, int n_threads, int channels, int taps, int filters, float lowpass,
                          int flags, float advance, const float *in, size_t in_stride, int n_in, float *out,
                          size_t out_stride, int n_out, float ratio, unsigned long long *frames_generated);

#ifdef __cplusplus
}
#endif
#endif
