/* TEST INFRASTRUCTURE — CPU oracle for the B200 resampler path (see art_oracle.h).
 *
 * Plain-C restatement of the reference algorithm; every function names the
 * reference lines it follows (paths relative to /root/reference).  Arithmetic is
 * FP32, un-fused, in the reference's evaluation order, except for the opt-in fmaf
 * chain of orc_resample_set_fused.  Compile with -ffp-contract=off.  Never linked
 * into the product.
 */
#define _GNU_SOURCE
#include "art_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#ifndef M_PI
#define M_PI 3.14159265358979324
#endif

/* ------------------------------------------------------------------------- */
/* ART resampler — src/resample/art_resampler.cpp                             */
/* ------------------------------------------------------------------------- */

struct OrcResampler {
  int channels, ring_len, n_filters, taps, input_index, flags; /* include/art_resampler.h:25-29 */
  int fused; /* not in the reference: orc_resample_set_fused */
  float output_offset;
  float *ring; /* channels x ring_len history (reference: buffers[ch]) */
  float *bank; /* (n_filters+1) x taps (reference: filters[i])       */
};

/* src/dsp/dsps_dotprod_f32_ansi.c:17-25 — sequential, separate multiply and add.  With `fused` set, the same
 * sequence with each multiply-add rounded once (correctly rounded fmaf): the library's fast mode (DESIGN.md §2.2). */
static float orc_dot(const float *a, const float *b, int n, int fused) {
  float acc = 0;
  if (fused)
    for (int i = 0; i < n; i++)
      acc = fmaf(a[i], b[i], acc);
  else
    for (int i = 0; i < n; i++)
      acc += a[i] * b[i];
  return acc;
}

/* art_resampler.cpp:379-419 (init_filter).  `scratch` plays tempFilter. */
static void orc_build_phase(float *dst, float *scratch, int taps, int flags, float fraction, float lowpass) {
  const float a0 = 0.35875f, a1 = 0.48829f, a2 = 0.14128f, a3 = 0.01168f;
  const int half = taps / 2;
  float sum = 0.0f;

  for (int i = 0; i < taps; ++i) {
    /* :394 — float subtraction, one double multiply by pi, back to float */
    float rel = (float) (half - 1) + fraction - (float) i;
    float dist = (float) (fabs((double) rel) * M_PI);
    float ratio = dist / (float) half; /* :395 */
    float v;
    if (dist != 0.0f) {
      v = sinf(dist * lowpass) / (dist * lowpass); /* :399 */
      if (flags & ORC_BLACKMAN_HARRIS)
        v *= a0 + a1 * cosf(ratio) + a2 * cosf(2 * ratio) + a3 * cosf(3 * ratio); /* :402 */
      else
        v *= 0.5f * (1.0f + cosf(ratio)); /* :404 */
    } else
      v = 1.0f;
    scratch[i] = v;
    sum += v; /* :408 */
  }

  /* :413-418 — unity DC gain, error feedback walking outward from the centre */
  float scaler = 1.0f / sum, err = 0.0f;
  for (int i = half; i < taps; i = taps - i - (i >= half)) {
    scratch[i] *= scaler;
    dst[i] = scratch[i] - err;
    err += dst[i] - scratch[i];
  }
}

/* art_resampler.cpp:78-139 */
OrcResampler *orc_resample_init(int channels, int taps, int filters, float lowpass_ratio, int flags) {
  if (lowpass_ratio > 0.0f && lowpass_ratio < 1.0f) /* :82-87 */
    flags |= ORC_INCLUDE_LOWPASS;
  else {
    flags &= ~ORC_INCLUDE_LOWPASS;
    lowpass_ratio = 1.0f;
  }
  if ((taps & 3) || taps <= 0 || taps > 1024) { /* :89-92 */
    fprintf(stderr, "must 4-1024 filter taps, and a multiple of 4!\n");
    return NULL;
  }
  if (filters < 2 || filters > 1024) { /* :94-97 */
    fprintf(stderr, "must be 2-1024 filters!\n");
    return NULL;
  }
  OrcResampler *r = (OrcResampler *) calloc(1, sizeof *r);
  if (!r)
    return NULL;
  r->channels = channels;
  r->ring_len = taps * 16; /* :100 */
  r->n_filters = filters;
  r->taps = taps;
  r->flags = flags;
  r->bank = (float *) calloc((size_t) (filters + 1) * taps, sizeof(float));
  r->ring = (float *) calloc((size_t) channels * r->ring_len, sizeof(float));
  float *scratch = (float *) malloc(taps * sizeof(float));
  if (!r->bank || !r->ring || !scratch) {
    free(scratch);
    orc_resample_free(r);
    return NULL;
  }
  for (int i = 0; i <= filters; ++i) /* :114-121, fraction = (float) i / numFilters */
    orc_build_phase(r->bank + (size_t) i * taps, scratch, taps, flags, (float) i / (float) filters, lowpass_ratio);
  free(scratch);
  r->output_offset = (float) (taps / 2); /* :135 */
  r->input_index = taps;                 /* :136 */
  return r;
}

/* art_resampler.cpp:353-366 */
void orc_resample_free(OrcResampler *r) {
  if (!r)
    return;
  free(r->bank);
  free(r->ring);
  free(r);
}

/* art_resampler.cpp:144-152 */
void orc_resample_reset(OrcResampler *r) {
  memset(r->ring, 0, (size_t) r->channels * r->ring_len * sizeof(float));
  r->output_offset = (float) (r->taps / 2);
  r->input_index = r->taps;
}

/* art_resampler.cpp:313-318 */
void orc_resample_advance(OrcResampler *r, float delta) {
  if (delta < 0.0f)
    fprintf(stderr, "resampleAdvancePosition() can only advance forward!\n");
  else
    r->output_offset += delta;
}

/* art_resampler.cpp:348 */
float orc_resample_position(const OrcResampler *r) {
  return r->output_offset + ((float) r->taps / 2.0f) - (float) r->input_index;
}

/* art_resampler.cpp:421-451 (subsample / _interpolate / _no_interpolate) */
static float orc_subsample(const OrcResampler *r, const float *hist, float offset) {
  const int taps = r->taps, lowpass = r->flags & ORC_INCLUDE_LOWPASS;
  const float *src = hist + (int) floorf(offset); /* :422 / :436 */
  offset -= floorf(offset);
  if (offset == 0.0f && !lowpass) /* :425 / :439 */
    return *src;
  const float *win = src - taps / 2 + 1;
  if (!(r->flags & ORC_SUBSAMPLE_INTERPOLATE)) /* :428 nearest phase (may equal n_filters) */
    return orc_dot(r->bank + (size_t) ((int) floorf(offset * (float) r->n_filters + 0.5f)) * taps, win, taps,
                   r->fused);

  offset *= (float) r->n_filters; /* :442 */
  int i = (int) floorf(offset);
  float sum1 = orc_dot(r->bank + (size_t) i * taps, win, taps, r->fused); /* :443 */
  offset -= (float) i;
  if (offset == 0.0f && !lowpass) /* :445 */
    return sum1;
  float sum2 = orc_dot(r->bank + (size_t) (i + 1) * taps, win, taps, r->fused); /* :448 */
  return sum2 * offset + sum1 * (1.0f - offset);                       /* :450 */
}

/* The "consume one frame" half of the loop: ring rebase, art_resampler.cpp:175-181 / :216-222 */
static void orc_make_room(OrcResampler *r) {
  if (r->input_index == r->ring_len) {
    const int keep = r->taps, drop = r->ring_len - r->taps;
    for (int c = 0; c < r->channels; ++c)
      memmove(r->ring + (size_t) c * r->ring_len, r->ring + (size_t) c * r->ring_len + drop, keep * sizeof(float));
    r->output_offset -= (float) drop;
    r->input_index -= drop;
  }
}

/* art_resampler.cpp:208-243.  in/out strides let one body serve both layouts:
 * interleaved = (frame stride channels, channel stride 1); planar uses the pointer tables. */
static void orc_run(OrcResampler *r, const float *in_i, const float *const *in_p, int n_in, float *out_i,
                    float *const *out_p, int n_out, float ratio, unsigned *used, unsigned *generated) {
  const int half = r->taps / 2, ch = r->channels;
  unsigned u = 0, g = 0;
  while (n_out > 0) {
    if (r->output_offset >= (float) (r->input_index - half)) { /* :214 (int converted to float) */
      if (n_in <= 0)
        break;
      orc_make_room(r);
      for (int c = 0; c < ch; ++c)
        r->ring[(size_t) c * r->ring_len + r->input_index] = in_p ? in_p[c][u] : in_i[(size_t) u * ch + c];
      r->input_index++;
      u++;
      n_in--;
    } else {
      for (int c = 0; c < ch; ++c) {
        float v = orc_subsample(r, r->ring + (size_t) c * r->ring_len, r->output_offset);
        if (out_p)
          out_p[c][g] = v;
        else
          out_i[(size_t) g * ch + c] = v;
      }
      r->output_offset += (1.0f / ratio); /* :236 */
      g++;
      n_out--;
    }
  }
  *used = u;
  *generated = g;
}

void orc_resample_interleaved(OrcResampler *r, const float *in, int n_in, float *out, int n_out, float ratio,
                              unsigned *used, unsigned *generated) {
  orc_run(r, in, NULL, n_in, out, NULL, n_out, ratio, used, generated);
}

/* art_resampler.cpp:167-202 */
void orc_resample_planar(OrcResampler *r, const float *const *in, int n_in, float *const *out, int n_out,
                         float ratio, unsigned *used, unsigned *generated) {
  orc_run(r, NULL, in, n_in, NULL, out, n_out, ratio, used, generated);
}

/* art_resampler.cpp:257-279 */
unsigned orc_resample_required(const OrcResampler *r, int n_out, float ratio) {
  const int half = r->taps / 2, drop = r->ring_len - r->taps;
  int idx = r->input_index;
  float off = r->output_offset;
  unsigned used = 0;
  while (n_out > 0) {
    if (off >= (float) (idx - half)) {
      if (idx == r->ring_len) {
        off -= (float) drop;
        idx -= drop;
      }
      idx++;
      used++;
    } else {
      off += (1.0f / ratio);
      n_out--;
    }
  }
  return used;
}

/* art_resampler.cpp:281-306 */
unsigned orc_resample_expected(const OrcResampler *r, int n_in, float ratio) {
  const int half = r->taps / 2, drop = r->ring_len - r->taps;
  int idx = r->input_index;
  float off = r->output_offset;
  unsigned gen = 0;
  for (;;) {
    if (off >= (float) (idx - half)) {
      if (n_in <= 0)
        break;
      if (idx == r->ring_len) {
        off -= (float) drop;
        idx -= drop;
      }
      idx++;
      n_in--;
    } else {
      off += (1.0f / ratio);
      gen++;
    }
  }
  return gen;
}

int orc_resample_flags(const OrcResampler *r) { return r->flags; }
void orc_resample_set_fused(OrcResampler *r, int fused) { r->fused = fused != 0; }
void orc_resample_copy_filter(const OrcResampler *r, int idx, float *dst) {
  memcpy(dst, r->bank + (size_t) idx * r->taps, r->taps * sizeof(float));
}
void orc_resample_state(const OrcResampler *r, float *output_offset, int *input_index) {
  *output_offset = r->output_offset;
  *input_index = r->input_index;
}

/* ------------------------------------------------------------------------- */
/* art_biquad — src/resample/art_biquad.cpp                                   */
/* ------------------------------------------------------------------------- */

/* art_biquad.cpp:16-25 — design in double, stored as float */
void orc_biquad_lowpass(OrcBiquadCoeffs *c, double frequency) {
  double Q = sqrt(0.5), K = tan(M_PI * frequency);
  double norm = 1.0 / (1.0 + K / Q + K * K);
  c->a0 = (float) (K * K * norm);
  c->a1 = 2 * c->a0;
  c->a2 = c->a0;
  c->b1 = (float) (2.0 * (K * K - 1.0) * norm);
  c->b2 = (float) ((1.0 - K / Q + K * K) * norm);
}

/* art_biquad.cpp:29-38 */
void orc_biquad_highpass(OrcBiquadCoeffs *c, double frequency) {
  double Q = sqrt(0.5), K = tan(M_PI * frequency);
  double norm = 1.0 / (1.0 + K / Q + K * K);
  c->a0 = (float) norm;
  c->a1 = (float) (-2.0 * norm);
  c->a2 = c->a0;
  c->b1 = (float) (2.0 * (K * K - 1.0) * norm);
  c->b2 = (float) ((1.0 - K / Q + K * K) * norm);
}

/* art_biquad.cpp:43-51 */
void orc_biquad_init(OrcBiquad *f, const OrcBiquadCoeffs *c, float gain) {
  f->c = *c;
  f->c.a0 *= gain;
  f->c.a1 *= gain;
  f->c.a2 *= gain;
  f->in_d1 = f->in_d2 = 0.0f;
  f->out_d1 = f->out_d2 = 0.0f;
  f->first_order = (c->a2 == 0.0f && c->b2 == 0.0f);
}

/* art_biquad.cpp:55-69 — Direct Form I, left to right, every product and sum rounded */
float orc_biquad_apply_sample(OrcBiquad *f, float x) {
  float sum;
  if (f->first_order)
    sum = (x * f->c.a0) + (f->in_d1 * f->c.a1) - (f->c.b1 * f->out_d1);
  else
    sum = (x * f->c.a0) + (f->in_d1 * f->c.a1) + (f->in_d2 * f->c.a2) - (f->c.b1 * f->out_d1) -
          (f->c.b2 * f->out_d2);
  f->out_d2 = f->out_d1;
  f->out_d1 = sum;
  f->in_d2 = f->in_d1;
  f->in_d1 = x;
  return sum;
}

/* art_biquad.cpp:73-93 — in place, strided */
void orc_biquad_apply_buffer(OrcBiquad *f, float *buf, int n, int stride) {
  for (int k = 0; k < n; ++k, buf += stride)
    *buf = orc_biquad_apply_sample(f, *buf);
}

/* ------------------------------------------------------------------------- */
/* quantization_utils — src/quantization_utils.cpp                            */
/* ------------------------------------------------------------------------- */

/* quantization_utils.cpp:6-48.  Little-endian packed PCM; byte-wise reads.  The
 * 32-bit branch sign-extends byte 2 as well as byte 3 (:43) — reproduced. */
void orc_quantized_to_float(const uint8_t *in, float *out, uint32_t n, uint8_t bits, float gain_db) {
  float gain = powf(10.0f, gain_db / 20.0f);
  if (bits <= 8) {
    float k = gain / 128.0f;
    for (uint32_t i = 0; i < n; ++i)
      out[i] = (float) ((int) in[i] - 128) * k;
  } else if (bits <= 16) {
    float k = gain / 32768.0f;
    for (uint32_t i = 0; i < n; ++i) {
      int16_t v = (int16_t) (in[2 * i] | (in[2 * i + 1] << 8));
      out[i] = (float) v * k;
    }
  } else if (bits <= 24) {
    float k = gain / 8388608.0f;
    for (uint32_t i = 0; i < n; ++i) {
      const uint8_t *p = in + 3 * (size_t) i;
      int32_t v = (int32_t) p[0] + ((int32_t) p[1] << 8) + ((int32_t) (int8_t) p[2]) * 65536;
      out[i] = (float) v * k;
    }
  } else if (bits <= 32) {
    float k = gain / 2147483648.0f;
    for (uint32_t i = 0; i < n; ++i) {
      const uint8_t *p = in + 4 * (size_t) i;
      /* sums wrap modulo 2^32 exactly like the reference's int32 additions */
      uint32_t v = (uint32_t) p[0] + ((uint32_t) p[1] << 8) + (uint32_t) ((int32_t) (int8_t) p[2] * 65536) +
                   ((uint32_t) (int32_t) (int8_t) p[3] << 24);
      out[i] = (float) (int32_t) v * k;
    }
  }
}

/* quantization_utils.cpp:50-94.  Round half up in FP32, clip + count, pack LE. */
uint32_t orc_float_to_quantized(const float *in, uint8_t *out, uint32_t n, uint8_t bits) {
  float scalar = (float) ((uint64_t) 1 << bits) / 2.0f;
  int32_t offset = (bits <= 8) * 128;
  int32_t hi = (int32_t) ((1u << (bits - 1)) - 1u);
  int32_t lo = ~hi;
  int shift = (32 - bits) % 8;
  uint32_t clipped = 0;
  size_t j = 0;
  for (uint32_t i = 0; i < n; ++i) {
    int32_t v = (int32_t) floorf((in[i] * scalar) + 0.5f);
    if (bits < 32) {
      if (v > hi) {
        ++clipped;
        v = hi;
      } else if (v < lo) {
        ++clipped;
        v = lo;
      }
    } else {
      if (in[i] >= 1.0f) {
        ++clipped;
        v = hi;
      } else if (in[i] < -1.0f) {
        ++clipped;
        v = lo;
      }
    }
    v = (int32_t) ((uint32_t) v << shift) + offset;
    out[j++] = (uint8_t) v;
    if (bits > 8) {
      out[j++] = (uint8_t) (v >> 8);
      if (bits > 16)
        out[j++] = (uint8_t) (v >> 16);
      if (bits > 24)
        out[j++] = (uint8_t) (v >> 24);
    }
  }
  return clipped;
}

/* ------------------------------------------------------------------------- */
/* Q15 mix / volume — src/dsp/dsps_add_s16_ansi.c, src/dsp/dsps_mulc_s16_ansi.c */
/* ------------------------------------------------------------------------- */

/* dsps_add_s16_ansi.c:10-27 — 32-bit sum, arithmetic shift, truncated to int16 */
int orc_add_s16(const int16_t *in1, const int16_t *in2, int16_t *out, int len, int step1, int step2, int step_out,
                int shift) {
  if (!in1 || !in2 || !out)
    return -1;
  for (int i = 0; i < len; i++) {
    int32_t acc = (int32_t) in1[i * step1] + (int32_t) in2[i * step2];
    out[i * step_out] = (int16_t) (acc >> shift);
  }
  return 0;
}

/* dsps_mulc_s16_ansi.c:18-31 — Q15 multiply by a constant */
int orc_mulc_s16(const int16_t *in, int16_t *out, int len, int16_t c, int step_in, int step_out) {
  if (!in || !out)
    return -1;
  for (int i = 0; i < len; i++) {
    int32_t acc = (int32_t) in[i * step_in] * (int32_t) c;
    out[i * step_out] = (int16_t) (acc >> 15);
  }
  return 0;
}

/* ------------------------------------------------------------------------- */
/* WAV header parser — src/decode/wav_decoder.cpp                                */
/* ------------------------------------------------------------------------- */

/* include/wav_decoder.h:78-88 — member initialisers (bytes_processed_ has none) */
void orc_wav_init(OrcWav *w) {
  memset(w, 0, sizeof *w);
  w->state = 0;
  w->bytes_needed = 8;
}

/* wav_decoder.cpp:61-65 etc.: memcpy of a uint32 into a size_t member — only the low four bytes change — then the
 * RIFF pad byte */
static void wav_chunk_size(OrcWav *w, const uint8_t *p) {
  uint32_t v;
  memcpy(&v, p, 4);
  memcpy(&w->chunk_bytes_left, &v, 4);
  if (w->chunk_bytes_left % 2 != 0)
    w->chunk_bytes_left++;
}

/* wav_decoder.cpp:48-149 */
int orc_wav_next(OrcWav *w, const uint8_t *buffer) {
  w->bytes_to_skip = 0;
  switch (w->state) {
    case 0: /* BEFORE_RIFF :52-68 */
      memcpy(w->chunk_name, buffer, 4);
      if (memcmp(w->chunk_name, "RIFF", 4) != 0)
        return 3;
      wav_chunk_size(w, buffer + 4);
      w->state = 1;
      w->bytes_needed = 4;
      break;
    case 1: /* BEFORE_WAVE :70-80 */
      memcpy(w->chunk_name, buffer, 4);
      if (memcmp(w->chunk_name, "WAVE", 4) != 0)
        return 4;
      w->state = 2;
      w->bytes_needed = 8;
      break;
    case 2: /* BEFORE_FMT :82-100 */
      memcpy(w->chunk_name, buffer, 4);
      wav_chunk_size(w, buffer + 4);
      if (memcmp(w->chunk_name, "fmt ", 4) == 0) {
        w->state = 3;
        w->bytes_needed = w->chunk_bytes_left;
      } else {
        w->bytes_to_skip = w->chunk_bytes_left;
        w->bytes_needed = 8;
      }
      break;
    case 3: /* IN_FMT :102-120 */
      memcpy(&w->num_channels, buffer + 2, 2);
      memcpy(&w->sample_rate, buffer + 4, 4);
      memcpy(&w->bits_per_sample, buffer + 14, 2);
      w->state = 4;
      w->bytes_needed = 8;
      break;
    case 4: /* BEFORE_DATA :122-141 */
      memcpy(w->chunk_name, buffer, 4);
      wav_chunk_size(w, buffer + 4);
      if (memcmp(w->chunk_name, "data", 4) == 0) {
        w->state = 5;
        w->bytes_needed = 0;
        return 1;
      }
      w->bytes_to_skip = w->chunk_bytes_left;
      w->bytes_needed = 8;
      break;
    default: /* IN_DATA :143-146 */
      return 1;
  }
  return 0;
}

/* wav_decoder.cpp:8-46 */
int orc_wav_decode_header(OrcWav *w, const uint8_t *buffer, size_t bytes_available) {
  size_t to_skip = w->bytes_to_skip, to_read = w->bytes_needed;
  w->bytes_processed = 0;
  while (to_skip + to_read > 0) {
    if (to_skip > bytes_available || to_read > bytes_available)
      return 2;
    if (to_skip > 0) {
      buffer += to_skip;
      w->bytes_processed += to_skip;
      bytes_available -= to_skip;
      to_skip = 0;
    } else if (to_read > 0) {
      int r = orc_wav_next(w, buffer);
      buffer += to_read;
      w->bytes_processed += to_read;
      bytes_available -= to_read;
      if (r == 1)
        return r;
      if (r != 0)
        return r;
      to_skip = w->bytes_to_skip;
      to_read = w->bytes_needed;
    }
  }
  return 5;
}

/* wav_decoder.cpp:151-161 — bytes_needed_ and bytes_processed_ are NOT restored */
void orc_wav_reset(OrcWav *w) {
  w->state = 0;
  w->bytes_to_skip = 0;
  memset(w->chunk_name, 0, sizeof w->chunk_name);
  w->chunk_bytes_left = 0;
  w->sample_rate = 0;
  w->num_channels = 0;
  w->bits_per_sample = 0;
}

void *orc_wav_create(void) {
  OrcWav *w = (OrcWav *) malloc(sizeof *w);
  if (w)
    orc_wav_init(w);
  return w;
}
void orc_wav_free(void *w) { free(w); }
void orc_wav_snapshot(const void *p, uint64_t out[8], char name[5]) {
  const OrcWav *w = (const OrcWav *) p;
  out[0] = (uint64_t) w->state;
  out[1] = w->bytes_processed;
  out[2] = w->bytes_needed;
  out[3] = w->bytes_to_skip;
  out[4] = w->chunk_bytes_left;
  out[5] = w->sample_rate;
  out[6] = w->num_channels;
  out[7] = w->bits_per_sample;
  memcpy(name, w->chunk_name, 4);
  name[4] = 0;
}

/* ------------------------------------------------------------------------- */
/* Resampler wrapper — src/resample/resampler.cpp, include/resampler.h         */
/* ------------------------------------------------------------------------- */

struct OrcWrapper {
  float *fin, *fout;
  size_t fin_samples, fout_samples;
  OrcResampler *art;
  OrcBiquad lp[2][2]; /* include/resampler.h:64 — two channels, two sections */
  OrcBiquadCoeffs lp_coeff;
  float sample_ratio, lowpass_ratio, art_lowpass;
  int pre, post, resampling, in_bits, out_bits, channels, art_flags;
};

/* resampler.cpp:21-98 */
OrcWrapper *orc_wrapper_create(size_t in_samples, size_t out_samples, float src_rate, float dst_rate, int src_bits,
                               int dst_bits, int channels, int use_filter, int interpolate, int taps, int filters) {
  OrcWrapper *w = (OrcWrapper *) calloc(1, sizeof *w);
  if (!w)
    return NULL;
  w->in_bits = src_bits;
  w->out_bits = dst_bits;
  w->channels = channels;
  w->sample_ratio = 1.0f;
  w->lowpass_ratio = 1.0f;
  w->art_lowpass = 1.0f;
  w->fin_samples = in_samples;
  w->fout_samples = out_samples;
  w->fin = (float *) malloc((in_samples ? in_samples : 1) * sizeof(float));
  w->fout = (float *) malloc((out_samples ? out_samples : 1) * sizeof(float));
  if (!w->fin || !w->fout) {
    orc_wrapper_free(w);
    return NULL;
  }
  if (src_rate != dst_rate) { /* :38 */
    w->resampling = 1;
    int flags = interpolate ? ORC_SUBSAMPLE_INTERPOLATE : 0;
    w->sample_ratio = dst_rate / src_rate; /* :46 */
    if (w->sample_ratio < 1.0f) {           /* :48-59 */
      w->lowpass_ratio -= (10.24f / (float) taps);
      if (w->lowpass_ratio < 0.84f)
        w->lowpass_ratio = 0.84f;
      if (w->lowpass_ratio < w->sample_ratio)
        w->lowpass_ratio = w->sample_ratio;
    }
    if (w->lowpass_ratio * w->sample_ratio < 0.98f && use_filter) { /* :60-64 */
      float cutoff = w->lowpass_ratio * w->sample_ratio / 2.0f;
      orc_biquad_lowpass(&w->lp_coeff, cutoff);
      w->pre = 1;
    }
    if (w->lowpass_ratio / w->sample_ratio < 0.98f && use_filter && !w->pre) { /* :66-70 */
      float cutoff = w->lowpass_ratio / w->sample_ratio / 2.0f;
      orc_biquad_lowpass(&w->lp_coeff, cutoff);
      w->post = 1;
    }
    if (w->pre || w->post) /* :72-77 (the reference indexes lowpass_[channel] without a bound check) */
      for (int c = 0; c < channels && c < 2; ++c) {
        orc_biquad_init(&w->lp[c][0], &w->lp_coeff, 1.0f);
        orc_biquad_init(&w->lp[c][1], &w->lp_coeff, 1.0f);
      }
    if (w->sample_ratio < 1.0f) { /* :79-89 */
      w->art_lowpass = w->sample_ratio * w->lowpass_ratio;
      w->art_flags = flags | ORC_INCLUDE_LOWPASS;
    } else if (w->lowpass_ratio < 1.0f) {
      w->art_lowpass = w->lowpass_ratio;
      w->art_flags = flags | ORC_INCLUDE_LOWPASS;
    } else {
      w->art_lowpass = 1.0f;
      w->art_flags = flags;
    }
    w->art = orc_resample_init(channels, taps, filters, w->art_lowpass, w->art_flags);
    if (!w->art) {
      orc_wrapper_free(w);
      return NULL;
    }
    orc_resample_advance(w->art, (float) taps / 2.0f); /* :94 */
  }
  return w;
}

void orc_wrapper_free(OrcWrapper *w) {
  if (!w)
    return;
  orc_resample_free(w->art);
  free(w->fin);
  free(w->fout);
  free(w);
}

void orc_wrapper_set_fused(OrcWrapper *w, int fused) {
  if (w->art)
    orc_resample_set_fused(w->art, fused);
}

int orc_wrapper_policy(const OrcWrapper *w, float coeffs[5], float *sample_ratio, float *art_lowpass,
                       int *art_flags) {
  memcpy(coeffs, &w->lp_coeff, 5 * sizeof(float));
  *sample_ratio = w->sample_ratio;
  *art_lowpass = w->art_lowpass;
  *art_flags = w->art ? orc_resample_flags(w->art) : 0;
  return w->pre ? 1 : (w->post ? 2 : 0);
}

/* resampler.cpp:100-160 */
void orc_wrapper_resample(OrcWrapper *w, const uint8_t *in, uint8_t *out, size_t in_frames, size_t out_free,
                          float gain_db, uint64_t results[4]) {
  size_t todo = in_frames;
  const int ch = w->channels;
  if (w->resampling) { /* :104-107 */
    size_t need = orc_resample_required(w->art, (int) out_free, w->sample_ratio);
    if (need < todo)
      todo = need;
  } else if (out_free < todo)
    todo = out_free;

  orc_quantized_to_float(in, w->resampling ? w->fin : w->fout, (uint32_t) (todo * ch), (uint8_t) w->in_bits,
                         gain_db); /* :112-119 */
  size_t used = todo, generated = todo;
  if (w->resampling) {
    if (w->pre) /* :126-133 */
      for (int c = 0; c < ch; ++c) {
        orc_biquad_apply_buffer(&w->lp[c][0], w->fin + c, (int) todo, ch);
        orc_biquad_apply_buffer(&w->lp[c][1], w->fin + c, (int) todo, ch);
      }
    unsigned u, g;
    orc_resample_interleaved(w->art, w->fin, (int) todo, w->fout, (int) out_free, w->sample_ratio, &u, &g);
    used = u;
    generated = g;
    if (w->post) /* :142-149 */
      for (int c = 0; c < ch; ++c) {
        orc_biquad_apply_buffer(&w->lp[c][0], w->fout + c, (int) generated, ch);
        orc_biquad_apply_buffer(&w->lp[c][1], w->fout + c, (int) generated, ch);
      }
  }
  uint32_t clipped = orc_float_to_quantized(w->fout, out, (uint32_t) (generated * ch), (uint8_t) w->out_bits);
  results[0] = used;
  results[1] = generated;
  results[2] = todo;
  results[3] = clipped;
}

/* ------------------------------------------------------------------------- */
/* CPU-baseline driver (bench.py, kind "port")                                */
/* ------------------------------------------------------------------------- */

typedef struct {
  int first, step, n_streams;
  OrcResampler **ctx;
  const float *in;
  size_t in_stride;
  int n_in;
  float *out;
  size_t out_stride;
  int n_out;
  float ratio;
  unsigned long long generated;
} OrcJob;

static void *orc_bench_thread(void *p) {
  OrcJob *j = (OrcJob *) p;
  unsigned long long g = 0;
  for (int s = j->first; s < j->n_streams; s += j->step) {
    unsigned u, gen;
    orc_resample_interleaved(j->ctx[s], j->in + s * j->in_stride, j->n_in, j->out + s * j->out_stride, j->n_out,
                             j->ratio, &u, &gen);
    g += gen;
  }
  j->generated = g;
  return NULL;
}

double orc_bench_resample(int n_streams, int n_threads, int channels, int taps, int filters, float lowpass,
                          int flags, float advance, const float *in, size_t in_stride, int n_in, float *out,
                          size_t out_stride, int n_out, float ratio, unsigned long long *frames_generated) {
  if (n_threads < 1)
    n_threads = 1;
  OrcResampler **ctx = (OrcResampler **) calloc(n_streams, sizeof *ctx);
  OrcJob *jobs = (OrcJob *) calloc(n_threads, sizeof *jobs);
  pthread_t *tids = (pthread_t *) calloc(n_threads, sizeof *tids);
  for (int s = 0; s < n_streams; ++s) {
    ctx[s] = orc_resample_init(channels, taps, filters, lowpass, flags);
    if (!ctx[s])
      return -1.0;
    if (advance > 0.0f)
      orc_resample_advance(ctx[s], advance);
  }
  struct timespec t0, t1;
  clock_gettime(CLOCK_MONOTONIC, &t0);
  for (int t = 0; t < n_threads; ++t) {
    OrcJob j = {t, n_threads, n_streams, ctx, in, in_stride, n_in, out, out_stride, n_out, ratio, 0};
    jobs[t] = j;
    pthread_create(&tids[t], NULL, orc_bench_thread, &jobs[t]);
  }
  unsigned long long total = 0;
  for (int t = 0; t < n_threads; ++t) {
    pthread_join(tids[t], NULL);
    total += jobs[t].generated;
  }
  clock_gettime(CLOCK_MONOTONIC, &t1);
  for (int s = 0; s < n_streams; ++s)
    orc_resample_free(ctx[s]);
  free(ctx);
  free(jobs);
  free(tids);
  if (frames_generated)
    *frames_generated = total;
  return (double) (t1.tv_sec - t0.tv_sec) + 1e-9 * (double) (t1.tv_nsec - t0.tv_nsec);
}
