// Host-side planning (see plan.hpp).  Compiled with -ffp-contract=off: the reference
// arithmetic is un-fused FP32 and the bank/schedule must match it bit for bit.
#include "plan.hpp"

#include <math.h>
#include <stdio.h>

namespace espb {

bool normalise_init(int taps, int filters, float *lowpass, int *flags) {
  if (*lowpass > 0.0f && *lowpass < 1.0f)
    *flags |= kFlagLowpass;
  else {
    *flags &= ~kFlagLowpass;
    *lowpass = 1.0f;
  }
  if ((taps & 3) || taps <= 0 || taps > 1024) {
    fprintf(stderr, "must 4-1024 filter taps, and a multiple of 4!\n");
    return false;
  }
  if (filters < 2 || filters > 1024) {
    fprintf(stderr, "must be 2-1024 filters!\n");
    return false;
  }
  return true;
}

namespace {

// Window value at normalised distance `r` (pi at the window edge).
inline float window_at(float r, bool blackman_harris) {
  if (blackman_harris)
    return 0.35875f + 0.48829f * cosf(r) + 0.14128f * cosf(2 * r) + 0.01168f * cosf(3 * r);
  return 0.5f * (1.0f + cosf(r));
}

// One phase of the bank.  raw[] receives the un-normalised taps; row[] the final ones.
void build_phase(float *row, float *raw, int taps, bool bh, float fraction, float lowpass) {
  const int half = taps / 2;
  const double pi = 3.14159265358979323846;
  float total = 0.0f;
  for (int t = 0; t < taps; ++t) {
    const float rel = (float) (half - 1) + fraction - (float) t;
    const float dist = (float) (fabs((double) rel) * pi);
    float v = 1.0f;
    if (dist != 0.0f) {
      const float arg = dist * lowpass;
      v = sinf(arg) / arg;
      v *= window_at(dist / (float) half, bh);
    }
    raw[t] = v;
    total += v;
  }
  // unity DC gain; rounding error of each scaled tap is fed to the next one, visiting
  // taps centre-out: half, half-1, half+1, half-2, ...
  const float scale = 1.0f / total;
  float carry = 0.0f;
  int t = half;
  for (int visited = 0; visited < taps; ++visited) {
    raw[t] *= scale;
    row[t] = raw[t] - carry;
    carry += row[t] - raw[t];
    t = taps - t - (t >= half ? 1 : 0);
  }
}

}  // namespace

void build_filter_bank(const ArtGeometry &g, float lowpass, std::vector<float> &bank) {
  bank.assign((size_t) (g.filters + 1) * g.taps, 0.0f);
  std::vector<float> raw(g.taps);
  for (int i = 0; i <= g.filters; ++i)
    build_phase(bank.data() + (size_t) i * g.taps, raw.data(), g.taps, (g.flags & kFlagBlackmanHarris) != 0,
                (float) i / (float) g.filters, lowpass);
}

ArtState initial_state(int taps) { return ArtState{(float) (taps / 2), taps}; }

float position_of(const ArtGeometry &g, ArtState st) { return st.offset + ((float) g.taps / 2.0f) - (float) st.index; }

namespace {

// The signal-independent core of the reference loop.  `emit(offset, base)` is called for every output with
// the pre-increment offset and the accumulated ring rebase.  (A closed-form jump over runs of "consume"
// steps was measured slower than this loop: the steps are cheap and well predicted.)
template <typename Emit>
inline void run_machine(const ArtGeometry &g, ArtState &st, int n_in, int n_out, float ratio, bool stop_on_input,
                        bool stop_on_output, unsigned *used, unsigned *generated, Emit emit) {
  const int half = g.taps / 2, ring = g.taps * 16, drop = ring - g.taps;
  const float step = 1.0f / ratio;
  float off = st.offset;
  int idx = st.index;
  long long base = 0;
  unsigned u = 0, gcount = 0;
  for (;;) {
    if (stop_on_output && n_out <= 0)
      break;
    if (off >= (float) (idx - half)) {
      if (stop_on_input && n_in <= 0)
        break;
      if (idx == ring) {
        off -= (float) drop;
        idx -= drop;
        base += drop;
      }
      ++idx;
      ++u;
      --n_in;
    } else {
      emit(off, base);
      off += step;
      ++gcount;
      --n_out;
    }
  }
  st.offset = off;
  st.index = idx;
  *used = u;
  *generated = gcount;
}

}  // namespace

// floorf for the non-negative values of the state machine (offsets live in [0, 16*taps), phase products in
// [0, filters]): truncation is the same value and avoids a libm call per output.
static inline float floor_nonneg(float v) { return (float) (int) v; }

void build_schedule(const ArtGeometry &g, ArtState start, int n_in, int n_out, float ratio, Schedule &s) {
  // Upper bound on the outputs of this call: capacity, and what the input can feed — every output moves the
  // offset by 1/ratio, and the offset can run at most (frames available + what is already buffered) ahead.
  size_t cap = n_out > 0 ? (size_t) n_out : 0;
  {
    const double room = (double) (n_in > 0 ? n_in : 0) + (double) start.index - (double) start.offset + 2.0;
    const double feed = room * (double) ratio + 16.0;
    if (feed < (double) cap)
      cap = feed > 0.0 ? (size_t) feed : 0;
  }
  s.outs.clear();
  s.outs.reserve(cap + 1);
  // Pass 1 (sequential, branchy): the state machine records, per output, the offset (in .w) and the ring
  // rebase folded into a window-start base (in .ws).  Pass 2 (finalize_entries, independent per output): window
  // start, phase, weight and kind from the offset (art_resampler.cpp:421-451), written into the same 16-byte entries.
  const int half = g.taps / 2, idx0 = start.index;
  ArtState st = start;
  run_machine(g, st, n_in, n_out, ratio, true, true, &s.used, &s.generated, [&](float off, long long base) {
    OutEntry e;
    e.ws = (int32_t) (base - half + 1 - idx0);
    e.w = off;
    s.outs.push_back(e);  // grows if the bound above was ever too small
  });
  s.end = st;
  finalize_entries(g, s.outs.data(), s.outs.size());
}

void finalize_entries(const ArtGeometry &g, OutEntry *out, size_t n) {
  const bool lowpass = (g.flags & kFlagLowpass) != 0, interp = (g.flags & kFlagInterpolate) != 0;
  const float nf = (float) g.filters;
  for (size_t k = 0; k < n; ++k) {
    const float off = out[k].w;
    const float fl = floor_nonneg(off);
    float frac = off - fl;
    OutEntry e;
    e.ws = out[k].ws + (int32_t) fl;
    e.phase = 0;
    e.w = 0.0f;
    if (frac == 0.0f && !lowpass) {
      e.kind = kKindPass;
    } else if (!interp) {
      e.kind = kKindSingle;
      e.phase = (int) floor_nonneg(frac * nf + 0.5f);
    } else {
      frac *= nf;
      const int i = (int) floor_nonneg(frac);
      frac -= (float) i;
      e.phase = i;
      e.w = frac;
      e.kind = (frac == 0.0f && !lowpass) ? kKindSingle : kKindBlend;
    }
    out[k] = e;
  }
}

void build_schedule_segments(const ArtGeometry &g, ArtState start, int n_in, int n_out, float ratio, Schedule &s) {
  const int half = g.taps / 2, ring = g.taps * 16, drop = ring - g.taps, idx0 = start.index;
  const float thr = (float) (ring - half);  // an output whose offset has reached this needs the ring rebase first
  const float step = 1.0f / ratio;
  s.outs.clear();
  s.segs.clear();
  s.segmented = true;
  float off = start.offset;
  int idx = start.index;
  long long base = 0, in_left = n_in > 0 ? n_in : 0, out_left = n_out > 0 ? n_out : 0;
  unsigned used = 0, gen = 0;
  // The reference machine itself, for at most max_emit outputs from the current state (which is always "between
  // two emissions").  false: the call has ended (output space or input exhausted).
  auto emit_seq = [&](long long max_emit) -> bool {
    long long emitted = 0;
    for (;;) {
      if (out_left <= 0)
        return false;
      if (emitted >= max_emit)
        return true;
      if (off >= (float) (idx - half)) {
        if (in_left <= 0)
          return false;
        if (idx == ring) {
          off -= (float) drop;
          idx -= drop;
          base += drop;
        }
        ++idx;
        ++used;
        --in_left;
      } else {
        s.segs.push_back(SchedSegment{(int32_t) gen, 1, (int32_t) (base - half + 1 - idx0), off, 0.0f});
        off += step;
        ++gen;
        --out_left;
        ++emitted;
      }
    }
  };
  // the closed form needs a sane step: positive, and small against the ring (ratios below ~4 / taps fall back)
  const bool closed_form_ok = step > 0.0f && step < (float) g.taps * 0.25f && off >= 0.0f;
  for (;;) {
    if (out_left <= 0)
      break;
    if (!closed_form_ok) {
      emit_seq(1LL << 62);
      break;
    }
    // ---- one piece, tentatively (committed only if the input covers all of it)
    float o = off;
    int id = idx;
    long long b = base, il = in_left;
    unsigned consumed = 0;
    if (o >= thr) {  // consume up to idx == ring, then the consume that rebases (art_resampler.cpp:175-181)
      const long long c = (long long) (ring - id) + 1;
      if (il < c) {
        emit_seq(1LL << 62);
        break;
      }
      il -= c;
      consumed += (unsigned) c;
      id = g.taps + 1;
      o -= (float) drop;
      b += drop;
    }
    if (!(o >= 1.0f)) {  // (sub-unit offsets only occur for tiny filters: not worth a closed form)
      if (!emit_seq(1))
        break;
      continue;
    }
    const int ex = ilogbf(o);
    const float top = ldexpf(1.0f, ex + 1);
    const double u = ldexp(1.0, ex - 23);      // one ulp of this binade
    const float lim = top < thr ? top : thr;   // offsets below it continue the progression
    const float o1 = o + step;
    const float o2 = o1 + step;
    const float inc = o1 - o;
    if (!(o1 < lim) || !(inc > 0.0f) || (o2 < lim && (o2 - o1) != inc)) {
      // a one-output piece, or a tie whose first rounding differs from the following ones: one exact step
      if (!emit_seq(1))
        break;
      continue;
    }
    const long long O = (long long) ((double) o / u), I = (long long) ((double) inc / u),
                    Lm = (long long) ((double) lim / u);
    // o2 < lim: the first two increments agree, so all do (a tie rounding can only differ on its first step), and the
    // piece holds the offsets O + j I < Lm.  Otherwise the piece is {o, o1} and o2 (a real float sum) starts the next.
    const long long nj = o2 < lim ? (Lm - O + I - 1) / I : 2;
    const long long m = nj < out_left ? nj : out_left;
    const double o_last = (double) (O + (m - 1) * I) * u;
    long long need = (long long) o_last + half + 1 - id;  // o_last >= 0: truncation == floor
    if (need < 0)
      need = 0;
    if (need > il) {
      // the input ends inside this piece: the outputs it can still feed (offset < idx + input - half) leave as a
      // run, the reference machine then consumes what is left and ends the call
      const long long F1 = il + id - half;
      long long cnt = ((long long) ((double) F1 / u) - O + I - 1) / I;
      cnt = cnt < 0 ? 0 : (cnt > m ? m : cnt);
      if (cnt > 0) {
        const double o_fed = (double) (O + (cnt - 1) * I) * u;
        long long nd = (long long) o_fed + half + 1 - id;
        nd = nd < 0 ? 0 : nd;
        in_left = il - nd;
        used += consumed + (unsigned) nd;
        idx = id + (int) nd;
        base = b;
        s.segs.push_back(SchedSegment{(int32_t) gen, (int32_t) cnt, (int32_t) (b - half + 1 - idx0), o, inc});
        gen += (unsigned) cnt;
        out_left -= cnt;
        off = (float) o_fed + step;
      }
      emit_seq(1LL << 62);
      break;
    }
    in_left = il - need;
    used += consumed + (unsigned) need;
    idx = id + (int) need;
    base = b;
    s.segs.push_back(SchedSegment{(int32_t) gen, (int32_t) m, (int32_t) (b - half + 1 - idx0), o, inc});
    gen += (unsigned) m;
    out_left -= m;
    off = (float) o_last + step;
  }
  s.used = used;
  s.generated = gen;
  s.end = ArtState{off, idx};
}

static inline float segment_offset(const SchedSegment &sg, int j) {
  return (float) ((double) sg.off0 + (double) j * (double) sg.inc);  // exact: every term is a multiple of one ulp
}

int32_t schedule_ws(const Schedule &s, int k, int *cursor) {
  if (!s.segmented)
    return s.outs[k].ws;
  int c = cursor ? *cursor : 0;
  const int n = (int) s.segs.size();
  if (c < 0 || c >= n || s.segs[c].n0 > k) {  // not a forward walk: binary search
    int lo = 0, hi = n - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (s.segs[mid].n0 <= k)
        lo = mid;
      else
        hi = mid - 1;
    }
    c = lo;
  }
  while (c + 1 < n && s.segs[c + 1].n0 <= k)
    ++c;
  if (cursor)
    *cursor = c;
  const SchedSegment &sg = s.segs[c];
  return sg.ws_base + (int32_t) segment_offset(sg, k - sg.n0);
}

void expand_segments(const ArtGeometry &g, const Schedule &s, OutEntry *out) {
  for (size_t i = 0; i < s.segs.size(); ++i) {
    const SchedSegment &sg = s.segs[i];
    for (int j = 0; j < sg.count; ++j) {
      out[sg.n0 + j].ws = sg.ws_base;
      out[sg.n0 + j].w = segment_offset(sg, j);
    }
  }
  finalize_entries(g, out, s.generated);
}

unsigned required_samples(const ArtGeometry &g, ArtState st, int n_out, float ratio) {
  unsigned used, gen;
  run_machine(g, st, 0, n_out, ratio, false, true, &used, &gen, [](float, long long) {});
  return used;
}

unsigned expected_output(const ArtGeometry &g, ArtState st, int n_in, float ratio) {
  unsigned used, gen;
  run_machine(g, st, n_in, 0, ratio, true, false, &used, &gen, [](float, long long) {});
  return gen;
}


void build_pass_plan(const Schedule &s, int taps, int blocks_per_pass, int chunk_rows, PassPlan &p) {
  const int opp = blocks_per_pass * kOutputsPerBlock;
  const int n = (int) s.generated;
  int cursor = 0;
  auto entry_ws = [&](const Schedule &sc, int k) { return schedule_ws(sc, k, &cursor); };
  p.outputs_per_pass = opp;
  p.chunks.clear();
  p.pass_chunk_begin.clear();
  if (n > 0) {  // windows advance monotonically: the last pass's span bounds the chunk count per pass well enough
    const size_t n_passes = ((size_t) n + opp - 1) / opp;
    const long long span = (long long) entry_ws(s, n - 1) - entry_ws(s, 0);
    const size_t per_pass = (size_t) ((span / (long long) n_passes + taps) / chunk_rows + 4);
    p.chunks.reserve(n_passes * per_pass);
    p.pass_chunk_begin.reserve(n_passes + 1);
  }
  p.pass_chunk_begin.push_back(0);
  for (int first = 0, pass = 0; first < n; first += opp, ++pass) {
    const int last = (first + opp < n ? first + opp : n) - 1;
    const int j0 = entry_ws(s, first), j1 = entry_ws(s, last) + taps;
    for (int j = j0; j < j1; j += chunk_rows)
      p.chunks.push_back(ChunkEntry{j, pass});
    p.pass_chunk_begin.push_back((int32_t) p.chunks.size());
  }
}

void design_lowpass(BiquadCoeffs *c, double frequency) {
  const double pi = 3.14159265358979323846;
  const double q = sqrt(0.5), k = tan(pi * frequency);
  const double norm = 1.0 / (1.0 + k / q + k * k);
  c->a0 = (float) (k * k * norm);
  c->a1 = 2 * c->a0;
  c->a2 = c->a0;
  c->b1 = (float) (2.0 * (k * k - 1.0) * norm);
  c->b2 = (float) ((1.0 - k / q + k * k) * norm);
}

void design_highpass(BiquadCoeffs *c, double frequency) {
  const double pi = 3.14159265358979323846;
  const double q = sqrt(0.5), k = tan(pi * frequency);
  const double norm = 1.0 / (1.0 + k / q + k * k);
  c->a0 = (float) norm;
  c->a1 = (float) (-2.0 * norm);
  c->a2 = c->a0;
  c->b1 = (float) (2.0 * (k * k - 1.0) * norm);
  c->b2 = (float) ((1.0 - k / q + k * k) * norm);
}

void decide_policy(float src_rate, float dst_rate, int taps, bool use_filter, bool interpolate, WrapperPolicy *p) {
  *p = WrapperPolicy{};
  if (src_rate == dst_rate)
    return;
  p->resampling = true;
  const int flags = interpolate ? kFlagInterpolate : 0;
  p->sample_ratio = dst_rate / src_rate;
  if (p->sample_ratio < 1.0f) {
    p->lowpass_ratio -= (10.24f / (float) taps);
    if (p->lowpass_ratio < 0.84f)
      p->lowpass_ratio = 0.84f;
    if (p->lowpass_ratio < p->sample_ratio)
      p->lowpass_ratio = p->sample_ratio;
  }
  if (p->lowpass_ratio * p->sample_ratio < 0.98f && use_filter) {
    const float cutoff = p->lowpass_ratio * p->sample_ratio / 2.0f;
    design_lowpass(&p->coeffs, cutoff);
    p->pre = true;
  }
  if (p->lowpass_ratio / p->sample_ratio < 0.98f && use_filter && !p->pre) {
    const float cutoff = p->lowpass_ratio / p->sample_ratio / 2.0f;
    design_lowpass(&p->coeffs, cutoff);
    p->post = true;
  }
  if (p->sample_ratio < 1.0f) {
    p->art_lowpass = p->sample_ratio * p->lowpass_ratio;
    p->art_flags = flags | kFlagLowpass;
  } else if (p->lowpass_ratio < 1.0f) {
    p->art_lowpass = p->lowpass_ratio;
    p->art_flags = flags | kFlagLowpass;
  } else {
    p->art_lowpass = 1.0f;
    p->art_flags = flags;
  }
}

float q2f_gain_factor(int bits, float gain_db) {
  const float gain = powf(10.0f, gain_db / 20.0f);
  if (bits <= 8)
    return gain / 128.0f;
  if (bits <= 16)
    return gain / 32768.0f;
  if (bits <= 24)
    return gain / 8388608.0f;
  return gain / 2147483648.0f;
}

}  // namespace espb
