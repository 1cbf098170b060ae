"""TEST INFRASTRUCTURE — ctypes bindings for the two CPU checkers.

`Oracle`  : oracle/libart_oracle.so  (plain-C restatement, oracle/art_oracle.c)
`Reference`: oracle/_ref/libesp_audio_ref.so (the unmodified reference compiled from
            /root/reference by oracle/Makefile; may be absent)

Both expose the same Python surface so tests can run the same case through either.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs import this module.  The product package never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "libart_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libesp_audio_ref.so")

SUBSAMPLE_INTERPOLATE = 0x1
BLACKMAN_HARRIS = 0x2
INCLUDE_LOWPASS = 0x4

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS")


def build_oracle():
    """Compile the checkers (building the checker is not using it)."""
    subprocess.run(["make", "-s", "-f", os.path.join(ROOT, "oracle", "Makefile")], check=True, cwd=ROOT)


def _bind(lib, prefix, names):
    """names: pythonic name -> (symbol suffix, restype, argtypes)"""
    out = {}
    for key, (sym, res, args) in names.items():
        fn = getattr(lib, prefix + sym)
        fn.restype = res
        fn.argtypes = args
        out[key] = fn
    return out


class _Backend:
    """Common surface; subclasses fill self.f with bound functions."""

    name = "?"

    # ---- ART resampler ----
    def resampler(self, channels, taps, filters, lowpass, flags, fused=False):
        """fused=True: every dot product is an fmaf chain in tap order, the library's fast mode (oracle only)."""
        self._check_fused(fused)
        h = self.f["init"](channels, taps, filters, lowpass, flags)
        if h and fused:
            self.lib.orc_resample_set_fused(h, 1)
        return ArtContext(self, h, channels, taps, filters) if h else None

    def _check_fused(self, fused):
        if fused:
            raise ValueError(f"{self.name}: fused=True needs the oracle (the reference has no fused form)")

    # ---- quantisers ----
    def quantized_to_float(self, data, n, bits, gain_db=0.0):
        data = np.ascontiguousarray(data, np.uint8)
        out = np.empty(n, np.float32)
        self.f["q2f"](data, out, n, bits, gain_db)
        return out

    def float_to_quantized(self, x, bits):
        x = np.ascontiguousarray(x, np.float32)
        nbytes = (bits + 7) // 8
        out = np.zeros(x.size * nbytes, np.uint8)
        clipped = self.f["f2q"](x, out, x.size, bits)
        return out, int(clipped)

    # ---- biquad ----
    def biquad_lowpass(self, f):
        c = np.zeros(5, np.float32)
        self.f["bq_lowpass"](c, f)
        return c

    def biquad_highpass(self, f):
        c = np.zeros(5, np.float32)
        self.f["bq_highpass"](c, f)
        return c

    def biquad(self, coeffs, gain=1.0):
        return BiquadState(self, np.ascontiguousarray(coeffs, np.float32), gain)

    # ---- wrapper ----
    def wrapper(self, in_samples, out_samples, src_rate, dst_rate, src_bits, dst_bits, channels, use_filter=True,
                interpolate=True, taps=256, filters=256, fused=False):
        """fused=True: the wrapper's resampler runs the fmaf chain (see resampler())."""
        self._check_fused(fused)
        h = self.f["w_create"](in_samples, out_samples, src_rate, dst_rate, src_bits, dst_bits, channels,
                               int(use_filter), int(interpolate), taps, filters)
        if h and fused:
            self.lib.orc_wrapper_set_fused(h, 1)
        return WrapperContext(self, h, channels, src_bits, dst_bits) if h else None

    # ---- Q15 helpers ----
    def add_s16(self, a, b, n, step1=1, step2=1, step_out=1, shift=0):
        a, b = np.ascontiguousarray(a, np.int16), np.ascontiguousarray(b, np.int16)
        out = np.zeros(max(n * step_out, 1), np.int16)
        rc = self.f["add_s16"](a, b, out, n, step1, step2, step_out, shift)
        return out, rc

    def mulc_s16(self, a, n, c, step_in=1, step_out=1):
        a = np.ascontiguousarray(a, np.int16)
        out = np.zeros(max(n * step_out, 1), np.int16)
        rc = self.f["mulc_s16"](a, out, n, c, step_in, step_out)
        return out, rc

    # ---- WAV header parser ----
    def wav(self):
        return WavContext(self)

    def bench_resample(self, n_threads, channels, taps, filters, lowpass, flags, advance, x, n_out, ratio):
        """x: (n_streams, n_in*channels) float32.  Returns (seconds, frames_generated, out)."""
        x = np.ascontiguousarray(x, np.float32)
        n_streams, row = x.shape
        n_in = row // channels
        out = np.zeros((n_streams, n_out * channels), np.float32)
        gen = C.c_ulonglong(0)
        secs = self.f["bench"](n_streams, n_threads, channels, taps, filters, lowpass, flags, advance, x, row, n_in,
                               out, n_out * channels, n_out, ratio, C.byref(gen))
        return secs, int(gen.value), out


class ArtContext:
    def __init__(self, be, handle, channels, taps, filters):
        self.be, self.h, self.channels, self.taps, self.filters = be, handle, channels, taps, filters

    def __del__(self):
        if getattr(self, "h", None):
            self.be.f["free"](self.h)
            self.h = None

    def reset(self):
        self.be.f["reset"](self.h)

    def advance(self, delta):
        self.be.f["advance"](self.h, delta)

    def position(self):
        return float(self.be.f["position"](self.h))

    def required(self, n_out, ratio):
        return int(self.be.f["required"](self.h, n_out, ratio))

    def expected(self, n_in, ratio):
        return int(self.be.f["expected"](self.h, n_in, ratio))

    def flags(self):
        return int(self.be.f["flags"](self.h))

    def state(self):
        off, idx = C.c_float(0), C.c_int(0)
        self.be.f["state"](self.h, C.byref(off), C.byref(idx))
        return np.float32(off.value), int(idx.value)

    def bank(self):
        out = np.empty((self.filters + 1, self.taps), np.float32)
        row = np.empty(self.taps, np.float32)
        for i in range(self.filters + 1):
            self.be.f["copy_filter"](self.h, i, row)
            out[i] = row
        return out

    def process_interleaved(self, x, n_out, ratio, n_in=None):
        """x: float32 (n_in*channels,) interleaved.  Returns (out[:gen*ch], used, generated)."""
        x = np.ascontiguousarray(x, np.float32).reshape(-1)
        if n_in is None:
            n_in = x.size // self.channels
        out = np.zeros(max(n_out, 1) * self.channels, np.float32)
        used, gen = C.c_uint(0), C.c_uint(0)
        xin = x if x.size else np.zeros(1, np.float32)
        self.be.f["interleaved"](self.h, xin, n_in, out, n_out, ratio, C.byref(used), C.byref(gen))
        return out[: gen.value * self.channels].copy(), int(used.value), int(gen.value)

    def process_planar(self, x, n_out, ratio):
        """x: float32 (channels, n_in).  Returns (out (channels, gen), used, generated)."""
        x = np.ascontiguousarray(x, np.float32)
        ch, n_in = x.shape
        out = np.zeros((ch, max(n_out, 1)), np.float32)
        ptr_t = C.POINTER(C.c_float) * ch
        inp = ptr_t(*[x[c].ctypes.data_as(C.POINTER(C.c_float)) for c in range(ch)])
        outp = ptr_t(*[out[c].ctypes.data_as(C.POINTER(C.c_float)) for c in range(ch)])
        used, gen = C.c_uint(0), C.c_uint(0)
        self.be.f["planar"](self.h, inp, n_in, outp, n_out, ratio, C.byref(used), C.byref(gen))
        return out[:, : gen.value].copy(), int(used.value), int(gen.value)


class BiquadState:
    def __init__(self, be, coeffs, gain):
        self.be = be
        self.buf = C.create_string_buffer(64)
        be.f["bq_init"](self.buf, coeffs, gain)

    def apply_buffer(self, x, stride=1, n=None):
        x = np.ascontiguousarray(x, np.float32)
        if n is None:
            n = x.size // stride
        self.be.f["bq_apply"](self.buf, x, n, stride)
        return x

    def apply_sample(self, v):
        return np.float32(self.be.f["bq_sample"](self.buf, v))


class WrapperContext:
    def __init__(self, be, handle, channels, src_bits, dst_bits):
        self.be, self.h, self.channels = be, handle, channels
        self.src_bytes, self.dst_bytes = (src_bits + 7) // 8, (dst_bits + 7) // 8

    def __del__(self):
        if getattr(self, "h", None):
            self.be.f["w_free"](self.h)
            self.h = None

    def resample(self, data, in_frames, out_free, gain_db=0.0):
        data = np.ascontiguousarray(data, np.uint8)
        out = np.zeros(max(out_free, 1) * self.channels * self.dst_bytes, np.uint8)
        res = (C.c_uint64 * 4)()
        self.be.f["w_resample"](self.h, data if data.size else np.zeros(1, np.uint8), out, in_frames, out_free,
                                gain_db, res)
        used, gen, pred, clipped = (int(v) for v in res)
        return out[: gen * self.channels * self.dst_bytes].copy(), dict(
            frames_used=used, frames_generated=gen, predicted_frames_used=pred, clipped_samples=clipped)


_vp, _i, _f, _u = C.c_void_p, C.c_int, C.c_float, C.c_uint
_pu = C.POINTER(C.c_uint)
_BENCH_ARGS = [_i, _i, _i, _i, _i, _f, _i, _f, _f32p, C.c_size_t, _i, _f32p, C.c_size_t, _i, _f,
               C.POINTER(C.c_ulonglong)]
_W_ARGS = [C.c_size_t, C.c_size_t, _f, _f, _i, _i, _i, _i, _i, _i, _i]


def _table(n):
    """symbol names per backend: n maps logical name -> suffix"""
    pp = C.POINTER(C.POINTER(C.c_float))
    return {
        "init": (n["init"], _vp, [_i, _i, _i, _f, _i]),
        "free": (n["free"], None, [_vp]),
        "reset": (n["reset"], None, [_vp]),
        "advance": (n["advance"], None, [_vp, _f]),
        "position": (n["position"], _f, [_vp]),
        "required": (n["required"], _u, [_vp, _i, _f]),
        "expected": (n["expected"], _u, [_vp, _i, _f]),
        "interleaved": (n["interleaved"], None, [_vp, _f32p, _i, _f32p, _i, _f, _pu, _pu]),
        "planar": (n["planar"], None, [_vp, pp, _i, pp, _i, _f, _pu, _pu]),
        "flags": (n["flags"], _i, [_vp]),
        "copy_filter": (n["copy_filter"], None, [_vp, _i, _f32p]),
        "state": (n["state"], None, [_vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
        "bq_lowpass": (n["bq_lowpass"], None, [_f32p, C.c_double]),
        "bq_highpass": (n["bq_highpass"], None, [_f32p, C.c_double]),
        "bq_init": (n["bq_init"], None, [C.c_char_p, _f32p, _f]),
        "bq_apply": (n["bq_apply"], None, [C.c_char_p, _f32p, _i, _i]),
        "bq_sample": (n["bq_sample"], _f, [C.c_char_p, _f]),
        "q2f": (n["q2f"], None, [_u8p, _f32p, C.c_uint32, C.c_uint8, _f]),
        "f2q": (n["f2q"], C.c_uint32, [_f32p, _u8p, C.c_uint32, C.c_uint8]),
        "w_create": (n["w_create"], _vp, _W_ARGS),
        "w_free": (n["w_free"], None, [_vp]),
        "w_resample": (n["w_resample"], None, [_vp, _u8p, _u8p, C.c_size_t, C.c_size_t, _f,
                                               C.POINTER(C.c_uint64)]),
        "bench": (n["bench"], C.c_double, _BENCH_ARGS),
        "add_s16": (n["add_s16"], _i, [_i16p, _i16p, _i16p, _i, _i, _i, _i, _i]),
        "mulc_s16": (n["mulc_s16"], _i, [_i16p, _i16p, _i, C.c_int16, _i, _i]),
    }


class WavContext:
    """WAVDecoder handle of a backend; snapshot() = (state, processed, needed, skip, chunk_left, rate, channels,
    bits, chunk_name)."""

    def __init__(self, backend):
        self.L, self.pre = backend.lib, backend.prefix
        g = lambda n: getattr(self.L, self.pre + "wav_" + n)  # noqa: E731
        g("create").restype = _vp
        g("create").argtypes = []
        g("free").argtypes = [_vp]
        g("next").restype = _i
        g("next").argtypes = [_vp, _u8p]
        g("decode_header").restype = _i
        g("decode_header").argtypes = [_vp, _u8p, C.c_size_t]
        g("reset").argtypes = [_vp]
        g("snapshot").argtypes = [_vp, C.POINTER(C.c_uint64), C.c_char_p]
        self.g = g
        self.h = g("create")()

    def decode_header(self, data):
        buf = np.frombuffer(bytes(data), np.uint8) if len(data) else np.zeros(1, np.uint8)
        return self.g("decode_header")(self.h, np.ascontiguousarray(buf), len(data))

    def next(self, data):
        return self.g("next")(self.h, np.frombuffer(bytes(data) + b"\0" * 16, np.uint8).copy())

    def reset(self):
        self.g("reset")(self.h)

    def snapshot(self):
        out = (C.c_uint64 * 8)()
        name = C.create_string_buffer(5)
        self.g("snapshot")(self.h, out, name)
        return tuple(int(v) for v in out) + (name.raw[:4],)

    def __del__(self):
        try:
            self.g("free")(self.h)
        except Exception:
            pass


class Oracle(_Backend):
    name = "oracle-port"
    prefix = "orc_"

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            build_oracle()
        self.lib = C.CDLL(ORACLE_SO)
        names = dict(init="resample_init", free="resample_free", reset="resample_reset", advance="resample_advance",
                     position="resample_position", required="resample_required", expected="resample_expected",
                     interleaved="resample_interleaved", planar="resample_planar", flags="resample_flags",
                     copy_filter="resample_copy_filter", state="resample_state", bq_lowpass="biquad_lowpass",
                     bq_highpass="biquad_highpass", bq_init="biquad_init", bq_apply="biquad_apply_buffer",
                     bq_sample="biquad_apply_sample", q2f="quantized_to_float", f2q="float_to_quantized",
                     w_create="wrapper_create", w_free="wrapper_free", w_resample="wrapper_resample",
                     bench="bench_resample", add_s16="add_s16", mulc_s16="mulc_s16")
        self.f = _bind(self.lib, "orc_", _table(names))
        self.lib.orc_wrapper_policy.restype = _i
        self.lib.orc_wrapper_policy.argtypes = [_vp, _f32p, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                                C.POINTER(C.c_int)]
        for fn in (self.lib.orc_resample_set_fused, self.lib.orc_wrapper_set_fused):
            fn.restype = None
            fn.argtypes = [_vp, _i]

    def _check_fused(self, fused):
        pass

    def wrapper_policy(self, w):
        coeffs = np.zeros(5, np.float32)
        ratio, lp, flags = C.c_float(0), C.c_float(0), C.c_int(0)
        kind = self.lib.orc_wrapper_policy(w.h, coeffs, C.byref(ratio), C.byref(lp), C.byref(flags))
        return dict(filter={0: "none", 1: "pre", 2: "post"}[kind], coeffs=coeffs, sample_ratio=np.float32(ratio.value),
                    art_lowpass=np.float32(lp.value), art_flags=int(flags.value))


class Reference(_Backend):
    name = "reference"
    prefix = "ref_"

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO)
        self.lib = C.CDLL(REF_SO)
        names = dict(init="resampleInit", free="resampleFree", reset="resampleReset",
                     advance="resampleAdvancePosition", position="resampleGetPosition",
                     required="resampleGetRequiredSamples", expected="resampleGetExpectedOutput",
                     interleaved="resampleProcessInterleaved", planar="resampleProcess", flags="resampleFlags",
                     copy_filter="resampleCopyFilter", state="resampleState", bq_lowpass="biquad_lowpass",
                     bq_highpass="biquad_highpass", bq_init="biquad_init", bq_apply="biquad_apply_buffer",
                     bq_sample="biquad_apply_sample", q2f="quantized_to_float", f2q="float_to_quantized",
                     w_create="wrapper_create", w_free="wrapper_free", w_resample="wrapper_resample",
                     bench="bench_resample", add_s16="add_s16", mulc_s16="mulc_s16")
        self.f = _bind(self.lib, "ref_", _table(names))


def have_reference():
    return os.path.exists(REF_SO)


# Synthetic signals (SURVEY.md §8d) live in tests/signals.py (no oracle involved); re-exported for the tests.
from signals import multitone, noise  # noqa: E402,F401

DYADIC_K = (-14, 0)  # exponents of dyadic(): every bank entry times 2^k stays a normal float32


def dyadic(frames, channels, stream, kmin=DYADIC_K[0], kmax=DYADIC_K[1]):
    """Interleaved float32 samples s * 2^k, s in {-1, -0, +0, +1}, k in [kmin, kmax], seeded by `stream`.  Every
    product of such a sample with a filter tap is exact in FP32, so a multiply-add rounds the same fused or not: on
    this input the fused (fast-mode) and plain (exact-mode) dot products give the same bits."""
    rng = np.random.default_rng(0xD1AD1C + stream)
    n = frames * channels
    s = rng.choice(np.array([-1.0, -0.0, 0.0, 1.0]), size=n, p=[0.4, 0.1, 0.1, 0.4])
    return (s * np.ldexp(1.0, rng.integers(kmin, kmax + 1, size=n))).astype(np.float32)
