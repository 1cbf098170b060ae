"""TEST INFRASTRUCTURE — generates tests/golden/*.npz from the UNMODIFIED reference.

Run in the build container (needs oracle/_ref, i.e. /root/reference present):
    python oracle/gen_golden.py
Every array written here is an output of the real reference library
(oracle/_ref/libesp_audio_ref.so, built by oracle/Makefile from /root/reference),
never of the oracle port or of the CUDA path.  Inputs drawn from the seeded
generators in tests/signals.py are stored as their recipe and SHA-256 digest
(meta "inputs"; tests/conftest.py regenerates them), other inputs next to the
outputs; the large cases store SHA-256 digests, frame counts and final state,
with inputs regenerated from the same generators (an input digest guards
against generator drift).
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle_lib import BLACKMAN_HARRIS, INCLUDE_LOWPASS, SUBSAMPLE_INTERPOLATE, Reference, noise  # noqa: E402
from signals import from_recipe  # noqa: E402

R = Reference()
OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
f32 = np.float32


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


arrays, meta = {}, {"inputs": {}}


def seeded_input(name, **recipe):
    """A signal of tests/signals.py: stored as its recipe and digest (tests/conftest.py regenerates it), not as data."""
    x = from_recipe(recipe)
    meta["inputs"][name] = dict(recipe, sha256=sha(x))
    return x

# ---- 1. filter banks ---------------------------------------------------------
BANKS = [  # taps, filters, lowpass, flags
    (256, 256, 1.0, SUBSAMPLE_INTERPOLATE | BLACKMAN_HARRIS),
    (256, 256, float(f32(44100) / f32(48000) * f32(0.96)), SUBSAMPLE_INTERPOLATE),
    (1024, 256, float(f32(44100) / f32(96000) * (f32(1.0) - f32(10.24) / f32(1024))), SUBSAMPLE_INTERPOLATE),
    (1024, 1024, 0.45, SUBSAMPLE_INTERPOLATE | BLACKMAN_HARRIS),
    (32, 16, 1.0, 0),
    (4, 2, 0.5, BLACKMAN_HARRIS),
    (64, 1024, 1.0, BLACKMAN_HARRIS),
]
meta["banks"] = []
for k, (taps, filters, lp, flags) in enumerate(BANKS):
    ctx = R.resampler(1, taps, filters, lp, flags)
    bank = ctx.bank()
    meta["banks"].append(dict(taps=taps, filters=filters, lowpass=lp, flags=flags, eff_flags=ctx.flags(),
                              sha256=sha(bank), centre=float(bank[0, taps // 2 - 1]),
                              next=float(bank[0, taps // 2]), sum0=float(bank[0].astype(np.float64).sum())))
    if taps <= 32:
        arrays[f"bank{k}"] = bank
    else:  # a few rows of the big ones
        arrays[f"bank{k}_rows"] = bank[[0, 1, filters // 2, filters]]

# ---- 2. small fully-stored resampler cases ------------------------------------
SMALL = [  # name, channels, taps, filters, lowpass, flags, ratio, n_in, advance, signal
    ("up_441_48_bh", 2, 256, 256, 1.0, 3, f32(48000) / f32(44100), 3000, 128.0, "multitone"),
    ("down_48_441_lp", 2, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 3000,
     128.0, "noise"),
    ("up3_mono_hann", 1, 256, 256, 1.0, 1, f32(3.0), 1200, 128.0, "noise"),
    ("down_96_441_t1024", 8, 1024, 256, float(f32(44100) / f32(96000) * (f32(1.0) - f32(10.24) / f32(1024))), 1,
     f32(44100) / f32(96000), 2600, 512.0, "noise"),
    ("nointerp_t32", 3, 32, 16, 1.0, 0, f32(1.37), 700, 0.0, "noise"),
    ("nointerp_lp_t64", 2, 64, 64, 0.7, BLACKMAN_HARRIS, f32(0.75), 900, 32.0, "multitone"),
    ("unity_t16", 1, 16, 8, 1.0, 3, f32(1.0), 400, 8.0, "noise"),
    ("tiny_t4", 2, 4, 2, 1.0, 1, f32(2.5), 300, 2.0, "noise"),
    ("ring_rebase_t8", 1, 8, 32, 1.0, 3, f32(1.3), 1000, 4.0, "noise"),
]
meta["small"] = []
for name, ch, taps, filters, lp, flags, ratio, n_in, adv, sig in SMALL:
    if sig == "multitone":
        x = seeded_input(f"small_{name}_x", signal=sig, frames=n_in, channels=ch, stream=5, amp=0.9, fs=44100.0)
    else:
        x = seeded_input(f"small_{name}_x", signal=sig, frames=n_in, channels=ch, stream=11, amp=0.9)
    ctx = R.resampler(ch, taps, filters, lp, flags)
    if adv:
        ctx.advance(adv)
    cap = int(n_in * float(ratio)) + 64
    y, used, gen = ctx.process_interleaved(x, cap, ratio)
    off, idx = ctx.state()
    arrays[f"small_{name}_y"] = y
    meta["small"].append(dict(name=name, channels=ch, taps=taps, filters=filters, lowpass=lp, flags=flags,
                              ratio=float(ratio), n_in=n_in, advance=adv, cap=cap, used=used, generated=gen,
                              final_offset=float(off), final_index=idx, position=ctx.position()))

# chunked == one-shot (KAT 7) and output-capacity-limited calls: store the chunk plan + per-call results
rng = np.random.default_rng(2024)
ch, taps, filters, ratio = 2, 64, 64, f32(48000) / f32(44100)
x = seeded_input("chunked_x", signal="noise", frames=6000, channels=ch, stream=2, amp=0.8)
ctx = R.resampler(ch, taps, filters, 1.0, 3)
ctx.advance(taps / 2)
plan, outs, pos = [], [], 0
while pos < 6000:
    n_in = int(min(rng.integers(0, 700), 6000 - pos))
    n_out = int(rng.integers(0, 900))
    y, used, gen = ctx.process_interleaved(x[pos * ch:(pos + n_in) * ch], n_out, ratio, n_in=n_in)
    plan.append((n_in, n_out, used, gen))
    outs.append(y)
    pos += used
arrays["chunked_plan"] = np.array(plan, np.int64)
arrays["chunked_y"] = np.concatenate(outs)
meta["chunked"] = dict(channels=ch, taps=taps, filters=filters, ratio=float(ratio), flags=3, advance=taps / 2)

# planar entry point
ctx = R.resampler(3, 32, 32, 1.0, 3)
xp = noise(500, 3, stream=4, amp=0.7).reshape(500, 3).T.copy()
yp, used, gen = ctx.process_planar(xp, 800, f32(1.25))
arrays["planar_x"], arrays["planar_y"] = xp, yp
meta["planar"] = dict(channels=3, taps=32, filters=32, ratio=1.25, flags=3, used=used, generated=gen)

# ---- 3. large cases: counts, final state, digests (BASELINE.json configs, 1 s / 10 s units) ----
LARGE = [  # name, ch, taps, filters, lowpass, flags, ratio, n_in
    ("C1_10s", 2, 256, 256, 1.0, 3, f32(48000) / f32(44100), 441000),
    ("C3_unit_10s", 1, 256, 256, 1.0, 1, f32(48000) / f32(16000), 160000),
    ("C4_unit_1s", 8, 1024, 256, float(f32(44100) / f32(96000) * (f32(1.0) - f32(10.24) / f32(1024))), 1,
     f32(44100) / f32(96000), 96000),
    ("C5_unit_10s", 2, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 480000),
]
meta["large"] = []
for name, ch, taps, filters, lp, flags, ratio, n_in in LARGE:
    x = noise(n_in, ch, stream=1, amp=0.5)
    ctx = R.resampler(ch, taps, filters, lp, flags)
    ctx.advance(taps / 2)
    cap = int(n_in * float(ratio)) + 256
    y, used, gen = ctx.process_interleaved(x, cap, ratio)
    off, idx = ctx.state()
    meta["large"].append(dict(name=name, channels=ch, taps=taps, filters=filters, lowpass=lp, flags=flags,
                              ratio=float(ratio), n_in=n_in, cap=cap, used=used, generated=gen,
                              final_offset=float(off), final_index=idx, x_sha256=sha(x), y_sha256=sha(y),
                              y_head=[float(v) for v in y[:8]], y_tail=[float(v) for v in y[-8:]]))

# schedule KATs (SURVEY.md §8c (2)): 1/ratio and first offsets
meta["kat"] = dict(inv_ratio_441_48=float(f32(1.0) / (f32(48000) / f32(44100))))

# ---- 4. quantisers ---------------------------------------------------------------
rng = np.random.default_rng(77)
meta["quant"] = []
for bits in (8, 12, 16, 20, 24, 32):
    nb = (bits + 7) // 8
    n = 4096
    raw = rng.integers(0, 256, size=n * nb, dtype=np.uint8)
    for gain in (0.0, -6.5):
        arrays[f"q2f_{bits}_{gain}"] = R.quantized_to_float(raw, n, bits, gain)
    arrays[f"q2f_{bits}_raw"] = raw
    x = (rng.random(n) * 2.6 - 1.3).astype(f32)
    edge = np.array([0, 1, -1, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768, np.nextafter(f32(1), f32(0)), -1.0000001,
                     0.99999, -0.99999, 1e-9, -1e-9], f32)
    x[:edge.size] = edge
    q, clipped = R.float_to_quantized(x, bits)
    arrays[f"f2q_{bits}_x"], arrays[f"f2q_{bits}_q"] = x, q
    meta["quant"].append(dict(bits=bits, clipped=clipped))
q, clipped = R.float_to_quantized(np.array([0, 1, -1, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768], f32), 16)
meta["kat"]["f2q16"] = dict(values=[int(v) for v in q.view(np.int16)], clipped=clipped)
meta["kat"]["q2f32_quirk"] = float(R.quantized_to_float(np.array([0, 0, 0x80, 1], np.uint8), 1, 32)[0])

# ---- 5. biquad --------------------------------------------------------------------
meta["biquad"] = []
x = seeded_input("biquad_x", signal="noise", frames=4000, channels=2, stream=9, amp=0.9)
for k, (kind, f, gain) in enumerate([("lp", 0.2274, 1.0), ("lp", 1.0 / 6.0, 1.0), ("lp", 0.441, 0.5),
                                     ("lp", 0.02, 1.0), ("hp", 0.1, 1.0), ("hp", 0.3, 2.0)]):
    c = R.biquad_lowpass(f) if kind == "lp" else R.biquad_highpass(f)
    y = x.copy()
    for chn in range(2):  # two cascaded sections per channel, like resampler.cpp:126-133
        s0, s1 = R.biquad(c, gain), R.biquad(c, gain)
        s0.apply_buffer(y[chn:], 2, n=4000)
        s1.apply_buffer(y[chn:], 2, n=4000)
    arrays[f"biquad_{k}_c"], arrays[f"biquad_{k}_y"] = c, y
    meta["biquad"].append(dict(kind=kind, f=f, gain=gain, hex=[float(v).hex() for v in c]))
# first-order section (a2 == b2 == 0) through the public init
c1 = np.array([0.25, 0.25, 0.0, -0.5, 0.0], f32)
s = R.biquad(c1, 1.0)
arrays["biquad_fo_c"], arrays["biquad_fo_y"] = c1, s.apply_buffer(x[:2000].copy(), 1)

# ---- 6. Resampler wrapper, chunked -----------------------------------------------
meta["wrapper"] = []
rng = np.random.default_rng(5)
for k, (sr, dr, sb, db, chn, use_f, interp, taps, filters, gain) in enumerate([
        (16000, 48000, 16, 16, 1, 1, 1, 256, 256, 0.0),
        (44100, 48000, 16, 24, 2, 1, 1, 256, 256, -3.0),
        (48000, 44100, 24, 16, 2, 1, 1, 256, 256, 0.0),
        (96000, 44100, 32, 32, 2, 1, 1, 64, 64, -1.0),
        (48000, 48000, 16, 8, 2, 1, 1, 32, 32, 0.0),
        (44100, 48000, 16, 16, 2, 0, 0, 32, 32, 2.0)]):
    nb = (sb + 7) // 8
    w = R.wrapper(1024 * chn, 4096 * chn, float(sr), float(dr), sb, db, chn, use_f, interp, taps, filters)
    # band-limited-ish PCM so clipping is rare but present
    pcm = (rng.normal(0, 0.35, size=1024 * 3 * chn).clip(-1, 0.99999) * (2 ** (8 * nb - 1))).astype(np.int64)
    raw = np.zeros(pcm.size * nb, np.uint8)
    for b in range(nb):
        raw[b::nb] = (pcm >> (8 * b)) & 0xFF
    outs, res = [], []
    for it in range(3):
        y, r = w.resample(raw[it * 1024 * chn * nb:(it + 1) * 1024 * chn * nb], 1024, 4096 if it != 1 else 700, gain)
        outs.append(y)
        res.append([r["frames_used"], r["frames_generated"], r["predicted_frames_used"], r["clipped_samples"]])
    arrays[f"wrap_{k}_raw"], arrays[f"wrap_{k}_y"] = raw, np.concatenate(outs)
    arrays[f"wrap_{k}_res"] = np.array(res, np.int64)
    meta["wrapper"].append(dict(src_rate=sr, dst_rate=dr, src_bits=sb, dst_bits=db, channels=chn, use_filter=use_f,
                                interpolate=interp, taps=taps, filters=filters, gain_db=gain,
                                out_free=[4096, 700, 4096]))

np.savez_compressed(os.path.join(OUT, "golden_v1.npz"), **arrays)
with open(os.path.join(OUT, "golden_v1.json"), "w") as fh:
    json.dump(meta, fh, indent=1, sort_keys=True)
print("wrote", len(arrays), "arrays;", os.path.getsize(os.path.join(OUT, "golden_v1.npz")) // 1024, "KiB")
