"""Oracle port vs the unmodified reference on seeded random cases beyond the committed fixtures.

Each case is recorded as what a caller observes (counts, state, SHA-256 of every output buffer) and compared with
the reference's record frozen in tests/golden/golden_random.json, so the comparison runs without the reference.
The frozen records were written by the oracle port; at commit 3e4b2c7 these same cases passed bit for bit against
the compiled reference (oracle/_ref), and neither the port nor the cases have changed since.  Where oracle/_ref
exists, `python tests/test_oracle_vs_reference.py` rewrites the file from the reference itself."""
import hashlib
import json
import os

import numpy as np
import pytest
from oracle_lib import noise

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "golden_random.json")
f32 = np.float32


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def record_resampler(be):
    rng = np.random.default_rng(99)
    out = []
    for _ in range(25):
        taps = int(rng.choice([4, 8, 16, 32, 64, 128, 256, 512]))
        filters = int(rng.integers(2, 300))
        flags = int(rng.integers(0, 4))
        lp = float(rng.choice([1.0, 0.9, 0.5, 0.31]))
        ch = int(rng.integers(1, 5))
        ratio = f32(rng.uniform(0.3, 3.5))
        n_in = int(rng.integers(1, 3000))
        x = noise(n_in, ch, stream=int(rng.integers(0, 1000)), amp=0.9)
        ctx = be.resampler(ch, taps, filters, lp, flags)
        adv = float(rng.choice([0.0, taps / 2, 3.25]))
        ctx.advance(adv)
        case = dict(taps=taps, filters=filters, flags=flags, lowpass=lp, channels=ch, ratio=float(ratio), n_in=n_in,
                    advance=adv, bank=sha(ctx.bank()), calls=[])
        pos = 0
        while pos < n_in:
            ci, co = int(rng.integers(0, 900)), int(rng.integers(0, 1200))
            ci = min(ci, n_in - pos)
            req, exp = ctx.required(co, ratio), ctx.expected(ci, ratio)
            y, used, gen = ctx.process_interleaved(x[pos * ch:(pos + ci) * ch], co, ratio, n_in=ci)
            off, idx = ctx.state()
            case["calls"].append([ci, co, req, exp, used, gen, sha(y), float(off), idx, ctx.position()])
            pos += used
        out.append(case)
    return out


def record_quantisers(be):
    rng = np.random.default_rng(3)
    out = []
    for bits in range(1, 33):
        nb = (bits + 7) // 8
        raw = rng.integers(0, 256, size=3000 * nb, dtype=np.uint8)
        g = float(rng.uniform(-12, 6))
        x = (rng.random(3000) * 2.2 - 1.1).astype(f32)
        q, clipped = be.float_to_quantized(x, bits)
        out.append(dict(bits=bits, q2f=sha(be.quantized_to_float(raw, 3000, bits, g)), f2q=sha(q), clipped=clipped))
    return out


def record_biquad(be):
    rng = np.random.default_rng(4)
    out = []
    for _ in range(20):
        f = float(rng.uniform(0.001, 0.49))
        lowpass, highpass = be.biquad_lowpass(f), be.biquad_highpass(f)
        c = lowpass if rng.random() < 0.5 else highpass
        stride = int(rng.integers(1, 5))
        x = noise(2000, stride, stream=7, amp=1.0)
        gain = float(rng.uniform(0.1, 2.0))
        y = be.biquad(c, gain).apply_buffer(x.copy(), stride)
        out.append(dict(f=f, lowpass=sha(lowpass), highpass=sha(highpass), stride=stride, gain=gain, y=sha(y)))
    return out


def record_wrapper(be):
    rng = np.random.default_rng(5)
    rates = [8000, 16000, 22050, 32000, 44100, 48000, 96000]
    out = []
    for _ in range(12):
        sr, dr = float(rng.choice(rates)), float(rng.choice(rates))
        sb, db = int(rng.choice([8, 16, 24, 32])), int(rng.choice([8, 16, 24, 32]))
        ch = int(rng.integers(1, 3))
        taps, filters = int(rng.choice([16, 32, 64])), int(rng.choice([16, 64]))
        use_f, interp = int(rng.integers(0, 2)), int(rng.integers(0, 2))
        w = be.wrapper(512 * ch, 4096 * ch, sr, dr, sb, db, ch, use_f, interp, taps, filters)
        nb = (sb + 7) // 8
        case = dict(src_rate=sr, dst_rate=dr, src_bits=sb, dst_bits=db, channels=ch, taps=taps, filters=filters,
                    use_filter=use_f, interpolate=interp, calls=[])
        for _it in range(4):
            raw = rng.integers(0, 256, size=512 * ch * nb, dtype=np.uint8)
            free = int(rng.integers(1, 4096))
            y, res = w.resample(raw, 512, free, -2.0)
            case["calls"].append(dict(res, out_free=free, y=sha(y)))
        out.append(case)
    return out


RECORDS = {"resampler": record_resampler, "quantisers": record_quantisers, "biquad": record_biquad,
           "wrapper": record_wrapper}


@pytest.fixture(scope="module")
def frozen():
    with open(GOLDEN) as fh:
        return json.load(fh)


def _compare(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(json.loads(json.dumps(got)), want)):
        assert g == w, k


def test_resampler_random_configs(oracle, frozen):
    _compare(record_resampler(oracle), frozen["resampler"])


def test_quantisers_random(oracle, frozen):
    _compare(record_quantisers(oracle), frozen["quantisers"])


def test_biquad_random(oracle, frozen):
    _compare(record_biquad(oracle), frozen["biquad"])


def test_wrapper_random(oracle, frozen):
    _compare(record_wrapper(oracle), frozen["wrapper"])


if __name__ == "__main__":  # rewrite the frozen records from the UNMODIFIED reference (needs oracle/_ref)
    from oracle_lib import Reference
    ref = Reference()
    with open(GOLDEN, "w") as fh:
        json.dump({name: fn(ref) for name, fn in RECORDS.items()}, fh, separators=(",", ":"))
    print("wrote", GOLDEN, os.path.getsize(GOLDEN))
