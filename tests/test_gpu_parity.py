"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle and the
golden fixtures from the unmodified reference.  Integer/byte work is bit-exact; the FP32
resampler is bit-exact in exact mode and within 1e-6 max-abs full scale in fast mode
(the tolerance BASELINE.json states); the biquad is bit-exact."""
import numpy as np
import pytest
from conftest import bits_equal
from oracle_lib import multitone, noise

import esp_audio_libs_b200 as espb

pytestmark = pytest.mark.gpu
f32 = np.float32
TOL = 1e-6  # BASELINE.json north_star: max-abs error of 1e-6 full scale for the FP32 resampler


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert espb.device_count() > 0, "GPU tests need a GPU: the product has no CPU path"
    espb.set_device(0)
    info = espb.device_info()
    assert info["cc"][0] == 10, f"built for sm_100a, found {info}"


def oracle_rows(oracle, x, channels, taps, filters, lowpass, flags, adv, cap, ratio):
    ys = []
    res = None
    for row in x:
        o = oracle.resampler(channels, taps, filters, lowpass, flags)
        if adv:
            o.advance(adv)
        y, u, g = o.process_interleaved(row, cap, ratio)
        ys.append(y)
        res = (u, g)
    return np.stack(ys), res


# ---------------------------------------------------------------- quantisers
@pytest.mark.parametrize("bits", [1, 5, 8, 9, 12, 16, 17, 20, 24, 25, 31, 32])
def test_quantisers_bit_exact(oracle, bits):
    rng = np.random.default_rng(bits)
    nb = (bits + 7) // 8
    for n in (0, 1, 3, 4, 5, 1023, 4096, 100003):
        raw = rng.integers(0, 256, size=max(n * nb, 1), dtype=np.uint8)
        for gain in (0.0, -7.25):
            a = espb.quantized_to_float(raw, n, bits, gain)
            b = oracle.quantized_to_float(raw, n, bits, gain) if n else np.zeros(0, f32)
            assert bits_equal(a, b), (bits, n, gain)
        x = (rng.random(n) * 2.6 - 1.3).astype(f32)
        if n >= 12:
            x[:12] = [0, 1, -1, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768, np.nextafter(f32(1), f32(0)), -1.0000001,
                      0.99999, -0.99999, 1e-9, -1e-9]
        qa, ca = espb.float_to_quantized(x, bits)
        qb, cb = oracle.float_to_quantized(x, bits) if n else (np.zeros(0, np.uint8), 0)
        assert ca == cb and bits_equal(qa, qb), (bits, n)


def test_quantisers_golden(golden):
    arrays, meta = golden
    for q in meta["quant"]:
        bits = q["bits"]
        for gain in (0.0, -6.5):
            assert bits_equal(espb.quantized_to_float(arrays[f"q2f_{bits}_raw"], 4096, bits, gain),
                              arrays[f"q2f_{bits}_{gain}"])
        out, clipped = espb.float_to_quantized(arrays[f"f2q_{bits}_x"], bits)
        assert clipped == q["clipped"] and bits_equal(out, arrays[f"f2q_{bits}_q"])
    out, clipped = espb.float_to_quantized(np.array([0, 1, -1, 0.5 / 32768, -0.5 / 32768, 1.5 / 32768], f32), 16)
    assert list(out.view(np.int16)) == [0, 32767, -32768, 1, 0, 2] and clipped == 1
    assert float(espb.quantized_to_float(np.array([0, 0, 0x80, 1], np.uint8), 1, 32)[0]) == 0.00390625


def test_quantiser_unaligned_buffers(oracle):
    # the reference reads byte-wise with no alignment assumption: offset device pointers by 1..3 bytes
    rng = np.random.default_rng(12)
    L = espb.lib()
    for bits in (16, 24, 32):
        nb = (bits + 7) // 8
        n = 5001
        raw = rng.integers(0, 256, size=n * nb + 8, dtype=np.uint8)
        d_in = espb.DeviceBuffer.from_numpy(raw)
        d_out = espb.DeviceBuffer((n + 4) * 4)
        for off in (1, 2, 3):
            assert L.espb_quantized_to_float(d_in.ptr + off, d_out.ptr + 4, n, bits, 0.0, None) == 0
            got = d_out.download(f32)[1:n + 1]
            assert bits_equal(got, oracle.quantized_to_float(raw[off:], n, bits, 0.0)), (bits, off)


# ---------------------------------------------------------------- biquad
@pytest.mark.parametrize("channels,streams", [(1, 70), (2, 37), (3, 11), (8, 5)])
def test_biquad_bit_exact(oracle, channels, streams):
    n = 3000
    x = np.stack([noise(n, channels, stream=s, amp=0.9) for s in range(streams)])
    for f, gain, sections in ((0.2274, 1.0, 2), (1.0 / 6.0, 1.0, 2), (0.441, 0.5, 1), (0.02, 1.0, 3)):
        c = espb.biquad_lowpass(f)
        assert bits_equal(c, oracle.biquad_lowpass(f))
        bq = espb.BiquadBatch(streams * channels, sections, c, gain)
        # two calls: state carries across calls exactly like the reference's Biquad struct
        y1 = bq.apply_interleaved(x[:, : 1234 * channels], channels)
        y2 = bq.apply_interleaved(x[:, 1234 * channels:], channels)
        y = np.concatenate([y1, y2], axis=1)
        for s in range(streams):
            ref = x[s].copy()
            for ch in range(channels):
                for _ in range(sections):
                    oracle.biquad(c, gain).apply_buffer(ref[ch:], channels, n=n)
            assert bits_equal(y[s], ref), (channels, s, f)
        bq.free()


def test_biquad_first_order_and_highpass(oracle, golden):
    arrays, _ = golden
    x = arrays["biquad_x"][:2000].copy().reshape(1, -1)
    bq = espb.BiquadBatch(1, 1, arrays["biquad_fo_c"], 1.0)
    assert bits_equal(bq.apply_interleaved(x, 1)[0], arrays["biquad_fo_y"])
    c = espb.biquad_highpass(0.1)
    assert bits_equal(c, oracle.biquad_highpass(0.1))
    xs = np.stack([noise(2500, 2, stream=s) for s in range(9)])
    y = espb.BiquadBatch(18, 2, c, 2.0).apply_interleaved(xs, 2)
    for s in range(9):
        ref = xs[s].copy()
        for ch in range(2):
            for _ in range(2):
                oracle.biquad(c, 2.0).apply_buffer(ref[ch:], 2, n=2500)
        assert bits_equal(y[s], ref)


@pytest.mark.parametrize("f", [0.2274, 1.0 / 6.0, 0.441])
def test_biquad_time_blocks_merge_bit_exactly(oracle, f):
    """Block-parallel state carry for long single streams: blocks of 4096 frames, each after a 1024-frame warm-up
    from a zero state, give the sequential result bit for bit at the cutoffs the Resampler policy produces (the
    trajectories merge); the formal bar for this mode is 1e-6."""
    channels, streams, n = 8, 3, 30000
    x = np.stack([noise(n, channels, stream=s, amp=0.9) for s in range(streams)])
    c = espb.biquad_lowpass(f)
    bq = espb.BiquadBatch(streams * channels, 2, c, 1.0)
    bq.set_time_blocks(4096, 1024)
    y1 = bq.apply_interleaved(x[:, : 17000 * channels], channels)   # state carries across calls in this mode too
    y2 = bq.apply_interleaved(x[:, 17000 * channels:], channels)
    y = np.concatenate([y1, y2], axis=1)
    for s in range(streams):
        ref = x[s].copy()
        for ch in range(channels):
            for _ in range(2):
                oracle.biquad(c, 1.0).apply_buffer(ref[ch:], channels, n=n)
        assert np.max(np.abs(y[s].astype(np.float64) - ref)) <= TOL
        assert bits_equal(y[s], ref), f
    bq.free()


@pytest.mark.parametrize("f,warm", [(0.02, 1024), (0.005, 1024), (0.005, 32), (0.0007, 256), (0.2274, 32)])
def test_biquad_time_blocks_are_exact_by_construction(oracle, f, warm):
    """Low cutoffs (pole radius 0.92 .. 0.997) and warm-ups far too short for the trajectories to merge: the device
    compares every block's start state with its predecessor's end state and re-filters the block where they differ,
    so the output and the saved state are still the sequential ones (art_biquad.cpp:73-93) bit for bit — over two
    calls, with the automatic default (blocks of 8192 rows) and with explicit small blocks."""
    channels, streams, n = 2, 3, 70000
    x = np.stack([noise(n, channels, stream=20 + s, amp=0.9) for s in range(streams)])
    c = espb.biquad_lowpass(f)
    ref = x.copy()
    states = []
    for s in range(streams):
        for ch in range(channels):
            st = []
            for _ in range(2):
                b = oracle.biquad(c, 1.0)
                b.apply_buffer(ref[s][ch:], channels, n=n)
                st.append(b)
            states.append(st)
    for blocks in (-1, 2048):
        bq = espb.BiquadBatch(streams * channels, 2, c, 1.0)
        bq.set_time_blocks(blocks, warm)
        y1 = bq.apply_interleaved(x[:, : 41000 * channels], channels)
        y2 = bq.apply_interleaved(x[:, 41000 * channels:], channels)
        y = np.concatenate([y1, y2], axis=1)
        assert bits_equal(y, ref), (f, warm, blocks)
        repaired, warm_now = bq.block_stats()
        if f <= 0.005:   # these cannot merge within the warm-up: the repair path is what made the result exact
            assert repaired > 0 and warm_now > warm
        # the saved state is the sequential one too: a third (short, sequential) call continues identically
        tail = noise(500, channels, stream=99, amp=0.5).reshape(1, -1).repeat(streams, axis=0)
        y3 = bq.apply_interleaved(tail, channels)
        bq2 = espb.BiquadBatch(streams * channels, 2, c, 1.0)
        bq2.set_time_blocks(0, 0)
        bq2.apply_interleaved(x, channels)
        assert bits_equal(y3, bq2.apply_interleaved(tail, channels))
        bq.free()
        bq2.free()


def test_wrapper_with_biquad_time_blocks(oracle):
    """C4-like call (96 -> 44.1 kHz, 8 channels, 24-bit, pre-filter) with the pre-filter in time-block mode."""
    ns, ch, frames = 2, 8, 20000
    rng = np.random.default_rng(4)
    pcm = (rng.normal(0, 0.3, size=(ns, frames * ch)).clip(-1, 0.99999) * (2 ** 23)).astype(np.int64)
    raw = np.zeros((ns, frames * ch * 3), np.uint8)
    for b in range(3):
        raw[:, b::3] = (pcm >> (8 * b)) & 0xFF
    cap = int(frames * 44100 / 96000) + 64
    r = espb.Resampler(ns, frames * ch, cap * ch, 96000, 44100, 24, 24, ch, True, True, 256, 64, mode=espb.MODE_EXACT)
    assert r.policy()["filter"] == "pre"
    r.set_biquad_time_blocks(4096, 1024)
    out, res = r.resample(raw, frames, cap, 0.0)
    # the oracle wrapper handles at most 2 channels (include/resampler.h:64): compose the stages directly
    pol = r.policy()
    for s in range(ns):
        xf = oracle.quantized_to_float(raw[s], frames * ch, 24, 0.0)
        for c in range(ch):
            for _ in range(2):
                oracle.biquad(pol["coeffs"], 1.0).apply_buffer(xf[c:], ch, n=frames)
        o = oracle.resampler(ch, 256, 64, float(pol["art_lowpass"]), pol["art_flags"])
        o.advance(128.0)
        yf, used, gen = o.process_interleaved(xf, cap, pol["sample_ratio"])
        q, clipped = oracle.float_to_quantized(yf, 24)
        assert gen == res["frames_generated"] and bits_equal(out[s], q)
    r.free()


def test_biquad_golden(golden):
    arrays, meta = golden
    x = arrays["biquad_x"].reshape(1, -1)
    for k, b in enumerate(meta["biquad"]):
        bq = espb.BiquadBatch(2, 2, arrays[f"biquad_{k}_c"], b["gain"])
        assert bits_equal(bq.apply_interleaved(x, 2)[0], arrays[f"biquad_{k}_y"]), b


# ---------------------------------------------------------------- resampler
def test_resampler_golden_small_cases(golden):
    arrays, meta = golden
    for c in meta["small"]:
        x = arrays[f"small_{c['name']}_x"]
        ns = 3
        xb = np.stack([x] * ns)
        for mode in (espb.MODE_EXACT, espb.MODE_FAST):
            b = espb.ResampleBatch(ns, c["channels"], c["taps"], c["filters"], c["lowpass"], c["flags"], mode=mode)
            if c["advance"]:
                b.advance(c["advance"])
            y, used, gen = b.process_interleaved(xb, c["cap"], f32(c["ratio"]))
            assert (used, gen) == (c["used"], c["generated"]), c["name"]
            off, idx = b.state()
            assert (float(off), idx) == (c["final_offset"], c["final_index"]) and b.position() == c["position"]
            ref = arrays[f"small_{c['name']}_y"]
            for s in range(ns):
                if mode == espb.MODE_EXACT:
                    assert bits_equal(y[s], ref), c["name"]
                else:
                    assert np.max(np.abs(y[s].astype(np.float64) - ref)) <= TOL, c["name"]
            b.free()


@pytest.mark.parametrize("case", [
    # channels, streams, taps, filters, lowpass, flags, ratio, n_in   (series counts straddle the 128-series CTA groups)
    (2, 70, 256, 256, 1.0, 3, f32(48000) / f32(44100), 2500),
    (2, 65, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 2500),
    (1, 131, 256, 256, 1.0, 1, f32(3.0), 900),
    (8, 17, 1024, 256, 0.45, 1, f32(44100) / f32(96000), 3000),
    (3, 45, 32, 16, 1.0, 0, f32(1.37), 1500),
    (1, 1, 4, 2, 1.0, 3, f32(2.5), 300),
    (5, 30, 64, 1024, 0.7, 2, f32(0.61), 2000),
])
def test_resampler_vs_oracle(oracle, case):
    ch, ns, taps, filters, lp, flags, ratio, n_in = case
    x = np.stack([noise(n_in, ch, stream=s, amp=0.9) for s in range(ns)])
    cap = int(n_in * float(ratio)) + 40
    ref, (uo, go) = oracle_rows(oracle, x, ch, taps, filters, lp, flags, taps / 2, cap, ratio)
    for mode in (espb.MODE_EXACT, espb.MODE_FAST):
        b = espb.ResampleBatch(ns, ch, taps, filters, lp, flags, mode=mode)
        b.advance(taps / 2)
        assert bits_equal(b.bank(), oracle.resampler(1, taps, filters, lp, flags).bank())
        y, used, gen = b.process_interleaved(x, cap, ratio)
        assert (used, gen) == (uo, go)
        if mode == espb.MODE_EXACT:
            assert bits_equal(y, ref)
        else:
            assert np.max(np.abs(y.astype(np.float64) - ref)) <= TOL
        b.free()


def test_resampler_high_amplitude_fast_mode_tolerance(oracle):
    # SURVEY §8a R5 stress case: amplitude 0.9 noise and multitone, T=256 and T=1024
    for taps, ch, ratio, lp in ((256, 2, f32(48000) / f32(44100), 1.0), (1024, 2, f32(44100) / f32(96000), 0.45)):
        x = np.stack([noise(6000, ch, stream=1, amp=0.9), multitone(6000, ch, 44100.0, stream=2, amp=0.9)])
        cap = int(6000 * float(ratio)) + 40
        ref, _ = oracle_rows(oracle, x, ch, taps, 256, lp, 3, taps / 2, cap, ratio)
        b = espb.ResampleBatch(2, ch, taps, 256, lp, 3)
        b.advance(taps / 2)
        y, _, _ = b.process_interleaved(x, cap, ratio)
        err = float(np.max(np.abs(y.astype(np.float64) - ref)))
        assert err <= TOL, (taps, err)


def test_resampler_chunked_streaming_is_bit_identical(oracle, golden):
    arrays, meta = golden
    m = meta["chunked"]
    x, plan, ch = arrays["chunked_x"], arrays["chunked_plan"], m["channels"]
    ns = 4
    b = espb.ResampleBatch(ns, ch, m["taps"], m["filters"], 1.0, m["flags"], mode=espb.MODE_EXACT)
    b.advance(m["advance"])
    o_dry = oracle.resampler(ch, m["taps"], m["filters"], 1.0, m["flags"])
    o_dry.advance(m["advance"])
    outs, pos = [], 0
    for n_in, n_out, used, gen in plan:
        seg = np.stack([x[pos * ch:(pos + int(n_in)) * ch]] * ns)
        # dry runs on a context with carried state (art_resampler.cpp:257-306) against the oracle in the same state
        assert b.required(int(n_out), f32(m["ratio"])) == o_dry.required(int(n_out), f32(m["ratio"]))
        assert b.expected(int(n_in), f32(m["ratio"])) == o_dry.expected(int(n_in), f32(m["ratio"]))
        assert b.position() == o_dry.position()
        o_dry.process_interleaved(x[pos * ch:(pos + int(n_in)) * ch], int(n_out), f32(m["ratio"]), n_in=int(n_in))
        y, u, g = b.process_interleaved(seg.reshape(ns, -1), int(n_out), f32(m["ratio"]), n_in=int(n_in))
        assert (u, g) == (used, gen)
        outs.append(y)
        pos += u
    y = np.concatenate(outs, axis=1)
    for s in range(ns):
        assert bits_equal(y[s], arrays["chunked_y"])
    # reset returns to the initial state and output
    b.reset()
    b.advance(m["advance"])
    y2, _, _ = b.process_interleaved(np.stack([x] * ns), y.shape[1] // ch, f32(m["ratio"]))
    assert bits_equal(y2[0], arrays["chunked_y"])


def test_resampler_empty_and_capacity_limited_calls(oracle):
    ch, taps = 2, 64
    ratio = f32(1.5)
    x = np.stack([noise(500, ch, stream=s) for s in range(3)])
    b = espb.ResampleBatch(3, ch, taps, 64, 1.0, 3, mode=espb.MODE_EXACT)
    o = [oracle.resampler(ch, taps, 64, 1.0, 3) for _ in range(3)]
    # no input, no output space
    assert b.process_interleaved(np.zeros((3, 0), f32), 0, ratio, n_in=0)[1:] == (0, 0)
    # no input but output space: the initial half-window of silence can be emitted
    y, u, g = b.process_interleaved(np.zeros((3, 0), f32), 100, ratio, n_in=0)
    yo, uo, go = o[0].process_interleaved(np.zeros(0, f32), 100, ratio, n_in=0)
    for k in (1, 2):
        o[k].process_interleaved(np.zeros(0, f32), 100, ratio, n_in=0)
    assert (u, g) == (uo, go) and bits_equal(y[0], yo)
    # output capacity smaller than what the input could produce
    y, u, g = b.process_interleaved(x, 37, ratio)
    for k in range(3):
        yo, uo, go = o[k].process_interleaved(x[k], 37, ratio)
        assert (u, g) == (uo, go) and bits_equal(y[k], yo)
    # the rest of that input after the capacity-limited call
    y, u2, g2 = b.process_interleaved(x[:, u * ch:], 2000, ratio)
    for k in range(3):
        yo, uo, go = o[k].process_interleaved(x[k][u * ch:], 2000, ratio)
        assert (u2, g2) == (uo, go) and bits_equal(y[k], yo)
    assert b.state() == o[0].state()


def test_resampler_planar(golden):
    arrays, meta = golden
    m = meta["planar"]
    b = espb.ResampleBatch(2, m["channels"], m["taps"], m["filters"], 1.0, m["flags"], mode=espb.MODE_EXACT)
    y, used, gen = b.process_planar(np.stack([arrays["planar_x"]] * 2), 800, f32(m["ratio"]))
    assert (used, gen) == (m["used"], m["generated"])
    assert bits_equal(y[0], arrays["planar_y"]) and bits_equal(y[1], arrays["planar_y"])


def test_resampler_host_buffer_path(oracle):
    ch, taps, ns, n_in = 2, 64, 50, 1500
    ratio = f32(48000) / f32(44100)
    x = np.stack([noise(n_in, ch, stream=s) for s in range(ns)])
    cap = int(n_in * float(ratio)) + 20
    hin = espb.PinnedBuffer(x.size, f32)
    hin.array[:] = x.reshape(-1)
    hout = espb.PinnedBuffer(ns * cap * ch, f32)
    hout.array[:] = 0
    b = espb.ResampleBatch(ns, ch, taps, 64, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(taps / 2)
    used, gen = b.process_interleaved_host(hin.ptr, n_in * ch, n_in, hout.ptr, cap * ch, cap, ratio)
    ref, (uo, go) = oracle_rows(oracle, x, ch, taps, 64, 1.0, 3, taps / 2, cap, ratio)
    assert (used, gen) == (uo, go)
    got = hout.array.reshape(ns, cap * ch)[:, : gen * ch]
    assert bits_equal(np.ascontiguousarray(got), ref)


def test_invalid_init_returns_null():
    for taps, filters in ((30, 16), (0, 16), (1028, 16), (32, 1), (32, 1025)):
        with pytest.raises(espb.EspbError):
            espb.ResampleBatch(1, 1, taps, filters, 1.0, 0)


# ---------------------------------------------------------------- wrapper, end to end
def test_wrapper_golden(golden):
    arrays, meta = golden
    for k, m in enumerate(meta["wrapper"]):
        chn, nb = m["channels"], (m["src_bits"] + 7) // 8
        ns = 3
        r = espb.Resampler(ns, 1024 * chn, 4096 * chn, m["src_rate"], m["dst_rate"], m["src_bits"], m["dst_bits"],
                           chn, m["use_filter"], m["interpolate"], m["taps"], m["filters"], mode=espb.MODE_EXACT)
        raw, outs, res = arrays[f"wrap_{k}_raw"], [], []
        for it in range(3):
            seg = raw[it * 1024 * chn * nb:(it + 1) * 1024 * chn * nb]
            y, rr = r.resample(np.stack([seg] * ns), 1024, m["out_free"][it], m["gain_db"], host_path=(it == 2))
            outs.append(y)
            res.append([rr["frames_used"], rr["frames_generated"], rr["predicted_frames_used"],
                        int(rr["clipped_per_stream"][1])])
            assert rr["clipped_samples"] == ns * int(rr["clipped_per_stream"][0])
        assert np.array_equal(np.array(res, np.int64), arrays[f"wrap_{k}_res"]), m
        y = np.concatenate(outs, axis=1)
        for s in range(ns):
            assert bits_equal(y[s], arrays[f"wrap_{k}_y"]), (m, s)
        r.free()


@pytest.mark.parametrize("cfg", [
    # src_rate, dst_rate, src_bits, dst_bits, channels, streams  (C3- and C4-like paths)
    (16000, 48000, 16, 16, 1, 133),
    (96000, 44100, 24, 24, 2, 20),
    (48000, 44100, 32, 16, 2, 40),
])
def test_wrapper_vs_oracle_fast_mode_within_one_lsb(oracle, cfg):
    sr, dr, sb, db, ch, ns = cfg
    nb = (sb + 7) // 8
    frames = 2048
    rng = np.random.default_rng(sr + db)
    pcm = (rng.normal(0, 0.3, size=(ns, frames * ch)).clip(-1, 0.99999) * (2 ** (8 * nb - 1))).astype(np.int64)
    raw = np.zeros((ns, frames * ch * nb), np.uint8)
    for b in range(nb):
        raw[:, b::nb] = (pcm >> (8 * b)) & 0xFF
    cap = int(frames * dr / sr) + 64
    for mode in (espb.MODE_EXACT, espb.MODE_FAST):
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 256, 256, mode=mode)
        out, res = r.resample(raw, frames, cap, -1.5)
        ob = (db + 7) // 8
        for s in range(0, ns, 7):
            w = oracle.wrapper(frames * ch, cap * ch, float(sr), float(dr), sb, db, ch, True, True, 256, 256)
            yo, ro = w.resample(raw[s], frames, cap, -1.5)
            assert res["frames_generated"] == ro["frames_generated"] and res["frames_used"] == ro["frames_used"]
            if mode == espb.MODE_EXACT:
                assert bits_equal(out[s], yo)
                assert int(res["clipped_per_stream"][s]) == ro["clipped_samples"]
            else:
                a = _le_to_int(out[s], ob)
                bb = _le_to_int(yo, ob)
                assert np.max(np.abs(a - bb)) <= (1 << ((32 - db) % 8)), (cfg, s)
        r.free()


@pytest.mark.parametrize("cfg", [
    # src_rate, dst_rate, src_bits, dst_bits, channels, streams, frames: channel counts / frame counts that take the
    # generic layout kernels, the < 64-frame tails and unaligned PCM rows (odd bytes per row)
    (44100, 48000, 24, 16, 3, 45, 1001),
    (48000, 32000, 16, 24, 6, 22, 777),
    (22050, 44100, 8, 32, 5, 27, 63),
    (32000, 48000, 16, 16, 2, 3, 130),
])
def test_wrapper_odd_shapes_vs_composed_oracle(oracle, cfg):
    """The oracle wrapper is limited to 2 channels (include/resampler.h:64), so the reference pipeline is composed
    from the oracle's stages with the policy the library reports."""
    sr, dr, sb, db, ch, ns, frames = cfg
    nb, ob = (sb + 7) // 8, (db + 7) // 8
    rng = np.random.default_rng(frames)
    raw = rng.integers(0, 256, size=(ns, frames * ch * nb), dtype=np.uint8)
    cap = int(frames * dr / sr) + 40
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 64, 64, mode=espb.MODE_EXACT)
    pol = r.policy()
    outs = []
    for it in range(2):  # two calls: state carries through every stage
        out, res = r.resample(raw, frames, cap, -2.5)
        outs.append((out, res))
    states = {}
    for s in range(0, ns, 4):
        o = oracle.resampler(ch, 64, 64, float(pol["art_lowpass"]), pol["art_flags"])
        o.advance(32.0)
        bq = [[oracle.biquad(pol["coeffs"], 1.0) for _ in range(2)] for _ in range(ch)]
        for it in range(2):
            xf = oracle.quantized_to_float(raw[s], frames * ch, sb, -2.5)
            if pol["filter"] == "pre":
                for c in range(ch):
                    for k in range(2):
                        bq[c][k].apply_buffer(xf[c:], ch, n=frames)
            yf, used, gen = o.process_interleaved(xf, cap, pol["sample_ratio"])
            yf = np.ascontiguousarray(yf)
            if pol["filter"] == "post":
                for c in range(ch):
                    for k in range(2):
                        bq[c][k].apply_buffer(yf[c:], ch, n=gen)
            q, clipped = oracle.float_to_quantized(yf, db)
            out, res = outs[it]
            assert (res["frames_used"], res["frames_generated"]) == (used, gen)
            assert bits_equal(out[s], q), (cfg, s, it)
            assert int(res["clipped_per_stream"][s]) == clipped
    r.free()


def _le_to_int(bytes_, nb):
    b = bytes_.reshape(-1, nb).astype(np.int64)
    v = np.zeros(b.shape[0], np.int64)
    for k in range(nb):
        v |= b[:, k] << (8 * k)
    sign = 1 << (8 * nb - 1)
    return (v ^ sign) - sign


# ---------------------------------------------------------------- full-size properties (BASELINE configs[1])
@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_full_size_batch_properties(oracle, mode):
    """4096 stereo streams, 256 taps, 44.1 -> 48 kHz (0.25 s each to keep the test short): every stream
    with the same input gives the same output (a checksum of checksums), sampled streams match the
    oracle (bit for bit in exact mode), and the device checksum equals the host's.  Run three times on fresh
    contexts: the checksum must not move (the kernel's stage hand-over — a relaxed shared-memory counter and
    mbarriers, resample_kernel.cu — would show up here as run-to-run differences; compute-sanitizer is closed on
    this pool, see profiles/r02_sanitizer_note.md)."""
    ns, ch, taps, n_in = 4096, 2, 256, 11025
    exact = mode == "exact"
    ratio = f32(48000) / f32(44100)
    base = [noise(n_in, ch, stream=s, amp=0.5) for s in range(8)]
    x = np.stack([base[s % 8] for s in range(ns)])
    cap = int(n_in * float(ratio)) + 16
    d_in = espb.DeviceBuffer.from_numpy(x)
    d_out = espb.DeviceBuffer(ns * cap * ch * 4)
    sums_seen = set()
    for _run in range(3):
        b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=espb.MODE_EXACT if exact else espb.MODE_FAST)
        b.advance(taps / 2)
        d_out.zero()
        used, gen = b.process_interleaved_dev(d_in.ptr, n_in * ch, n_in, d_out.ptr, cap * ch, cap, ratio)
        dev_sum = espb.checksum_u32(d_out.ptr, ns * cap * ch)
        sums_seen.add(dev_sum)
        b.free()
    assert len(sums_seen) == 1
    y = d_out.download(f32).reshape(ns, cap * ch)
    assert dev_sum == int(y.view(np.uint32).astype(np.uint64).sum() & np.uint64(0xFFFFFFFFFFFFFFFF))
    o = oracle.resampler(ch, taps, 256, 1.0, 3)
    o.advance(taps / 2)
    assert gen == o.expected(n_in, ratio) and used == n_in
    sums = y[:, : gen * ch].view(np.uint32).astype(np.uint64).sum(axis=1)
    for s in range(8):
        assert np.all(sums[s::8] == sums[s])  # identical inputs -> identical outputs, wherever they sit in the batch
        oo = oracle.resampler(ch, taps, 256, 1.0, 3)
        oo.advance(taps / 2)
        yo, _, _ = oo.process_interleaved(base[s], cap, ratio)
        if exact:
            assert bits_equal(y[s, : gen * ch], yo[: gen * ch]) and bits_equal(y[ns - 8 + s, : gen * ch], yo[: gen * ch])
        else:
            assert np.max(np.abs(y[s, : gen * ch].astype(np.float64) - yo)) <= TOL
    assert np.all(y[:, gen * ch:] == 0)  # nothing written past the generated frames


@pytest.mark.parametrize("mode", ["exact", "fast"])
def test_ratio_groups_drifting_ratios_chunked(oracle, mode):
    """SURVEY §8f N1: per-group, per-call ratios (ASRC) with persistent device-side state.  Three groups of
    streams follow three clocks; every call each group gets its own chunk sizes and a slightly different ratio.
    Each stream is compared with its own reference-style context fed the same sequence of calls."""
    ch, taps, filters, flags = 2, 64, 128, 3
    sizes = [5, 130, 1]
    base = [f32(48000) / f32(44100), f32(44100) / f32(48000) * f32(0.999), f32(2.0)]
    g = espb.ResampleGroups(sizes, ch, taps, filters, 1.0, flags,
                            mode=espb.MODE_EXACT if mode == "exact" else espb.MODE_FAST)
    ns = sum(sizes)
    group_of = np.repeat(np.arange(len(sizes)), sizes)
    orc = [oracle.resampler(ch, taps, filters, 1.0, flags) for _ in range(ns)]
    for k in range(len(sizes)):
        g.advance(k, taps / 2)
    for o in orc:
        o.advance(taps / 2)
    rng = np.random.default_rng(42)
    total = 2600
    x = np.stack([noise(total, ch, stream=300 + s, amp=0.7) for s in range(ns)])
    pos = [0] * len(sizes)
    worst = 0.0
    for call in range(9):
        n_in = [int(min(rng.integers(0, 400), total - pos[k])) for k in range(len(sizes))]
        n_out = [int(rng.integers(0, 700)) for _ in sizes]
        ratios = [f32(base[k] * f32(1.0 + 2e-4 * np.sin(call + k))) for k in range(len(sizes))]
        row = max(max(n_in), 1) * ch
        xin = np.zeros((ns, row), f32)
        for s in range(ns):
            k = group_of[s]
            xin[s, : n_in[k] * ch] = x[s, pos[k] * ch:(pos[k] + n_in[k]) * ch]
        y, res = g.process_interleaved(xin, n_in, n_out, ratios)
        for s in range(ns):
            k = group_of[s]
            yo, uo, go = orc[s].process_interleaved(xin[s, : n_in[k] * ch], n_out[k], ratios[k], n_in=n_in[k])
            assert res[k] == (uo, go), (call, s, res[k], uo, go)
            got = y[s, : go * ch]
            if mode == "exact":
                assert bits_equal(got, yo), (call, s)
            elif go:
                worst = max(worst, float(np.max(np.abs(got.astype(np.float64) - yo))))
        for k in range(len(sizes)):
            pos[k] += res[k][0]
            assert g.state(k) == orc[int(np.argmax(group_of == k))].state()
    assert worst <= 1e-6  # fast mode: the north star's tolerance (max-abs, full scale)
    g.free()


@pytest.mark.parametrize("mode", ["exact", "fast"])
def test_direct_input_path_stereo(oracle, mode):
    """Interleaved stereo float input in chunked calls of changing size (some below numTaps: the carried frames come
    from more than one earlier call), capacity-limited calls, an empty call, a partial last series group."""
    ch, taps, filters = 2, 64, 64
    ns = 70  # one full group of 64 streams and a partial one
    ratio = f32(48000) / f32(44100)
    total = 5000
    x = np.stack([noise(total, ch, stream=500 + s, amp=0.8) for s in range(ns)])
    b = espb.ResampleBatch(ns, ch, taps, filters, 1.0, 3, mode=espb.MODE_EXACT if mode == "exact" else espb.MODE_FAST)
    b.advance(taps / 2)
    probes = [0, 31, 32, 63, 64, ns - 1]
    orc = {s: oracle.resampler(ch, taps, filters, 1.0, 3) for s in probes}
    for o in orc.values():
        o.advance(taps / 2)
    pos, worst = 0, 0.0
    for n_in, cap in [(1000, 2000), (10, 50), (900, 300), (64, 500), (2, 9), (1500, 4000), (700, 4000)]:
        n_in = min(n_in, total - pos)
        seg = np.ascontiguousarray(x[:, pos * ch:(pos + n_in) * ch])
        if n_in == 0:
            seg = np.zeros((ns, 0), f32)
        y, used, gen = b.process_interleaved(seg, cap, ratio, n_in=n_in)
        for s in probes:
            yo, uo, go = orc[s].process_interleaved(seg[s], cap, ratio, n_in=n_in)
            assert (used, gen) == (uo, go)
            if mode == "exact":
                assert bits_equal(y[s], yo), (n_in, cap, s)
            elif go:
                worst = max(worst, float(np.max(np.abs(y[s].astype(np.float64) - yo))))
        pos += used
    assert b.state() == orc[0].state()
    assert worst <= 1e-6
    b.free()


@pytest.mark.parametrize("ch,pad,skew", [(2, 2, 0), (2, 1, 1), (1, 1, 0), (1, 3, 1), (4, 2, 2), (8, 4, 1), (1, 4, 0), (2, 4, 0),
                                         (4, 4, 0), (8, 8, 4)])
def test_resampler_float_rows_of_any_alignment(oracle, ch, pad, skew):
    """Stream rows that are 16-, 8- or only 4-byte aligned (row stride = frames*channels + pad floats, buffers offset
    by `skew` floats) go through the vectorised, the 8-byte and the scalar form of the layout stages."""
    taps, filters, ns, n_in = 64, 32, 9, 300
    ratio = f32(1.25)
    cap = int(n_in * 1.25) + 8
    x = np.stack([noise(n_in, ch, stream=700 + s, amp=0.8) for s in range(ns)])
    in_stride, out_stride = n_in * ch + pad, cap * ch + pad
    hin = np.zeros(ns * in_stride + skew, f32)
    for s in range(ns):
        hin[skew + s * in_stride: skew + s * in_stride + n_in * ch] = x[s]
    d_in = espb.DeviceBuffer.from_numpy(hin)
    d_out = espb.DeviceBuffer((ns * out_stride + skew) * 4)
    d_out.zero()
    b = espb.ResampleBatch(ns, ch, taps, filters, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(taps / 2)
    used, gen = b.process_interleaved_dev(d_in.ptr + 4 * skew, in_stride, n_in, d_out.ptr + 4 * skew, out_stride, cap,
                                          ratio)
    got = d_out.download(f32)
    for s in range(ns):
        o = oracle.resampler(ch, taps, filters, 1.0, 3)
        o.advance(taps / 2)
        yo, uo, go = o.process_interleaved(x[s], cap, ratio)
        assert (used, gen) == (uo, go)
        row = got[skew + s * out_stride: skew + (s + 1) * out_stride]
        assert bits_equal(row[: gen * ch], yo), (s, ch, pad, skew)
        assert not row[gen * ch:].any()  # nothing written past the generated frames
    b.free()
    d_in.free()
    d_out.free()


def test_biquad_apply_samples_matches_sample_by_sample_reference(oracle):
    """biquad_apply_sample (art_biquad.cpp:55-69) for a bank of series, one sample per call, bit-exact, and
    interchangeable with apply_buffer (same state)."""
    n_series, steps = 300, 40
    c = espb.biquad_lowpass(0.2274)
    bank = espb.BiquadBatch(n_series, 2, c)
    x = np.stack([noise(steps, 1, stream=900 + q, amp=0.9) for q in range(n_series)])  # (series, steps)
    got = np.stack([bank.apply_samples(x[:, t]) for t in range(steps)], axis=1)
    for q in (0, 1, 127, 128, 299):
        s1, s2 = oracle.biquad(c), oracle.biquad(c)  # the wrapper's cascade: two sections, sample by sample
        want = np.array([s2.apply_sample(s1.apply_sample(v)) for v in x[q]], np.float32)
        assert bits_equal(got[q], want), q
    bank.free()


def test_wrapper_async_calls_match_synchronous_ones(oracle):
    """espb_resampler_resample_async: a stream of calls enqueued without synchronising gives the same bytes, frame
    counts and (device-side) clip counts as the synchronous call."""
    ns, ch, frames, cap = 50, 2, 1500, 1800
    rng = np.random.default_rng(5)
    pcm = (rng.normal(0, 0.5, (ns, frames * ch)).clip(-1.2, 1.2) * 30000).clip(-32768, 32767).astype(np.int16)
    outs = {}
    for kind in ("sync", "async"):
        r = espb.Resampler(ns, frames * ch, cap * ch, 44100, 48000, 16, 16, ch, True, True, 64, 64, mode=espb.MODE_EXACT)
        d_in = espb.DeviceBuffer.from_numpy(pcm.view(np.uint8))
        d_out = espb.DeviceBuffer(ns * cap * ch * 2)
        got = []
        for call in range(3):
            d_out.zero()
            if kind == "sync":
                res = r.resample_dev(d_in.ptr, frames * ch * 2, d_out.ptr, cap * ch * 2, frames, cap, 3.0)
                clips = res["clipped_per_stream"].copy()
            else:
                res = r.resample_dev_async(d_in.ptr, frames * ch * 2, d_out.ptr, cap * ch * 2, frames, cap, 3.0)
                clips = np.zeros(ns, np.uint32)
                espb.capi._check(espb.lib().espb_memcpy_d2h(clips.ctypes.data, r.clipped_dev(), ns * 4, None), "d2h")
                espb.capi._check(espb.lib().espb_stream_sync(None), "sync")
            got.append((res["frames_used"], res["frames_generated"], clips, d_out.download(np.uint8)))
        outs[kind] = got
        r.free()
    for a, b in zip(outs["sync"], outs["async"]):
        assert a[0] == b[0] and a[1] == b[1] and bits_equal(a[2], b[2]) and bits_equal(a[3], b[3])
    assert sum(int(c[2].sum()) for c in outs["sync"]) > 0  # the +3 dB gain does clip some samples


# ---------------------------------------------------------------- full-size properties (BASELINE configs[2..4])
def _composed_oracle(oracle, raw_row, frames, ch, sb, db, taps, filters, pol, cap, gain_db=0.0):
    """One stream through the oracle's stages with the policy the library reports (any channel count)."""
    o = oracle.resampler(ch, taps, filters, float(pol["art_lowpass"]), pol["art_flags"])
    o.advance(taps / 2.0)
    xf = oracle.quantized_to_float(raw_row, frames * ch, sb, gain_db)
    if pol["filter"] == "pre":
        for c in range(ch):
            for _ in range(2):
                oracle.biquad(pol["coeffs"], 1.0).apply_buffer(xf[c:], ch, n=frames)
    yf, used, gen = o.process_interleaved(xf, cap, pol["sample_ratio"])
    yf = np.ascontiguousarray(yf)
    if pol["filter"] == "post":
        for c in range(ch):
            for _ in range(2):
                oracle.biquad(pol["coeffs"], 1.0).apply_buffer(yf[c:], ch, n=gen)
    q, clipped = oracle.float_to_quantized(yf, db)
    return q, used, gen, clipped


@pytest.mark.parametrize("name,ns,ch,sr,dr,bits,frames", [
    ("C3", 16384, 1, 16000, 48000, 16, 16000),   # 16 kHz -> 48 kHz mono voice, int16 in / out, post biquad
    ("C5 shard", 8192, 2, 48000, 44100, 32, 24000),  # 65536 / 8 stereo streams 48 -> 44.1 kHz (0.5 s per call)
])
def test_full_size_wrapper_configs(oracle, name, ns, ch, sr, dr, bits, frames):
    """BASELINE configs[2] and [4] at their stream counts, exact mode: streams with identical input give identical
    bytes wherever they sit in the batch, sampled streams are bit-exact with the composed CPU pipeline (PCM bytes and
    clip counts), nothing is written past the generated frames, and the batch clip total is the sum of the rows."""
    nb = bits // 8
    rng = np.random.default_rng(ns)
    distinct = 8
    amp = 2 ** (bits - 1) * 0.6
    base = (rng.normal(0, 0.45, (distinct, frames * ch)) * amp).clip(-2 ** (bits - 1), 2 ** (bits - 1) - 1).astype(np.int64)
    raw8 = np.zeros((distinct, frames * ch * nb), np.uint8)
    for b in range(nb):
        raw8[:, b::nb] = (base >> (8 * b)) & 0xFF
    raw = np.tile(raw8, (ns // distinct, 1))
    cap = int(frames * dr / sr) + 64
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, bits, bits, ch, True, True, 256, 256, mode=espb.MODE_EXACT)
    pol = r.policy()
    out, res = r.resample(raw, frames, cap, 2.0)   # +2 dB: some samples clip
    gen = res["frames_generated"]
    assert res["frames_used"] == frames and gen > 0
    row_bytes = gen * ch * nb
    sums = out[:, :row_bytes].astype(np.uint64).sum(axis=1)
    for s in range(distinct):
        assert np.all(sums[s::distinct] == sums[s])
        assert np.all(res["clipped_per_stream"][s::distinct] == res["clipped_per_stream"][s])
    assert not out[:, row_bytes:].any()
    assert int(res["clipped_per_stream"].astype(np.uint64).sum()) == res["clipped_samples"] > 0
    for s in (0, 3, ns - 1):
        q, used, g2, clipped = _composed_oracle(oracle, raw[s], frames, ch, bits, bits, 256, 256, pol, cap, 2.0)
        assert (used, g2) == (frames, gen)
        assert bits_equal(out[s, :row_bytes], q), (name, s)
        assert int(res["clipped_per_stream"][s]) == clipped
    r.free()


def test_full_size_long_stream_config(oracle):
    """BASELINE configs[3]: 96 -> 44.1 kHz, 8 channels, 24-bit, 1024 taps, long streams.  Ten seconds per call: the
    time-block form of the pre-filter gives the same bytes as the sequential one (exact mode), chunked calls give the
    same bytes as one call, and the first second is bit-exact with the composed CPU pipeline."""
    ns, ch, sr, dr, bits, taps, frames = 4, 8, 96000, 44100, 24, 1024, 960000
    rng = np.random.default_rng(4)
    base = (rng.normal(0, 0.3, (ns, frames * ch)) * 2 ** 23).clip(-2 ** 23, 2 ** 23 - 1).astype(np.int64)
    raw = np.zeros((ns, frames * ch * 3), np.uint8)
    for b in range(3):
        raw[:, b::3] = (base >> (8 * b)) & 0xFF
    del base
    cap = int(frames * dr / sr) + 64

    def run(blocks, chunks):
        r = espb.Resampler(ns, (frames // chunks) * ch, (cap // chunks + 64) * ch, sr, dr, bits, bits, ch, True, True,
                           taps, 256, mode=espb.MODE_EXACT)
        if blocks:
            r.set_biquad_time_blocks(*blocks)
        parts, per = [], frames // chunks
        for k in range(chunks):
            seg = np.ascontiguousarray(raw[:, k * per * ch * 3:(k + 1) * per * ch * 3])
            out, res = r.resample(seg, per, cap // chunks + 64, 0.0)
            assert res["frames_used"] == per
            parts.append(out[:, : res["frames_generated"] * ch * 3])
        pol = r.policy()
        r.free()
        return np.concatenate(parts, axis=1), pol

    seq, pol = run(None, 1)
    blk, _ = run((8192, 1024), 1)
    assert seq.shape == blk.shape and bits_equal(seq, blk)
    chunked, _ = run(None, 10)
    assert bits_equal(seq, chunked)
    # the first second against the CPU pipeline (one stream; 8 channels x 44100 outputs x 2048 taps on the host)
    one = 96000
    q, used, gen, _ = _composed_oracle(oracle, raw[1, : one * ch * 3], one, ch, bits, bits, taps, 256, pol,
                                       int(one * dr / sr) + 64)
    settle = gen - 600  # the one-shot CPU run has no frames after `one`, the 10 s run has: compare what both know
    assert bits_equal(seq[1, : settle * ch * 3], q[: settle * ch * 3])


@pytest.mark.parametrize("flags,lowpass", [(0, 1.0), (espb.BLACKMAN_HARRIS, 1.0), (espb.INCLUDE_LOWPASS, 0.7)])
def test_non_interpolating_kernel(oracle, flags, lowpass, monkeypatch):
    """Flags without SUBSAMPLE_INTERPOLATE take the dedicated one-filter kernel (art_resampler.cpp:421-430): bit-exact
    with the oracle in exact mode, <= 1e-6 in fast mode, and identical to the route through the interpolating kernel
    (ESPB_NI=0), over chunked calls and a partial series group."""
    ns, ch, taps, filters = 70, 2, 128, 37
    ratio = f32(44100) / f32(48000)
    total = 3000
    x = np.stack([noise(total, ch, stream=40 + s, amp=0.8) for s in range(ns)])
    results = {}
    for label, env in (("dedicated", "1"), ("via-interp", "0")):
        monkeypatch.setenv("ESPB_NI", env)
        for mode in (espb.MODE_EXACT, espb.MODE_FAST):
            b = espb.ResampleBatch(ns, ch, taps, filters, lowpass, flags, mode=mode)
            b.advance(taps / 2)
            outs, pos = [], 0
            for n_in, cap in ((1000, 2000), (7, 30), (1993, 4000)):
                y, used, gen = b.process_interleaved(x[:, pos * ch:(pos + n_in) * ch], cap, ratio, n_in=n_in)
                outs.append(y)
                pos += used
            results[(label, mode)] = np.concatenate(outs, axis=1)
            b.free()
    assert bits_equal(results[("dedicated", espb.MODE_EXACT)], results[("via-interp", espb.MODE_EXACT)])
    assert bits_equal(results[("dedicated", espb.MODE_FAST)], results[("via-interp", espb.MODE_FAST)])
    for s in (0, 63, 64, ns - 1):
        o = oracle.resampler(ch, taps, filters, lowpass, flags)
        o.advance(taps / 2)
        yo = np.concatenate([o.process_interleaved(x[s, a * ch:(a + n) * ch], cap, ratio, n_in=n)[0]
                             for a, n, cap in ((0, 1000, 2000), (1000, 7, 30), (1007, 1993, 4000))])
        assert bits_equal(results[("dedicated", espb.MODE_EXACT)][s], yo), s
        assert np.max(np.abs(results[("dedicated", espb.MODE_FAST)][s].astype(np.float64) - yo)) <= TOL


@pytest.mark.parametrize("ns", [3, 150])
def test_growing_calls_without_synchronisation(oracle, ns):
    """Calls of growing size enqueued back to back on a non-blocking stream with no host synchronisation in between:
    the staging buffers are re-allocated (and the carried frames moved) while earlier calls may still be running.
    Everything must come out as from one reference context per stream (the re-allocation waits for the device)."""
    L = espb.lib()
    ch, taps = 2, 64
    ratio = f32(48000) / f32(44100)
    sizes = [100, 300, 900, 2700, 8100]
    total = sum(sizes)
    x = np.stack([noise(total, ch, stream=700 + s, amp=0.8) for s in range(ns)])
    stream = L.espb_stream_create()
    b = espb.ResampleBatch(ns, ch, taps, 64, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(taps / 2)
    d_in = espb.DeviceBuffer.from_numpy(x)
    caps = [int(n * float(ratio)) + 8 for n in sizes]
    d_outs = [espb.DeviceBuffer(ns * c * ch * 4) for c in caps]
    results, pos = [], 0
    for n, cap, d_out in zip(sizes, caps, d_outs):
        results.append(b.process_interleaved_dev(d_in.ptr + pos * ch * 4, total * ch, n, d_out.ptr, cap * ch, cap,
                                                 ratio, stream))
        pos += n
    espb.capi._check(L.espb_stream_sync(stream), "sync")
    for s in (0, ns - 1):
        o = oracle.resampler(ch, taps, 64, 1.0, 3)
        o.advance(taps / 2)
        pos = 0
        for n, cap, d_out, (used, gen) in zip(sizes, caps, d_outs, results):
            yo, uo, go = o.process_interleaved(x[s, pos * ch:(pos + n) * ch], cap, ratio)
            assert (used, gen) == (uo, go)
            got = d_out.download(f32).reshape(ns, cap * ch)[s, : go * ch]
            assert bits_equal(got, yo), (s, n)
            pos += n
    b.free()
    L.espb_stream_destroy(stream)


def test_bad_ratios_are_refused_not_executed():
    """A NaN / non-positive / infinite ratio, or one so small that a single pass of 32 outputs spans more input than
    the kernel's per-CTA chunk table, must fail the call (ESPB_ERR_ARG through espb_last_status) and leave the context
    usable — not index shared memory out of bounds (ADVICE r1)."""
    L = espb.lib()
    ns, ch, taps = 70, 2, 256          # 140 series: the standard kernel (chunk table in shared memory)
    x = np.stack([noise(3000, ch, stream=s) for s in range(ns)])
    b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(taps / 2)
    d_in, d_out = espb.DeviceBuffer.from_numpy(x), espb.DeviceBuffer(ns * 4000 * ch * 4)
    for bad in (float("nan"), 0.0, -1.0, float("inf")):
        with pytest.raises(espb.EspbError):
            b.process_interleaved_dev(d_in.ptr, 3000 * ch, 3000, d_out.ptr, 4000 * ch, 4000, f32(bad))
        assert L.espb_last_status() == -1  # ESPB_ERR_ARG
    # ratio 0.002 over 40000 frames: 80 outputs, a pass of 32 of them spans 16000 input rows = 500 chunks > 320
    d_long = espb.DeviceBuffer(ns * 40000 * ch * 4)
    d_long.zero()
    with pytest.raises(espb.EspbError):
        b.process_interleaved_dev(d_long.ptr, 40000 * ch, 40000, d_out.ptr, 4000 * ch, 4000, f32(0.002))
    assert L.espb_last_status() == -1
    # the context is untouched: the next good call equals a fresh oracle context
    y, used, gen = b.process_interleaved(x, 3300, f32(48000) / f32(44100))
    o = espb  # noqa: F841
    from oracle_lib import Oracle
    oc = Oracle().resampler(ch, taps, 256, 1.0, 3)
    oc.advance(taps / 2)
    yo, uo, go = oc.process_interleaved(x[5], 3300, f32(48000) / f32(44100))
    assert (used, gen) == (uo, go) and bits_equal(y[5], yo)
    assert L.espb_last_status() == 0
    b.free()


@pytest.mark.parametrize("ch,planar,ns,flags", [(2, False, 200, 3), (1, False, 300, 3), (4, False, 70, 3),
                                                (2, True, 130, 3), (8, False, 40, 3),
                                                (2, False, 140, 2), (1, False, 150, 0)])  # (last two: non-interpolating)
def test_staging_overlap_is_bit_identical(oracle, ch, planar, ns, flags):
    """Long device-buffer calls launch the resampler kernel as a programmatic dependent of the transposing kernel and
    synchronise per CTA on per-row-tile counters (ESPB_OPT_OVERLAP_STAGING, default on).  Three chained calls of
    uneven length (not multiples of the 32-row tile, so the tail and the padding take the generic kernel) must give
    the bytes of the serial order, and sampled streams the oracle's bytes (exact mode)."""
    taps, filters = 64, 128
    ratio = f32(48000) / f32(44100)
    sizes = [4111, 6000, 4500]  # > 4096 frames: the fused small-call staging does not take them
    total = sum(sizes)
    x = np.stack([noise(total, ch, stream=900 + s, amp=0.7) for s in range(ns)])  # (ns, total*ch) interleaved
    outs = {}
    for overlap in (1, 0):
        b = espb.ResampleBatch(ns, ch, taps, filters, 1.0, flags, mode=espb.MODE_EXACT)
        b.set_option(espb.OPT_OVERLAP_STAGING, overlap)
        b.set_option(espb.OPT_PLAN_CACHE, 0)
        b.advance(taps / 2)
        got, pos = [], 0
        for n in sizes:
            cap = int(n * float(ratio)) + 8
            seg = x.reshape(ns, total, ch)[:, pos:pos + n, :]
            if planar:
                y, used, gen = b.process_planar(np.ascontiguousarray(seg.transpose(0, 2, 1)), cap, ratio)
                y = np.ascontiguousarray(y.transpose(0, 2, 1)).reshape(ns, -1)
            else:
                y, used, gen = b.process_interleaved(seg.reshape(ns, n * ch), cap, ratio)
            got.append((np.array(y, copy=True), used, gen))
            pos += n
        outs[overlap] = got
        b.free()
    for (y1, u1, g1), (y0, u0, g0) in zip(outs[1], outs[0]):
        assert (u1, g1) == (u0, g0) and bits_equal(y1, y0)
    for s in (0, ns // 2, ns - 1):
        o = oracle.resampler(ch, taps, filters, 1.0, flags)
        o.advance(taps / 2)
        pos = 0
        for n, (y1, u1, g1) in zip(sizes, outs[1]):
            cap = int(n * float(ratio)) + 8
            yo, uo, go = o.process_interleaved(x[s, pos * ch:(pos + n) * ch], cap, ratio)
            assert (u1, g1) == (uo, go)
            assert bits_equal(y1[s][: go * ch], yo), (s, n)
            pos += n


@pytest.mark.parametrize("db,frames", [(16, 2048), (8, 1000), (24, 777), (32, 1500)])
def test_fused_post_filter_quantiser_mono(oracle, db, frames, monkeypatch):
    """Mono up-sampling through the wrapper: the post-filter's thread quantises and packs its own results
    (espb_biquad_tm_pcm_kernel) instead of a filter pass followed by a quantising layout pass.  Same bytes and clip
    counts as the two-pass form (ESPB_FUSE_POST=0) over three chained calls, loud enough to clip, frame counts that
    leave a partial last chunk; and bit-exact against the oracle wrapper in exact mode."""
    sr, dr, sb, ch, ns = 16000, 48000, 16, 1, 150
    rng = np.random.default_rng(db + frames)
    calls = [(rng.normal(0, 0.45, size=(ns, frames)).clip(-1, 0.99997) * 32768).astype(np.int16) for _ in range(3)]
    cap = frames * 3 + 64
    results = {}
    monkeypatch.setenv("ESPB_FUSE_POST_GROUPS", "1")  # (by default only batches of >= 96 groups take the fused kernel)
    for fused in ("1", "0"):
        monkeypatch.setenv("ESPB_FUSE_POST", fused)
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 64, 64, mode=espb.MODE_EXACT)
        got = []
        for pcm in calls:
            out, res = r.resample(pcm.view(np.uint8).reshape(ns, -1), frames, cap, 3.0)
            got.append((out.copy(), res["frames_generated"], np.array(res["clipped_per_stream"]).copy()))
        results[fused] = got
        r.free()
    clipped_any = 0
    for (o1, g1, c1), (o0, g0, c0) in zip(results["1"], results["0"]):
        assert g1 == g0 and bits_equal(o1, o0) and np.array_equal(c1, c0)
        clipped_any += int(c1.sum())
    assert clipped_any > 0  # the clip-count path was exercised
    for s in (0, 77, ns - 1):
        w = oracle.wrapper(frames * ch, cap * ch, float(sr), float(dr), sb, db, ch, True, True, 64, 64)
        for pcm, (o1, g1, c1) in zip(calls, results["1"]):
            yo, ro = w.resample(pcm[s].view(np.uint8), frames, cap, 3.0)
            assert g1 == ro["frames_generated"] and bits_equal(o1[s], yo) and int(c1[s]) == ro["clipped_samples"]
