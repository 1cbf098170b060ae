"""Fast mode bit for bit.  DESIGN.md §2.2 defines fast mode as the reference loop with each multiply-add rounded once:
`acc = fmaf(h[k], x[k], acc)` for k = 0 ... T-1, one accumulator per dot product, and the blend un-fused as in exact
mode.  The oracle's fused form (oracle.resampler(..., fused=True), checked on the CPU by test_oracle_fused.py) is that
loop, so every fast-mode path must reproduce it exactly: output bytes, frames used and generated, final state and clip
counts.  The 1e-6 max-abs (and 1 LSB) checks elsewhere in the suite stay: they are the contract against the
reference; this file checks the arithmetic, where a dropped, added or re-ordered term of 1e-7 would pass that bar.

Each check also runs exact mode on the same generic input (noise and multitone at amplitude 0.9 and 1e-3) and
asserts that the fast output differs from it somewhere, so the FFMA path is the one under test.  The dyadic checks at
the end need no fused oracle: on samples 0, -0 and +-2^k every product is exact, so fast == exact == plain oracle.

Switches cached in a static (ESPB_FS_STAGES) and the ESPB_DEBUG instantiation report run in a child process that
writes its results under tmp_path; the parent compares them with the oracle."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
from conftest import bits_equal
from oracle_lib import dyadic, multitone, noise

import esp_audio_libs_b200 as espb

pytestmark = pytest.mark.gpu
f32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FAST, EXACT = espb.MODE_FAST, espb.MODE_EXACT
R48 = f32(48000) / f32(44100)


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert espb.device_count() > 0, "GPU tests need a GPU: the product has no CPU path"
    espb.set_device(0)


# ---------------------------------------------------------------- helpers
def sig(frames, ch, s, seed):
    """Stream s of a batch: noise / multitone at amplitude 0.9 / 1e-3, by s % 4 (interleaved float32)."""
    amp = 0.9 if s % 4 < 2 else 1e-3
    if s % 2 == 0:
        return noise(frames, ch, stream=seed + s, amp=amp)
    return multitone(frames, ch, 44100.0, stream=seed + s, amp=amp)


def sigs(ns, frames, ch, seed):
    return np.stack([sig(frames, ch, s, seed) for s in range(ns)])


def probes_of(ns):
    """the four signal kinds, the 128-series group edges, the last stream"""
    return sorted({s for s in (0, 1, 2, 3, 31, 32, 63, 64, 127, 128, ns - 2, ns - 1) if 0 <= s < ns})


def run_child(tmp_path, func, env, timeout=900):
    """Run `func(out_dir)` of this module in a fresh interpreter with `env` added; returns its stderr."""
    code = (f"import sys; sys.path[:0] = [{HERE!r}, {ROOT!r}]; import test_gpu_fast_mode as t; "
            f"t.{func}({str(tmp_path)!r})")
    p = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=timeout)
    assert p.returncode == 0, p.stderr[-4000:]
    return p.stderr


def oracle_chain(oracle, row, ch, geo, calls, ratios, fused=True, adv=None):
    """One oracle context fed `calls` [(n_in, cap)] from `row`, each call's input starting at the first frame the
    previous call did not use.  Returns ([(y, used, generated)], final state)."""
    taps, filters, lp, flags = geo
    o = oracle.resampler(ch, taps, filters, lp, flags, fused=fused)
    o.advance(taps / 2 if adv is None else adv)
    out, pos = [], 0
    for (n_in, cap), ratio in zip(calls, ratios):
        assert (pos + n_in) * ch <= row.size  # the oracle reads n_in frames, whatever the slice holds
        y, u, g = o.process_interleaved(row[pos * ch:(pos + n_in) * ch], cap, ratio, n_in=n_in)
        out.append((y, u, g))
        pos += u
    return out, o.state()


def device_chain(b, x, calls, ratios):
    ch = b.channels
    out, pos = [], 0
    for (n_in, cap), ratio in zip(calls, ratios):
        seg = np.ascontiguousarray(x[:, pos * ch:(pos + n_in) * ch])
        assert seg.shape[1] == n_in * ch
        y, u, g = b.process_interleaved(seg, cap, ratio, n_in=n_in)
        out.append((np.array(y, copy=True), u, g))
        pos += u
    return out


def batch(ns, ch, geo, mode, adv=None):
    taps, filters, lp, flags = geo
    b = espb.ResampleBatch(ns, ch, taps, filters, lp, flags, mode=mode)
    b.advance(taps / 2 if adv is None else adv)
    return b


def run_modes(ns, ch, geo, x, calls, ratios, adv=None):
    """The same chained calls in fast and exact mode: {mode: (chain, final state)}."""
    out = {}
    for mode in (FAST, EXACT):
        b = batch(ns, ch, geo, mode, adv)
        out[mode] = (device_chain(b, x, calls, ratios), b.state())
        b.free()
    return out


def assert_chain(got, ref, probes, what):
    """got: device chain (all streams); ref: {stream: oracle chain}; bytes and counts, call by call."""
    for s in probes:
        for k, ((y, u, g), (yo, uo, go)) in enumerate(zip(got, ref[s])):
            assert (u, g) == (uo, go), (what, s, k, (u, g), (uo, go))
            assert bits_equal(y[s], yo), (what, s, k, float(np.max(np.abs(y[s].astype(np.float64) - yo))))


def assert_fast_path(fast, exact, what):
    """the fast chain is not the exact one: the FFMA path ran"""
    assert any(not bits_equal(a[0], b[0]) for a, b in zip(fast, exact)), (what, "fast output == exact output")


def check_modes(oracle, ns, ch, geo, x, calls, ratios, what, probes=None, adv=None):
    """Fast mode bit-exact against the fused oracle (bytes, counts, state), and different from exact mode."""
    probes = probes_of(ns) if probes is None else probes
    runs = run_modes(ns, ch, geo, x, calls, ratios, adv)
    ref = {s: oracle_chain(oracle, x[s], ch, geo, calls, ratios, adv=adv) for s in probes}
    assert_chain(runs[FAST][0], {s: r[0] for s, r in ref.items()}, probes, what)
    assert runs[FAST][1] == ref[probes[0]][1], what
    assert_fast_path(runs[FAST][0], runs[EXACT][0], what)
    return runs


def split3(n_in, ratio):
    """three chained calls over at most n_in frames: a third, a capacity-limited one, the rest of the input"""
    a, b = n_in // 3 + 1, n_in // 3
    return [(a, int(a * float(ratio)) + 40), (b, 37), (n_in - a - b, int(n_in * float(ratio)) + 40)]


def pcm_bytes(codes, nb):
    raw = np.zeros(codes.shape[:-1] + (codes.shape[-1] * nb,), np.uint8)
    for b in range(nb):
        raw[..., b::nb] = (codes >> (8 * b)) & 0xFF
    return raw


def pcm_noise(rng, ns, n, bits, std=0.3, amp=1.0):
    nb = (bits + 7) // 8
    codes = (rng.normal(0, std, size=(ns, n)).clip(-1, 0.99999) * amp * (2 ** (8 * nb - 1))).astype(np.int64)
    return pcm_bytes(codes, nb)


def composed_fused(oracle, pol, ch, sb, db, taps, filters, raws, frames, cap, gain_db, fused=True):
    """One stream through the oracle's stages with the policy the library reports, state carried over the calls in
    `raws` (any channel count; the oracle wrapper holds filters for two channels only).  Returns [(q, used, gen,
    clipped)]."""
    o = oracle.resampler(ch, taps, filters, float(pol["art_lowpass"]), pol["art_flags"], fused=fused)
    o.advance(taps / 2.0)
    bq = [[oracle.biquad(pol["coeffs"], 1.0) for _ in range(2)] for _ in range(ch)]
    out = []
    for raw in raws:
        xf = oracle.quantized_to_float(raw, frames * ch, sb, gain_db)
        if pol["filter"] == "pre":
            for c in range(ch):
                for k in range(2):
                    bq[c][k].apply_buffer(xf[c:], ch, n=frames)
        yf, used, gen = o.process_interleaved(xf, cap, pol["sample_ratio"], n_in=frames)
        assert used == frames  # (the stages above took every frame: the wrapper's call must have too)
        yf = np.ascontiguousarray(yf)
        if pol["filter"] == "post":
            for c in range(ch):
                for k in range(2):
                    bq[c][k].apply_buffer(yf[c:], ch, n=gen)
        q, clipped = oracle.float_to_quantized(yf, db)
        out.append((q, used, gen, clipped))
    return out


# ---------------------------------------------------------------- 1. standard kernel, default geometry
VS_ORACLE = [  # test_gpu_parity.py::test_resampler_vs_oracle
    (2, 70, 256, 256, 1.0, 3, f32(48000) / f32(44100), 2500),
    (2, 65, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 2500),
    (1, 131, 256, 256, 1.0, 1, f32(3.0), 900),
    (8, 17, 1024, 256, 0.45, 1, f32(44100) / f32(96000), 3000),
    (3, 45, 32, 16, 1.0, 0, f32(1.37), 1500),
    (1, 1, 4, 2, 1.0, 3, f32(2.5), 300),
    (5, 30, 64, 1024, 0.7, 2, f32(0.61), 2000),
]


@pytest.mark.parametrize("case", VS_ORACLE)
def test_resampler_cases(oracle, case):
    """The seven geometries of test_resampler_vs_oracle, one call, every stream against the fused oracle."""
    ch, ns, taps, filters, lp, flags, ratio, n_in = case
    x = sigs(ns, n_in, ch, seed=100)
    cap = int(n_in * float(ratio)) + 40
    check_modes(oracle, ns, ch, (taps, filters, lp, flags), x, [(n_in, cap)], [ratio], case, probes=range(ns))


def test_chained_capacity_limited_and_empty_calls(oracle):
    """Chained uneven calls with empty calls (no input, no room; no input, room for the leading half window) and
    capacity-limited ones, on 70 stereo streams at T = 256 and 3 mono streams at T = 64."""
    for ns, ch, taps in ((70, 2, 256), (3, 1, 64)):
        geo = (taps, taps, 1.0, 3)
        ratio = f32(1.5)
        calls = [(0, 0), (0, 100), (500, 37), (1200, 300), (10, 9), (2000, 4000), (0, 50)]
        x = sigs(ns, sum(c[0] for c in calls), ch, seed=200)
        check_modes(oracle, ns, ch, geo, x, calls, [ratio] * len(calls), (ns, ch, taps))


def test_planar_io_and_pointer_tables(oracle):
    """Planar buffers (process_planar) and one buffer per (stream, channel) plane (process_planes), two calls each, on
    the standard kernel (140 series) and the few-series one (2 x 5 channels)."""
    taps, filters = 64, 32
    geo = (taps, filters, 1.0, 3)
    for ns, ch in ((70, 2), (2, 5)):
        n_in = 1500
        x = sigs(ns, n_in, ch, seed=300)  # interleaved
        ref = {s: oracle_chain(oracle, x[s], ch, geo, [(700, 1000), (800, 1000)], [R48] * 2)[0] for s in range(ns)}
        ys = {}
        for mode in (FAST, EXACT):
            for form in ("planar", "planes"):
                b = batch(ns, ch, geo, mode)
                got = []
                for a, e in ((0, 700), (700, n_in)):
                    seg = x.reshape(ns, n_in, ch)[:, a:e, :].transpose(0, 2, 1)  # (ns, ch, frames)
                    if form == "planar":
                        y, u, g = b.process_planar(np.ascontiguousarray(seg), 1000, R48)
                        y = np.ascontiguousarray(np.asarray(y)[:, :, :g].transpose(0, 2, 1)).reshape(ns, -1)
                    else:
                        planes = [np.ascontiguousarray(seg[s, c]) for s in range(ns) for c in range(ch)]
                        yp, u, g = b.process_planes(planes, 1000, R48)
                        y = np.stack([np.stack([yp[s * ch + c][:g] for c in range(ch)], axis=1).reshape(-1)
                                      for s in range(ns)])
                    got.append((y, u, g))
                b.free()
                ys[(mode, form)] = got
        for form in ("planar", "planes"):
            assert_chain(ys[(FAST, form)], ref, range(ns), (ns, ch, form))
            assert_fast_path(ys[(FAST, form)], ys[(EXACT, form)], (ns, ch, form))


@pytest.mark.parametrize("ch,pad,skew", [(2, 2, 0), (2, 1, 1), (1, 1, 0), (1, 3, 1), (4, 2, 2), (8, 4, 1), (1, 4, 0),
                                         (2, 4, 0), (4, 4, 0), (8, 8, 4)])
def test_float_rows_of_any_alignment(oracle, ch, pad, skew):
    """The row shapes of test_resampler_float_rows_of_any_alignment (16-, 8- and 4-byte aligned rows, buffers offset by
    `skew` floats): the vectorised, 8-byte and scalar forms of the layout stages around the fast kernel."""
    taps, filters, ns, n_in = 64, 32, 9, 300
    ratio = f32(1.25)
    cap = int(n_in * 1.25) + 8
    x = sigs(ns, n_in, ch, seed=700)
    in_stride, out_stride = n_in * ch + pad, cap * ch + pad
    hin = np.zeros(ns * in_stride + skew, f32)
    for s in range(ns):
        hin[skew + s * in_stride: skew + s * in_stride + n_in * ch] = x[s]
    d_in = espb.DeviceBuffer.from_numpy(hin)
    d_out = espb.DeviceBuffer((ns * out_stride + skew) * 4)
    got = {}
    for mode in (FAST, EXACT):
        d_out.zero()
        b = batch(ns, ch, (taps, filters, 1.0, 3), mode)
        used, gen = b.process_interleaved_dev(d_in.ptr + 4 * skew, in_stride, n_in, d_out.ptr + 4 * skew, out_stride,
                                              cap, ratio)
        b.free()
        raw = d_out.download(f32)[skew:skew + ns * out_stride].reshape(ns, out_stride)
        assert not raw[:, gen * ch:].any()  # nothing written past the generated frames
        got[mode] = [(raw[:, : gen * ch].copy(), used, gen)]
    d_in.free()
    d_out.free()
    ref = {s: oracle_chain(oracle, x[s], ch, (taps, filters, 1.0, 3), [(n_in, cap)], [ratio])[0] for s in range(ns)}
    assert_chain(got[FAST], ref, range(ns), (ch, pad, skew))
    assert_fast_path(got[FAST], got[EXACT], (ch, pad, skew))


@pytest.mark.parametrize("slabs", [None, "1", "3"])
def test_host_buffer_path(oracle, monkeypatch, slabs):
    """process_interleaved_host over two chained calls, with the default stream slabs and ESPB_HOST_SLABS = 1 and 3
    (150 stereo streams: two 128-series groups per slab at most)."""
    if slabs:
        monkeypatch.setenv("ESPB_HOST_SLABS", slabs)
    ch, ns = 2, 150
    geo = (64, 64, 1.0, 3)
    calls = [(1500, 1700), (1300, 1000)]
    x = sigs(ns, sum(c[0] for c in calls), ch, seed=400)
    got = {}
    for mode in (FAST, EXACT):
        b = batch(ns, ch, geo, mode)
        chain, pos = [], 0
        for n_in, cap in calls:
            hin = espb.PinnedBuffer(ns * n_in * ch, f32)
            hin.array[:] = x[:, pos * ch:(pos + n_in) * ch].reshape(-1)
            hout = espb.PinnedBuffer(ns * cap * ch, f32)
            hout.array[:] = 0
            u, g = b.process_interleaved_host(hin.ptr, n_in * ch, n_in, hout.ptr, cap * ch, cap, R48)
            chain.append((hout.array.reshape(ns, cap * ch)[:, : g * ch].copy(), u, g))
            pos += u
            hin.free()
            hout.free()
        got[mode] = (chain, b.state())
        b.free()
    probes = probes_of(ns)
    ref = {s: oracle_chain(oracle, x[s], ch, geo, calls, [R48] * 2) for s in probes}
    assert_chain(got[FAST][0], {s: r[0] for s, r in ref.items()}, probes, slabs)
    assert got[FAST][1] == ref[0][1]
    assert_fast_path(got[FAST][0], got[EXACT][0], slabs)


@pytest.mark.parametrize("overlap", [1, 0])
def test_staging_overlap(oracle, overlap):
    """Long device-buffer calls (> 4096 frames) with the resampler launched while the staging kernel still writes
    (ESPB_OPT_OVERLAP_STAGING = 1) and in the serial order (0); three chained calls, stereo and 4-channel."""
    for ns, ch in ((200, 2), (70, 4)):
        geo = (64, 128, 1.0, 3)
        calls = [(4111, 4500), (6000, 6540), (4500, 4900)]
        x = sigs(ns, sum(c[0] for c in calls), ch, seed=500)
        runs = {}
        for mode in (FAST, EXACT):
            b = batch(ns, ch, geo, mode)
            b.set_option(espb.OPT_OVERLAP_STAGING, overlap)
            b.set_option(espb.OPT_PLAN_CACHE, 0)
            runs[mode] = device_chain(b, x, calls, [R48] * 3)
            b.free()
        probes = probes_of(ns)
        ref = {s: oracle_chain(oracle, x[s], ch, geo, calls, [R48] * 3)[0] for s in probes}
        assert_chain(runs[FAST], ref, probes, (ns, ch, overlap))
        assert_fast_path(runs[FAST], runs[EXACT], (ns, ch, overlap))


@pytest.mark.parametrize("env", [{"ESPB_G_MBYTES": "1"}, {"ESPB_PPC": "7"}, {"ESPB_SCHED": "seq"}],
                         ids=["g_slabs", "ppc7", "sched_seq"])
def test_host_switches(oracle, monkeypatch, env):
    """G made resident in 1 MB time slabs (several resampler launches per call), 7 passes per CTA (a partial last
    pass range), and the host-built sequential schedule: 150 stereo streams, T = 256, three chained calls."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ns, ch = 150, 2
    geo = (256, 256, 1.0, 3)
    calls = [(4500, 5000), (900, 300), (1202, 1400)]
    x = sigs(ns, sum(c[0] for c in calls), ch, seed=600)
    check_modes(oracle, ns, ch, geo, x, calls, [R48] * 3, env)


def test_full_size_batch(oracle):
    """BASELINE configs[1] in fast mode: 4096 stereo streams, 256 taps, 44.1 -> 48 kHz, 0.25 s each, every stream its
    own input; the first, the last and eight seeded streams bit-exact against the fused oracle."""
    ns, ch, taps, n_in = 4096, 2, 256, 11025
    rng = np.random.default_rng(41)
    x = rng.standard_normal((ns, n_in * ch), dtype=f32)
    x *= np.where(np.arange(ns) % 2 == 0, f32(0.3), f32(3e-4))[:, None]  # loud and quiet rows
    cap = int(n_in * float(R48)) + 16
    d_in = espb.DeviceBuffer.from_numpy(x)
    d_out = espb.DeviceBuffer(ns * cap * ch * 4)
    got = {}
    for mode in (FAST, EXACT):
        d_out.zero()
        b = batch(ns, ch, (taps, 256, 1.0, 3), mode)
        used, gen = b.process_interleaved_dev(d_in.ptr, n_in * ch, n_in, d_out.ptr, cap * ch, cap, R48)
        b.free()
        y = d_out.download(f32).reshape(ns, cap * ch)
        assert not y[:, gen * ch:].any()
        got[mode] = (y[:, : gen * ch], used, gen)
    d_in.free()
    d_out.free()
    sampled = sorted({0, 1, ns - 1} | set(int(s) for s in rng.choice(ns, 8, replace=False)))
    ref = {s: oracle_chain(oracle, x[s], ch, (taps, 256, 1.0, 3), [(n_in, cap)], [R48])[0] for s in sampled}
    assert_chain([got[FAST]], ref, sampled, "configs[1]")
    assert_fast_path([got[FAST]], [got[EXACT]], "configs[1]")


# ---------------------------------------------------------------- 2. all geometries of the standard kernel (child)
GEOMETRIES = [(4, 32), (8, 32), (4, 16), (8, 16), (4, 24), (4, 36)]  # (ESPB_BPP, ESPB_CHUNK_ROWS)
GEO_CALLS = [(4500, 5000), (900, 300), (1202, 1400)]
GEO_SHAPE = (70, 2, (256, 256, 1.0, 3))  # 140 series: a full 128-series group and a partial one
WRAP_CALLS = [(4500, 4950), (900, 300), (1202, 1400)]  # 44.1 -> 48 kHz stereo int16: post-filter, time-major output


def _wrap_raw():
    rng = np.random.default_rng(77)
    return pcm_noise(rng, 70, sum(c[0] for c in WRAP_CALLS) * 2, 16, std=0.45)


def _wrapper_chain(r, raw, ch, nb, calls, gain_db, host_path=False):
    out, pos = [], 0
    for n_in, cap in calls:
        seg = np.ascontiguousarray(raw[:, pos * ch * nb:(pos + n_in) * ch * nb])
        y, res = r.resample(seg, n_in, cap, gain_db, host_path=host_path)
        out.append((y, res["frames_used"], res["frames_generated"], np.array(res["clipped_per_stream"]).copy()))
        pos += res["frames_used"]
    return out


def _oracle_wrapper_chain(oracle, raw_row, ch, nb, sr, dr, sb, db, calls, gain_db, taps=256, filters=256, fused=True):
    w = oracle.wrapper(max(c[0] for c in calls) * ch, max(c[1] for c in calls) * ch, float(sr), float(dr), sb, db, ch,
                       True, True, taps, filters, fused=fused)
    out, pos = [], 0
    for n_in, cap in calls:
        y, ro = w.resample(np.ascontiguousarray(raw_row[pos * ch * nb:(pos + n_in) * ch * nb]), n_in, cap, gain_db)
        out.append((y, ro["frames_used"], ro["frames_generated"], ro["clipped_samples"]))
        pos += ro["frames_used"]
    return out


def _assert_wrapper(got, ref, probes, what):
    for s in probes:
        for k, ((y, u, g, clips), (yo, uo, go, co)) in enumerate(zip(got, ref[s])):
            assert (u, g) == (uo, go), (what, s, k)
            assert bits_equal(y[s], yo), (what, s, k)
            assert int(clips[s]) == co, (what, s, k)


def _assert_wrapper_fast_path(fast, exact, what):
    assert any(not bits_equal(a[0], b[0]) for a, b in zip(fast, exact)), (what, "fast PCM == exact PCM")


def _child_geometries(out_dir):
    espb.set_device(0)
    ns, ch, geo = GEO_SHAPE
    x = sigs(ns, sum(c[0] for c in GEO_CALLS), ch, seed=800)
    raw = _wrap_raw()
    saved = {}
    for bpp, rows in GEOMETRIES:
        os.environ["ESPB_BPP"], os.environ["ESPB_CHUNK_ROWS"] = str(bpp), str(rows)
        for mode in (FAST, EXACT):
            b = batch(ns, ch, geo, mode)
            for k, (y, u, g) in enumerate(device_chain(b, x, GEO_CALLS, [R48] * 3)):
                saved[f"{bpp}_{rows}_{mode}_{k}_y"] = y
                saved[f"{bpp}_{rows}_{mode}_{k}_n"] = np.array([u, g], np.int64)
            st = b.state()
            saved[f"{bpp}_{rows}_{mode}_state"] = np.array([st[0], st[1]], np.float64)
            b.free()
            r = espb.Resampler(ns, 4500 * 2, 4950 * 2, 44100, 48000, 16, 16, 2, True, True, 256, 256, mode=mode)
            assert r.policy()["filter"] == "post"
            for k, (y, u, g, clips) in enumerate(_wrapper_chain(r, raw, 2, 2, WRAP_CALLS, 2.0)):
                saved[f"w_{bpp}_{rows}_{mode}_{k}_y"] = y
                saved[f"w_{bpp}_{rows}_{mode}_{k}_res"] = np.concatenate([[u, g], clips]).astype(np.int64)
            r.free()
    np.savez(os.path.join(out_dir, "geo.npz"), **saved)


def _load_chain(m, key):
    return [(m[f"{key}_{k}_y"], *[int(v) for v in m[f"{key}_{k}_n"]]) for k in range(3)]


def _load_wrapper_chain(m, key):
    out = []
    for k in range(3):
        res = m[f"{key}_{k}_res"]
        out.append((m[f"{key}_{k}_y"], int(res[0]), int(res[1]), res[2:]))
    return out


def test_all_geometries(oracle, tmp_path):
    """All six (ESPB_BPP, ESPB_CHUNK_ROWS) geometries in fast mode, on caller-layout output (70 stereo streams, T =
    256, three chained calls) and on time-major output (the wrapper's post-filter, 16-bit PCM, +2 dB so some samples
    clip): every fast instantiation resample<BPP, NST, ROWS, 0, TMCAP> — twelve, named by the ESPB_DEBUG report of the
    child — bit-exact against the fused oracle."""
    err = run_child(tmp_path, "_child_geometries", {"ESPB_DEBUG": "1"})
    seen = set(re.findall(r"\[espb\] resample<(\d+),(\d+),(\d+),0,(\d)>", err))
    stages = {(4, 32): 2, (8, 32): 3, (4, 16): 4, (8, 16): 6, (4, 24): 3, (4, 36): 2}
    want = {(str(b), str(stages[(b, r)]), str(r), str(t)) for b, r in GEOMETRIES for t in (0, 1)}
    assert seen >= want, sorted(want - seen)
    m = np.load(tmp_path / "geo.npz")
    ns, ch, geo = GEO_SHAPE
    x = sigs(ns, sum(c[0] for c in GEO_CALLS), ch, seed=800)
    probes = probes_of(ns)
    ref = {s: oracle_chain(oracle, x[s], ch, geo, GEO_CALLS, [R48] * 3) for s in probes}
    raw = _wrap_raw()
    wprobes = (0, 1, 2, 3, 31, 32, 63, 64, 69)
    wref = {s: _oracle_wrapper_chain(oracle, raw[s], 2, 2, 44100, 48000, 16, 16, WRAP_CALLS, 2.0) for s in wprobes}
    assert sum(c[3] for chain in wref.values() for c in chain) > 0  # clip counts were compared
    for bpp, rows in GEOMETRIES:
        key = f"{bpp}_{rows}"
        fast, exact = _load_chain(m, f"{key}_{FAST}"), _load_chain(m, f"{key}_{EXACT}")
        assert_chain(fast, {s: r[0] for s, r in ref.items()}, probes, key)
        sv = m[f"{key}_{FAST}_state"]
        assert (f32(sv[0]), int(sv[1])) == ref[0][1], key
        assert_fast_path(fast, exact, key)
        wf, we = _load_wrapper_chain(m, f"w_{key}_{FAST}"), _load_wrapper_chain(m, f"w_{key}_{EXACT}")
        _assert_wrapper(wf, wref, wprobes, ("wrapper", key))
        _assert_wrapper_fast_path(wf, we, ("wrapper", key))


# ---------------------------------------------------------------- 3. non-interpolating kernel, direct input
@pytest.mark.parametrize("flags,lowpass", [(0, 1.0), (espb.BLACKMAN_HARRIS, 1.0), (espb.INCLUDE_LOWPASS, 0.7),
                                           (espb.BLACKMAN_HARRIS | espb.INCLUDE_LOWPASS, 0.7)])
def test_non_interpolating_kernel(oracle, flags, lowpass):
    """Flags without SUBSAMPLE_INTERPOLATE (0, 2, 4, 6): the one-filter kernel, nearest phase including phase F (the
    extra bank row), chunked calls, a partial series group."""
    ns, ch, taps, filters = 70, 2, 128, 37
    ratio = f32(44100) / f32(48000)
    geo = (taps, filters, lowpass, flags)
    calls = [(1000, 2000), (7, 30), (1993, 4000)]
    eff = flags | espb.INCLUDE_LOWPASS if lowpass < 1 else flags
    s = espb.plan_schedule(taps, filters, eff, f32(taps), taps, 1000, 2000, ratio)
    assert int(s["phase"].max()) == filters and set(np.unique(s["kind"])) <= {1, 2}  # nearest phase F is reached
    x = sigs(ns, sum(c[0] for c in calls), ch, seed=900)
    check_modes(oracle, ns, ch, geo, x, calls, [ratio] * 3, (flags, lowpass))


@pytest.mark.parametrize("taps", [64, 256])
def test_direct_input(oracle, monkeypatch, taps):
    """ESPB_DIRECT=1: interleaved stereo read by the kernel through a TMA tensor map; chunked calls of changing size
    (some shorter than T, which take the staged path and hand the history over), capacity-limited calls."""
    monkeypatch.setenv("ESPB_DIRECT", "1")
    ns, ch = 70, 2
    geo = (taps, 64, 1.0, 3)
    calls = [(1000, 2000), (10, 50), (900, 300), (64, 500), (2, 9), (1500, 4000), (700, 4000)]
    x = sigs(ns, sum(c[0] for c in calls), ch, seed=1000)
    check_modes(oracle, ns, ch, geo, x, calls, [R48] * len(calls), ("direct", taps))


# ---------------------------------------------------------------- 4. few-series kernel
FEW = [
    # channels, streams, taps, filters, lowpass, flags, ratio, n_in     series -> series per lane
    (1, 1, 256, 256, 1.0, 3, R48, 5000),                              # 1 -> 2
    (2, 1, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 5000),  # 2 -> 2
    (1, 2, 4, 2, 1.0, 3, f32(2.5), 300),                              # 2 -> 2
    (3, 1, 64, 16, 1.0, 0, f32(1.37), 3000),                          # 3 -> 4
    (2, 2, 128, 37, 0.7, 4, f32(0.61), 4000),                         # 4 -> 4
    (1, 4, 256, 256, 1.0, 3, f32(3.0), 1500),                         # 4 -> 4
    (8, 1, 1024, 256, 0.45, 1, f32(44100) / f32(96000), 9000),        # 8 -> 8
    (5, 3, 32, 1024, 1.0, 2, f32(0.61), 2000),                        # 15 -> 8
    (2, 9, 256, 256, 1.0, 3, R48, 2500),                              # 18 -> 8
    (8, 4, 256, 64, 1.0, 1, f32(2.0), 1500),                          # 32 -> 8, pass-through / single-filter outputs
    (1, 16, 256, 256, 1.0, 3, R48, 2000),                             # 16 -> 8
    (2, 16, 64, 64, 1.0, 3, f32(0.21), 6000),                         # 32 -> 8, strong down-sampling
    (6, 1, 256, 1024, 1.0, 3, f32(1.0001), 3000),                     # 6 -> 8
]


@pytest.mark.parametrize("case", FEW)
def test_few_series_forms(oracle, case):
    """<= 32 series: the lanes-over-time kernel in its 2-, 4- and 8-series-per-lane forms (1-8 channels, 1-16
    streams), three chained calls; every stream against the fused oracle."""
    ch, ns, taps, filters, lp, flags, ratio, n_in = case
    x = sigs(ns, n_in, ch, seed=1100)
    check_modes(oracle, ns, ch, (taps, filters, lp, flags), x, split3(n_in, ratio), [ratio] * 3, case,
                probes=range(ns))


SWITCH_SHAPES = [(1, 2), (4, 8)]
R_LOW = f32(0.015)


def _switch_calls(ch):
    # 48/44.1 (few-series), 0.015 (its input tile no longer fits: the standard kernel), 48/44.1 again
    return [(2000, 2300), (30000 if ch == 2 else 3000, 600), (2000, 2300)], [R48, R_LOW, R48]


def _switch_runs(ns, ch):
    calls, ratios = _switch_calls(ch)
    x = sigs(ns, sum(c[0] for c in calls), ch, seed=1200 + ch)
    return x, run_modes(ns, ch, (256, 256, 1.0, 3), x, calls, ratios)


def _check_switch(oracle, runs, x, ns, ch, what):
    calls, ratios = _switch_calls(ch)
    ref = {s: oracle_chain(oracle, x[s], ch, (256, 256, 1.0, 3), calls, ratios) for s in range(ns)}
    assert_chain(runs[FAST][0], {s: r[0] for s, r in ref.items()}, range(ns), what)
    assert runs[FAST][1] == ref[0][1], what
    assert_fast_path(runs[FAST][0], runs[EXACT][0], what)


@pytest.mark.parametrize("slice_kb", [None, "1", "1000"])
def test_few_series_slices_and_kernel_switch(oracle, monkeypatch, slice_kb):
    """One stereo stream and 4 x 8 channels switching few-series -> standard -> few-series kernel within one context,
    with the default slice width, kt = 4 (ESPB_FS_SLICE_KB=1) and kt = 64 (ESPB_FS_SLICE_KB=1000)."""
    if slice_kb:
        monkeypatch.setenv("ESPB_FS_SLICE_KB", slice_kb)
    for ns, ch in SWITCH_SHAPES:
        x, runs = _switch_runs(ns, ch)
        _check_switch(oracle, runs, x, ns, ch, (ns, ch, slice_kb))


def _child_fs_stages(out_dir):
    espb.set_device(0)
    saved = {}
    for ns, ch in SWITCH_SHAPES:
        _, runs = _switch_runs(ns, ch)
        for mode in (FAST, EXACT):
            for k, (y, u, g) in enumerate(runs[mode][0]):
                saved[f"{ns}_{ch}_{mode}_{k}_y"] = y
                saved[f"{ns}_{ch}_{mode}_{k}_n"] = np.array([u, g], np.int64)
            saved[f"{ns}_{ch}_{mode}_state"] = np.array(runs[mode][1], np.float64)
    np.savez(os.path.join(out_dir, "fs.npz"), **saved)


@pytest.mark.parametrize("stages", ["3", "4"])
def test_few_series_ring_depth(oracle, tmp_path, stages):
    """ESPB_FS_STAGES (read once per process) = 3 and 4, over the kernel-switching calls, in a child process."""
    run_child(tmp_path, "_child_fs_stages", {"ESPB_FS_STAGES": stages})
    m = np.load(tmp_path / "fs.npz")
    for ns, ch in SWITCH_SHAPES:
        calls, _ = _switch_calls(ch)
        x = sigs(ns, sum(c[0] for c in calls), ch, seed=1200 + ch)
        runs = {}
        for mode in (FAST, EXACT):
            sv = m[f"{ns}_{ch}_{mode}_state"]
            runs[mode] = (_load_chain(m, f"{ns}_{ch}_{mode}"), (f32(sv[0]), int(sv[1])))
        _check_switch(oracle, runs, x, ns, ch, (ns, ch, stages))


def test_c1_ten_seconds_both_kernels(oracle, golden, monkeypatch):
    """C1: 10 s of 44.1 -> 48 kHz stereo (479880 frames, one call) through the few-series kernel (ESPB_FS=1) and the
    standard one (ESPB_FS=0): both bit-exact against the fused oracle and byte-identical to each other."""
    _, meta = golden
    c = [m for m in meta["large"] if m["name"] == "C1_10s"][0]
    x = noise(c["n_in"], c["channels"], stream=1, amp=0.5)
    geo = (c["taps"], c["filters"], c["lowpass"], c["flags"])
    calls, ratios = [(c["n_in"], c["cap"])], [f32(c["ratio"])]
    got = {}
    for fs in ("1", "0"):
        monkeypatch.setenv("ESPB_FS", fs)
        got[fs] = run_modes(1, c["channels"], geo, x.reshape(1, -1), calls, ratios)
    ref, state = oracle_chain(oracle, x, c["channels"], geo, calls, ratios)
    assert ref[0][1:] == (c["used"], c["generated"])
    for fs in ("1", "0"):
        assert_chain(got[fs][FAST][0], {0: ref}, [0], ("C1", fs))
        assert got[fs][FAST][1] == state
        assert_fast_path(got[fs][FAST][0], got[fs][EXACT][0], ("C1", fs))
    assert bits_equal(got["1"][FAST][0][0][0], got["0"][FAST][0][0][0])


# ---------------------------------------------------------------- 5. clock groups
def _group_calls(n_groups, seed):
    rng = np.random.default_rng(seed)
    base = [f32(rng.choice([48000 / 44100, 44100 / 48000, 2.0, 0.5, 1.0, 1.37])) for _ in range(n_groups)]
    calls = []
    for call in range(6):
        n_in = [int(rng.integers(0, 500)) for _ in range(n_groups)]
        n_out = [int(rng.integers(0, 900)) for _ in range(n_groups)]
        ratios = [f32(base[k] * f32(1.0 + 3e-4 * np.sin(call + k))) for k in range(n_groups)]
        calls.append((n_in, n_out, ratios))
    return calls


def _run_groups(shape, x, calls, mode, fused, geo):
    n_groups, spg, ch = shape
    taps, filters, lp, flags = geo
    os.environ["ESPB_GROUPS_FUSED"] = "1" if fused else "0"
    try:
        g = espb.ResampleGroups([spg] * n_groups, ch, taps, filters, lp, flags, mode=mode)
    finally:
        del os.environ["ESPB_GROUPS_FUSED"]
    assert g.is_fused() == fused
    for k in range(n_groups):
        g.advance(k, taps / 2)
    ns, total = n_groups * spg, x.shape[1] // ch
    pos, outs = [0] * n_groups, []
    for n_in, n_out, ratios in calls:
        n_in = [min(n_in[k], total - pos[k]) for k in range(n_groups)]
        xin = np.zeros((ns, max(max(n_in), 1) * ch), f32)
        for s in range(ns):
            k = s // spg
            xin[s, : n_in[k] * ch] = x[s, pos[k] * ch:(pos[k] + n_in[k]) * ch]
        y, res = g.process_interleaved(xin, n_in, n_out, ratios)
        outs.append((xin, n_in, np.array(y, copy=True), res))
        for k in range(n_groups):
            pos[k] += res[k][0]
    states = [g.state(k) for k in range(n_groups)]
    g.free()
    return outs, states


@pytest.mark.parametrize("shape", [(40, 1, 2), (9, 4, 3), (5, 2, 1)])  # groups, streams per group, channels
def test_clock_groups(oracle, shape):
    """Per-group ratios drifting from call to call and per-group chunk sizes, in the fused form (one launch for all
    groups) and with one context per group: fast mode bit-exact against one fused-oracle context per stream, the two
    forms byte-identical."""
    n_groups, spg, ch = shape
    geo = (64, 128, 1.0, 3)
    ns = n_groups * spg
    x = sigs(ns, 3000, ch, seed=1300)
    calls = _group_calls(n_groups, seed=7)
    runs = {(mode, fused): _run_groups(shape, x, calls, mode, fused, geo) for mode in (FAST, EXACT)
            for fused in (True, False)}
    orc = [oracle.resampler(ch, *geo, fused=True) for _ in range(ns)]
    for o in orc:
        o.advance(geo[0] / 2)
    differ = False
    for c, (xin, n_in, y, res) in enumerate(runs[(FAST, True)][0]):
        _, _, yp, resp = runs[(FAST, False)][0][c]
        assert res == resp and bits_equal(y, yp), (shape, c)  # fused form == one context per group
        ye = runs[(EXACT, True)][0][c][2]
        n_out, ratios = calls[c][1], calls[c][2]
        for s in range(ns):
            k = s // spg
            yo, uo, go = orc[s].process_interleaved(xin[s, : n_in[k] * ch], n_out[k], ratios[k], n_in=n_in[k])
            assert res[k] == (uo, go), (shape, c, s)
            assert bits_equal(y[s, : go * ch], yo), (shape, c, s)
            differ |= not bits_equal(y[s, : go * ch], ye[s, : go * ch])
    assert runs[(FAST, True)][1] == runs[(FAST, False)][1] == [orc[k * spg].state() for k in range(n_groups)]
    assert differ, (shape, "fast output == exact output")


# ---------------------------------------------------------------- 6. the wrapper
@pytest.mark.parametrize("cfg", [
    # src_rate, dst_rate, src_bits, dst_bits, channels, streams   (test_wrapper_vs_oracle_fast_mode_within_one_lsb)
    (16000, 48000, 16, 16, 1, 133),
    (96000, 44100, 24, 24, 2, 20),
    (48000, 44100, 32, 16, 2, 40),
])
def test_wrapper_pcm_exact(oracle, cfg):
    """PCM in -> filter -> fast resampler -> PCM out: codes and clip counts equal to the oracle wrapper with the fused
    resampler, over two chained calls, where the existing check allows one LSB."""
    sr, dr, sb, db, ch, ns = cfg
    frames = 2048
    rng = np.random.default_rng(sr + db)
    raw = pcm_noise(rng, ns, 2 * frames * ch, sb, std=0.4)
    cap = int(frames * dr / sr) + 64
    calls = [(frames, cap), (frames, cap)]
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 256, 256, mode=mode)
        got[mode] = _wrapper_chain(r, raw, ch, (sb + 7) // 8, calls, 1.5)
        r.free()
    probes = sorted({0, 1, 2, 3, ns // 2, ns - 1})
    ref = {s: _oracle_wrapper_chain(oracle, raw[s], ch, (sb + 7) // 8, sr, dr, sb, db, calls, 1.5) for s in probes}
    assert sum(c[3] for chain in ref.values() for c in chain) > 0  # +1.5 dB at 0.4 std: some samples clip
    _assert_wrapper(got[FAST], ref, probes, cfg)
    _assert_wrapper_fast_path(got[FAST], got[EXACT], cfg)


@pytest.mark.parametrize("db,frames", [(8, 1000), (16, 2048), (24, 777), (32, 1500)])
def test_fused_post_filter_quantiser_mono(oracle, monkeypatch, db, frames):
    """Mono 16 -> 48 kHz: the post-filter's threads quantise and pack their own results (espb_biquad_tm_pcm_kernel),
    three chained calls, loud enough to clip."""
    monkeypatch.setenv("ESPB_FUSE_POST_GROUPS", "1")
    monkeypatch.setenv("ESPB_FUSE_POST", "1")
    sr, dr, sb, ch, ns = 16000, 48000, 16, 1, 150
    rng = np.random.default_rng(db + frames)
    raw = pcm_noise(rng, ns, 3 * frames, 16, std=0.45)
    cap = frames * 3 + 64
    calls = [(frames, cap)] * 3
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 64, 64, mode=mode)
        got[mode] = _wrapper_chain(r, raw, ch, 2, calls, 3.0)
        r.free()
    probes = (0, 1, 2, 3, 77, ns - 1)
    ref = {s: _oracle_wrapper_chain(oracle, raw[s], ch, 2, sr, dr, sb, db, calls, 3.0, 64, 64) for s in probes}
    assert sum(c[3] for chain in ref.values() for c in chain) > 0
    _assert_wrapper(got[FAST], ref, probes, db)
    if db >= 16:  # 8-bit codes are too coarse for the last-bit differences to show in 150 x 9000 samples
        _assert_wrapper_fast_path(got[FAST], got[EXACT], db)


def test_c4_like_pre_filter_time_blocks(oracle):
    """96 -> 44.1 kHz, 8 channels, 24-bit, T = 1024, pre-filter in time blocks, two calls: composed from the oracle's
    stages with the fused resampler (the oracle wrapper holds filters for two channels only)."""
    ns, ch, frames, sb = 3, 8, 12000, 24
    rng = np.random.default_rng(4)
    raw = pcm_noise(rng, ns, 2 * frames * ch, sb, std=0.3)
    cap = int(frames * 44100 / 96000) + 64
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, 96000, 44100, sb, sb, ch, True, True, 1024, 256, mode=mode)
        assert r.policy()["filter"] == "pre"
        r.set_biquad_time_blocks(4096, 1024)
        got[mode] = _wrapper_chain(r, raw, ch, 3, [(frames, cap)] * 2, 0.0)
        pol = r.policy()
        r.free()
    for s in range(ns):
        segs = [raw[s, k * frames * ch * 3:(k + 1) * frames * ch * 3] for k in range(2)]
        ref = composed_fused(oracle, pol, ch, sb, sb, 1024, 256, segs, frames, cap, 0.0)
        for k, ((y, u, g, clips), (q, uo, go, co)) in enumerate(zip(got[FAST], ref)):
            assert (u, g) == (uo, go) and bits_equal(y[s], q) and int(clips[s]) == co, (s, k)
    _assert_wrapper_fast_path(got[FAST], got[EXACT], "C4-like")


@pytest.mark.parametrize("cfg", [
    # src_rate, dst_rate, src_bits, dst_bits, channels, streams, frames (test_wrapper_odd_shapes_vs_composed_oracle)
    (44100, 48000, 24, 16, 3, 45, 1001),
    (48000, 32000, 16, 24, 6, 22, 777),
    (22050, 44100, 8, 32, 5, 27, 63),
    (32000, 48000, 16, 16, 2, 3, 130),
])
def test_wrapper_odd_shapes(oracle, cfg):
    """Channel and frame counts that take the generic layout kernels, tails under 64 frames and unaligned PCM rows;
    two calls, against the composed fused pipeline."""
    sr, dr, sb, db, ch, ns, frames = cfg
    nb = (sb + 7) // 8
    rng = np.random.default_rng(frames)
    raw = rng.integers(0, 256, size=(ns, frames * ch * nb), dtype=np.uint8)
    cap = int(frames * dr / sr) + 40
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, sb, db, ch, True, True, 64, 64, mode=mode)
        pol = r.policy()
        got[mode] = [r.resample(raw, frames, cap, -2.5) for _ in range(2)]
        r.free()
    for s in range(0, ns, 4):
        ref = composed_fused(oracle, pol, ch, sb, db, 64, 64, [raw[s]] * 2, frames, cap, -2.5)
        for k, ((out, res), (q, used, gen, clipped)) in enumerate(zip(got[FAST], ref)):
            assert (res["frames_used"], res["frames_generated"]) == (used, gen), (cfg, s, k)
            assert bits_equal(out[s], q), (cfg, s, k)
            assert int(res["clipped_per_stream"][s]) == clipped, (cfg, s, k)
    if ns * frames > 1000:  # (3 streams x 130 frames of 16-bit codes are too few for a last-bit difference to show)
        assert any(not bits_equal(a[0], b[0]) for a, b in zip(got[FAST], got[EXACT])), cfg


def test_wrapper_async_calls(oracle):
    """espb_resampler_resample_async, three calls enqueued without synchronising: bytes, frame counts and the
    device-side clip counts of every call against the fused oracle wrapper."""
    ns, ch, frames, cap = 50, 2, 1500, 1800
    rng = np.random.default_rng(5)
    pcm = (rng.normal(0, 0.5, (ns, 3 * frames * ch)).clip(-1.2, 1.2) * 30000).clip(-32768, 32767).astype(np.int16)
    raw = pcm.view(np.uint8)
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, 44100, 48000, 16, 16, ch, True, True, 64, 64, mode=mode)
        d_in = espb.DeviceBuffer.from_numpy(np.ascontiguousarray(raw))
        d_outs = [espb.DeviceBuffer(ns * cap * ch * 2) for _ in range(3)]
        clips = [np.zeros(ns, np.uint32) for _ in range(3)]
        results = []
        for call in range(3):
            d_outs[call].zero()
            res = r.resample_dev_async(d_in.ptr + call * frames * ch * 2, 3 * frames * ch * 2, d_outs[call].ptr,
                                       cap * ch * 2, frames, cap, 3.0)
            espb.capi._check(espb.lib().espb_memcpy_d2h(clips[call].ctypes.data, r.clipped_dev(), ns * 4, None), "d2h")
            results.append(res)
        espb.capi._check(espb.lib().espb_stream_sync(None), "sync")
        chain = []
        for call, res in enumerate(results):
            g = res["frames_generated"]
            assert res["frames_used"] == frames
            y = d_outs[call].download(np.uint8).reshape(ns, cap * ch * 2)
            assert not y[:, g * ch * 2:].any()
            chain.append((y[:, : g * ch * 2].copy(), res["frames_used"], g, clips[call]))
            d_outs[call].free()
        d_in.free()
        r.free()
        got[mode] = chain
    calls = [(frames, cap)] * 3
    probes = (0, 1, 25, ns - 1)
    ref = {s: _oracle_wrapper_chain(oracle, raw[s], ch, 2, 44100, 48000, 16, 16, calls, 3.0, 64, 64) for s in probes}
    _assert_wrapper(got[FAST], ref, probes, "async")
    assert sum(c[3] for chain in ref.values() for c in chain) > 0
    _assert_wrapper_fast_path(got[FAST], got[EXACT], "async")


@pytest.mark.parametrize("name,ns,ch,sr,dr,bits,frames", [
    ("C3", 16384, 1, 16000, 48000, 16, 16000),       # BASELINE configs[2]
    ("C5 shard", 8192, 2, 48000, 44100, 32, 24000),  # BASELINE configs[4]
])
def test_full_size_wrapper_configs(oracle, name, ns, ch, sr, dr, bits, frames):
    """BASELINE configs[2] and [4] at their stream counts in fast mode (+2 dB: some samples clip): the first, the last
    and seeded sampled streams bit-exact (PCM and clip counts) against the fused oracle wrapper."""
    nb = bits // 8
    rng = np.random.default_rng(ns)
    distinct = 64
    amp = 2 ** (bits - 1) * 0.6
    base = (rng.normal(0, 0.45, (distinct, frames * ch)) * amp).clip(-2 ** (bits - 1), 2 ** (bits - 1) - 1)
    raw = np.tile(pcm_bytes(base.astype(np.int64), nb), (ns // distinct, 1))
    cap = int(frames * dr / sr) + 64
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, bits, bits, ch, True, True, 256, 256, mode=FAST)
    fast, res = r.resample(raw, frames, cap, 2.0)
    r.free()
    got = [(fast, res["frames_used"], res["frames_generated"], np.array(res["clipped_per_stream"]))]
    r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, bits, bits, ch, True, True, 256, 256, mode=EXACT)
    exact, res_e = r.resample(raw, frames, cap, 2.0)
    r.free()
    assert res_e["frames_generated"] == res["frames_generated"]
    assert not np.array_equal(fast, exact), (name, "fast PCM == exact PCM")
    del exact
    sampled = sorted({0, ns - 1} | set(int(s) for s in rng.choice(ns, 6, replace=False)))
    ref = {s: _oracle_wrapper_chain(oracle, raw[s], ch, nb, sr, dr, bits, bits, [(frames, cap)], 2.0) for s in sampled}
    assert sum(c[3] for chain in ref.values() for c in chain) > 0
    _assert_wrapper(got, ref, sampled, name)


# ---------------------------------------------------------------- 7. dyadic input: fast == exact == plain oracle
def _dyadic_batch(n, frames, ch, seed):
    return np.stack([dyadic(frames, ch, stream=seed + s) for s in range(n)])


def _assert_dyadic(oracle, ns, ch, geo, x, calls, ratios, probes, what, adv=None):
    runs = run_modes(ns, ch, geo, x, calls, ratios, adv)
    assert len(runs[FAST][0]) == len(runs[EXACT][0])
    for (yf, uf, gf), (ye, ue, ge) in zip(runs[FAST][0], runs[EXACT][0]):
        assert (uf, gf) == (ue, ge) and bits_equal(yf, ye), what  # fast == exact, all streams
    assert runs[FAST][1] == runs[EXACT][1]
    ref = {s: oracle_chain(oracle, x[s], ch, geo, calls, ratios, fused=False, adv=adv)[0] for s in probes}
    assert_chain(runs[FAST][0], ref, probes, what)  # == the plain oracle
    assert any(np.count_nonzero(y) for y, _, _ in runs[FAST][0]), what


def test_dyadic_standard_kernel(oracle, monkeypatch):
    """Dyadic input (samples 0, -0, +-2^k, k in [-14, 0]) on the default standard kernel and on ESPB_BPP=8,
    ESPB_CHUNK_ROWS=16: fast == exact == plain oracle, bit for bit, with no fused oracle involved."""
    ns, ch = 70, 2
    calls = split3(3000, R48)
    x = _dyadic_batch(ns, 3000, ch, seed=0)
    _assert_dyadic(oracle, ns, ch, (256, 256, 1.0, 3), x, calls, [R48] * 3, probes_of(ns), "default")
    monkeypatch.setenv("ESPB_BPP", "8")
    monkeypatch.setenv("ESPB_CHUNK_ROWS", "16")
    _assert_dyadic(oracle, ns, ch, (1024, 256, 0.45, 3), x, calls, [f32(44100) / f32(96000)] * 3, probes_of(ns),
                   "bpp 8 rows 16")


def test_dyadic_non_interpolating_and_direct(oracle, monkeypatch):
    """Dyadic input on the non-interpolating kernel (flags 2, nearest phase up to F) and on direct input
    (ESPB_DIRECT=1, stereo)."""
    ns, ch = 70, 2
    x = _dyadic_batch(ns, 3000, ch, seed=100)
    ratio = f32(44100) / f32(48000)
    _assert_dyadic(oracle, ns, ch, (128, 37, 1.0, 2), x, split3(3000, ratio), [ratio] * 3, probes_of(ns), "ni")
    monkeypatch.setenv("ESPB_DIRECT", "1")
    calls = [(1000, 2000), (10, 50), (900, 300), (64, 500), (1000, 4000)]
    _assert_dyadic(oracle, ns, ch, (64, 64, 1.0, 3), x, calls, [R48] * len(calls), probes_of(ns), "direct")


@pytest.mark.parametrize("ns,ch", [(1, 2), (4, 8)])  # 2 and 8 series per lane
def test_dyadic_few_series(oracle, ns, ch):
    """Dyadic input on the few-series kernel in its 2- and 8-series-per-lane forms."""
    x = _dyadic_batch(ns, 4000, ch, seed=200)
    _assert_dyadic(oracle, ns, ch, (256, 256, 1.0, 3), x, split3(4000, R48), [R48] * 3, range(ns), (ns, ch))


def test_dyadic_clock_groups(oracle):
    """Dyadic input on the fused clock groups (9 groups x 4 streams x 3 channels), drifting ratios."""
    shape = (9, 4, 3)
    n_groups, spg, ch = shape
    geo = (64, 128, 1.0, 3)
    ns = n_groups * spg
    x = _dyadic_batch(ns, 3000, ch, seed=300)
    calls = _group_calls(n_groups, seed=11)
    fast, st_f = _run_groups(shape, x, calls, FAST, True, geo)
    exact, st_e = _run_groups(shape, x, calls, EXACT, True, geo)
    assert st_f == st_e
    orc = [oracle.resampler(ch, *geo) for _ in range(ns)]
    for o in orc:
        o.advance(geo[0] / 2)
    nonzero = 0
    for c, ((xin, n_in, y, res), (_, _, ye, rese)) in enumerate(zip(fast, exact)):
        assert res == rese and bits_equal(y, ye), c
        n_out, ratios = calls[c][1], calls[c][2]
        for s in range(ns):
            k = s // spg
            yo, uo, go = orc[s].process_interleaved(xin[s, : n_in[k] * ch], n_out[k], ratios[k], n_in=n_in[k])
            assert res[k] == (uo, go) and bits_equal(y[s, : go * ch], yo), (c, s)
            nonzero += int(np.count_nonzero(yo))
    assert nonzero > 0


@pytest.mark.parametrize("use_filter", [True, False])
def test_dyadic_wrapper(oracle, use_filter):
    """The wrapper with its post-filter (16 -> 48 kHz mono) and with no filter (44.1 -> 48 kHz stereo), 16-bit PCM
    codes 0 and +-2^j (j in [1, 14]: samples +-2^(j-15) after the gain of 0 dB): fast == exact == plain oracle wrapper,
    PCM codes and clip counts.  Pre-filter paths cannot be dyadic: the biquad's output is not."""
    sr, dr, ch = (16000, 48000, 1) if use_filter else (44100, 48000, 2)
    ns, frames = 40, 2000
    rng = np.random.default_rng(17 + use_filter)
    n = 2 * frames * ch
    codes = (rng.choice([-1, 0, 1], size=(ns, n), p=[0.45, 0.1, 0.45]) << rng.integers(1, 15, size=(ns, n)))
    raw = pcm_bytes(codes.astype(np.int64), 2)
    cap = int(frames * dr / sr) + 64
    calls = [(frames, cap)] * 2
    got = {}
    for mode in (FAST, EXACT):
        r = espb.Resampler(ns, frames * ch, cap * ch, sr, dr, 16, 16, ch, use_filter, True, 64, 64, mode=mode)
        assert r.policy()["filter"] == ("post" if use_filter else "none")
        got[mode] = _wrapper_chain(r, raw, ch, 2, calls, 0.0)
        r.free()
    for (yf, uf, gf, cf), (ye, ue, ge, ce) in zip(got[FAST], got[EXACT]):
        assert (uf, gf) == (ue, ge) and bits_equal(yf, ye) and np.array_equal(cf, ce)
    for s in (0, 1, ns - 1):
        w = oracle.wrapper(frames * ch, cap * ch, float(sr), float(dr), 16, 16, ch, use_filter, True, 64, 64)
        for k, (y, u, g, clips) in enumerate(got[FAST]):
            yo, ro = w.resample(np.ascontiguousarray(raw[s, k * frames * ch * 2:(k + 1) * frames * ch * 2]), frames,
                                cap, 0.0)
            assert (u, g) == (ro["frames_used"], ro["frames_generated"]), (s, k)
            assert bits_equal(y[s], yo) and int(clips[s]) == ro["clipped_samples"], (s, k)
    assert any(np.count_nonzero(y) for y, *_ in got[FAST])
