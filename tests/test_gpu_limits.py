"""Sizes along the y axis of the launch grid.  CUDA caps gridDim.y at 65,535; the launchers put frames (tiles of 32 or
64), outputs, biquad time blocks, CTAs of passes and clock groups on y, and slice a launch that would exceed the cap
(kernels.hpp: for_each_y_slice).  A wrong slice offset shows as a block of 32 or 64 rows at one place in the output, so
every check here compares whole series: bit-exact against the oracle in exact mode (bytes, frame counts, end state,
clip counts), bit-exact against the oracle's FMA chain (fused=True) in fast mode.

Switch                 read                         covered by
ESPB_GRID_Y_MAX        per process (static)         test_sliced_launches (child process, = 3 and = 1)
ESPB_GROUPS_FUSED      per context                  test_sliced_launches, test_real_size_clock_groups
ESPB_FUSE_POST_GROUPS  per call                     test_sliced_launches (mono wrapper: fused post-filter quantiser)
ESPB_PPC               per call                     test_sliced_launches

Part a runs every sliced launcher at ordinary sizes with the limit lowered to 3 and to 1 in a child process; each
call is long enough that each launcher it reaches is split at least twice.  Part b runs real sizes past the limit
once each; each docstring states the test's peak device memory (time-major staging is 2 x rows x 512 B per 128-series
group)."""
import os
import subprocess
import sys

import numpy as np
import pytest
from conftest import bits_equal
from oracle_lib import noise

import esp_audio_libs_b200 as espb

pytestmark = pytest.mark.gpu
f32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
R48 = f32(48000) / f32(44100)
T, F = 32, 32  # small taps: the limits concern frames, and the CPU oracle stays cheap


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert espb.device_count() > 0, "GPU tests need a GPU: the product has no CPU path"
    espb.set_device(0)


def _set_env(env):
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)


def signal(ns, frames, ch, seed):
    return np.stack([noise(frames, ch, stream=seed + s, amp=0.8) for s in range(ns)])


def pcm(ns, frames, ch, bits, seed, amp=0.5):
    """Little-endian packed PCM rows of `bits` (16 or 24), loud enough that a few samples clip after gain."""
    rng = np.random.default_rng(seed)
    full = 2 ** (bits - 1)
    v = (rng.normal(0, amp, (ns, frames * ch)).clip(-1, 1 - 1 / full) * full).astype(np.int32)
    b = v.astype("<i4").view(np.uint8).reshape(ns, frames * ch, 4)[:, :, : bits // 8]
    return np.ascontiguousarray(b).reshape(ns, frames * ch * (bits // 8))


def oracle_chain(oracle, row, ch, calls, ratio, flags=3, fused=False):
    o = oracle.resampler(ch, T, F, 1.0, flags, fused=fused)
    o.advance(T / 2)
    out, pos = [], 0
    for n_in, cap in calls:
        y, u, g = o.process_interleaved(row[pos * ch:(pos + n_in) * ch], cap, ratio, n_in=n_in)
        out.append((y, u, g))
        pos += u
    return out, o.state()


def check_streams(got, x, ch, calls, ratio, oracle, streams, flags=3, fused=False, what=""):
    """got: [(y (ns, gen*ch), used, gen)] per call, state; every listed stream against its own oracle context."""
    chain, st = got
    for s in streams:
        ref, ost = oracle_chain(oracle, x[s], ch, calls, ratio, flags, fused)
        for k, ((y, u, g), (yo, uo, go)) in enumerate(zip(chain, ref)):
            assert (u, g) == (uo, go), (what, s, k, (u, g), (uo, go))
            assert bits_equal(y[s, : g * ch], yo), (what, s, k)
        assert st == ost, (what, st, ost)


def layout_call(b, x, n_in, cap, ratio, in_fs=None, out_skew=0):
    """One call through espb_resampleProcessLayout: input frames of `in_fs` floats (default: channels, interleaved),
    output rows of cap*ch + out_skew floats starting out_skew floats into the buffer (out_skew = 1: the generic store
    path).  Returns (y (ns, gen*ch), used, gen)."""
    L = espb.lib()
    ns, ch = b.num_streams, b.channels
    fs = in_fs or ch
    xin = np.zeros((ns, max(n_in, 1) * fs), f32)
    for c in range(ch):
        xin[:, c::fs][:, :n_in] = x[:, c::ch][:, :n_in]
    il = espb.capi._Layout(xin.shape[1], 1, fs)
    ol = espb.capi._Layout(cap * ch + out_skew, 1, ch)
    d_in = espb.DeviceBuffer.from_numpy(xin)
    d_out = espb.DeviceBuffer((ns * ol.stream_stride + out_skew) * 4)
    d_out.zero()
    r = L.espb_resampleProcessLayout(b.h, d_in.ptr, il, n_in, d_out.ptr + 4 * out_skew, ol, cap, ratio, None)
    if r.input_used == 0 and r.output_generated == 0 and espb.capi._err():
        raise espb.EspbError(espb.capi._err())
    used, gen = int(r.input_used), int(r.output_generated)
    y = d_out.download(f32)[out_skew: out_skew + ns * ol.stream_stride].reshape(ns, -1)[:, : gen * ch].copy()
    d_in.free()
    d_out.free()
    return y, used, gen


def chain_calls(b, x, calls, ratio, call):
    ch, out, pos = b.channels, [], 0
    for n_in, cap in calls:
        y, u, g = call(b, np.ascontiguousarray(x[:, pos * ch:(pos + n_in) * ch]), n_in, cap, ratio)
        out.append((y, u, g))
        pos += u
    return out, b.state()


def _interleaved(b, seg, n_in, cap, ratio):
    return b.process_interleaved(seg, cap, ratio, n_in=n_in)


def _planar(b, seg, n_in, cap, ratio):
    ns, ch = b.num_streams, b.channels
    y, u, g = b.process_planar(seg.reshape(ns, n_in, ch).transpose(0, 2, 1), cap, ratio)
    return np.ascontiguousarray(y.transpose(0, 2, 1)).reshape(ns, -1), u, g


def _planes(b, seg, n_in, cap, ratio):
    ns, ch = b.num_streams, b.channels
    planes = [np.ascontiguousarray(seg[s, c::ch]) for s in range(ns) for c in range(ch)]
    ys, u, g = b.process_planes(planes, cap, ratio)
    return np.stack([np.stack(ys[s * ch:(s + 1) * ch], 1).reshape(-1) for s in range(ns)]), u, g


def _host(b, seg, n_in, cap, ratio):
    ns, ch = b.num_streams, b.channels
    hin = espb.PinnedBuffer(ns * n_in * ch, f32)
    hin.array[:] = seg.reshape(-1)
    hout = espb.PinnedBuffer(ns * cap * ch, f32)
    hout.array[:] = 0
    u, g = b.process_interleaved_host(hin.ptr, n_in * ch, n_in, hout.ptr, cap * ch, cap, ratio)
    y = hout.array.reshape(ns, cap * ch)[:, : g * ch].copy()
    hin.free()
    hout.free()
    return y, u, g


def _general_stride(b, seg, n_in, cap, ratio):
    return layout_call(b, seg, n_in, cap, ratio, in_fs=b.channels + 1, out_skew=1)


# ---------------------------------------------------------------- a. slicing at ordinary sizes
# 20,000 frames at 48/44.1: 313 fast tiles, 626 generic tiles, ~680 passes — every launcher splits many times at 3
CALLS = [(20000, 21900), (1500, 1700)]
# (name, channels, streams, flags, call form, batch env, options, modes)
RESAMPLE_CASES = [
    ("ch1", 1, 40, 3, _interleaved, {}, {}, "ef"),
    ("ch2", 2, 20, 3, _interleaved, {}, {}, "ef"),
    ("ch3", 3, 14, 3, _interleaved, {}, {}, "e"),
    ("ch4", 4, 10, 3, _interleaved, {}, {}, "e"),
    ("ch6", 6, 7, 3, _interleaved, {}, {}, "e"),
    ("ch8", 8, 5, 3, _interleaved, {}, {}, "e"),
    ("few", 2, 3, 3, _interleaved, {}, {}, "ef"),              # 6 series: the few-series kernel
    ("planar", 2, 20, 3, _planar, {}, {}, "e"),
    ("stride", 2, 20, 3, _general_stride, {}, {}, "e"),
    ("serial", 2, 20, 3, _interleaved, {}, {espb.OPT_OVERLAP_STAGING: 0}, "e"),
    ("timing", 2, 20, 3, _interleaved, {}, {espb.OPT_KERNEL_TIMING: 1}, "e"),
    ("planes", 1, 40, 3, _planes, {}, {}, "e"),
    ("host", 2, 20, 3, _host, {}, {}, "e"),
    ("flags0", 2, 20, 0, _interleaved, {}, {}, "e"),          # the non-interpolating kernel
    ("ppc1", 2, 20, 3, _interleaved, {"ESPB_PPC": "1"}, {}, "e"),
]
# wrapper: (name, streams, channels, src rate, dst rate, bits, filter position, env)
WRAP_FRAMES = 20000
WRAP_CASES = [("w16post", 6, 2, 44100, 48000, 16, "post", {}),
              ("w24post", 6, 2, 44100, 48000, 24, "post", {}),
              ("w16pre", 6, 2, 48000, 44100, 16, "pre", {}),
              ("w16fuse", 40, 1, 44100, 48000, 16, "post", {"ESPB_FUSE_POST_GROUPS": "1"})]
BQ_CASES = [(1, 4000), (40, 4000)]  # (series, samples): blocks of 32 rows, the few-series and the 128-thread form
GROUPS7 = (7, 1500)                 # 7 mono clock groups (fused), frames per call
ROWS10 = (10, 3001)                 # rows, samples per row


def _mode_list(m):
    return [md for c, md in (("e", espb.MODE_EXACT), ("f", espb.MODE_FAST)) if c in m]


def _wrapper_inputs(ns, ch, bits, seed):
    return pcm(ns, WRAP_FRAMES + 600, ch, bits, seed)


def _group_inputs():
    n, frames = GROUPS7
    rng = np.random.default_rng(77)
    ratios = [f32(R48 * f32(1.0 + 1e-3 * rng.standard_normal())) for _ in range(n)]
    return signal(n, frames, 1, seed=7700), ratios


def run_sliced_cases():
    """Every case of part a with the current process's limit; returns {key: array}."""
    saved = {}
    for name, ch, ns, flags, form, env, opts, modes in RESAMPLE_CASES:
        x = signal(ns, sum(c[0] for c in CALLS), ch, seed=sum(map(ord, name)))
        for mode in _mode_list(modes):
            _set_env(env)
            b = espb.ResampleBatch(ns, ch, T, F, 1.0, flags, mode=mode)
            _set_env({k: None for k in env if k != "ESPB_PPC"})
            for o, v in opts.items():
                b.set_option(o, v)
            b.advance(T / 2)
            chain, st = chain_calls(b, x, CALLS, R48, form)
            _set_env({k: None for k in env})
            b.free()
            for k, (y, u, g) in enumerate(chain):
                saved[f"{name}_{mode}_{k}_y"] = y
                saved[f"{name}_{mode}_{k}_n"] = np.array([u, g], np.int64)
            saved[f"{name}_{mode}_st"] = np.array([st[0]], f32)
            saved[f"{name}_{mode}_idx"] = np.array([st[1]], np.int64)
    for name, ns, ch, sr, dr, bits, where, env in WRAP_CASES:
        raw = _wrapper_inputs(ns, ch, bits, seed=len(name) * 31 + bits)
        _set_env(env)
        r = espb.Resampler(ns, (WRAP_FRAMES + 600) * ch, (WRAP_FRAMES + 2000) * ch, sr, dr, bits, bits, ch, True, True,
                           T, F, mode=espb.MODE_EXACT)
        assert r.policy()["filter"] == where, name
        y, res = r.resample(raw, WRAP_FRAMES, WRAP_FRAMES + 2000, 3.0)
        _set_env({k: None for k in env})
        r.free()
        saved[f"{name}_y"] = y
        saved[f"{name}_res"] = np.concatenate([[res["frames_used"], res["frames_generated"]],
                                               res["clipped_per_stream"]]).astype(np.int64)
    for nser, n in BQ_CASES:
        x = signal(nser, n, 1, seed=8800 + nser)
        bq = espb.BiquadBatch(nser, 2, espb.biquad_lowpass(0.2274))
        bq.set_time_blocks(32, 32)
        saved[f"bq{nser}_y"] = bq.apply_interleaved(x, 1)
        saved[f"bq{nser}_st"] = bq.state()
        bq.free()
    x, ratios = _group_inputs()
    n, frames = GROUPS7
    _set_env({"ESPB_GROUPS_FUSED": "1"})
    g = espb.ResampleGroups([1] * n, 1, T, F, 1.0, 3, mode=espb.MODE_EXACT)
    _set_env({"ESPB_GROUPS_FUSED": None})
    assert g.is_fused()
    for k in range(n):
        g.advance(k, T / 2)
    y, res = g.process_interleaved(x, [frames] * n, [frames + 200] * n, ratios)
    saved["groups_y"] = y
    saved["groups_n"] = np.array(res, np.int64)
    saved["groups_st"] = np.array([g.state(k)[0] for k in range(n)], f32)
    g.free()
    rows, n = ROWS10
    q, clipped, back = rows_roundtrip(rows, n)
    saved["rows_q"], saved["rows_clipped"], saved["rows_f"] = q, clipped, back
    return saved


def rows_inputs(rows, n):
    rng = np.random.default_rng(1010)
    return (rng.standard_normal((rows, n)) * 0.8).astype(f32)  # loud: some samples clip


def rows_roundtrip(rows, n, bits=24):
    """espb_float_to_quantized_rows then espb_quantized_to_float_rows over `rows` padded rows."""
    L = espb.lib()
    nb = bits // 8
    x = rows_inputs(rows, n)
    in_row, q_row, f_row = n + 3, n * nb + 5, n + 7
    xin = np.zeros((rows, in_row), f32)
    xin[:, :n] = x
    d_x = espb.DeviceBuffer.from_numpy(xin)
    d_q = espb.DeviceBuffer(rows * q_row)
    d_q.zero()
    d_c = espb.DeviceBuffer(rows * 4)
    d_c.zero()
    assert L.espb_float_to_quantized_rows(d_x.ptr, in_row, d_q.ptr, q_row, rows, n, bits, d_c.ptr, None) == 0
    d_f = espb.DeviceBuffer(rows * f_row * 4)
    d_f.zero()
    assert L.espb_quantized_to_float_rows(d_q.ptr, q_row, d_f.ptr, f_row, rows, n, bits, -1.5, None) == 0
    q = d_q.download(np.uint8).reshape(rows, q_row)[:, : n * nb].copy()
    clipped = d_c.download(np.uint32, rows).astype(np.int64)
    back = d_f.download(f32).reshape(rows, f_row)[:, :n].copy()
    for d in (d_x, d_q, d_c, d_f):
        d.free()
    return q, clipped, back


def _child_sliced(out_dir):
    espb.set_device(0)
    np.savez(os.path.join(out_dir, "sliced.npz"), **run_sliced_cases())


@pytest.fixture(scope="module")
def default_limit_run():
    assert "ESPB_GRID_Y_MAX" not in os.environ
    return run_sliced_cases()


def check_sliced_against_oracle(m, oracle):
    for name, ch, ns, flags, form, env, opts, modes in RESAMPLE_CASES:
        x = signal(ns, sum(c[0] for c in CALLS), ch, seed=sum(map(ord, name)))
        for mode in _mode_list(modes):
            chain = [(m[f"{name}_{mode}_{k}_y"], *[int(v) for v in m[f"{name}_{mode}_{k}_n"]]) for k in range(len(CALLS))]
            st = (f32(m[f"{name}_{mode}_st"][0]), int(m[f"{name}_{mode}_idx"][0]))
            check_streams((chain, st), x, ch, CALLS, R48, oracle, range(ns), flags, fused=mode == espb.MODE_FAST,
                          what=(name, mode))
    for name, ns, ch, sr, dr, bits, where, env in WRAP_CASES:
        raw = _wrapper_inputs(ns, ch, bits, seed=len(name) * 31 + bits)
        res = m[f"{name}_res"]
        assert res[2:].sum() > 0, name  # the gain makes some samples clip
        for s in range(ns):
            w = oracle.wrapper((WRAP_FRAMES + 600) * ch, (WRAP_FRAMES + 2000) * ch, float(sr), float(dr), bits, bits, ch,
                               True, True, T, F)
            yo, ro = w.resample(raw[s], WRAP_FRAMES, WRAP_FRAMES + 2000, 3.0)
            assert (int(res[0]), int(res[1])) == (ro["frames_used"], ro["frames_generated"]), (name, s)
            assert int(res[2 + s]) == ro["clipped_samples"], (name, s)
            assert bits_equal(m[f"{name}_y"][s][: yo.size], yo), (name, s)
    for nser, n in BQ_CASES:
        x = signal(nser, n, 1, seed=8800 + nser)
        coeffs = espb.biquad_lowpass(0.2274)
        for s in range(nser):
            ref = np.ascontiguousarray(x[s])
            for k in range(2):
                o = oracle.biquad(coeffs)
                o.apply_buffer(ref)
                assert bits_equal(m[f"bq{nser}_st"][s, k], np.frombuffer(o.buf, f32)[5:9]), (nser, s, k)
            assert bits_equal(m[f"bq{nser}_y"][s], ref), (nser, s)
    x, ratios = _group_inputs()
    n, frames = GROUPS7
    for k in range(n):
        (yo, uo, go), = oracle_chain(oracle, x[k], 1, [(frames, frames + 200)], ratios[k])[0]
        assert tuple(m["groups_n"][k]) == (uo, go) and bits_equal(m["groups_y"][k][:go], yo), k
        assert bits_equal(m["groups_st"][k:k + 1], np.array([oracle_chain(oracle, x[k], 1, [(frames, frames + 200)],
                                                                          ratios[k])[1][0]], f32)), k
    rows, n = ROWS10
    x = rows_inputs(rows, n)
    for r in range(rows):
        q, clipped = oracle.float_to_quantized(x[r], 24)
        assert bits_equal(m["rows_q"][r], q) and int(m["rows_clipped"][r]) == clipped, r
        assert bits_equal(m["rows_f"][r], oracle.quantized_to_float(q, n, 24, -1.5)), r


@pytest.mark.parametrize("limit", ["3", "1"])
def test_sliced_launches(oracle, tmp_path, default_limit_run, limit):
    """ESPB_GRID_Y_MAX = 3 and 1 (read once per process, in a child): every sliced launcher at ordinary sizes, each
    split at least twice — float interleaved 1/2/3/4/6/8 channels, planar, a general stride (frames of channels + 1
    floats, unaligned output rows), few-series and standard kernels, staging overlap on and off, kernel timing on,
    pointer tables, the host-buffer path, the non-interpolating kernel, ESPB_PPC=1, the wrapper (int16
    and int24, pre- and post-filter, the fused mono post-filter quantiser), the stand-alone biquad in 32-row time
    blocks, a fused set of 7 clock groups and the *_rows quantisers over 10 rows.  The bytes must equal the default
    limit's run in this process, and the oracle (fast mode: its FMA chain) on every series."""
    p = subprocess.run([sys.executable, "-c", f"import sys; sys.path[:0] = [{HERE!r}, {ROOT!r}]; "
                        f"import test_gpu_limits as t; t._child_sliced({str(tmp_path)!r})"],
                       env=dict(os.environ, ESPB_GRID_Y_MAX=limit), capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, p.stderr[-4000:]
    m = np.load(tmp_path / "sliced.npz")
    assert sorted(m.files) == sorted(default_limit_run)
    for k in m.files:
        assert bits_equal(m[k], default_limit_run[k]), k
    check_sliced_against_oracle(m, oracle)


# ---------------------------------------------------------------- b. real sizes past the limit
def test_real_size_generic_transpose_few_series(oracle):
    """One 6-channel interleaved stream, n_in = 2,100,000 at 48/44.1 (65,626 generic 32-row tiles on y; the few-series
    kernel), exact and fast.  Peak device memory about 0.2 GB (input 50 MB, output 55 MB, staging 2 x 2.1 M x 512 B of
    one group when the standard kernel's buffers are sized)."""
    ch, n = 6, 2_100_000
    calls = [(n, int(n * float(R48)) + 64)]
    x = signal(1, n, ch, seed=2100)
    for mode in (espb.MODE_EXACT, espb.MODE_FAST):
        b = espb.ResampleBatch(1, ch, T, F, 1.0, 3, mode=mode)
        b.advance(T / 2)
        got = chain_calls(b, x, calls, R48, _interleaved)
        b.free()
        check_streams(got, x, ch, calls, R48, oracle, [0], fused=mode == espb.MODE_FAST, what=("b1", mode))


def test_real_size_fast_transpose_standard_kernel(oracle):
    """17 stereo streams (34 series: the standard kernel), n_in = 4,200,000 (65,625 fast 64-row tiles on y), with
    default options and with kernel timing on (the non-overlapped staging): identical bytes; 3 streams against the
    oracle; calls of 1,000,000 frames over the same input give the same bytes.  Peak device memory about 4.9 GB
    (staging 2 x 4.2 M x 512 B = 4.3 GB, input 0.57 GB, output 0.62 GB)."""
    ns, ch, n = 17, 2, 4_200_000
    cap = int(n * float(R48)) + 64
    x = signal(ns, n, ch, seed=4200)
    runs = {}
    for label in ("default", "timing"):
        b = espb.ResampleBatch(ns, ch, T, F, 1.0, 3, mode=espb.MODE_EXACT)
        if label == "timing":
            b.set_option(espb.OPT_KERNEL_TIMING, 1)
        b.advance(T / 2)
        runs[label] = chain_calls(b, x, [(n, cap)], R48, _interleaved)
        b.free()
    (y, u, g), = runs["default"][0]
    (yt, ut, gt), = runs["timing"][0]
    assert (u, g) == (ut, gt) and bits_equal(y, yt) and runs["default"][1] == runs["timing"][1]
    check_streams(runs["default"], x, ch, [(n, cap)], R48, oracle, [0, 8, ns - 1], what="b2")
    # the same input in calls of 1,000,000 frames: the concatenated output is the same
    b = espb.ResampleBatch(ns, ch, T, F, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(T / 2)
    pieces, pos = [], 0
    while pos < n:
        m = min(1_000_000, n - pos)
        yy, uu, gg = b.process_interleaved(np.ascontiguousarray(x[:, pos * ch:(pos + m) * ch]),
                                           int(m * float(R48)) + 64, R48, n_in=m)
        assert uu == m
        pieces.append(yy)
        pos += uu
    st = b.state()
    b.free()
    yc = np.concatenate(pieces, axis=1)
    assert yc.shape[1] == g * ch and bits_equal(yc, y) and st == runs["default"][1]


def test_real_size_pointer_tables(oracle):
    """Pointer tables, 2 mono planes, n_in = 2,000,000 at 48/44.1 (2,176,870 outputs: launch_untranspose_ptrs splits
    at 65,535 x 32 rows).  Peak device memory about 2.3 GB (staging 2 x 2 M x 512 B, time-major output 2.2 M x 512 B,
    the planes 34 MB)."""
    ns, n = 2, 2_000_000
    cap = int(n * float(R48)) + 64
    x = signal(ns, n, 1, seed=2000)
    b = espb.ResampleBatch(ns, 1, T, F, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(T / 2)
    got = chain_calls(b, x, [(n, cap)], R48, _planes)
    b.free()
    assert got[0][0][2] > 65535 * 32
    check_streams(got, x, 1, [(n, cap)], R48, oracle, range(ns), what="b3")


def test_real_size_wrapper(oracle):
    """Wrapper: one stereo int16 stream 44.1 -> 48 kHz with the post-filter, 4,200,000 frames: pcm_to_tm and tm_to_pcm
    (65,625 64-frame tiles), the post-filter's time blocks and the untranspose.  Bytes, counts and clip counts against
    the oracle.  Peak device memory about 7 GB (staging 4.3 GB, time-major output and its filtered copy 2 x 2.3 GB,
    the PCM buffers 35 MB)."""
    ch, n = 2, 4_200_000
    out_cap = int(n * 48000 / 44100) + 64
    raw = pcm(1, n, ch, 16, seed=4242, amp=0.6)
    r = espb.Resampler(1, n * ch, out_cap * ch, 44100, 48000, 16, 16, ch, True, True, T, F, mode=espb.MODE_EXACT)
    assert r.policy()["filter"] == "post"
    y, res = r.resample(raw, n, out_cap, 3.0)
    r.free()
    w = oracle.wrapper(n * ch, out_cap * ch, 44100.0, 48000.0, 16, 16, ch, True, True, T, F)
    yo, ro = w.resample(raw[0], n, out_cap, 3.0)
    assert (res["frames_used"], res["frames_generated"]) == (ro["frames_used"], ro["frames_generated"])
    assert ro["frames_generated"] > 65535 * 64
    assert int(res["clipped_per_stream"][0]) == ro["clipped_samples"] > 0
    assert bits_equal(y[0][: yo.size], yo)


def test_real_size_standalone_biquad(oracle):
    """Stand-alone biquad: one mono series of 4,200,000 samples in automatic time-block mode (the transposes to and
    from the time-major route split at 65,535 tiles).  Output and saved state bit-exact against the oracle.  Peak
    device memory about 4.4 GB (two time-major copies of 4.2 M x 512 B and the 17 MB buffer)."""
    n = 4_200_000
    x = signal(1, n, 1, seed=4300)
    coeffs = espb.biquad_lowpass(0.2274)
    bq = espb.BiquadBatch(1, 2, coeffs)
    y = bq.apply_interleaved(x, 1)
    st = bq.state()
    bq.free()
    ref = np.ascontiguousarray(x[0])
    for k in range(2):
        o = oracle.biquad(coeffs)
        o.apply_buffer(ref)
        assert bits_equal(st[0, k], np.frombuffer(o.buf, f32)[5:9]), k
    assert bits_equal(y[0], ref)


def test_real_size_clock_groups(oracle):
    """Fused clock groups: 65,600 groups of one mono stream, two calls of about 256 frames, a seeded ratio per group
    (groups on y of the staging, schedule and resampler launches).  Group k + 65,536 gets the input and ratios of group
    k, so its bytes must be identical; the oracle runs on groups 0, 65,534, 65,535, 65,536, 65,599 and 250 seeded
    others; every group's state equals espb.plan_schedule's on the host.  Peak device memory about 0.3 GB (input and
    output 2 x 65,600 x 300 x 4 B, staging and schedule tables)."""
    n_groups, base = 65_600, 65_536
    calls = [(256, 300), (250, 300)]
    rng = np.random.default_rng(656)
    ratios_base = [(R48 * (1.0 + 2e-3 * rng.standard_normal((base,)))).astype(f32) for _ in calls]
    ratios = [np.concatenate([r, r[: n_groups - base]]) for r in ratios_base]
    x0 = (rng.standard_normal((base, sum(c[0] for c in calls))) * 0.5).astype(f32)
    x = np.concatenate([x0, x0[: n_groups - base]])
    os.environ["ESPB_GROUPS_FUSED"] = "1"
    try:
        g = espb.ResampleGroups([1] * n_groups, 1, T, F, 1.0, 3, mode=espb.MODE_EXACT)
    finally:
        os.environ.pop("ESPB_GROUPS_FUSED")
    assert g.is_fused()
    for k in range(n_groups):
        g.advance(k, T / 2)
    outs, pos = [], np.zeros(n_groups, np.int64)
    for c, (n_in, cap) in enumerate(calls):
        xin = np.stack([x[k, pos[k]: pos[k] + n_in] for k in range(n_groups)]) if c else x[:, :n_in]
        y, res = g.process_interleaved(np.ascontiguousarray(xin), [n_in] * n_groups, [cap] * n_groups, ratios[c])
        res = np.array(res, np.int64)
        outs.append((y, res))
        pos += res[:, 0]
    states = [g.state(k) for k in range(n_groups)]
    g.free()
    for y, res in outs:
        assert bits_equal(y[base:], y[: n_groups - base]) and np.array_equal(res[base:], res[: n_groups - base])
    probes = sorted({0, 65_534, 65_535, 65_536, 65_599} | set(int(v) for v in rng.choice(n_groups, 250, replace=False)))
    for k in probes:
        o = oracle.resampler(1, T, F, 1.0, 3)
        o.advance(T / 2)
        p = 0
        for c, (n_in, cap) in enumerate(calls):
            yo, uo, go = o.process_interleaved(x[k, p: p + n_in], cap, ratios[c][k], n_in=n_in)
            y, res = outs[c]
            assert tuple(res[k]) == (uo, go) and bits_equal(y[k, :go], yo), (k, c)
            p += uo
        assert states[k] == o.state(), k
    for k in range(n_groups):
        off, idx = f32(f32(T // 2) + f32(T / 2)), T
        p = 0
        for c, (n_in, cap) in enumerate(calls):
            s = espb.plan_schedule(T, F, 3, off, idx, n_in, cap, ratios[c][k], want_entries=False)
            off, idx = s["end_offset"], s["end_index"]
        assert states[k] == (f32(off), int(idx)), k
