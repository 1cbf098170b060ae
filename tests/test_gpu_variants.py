"""The kernel instantiations and host paths the default configuration never reaches, held to the same bar as the
default: bit-exact against the oracle in exact mode (frame counts, state, bytes, clip counts), <= 1e-6 max-abs in fast
mode, and byte-identical to the default path in both modes wherever the two must agree.

Switch                 read                         covered by
ESPB_BPP               per context (resampleInit)   test_geometry_matrix, test_chunk_table_limit_per_geometry
ESPB_CHUNK_ROWS        per context (resampleInit)   test_geometry_matrix, test_chunk_table_limit_per_geometry
ESPB_G_MBYTES          per context (resampleInit)   test_g_time_slabs*
ESPB_DIRECT            per context (resampleInit)   test_g_time_slabs_paths
ESPB_NI                per context (resampleInit)   test_g_time_slabs_paths (on, its default)
ESPB_SCHED             per context (resampleInit)   test_sequential_schedule*
ESPB_FS_SLICE_KB       per context (resampleInit)   test_few_series_kernel_switch
ESPB_STAGE_CTAS        per context (resampleInit)   test_staging_grid_size
ESPB_OVERLAP           per context (resampleInit)   test_staging_grid_size, test_g_time_slabs
ESPB_BIQUAD_ONEPASS    per context (biquad_init)    test_standalone_biquad
ESPB_PPC               per call                     test_passes_per_cta, test_chunk_table_limit_per_geometry
ESPB_HOST_SLABS        per call                     test_host_pipeline_slabs
ESPB_FS_STAGES         per process (static)         test_few_series_ring_depth (child process)
ESPB_PCM_CTAS          per process (static)         test_grid_stride_loops (child process)
ESPB_Q15_CTAS          per process (static)         test_grid_stride_loops (child process)
ESPB_EXPAND_CTAS       per process (static)         test_grid_stride_loops (child process)
ESPB_DEBUG             per process                  test_geometry_matrix (names every instantiation it launches)

Switches that are cached in a static, and the instantiation report of ESPB_DEBUG (printed once per process), are
exercised in a child process that writes its results under tmp_path; the parent compares them with the oracle."""
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest
from conftest import bits_equal
from oracle_lib import noise

import esp_audio_libs_b200 as espb

pytestmark = pytest.mark.gpu
f32 = np.float32
TOL = 1e-6  # BASELINE.json north_star: max-abs 1e-6 full scale (fast mode)
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
MODES = (espb.MODE_EXACT, espb.MODE_FAST)
R48 = f32(48000) / f32(44100)
# (ESPB_BPP, ESPB_CHUNK_ROWS) -> pipeline stages of that instantiation (resample_kernel.cu:launch_resample)
GEOMETRIES = {(4, 32): 2, (8, 32): 3, (4, 16): 4, (8, 16): 6, (4, 24): 3, (4, 36): 2}
TABLE = {(4, 32): 320, (8, 32): 768, (4, 16): 320, (8, 16): 768, (4, 24): 120, (4, 36): 120}  # max_chunks_per_cta
# three chained calls: long (> 4096 frames: the staging-overlap path), capacity-limited, uneven
CALLS = [(4500, 5000), (900, 300), (1202, 1400)]


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert espb.device_count() > 0, "GPU tests need a GPU: the product has no CPU path"
    espb.set_device(0)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _set_env(env):
    for k, v in env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)


def run_child(tmp_path, func, env, timeout=900):
    """Run `func(out_dir)` of this module in a fresh interpreter with `env` added; returns its stderr."""
    code = (f"import sys; sys.path[:0] = [{HERE!r}, {ROOT!r}]; import test_gpu_variants as t; "
            f"t.{func}({str(tmp_path)!r})")
    p = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=timeout)
    assert p.returncode == 0, p.stderr[-4000:]
    return p.stderr


def signal(ns, frames, ch, seed):
    return np.stack([noise(frames, ch, stream=seed + s, amp=0.8) for s in range(ns)])


def oracle_chain(oracle, row, ch, taps, filters, lp, flags, calls, ratios):
    """One reference context fed `calls` [(n_in, cap)] from `row`, the input of each call starting at the first frame
    the previous call did not use.  Returns ([(y, used, generated)], final state)."""
    o = oracle.resampler(ch, taps, filters, lp, flags)
    o.advance(taps / 2)
    out, pos = [], 0
    for (n_in, cap), ratio in zip(calls, ratios):
        y, u, g = o.process_interleaved(row[pos * ch:(pos + n_in) * ch], cap, ratio, n_in=n_in)
        out.append((y, u, g))
        pos += u
    return out, o.state()


def process_layout(b, seg, n_in, cap, ratio, form):
    """One device call with interleaved input and the output layout `form`; returns (y interleaved, used, gen).
    stereo / frame4: interleaved rows of a multiple of 4 floats (kOutVecStereo / kOutVecFrame4); planar: channel planes
    of a multiple of 4 floats (kOutVecPlanar); scalar: rows of cap*ch + 1 floats, buffer offset by 4 bytes."""
    L = espb.lib()
    ns, ch = b.num_streams, b.channels
    skew = 0
    if form == "planar":
        cs = (cap + 3) & ~3
        ol = espb.capi._Layout(ch * cs, cs, 1)
    elif form == "scalar":
        ol, skew = espb.capi._Layout(cap * ch + 1, 1, ch), 1
    else:
        ol = espb.capi._Layout(((cap * ch) + 3) & ~3, 1, ch)
    il = espb.capi._Layout(max(n_in * ch, 1), 1, ch)
    d_in = espb.DeviceBuffer.from_numpy(seg if seg.size else np.zeros(ns, f32))
    d_out = espb.DeviceBuffer((ns * ol.stream_stride + skew) * 4)
    d_out.zero()
    r = L.espb_resampleProcessLayout(b.h, d_in.ptr, il, n_in, d_out.ptr + 4 * skew, ol, cap, ratio, None)
    if r.input_used == 0 and r.output_generated == 0 and espb.capi._err():
        raise espb.EspbError(espb.capi._err())
    used, gen = int(r.input_used), int(r.output_generated)
    raw = d_out.download(f32)[skew: skew + ns * ol.stream_stride].reshape(ns, ol.stream_stride)
    if form == "planar":
        y = raw[:, : ch * ol.channel_stride].reshape(ns, ch, ol.channel_stride)[:, :, :gen]
        y = np.ascontiguousarray(y.transpose(0, 2, 1)).reshape(ns, gen * ch)
    else:
        y = raw[:, : gen * ch].copy()
        assert not raw[:, gen * ch: cap * ch].any()  # nothing written past the generated frames
    d_in.free()
    d_out.free()
    return y, used, gen


def device_chain(b, x, calls, ratios, form="stereo"):
    ch = b.channels
    out, pos = [], 0
    for (n_in, cap), ratio in zip(calls, ratios):
        seg = np.ascontiguousarray(x[:, pos * ch:(pos + n_in) * ch])
        y, u, g = process_layout(b, seg, n_in, cap, ratio, form)
        out.append((y, u, g))
        pos += u
    return out


def check_against_oracle(got, ref, probes, mode, what):
    """got: device chain (all streams); ref: {stream: oracle chain}."""
    for s in probes:
        for k, ((y, u, g), (yo, uo, go)) in enumerate(zip(got, ref[s])):
            assert (u, g) == (uo, go), (what, s, k)
            if mode == espb.MODE_EXACT:
                assert bits_equal(y[s], yo), (what, s, k)
            elif go:
                err = float(np.max(np.abs(y[s].astype(np.float64) - yo)))
                assert err <= TOL, (what, s, k, err)


def same_chain(a, b, what):
    assert len(a) == len(b)
    for k, ((ya, ua, ga), (yb, ub, gb)) in enumerate(zip(a, b)):
        assert (ua, ga) == (ub, gb) and bits_equal(ya, yb), (what, k)


def pcm16(ns, frames, ch, seed, amp=0.45):
    rng = np.random.default_rng(seed)
    return (rng.normal(0, amp, (ns, frames * ch)).clip(-1, 0.99997) * 32768).astype(np.int16).view(np.uint8)


def wrapper_chain(r, raw, ch, calls, host_path=False, gain_db=0.0):
    """Chained wrapper calls; the input of a call starts at the first frame the previous one did not use."""
    out, pos = [], 0
    for n_in, cap in calls:
        seg = np.ascontiguousarray(raw[:, pos * ch * 2:(pos + n_in) * ch * 2])
        y, res = r.resample(seg, n_in, cap, gain_db, host_path=host_path)
        out.append((y, res["frames_used"], res["frames_generated"], np.array(res["clipped_per_stream"]).copy()))
        pos += res["frames_used"]
    return out


def oracle_wrapper_chain(oracle, raw_row, ch, sr, dr, calls, taps=256, filters=256, gain_db=0.0):
    w = oracle.wrapper(max(c[0] for c in calls) * ch, max(c[1] for c in calls) * ch, float(sr), float(dr), 16, 16, ch,
                       True, True, taps, filters)
    out, pos = [], 0
    for n_in, cap in calls:
        y, ro = w.resample(np.ascontiguousarray(raw_row[pos * ch * 2:(pos + n_in) * ch * 2]), n_in, cap, gain_db)
        out.append((y, ro["frames_used"], ro["frames_generated"], ro["clipped_samples"]))
        pos += ro["frames_used"]
    return out


def same_wrapper_chain(a, b, what):
    for k, (ra, rb) in enumerate(zip(a, b)):
        assert ra[1:3] == rb[1:3] and bits_equal(ra[0], rb[0]) and np.array_equal(ra[3], rb[3]), (what, k)


def _le16(b):
    return np.ascontiguousarray(b).view(np.int16).astype(np.int64)


# ---------------------------------------------------------------- 1. resampler geometry matrix
# (ch, streams, taps, flags, forms): 140 series = one full 128-series group and a partial one
MATRIX = [(2, 70, 256, 3, ("stereo", "planar", "scalar")), (4, 35, 256, 3, ("frame4",)),
          (2, 70, 256, 0, ("stereo",)), (2, 70, 1024, 3, ("stereo",))]
WRAP_SR, WRAP_DR, WRAP_CALLS = 44100, 48000, [(4500, 4950), (900, 300), (1202, 1400)]  # post-filter: TMCAP output


def _matrix_cases():
    for bpp, rows in GEOMETRIES:
        for ch, ns, taps, flags, forms in MATRIX:
            if taps == 1024 and (bpp, rows) not in ((4, 32), (4, 24), (4, 36)):
                continue  # T=1024: the most rows per pass against the 120-entry table of the 24- and 36-row variants
            for form in forms:
                yield bpp, rows, ch, ns, taps, flags, form


def _probes(ns, ch):
    return sorted({0, 64 // ch - 1, 128 // ch, ns - 1})


def _child_geometry_matrix(out_dir):
    """Every geometry x mode x output form (and the wrapper's time-major output); saves digests + probe rows."""
    espb.set_device(0)
    saved = {}
    for bpp, rows, ch, ns, taps, flags, form in _matrix_cases():
        _set_env({"ESPB_BPP": bpp, "ESPB_CHUNK_ROWS": rows})
        x = signal(ns, sum(c[0] for c in CALLS), ch, seed=1000 + ch)
        for mode in MODES:
            b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, flags, mode=mode)
            b.advance(taps / 2)
            got = device_chain(b, x, CALLS, [R48] * 3, form)
            key = f"{bpp}_{rows}_{ch}_{taps}_{flags}_{form}_{mode}"
            saved[key + "_counts"] = np.array([[u, g] for _, u, g in got] + [[int(b.state()[1]), 0]], np.int64)
            saved[key + "_offset"] = np.array([b.state()[0]], f32)
            for k, (y, _, _) in enumerate(got):
                saved[f"{key}_{k}_sha"] = np.frombuffer(hashlib.sha256(y.tobytes()).digest(), np.uint8)
                saved[f"{key}_{k}_probes"] = y[_probes(ns, ch)]
            b.free()
    for bpp, rows in GEOMETRIES:
        _set_env({"ESPB_BPP": bpp, "ESPB_CHUNK_ROWS": rows})
        raw = pcm16(70, sum(c[0] for c in WRAP_CALLS), 2, seed=77)
        for mode in MODES:
            r = espb.Resampler(70, 4500 * 2, 4950 * 2, WRAP_SR, WRAP_DR, 16, 16, 2, True, True, 256, 256, mode=mode)
            assert r.policy()["filter"] == "post"
            got = wrapper_chain(r, raw, 2, WRAP_CALLS, gain_db=2.0)
            for k, (y, u, g, clips) in enumerate(got):
                key = f"w_{bpp}_{rows}_{mode}_{k}"
                saved[key + "_y"] = y
                saved[key + "_res"] = np.concatenate([[u, g], clips]).astype(np.int64)
            r.free()
    np.savez(os.path.join(out_dir, "matrix.npz"), **saved)


def test_geometry_matrix(oracle, tmp_path):
    """All six (ESPB_BPP, ESPB_CHUNK_ROWS) geometries, exact and fast, over three chained calls (long / capacity-limited
    / uneven) of 70 stereo streams, through the interleaved-stereo, planar, 4-channel and scalar (unaligned row) output
    forms and the wrapper's post-filter path (TMCAP), plus T=1024 and flags=0 (no interpolation: the interpolating
    kernel with an idle filter, except at (4,32) where the dedicated kernel runs).  Run in a child with ESPB_DEBUG=1:
    its report must name all 24 resample<BPP,NST,CJ,EXACT,TMCAP> instantiations."""
    err = run_child(tmp_path, "_child_geometry_matrix", {"ESPB_DEBUG": "1"})
    seen = set(re.findall(r"\[espb\] resample<(\d+),(\d+),(\d+),(\d),(\d)>", err))
    want = {(str(b), str(n), str(r), str(e), str(t)) for (b, r), n in GEOMETRIES.items() for e in (0, 1) for t in (0, 1)}
    assert seen == want, sorted(want - seen)
    m = np.load(tmp_path / "matrix.npz")
    refs = {}
    for ch, ns, taps, flags, _ in MATRIX:
        x = signal(ns, sum(c[0] for c in CALLS), ch, seed=1000 + ch)
        refs[(ch, taps, flags)] = {s: oracle_chain(oracle, x[s], ch, taps, 256, 1.0, flags, CALLS, [R48] * 3)
                                   for s in _probes(ns, ch)}
    for bpp, rows, ch, ns, taps, flags, form in _matrix_cases():
        ref = refs[(ch, taps, flags)]
        probes = _probes(ns, ch)
        for mode in MODES:
            key = f"{bpp}_{rows}_{ch}_{taps}_{flags}_{form}_{mode}"
            base = f"4_32_{ch}_{taps}_{flags}_stereo_{mode}" if form != "frame4" else f"4_32_{ch}_{taps}_{flags}_frame4_{mode}"
            counts = m[key + "_counts"]
            ochain, ostate = ref[probes[0]]
            assert [tuple(c) for c in counts[:3]] == [(u, g) for _, u, g in ochain], key
            assert (m[key + "_offset"][0], int(counts[3][0])) == ostate, key
            for k in range(3):
                # identical bytes to the default geometry (and, for the other layouts, to its interleaved output)
                assert bits_equal(m[f"{key}_{k}_sha"], m[f"{base}_{k}_sha"]), (key, k)
                for i, s in enumerate(probes):
                    yo = ref[s][0][k][0]
                    y = m[f"{key}_{k}_probes"][i]
                    if mode == espb.MODE_EXACT:
                        assert bits_equal(y, yo), (key, k, s)
                    elif yo.size:
                        assert float(np.max(np.abs(y.astype(np.float64) - yo))) <= TOL, (key, k, s)
    raw = pcm16(70, sum(c[0] for c in WRAP_CALLS), 2, seed=77)
    wref = {s: oracle_wrapper_chain(oracle, raw[s], 2, WRAP_SR, WRAP_DR, WRAP_CALLS, gain_db=2.0)
            for s in (0, 31, 32, 69)}
    clipped = 0
    for bpp, rows in GEOMETRIES:
        for mode in MODES:
            for k in range(3):
                key, base = f"w_{bpp}_{rows}_{mode}_{k}", f"w_4_32_{mode}_{k}"
                y, res = m[key + "_y"], m[key + "_res"]
                assert bits_equal(y, m[base + "_y"]) and np.array_equal(res, m[base + "_res"]), key
                for s, chain in wref.items():
                    yo, uo, go, co = chain[k]
                    assert (int(res[0]), int(res[1])) == (uo, go), (key, s)
                    if mode == espb.MODE_EXACT:
                        assert bits_equal(y[s], yo) and int(res[2 + s]) == co, (key, s)
                        clipped += co
                    else:  # fast mode: within one LSB of the 16-bit output
                        assert np.max(np.abs(_le16(y[s]) - _le16(yo))) <= 1, (key, s)
    assert clipped > 0  # the +2 dB gain clips: the clip counts were compared


# ---------------------------------------------------------------- 2. chunk-table limit per geometry
def _max_chunks(taps, state, n_in, n_out, ratio, bpp, rows):
    _, _, pcb = espb.plan_passes(taps, 256, 3, float(state[0]), state[1], n_in, n_out, ratio, bpp, rows, False)
    return int(np.max(np.diff(pcb)))


def _threshold(taps, state, n_in, n_out, bpp, rows):
    """(accepted, refused) float32 ratios either side of the table limit of this geometry, for this call's plan."""
    limit = TABLE[(bpp, rows)]
    lo, hi = f32(0.0005), f32(0.05)
    assert _max_chunks(taps, state, n_in, n_out, lo, bpp, rows) > limit >= _max_chunks(taps, state, n_in, n_out, hi,
                                                                                        bpp, rows)
    for _ in range(60):
        mid = f32((float(lo) + float(hi)) / 2)
        if mid in (lo, hi):
            break
        if _max_chunks(taps, state, n_in, n_out, mid, bpp, rows) > limit:
            lo = mid
        else:
            hi = mid
    return hi, lo


@pytest.mark.parametrize("bpp,rows", list(GEOMETRIES))
def test_chunk_table_limit_per_geometry(oracle, monkeypatch, bpp, rows):
    """Per geometry, the ratio where one pass's chunks first exceed the CTA's chunk table (320 / 768 / 120 entries):
    just above it the call is refused (ESPB_ERR_ARG) before anything runs and the context stays usable; just below
    it the call runs and is bit-exact.  ESPB_PPC=64 at the accepted ratio exercises the clamp ppc * chunks <= table."""
    monkeypatch.setenv("ESPB_BPP", str(bpp))
    monkeypatch.setenv("ESPB_CHUNK_ROWS", str(rows))
    L = espb.lib()
    ns, ch, taps, n_in = 70, 2, 256, 60000
    n_out = 4000
    x = signal(ns, n_in, ch, seed=2000)
    probe = ns - 1
    b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=espb.MODE_EXACT)
    b.advance(taps / 2)
    ok, bad = _threshold(taps, b.state(), n_in, n_out, bpp, rows)
    assert float(ok) / float(bad) < 1.001
    d_in = espb.DeviceBuffer.from_numpy(x)
    d_out = espb.DeviceBuffer(ns * n_out * ch * 4)
    with pytest.raises(espb.EspbError, match="chunk table"):
        b.process_interleaved_dev(d_in.ptr, n_in * ch, n_in, d_out.ptr, n_out * ch, n_out, bad)
    assert L.espb_last_status() == -1  # ESPB_ERR_ARG
    results = {}
    for ppc in ("0", "64"):
        monkeypatch.setenv("ESPB_PPC", ppc)
        if ppc != "0":
            b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=espb.MODE_EXACT)
            b.advance(taps / 2)
        d_out.zero()
        used, gen = b.process_interleaved_dev(d_in.ptr, n_in * ch, n_in, d_out.ptr, n_out * ch, n_out, ok)
        assert L.espb_last_status() == 0 and gen > 32
        results[ppc] = (used, gen, d_out.download(f32).reshape(ns, n_out * ch)[:, : gen * ch], b.state())
        b.free()
    assert results["0"][:2] == results["64"][:2] and bits_equal(results["0"][2], results["64"][2])
    for s in (0, 64, probe):
        (yo, uo, go), = oracle_chain(oracle, x[s], ch, taps, 256, 1.0, 3, [(n_in, n_out)], [ok])[0]
        assert (results["0"][0], results["0"][1]) == (uo, go) and bits_equal(results["0"][2][s], yo), s
    d_in.free()
    d_out.free()


# ---------------------------------------------------------------- 3. G time slabs
def _resample_launches(b, seg, n_in, cap, ratio):
    b.set_option(espb.OPT_KERNEL_TIMING, 1)
    y, u, g = process_layout(b, seg, n_in, cap, ratio, "stereo")
    _, launches = b.kernel_time()
    b.set_option(espb.OPT_KERNEL_TIMING, 0)
    return (y, u, g), launches


@pytest.mark.parametrize("mode", ["exact", "fast"])
def test_g_time_slabs(oracle, monkeypatch, mode):
    """ESPB_G_MBYTES=1: the expanded coefficients of a call (8 KB per chunk, ~12 MB here) are made resident one slab
    of passes at a time and the resampler is launched once per slab.  Device buffers with staging overlap on and off;
    bytes equal to the default budget and to the oracle; kernel timing shows several launches per call; a plan-cache
    hit after reset() re-expands the first slab and gives the same bytes again."""
    md = espb.MODE_EXACT if mode == "exact" else espb.MODE_FAST
    ns, ch, taps = 70, 2, 256
    x = signal(ns, sum(c[0] for c in CALLS), ch, seed=3000)
    runs = {}
    for label, gmb, overlap in (("default", None, 1), ("slabs", "1", 1), ("slabs-serial", "1", 0)):
        if gmb:
            monkeypatch.setenv("ESPB_G_MBYTES", gmb)
        else:
            monkeypatch.delenv("ESPB_G_MBYTES", raising=False)
        b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=md)
        b.set_option(espb.OPT_OVERLAP_STAGING, overlap)
        b.advance(taps / 2)
        runs[label] = (device_chain(b, x, CALLS, [R48] * 3), b.state())
        if label == "slabs":
            # slabs happened: more than one resampler launch per call, first call again and a plan-cache hit of it
            b.reset()
            b.advance(taps / 2)
            first, n1 = _resample_launches(b, x[:, : CALLS[0][0] * ch], CALLS[0][0], CALLS[0][1], R48)
            b.reset()
            b.advance(taps / 2)
            again, n2 = _resample_launches(b, x[:, : CALLS[0][0] * ch], CALLS[0][0], CALLS[0][1], R48)
            assert n1 > 1 and n2 == n1, (n1, n2)
            same_chain([first, again], [runs["default"][0][0]] * 2, "slabs after reset / plan-cache hit")
        b.free()
    for label in ("slabs", "slabs-serial"):
        same_chain(runs[label][0], runs["default"][0], label)
        assert runs[label][1] == runs["default"][1]
    ref = {s: oracle_chain(oracle, x[s], ch, taps, 256, 1.0, 3, CALLS, [R48] * 3)[0] for s in (0, 63, 64, ns - 1)}
    check_against_oracle(runs["slabs"][0], ref, ref, md, "G slabs")


def test_g_time_slabs_paths(oracle, monkeypatch):
    """G slabs on the other kernels and entry points, each against the same configuration with the default budget
    and against the oracle: the non-interpolating kernel (half-size G rows), direct input (ESPB_DIRECT=1, split pass
    plan), the host-buffer pipeline (stream slabs serial on one CUDA stream, G re-expanded per slab) and the wrapper
    (device and host path)."""
    ns, ch, taps = 70, 2, 256
    total = sum(c[0] for c in CALLS)
    x = signal(ns, total, ch, seed=3100)
    probes = (0, 63, 64, ns - 1)

    def batch(flags, env, mode):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, flags, mode=mode)
        b.advance(taps / 2)
        for k in env:
            monkeypatch.delenv(k)
        return b

    for flags, env in ((espb.BLACKMAN_HARRIS, {}), (3, {"ESPB_DIRECT": "1"})):
        ref = {s: oracle_chain(oracle, x[s], ch, taps, 256, 1.0, flags, CALLS, [R48] * 3)[0] for s in probes}
        for mode in MODES:
            base = device_chain(batch(flags, env, mode), x, CALLS, [R48] * 3)
            b = batch(flags, dict(env, ESPB_G_MBYTES="1"), mode)
            (y, u, g), launches = _resample_launches(b, x[:, : CALLS[0][0] * ch], *CALLS[0], R48)
            assert launches > 1
            got = [(y, u, g)] + device_chain(b, x[:, u * ch:], CALLS[1:], [R48] * 2)
            same_chain(got, base, (flags, env, mode))
            check_against_oracle(got, ref, probes, mode, (flags, env))
    # host-buffer pipeline: every stream slab re-expands its G slabs on the one CUDA stream
    ref = {s: oracle_chain(oracle, x[s], ch, taps, 256, 1.0, 3, CALLS, [R48] * 3)[0] for s in probes}
    for mode in MODES:
        base = device_chain(batch(3, {}, mode), x, CALLS, [R48] * 3)
        b = batch(3, {"ESPB_G_MBYTES": "1"}, mode)
        monkeypatch.setenv("ESPB_HOST_SLABS", "3")
        got, pos = [], 0
        for n_in, cap in CALLS:
            hin = espb.PinnedBuffer(ns * n_in * ch, f32)
            hin.array[:] = x[:, pos * ch:(pos + n_in) * ch].reshape(-1)
            hout = espb.PinnedBuffer(ns * cap * ch, f32)
            hout.array[:] = 0
            u, g = b.process_interleaved_host(hin.ptr, n_in * ch, n_in, hout.ptr, cap * ch, cap, R48)
            got.append((hout.array.reshape(ns, cap * ch)[:, : g * ch].copy(), u, g))
            pos += u
            hin.free()
            hout.free()
        monkeypatch.delenv("ESPB_HOST_SLABS")
        same_chain(got, base, ("host", mode))
        check_against_oracle(got, ref, probes, mode, "host")
    # the wrapper, device and host path (44.1 -> 48 kHz stereo int16, post-filter)
    raw = pcm16(ns, sum(c[0] for c in WRAP_CALLS), 2, seed=3200)
    wref = {s: oracle_wrapper_chain(oracle, raw[s], 2, WRAP_SR, WRAP_DR, WRAP_CALLS, gain_db=1.0) for s in probes}
    results = {}
    for label, gmb, host in (("default", None, False), ("dev", "1", False), ("host", "1", True)):
        if gmb:
            monkeypatch.setenv("ESPB_G_MBYTES", gmb)
        r = espb.Resampler(ns, 4500 * 2, 4950 * 2, WRAP_SR, WRAP_DR, 16, 16, 2, True, True, 256, 256,
                           mode=espb.MODE_EXACT)
        monkeypatch.delenv("ESPB_G_MBYTES", raising=False)
        if label == "dev":
            r.set_option(espb.OPT_KERNEL_TIMING, 1)
        results[label] = wrapper_chain(r, raw, 2, WRAP_CALLS, host_path=host, gain_db=1.0)
        if label == "dev":
            assert r.kernel_time()[1] > len(WRAP_CALLS)
        r.free()
    for label in ("dev", "host"):
        same_wrapper_chain(results[label], results["default"], label)
    for s, chain in wref.items():
        for (y, u, g, clips), (yo, uo, go, co) in zip(results["host"], chain):
            assert (u, g) == (uo, go) and bits_equal(y[s], yo) and int(clips[s]) == co, s


# ---------------------------------------------------------------- 4. passes per CTA
def test_passes_per_cta(oracle, monkeypatch):
    """ESPB_PPC in {2, 3, 7, 64} over calls of 47, 53 and 1 passes (none a multiple of ppc, so the last CTA has a
    partial pass range; 64 is clamped by the chunk table) and three series groups: bytes equal ppc = 1 and the
    oracle."""
    ns, ch, taps = 150, 2, 256
    calls = [(1600, 1500), (1700, 1690), (20, 100)]  # 1500 / 1690 / ~21 outputs: 47, 53 and 1 passes of 32
    x = signal(ns, sum(c[0] for c in calls), ch, seed=4000)
    probes = (0, 63, 64, 127, ns - 1)
    ref = {s: oracle_chain(oracle, x[s], ch, taps, 256, 1.0, 3, calls, [R48] * 3)[0] for s in probes}
    assert [g for _, _, g in ref[0]][:2] == [1500, 1690]
    for mode in MODES:
        runs = {}
        for ppc in ("1", "2", "3", "7", "64"):
            monkeypatch.setenv("ESPB_PPC", ppc)
            b = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=mode)
            b.advance(taps / 2)
            runs[ppc] = device_chain(b, x, calls, [R48] * 3)
            b.free()
        for ppc in ("2", "3", "7", "64"):
            same_chain(runs[ppc], runs["1"], (ppc, mode))
        check_against_oracle(runs["7"], ref, probes, mode, "ppc")


# ---------------------------------------------------------------- 5. host pipeline slabs
@pytest.mark.parametrize("ns,ch", [(300, 1), (97, 2), (45, 3)])
def test_host_pipeline_slabs(oracle, monkeypatch, ns, ch):
    """ESPB_HOST_SLABS in {1, 3, 7, 32}: stream slabs of the host-buffer entry points, rounded to whole 128-series
    groups, uneven and with a partial last slab; process_interleaved_host and the wrapper host path must give the
    bytes (and clip counts) of the device-buffer call over two chained calls."""
    taps = 64
    calls = [(2000, 2300), (1500, 900)]
    x = signal(ns, sum(c[0] for c in calls), ch, seed=5000 + ch)
    raw = pcm16(ns, sum(c[0] for c in calls), ch, seed=5100 + ch, amp=0.6)
    sr, dr = 44100, 48000
    for mode in MODES:
        b = espb.ResampleBatch(ns, ch, taps, 64, 1.0, 3, mode=mode)
        b.advance(taps / 2)
        base = device_chain(b, x, calls, [R48] * 2, "stereo" if ch != 3 else "scalar")
        b.free()
        if mode == espb.MODE_EXACT:
            ref = {s: oracle_chain(oracle, x[s], ch, taps, 64, 1.0, 3, calls, [R48] * 2)[0] for s in (0, ns - 1)}
            check_against_oracle(base, ref, ref, mode, "device")
        r = espb.Resampler(ns, 2000 * ch, 2300 * ch, sr, dr, 16, 16, ch, True, True, taps, 64, mode=mode)
        wbase = wrapper_chain(r, raw, ch, calls, gain_db=3.0)
        r.free()
        assert sum(int(c[3].sum()) for c in wbase) > 0
        for slabs in ("1", "3", "7", "32"):
            monkeypatch.setenv("ESPB_HOST_SLABS", slabs)
            b = espb.ResampleBatch(ns, ch, taps, 64, 1.0, 3, mode=mode)
            b.advance(taps / 2)
            got, pos = [], 0
            for n_in, cap in calls:
                hin = espb.PinnedBuffer(ns * n_in * ch, f32)
                hin.array[:] = x[:, pos * ch:(pos + n_in) * ch].reshape(-1)
                hout = espb.PinnedBuffer(ns * cap * ch, f32)
                hout.array[:] = 0
                u, g = b.process_interleaved_host(hin.ptr, n_in * ch, n_in, hout.ptr, cap * ch, cap, R48)
                got.append((hout.array.reshape(ns, cap * ch)[:, : g * ch].copy(), u, g))
                pos += u
                hin.free()
                hout.free()
            b.free()
            same_chain(got, base, ("host", slabs, mode))
            r = espb.Resampler(ns, 2000 * ch, 2300 * ch, sr, dr, 16, 16, ch, True, True, taps, 64, mode=mode)
            same_wrapper_chain(wrapper_chain(r, raw, ch, calls, host_path=True, gain_db=3.0), wbase,
                               ("wrapper host", slabs, mode))
            r.free()
            monkeypatch.delenv("ESPB_HOST_SLABS")


# ---------------------------------------------------------------- 6. sequential schedule
VS_ORACLE = [  # the geometries of test_gpu_parity.py::test_resampler_vs_oracle
    (2, 70, 256, 256, 1.0, 3, f32(48000) / f32(44100), 2500),
    (2, 65, 256, 256, float(f32(44100) / f32(48000) * f32(0.96)), 1, f32(44100) / f32(48000), 2500),
    (1, 131, 256, 256, 1.0, 1, f32(3.0), 900),
    (8, 17, 1024, 256, 0.45, 1, f32(44100) / f32(96000), 3000),
    (3, 45, 32, 16, 1.0, 0, f32(1.37), 1500),
    (1, 1, 4, 2, 1.0, 3, f32(2.5), 300),
    (5, 30, 64, 1024, 0.7, 2, f32(0.61), 2000),
    (2, 70, 256, 256, 1.0, 3, f32(48000) / f32(44100), 20000),  # tables far beyond the 48 KB single upload
    (2, 1, 256, 256, 1.0, 3, f32(48000) / f32(44100), 5000),    # few-series kernel
]


@pytest.mark.parametrize("case", VS_ORACLE)
def test_sequential_schedule(oracle, monkeypatch, case):
    """ESPB_SCHED=seq: the per-output schedule built on the host and finished by espb_finalize_kernel instead of the
    closed form expanded on the device.  Two chained calls; bytes, counts and state equal the closed form's and the
    oracle's."""
    ch, ns, taps, filters, lp, flags, ratio, n_in = case
    calls = [(n_in // 3 + 1, int((n_in // 3 + 1) * float(ratio)) + 40), (n_in - n_in // 3 - 1, int(n_in * float(ratio)))]
    x = signal(ns, n_in, ch, seed=6000 + ns)
    probes = sorted({0, ns - 1})
    ref = {s: oracle_chain(oracle, x[s], ch, taps, filters, lp, flags, calls, [ratio] * 2) for s in probes}
    for mode in MODES:
        runs = {}
        for sched in ("seq", None):
            if sched:
                monkeypatch.setenv("ESPB_SCHED", sched)
            else:
                monkeypatch.delenv("ESPB_SCHED", raising=False)
            b = espb.ResampleBatch(ns, ch, taps, filters, lp, flags, mode=mode)
            b.advance(taps / 2)
            runs[sched] = (device_chain(b, x, calls, [ratio] * 2, "scalar" if ch % 2 else "stereo"), b.state())
            b.free()
        same_chain(runs["seq"][0], runs[None][0], ("seq", mode))
        assert runs["seq"][1] == runs[None][1] == ref[0][1]
        check_against_oracle(runs["seq"][0], {s: r[0] for s, r in ref.items()}, probes, mode, "seq")


# ---------------------------------------------------------------- 7. few-series <-> standard kernel in one context
R_LOW = f32(0.015)


def _switch_calls(ch):
    # 48/44.1, then a ratio at which the few-series kernel's input tile exceeds 200 KB, then 48/44.1 again
    return [(2000, 2300), (30000 if ch == 2 else 3000, 600), (2000, 2300)], [R48, R_LOW, R48]


SWITCH_SHAPES = [(1, 2), (4, 8)]


def _run_switch(ns, ch, mode):
    calls, ratios = _switch_calls(ch)
    x = signal(ns, sum(c[0] for c in calls), ch, seed=7000 + ch)
    b = espb.ResampleBatch(ns, ch, 256, 256, 1.0, 3, mode=mode)
    b.advance(128.0)
    got = device_chain(b, x, calls, ratios)
    st = b.state()
    b.free()
    return got, st


def _child_fs_switch(out_dir):
    espb.set_device(0)
    saved = {}
    for ns, ch in SWITCH_SHAPES:
        for mode in MODES:
            got, st = _run_switch(ns, ch, mode)
            for k, (y, u, g) in enumerate(got):
                saved[f"{ns}_{ch}_{mode}_{k}_y"] = y
                saved[f"{ns}_{ch}_{mode}_{k}_n"] = np.array([u, g], np.int64)
            saved[f"{ns}_{ch}_{mode}_state"] = np.array([st[0], st[1]], np.float64)
    np.savez(os.path.join(out_dir, "fs.npz"), **saved)


def _switch_refs(oracle):
    refs = {}
    for ns, ch in SWITCH_SHAPES:
        calls, ratios = _switch_calls(ch)
        x = signal(ns, sum(c[0] for c in calls), ch, seed=7000 + ch)
        refs[(ns, ch)] = {s: oracle_chain(oracle, x[s], ch, 256, 256, 1.0, 3, calls, ratios) for s in range(ns)}
    return refs


def _check_switch(got, st, ref, ns, mode, what):
    check_against_oracle(got, {s: r[0] for s, r in ref.items()}, range(ns), mode, what)
    assert st == ref[0][1], what


@pytest.mark.parametrize("slice_kb", [None, "1", "1000"])
def test_few_series_kernel_switch(oracle, monkeypatch, slice_kb):
    """One stereo stream and 4 x 8 channels (<= 32 series: the few-series kernel) chained at 48/44.1, then at a ratio
    of 0.015 where its input tile no longer fits and the call takes the standard kernel, then back: the carried
    history and the state cross both switches.  Each stream against its own oracle context; with the default slice
    width, kt = 4 (ESPB_FS_SLICE_KB=1) and the widest kt = 64 (ESPB_FS_SLICE_KB=1000); bytes identical to the default
    slice width."""
    refs = _switch_refs(oracle)
    for ns, ch in SWITCH_SHAPES:
        for mode in MODES:
            monkeypatch.delenv("ESPB_FS_SLICE_KB", raising=False)
            base, _ = _run_switch(ns, ch, mode)
            if slice_kb:
                monkeypatch.setenv("ESPB_FS_SLICE_KB", slice_kb)
            got, st = _run_switch(ns, ch, mode)
            _check_switch(got, st, refs[(ns, ch)], ns, mode, (ns, ch, slice_kb))
            same_chain(got, base, (ns, ch, slice_kb, mode))


@pytest.mark.parametrize("stages", ["3", "4"])
def test_few_series_ring_depth(oracle, tmp_path, stages):
    """ESPB_FS_STAGES (read once per process): the few-series kernel with a 3- and a 4-stage ring, over the same
    kernel-switching calls, in a child process."""
    run_child(tmp_path, "_child_fs_switch", {"ESPB_FS_STAGES": stages})
    m = np.load(tmp_path / "fs.npz")
    refs = _switch_refs(oracle)
    for ns, ch in SWITCH_SHAPES:
        for mode in MODES:
            got = [(m[f"{ns}_{ch}_{mode}_{k}_y"], *[int(v) for v in m[f"{ns}_{ch}_{mode}_{k}_n"]]) for k in range(3)]
            sv = m[f"{ns}_{ch}_{mode}_state"]
            _check_switch(got, (f32(sv[0]), int(sv[1])), refs[(ns, ch)], ns, mode, (ns, ch, stages))
            base, _ = _run_switch(ns, ch, mode)
            same_chain(got, base, (ns, ch, stages, mode))


# ---------------------------------------------------------------- 8. staging grid size
def test_staging_grid_size(oracle, monkeypatch):
    """ESPB_STAGE_CTAS = -1 (one staging CTA in all) and 1 (one per SM) on long overlapped calls: the resampler's CTAs
    wait longer for their row tiles; the bytes must equal the serial order (ESPB_OVERLAP=0) and the oracle."""
    ns, ch, taps = 200, 2, 64
    calls = [(4111, 4500), (6000, 6540), (4500, 4900)]
    x = signal(ns, sum(c[0] for c in calls), ch, seed=8000)
    ref = {s: oracle_chain(oracle, x[s], ch, taps, 128, 1.0, 3, calls, [R48] * 3)[0] for s in (0, 63, 64, ns - 1)}
    for mode in MODES:
        runs = {}
        for label, env in (("serial", {"ESPB_OVERLAP": "0"}), ("-1", {"ESPB_STAGE_CTAS": "-1"}),
                           ("1", {"ESPB_STAGE_CTAS": "1"})):
            for k in ("ESPB_OVERLAP", "ESPB_STAGE_CTAS"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            b = espb.ResampleBatch(ns, ch, taps, 128, 1.0, 3, mode=mode)
            b.set_option(espb.OPT_PLAN_CACHE, 0)
            b.advance(taps / 2)
            runs[label] = device_chain(b, x, calls, [R48] * 3)
            b.free()
        same_chain(runs["-1"], runs["serial"], ("-1", mode))
        same_chain(runs["1"], runs["serial"], ("1", mode))
        check_against_oracle(runs["-1"], ref, ref, mode, "stage ctas")


# ---------------------------------------------------------------- 9. stand-alone biquad
FIRST_ORDER = np.array([0.13, 0.13, 0.0, -0.74, 0.0], f32)  # a2 = b2 = 0: the first-order form


def _biquad_cases():
    lp, hp = espb.biquad_lowpass(0.2274), espb.biquad_highpass(0.1)
    for layout, ch in (("interleaved", 2), ("interleaved", 4), ("interleaved", 8), ("planar4", 2), ("planar", 3)):
        for sections in (1, 2, 3, 4):
            yield layout, ch, sections, lp, 1.0, 0
    yield "interleaved", 2, 1, FIRST_ORDER, 1.0, 0
    yield "interleaved", 4, 3, FIRST_ORDER, 0.5, 0
    yield "planar", 2, 3, FIRST_ORDER, 1.0, 0
    yield "interleaved", 2, 2, hp, 2.0, 0
    yield "planar4", 4, 2, hp, 1.0, 0
    yield "interleaved", 2, 2, lp, 1.0, 1   # buffer offset by 4 bytes: the unaligned (non-vector) form
    yield "interleaved", 8, 3, lp, 1.0, 1
    yield "planar4", 1, 2, lp, 1.0, 1


@pytest.mark.parametrize("onepass", ["1", "0"])
def test_standalone_biquad(oracle, monkeypatch, onepass):
    """espb_biquad_apply_buffer on its own: interleaved 2/4/8 channels and planar layouts (channel stride a multiple of
    4 floats and not), 1-4 sections, the first-order form with 1 and 3 sections, high-pass, gain; 300+ series (several
    128-series CTAs, a partial last one); 1000 frames (not a multiple of the 64-frame chunk) split 437 + 563 over two
    calls; buffers offset by 4 bytes; and ESPB_BIQUAD_ONEPASS=0 (the time-major route).  Every series against the
    oracle's apply_buffer, bit for bit, and the saved state against the oracle's."""
    monkeypatch.setenv("ESPB_BIQUAD_ONEPASS", onepass)
    n, split = 1000, 437
    for layout, ch, sections, coeffs, gain, skew in _biquad_cases():
        ns = -(-301 // ch)
        x = np.stack([noise(n, ch, stream=9000 + s, amp=0.9) for s in range(ns)])  # (ns, n*ch) interleaved
        bq = espb.BiquadBatch(ns * ch, sections, coeffs, gain)
        got = np.zeros((ns, ch, n), f32)
        for a, e in ((0, split), (split, n)):
            m = e - a
            seg = x.reshape(ns, n, ch)[:, a:e, :]
            if layout == "interleaved":
                ss = m * ch + (4 - (m * ch) % 4) % 4
                buf = np.zeros((ns, ss), f32)
                buf[:, : m * ch] = seg.reshape(ns, m * ch)
                lay = (ss, 1, ch)
            else:
                cs = (m + 3) & ~3 if layout == "planar4" else m + 1
                ss = ch * cs + 4
                buf = np.zeros((ns, ss), f32)
                for c in range(ch):
                    buf[:, c * cs: c * cs + m] = seg[:, :, c]
                lay = (ss, cs, 1)
            flat = np.concatenate([np.zeros(skew, f32), buf.reshape(-1)])
            d = espb.DeviceBuffer.from_numpy(flat)
            bq.apply_dev(d.ptr + 4 * skew, lay, ch, m)
            res = d.download(f32)[skew:].reshape(ns, ss)
            d.free()
            if layout == "interleaved":
                got[:, :, a:e] = res[:, : m * ch].reshape(ns, m, ch).transpose(0, 2, 1)
                assert bits_equal(res[:, m * ch:], buf[:, m * ch:])
            else:
                for c in range(ch):
                    got[:, c, a:e] = res[:, c * cs: c * cs + m]
                    assert bits_equal(res[:, c * cs + m: (c + 1) * cs], buf[:, c * cs + m: (c + 1) * cs])
        state = bq.state()
        bq.free()
        what = (layout, ch, sections, gain, skew, onepass)
        for s in range(ns):
            for c in range(ch):
                ref = np.ascontiguousarray(x[s, c::ch])
                for k in range(sections):
                    o = oracle.biquad(coeffs, gain)
                    o.apply_buffer(ref)
                    assert bits_equal(state[s * ch + c, k], np.frombuffer(o.buf, f32)[5:9]), (what, s, c, k)
                assert bits_equal(got[s, c], ref), (what, s, c)


# ---------------------------------------------------------------- 10. grid-stride loops
N_BIG = 2_500_000 + 13
PCM_BITS = (8, 16, 24, 32)


def _big_inputs(bits):
    rng = np.random.default_rng(bits)
    raw = rng.integers(0, 256, N_BIG * (bits // 8), dtype=np.uint8)
    x = (rng.standard_normal(N_BIG) * 0.7).astype(f32)  # loud: a few percent clip, in every thread's iterations
    return raw, x


def _q15_inputs():
    rng = np.random.default_rng(15)
    return rng.integers(-32768, 32768, N_BIG + 1).astype(np.int16), rng.integers(-32768, 32768, N_BIG + 1).astype(np.int16)


GS_RESAMPLE = (140, 2, 256, [(6000, 6600)])


def _child_grid_stride(out_dir):
    espb.set_device(0)
    L = espb.lib()
    saved = {}
    for bits in PCM_BITS:
        raw, x = _big_inputs(bits)
        saved[f"q2f_{bits}"] = espb.quantized_to_float(raw, N_BIG, bits, -1.5)
        q, clipped = espb.float_to_quantized(x, bits)
        saved[f"f2q_{bits}"] = q
        saved[f"f2q_{bits}_clipped"] = np.array([clipped], np.int64)
    a, b = _q15_inputs()
    for off in (0, 1):  # element offset 1: 2-byte aligned buffers
        d_a, d_b, d_o = espb.DeviceBuffer.from_numpy(a), espb.DeviceBuffer.from_numpy(b), espb.DeviceBuffer(2 * a.size)
        d_o.zero()
        assert L.espb_dsps_add_s16(d_a.ptr + 2 * off, d_b.ptr + 2 * off, d_o.ptr + 2 * off, N_BIG, 1, 1, 1, 1, None) == 0
        saved[f"add_{off}"] = d_o.download(np.int16)[off: off + N_BIG]
        assert L.espb_dsps_mulc_s16(d_a.ptr + 2 * off, d_o.ptr + 2 * off, N_BIG, -23170, 1, 1, None) == 0
        saved[f"mulc_{off}"] = d_o.download(np.int16)[off: off + N_BIG]
        for d in (d_a, d_b, d_o):
            d.free()
    ns, ch, taps, calls = GS_RESAMPLE
    x = signal(ns, calls[0][0], ch, seed=10000)
    rb = espb.ResampleBatch(ns, ch, taps, 256, 1.0, 3, mode=espb.MODE_EXACT)
    rb.advance(taps / 2)
    (y, u, g), = device_chain(rb, x, calls, [R48])
    saved["resample"] = y
    saved["resample_n"] = np.array([u, g], np.int64)
    np.savez(os.path.join(out_dir, "gs.npz"), **saved)


def test_grid_stride_loops(oracle, tmp_path):
    """ESPB_PCM_CTAS=1, ESPB_Q15_CTAS=1, ESPB_EXPAND_CTAS=1 (read once per process, in a child): one CTA per SM, so
    each thread runs its grid-stride loop ~60 times plus a ragged tail of 13 elements.  Quantisers both ways at 8/16/24
    and 32 bits with loud input (clip counts accumulate across iterations), Q15 add / mulc on aligned and offset
    buffers, and a standard-kernel resample (coefficient expansion over ~2000 chunks), each bit-exact with the oracle."""
    run_child(tmp_path, "_child_grid_stride", {"ESPB_PCM_CTAS": "1", "ESPB_Q15_CTAS": "1", "ESPB_EXPAND_CTAS": "1"})
    m = np.load(tmp_path / "gs.npz")
    for bits in PCM_BITS:
        raw, x = _big_inputs(bits)
        assert bits_equal(m[f"q2f_{bits}"], oracle.quantized_to_float(raw, N_BIG, bits, -1.5)), bits
        q, clipped = oracle.float_to_quantized(x, bits)
        assert clipped > 10000 and int(m[f"f2q_{bits}_clipped"][0]) == clipped, bits
        assert bits_equal(m[f"f2q_{bits}"], q), bits
    a, b = _q15_inputs()
    for off in (0, 1):
        assert bits_equal(m[f"add_{off}"], oracle.add_s16(a[off:], b[off:], N_BIG, shift=1)[0][:N_BIG]), off
        assert bits_equal(m[f"mulc_{off}"], oracle.mulc_s16(a[off:], N_BIG, -23170)[0][:N_BIG]), off
    ns, ch, taps, calls = GS_RESAMPLE
    x = signal(ns, calls[0][0], ch, seed=10000)
    for s in (0, 63, 64, ns - 1):
        (yo, uo, go), = oracle_chain(oracle, x[s], ch, taps, 256, 1.0, 3, calls, [R48])[0]
        assert tuple(int(v) for v in m["resample_n"]) == (uo, go) and bits_equal(m["resample"][s], yo), s
