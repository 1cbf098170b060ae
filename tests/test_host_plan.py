"""Host-side logic of the product (no GPU): the C-ABI library loads and exports every
declared symbol, and its planning code (filter bank, position schedule, wrapper policy)
matches the golden fixtures made from the unmodified reference.  The schedule is
additionally proven by replaying it in numpy with the kernel's arithmetic (one
accumulator per dot product, taps in order, FMUL+FADD) against the golden outputs."""
import hashlib
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
from conftest import bits_equal

import esp_audio_libs_b200 as espb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_library_loads_and_exports_every_declared_symbol():
    L = espb.lib()
    names = espb.declared_symbols()
    assert len(names) >= 50
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert L.espb_abi_version() == 1
    assert os.path.basename(espb.library_path()) == "libesp_audio_b200.so"


def test_no_cpu_fallback_fails_loudly():
    """Run in a child process with every CUDA device hidden, so that a machine with a GPU checks it too."""
    code = textwrap.dedent(f"""
        import sys
        sys.path.insert(0, {ROOT!r})
        import pytest
        import esp_audio_libs_b200 as espb
        assert espb.device_count() == 0
        with pytest.raises(espb.EspbError, match="no CUDA device"):
            espb.ResampleBatch(2, 2, 64, 64, 1.0, 3)
        with pytest.raises(espb.EspbError):
            espb.BiquadBatch(4, 2, espb.biquad_lowpass(0.2))
        with pytest.raises(espb.EspbError):
            espb.Resampler(2, 1024, 4096, 44100, 48000, 16, 16, 2)
    """)
    p = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr[-2000:]


def test_invalid_init_parameters():
    assert espb.plan_filter_bank(30, 16, 1.0, 0) is None
    assert espb.plan_filter_bank(0, 16, 1.0, 0) is None
    assert espb.plan_filter_bank(1028, 16, 1.0, 0) is None
    assert espb.plan_filter_bank(32, 1, 1.0, 0) is None
    assert espb.plan_filter_bank(32, 1025, 1.0, 0) is None


def test_filter_bank_matches_reference(golden):
    arrays, meta = golden
    for k, b in enumerate(meta["banks"]):
        bank, eff = espb.plan_filter_bank(b["taps"], b["filters"], b["lowpass"], b["flags"])
        assert eff == b["eff_flags"]
        assert sha(bank) == b["sha256"], b
        if f"bank{k}" in arrays:
            assert bits_equal(bank, arrays[f"bank{k}"])


def test_schedule_counts_and_state_match_reference(golden):
    _, meta = golden
    for c in meta["large"] + meta["small"]:
        taps = c["taps"]
        adv = c.get("advance", taps / 2)
        off = f32(f32(taps // 2) + f32(adv))
        s = espb.plan_schedule(taps, c["filters"], _eff_flags(c), off, taps, c["n_in"], c["cap"], f32(c["ratio"]),
                               want_entries=False)
        assert (s["used"], s["generated"]) == (c["used"], c["generated"]), c["name"]
        assert (float(s["end_offset"]), s["end_index"]) == (c["final_offset"], c["final_index"]), c["name"]


def _eff_flags(c):
    fl = c["flags"]
    return (fl | 4) if 0.0 < c["lowpass"] < 1.0 else (fl & ~4)


def replay(bank, sched, x, channels, taps):
    """out[n, c] from the schedule with the kernel's arithmetic: for k in taps: acc = acc + h[k]*x[ws+k]."""
    n = sched["generated"]
    xin = np.ascontiguousarray(x, f32).reshape(-1, channels)
    xpad = np.concatenate([np.zeros((taps, channels), f32), xin, np.zeros((taps, channels), f32)])
    ws = sched["ws"].astype(np.int64) + taps
    out = np.zeros((n, channels), f32)
    acc1 = np.zeros((n, channels), f32)
    acc2 = np.zeros((n, channels), f32)
    h1 = bank[sched["phase"]]
    h2 = bank[np.minimum(sched["phase"] + 1, bank.shape[0] - 1)]
    for k in range(taps):
        xs = xpad[ws + k]
        acc1 = acc1 + (h1[:, k:k + 1] * xs).astype(f32)
        acc2 = acc2 + (h2[:, k:k + 1] * xs).astype(f32)
    w = sched["w"][:, None]
    blend = (acc2 * w).astype(f32) + (acc1 * (f32(1.0) - w)).astype(f32)
    kind = sched["kind"][:, None]
    passthrough = xpad[ws + taps // 2 - 1]
    out = np.where(kind == 3, blend, np.where(kind == 2, acc1, passthrough)).astype(f32)
    return out.reshape(-1)


def test_schedule_replay_is_bit_exact(golden):
    arrays, meta = golden
    for c in meta["small"]:
        taps = c["taps"]
        bank, eff = espb.plan_filter_bank(taps, c["filters"], c["lowpass"], c["flags"])
        off = f32(f32(taps // 2) + f32(c["advance"]))
        s = espb.plan_schedule(taps, c["filters"], eff, off, taps, c["n_in"], c["cap"], f32(c["ratio"]))
        y = replay(bank, s, arrays[f"small_{c['name']}_x"], c["channels"], taps)
        assert bits_equal(y, arrays[f"small_{c['name']}_y"]), c["name"]
        assert np.all(np.diff(s["ws"]) >= 0)
        assert s["ws"].min() >= -taps


def test_schedule_kinds(golden):
    # KAT: over C1's 479880 outputs the fractional offset is exactly 0 for 93 and the blend weight 0 for 24139
    s = espb.plan_schedule(256, 256, 3, f32(256.0), 256, 441000, 480016, f32(48000) / f32(44100))
    assert s["generated"] == 479880
    assert int((s["kind"] == 1).sum()) == 93
    assert int((s["kind"] == 2).sum()) == 24139
    # with the low-pass on there are no shortcuts
    s = espb.plan_schedule(256, 256, 5, f32(256.0), 256, 48000, 48000, f32(44100) / f32(48000))
    assert set(np.unique(s["kind"])) == {3}
    # non-interpolating: nearest phase may equal numFilters
    s = espb.plan_schedule(32, 16, 0, f32(16.0), 32, 5000, 8000, f32(1.37))
    assert set(np.unique(s["kind"])) <= {1, 2} and s["phase"].max() == 16


def test_required_and_expected_follow_the_oracle(oracle):
    rng = np.random.default_rng(8)
    for _ in range(30):
        taps = int(rng.choice([4, 16, 64, 256, 1024]))
        ratio = f32(rng.uniform(0.3, 3.2))
        n = int(rng.integers(0, 5000))
        ctx = oracle.resampler(1, taps, 32, 1.0, 3)
        adv = float(rng.choice([0.0, taps / 2, 1.75]))
        ctx.advance(adv)
        off, idx = ctx.state()
        s = espb.plan_schedule(taps, 32, 3, off, idx, n, 10 ** 7, ratio, want_entries=False)
        assert s["generated"] == ctx.expected(n, ratio)
        s = espb.plan_schedule(taps, 32, 3, off, idx, 10 ** 7, n, ratio, want_entries=False)
        assert s["used"] == ctx.required(n, ratio)


def test_wrapper_policy_matches_oracle(oracle):
    rates = [8000, 16000, 22050, 32000, 44100, 48000, 88200, 96000]
    for sr in rates:
        for dr in rates:
            for taps in (32, 256, 1024):
                for use_f in (0, 1):
                    w = oracle.wrapper(64, 64, float(sr), float(dr), 16, 16, 2, use_f, 1, taps, 64)
                    a = oracle.wrapper_policy(w)
                    b = espb.plan_policy(sr, dr, 16, 16, 2, use_f, 1, taps, 64)
                    assert a["filter"] == b["filter"], (sr, dr, taps)
                    assert a["sample_ratio"] == b["sample_ratio"] and a["art_lowpass"] == b["art_lowpass"]
                    assert a["art_flags"] == b["art_flags"], (sr, dr, taps, a, b)
                    if a["filter"] != "none":
                        assert bits_equal(a["coeffs"], b["coeffs"])
    # SURVEY §8a R7: which branch each BASELINE config takes
    assert espb.plan_policy(44100, 48000, 32, 32, 2, 1, 1, 256, 256)["filter"] == "post"
    assert espb.plan_policy(16000, 48000, 16, 16, 1, 1, 1, 256, 256)["filter"] == "post"
    assert espb.plan_policy(96000, 44100, 24, 24, 2, 1, 1, 1024, 256)["filter"] == "pre"
    assert espb.plan_policy(48000, 44100, 32, 32, 2, 1, 1, 256, 256)["filter"] == "pre"


def test_biquad_design_matches_golden(golden):
    arrays, meta = golden
    for k, b in enumerate(meta["biquad"]):
        c = espb.biquad_lowpass(b["f"]) if b["kind"] == "lp" else espb.biquad_highpass(b["f"])
        assert bits_equal(c, arrays[f"biquad_{k}_c"])


def test_cpp_shim_compiles_and_links(tmp_path):
    """include/esp_audio_b200.hpp (the reference's names over the C ABI) and the plain-C header build."""
    import shutil
    import subprocess
    if not shutil.which("g++"):
        pytest.skip("no g++")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "shim.cpp"
    src.write_text('#include "esp_audio_b200.hpp"\n'
                   "namespace b = esp_audio_libs_b200;\n"
                   "int main() { b::resampler::Resampler r(4, 1024, 4096); (void) r;\n"
                   "  b::art_resampler::BiquadCoefficients c; b::art_resampler::biquad_lowpass(&c, 0.2274);\n"
                   "  unsigned char h[44]; espb_wav_write_header(h, 48000, 2, 16, 960);\n"
                   "  b::wav_decoder::WAVDecoder d;\n"
                   "  if (d.decode_header(h, 44) != b::wav_decoder::WAV_DECODER_SUCCESS_IN_DATA) return 2;\n"
                   "  if (d.sample_rate() != 48000 || d.num_channels() != 2 || d.bits_per_sample() != 16 ||\n"
                   "      d.chunk_name() != \"data\" || d.chunk_bytes_left() != 960 || d.bytes_processed() != 44) return 3;\n"
                   "  if (b::dsps_add_s16(nullptr, nullptr, nullptr, 4, 1, 1, 1, 0) != -1) return 4;\n"
                   "  return (espb_abi_version() == ESPB_ABI_VERSION && c.a0 > 0.25f && c.a0 < 0.26f) ? 0 : 1; }\n")
    exe = tmp_path / "shim"
    libdir = os.path.dirname(espb.library_path())
    subprocess.run(["g++", "-std=c++11", "-I", os.path.join(root, "include"), str(src), "-o", str(exe), "-L", libdir,
                    "-lesp_audio_b200", f"-Wl,-rpath,{libdir}"], check=True)
    assert subprocess.run([str(exe)]).returncode == 0
    csrc = tmp_path / "hdr.c"
    csrc.write_text('#include "esp_audio_b200.h"\nint main(void) { return 0; }\n')
    subprocess.run(["gcc", "-std=c99", "-fsyntax-only", "-I", os.path.join(root, "include"), str(csrc)], check=True)


@pytest.mark.parametrize("taps,ratio,n_in,split", [(256, 48000 / 44100, 5000, False), (256, 48000 / 44100, 5000, True),
                                                  (64, 0.37, 3001, True), (1024, 44100 / 96000, 9000, True),
                                                  (32, 3.0, 700, True), (8, 1.0, 100, True),
                                                  # the call lengths of test_gpu_limits.py's real-size tests
                                                  (32, 48000 / 44100, 2_100_000, False),
                                                  (32, 48000 / 44100, 4_200_000, True)])
def test_pass_plan_covers_every_window(taps, ratio, n_in, split):
    """The chunk table the kernel sweeps (host logic, no GPU): every output's window lies inside the chunks of its
    pass, chunks of a pass are contiguous in time, and the split form the direct-input kernel needs never straddles
    input frame 0, starts history chunks on multiples of 4 rows and input chunks on even frames."""
    f32 = np.float32
    filters, flags, bpp, rows = 64, 3, 4, 32
    n_out = int(n_in * ratio) + 16
    sched = espb.plan_schedule(taps, filters, flags, float(taps // 2), taps, n_in, n_out, f32(ratio))
    cs, cp, pcb = espb.plan_passes(taps, filters, flags, float(taps // 2), taps, n_in, n_out, f32(ratio), bpp, rows, split)
    gen = sched["generated"]
    assert gen > 0 and len(pcb) == (gen + bpp * 8 - 1) // (bpp * 8) + 1 and pcb[0] == 0 and pcb[-1] == len(cs)
    ws = sched["ws"]
    for p in range(len(pcb) - 1):
        a, b = int(pcb[p]), int(pcb[p + 1])
        assert b > a and np.all(cp[a:b] == p)
        starts = cs[a:b].astype(np.int64)
        lo, hi = int(ws[p * bpp * 8]), int(ws[min((p + 1) * bpp * 8, gen) - 1]) + taps
        covered = np.zeros(hi - lo, bool)
        for k, j in enumerate(starts):
            end = j + rows
            if split and j < 0:
                assert j % 4 == 0
                end = min(end, 0)  # rows from frame 0 on belong to the chunk that starts there
                if hi > 0 >= lo:
                    pass
            elif split:
                assert j % 2 == 0 and j >= 0
            if k + 1 < len(starts):
                nxt = starts[k + 1]
                assert nxt == j + rows or (split and j < 0 <= j + rows and nxt == 0) or (split and j < 0 and nxt == 0)
            covered[max(j, lo) - lo: max(min(end, hi), lo) - lo] = True
        assert covered.all(), (p, lo, hi, starts)


def test_closed_form_schedule_is_the_sequential_machine():
    """The processing path plans with a closed form (plan.cpp:build_schedule_segments: the FP32 offset accumulator of
    art_resampler.cpp:195,236 advances by an exact constant inside one binade, so runs of outputs are arithmetic
    progressions) and expands it per output on the device.  Its host expansion must equal the reference's
    sequential state machine bit for bit — entries, counts and final state — for the BASELINE shapes and for random
    geometries, ratios (rational, near-unity, tie-prone steps, strong down-sampling) and chained calls."""
    rng = np.random.default_rng(5)

    def same(taps, filters, flags, off, idx, n_in, n_out, ratio):
        a = espb.plan_schedule(taps, filters, flags, off, idx, n_in, n_out, ratio)
        b = espb.plan_schedule_segments(taps, filters, flags, off, idx, n_in, n_out, ratio)
        assert (a["used"], a["generated"], a["end_index"]) == (b["used"], b["generated"], b["end_index"])
        assert a["end_offset"].tobytes() == b["end_offset"].tobytes()
        for k in ("ws", "phase", "w", "kind"):
            assert a[k].tobytes() == b[k].tobytes(), (k, taps, filters, flags, off, idx, n_in, n_out, float(ratio))
        return a, b

    a, b = same(256, 256, 3, 256.0, 256, 441000, 480016, f32(48000) / f32(44100))       # C1: 479880 outputs
    assert a["generated"] == 479880 and b["segments"] < 1000                             # ... in < 1000 runs
    same(1024, 256, 5, 1024.0, 1024, 960000, 441100, f32(44100) / f32(96000))            # C4 unit
    same(256, 256, 1, 256.0, 256, 480000, 441000, f32(44100) / f32(48000))               # C5 unit
    same(256, 256, 3, 256.0, 256, 160000, 480100, f32(3.0))                              # C3 unit
    # the call lengths of test_gpu_limits.py's real-size tests (thousands of 16 T ring cycles at T = 32)
    same(32, 32, 3, 32.0, 32, 2_100_000, 2_290_000, f32(48000) / f32(44100))
    same(32, 32, 3, 32.0, 32, 4_200_000, 4_580_000, f32(48000) / f32(44100))
    for _ in range(150):
        taps = int(rng.choice([4, 8, 16, 32, 64, 128, 256, 512, 1024, 12, 20, 36, 100, 260]))
        filters, flags = int(rng.integers(2, 1025)), int(rng.integers(0, 8))
        kind = rng.integers(0, 6)
        if kind == 0:
            ratio = f32(rng.uniform(0.3, 3.0))
        elif kind == 1:
            ratio = f32(rng.choice([0.5, 2.0, 1.0, 4.0, 0.25, 1.5, 3.0, 8.0, 0.125]))
        elif kind == 2:
            ratio = f32(rng.integers(1, 200)) / f32(rng.integers(1, 200))
        elif kind == 3:
            ratio = f32(1.0) + f32(rng.uniform(-1e-3, 1e-3))
        elif kind == 4:
            ratio = f32(1.0) / (f32(0.5) + f32(2.0 ** -int(rng.integers(10, 24))))  # steps that round on ties
        else:
            ratio = f32(rng.uniform(0.02, 0.3))
        off, idx = f32(taps / 2), taps
        if rng.random() < 0.7:
            off = f32(off + f32(taps / 2))
        if rng.random() < 0.3:
            off = f32(off + f32(rng.uniform(0, 3)))
        for _call in range(int(rng.integers(1, 5))):
            n_in = int(rng.choice([0, 1, 7, 441, 1000, 5000, 20000, 70000]))
            n_out = int(rng.choice([0, 1, 5, 480, 1200, 6000, 30000, 200000]))
            a, _ = same(taps, filters, flags, float(off), idx, n_in, n_out, ratio)
            off, idx = a["end_offset"], a["end_index"]


def test_shard_ranges_and_multi_gpu_symbols():
    """espb_shard_range (C) == the Python helper; contiguous, covering, sizes differ by at most one; NCCL resolves at
    run time (the library loads and these host-only entry points work without a GPU)."""
    import ctypes as C
    L = espb.lib()
    for n in (0, 1, 7, 4096, 65536, 65537):
        for world in (1, 2, 3, 8):
            nxt = 0
            for r in range(world):
                first, count = C.c_int64(0), C.c_int64(0)
                L.espb_shard_range(n, r, world, C.byref(first), C.byref(count))
                assert (first.value, count.value) == espb.shard_range(n, r, world)
                assert first.value == nxt and count.value in (n // world, n // world + 1)
                nxt += count.value
            assert nxt == n
    assert L.espb_nccl_version() >= 0          # 0: no NCCL on this machine; the single-GPU path does not need it
    assert L.espb_multi_size(None) == 0 and L.espb_dist_world(None) == 0
