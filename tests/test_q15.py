"""dsp.h Q15 helpers (SURVEY.md §8f N4): oracle vs golden vectors of the unmodified reference (CPU), oracle vs the
reference's frozen record of random cases (CPU), CUDA path vs oracle and golden (GPU)."""
import hashlib
import json
import os

import numpy as np
import pytest
from conftest import bits_equal

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_RANDOM = os.path.join(HERE, "golden", "golden_q15_random.json")


@pytest.fixture(scope="module")
def q15_golden():
    return np.load(os.path.join(HERE, "golden", "golden_q15.npz"))


def _cases(g):
    for row in g["cases"]:
        yield ("add" if row[0] == 0 else "mulc"), [int(v) for v in row[1:]]


def _run(backend, g, kind, args):
    if kind == "add":
        k, n, s1, s2, so, shift = args
        return backend.add_s16(g["a"], g["b"], n, s1, s2, so, shift), g[f"add_{k}"]
    k, n, c, si, so, _ = args
    return backend.mulc_s16(g["a"], n, c, si, so), g[f"mulc_{k}"]


def test_oracle_matches_reference_golden(oracle, q15_golden):
    for kind, args in _cases(q15_golden):
        (out, rc), want = _run(oracle, q15_golden, kind, args)
        assert rc == 0 and bits_equal(out, want), (kind, args)


def test_known_answers(oracle):
    # dsps_add_s16_ansi.c:23-24 — 32-bit sum, arithmetic shift, truncation (no saturation)
    out, _ = oracle.add_s16(np.array([32767, -32768, -1, 3], np.int16), np.array([1, -1, 0, -6], np.int16), 4)
    assert out.tolist() == [-32768, 32767, -1, -3]
    out, _ = oracle.add_s16(np.array([32767, -32768, -1, 3], np.int16), np.array([1, -1, 0, -6], np.int16), 4, shift=1)
    assert out.tolist() == [16384, -16385, -1, -2]
    # dsps_mulc_s16_ansi.c:27-28 — (x * C) >> 15: -32768 * -32768 wraps to -32768
    out, _ = oracle.mulc_s16(np.array([-32768, 32767, 1, -1], np.int16), 4, -32768)
    assert out.tolist() == [-32768, -32767, -1, 1]
    out, _ = oracle.mulc_s16(np.array([-32768, 32767, 1, -1], np.int16), 4, 16384)
    assert out.tolist() == [-16384, 16383, 0, -1]


def record_random(backend):
    """SHA-256 of every output of 200 seeded random add / mulc calls."""
    rng = np.random.default_rng(5)
    out = []
    for _ in range(200):
        n = int(rng.integers(0, 400))
        s1, s2, so = (int(v) for v in rng.integers(1, 4, 3))
        a = rng.integers(-32768, 32768, max(n * 3, 1)).astype(np.int16)
        b = rng.integers(-32768, 32768, max(n * 3, 1)).astype(np.int16)
        shift = int(rng.integers(0, 17))
        c = int(rng.integers(-32768, 32768))
        out.append([hashlib.sha256(backend.add_s16(a, b, n, s1, s2, so, shift)[0].tobytes()).hexdigest(),
                    hashlib.sha256(backend.mulc_s16(a, n, c, s1, so)[0].tobytes()).hexdigest()])
    return out


def test_oracle_vs_reference_random(oracle):
    """Against the reference's record of the same calls (tests/golden/golden_q15_random.json, written by the oracle
    port; at commit 3e4b2c7 these calls passed bit for bit against the compiled reference, and neither has changed
    since).  `python tests/test_q15.py` rewrites the record from oracle/_ref where it exists."""
    with open(GOLDEN_RANDOM) as fh:
        want = json.load(fh)
    got = record_random(oracle)
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert g == w, k


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_cuda_matches_golden(q15_golden):
    import esp_audio_libs_b200 as espb
    for kind, args in _cases(q15_golden):
        (out, rc), want = _run(espb._Q15Backend, q15_golden, kind, args)
        assert rc == 0 and bits_equal(out, want), (kind, args)


@pytest.mark.gpu
def test_cuda_vs_oracle_shapes_and_alignment(oracle):
    import esp_audio_libs_b200 as espb
    rng = np.random.default_rng(11)
    L = espb.lib()
    for n in (0, 1, 7, 8, 9, 1023, 4096, 100003, 1 << 20):
        a = rng.integers(-32768, 32768, max(n, 1)).astype(np.int16)
        b = rng.integers(-32768, 32768, max(n, 1)).astype(np.int16)
        for shift in (0, 1, 4):
            out, rc = espb.dsps_add_s16(a, b, n, shift=shift)
            assert rc == 0 and bits_equal(out, oracle.add_s16(a, b, n, shift=shift)[0]), (n, shift)
        for c in (32767, -32768, 23170, -7):
            out, rc = espb.dsps_mulc_s16(a, n, c)
            assert rc == 0 and bits_equal(out, oracle.mulc_s16(a, n, c)[0]), (n, c)
    # strides, and untouched gaps of a strided output keep their previous contents
    n = 5000
    a = rng.integers(-32768, 32768, n * 3).astype(np.int16)
    b = rng.integers(-32768, 32768, n * 3).astype(np.int16)
    init = rng.integers(-32768, 32768, n * 3).astype(np.int16)
    for s1, s2, so in ((2, 1, 1), (1, 3, 2), (3, 2, 3)):
        out, rc = espb.dsps_add_s16(a, b, n, s1, s2, so, 2, out_init=init[:n * so])
        want = init[:n * so].copy()
        want[::so] = oracle.add_s16(a, b, n, s1, s2, so, 2)[0][::so]
        assert rc == 0 and bits_equal(out, want), (s1, s2, so)
        out, rc = espb.dsps_mulc_s16(a, n, -20000, s1, so, out_init=init[:n * so])
        want = init[:n * so].copy()
        want[::so] = oracle.mulc_s16(a, n, -20000, s1, so)[0][::so]
        assert rc == 0 and bits_equal(out, want), (s1, so)
    # unaligned device pointers (2-byte offset) and in-place operation (output aliases input 1, as a mixer does)
    n = 40001
    a = rng.integers(-32768, 32768, n + 1).astype(np.int16)
    b = rng.integers(-32768, 32768, n + 1).astype(np.int16)
    d_a, d_b = espb.DeviceBuffer.from_numpy(a), espb.DeviceBuffer.from_numpy(b)
    assert L.espb_dsps_add_s16(d_a.ptr + 2, d_b.ptr + 2, d_a.ptr + 2, n, 1, 1, 1, 1, None) == 0
    got = d_a.download(np.int16, n + 1)
    assert got[0] == a[0] and bits_equal(got[1:], oracle.add_s16(a[1:], b[1:], n, shift=1)[0])
    assert L.espb_dsps_mulc_s16(d_b.ptr, d_b.ptr, n + 1, 12345, 1, 1, None) == 0
    assert bits_equal(d_b.download(np.int16, n + 1), oracle.mulc_s16(b, n + 1, 12345)[0])
    # the reference's ESP_FAIL cases
    assert L.espb_dsps_add_s16(None, d_b.ptr, d_a.ptr, 4, 1, 1, 1, 0, None) != 0
    assert L.espb_dsps_mulc_s16(d_a.ptr, None, 4, 1, 1, 1, None) != 0
    d_a.free()
    d_b.free()


@pytest.mark.gpu
def test_cuda_full_size_mix_properties():
    """C3-sized mix (16384 streams x 48005 int16 frames): linearity-style properties that need no oracle —
    (a + 0) >> 0 == a, mulc by 0x4000 twice == arithmetic >> 2 of the >> 1, add is commutative."""
    import esp_audio_libs_b200 as espb
    L = espb.lib()
    n = 16384 * 48005
    rng = np.random.default_rng(3)
    base = rng.integers(-32768, 32768, 1 << 22).astype(np.int16)
    a = np.tile(base, n // base.size + 1)[:n]
    d_a, d_z, d_o, d_p = espb.DeviceBuffer.from_numpy(a), espb.DeviceBuffer(2 * n), espb.DeviceBuffer(2 * n), espb.DeviceBuffer(2 * n)
    d_z.zero()
    assert L.espb_dsps_add_s16(d_a.ptr, d_z.ptr, d_o.ptr, n, 1, 1, 1, 0, None) == 0
    assert espb.checksum_u32(d_o.ptr, n // 2) == espb.checksum_u32(d_a.ptr, n // 2)
    assert L.espb_dsps_add_s16(d_a.ptr, d_o.ptr, d_p.ptr, n, 1, 1, 1, 1, None) == 0   # (a + a) >> 1 == a
    assert espb.checksum_u32(d_p.ptr, n // 2) == espb.checksum_u32(d_a.ptr, n // 2)
    assert L.espb_dsps_mulc_s16(d_a.ptr, d_o.ptr, n, 16384, 1, 1, None) == 0          # a >> 1
    assert L.espb_dsps_add_s16(d_a.ptr, d_z.ptr, d_p.ptr, n, 1, 1, 1, 1, None) == 0   # (a + 0) >> 1
    assert espb.checksum_u32(d_o.ptr, n // 2) == espb.checksum_u32(d_p.ptr, n // 2)
    for d in (d_a, d_z, d_o, d_p):
        d.free()


if __name__ == "__main__":  # rewrite the frozen record from the UNMODIFIED reference (needs oracle/_ref)
    from oracle_lib import Reference
    with open(GOLDEN_RANDOM, "w") as fh:
        json.dump(record_random(Reference()), fh, separators=(",", ":"))
    print("wrote", GOLDEN_RANDOM, os.path.getsize(GOLDEN_RANDOM))
