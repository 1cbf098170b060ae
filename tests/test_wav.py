"""WAV header parser / emitter (SURVEY.md §8f N3; include/wav_decoder.h, src/decode/wav_decoder.cpp).  Host code:
all of this runs without a GPU.  The oracle port is checked against frozen snapshots of the compiled reference
(tests/golden/golden_wav.json); the product's C ABI against the oracle."""
import json
import os
import struct

import numpy as np
import pytest

import esp_audio_libs_b200 as espb

HERE = os.path.dirname(os.path.abspath(__file__))


def chunk(tag, payload, pad=True):
    body = tag + struct.pack("<I", len(payload)) + payload
    return body + (b"\0" if pad and len(payload) % 2 else b"")


def fmt_chunk(rate, ch, bits, extra=b""):
    ba = ch * ((bits + 7) // 8)
    return chunk(b"fmt ", struct.pack("<HHIIHH", 1, ch, rate, rate * ba, ba, bits) + extra)


def wav_cases():
    """name -> bytes.  Canonical, with extra chunks (even and odd sizes), extensible fmt, bad magic, truncated."""
    data = bytes(range(64))
    riff = lambda body: b"RIFF" + struct.pack("<I", 4 + len(body)) + b"WAVE" + body  # noqa: E731
    cases = {
        "canonical_16k_mono": riff(fmt_chunk(16000, 1, 16) + chunk(b"data", data)),
        "stereo_44k1_24bit": riff(fmt_chunk(44100, 2, 24) + chunk(b"data", data)),
        "list_before_fmt": riff(chunk(b"LIST", b"INFOISFT\x05\0\0\0Lavf\0\0") + fmt_chunk(48000, 2, 16) + chunk(b"data", data)),
        "odd_chunks_between": riff(fmt_chunk(96000, 8, 24) + chunk(b"junk", b"abc") + chunk(b"fact", b"\x01\0\0\0") +
                                   chunk(b"PEAK", b"1234567") + chunk(b"data", data)),
        "extensible_fmt_40": riff(fmt_chunk(48000, 6, 32, extra=b"\x16\0" + bytes(22)) + chunk(b"data", data)),
        "odd_fmt_size_17": riff(fmt_chunk(22050, 1, 8, extra=b"\x07") + chunk(b"data", data)),
        "data_size_odd": riff(fmt_chunk(8000, 1, 8) + chunk(b"data", b"\x80" * 33)),
        "no_riff": b"RIFX" + bytes(60),
        "no_wave": b"RIFF" + struct.pack("<I", 100) + b"AVI " + bytes(60),
        "no_data_chunk": riff(fmt_chunk(16000, 1, 16) + chunk(b"LIST", bytes(10))),
        "empty": b"",
        "huge_chunk_size": riff(fmt_chunk(16000, 1, 16) + b"junk" + struct.pack("<I", 0xFFFFFFFF) + bytes(32)),
    }
    cases["written_by_espb"] = espb.wav_write_header(48000, 2, 16, 64) + data
    return cases


def drive(dec, blob):
    """Every observable of one decoder over one file: one-shot decode of every prefix length (fresh decoder state is
    simulated by reset + the documented restart), then the incremental skip/read/next protocol of wav_decoder.h:70-76."""
    log = []
    rc = dec.decode_header(blob)
    log.append(("oneshot", rc) + dec.snapshot())
    return log


def incremental(make, blob):
    """The protocol from include/wav_decoder.h:70-76 with exact reads."""
    dec = make()
    pos, log = 0, []
    for _ in range(64):
        st = dec.snapshot()
        skip, need = st[3], st[2]
        pos += skip
        if need == 0 or pos + need > len(blob):
            break
        rc = dec.next(blob[pos:pos + need])
        pos += need
        s = dec.snapshot()
        log.append((rc,) + s[:1] + s[2:])  # bytes_processed is not touched by next()
        if rc != 0:
            break
    return log, pos


def prefixes(make, blob):
    """decode_header on a fresh decoder for a set of truncated lengths: result + snapshot each."""
    out = []
    for n in sorted(set(list(range(0, min(len(blob), 60) + 1)) + [len(blob)])):
        dec = make()
        rc = dec.decode_header(blob[:n])
        out.append((n, rc) + dec.snapshot())
    return out


def resumed(make, blob, cut):
    """decode_header called twice as a streaming reader would: first with `cut` bytes, then — after dropping the
    bytes it processed — with the rest."""
    dec = make()
    rc1 = dec.decode_header(blob[:cut])
    used = dec.snapshot()[1]
    rc2 = dec.decode_header(blob[used:])
    return (rc1, used, rc2) + dec.snapshot()


def everything(make):
    res = {}
    for name, blob in wav_cases().items():
        inc, pos = incremental(make, blob)
        res[name] = dict(prefixes=[list(map(_j, t)) for t in prefixes(make, blob)],
                         incremental=[list(map(_j, t)) for t in inc], data_offset=pos,
                         resumed=[list(map(_j, resumed(make, blob, cut))) for cut in (8, 12, 20, 36, 43)])
        # reset keeps bytes_needed (wav_decoder.cpp:151-161): reuse after reaching the data chunk fails
        dec = make()
        dec.decode_header(blob)
        dec.reset()
        rc = dec.decode_header(blob)
        res[name]["after_reset"] = [rc] + list(map(_j, dec.snapshot()))
    return res


def _j(v):
    return v.decode("latin1") if isinstance(v, bytes) else int(v)


def test_oracle_vs_frozen_reference_snapshots(oracle):
    with open(os.path.join(HERE, "golden", "golden_wav.json")) as fh:
        want = json.load(fh)
    assert json.loads(json.dumps(everything(oracle.wav))) == want


def test_product_c_abi_vs_oracle(oracle):
    assert everything(espb.WavDecoder) == everything(oracle.wav)


def test_known_answers(oracle):
    blob = wav_cases()["odd_chunks_between"]
    d = espb.WavDecoder()
    assert d.decode_header(blob) == 1  # WAV_DECODER_SUCCESS_IN_DATA
    st = d.snapshot()
    assert st[0] == 5 and (st[5], st[6], st[7]) == (96000, 8, 24) and st[4] == 64 and st[8] == b"data"
    assert blob[st[1]:st[1] + 4] == bytes(range(4))  # bytes_processed() is the offset of the first sample
    assert espb.WavDecoder().decode_header(wav_cases()["no_riff"]) == 3
    assert espb.WavDecoder().decode_header(wav_cases()["no_wave"]) == 4
    assert espb.WavDecoder().decode_header(blob[:30]) == 2  # WARNING_INCOMPLETE_DATA


def test_writer_round_trip():
    for rate, ch, bits, nbytes in ((16000, 1, 16, 32000), (44100, 2, 24, 3 * 2 * 777), (96000, 8, 32, 0), (8000, 1, 8, 33)):
        h = espb.wav_write_header(rate, ch, bits, nbytes)
        assert len(h) == 44 and h[:4] == b"RIFF" and h[8:16] == b"WAVEfmt " and h[36:40] == b"data"
        riff_size, = struct.unpack("<I", h[4:8])
        assert riff_size == 36 + nbytes + (nbytes & 1)
        d = espb.WavDecoder()
        assert d.decode_header(h) == 1
        st = d.snapshot()
        assert (st[5], st[6], st[7]) == (rate, ch, bits) and st[1] == 44 and st[4] == nbytes + (nbytes & 1)


if __name__ == "__main__":  # regenerate the frozen snapshots from the UNMODIFIED reference (needs oracle/_ref)
    from oracle_lib import Reference
    path = os.path.join(HERE, "golden", "golden_wav.json")
    with open(path, "w") as fh:
        json.dump(everything(Reference().wav), fh, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path))
