"""The oracle's fused form (oracle.resampler(..., fused=True), orc_resample_set_fused): every dot product is an fmaf
chain in tap order, the arithmetic that defines the library's fast mode (DESIGN.md §2.2).  tests/test_gpu_fast_mode.py
holds every fast-mode path to it bit for bit, so the fused form is trusted only after these checks:

- libm's fmaf is correctly rounded (against exact rational arithmetic), so the chain is defined by IEEE alone;
- on dyadic input (samples 0, -0, +-2^k) every product is exact, so fused and plain must give the same bits, counts
  and state, over the golden geometries, T = 4 ... 1024, F = 2 ... 1024, all flag values, low-pass < 1, ratios
  0.21 ... 3 with the exact ratios 0.5, 1 and 2, and chained calls;
- on generic input fused differs from plain, and by no more than the 1e-6 bar;
- both stay within the forward-error bound of a float64 model of the same operation, built from the library's
  host-only filter bank and schedule;
- the switch is per context and off by default."""
import ctypes as C
import ctypes.util
from fractions import Fraction

import numpy as np
import pytest
from conftest import bits_equal
from oracle_lib import DYADIC_K, Reference, dyadic, multitone, noise

f32 = np.float32
TOL = 1e-6  # BASELINE.json north_star: max-abs 1e-6 full scale (fast mode)
FLT_MIN = 2.0 ** -126
R48, R44 = f32(48000) / f32(44100), f32(44100) / f32(48000)


# ---------------------------------------------------------------- libm fmaf
def _round_f32(q):
    """The float32 nearest to the rational q, ties to even (subnormals included), as a Python float; inf past the
    largest finite float32."""
    if q == 0:
        return 0.0
    m = abs(q)
    e = m.numerator.bit_length() - m.denominator.bit_length()
    while Fraction(2) ** e > m:
        e -= 1
    while Fraction(2) ** (e + 1) <= m:
        e += 1
    quantum = Fraction(2) ** (max(e, -126) - 23)
    scaled = m / quantum
    k = scaled.numerator // scaled.denominator
    rem = scaled - k
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and k % 2 == 1):
        k += 1
    v = k * quantum
    r = float("inf") if v >= Fraction(2) ** 128 else float(v)
    return -r if q < 0 else r


def _fma_exact(a, b, c):
    """IEEE fma(a, b, c) of float32 values: the exact a*b + c rounded once; an exact zero is -0 only when a*b and c
    are both -0 (round to nearest)."""
    fa, fb, fc = (Fraction(float(v)) for v in (a, b, c))
    q = fa * fb + fc
    if q == 0:
        prod_neg = (np.signbit(a) != np.signbit(b))
        both_neg = (fa * fb == 0) and prod_neg and (fc == 0) and np.signbit(c)
        return f32(-0.0) if both_neg else f32(0.0)
    return f32(_round_f32(q))


def _fmaf_triples(rng):
    """~10^4 float32 triples: random magnitudes, near-total cancellation, exact ties, signed zeros."""
    out = []
    for _ in range(4000):  # random, exponents -20 ... 20, both signs
        a, b, c = (f32(rng.choice([-1, 1]) * rng.uniform(1, 2) * 2.0 ** int(rng.integers(-20, 21))) for _ in range(3))
        out.append((a, b, c))
    for _ in range(3000):  # c = -fl(a*b) (+- a few ulps): the result is the product's rounding error (or near it)
        a, b = (f32(rng.choice([-1, 1]) * rng.uniform(1, 2) * 2.0 ** int(rng.integers(-30, 31))) for _ in range(2))
        c = -f32(np.float64(a) * np.float64(b))
        for _ in range(int(rng.integers(0, 3))):
            c = np.nextafter(c, f32(rng.choice([-np.inf, np.inf])))
        out.append((a, b, f32(c)))
    for _ in range(3000):  # exact ties: (1 + i/2^12)(1 + j/2^12), i, j odd, has a half-ulp bit 2^-24; c keeps it
        i, j = (int(rng.integers(0, 300)) * 2 + 1 for _ in range(2))
        ea, eb = (int(rng.integers(-40, 41)) for _ in range(2))
        sa, sb = rng.choice([-1, 1]), rng.choice([-1, 1])
        a = f32(sa * (1 + i / 4096) * 2.0 ** ea)
        b = f32(sb * (1 + j / 4096) * 2.0 ** eb)
        p = float(Fraction(float(a)) * Fraction(float(b)) / Fraction(2) ** (ea + eb))  # |p| in [1, 2)
        m = int(rng.integers(0, 2 ** 20))  # c: a multiple of 2^-23 that keeps |a*b + c| in [1, 2)
        c = (-1 if p < 0 else 1) * m * 2.0 ** -23
        if not 1 <= abs(p + c) < 2:
            c = 0.0
        out.append((a, b, f32(c * 2.0 ** (ea + eb))))
    for a in (f32(0.0), f32(-0.0), f32(1.5)):
        for b in (f32(0.0), f32(-0.0), f32(-3.0)):
            for c in (f32(0.0), f32(-0.0), f32(2.0 ** -140)):
                out.append((a, b, c))
    return out


def test_libm_fmaf_is_correctly_rounded():
    """The fused oracle calls libm's fmaf; glibc's is correctly rounded.  ~10^4 triples against exact rational
    arithmetic, bit for bit, including exact ties (round half to even), cancellation and signed zeros."""
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.fmaf.restype = C.c_float
    libm.fmaf.argtypes = [C.c_float] * 3
    rng = np.random.default_rng(2024)
    triples = _fmaf_triples(rng)
    assert len(triples) >= 10000
    ties = 0
    for a, b, c in triples:
        want = _fma_exact(a, b, c)
        got = f32(libm.fmaf(float(a), float(b), float(c)))
        assert bits_equal(np.array([got]), np.array([want])), (a, b, c, got, want)
        q = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
        if q != 0 and abs(q - Fraction(float(want))) * 2 == abs(Fraction(float(np.nextafter(want, f32(np.inf)))) -
                                                                 Fraction(float(want))):
            ties += 1
    assert ties > 500  # the tie cases did land on ties


# ---------------------------------------------------------------- dyadic input: fused == plain
def _chain(oracle, case, x, fused):
    ch, taps, filters, lp, flags, ratio, calls, adv = case
    o = oracle.resampler(ch, taps, filters, lp, flags, fused=fused)
    o.advance(adv)
    out, pos = [], 0
    for n_in, cap in calls:
        assert (pos + n_in) * ch <= x.size  # the oracle reads n_in frames, whatever the slice holds
        y, u, g = o.process_interleaved(x[pos * ch:(pos + n_in) * ch], cap, ratio, n_in=n_in)
        out.append((y, u, g))
        pos += u
    return out, o.state()


def _calls(n_in, ratio):
    """three chained calls over at most n_in frames: a third, a capacity-limited call, the rest of the input"""
    a, b = n_in // 3 + 1, n_in // 3
    return [(a, int(a * float(ratio)) + 20), (b, 7), (n_in - a - b, int(n_in * float(ratio)) + 20)]


def _dyadic_cases(golden_meta):
    # channels, taps, filters, lowpass, flags, ratio, calls, advance
    for c in golden_meta["small"]:
        yield ("golden " + c["name"], (c["channels"], c["taps"], c["filters"], c["lowpass"], c["flags"], f32(c["ratio"]),
                                       [(c["n_in"], c["cap"])], c["advance"]))
    for taps in (4, 8, 16, 32, 64, 128, 256, 512, 1024):
        yield f"T={taps}", (2, taps, 64, 1.0, 3, R48, _calls(700, R48), taps / 2)
    for filters in (2, 3, 16, 37, 256, 1024):
        yield f"F={filters}", (2, 64, filters, 1.0, 3, R44, _calls(700, R44), 32.0)
    for flags in range(8):
        for lp in (1.0, 0.7):
            yield f"flags={flags} lp={lp}", (3, 32, 16, lp, flags, f32(1.37), _calls(600, f32(1.37)), 16.0)
    for ratio in (0.21, 0.5, 0.61, 1.0, 1.37, 2.0, 3.0):
        for flags in (3, 2):
            r = f32(ratio)
            yield f"ratio={ratio} flags={flags}", (2, 64, 32, 1.0, flags, r, _calls(900, r), 32.0)
    yield "T=1024 lp=0.45 8 ch", (8, 1024, 256, 0.45, 1, f32(44100) / f32(96000), _calls(2500, f32(44100) / f32(96000)),
                                  512.0)
    yield "advance 0", (1, 64, 64, 1.0, 3, R48, _calls(500, R48), 0.0)
    yield "advance 77.25", (2, 64, 64, 1.0, 1, f32(2.0), _calls(500, f32(2.0)), 77.25)


def test_dyadic_products_are_exact(oracle, golden):
    """Every filter-bank entry of every geometry the dyadic checks use, times every 2^k of dyadic(), is a normal
    float32 (or 0): the products are exact, so a fused and an un-fused multiply-add round alike."""
    _, meta = golden
    kmin, kmax = DYADIC_K
    smallest = np.inf
    seen = set()
    for _, (ch, taps, filters, lp, flags, *_rest) in _dyadic_cases(meta):
        if (taps, filters, lp, flags) in seen:
            continue
        seen.add((taps, filters, lp, flags))
        bank = oracle.resampler(1, taps, filters, lp, flags).bank().astype(np.float64)
        nz = np.abs(bank[bank != 0])
        smallest = min(smallest, float(nz.min()))
        for k in range(kmin, kmax + 1):
            prod = nz * 2.0 ** k
            assert np.all(prod >= FLT_MIN), (taps, filters, lp, flags, k)
            assert np.array_equal(prod.astype(f32).astype(np.float64), prod)
    assert smallest * 2.0 ** kmin > 1e6 * FLT_MIN  # far above underflow (smallest tap ~3.9e-13)
    x = dyadic(5000, 2, stream=0)
    assert set(np.unique(np.abs(x[x != 0]))) == {f32(2.0 ** k) for k in range(kmin, kmax + 1)}
    assert np.any(np.signbit(x) & (x == 0)) and np.any(~np.signbit(x) & (x == 0))


def test_fused_equals_plain_on_dyadic_input(oracle, golden):
    """Fused and plain oracle on dyadic input: the same bytes, frame counts and final state, call by call."""
    _, meta = golden
    n_cases = 0
    for name, case in _dyadic_cases(meta):
        ch, calls = case[0], case[6]
        x = dyadic(sum(c[0] for c in calls), ch, stream=n_cases)
        plain, st_p = _chain(oracle, case, x, False)
        fused, st_f = _chain(oracle, case, x, True)
        assert st_p == st_f, name
        nonzero = 0
        for k, ((yp, up, gp), (yf, uf, gf)) in enumerate(zip(plain, fused)):
            assert (up, gp) == (uf, gf), (name, k)
            assert bits_equal(yp, yf), (name, k)
            nonzero += int(np.count_nonzero(yp))
        assert nonzero > 0, name
        n_cases += 1
    assert n_cases >= 50


# ---------------------------------------------------------------- generic input: fused != plain, within the bar
GENERIC = [  # channels, taps, filters, lowpass, flags, ratio
    (2, 256, 256, 1.0, 3, R48),
    (2, 1024, 256, 0.45, 3, f32(44100) / f32(96000)),
    (1, 32, 16, 1.0, 0, f32(1.37)),
    (3, 64, 1024, 0.7, 2, f32(0.61)),
    (2, 256, 256, 0.5, 2, f32(0.5)),  # whole-sample offsets with low-pass: the single-filter kind (phase 0)
]


def _signals(n, ch):
    for amp in (0.9, 1e-3):
        yield f"noise {amp}", noise(n, ch, stream=1, amp=amp)
        yield f"multitone {amp}", multitone(n, ch, 44100.0, stream=2, amp=amp)


def _one_call(oracle, geom, x, fused):
    ch, taps, filters, lp, flags, ratio = geom
    o = oracle.resampler(ch, taps, filters, lp, flags, fused=fused)
    o.advance(taps / 2)
    cap = int(x.size // ch * float(ratio)) + 40
    return o.process_interleaved(x, cap, ratio)


@pytest.mark.parametrize("geom", GENERIC)
def test_fused_differs_within_the_bar_on_generic_input(oracle, geom):
    """Noise and multitone at amplitude 0.9 and 1e-3: the fused chain changes some outputs (it is not the plain one),
    none by more than 1e-6, and the counts are the same."""
    ch = geom[0]
    for label, x in _signals(3000, ch):
        yp, up, gp = _one_call(oracle, geom, x, False)
        yf, uf, gf = _one_call(oracle, geom, x, True)
        assert (up, gp) == (uf, gf)
        assert np.any(yp != yf), (geom, label)
        assert float(np.max(np.abs(yp.astype(np.float64) - yf))) <= TOL, (geom, label)


def _model(geom, x):
    """float64 model of one call from a fresh context advanced by T/2, from the library's host-only filter bank and
    schedule: (value, forward-error bound) per output sample, interleaved."""
    import esp_audio_libs_b200 as espb
    ch, taps, filters, lp, flags, ratio = geom
    bank, eff = espb.plan_filter_bank(taps, filters, lp, flags)
    off = f32(f32(taps // 2) + f32(taps / 2))
    n_in = x.size // ch
    cap = int(n_in * float(ratio)) + 40
    s = espb.plan_schedule(taps, filters, eff, off, taps, n_in, cap, ratio)
    h = bank.astype(np.float64)
    xin = x.astype(np.float64).reshape(-1, ch)
    xpad = np.concatenate([np.zeros((taps, ch)), xin, np.zeros((taps, ch))])
    ws = s["ws"].astype(np.int64) + taps
    rows = ws[:, None] + np.arange(taps)[None, :]                     # (n, T)
    win = xpad[rows]                                                  # (n, T, ch)
    h1 = h[s["phase"]]
    h2 = h[np.minimum(s["phase"] + 1, filters)]
    s1 = np.einsum("nt,ntc->nc", h1, win)
    s2 = np.einsum("nt,ntc->nc", h2, win)
    a1 = np.einsum("nt,ntc->nc", np.abs(h1), np.abs(win))
    a2 = np.einsum("nt,ntc->nc", np.abs(h2), np.abs(win))
    kind = s["kind"][:, None]
    w = np.where(kind == 3, s["w"].astype(np.float64)[:, None], 0.0)
    u = 2.0 ** -24
    gamma = (taps + 3) * u / (1 - (taps + 3) * u)  # T roundings in the chain, up to three in the blend
    value = np.where(kind == 1, xpad[ws + taps // 2 - 1], (1 - w) * s1 + w * s2)
    bound = np.where(kind == 1, 0.0, gamma * ((1 - w) * a1 + w * a2))
    return value.reshape(-1), bound.reshape(-1), s["used"], s["generated"]


def test_both_oracles_within_forward_error_bound(oracle, record_property):
    """Plain and fused oracle against a float64 model of the same operation (the library's host-side bank and
    schedule, an exact-ish dot product): every output within gamma_{T+3} * ((1-w) sum|h_p x| + w sum|h_{p+1} x|) — the
    chain's T roundings and the blend's — and pass-through outputs exact.  The largest error / bound ratio is reported
    as the test property `worst_ratio`."""
    worst = {False: 0.0, True: 0.0}
    for geom in GENERIC:
        ch = geom[0]
        for label, x in _signals(2000, ch):
            value, bound, used, gen = _model(geom, x)
            for fused in (False, True):
                y, u, g = _one_call(oracle, geom, x, fused)
                assert (u, g) == (used, gen), (geom, fused)
                err = np.abs(y.astype(np.float64) - value)
                assert np.all(err <= bound), (geom, label, fused, float(np.max(err - bound)))
                nz = bound > 0
                if nz.any():
                    worst[fused] = max(worst[fused], float(np.max(err[nz] / bound[nz])))
    record_property("worst_ratio_plain", worst[False])
    record_property("worst_ratio_fused", worst[True])
    print(f"largest error / bound: plain {worst[False]:.3g}, fused {worst[True]:.3g}")
    assert 0 < worst[True] < 1 and 0 < worst[False] < 1


# ---------------------------------------------------------------- the switch
def test_fused_switch_is_per_context(oracle):
    """A fused and a plain context from the one session oracle, called in turn: each keeps its own arithmetic, and a
    context made without the argument is plain."""
    geom = GENERIC[0]
    ch, taps, filters, lp, flags, ratio = geom
    x = noise(1500, ch, stream=5, amp=0.9)
    ref_p = _one_call(oracle, geom, x, False)[0]
    ref_f = _one_call(oracle, geom, x, True)[0]
    assert not bits_equal(ref_p, ref_f)
    a = oracle.resampler(ch, taps, filters, lp, flags, fused=True)
    b = oracle.resampler(ch, taps, filters, lp, flags)
    a.advance(taps / 2)
    b.advance(taps / 2)
    ya, yb = [], []
    for lo, hi in ((0, 500), (500, 1500)):
        ya.append(a.process_interleaved(x[lo * ch:hi * ch], 2000, ratio)[0])
        yb.append(b.process_interleaved(x[lo * ch:hi * ch], 2000, ratio)[0])
    assert bits_equal(np.concatenate(ya), ref_f) and bits_equal(np.concatenate(yb), ref_p)
    # the wrapper's switch reaches its resampler; a plain wrapper stays plain
    pcm = (noise(2048, 2, stream=6, amp=0.5) * 32767).astype(np.int16).view(np.uint8)
    outs = {}
    for fused in (False, True):
        w = oracle.wrapper(2048 * 2, 2400 * 2, 44100.0, 48000.0, 16, 32, 2, True, True, 256, 256, fused=fused)
        outs[fused] = w.resample(pcm, 2048, 2400)[0]
    plain_again = oracle.wrapper(2048 * 2, 2400 * 2, 44100.0, 48000.0, 16, 32, 2, True, True, 256, 256)
    assert bits_equal(plain_again.resample(pcm, 2048, 2400)[0], outs[False])
    assert not bits_equal(outs[True], outs[False])


def test_reference_refuses_fused():
    """The compiled reference has no fused form: asking for one is an error, not a silent plain run."""
    ref = Reference.__new__(Reference)  # no library needed: the refusal comes first
    with pytest.raises(ValueError):
        ref.resampler(2, 64, 64, 1.0, 3, fused=True)
    with pytest.raises(ValueError):
        ref.wrapper(100, 100, 44100.0, 48000.0, 16, 16, 2, fused=True)

