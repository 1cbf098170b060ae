"""Synthetic test / bench signals (SURVEY.md §8d): deterministic, seeded by the stream index.  Pure numpy — nothing
here touches the oracle or the product."""
import numpy as np


def multitone(n_frames, channels, fs, stream=0, amp=0.5):
    """x[n,c] = A/8 * sum_{t=1..8} sin(2*pi*(997 t + 131 c + 7 s) n / fs + t), float32 interleaved."""
    n = np.arange(n_frames, dtype=np.float64)[:, None]
    c = np.arange(channels, dtype=np.float64)[None, :]
    acc = np.zeros((n_frames, channels), np.float64)
    for t in range(1, 9):
        acc += np.sin(2.0 * np.pi * (997.0 * t + 131.0 * c + 7.0 * stream) * n / fs + t)
    return (acc * (amp / 8.0)).astype(np.float32).reshape(-1)


def noise(n_frames, channels, stream=0, amp=0.5):
    """uniform in [-A, A], seeded by 0xC0FFEE ^ stream, float32 interleaved."""
    rng = np.random.default_rng(0xC0FFEE ^ (stream * 7919 + 1))
    return ((rng.random(n_frames * channels) * 2.0 - 1.0) * amp).astype(np.float32)


def from_recipe(r):
    """The signal a recipe names: {"signal": "multitone" | "noise", "frames", "channels", "stream", "amp"[, "fs"]}."""
    if r["signal"] == "multitone":
        return multitone(r["frames"], r["channels"], r["fs"], stream=r["stream"], amp=r["amp"])
    return noise(r["frames"], r["channels"], stream=r["stream"], amp=r["amp"])
