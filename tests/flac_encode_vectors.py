"""Inputs of the FLAC encoder tests: integer contents that exercise each choice of `encode_search` (tests/flac_encode_ref.py) (silence,
DC, a linear ramp, a sine, noise, a full-scale clipped square, content with wasted bits) and a sweep over channel counts,
bit depths, lengths around the block size and block sizes."""
import numpy as np

KINDS = ("silence", "dc", "ramp", "sine", "noise", "square", "wasted")
LENGTHS = (1, 15, 16, 4095, 4096, 4097, 3 * 4096 + 5)
BLOCKS = (16, 192, 4096, 4608)


def content(kind: str, n: int, channels: int, bps: int, seed: int = 0) -> np.ndarray:
    """[n, channels] integers within bps bits."""
    rng = np.random.default_rng(seed)
    lim = 1 << (bps - 1)
    t = np.arange(n)[:, None] + 37 * np.arange(channels)[None, :]
    if kind == "silence":
        x = np.zeros((n, channels))
    elif kind == "dc":
        x = np.full((n, channels), -lim // 3) + np.arange(channels)[None, :]
    elif kind == "ramp":
        x = (t * 7 - lim // 2) % (2 * lim) - lim
    elif kind == "sine":
        x = np.round(0.6 * lim * np.sin(t * 0.013))
    elif kind == "noise":
        x = rng.integers(-lim // 64, lim // 64, (n, channels))
    elif kind == "square":
        x = np.where((t // 50) % 2 == 0, lim - 1, -lim)
    elif kind == "wasted":
        x = np.round(0.4 * lim * np.sin(t * 0.021) / 32) * 32 + rng.integers(-4, 4, (n, channels)) * 32
    else:
        raise ValueError(kind)
    return np.clip(x, -lim, lim - 1).astype(np.int64)


def sweep():
    """(id, samples [N, C], bps, block size): every length x block size with content, channels and depth cycling, and
    every content at both depths on mono, stereo and three channels."""
    cases = []
    i = 0
    for n in LENGTHS:
        for bs in BLOCKS:
            kind, c, bps = KINDS[i % len(KINDS)], 1 + i % 3, (16, 24)[(i // 3) % 2]
            cases.append((f"n{n}_bs{bs}_{kind}_c{c}_{bps}", content(kind, n, c, bps, seed=i), bps, bs))
            i += 1
    for kind in KINDS:
        for bps in (16, 24):
            for c in (1, 2, 3):
                cases.append((f"{kind}_c{c}_{bps}", content(kind, 3000 + 17 * c, c, bps, seed=i), bps, 1024))
                i += 1
    return cases
