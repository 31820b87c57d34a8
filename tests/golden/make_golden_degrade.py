"""Golden vectors for the degradation generator, produced by the UNMODIFIED reference function
(`simulate_vinyl_artifacts`, src/utils/audio_processing.py:122-226 of the original project):

    python tests/golden/make_golden_degrade.py <original-project-dir>      ->  tests/golden/golden_degrade_v1.npz

`soundfile` (imported at audio_processing.py:3, not installed here) is stubbed; nothing else is touched.  Inputs are
regenerated from the seeds stored in the file; both global generators the reference uses are seeded per case
(`np.random.seed(seed)`, `torch.manual_seed(seed)`)."""
import os
import sys
import types

import numpy as np
import torch

# (seed, channels, samples, sample_rate, kwargs)
CASES = [
    (11, 1, 4410, 22050, {}),
    (12, 2, 6000, 22050, {"impulse_rate": 40.0}),
    (13, 1, 3000, 44100, {"add_rumble": False}),
    (14, 1, 2205, 22050, {"add_rolloff": False, "impulse_rate": 200.0}),
    (15, 2, 500, 22050, {"impulse_rate": 300.0, "impulse_amplitude": (0.2, 0.9)}),
    (16, 1, 16, 22050, {"impulse_rate": 5000.0}),          # shortest length filtfilt accepts (> padlen 15)
]


def make_input(seed, C, N):
    return (0.1 * np.random.default_rng(seed).standard_normal((C, N))).astype(np.float32)


def main():
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_golden_degrade.py <original-project-dir>")
    sys.modules.setdefault("soundfile", types.ModuleType("soundfile"))
    sys.path.insert(0, os.path.abspath(sys.argv[1]))
    from src.utils.audio_processing import simulate_vinyl_artifacts
    import scipy
    out = {"scipy_version": np.array(scipy.__version__), "n_cases": np.array(len(CASES))}
    for i, (seed, C, N, sr, kw) in enumerate(CASES):
        np.random.seed(seed)
        torch.manual_seed(seed)
        y = simulate_vinyl_artifacts(torch.from_numpy(make_input(seed, C, N)), sr, **kw)
        out[f"case{i}_y"] = y.numpy()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_degrade_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
