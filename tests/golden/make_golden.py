"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU.

Needs a checkout of the original project (its `src/` package):
        python tests/golden/make_golden.py <original-project-dir>

What it pins
  * the oracle `state_dict` factory has exactly the reference key set / shapes
    (`load_state_dict(strict=True)` into the reference modules);
  * reference outputs of the three forwards on seeded inputs incl. edge lengths
    (T=8 minimum, odd lengths that hit the floor-pool/right-pad branch of denoiser.py:121);
  * `normalize_audio` incl. the rms==0 and the peak-limit branches;
  * the whole-file chain of inference.py:45-98 and a trainer.py:652-681 style
    non-overlapping chunk loop built from the reference modules.
The resulting files are small (inputs are regenerated from seeds, outputs are a few KB).
"""
import os
import sys
import types

import numpy as np
import torch

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
if len(sys.argv) != 2:
    sys.exit("usage: python tests/golden/make_golden.py <original-project-dir>")
sys.path.insert(0, os.path.abspath(sys.argv[1]))
sys.modules.setdefault("soundfile", types.ModuleType("soundfile"))  # audio_processing.py:3

from src.models.denoiser import AudioDenoiser                      # noqa: E402  (reference)
from src.models.super_resolution import AudioSuperResolution       # noqa: E402
from src.models.stereo_separator import StereoSeparator            # noqa: E402
from src.utils.audio_processing import normalize_audio as ref_normalize  # noqa: E402

from oracle.weights import make_state_dict, make_input, state_dict_checksum  # noqa: E402

torch.set_num_threads(8)
SEED = 1234


def build():
    den, sr, st = AudioDenoiser(), AudioSuperResolution(upscale_factor=2), StereoSeparator()
    sds = {n: make_state_dict(n, SEED) for n in ("denoiser", "super_resolution", "stereo")}
    den.load_state_dict(sds["denoiser"], strict=True)
    sr.load_state_dict(sds["super_resolution"], strict=True)
    st.load_state_dict(sds["stereo"], strict=True)
    return den.eval(), sr.eval(), st.eval(), sds


def main():
    den, sr, st, sds = build()
    out = {"seed": np.int64(SEED)}
    for n, sd in sds.items():
        out[f"checksum_{n}"] = np.float64(state_dict_checksum(sd))
    with torch.no_grad():
        for T in (8, 9, 101, 1037, 2048):
            x = make_input(2, T, SEED)
            out[f"denoiser_T{T}"] = den(x).numpy()
        for T in (4, 65, 1000):
            x = make_input(3, T, SEED)
            out[f"super_resolution_T{T}"] = sr(x).numpy()
        for T in (7, 130, 1500):
            x = make_input(2, T, SEED)
            out[f"stereo_T{T}"] = st(x).numpy()
        # normalize_audio branches (audio_processing.py:72, :84)
        a = make_input(1, 4000, SEED)[0]
        out["normalize_plain"] = ref_normalize(a).numpy()
        out["normalize_silence"] = ref_normalize(torch.zeros(1, 100)).numpy()
        spiky = a.clone() * 0.01
        spiky[0, 17] = 5.0
        out["normalize_peak"] = ref_normalize(spiky).numpy()
        stereo_in = make_input(2, 3000, SEED)[:, 0]
        out["normalize_stereo"] = ref_normalize(stereo_in).numpy()
        # whole-file chain, inference.py:45-98 (tensor part)
        audio = make_input(1, 3001, SEED + 1, scale=0.3)[0]            # [1,N]
        a = ref_normalize(audio)
        d = den(a.unsqueeze(0)).squeeze(0)
        e = sr(d.unsqueeze(0)).squeeze(0)
        s = st(e.unsqueeze(0)).squeeze(0)
        out["chain_whole"] = ref_normalize(s).numpy()
        s1 = st(d.unsqueeze(0)).squeeze(0)
        out["chain_whole_nosr"] = ref_normalize(s1).numpy()
        # trainer.py:652-681 style loop (non-overlapping chunks, zero-padded tail), full chain per chunk
        chunk = 1000
        pieces = []
        for i in range(0, audio.shape[1], chunk):
            c = audio[:, i:i + chunk]
            valid = c.shape[1]
            if valid < chunk:
                c = torch.nn.functional.pad(c, (0, chunk - valid))
            y = st(sr(den(c.unsqueeze(0)))).squeeze(0)
            pieces.append(y[:, :2 * valid])
        out["chain_trainer_chunks"] = torch.cat(pieces, dim=1).numpy()

    np.savez_compressed(os.path.join(HERE, "golden_v1.npz"), **out)
    print("wrote golden_v1.npz:", {k: getattr(v, "shape", None) for k, v in out.items()})

    # Wiring anchors of SURVEY.md App. G (default init, torch RNG) -- printed, not stored.
    torch.manual_seed(0)
    m = AudioDenoiser().eval()
    g = torch.Generator().manual_seed(1234)
    x = 0.1 * torch.randn(2, 1, 44100, generator=g)
    with torch.no_grad():
        y = m(x)
    print("App.G denoiser anchor: x.sum=%.6f y.sum=%.6f (survey: +21.681887 / +773.360566)"
          % (x.double().sum(), y.double().sum()))


if __name__ == "__main__":
    main()
