"""Dump the pipeline trace of the fused-chain kernels (ar_debug_chain_trace) for one stereo forward.

Usage (on a B200):  python tools/chain_trace.py [B] [T]  ->  per launch, per tile pair: cycles between events.
Events: see the slot list above trace_ev() in csrc/conv_chain.cu.
"""
import sys
import os

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ml_audio_restoration_b200 import _lib  # noqa: E402
from ml_audio_restoration_b200.models import StereoSeparator, AudioSuperResolution, AudioDenoiser  # noqa: E402


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 148
    T = int(sys.argv[2]) if len(sys.argv) > 2 else 44100
    which = sys.argv[3] if len(sys.argv) > 3 else "stereo"
    fusion = int(sys.argv[4]) if len(sys.argv) > 4 else 1      # 0: layer by layer (nothing to trace)
    _lib.check(_lib.lib().ar_set_fusion(fusion))
    torch.manual_seed(0)
    m = {"stereo": StereoSeparator, "sr": lambda: AudioSuperResolution(upscale_factor=2), "denoiser": AudioDenoiser}[which]().cuda().eval()
    x = 0.1 * torch.randn(B, 1, T, device="cuda")
    with torch.no_grad():
        m(x)
    buf = torch.zeros(8 * 1024, dtype=torch.int64, device="cuda")
    L = _lib.lib()
    L.ar_debug_chain_trace(buf.data_ptr())
    with torch.no_grad():
        m(x)
    torch.cuda.synchronize()
    L.ar_debug_chain_trace(None)
    tr = buf.cpu().view(8, 64, 1, 16)
    names = ["G1i0", "G1i1", "G2rdy", "G2i", "E1b", "E1e", "ELb", "ELe", "full0", "fullN", "G3rdy", "G3i", "E2b", "E2e", "Pend", "Pbeg"]
    for k in range(8):
        t = tr[k]
        if int(t.max()) == 0:
            continue
        base = int(t[t > 0].min())
        print(f"--- chain launch {k}: leader CTA events (cycles since first event), then per-tile deltas")
        print("tile " + " ".join(f"{n:>7s}" for n in names))
        for it in range(8, 24):
            row = [int(v) - base if int(v) else -1 for v in t[it, 0]]
            print(f"{it:4d} " + " ".join(f"{v:7d}" for v in row))
        per = (int(t[40, 0, 0]) - int(t[8, 0, 0])) / 32.0
        print(f"period (G1 issue to G1 issue, tiles 8..40): {per:.0f} cycles")


if __name__ == "__main__":
    main()
