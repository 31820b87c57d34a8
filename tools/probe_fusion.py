"""Times the denoiser / super-resolution forwards at a bench sub-batch with ar_set_fusion off and on
(0 layer by layer, 1 every fused chain that fits, the product default), CUDA events, median of 5.
   python tools/probe_fusion.py [B] [T]"""
import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.weights import make_state_dict, make_input
from ml_audio_restoration_b200 import _lib
from ml_audio_restoration_b200.models import AudioDenoiser, AudioSuperResolution, StereoSeparator
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1184
T = int(sys.argv[2]) if len(sys.argv) > 2 else 44100
L = _lib.lib()
for name, cls in (("denoiser", AudioDenoiser), ("super_resolution", lambda: AudioSuperResolution(upscale_factor=2)), ("stereo", StereoSeparator)):
    x = make_input(B if name != "stereo" else B // 4, T).cuda()
    outs = {}
    for level in (0, 1):
        _lib.check(L.ar_set_fusion(level))
        m = cls(); m.load_state_dict(make_state_dict(name)); m = m.cuda().eval()
        with torch.no_grad():
            y = m(x)
            ts = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); y = m(x); e1.record(); e1.synchronize()
                ts.append(e0.elapsed_time(e1))
        outs[level] = y
        print(f"{name:17s} B={x.shape[0]} T={T} fusion={level}: {sorted(ts)[2]:.3f} ms   max|y - y(level 0)| = {float((y - outs[0]).abs().max()):.2e}")
    del m
L.ar_set_fusion(1)
