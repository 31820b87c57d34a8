"""Two forwards of one model (target of ncu captures).   python tools/probe_forward.py stereo|sr|denoiser [B] [T] [fusion 0|1]"""
import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.weights import make_state_dict, make_input
from ml_audio_restoration_b200 import _lib
from ml_audio_restoration_b200.models import StereoSeparator, AudioSuperResolution, AudioDenoiser
which = sys.argv[1] if len(sys.argv) > 1 else "stereo"
B, T = int(sys.argv[2]) if len(sys.argv) > 2 else 148, int(sys.argv[3]) if len(sys.argv) > 3 else 44100
_lib.check(_lib.lib().ar_set_fusion(int(sys.argv[4]) if len(sys.argv) > 4 else 1))
name, cls = {"stereo": ("stereo", StereoSeparator), "sr": ("super_resolution", lambda: AudioSuperResolution(upscale_factor=2)),
             "denoiser": ("denoiser", AudioDenoiser)}[which]
m = cls(); m.load_state_dict(make_state_dict(name)); m = m.cuda().eval()
x = make_input(B, T).cuda()
with torch.no_grad():
    for _ in range(2):
        y = m(x)
torch.cuda.synchronize()
print("ok", tuple(y.shape))
