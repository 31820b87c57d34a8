"""Helpers for the -m gpu parity tests (everything goes through the C-ABI library)."""
import ctypes as C

import torch

from ml_audio_restoration_b200 import _lib
from ml_audio_restoration_b200.models import AudioDenoiser, AudioSuperResolution, StereoSeparator

CLS = {"denoiser": AudioDenoiser, "super_resolution": AudioSuperResolution, "stereo": StereoSeparator}
MAX_ABS = 1e-3      # north_star tolerance: max abs error <= 1e-3 ...
MIN_SNR_DB = 60.0   # ... or >= 60 dB SNR; the tests demand both unless stated


def make_model(name, sd, engine=_lib.ENGINE_UMMA, device="cuda", fusion=1):
    """fusion: 0 layer by layer, 1 / True the product default, 2 every fused chain that fits (ar_set_fusion)."""
    m = CLS[name]()
    m.load_state_dict(sd, strict=True)
    m = m.to(device).eval()
    L = _lib.lib()
    _lib.check(L.ar_set_conv_engine(engine))
    _lib.check(L.ar_set_fusion(int(fusion)))
    try:
        m.native_handle(torch.device("cuda", torch.cuda.current_device()))
    finally:
        L.ar_set_conv_engine(_lib.ENGINE_UMMA)
        L.ar_set_fusion(1)
    return m


def snr_db(ref, got):
    ref = ref.double().cpu()
    got = got.double().cpu()
    den = ((ref - got) ** 2).sum()
    if den == 0:
        return float("inf")
    return float(10 * torch.log10((ref ** 2).sum() / den))


def assert_close(ref, got, what, max_abs=MAX_ABS, min_snr=MIN_SNR_DB):
    ref = ref.cpu()
    got = got.cpu()
    assert ref.shape == got.shape, f"{what}: shape {tuple(got.shape)} != {tuple(ref.shape)}"
    assert torch.isfinite(got).all(), f"{what}: non-finite output"
    err = float((ref - got).abs().max())
    snr = snr_db(ref, got)
    print(f"{what}: max|err|={err:.3e} snr={snr:.1f} dB")
    assert err <= max_abs, f"{what}: max abs err {err:.3e} > {max_abs}"
    if min_snr is not None:
        assert snr >= min_snr, f"{what}: SNR {snr:.1f} dB < {min_snr}"


def debug_conv(x, w, b, dilation=1, lrelu=0, engine=_lib.ENGINE_UMMA):
    B, Cin, T = x.shape
    Cout, _, k = w.shape
    y = torch.empty(B, Cout, T, device="cuda")
    wc = w.detach().cpu().contiguous()
    bc = b.detach().cpu().contiguous()
    xc = x.cuda().contiguous()
    _lib.check(_lib.lib().ar_debug_conv1d(xc.data_ptr(), wc.data_ptr(), bc.data_ptr(), y.data_ptr(), B, Cin, Cout, T, k,
                                          dilation, lrelu, engine, torch.cuda.current_stream().cuda_stream))
    return y.cpu()


def audit_taps(module, x, shapes):
    """Run `module`'s forward on x under the dynamic-range audit (layer by layer) with every tensor of `shapes`
    ({name: (channels, length)}) tapped through `ar_model_audit_tap`.  Returns ({name: fp32 [B, C, T] device tensor}, y,
    {name: max |value|}).  Tap buffers start as NaN, so a window the forward did not copy in full cannot pass a check."""
    x = module._check_input(x)
    B = x.shape[0]
    L = _lib.lib()
    taps = {n: torch.full((B, c, t), float("nan"), device=x.device) for n, (c, t) in shapes.items()}
    with torch.cuda.device(x.device):
        h = module.native_handle(x.device)
        for n, buf in taps.items():
            _lib.check(L.ar_model_audit_tap(h, n.encode(), buf.data_ptr(), buf.numel()))
        _lib.check(L.ar_model_audit_enable(h, 1))
        try:
            y = module.forward(x)
            vals = (C.c_float * _lib.AUDIT_MAX_LAYERS)()
            n = C.c_int()
            _lib.check(L.ar_model_audit_read(h, vals, _lib.AUDIT_MAX_LAYERS, C.byref(n)))
            audit = {L.ar_model_audit_name(h, i).decode(): float(vals[i]) for i in range(n.value)}
        finally:
            L.ar_model_audit_enable(h, 0)
            L.ar_model_audit_tap(h, None, None, 0)
    return taps, y, audit
