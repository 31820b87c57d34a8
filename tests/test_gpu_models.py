"""GPU: the three drop-in modules against the CPU oracle and the reference's golden vectors."""
import ctypes as C

import pytest
import torch

import oracle
from oracle.weights import make_input
from ml_audio_restoration_b200 import _lib
from gpu_util import make_model, assert_close

pytestmark = pytest.mark.gpu

FWD = {"denoiser": oracle.denoiser_forward, "super_resolution": oracle.super_resolution_forward,
       "stereo": oracle.stereo_forward}
GOLDEN = {"denoiser": (2, [8, 9, 101, 1037, 2048]), "super_resolution": (3, [4, 65, 1000]), "stereo": (2, [7, 130, 1500])}
ENGINES = {"simt": _lib.ENGINE_SIMT, "umma": _lib.ENGINE_UMMA}


@pytest.fixture(scope="module")
def models(state_dicts):
    cache = {}

    def get(name, engine):
        if (name, engine) not in cache:
            cache[(name, engine)] = make_model(name, state_dicts[name], ENGINES[engine])
        return cache[(name, engine)]
    return get


@pytest.mark.parametrize("engine", ["simt", "umma"])
@pytest.mark.parametrize("name", ["denoiser", "super_resolution", "stereo"])
def test_model_matches_reference_golden(models, golden, name, engine):
    B, lengths = GOLDEN[name]
    m = models(name, engine)
    for T in lengths:
        x = make_input(B, T)
        with torch.no_grad():
            y = m(x.cuda())
        assert_close(torch.from_numpy(golden[f"{name}_T{T}"]), y, f"{name}[{engine}] T={T} vs reference golden")


@pytest.mark.parametrize("engine", ["simt", "umma"])
@pytest.mark.parametrize("name,B,T", [("denoiser", 2, 44100), ("super_resolution", 16, 44100), ("stereo", 4, 44100)])
def test_model_baseline_config_vs_oracle(models, state_dicts, name, B, T, engine):
    """BASELINE.json configs 1-3 at full size."""
    if engine == "simt" and name != "denoiser":
        B = 2  # the CUDA-core engine is a cross-check, keep it short
    x = make_input(B, T)
    ref = FWD[name](state_dicts[name], x)
    with torch.no_grad():
        y = models(name, engine)(x.cuda())
    assert_close(ref, y, f"{name}[{engine}] B={B} T={T} vs oracle")


@pytest.mark.parametrize("T", [44096, 44101, 127, 128, 129, 255, 257])
def test_ragged_lengths(models, state_dicts, T):
    for name in ("denoiser", "super_resolution", "stereo"):
        x = make_input(1, T, seed=T)
        ref = FWD[name](state_dicts[name], x)
        with torch.no_grad():
            y = models(name, "umma")(x.cuda())
        assert_close(ref, y, f"{name} T={T}")


def test_impulse_and_silence_inputs(models, state_dicts):
    x = make_input(2, 4000)
    x[0, 0, 1000] = 0.9          # a pop (impulse-mask branch, denoiser.py:62-86)
    x[0, 0, 1001] = -0.8
    x[1] = 0.0                   # digital silence
    for name in ("denoiser", "super_resolution", "stereo"):
        ref = FWD[name](state_dicts[name], x)
        with torch.no_grad():
            y = models(name, "umma")(x.cuda())
        assert_close(ref, y, f"{name} impulse/silence", min_snr=None if name == "denoiser" else 60.0)


def test_noncontiguous_input_is_accepted(models, state_dicts):
    x = make_input(2, 2 * 1000)[:, :, ::2]   # stereo_separator.py:93 makes inputs contiguous
    ref = oracle.stereo_forward(state_dicts["stereo"], x.contiguous())
    with torch.no_grad():
        y = models("stereo", "umma")(x.cuda())
    assert_close(ref, y, "stereo non-contiguous")


def test_stereo_large_batch_tensor_core_lstm(models, state_dicts):
    """More than two sequences per SM switches the recurrence to the tensor-core (mma.sync fp16) kernel;
    ragged length (not a multiple of the 8-step block) and a batch that is not a multiple of 8."""
    m = models("stereo", "umma")
    x = make_input(301, 203, seed=11)
    ref, (hn, cn) = oracle.stereo_forward(state_dicts["stereo"], x, return_state=True)
    with torch.no_grad():
        y, st = m.forward_with_state(x.cuda())
    assert_close(ref, y, "stereo B=301 T=203 (tensor-core LSTM)")
    assert_close(hn[0], st[:, 0], "carried h (tensor-core LSTM)", max_abs=1e-3, min_snr=50.0)
    assert_close(cn[0], st[:, 1], "carried c (tensor-core LSTM)", max_abs=1e-3, min_snr=50.0)


@pytest.fixture(scope="module")
def weight_sets(state_dicts):
    from oracle.weights import calibrated_state_dicts
    return {"benign": state_dicts, "calibrated": calibrated_state_dicts()}


def assert_fused_equals_layer_by_layer(yp, yf, what):
    """DESIGN.md: a fused launch computes the same fp16 intermediates, in the same accumulation order, as its layers."""
    diff = float((yf - yp).abs().max())
    print(f"{what}: max|diff|={diff:.3e}  bitwise equal: {torch.equal(yf, yp)}")
    assert torch.equal(yf, yp), f"{what}: fused launches differ from layer by layer (max|diff| {diff:.3e})"


@pytest.mark.parametrize("weights", ["benign", "calibrated"])
@pytest.mark.parametrize("B,T", [(1, 100), (3, 129), (2, 1500), (5, 4099), (160, 1000)])
def test_fused_chains_match_layer_by_layer(weight_sets, B, T, weights):
    """The fused dilated-block launches (conv k3 -> conv k1 [-> LSTM input projection], conv_chain.cu) compute the
    same fp16-rounded intermediates as the layer-by-layer launches: bitwise equal outputs, and both agree with the oracle
    (benign weights; with calibrated ones the layer-by-layer path is pinned layer by layer, test_gpu_layers.py).
    B=160 gives every SM pair several tile pairs (steady-state pipeline)."""
    sd = weight_sets[weights]["stereo"]
    fused = make_model("stereo", sd, fusion=True)
    plain = make_model("stereo", sd, fusion=False)
    x = make_input(B, T, seed=B * 7 + T)
    with torch.no_grad():
        yf = fused(x.cuda())
        yp = plain(x.cuda())
    assert_fused_equals_layer_by_layer(yp, yf, f"stereo[{weights}] fused vs layer-by-layer B={B} T={T}")
    if B <= 5 and weights == "benign":
        assert_close(oracle.stereo_forward(sd, x), yf, f"stereo fused vs oracle B={B} T={T}")


@pytest.mark.parametrize("weights", ["benign", "calibrated"])
@pytest.mark.parametrize("name", ["denoiser", "super_resolution"])
@pytest.mark.parametrize("B,T", [(1, 8), (2, 125), (1, 126), (3, 127), (1, 252), (2, 253), (1, 1009), (5, 4099), (150, 1100)])
def test_fused_double_convs_match_layer_by_layer(weight_sets, name, B, T, weights):
    """The fused k3 -> k3 launches (U-Net double convs with the max-pool copy, super-resolution residual blocks with the
    skip add; conv_chain.cu, tile stride 126) compute the same fp16-rounded intermediates as the layer-by-layer launches.
    Lengths around the 126-row tile stride and its multiples (at every U-Net level: T, T/2, T/4), odd tile counts (idle peer
    CTA), and B=150 for the steady-state pipeline.  The denoiser is bitwise equal.  The super-resolution output head is
    the one fused path that legitimately differs: fused behind hf_emphasis it runs on the tensor core, layer by layer on
    CUDA cores (`final_k7`) -- same fp16 operands, another fp32 summation order -- so the fused output is held to the
    float64 head restatement of tests/layer_ref.py on the tapped hf_emphasis output of the layer-by-layer path, on every
    item of the batch, and (benign weights) to the layer-by-layer output within 2e-5 and 90 dB."""
    sd = weight_sets[weights][name]
    fused = make_model(name, sd, fusion=2)      # every pair that fits, not only the measured-faster ones
    plain = make_model(name, sd, fusion=0)
    x = make_input(B, T, seed=B * 11 + T)
    with torch.no_grad():
        yf = fused(x.cuda())
        yp = plain(x.cuda())
    what = f"{name}[{weights}] fused vs layer-by-layer B={B} T={T}"
    if name == "denoiser":
        assert_fused_equals_layer_by_layer(yp, yf, what)
    else:
        import layer_ref as R
        from gpu_util import audit_taps
        taps, yt, _ = audit_taps(plain, x.cuda(), {"hf": (32, 2 * T)})
        assert torch.equal(yt, yp), "the audited forward differs from the plain layer-by-layer forward"
        head = R.layers(name, R.Params(name, sd), T)[-1][1]
        val = head({"hf": taps["hf"].double().cpu()}, x.double(), {})          # every item of the batch
        st = R.compare(yf.double().cpu(), val, R.TAIL_SLACK)
        print(f"{what}: bitwise equal: {torch.equal(yf, yp)}; fused head vs float64 restatement: worst |dev-ref|/bound "
              f"{st['ratio']:.3g}, differing {100 * st['frac']:.2f} %")
        assert st["ratio"] <= 1.0 and st["nonfinite"] == 0
        if weights == "benign":
            assert_close(yp, yf, what, max_abs=2e-5, min_snr=90.0)
    if B <= 5 and weights == "benign":
        assert_close(FWD[name](sd, x), yf, f"{name} fused vs oracle B={B} T={T}")


def test_error_behaviour(models, state_dicts):
    den = models("denoiser", "umma")
    with pytest.raises(RuntimeError):          # reference: RuntimeError from max_pool1d for T < 8
        den(make_input(1, 7).cuda())
    with pytest.raises(RuntimeError):          # no CPU fallback
        den(make_input(1, 64))
    with pytest.raises(RuntimeError):
        den(make_input(1, 64).cuda().squeeze(1))
    for name, shape in (("denoiser", (0, 1, 64)), ("super_resolution", (0, 1, 128)), ("stereo", (0, 2, 64))):
        y = models(name, "umma")(torch.zeros(0, 1, 64, device="cuda"))      # reference: an empty batch gives an empty output
        assert tuple(y.shape) == shape and y.is_cuda and y.dtype == torch.float32
    den.train()
    with pytest.raises(NotImplementedError):
        den(make_input(1, 64).cuda())
    den.eval()
    from ml_audio_restoration_b200.models import AudioDenoiser
    bad = dict(state_dicts["denoiser"])
    bad.pop("final_conv.bias")
    with pytest.raises(RuntimeError):          # load_state_dict(strict) semantics
        AudioDenoiser().load_state_dict(bad)


def test_weight_update_repacks(state_dicts):
    m = make_model("super_resolution", state_dicts["super_resolution"])
    x = make_input(1, 500).cuda()
    with torch.no_grad():
        y0 = m(x)
        m.reconstruction.bias.add_(0.25)
        y1 = m(x)
    assert_close(y0.cpu() + 0.25, y1, "bias update visible after repack", max_abs=1e-6, min_snr=None)


@pytest.mark.parametrize("name,B,T", [("denoiser", 2, 44100), ("super_resolution", 3, 5000), ("stereo", 4, 4100)])
def test_cuda_graph_capture_replays_the_forward(models, name, B, T):
    """`module.capture(x)`: the forward's launch train captured into a CUDA graph (BASELINE configs 1-3 are launch-bound at
    their small batches); replays on new inputs give exactly what the eager forward gives."""
    m = models(name, "umma")
    xs = [make_input(B, T, seed=50 + i).cuda() for i in range(3)]
    with torch.no_grad():
        g = m.capture(xs[0])
        for x in xs:
            want = m(x)
            got = g(x).clone()
            assert torch.equal(want, got)
    with pytest.raises(RuntimeError):
        g(make_input(B, T + 8).cuda())


# ------------------------------------------------------------------------------------------------ workspace contents
# DESIGN.md section 2: rows outside [0, T) of a stored tensor are never written and consumers zero them in shared memory.
# Module forwards get `torch.empty` scratch, which mostly holds zeros or the previous identical forward's values, so the
# tests above cannot see a kernel that reads what nobody wrote.  These call the C ABI with a caller-owned workspace (and
# output) filled with 0x00, 0xFF (NaN in fp16 and fp32) and 0x7B (large finite values: a max-pool or an audit maximum
# would silently drop a NaN, not a 6e4): outputs must be finite and bitwise equal across the three fills.
FILLS = (0x00, 0xFF, 0x7B)


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _run_filled(call, need, y):
    """call(ws_ptr, ws_bytes) once per fill of workspace and output; returns the outputs."""
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    outs = []
    for fill in FILLS:
        ws.fill_(fill)
        y.view(torch.uint8).fill_(fill)
        _lib.check(call(ws.data_ptr(), ws.numel()))
        torch.cuda.synchronize()
        outs.append(y.clone())
    return outs


def _assert_fill_independent(outs, what):
    for fill, o in zip(FILLS, outs):
        assert torch.isfinite(o).all(), f"{what}: non-finite output with workspace fill 0x{fill:02X}"
    for fill, o in zip(FILLS[1:], outs[1:]):
        diff = float((o - outs[0]).abs().max())
        assert torch.equal(o, outs[0]), f"{what}: output with fill 0x{fill:02X} differs from fill 0x00 (max|diff| {diff:.3e})"


def _forward_filled(m, x, out_shape, audit=False, window=None):
    L = _lib.lib()
    B, _, T = x.shape
    h = m.native_handle(x.device)
    if audit:                                  # the audited forward runs layer by layer: its workspace is larger
        _lib.check(L.ar_model_audit_enable(h, 1))
    need = C.c_size_t()
    _lib.check(L.ar_model_workspace_bytes(h, B, T, C.byref(need)))
    y = torch.empty(out_shape, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    if window is None:
        call = lambda ws, n: L.ar_model_forward(h, x.data_ptr(), y.data_ptr(), B, T, ws, n, stream)
    else:
        lstm_start, state_pos, st_in, st_out = window
        call = lambda ws, n: L.ar_stereo_forward_window(h, x.data_ptr(), y.data_ptr(), B, T, lstm_start, state_pos,
                                                        st_in.data_ptr(), st_out.data_ptr(), ws, n, stream)
    try:
        return _run_filled(call, need.value, y)
    finally:
        if audit:
            L.ar_model_audit_enable(h, 0)


OUT = {"denoiser": lambda B, T: (B, 1, T), "super_resolution": lambda B, T: (B, 1, 2 * T), "stereo": lambda B, T: (B, 2, T)}


@pytest.mark.parametrize("mode", ["fusion0", "fusion1", "fusion2", "audit"])
@pytest.mark.parametrize("name", ["denoiser", "super_resolution", "stereo"])
def test_forwards_ignore_workspace_contents(state_dicts, name, mode):
    fusion = {"fusion0": 0, "fusion1": 1, "fusion2": 2, "audit": 1}[mode]
    m = make_model(name, state_dicts[name], fusion=fusion)
    batches = [2] if name != "stereo" else [3, 2 * _sm_count() + 8, 8 * _sm_count() + 13]
    for B in batches:
        for T in (8, 127, 1013):
            x = make_input(B, T, seed=B + T).cuda()
            outs = _forward_filled(m, x, OUT[name](B, T), audit=mode == "audit")
            _assert_fill_independent(outs, f"{name} {mode} B={B} T={T}")
    if name == "stereo":                       # a window: scan started inside the segment, state taken at an interior step
        B, T = 3, 1013
        x = make_input(B, T, seed=5).cuda()
        st_in = torch.randn(B, 2, 64, device="cuda") * 0.3
        st_out = torch.empty(B, 2, 64, device="cuda")
        outs = _forward_filled(m, x, (B, 2, T), audit=mode == "audit", window=(16, 504, st_in, st_out))
        _assert_fill_independent(outs, f"stereo window {mode}")


def test_chain_ignores_workspace_contents(state_dicts):
    """The chain beyond 8 chunks per SM: sub-batched conv phases around one scan that computes its own input projection."""
    from ml_audio_restoration_b200 import RestorationPipeline
    pipe = RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                state_dicts["stereo"], "cuda")
    B, T = 8 * _sm_count() + 13, 1037
    x = make_input(B, T, seed=9).cuda()
    L = _lib.lib()
    ch = pipe.chain()
    need = C.c_size_t()
    _lib.check(L.ar_chain_workspace_bytes(ch, B, T, C.byref(need)))
    y = torch.empty(B, 2, 2 * T, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    outs = _run_filled(lambda ws, n: L.ar_chain_forward(ch, x.data_ptr(), y.data_ptr(), B, T, ws, n, stream), need.value, y)
    _assert_fill_independent(outs, f"chain B={B} T={T}")
