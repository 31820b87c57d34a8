"""GPU: every stored fp16 tensor of the three models against the float64 per-layer restatement of tests/layer_ref.py.

Each layer is checked from the device's own inputs of that layer (taps of the audit path, `ar_model_audit_tap`), so the
check is as sharp with the suite's benign weights as with trained-like (BatchNorm-calibrated) ones, which the model-level
tests are not.  Both conv engines, both weight sets, shapes at the tile and pooling edges, and the three LSTM recurrence
kernels (selected by the batch: up to 2 sequences per SM `lstm_kernel<1, 8>`, up to 8 `lstm_mmaw_kernel<4>`, beyond
`lstm_mmaw_kernel<8>`; the audit runs layer by layer, so the scan reads stored pre-activations)."""
import pytest
import torch

from oracle.weights import calibrated_state_dicts, make_input
from ml_audio_restoration_b200 import _lib
import layer_ref as R
from gpu_util import audit_taps, make_model

pytestmark = pytest.mark.gpu

ENGINES = {"umma": _lib.ENGINE_UMMA, "simt": _lib.ENGINE_SIMT}
# The recurrence kernels: the tensor-core ones are checked teacher-forced (step t from the device's h_{t-1}), so every step
# is local and the common bound applies.  The CUDA-core kernel's fp32 h is not observable and the reference runs freely
# next to it, so its h is held to a looser magnitude slack.  Measured on a B200 (1000 W) over the shapes below, T <= 203:
# worst |dev - ref| / bound 0.30 with this slack, at most 0.45 % of the stored h differing from the rounded reference.
LSTM_FREE_SLACK = 2.0 ** -14


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


STEREO_B = {"3": lambda: 3, "2sm+8": lambda: 2 * sm_count() + 8, "8sm+13": lambda: 8 * sm_count() + 13}
SHAPES = ([("denoiser", str(B), T) for B, T in [(1, 8), (2, 127), (1, 129), (3, 1013), (150, 1100)]]
          + [("super_resolution", str(B), T) for B, T in [(3, 1), (2, 127), (1, 128), (1, 129), (2, 1000), (150, 1100)]]
          + [("stereo", b, T) for b, T in [("3", 203), ("2sm+8", 203), ("8sm+13", 203), ("3", 7), ("3", 130)]])


@pytest.fixture(scope="module")
def weight_sets(state_dicts):
    return {"benign": state_dicts, "calibrated": calibrated_state_dicts()}


def check_model(name, sd, engine, x, label):
    B, _, T = x.shape
    m = make_model(name, sd, ENGINES[engine], fusion=1)
    shapes = R.tap_shapes(name, B, T)
    if engine == "simt" and name == "denoiser":
        shapes.pop("td0")                       # the CUDA-core engine runs the whole transient detector in its tail kernel
    taps, y, audit = audit_taps(m, x.cuda(), shapes)
    assert set(audit) == set(shapes), f"audited tensors {sorted(audit)} != restated {sorted(shapes)}"
    picks = list(range(B)) if B <= 5 else sorted({0, 1, B // 2, B - 2, B - 1})
    S = {n: t[picks].double().cpu() for n, t in taps.items()}
    variant = R.lstm_variant_for(B, sm_count())
    P = R.Params(name, sd, rounding=True, engine=engine)
    stats = R.check_layers(name, P, x[picks], S, y[picks].double().cpu(), lstm_variant=variant,
                           lstm_slack=LSTM_FREE_SLACK if variant == "fp32" else None)
    print(f"{label} (lstm: {variant if name == 'stereo' else '-'})\n{R.report(stats)}")
    bad = [n for n, s in stats.items() if R.failed(s)]
    assert not bad, f"{label}: layers {bad} do not match the float64 restatement"


@pytest.mark.parametrize("weights", ["benign", "calibrated"])
@pytest.mark.parametrize("engine", ["umma", "simt"])
@pytest.mark.parametrize("name,B,T", SHAPES)
def test_every_layer_matches_float64_restatement(weight_sets, name, B, T, engine, weights):
    B = STEREO_B[B]() if name == "stereo" else int(B)
    x = make_input(B, T, seed=7 * B + T)
    check_model(name, weight_sets[weights][name], engine, x, f"{name}[{engine}, {weights}] B={B} T={T}")


def test_tap_window_larger_than_buffer_is_refused(state_dicts):
    """A tap whose buffer is smaller than the window fails the forward with AR_ERR_INVALID before anything is copied;
    with the audit off an armed tap is ignored and the forward is unchanged."""
    m = make_model("stereo", state_dicts["stereo"])
    x = make_input(2, 100, 3).cuda()
    L = _lib.lib()
    h = m.native_handle(x.device)
    small = torch.full((2 * 64 * 100 - 1,), float("nan"), device="cuda")
    with torch.no_grad():
        y0 = m(x)
        _lib.check(L.ar_model_audit_tap(h, b"lstm", small.data_ptr(), small.numel()))
        try:
            y1 = m(x)                                      # audit off: the tap does nothing
            torch.cuda.synchronize()
            assert torch.equal(y0, y1) and torch.isnan(small).all()
            with pytest.raises(RuntimeError, match="audit tap lstm"):
                m.audit(x)
            torch.cuda.synchronize()
            assert torch.isnan(small).all()
        finally:
            L.ar_model_audit_tap(h, None, None, 0)
    assert m.audit(x).keys() == R.tap_shapes("stereo", 2, 100).keys()
