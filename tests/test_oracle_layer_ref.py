"""CPU: the per-layer float64 restatement (tests/layer_ref.py) is the reference network, and its per-layer metric catches
the indexing and packing mistakes that the model-level tolerance misses with the suite's seeded weights."""
import pytest
import torch

import oracle
from oracle.weights import calibrated_state_dicts, make_input, make_state_dict
import layer_ref as R

FWD = {"denoiser": oracle.denoiser_forward, "super_resolution": oracle.super_resolution_forward,
       "stereo": oracle.stereo_forward}
MAX_ABS, MIN_SNR_DB = 1e-3, 60.0          # the model-level tolerance of the GPU parity tests


@pytest.fixture(scope="module")
def weight_sets():
    return {"benign": {n: make_state_dict(n, 1234) for n in oracle.MODEL_NAMES}, "calibrated": calibrated_state_dicts()}


@pytest.mark.parametrize("weights", ["benign", "calibrated"])
@pytest.mark.parametrize("name,T", [("denoiser", 1013), ("super_resolution", 129), ("stereo", 203)])
def test_restatement_without_rounding_is_the_oracle_network(weight_sets, name, T, weights):
    """Chained with rounding off, the per-layer functions reproduce the oracle forward in float64."""
    sd = weight_sets[weights][name]
    x = make_input(2, T, 5)
    for engine in ("umma", "simt"):
        _, y = R.run_layers(name, R.Params(name, sd, rounding=False, engine=engine), x, rounding=False)
        ref = FWD[name](sd, x, dtype=torch.float64)
        err = float((y - ref).abs().max())
        assert err <= 1e-10, f"{name}[{engine}, {weights}]: restatement vs oracle float64 max|diff| {err:.3e}"


@pytest.mark.parametrize("weights", ["benign", "calibrated"])
@pytest.mark.parametrize("name,T,variant", [("denoiser", 1013, "fp32"), ("super_resolution", 129, "fp32"),
                                            ("stereo", 203, "fp32"), ("stereo", 203, "mma")])
def test_rounded_chain_passes_its_own_checks(weight_sets, name, T, variant, weights):
    """No false alarms: the emulated device forward (every stored tensor rounded to fp16) passes every layer check, and
    stays within the model-level tolerance of the fp32 oracle with the suite's weights."""
    sd = weight_sets[weights][name]
    x = make_input(3, T, 6)
    for engine in ("umma", "simt"):
        P = R.Params(name, sd, rounding=True, engine=engine)
        S, y = R.run_layers(name, P, x, lstm_variant=variant)
        stats = R.check_layers(name, P, x, S, y, lstm_variant=variant)
        assert not [n for n, s in stats.items() if R.failed(s)], R.report(stats)
        if weights == "benign":
            assert float((y - FWD[name](sd, x)).abs().max()) <= MAX_ABS


# ------------------------------------------------------------------------------------------------ negative controls
def _shift(v):
    out = torch.zeros_like(v)
    out[..., 1:] = v[..., :-1]
    return out


def _zero_group(v):
    v[:, 8:16] = 0
    return v


def _swap_groups(v):
    a = v[:, 0:8].clone()
    v[:, 0:8] = v[:, 8:16]
    v[:, 8:16] = a
    return v


def _swap_phases(v):
    n = v.shape[-1] // 2 * 2
    a = v[..., 0:n:2].clone()
    v[..., 0:n:2] = v[..., 1:n:2]
    v[..., 1:n:2] = a
    return v


def _swap_gates_if(v):                         # stored [unit][i, f, g, o]: the i and f rows of every unit exchanged
    a = v[:, 0::4].clone()
    v[:, 0::4] = v[:, 1::4]
    v[:, 1::4] = a
    return v


def _zero_row127(v):                           # the last row of every 128-row tile
    v[..., 127::128] = 0
    return v


MUTATIONS = [
    ("denoiser", "bot_b", "output shifted by one sample", _shift, {}),
    ("stereo", "enc2a", "output shifted by one sample", _shift, {}),
    ("denoiser", "enc1b", "8-channel group zeroed", _zero_group, {}),
    ("stereo", "enc3b", "8-channel group zeroed", _zero_group, {}),
    ("denoiser", "enc2a", "two 8-channel groups swapped", _swap_groups, {}),
    ("stereo", "dec1R", "two 8-channel groups swapped", _swap_groups, {}),
    ("denoiser", "up0", "interleave phases swapped", _swap_phases, {}),
    ("super_resolution", "up", "interleave phases swapped", _swap_phases, {}),
    ("denoiser", "enc1b.pool", "pool window off by one", None, {"pool_off": True}),
    ("super_resolution", "rb1b", "residual dropped", None, {"no_res": True}),
    ("super_resolution", "middle", "residual dropped", None, {"no_res": True}),
    ("denoiser", "dec1a", "concat halves swapped", None, {"swap_cat": True}),
    ("denoiser", "dec0a", "concat halves swapped", None, {"swap_cat": True}),
    ("stereo", "xproj", "gates i and f permuted", _swap_gates_if, {}),
    ("super_resolution", "hf", "tile row 127 zeroed", _zero_row127, {}),
    ("denoiser", "enc0b", "tile row 127 zeroed", _zero_row127, {}),
]


def _model_level(y_ref, y):
    err = float((y - y_ref).abs().max())
    den = float(((y - y_ref) ** 2).sum())
    snr = float("inf") if den == 0 else float(10 * torch.log10((y_ref ** 2).sum() / den))
    return err, snr, err <= MAX_ABS and snr >= MIN_SNR_DB


def test_negative_controls_are_flagged_at_their_layer(weight_sets):
    """One mistake planted into one layer of the emulated forward, with the suite's benign weights: the per-layer metric
    flags exactly that layer, while the model output -- what the model-level parity tests look at -- mostly stays within
    their tolerance (max-abs 1e-3 and 60 dB against the unmutated forward).  This is the blind spot the per-layer GPU
    tests close."""
    sds = weight_sets["benign"]
    x = make_input(2, 2048, 5)
    clean, lines, hidden = {}, [], 0
    for name, layer, what, fn, opts in MUTATIONS:
        P = R.Params(name, sds[name], rounding=True, engine="umma")
        if name not in clean:
            clean[name] = R.run_layers(name, P, x)[1]
        S, y = R.run_layers(name, P, x, mutate=(layer, fn, opts))
        stats = R.check_layers(name, P, x, S, y)
        flagged = [n for n, s in stats.items() if R.failed(s)]
        err, snr, within = _model_level(clean[name], y)
        hidden += within
        lines.append(f"{name:16s} {layer:11s} {what:30s} flagged {flagged}  model output {snr:6.1f} dB, max-abs {err:.1e}"
                     f"{'  (within the model-level tolerance)' if within else ''}")
        assert layer in flagged, f"{name}.{layer} ({what}) not flagged:\n{R.report(stats)}"
        assert flagged[0] == layer, f"{name}.{layer} ({what}): first flagged layer is {flagged[0]}"
    print("\n".join(lines))
    print(f"{hidden} of {len(MUTATIONS)} mutations stay within the model-level tolerance")
    assert hidden >= len(MUTATIONS) // 2
