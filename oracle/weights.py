"""Deterministic `state_dict` factory for the three reference models (test infrastructure).

The reference ships no checkpoints (SURVEY.md section 2 #17), so parity runs need synthetic
weights.  Keys / shapes / dtypes follow the reference `state_dict` ABI exactly
(SURVEY.md App. C; denoiser.py:13-49, super_resolution.py:12-64,104-113,
stereo_separator.py:11-83) -- `tests/golden/make_golden.py` proves it by loading these
dicts into the real reference modules with `strict=True`.

Values come from numpy's PCG64 `default_rng(seed)` in a fixed key order, so they are the
same on every box without storing megabytes of weights in git.  Conv/LSTM weights use
PyTorch's default U(-1/sqrt(fan_in), 1/sqrt(fan_in)) scale; BatchNorm running stats and
affine terms are randomised (mean~N(0,.1), var~U(.5,1.5), gamma~U(.8,1.2), beta~N(0,.1),
SURVEY.md App. D) because default-init eval BN is ~identity and would hide folding bugs.
"""
from __future__ import annotations

import math
from collections import OrderedDict

import numpy as np
import torch

MODEL_NAMES = ("denoiser", "super_resolution", "stereo")


class _Gen:
    def __init__(self, seed: int):
        self.rng = np.random.default_rng(seed)
        self.sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()

    def uniform(self, key, shape, bound):
        a = self.rng.uniform(-bound, bound, size=shape).astype(np.float32)
        self.sd[key] = torch.from_numpy(a)

    def conv(self, prefix, cout, cin, k, transposed=False):
        fan_in = (cout if transposed else cin) * k  # torch: fan_in = weight.size(1) * k
        bound = 1.0 / math.sqrt(fan_in)
        shape = (cin, cout, k) if transposed else (cout, cin, k)
        self.uniform(prefix + ".weight", shape, bound)
        self.uniform(prefix + ".bias", (cout,), bound)

    def bn(self, prefix, c):
        r = self.rng
        self.sd[prefix + ".weight"] = torch.from_numpy(r.uniform(0.8, 1.2, c).astype(np.float32))
        self.sd[prefix + ".bias"] = torch.from_numpy((0.1 * r.standard_normal(c)).astype(np.float32))
        self.sd[prefix + ".running_mean"] = torch.from_numpy((0.1 * r.standard_normal(c)).astype(np.float32))
        self.sd[prefix + ".running_var"] = torch.from_numpy(r.uniform(0.5, 1.5, c).astype(np.float32))
        self.sd[prefix + ".num_batches_tracked"] = torch.tensor(100, dtype=torch.int64)


def _denoiser(g: _Gen):
    feats = [32, 64, 128]

    def block(prefix, cin, cout):  # denoiser.py:51-60
        g.conv(f"{prefix}.0", cout, cin, 3)
        g.bn(f"{prefix}.1", cout)
        g.conv(f"{prefix}.3", cout, cout, 3)
        g.bn(f"{prefix}.4", cout)

    cin = 1
    for i, f in enumerate(feats):
        block(f"encoder.{i}", cin, f)
        cin = f
    block("bottleneck", feats[-1], feats[-1] * 2)
    for i, f in enumerate(reversed(feats)):  # denoiser.py:29-35
        g.conv(f"decoder.{2 * i}", f, 2 * f, 2, transposed=True)
        block(f"decoder.{2 * i + 1}", 2 * f, f)
    g.conv("transient_detector.0", 16, 32, 3)
    g.conv("transient_detector.2", 8, 16, 3)
    g.conv("transient_detector.4", 1, 8, 3)
    g.conv("final_conv", 1, 32, 1)


def _super_resolution(g: _Gen):
    c = 32
    g.conv("initial.0", c, 1, 7)
    for i in range(4):  # super_resolution.py:104-113
        g.conv(f"residual_blocks.{i}.conv1", c, c, 3)
        g.bn(f"residual_blocks.{i}.bn1", c)
        g.conv(f"residual_blocks.{i}.conv2", c, c, 3)
        g.bn(f"residual_blocks.{i}.bn2", c)
    g.conv("middle.0", c, c, 3)
    g.bn("middle.1", c)
    g.conv("upsample_blocks.0.0", c, c, 4, transposed=True)
    g.conv("hf_emphasis.0", c, c, 5)
    g.conv("reconstruction", 1, c, 7)


def _stereo(g: _Gen):
    b, h = 32, 64
    g.conv("encoder.0.0", b, 1, 7)
    g.bn("encoder.0.1", b)
    dims = [(b, 2 * b), (2 * b, 4 * b), (4 * b, 4 * b), (4 * b, 4 * b)]
    for i, (ci, co) in enumerate(dims, start=1):  # stereo_separator.py:49-64
        g.conv(f"encoder.{i}.0", co, ci, 3)
        g.bn(f"encoder.{i}.1", co)
        g.conv(f"encoder.{i}.3", co, co, 1)
        g.bn(f"encoder.{i}.4", co)
    k = 1.0 / math.sqrt(h)  # nn.LSTM default init
    g.uniform("lstm.weight_ih_l0", (4 * h, 4 * b), k)
    g.uniform("lstm.weight_hh_l0", (4 * h, h), k)
    g.uniform("lstm.bias_ih_l0", (4 * h,), k)
    g.uniform("lstm.bias_hh_l0", (4 * h,), k)
    for side in ("left_decoder", "right_decoder"):  # stereo_separator.py:66-83
        g.conv(f"{side}.0", 4 * b, h, 7)
        g.bn(f"{side}.1", 4 * b)
        g.conv(f"{side}.3", 2 * b, 4 * b, 7)
        g.bn(f"{side}.4", 2 * b)
        g.conv(f"{side}.6", b, 2 * b, 7)
        g.bn(f"{side}.7", b)
        g.conv(f"{side}.9", 1, b, 7)


_BUILDERS = {"denoiser": _denoiser, "super_resolution": _super_resolution, "stereo": _stereo}
_SEED_OFFSET = {"denoiser": 0, "super_resolution": 1, "stereo": 2}


def make_state_dict(model: str, seed: int = 1234) -> "OrderedDict[str, torch.Tensor]":
    """state_dict for `model` in {"denoiser","super_resolution","stereo"} (App. C key set)."""
    g = _Gen(seed * 16 + _SEED_OFFSET[model])
    _BUILDERS[model](g)
    return g.sd


def make_input(batch: int, samples: int, seed: int = 1234, scale: float = 0.1) -> torch.Tensor:
    """Seeded synthetic chunk batch `[B,1,T]` at about -20 dBFS (SURVEY.md section 8c)."""
    rng = np.random.default_rng(seed * 7919 + batch * 131 + samples)
    return torch.from_numpy((scale * rng.standard_normal((batch, 1, samples))).astype(np.float32))


def calibrated_state_dicts():
    """Trained-like checkpoints: BatchNorm running stats = statistics of each layer's input on a calibration batch, so
    running_var is as small as 1e-4 and the BN folds carry gains of up to ~100 per layer (oracle.calibrate_batchnorm).
    Each model is calibrated on the previous model's output, as the chain feeds it."""
    from .models import calibrate_batchnorm, denoiser_forward, super_resolution_forward
    x = make_input(4, 8192, 5)
    sds, y = {}, x
    sds["denoiser"], _ = calibrate_batchnorm("denoiser", make_state_dict("denoiser"), y)
    y = denoiser_forward(sds["denoiser"], y)
    sds["super_resolution"], _ = calibrate_batchnorm("super_resolution", make_state_dict("super_resolution"), y)
    y = super_resolution_forward(sds["super_resolution"], y)
    sds["stereo"], _ = calibrate_batchnorm("stereo", make_state_dict("stereo"), y)
    return sds


def state_dict_checksum(sd) -> float:
    """Order-sensitive fp64 checksum used by the golden files to detect RNG drift."""
    tot = 0.0
    for i, (k, v) in enumerate(sd.items()):
        if v.dtype.is_floating_point:
            tot += float(v.double().sum()) * (1.0 + 1e-3 * (i % 17)) + float(v.double().abs().sum())
    return tot
