"""Float64 restatement of the three models, one function per fp16 tensor the device stores, with this repo's rounding points.

The model-level parity tests compare whole forwards with the fp32 oracle.  With the suite's seeded weights most layers
barely move the output (each layer's value is mostly its BatchNorm shift), so an indexing bug in one layer can hide below
the model-level tolerance.  Here each stored tensor is recomputed from the device's OWN fp16 inputs of that layer
(`ar_model_audit_tap`), so the check of a layer does not depend on what the layers behind it do with an error.

The restatement uses the reference ops (`F.conv1d`, `F.conv_transpose1d`, concatenation with the skip first, LSTM gates in
i, f, g, o order) and not the packed forms of `csrc/models.cu`, so a packing bug shows.  Rounding points mirrored from the
code:
  * BatchNorm fold in fp32 as `fold_bn`: s = g / sqrtf(var + eps), W*s, (b - mu)*s + beta; conv-engine weights rounded to
    fp16 (RNE, clamped to +-65504: `half_bits_host`), biases fp32;
  * stored activations: fp32 accumulation rounded once to fp16 (`cvt.rn.satfinite`), a residual is read as fp16 and added
    before that rounding; the max-pool copy is the max of the rounded values;
  * stems (Cin = 1) and the denoiser tail use fp32 weights; the super-resolution head uses fp16-rounded weights on both
    engines, the stereo heads fp16 on the tensor-core engine (`pack_final_umma`) and fp32 on the CUDA-core one;
  * LSTM: input projection (W_ih * sc) fp16, bias (b_ih + b_hh) * sc fp32, rows pre-scaled by log2(e) (2 log2(e) for the
    cell candidate), stored as fp16 in [unit][i, f, g, o] channel order; the recurrence keeps c in fp32 and takes
    W_hh * sc and the fed-back h in fp16 (`lstm_mmaw_kernel`) or both in fp32 (`lstm_kernel<1, 8>`).

Per element a stored value passes when |dev - ref| <= ulp16(ref) + 2^-18 * mag, where `mag` is the same op on |x|, |w|,
|b| (+ |residual|): fp32 accumulation of fp16 products can move the result by a small multiple of 2^-24 * mag, and the
final rounding by half an fp16 ulp.  Some checks are exact: the pool copy against max_pool1d of the device's un-pooled
tensor, the right zero-pad row of an up-conv, the zero padding channels of `td0`.

`run_layers(..., rounding=False)` chains the same functions without any rounding; that reproduces `oracle.*_forward` in
float64 (tests/test_oracle_layer_ref.py), so these functions are the reference network and not a second design.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle.models import detect_impulses

SLOPE = 0.2
HALF_MAX = 65504.0
L2E32 = float(torch.tensor(1.4426950408889634, dtype=torch.float32))   # the float constant of models.cu
SLACK = 2.0 ** -18          # accumulation slack per unit of `mag` (fp32 accumulation of fp16 products)
TAIL_SLACK = 2.0 ** -18     # fp32 tails (heads, denoiser tail): fp32 arithmetic throughout
MAX_DIFF_FRACTION = 0.01    # elements whose stored fp16 value differs from the correctly rounded reference ...
MIN_DIFF_COUNT = 2          # ... counted only beyond this many elements


# ------------------------------------------------------------------------------------------------ rounding
def r16(t):
    """fp32 value -> fp16 with round-to-nearest-even, clamped to the finite range (`half_bits_host`), as float64."""
    return t.float().clamp(-HALF_MAX, HALF_MAX).half().double()


def ulp16(v):
    e = torch.floor(torch.log2(v.abs())).clamp(min=-14.0)
    e = torch.where(torch.isfinite(e), e, torch.full_like(e, -14.0))
    return torch.pow(2.0, e - 10.0)


def _lrelu(v):
    return torch.where(v > 0, v, SLOPE * v)


# ------------------------------------------------------------------------------------------------ parameters
class Params:
    """Weights as each engine consumes them.  rounding=False: plain float64 (the reference network)."""

    def __init__(self, name, sd, rounding=True, engine="umma"):
        self.name, self.sd, self.rounding, self.engine = name, sd, rounding, engine

    def _f(self, t):
        return t.float() if self.rounding else t.double()

    def fold(self, conv, bn=None):
        """(W, b) of conv [+ BN] folded in the precision of `fold_bn` (fp32), returned as float64."""
        sd = self.sd
        W, b = self._f(sd[conv + ".weight"]), self._f(sd[conv + ".bias"])
        if bn:
            eps = self._f(sd[bn + ".eps"]).reshape(()) if bn + ".eps" in sd else self._f(torch.tensor(1e-5, dtype=torch.float64))
            s = self._f(sd[bn + ".weight"]) / torch.sqrt(self._f(sd[bn + ".running_var"]) + eps)
            W = W * s[:, None, None]
            b = (b - self._f(sd[bn + ".running_mean"])) * s + self._f(sd[bn + ".bias"])
        return W.double(), b.double()

    def w16(self, W):
        return r16(W) if self.rounding else W.double()

    def engine_conv(self, conv, bn=None):
        W, b = self.fold(conv, bn)
        return self.w16(W), b

    def raw(self, key):
        return self._f(self.sd[key]).double()


# ------------------------------------------------------------------------------------------------ ops (float64)
class Val:
    """A layer's float64 value before the final rounding, its magnitude term and optional exact-check positions."""

    def __init__(self, v, mag=None, exact=None, kind="fp16"):
        self.v, self.mag, self.exact, self.kind = v, mag, exact, kind


def conv(x, W, b, pad, dil=1, lrelu=True, res=None):
    v = F.conv1d(x, W, b, padding=pad, dilation=dil)
    mag = F.conv1d(x.abs(), W.abs(), b.abs(), padding=pad, dilation=dil)
    if lrelu:
        v = _lrelu(v)
    if res is not None:
        v = v + res
        mag = mag + res.abs()
    return Val(v, mag)


def conv_t(x, W, b, stride, padding, Tout, lrelu):
    """ConvTranspose1d through the reference op; a right zero-pad up to Tout (denoiser.py:121-122) is an exact zero."""
    v = F.conv_transpose1d(x, W, b, stride=stride, padding=padding)
    mag = F.conv_transpose1d(x.abs(), W.abs(), b.abs(), stride=stride, padding=padding)
    if lrelu:
        v = _lrelu(v)
    n = v.shape[2]
    exact = None
    if Tout > n:
        v = F.pad(v, (0, Tout - n))
        mag = F.pad(mag, (0, Tout - n))
        exact = torch.zeros(v.shape, dtype=torch.bool)
        exact[..., n:] = True
    return Val(v[..., :Tout], mag[..., :Tout], None if exact is None else exact[..., :Tout])


def pool(u, off=False):
    """MaxPool1d(2, 2), floor.  off=True pairs rows (2t+1, 2t+2) instead: a negative control."""
    if off:
        u = F.pad(u[..., 1:], (0, 1), mode="replicate")
    return Val(F.max_pool1d(u, 2, 2), kind="exact")


# ------------------------------------------------------------------------------------------------ model layers
# Each model is an ordered list of (name, fn(S, x, P, opts) -> Val).  S holds the stored tensors written so far (float64
# [B, C, T]); `opts` switches a deliberate mistake on for the negative controls of tests/test_oracle_layer_ref.py.

def _cat(S, skip, up, opts):
    return torch.cat((S[up], S[skip]) if opts.get("swap_cat") else (S[skip], S[up]), dim=1)


def denoiser_layers(P, T):
    T1, T2, T3 = T // 2, T // 4, T // 8
    L = []

    def add(name, fn):
        L.append((name, fn))

    W, b = P.fold("encoder.0.0", "encoder.0.1")       # fp32 stem
    add("stem", lambda S, x, o: conv(x, W, b, 1))

    def block(name, src, conv_, bn_, pool_name=None):
        Wq, bq = P.engine_conv(conv_, bn_)
        add(name, lambda S, x, o: conv(S[src] if not callable(src) else src(S, o), Wq, bq, 1))
        if pool_name:
            add(pool_name, lambda S, x, o: pool(S[name], o.get("pool_off", False)))

    block("enc0b", "stem", "encoder.0.3", "encoder.0.4", "enc0b.pool")
    block("enc1a", "enc0b.pool", "encoder.1.0", "encoder.1.1")
    block("enc1b", "enc1a", "encoder.1.3", "encoder.1.4", "enc1b.pool")
    block("enc2a", "enc1b.pool", "encoder.2.0", "encoder.2.1")
    block("enc2b", "enc2a", "encoder.2.3", "encoder.2.4", "enc2b.pool")
    block("bot_a", "enc2b.pool", "bottleneck.0", "bottleneck.1")
    block("bot_b", "bot_a", "bottleneck.3", "bottleneck.4")
    prev, skips, touts = "bot_b", ("enc2b", "enc1b", "enc0b"), (T2, T1, T)
    for i in range(3):
        Wu, bu = P.w16(P.raw(f"decoder.{2 * i}.weight")), P.raw(f"decoder.{2 * i}.bias")
        up, skip, Tout = f"up{i}", skips[i], touts[i]
        add(up, lambda S, x, o, Wu=Wu, bu=bu, prev=prev, Tout=Tout: conv_t(S[prev], Wu, bu, 2, 0, Tout, lrelu=False))
        block(f"dec{i}a", lambda S, o, skip=skip, up=up: _cat(S, skip, up, o), f"decoder.{2 * i + 1}.0", f"decoder.{2 * i + 1}.1")
        block(f"dec{i}b", f"dec{i}a", f"decoder.{2 * i + 1}.3", f"decoder.{2 * i + 1}.4")
        prev = f"dec{i}b"
    Wd, bd = P.fold("transient_detector.0")
    if P.engine == "umma":
        Wd16 = P.w16(Wd)

        def td0(S, x, o):
            v = conv(S["dec2b"], Wd16, bd, 1)
            z = torch.zeros_like(v.v)
            ex = torch.zeros(z.shape[0], 32, z.shape[2], dtype=torch.bool)
            ex[:, 16:] = True
            return Val(torch.cat((v.v, z), 1), torch.cat((v.mag, z), 1), ex)
        add("td0", td0)

    W1, b1 = P.fold("transient_detector.2")
    W2, b2 = P.fold("transient_detector.4")
    WF, BF = P.fold("final_conv")

    def tail(S, x, o):
        f = S["dec2b"]
        if P.engine == "umma":
            h1 = S["td0"][:, :16]
            m1 = h1.abs()
        else:
            v = conv(f, Wd, bd, 1)
            h1, m1 = v.v, v.mag
        v2 = conv(h1, W1, b1, 1)
        m2 = F.conv1d(m1, W1.abs(), b1.abs(), padding=1)
        v3 = conv(v2.v, W2, b2, 1, lrelu=False)
        m3 = F.conv1d(m2, W2.abs(), b2.abs(), padding=1)
        mask = torch.maximum(torch.sigmoid(v3.v), detect_impulses(x))
        yv = conv(f, WF, BF, 0, lrelu=False)
        return Val(yv.v * (1.0 - mask * 0.9), yv.mag * (2.0 + m3), kind="fp32")
    add("y", tail)
    return L


def super_resolution_layers(P, T):
    L = []

    def add(name, fn):
        L.append((name, fn))

    W0, b0 = P.fold("initial.0")
    add("stem", lambda S, x, o: conv(x, W0, b0, 3))
    prev = "stem"
    for i in range(4):
        p = f"residual_blocks.{i}"
        Wa, ba = P.engine_conv(p + ".conv1", p + ".bn1")
        Wb, bb = P.engine_conv(p + ".conv2", p + ".bn2")
        add(f"rb{i}a", lambda S, x, o, Wa=Wa, ba=ba, prev=prev: conv(S[prev], Wa, ba, 1))
        add(f"rb{i}b", lambda S, x, o, Wb=Wb, bb=bb, prev=prev, i=i:
            conv(S[f"rb{i}a"], Wb, bb, 1, lrelu=False, res=None if o.get("no_res") else S[prev]))
        prev = f"rb{i}b"
    Wm, bm = P.engine_conv("middle.0", "middle.1")
    add("middle", lambda S, x, o: conv(S["rb3b"], Wm, bm, 1, lrelu=False, res=None if o.get("no_res") else S["stem"]))
    Wu, bu = P.w16(P.raw("upsample_blocks.0.0.weight")), P.raw("upsample_blocks.0.0.bias")
    add("up", lambda S, x, o: conv_t(S["middle"], Wu, bu, 2, 1, 2 * T, lrelu=True))
    Wh, bh = P.engine_conv("hf_emphasis.0")
    add("hf", lambda S, x, o: conv(S["up"], Wh, bh, 2))
    WR, BR = P.w16(P.raw("reconstruction.weight")), P.raw("reconstruction.bias")

    def head(S, x, o):
        v = conv(S["hf"], WR, BR, 3, lrelu=False)
        up = F.interpolate(x, scale_factor=2, mode="linear", align_corners=False)
        mag_up = F.interpolate(x.abs(), scale_factor=2, mode="linear", align_corners=False)
        return Val(v.v + up, v.mag + mag_up, kind="fp32")
    add("y", head)
    return L


def _gate_scale(P):
    l2e = L2E32 if P.rounding else 1.0 / math.log(2.0)
    return torch.tensor([l2e, l2e, 2.0 * l2e, l2e], dtype=torch.float32 if P.rounding else torch.float64)


def stereo_lstm_params(P):
    """(W_ih * sc, (b_ih + b_hh) * sc, W_hh * sc) in gate-major rows (i, f, g, o), as the device packs them (models.cu)."""
    sc = _gate_scale(P).repeat_interleave(64)
    Wih = P.w16((P._f(P.sd["lstm.weight_ih_l0"]) * sc[:, None]).double())
    bias = ((P._f(P.sd["lstm.bias_ih_l0"]) + P._f(P.sd["lstm.bias_hh_l0"])) * sc).double()
    Whh = (P._f(P.sd["lstm.weight_hh_l0"]) * sc[:, None]).double()
    return Wih, bias, Whh


def unit_gate_order(v):
    """[B, 256, T] gate-major (row g*64 + u) -> the stored [unit][gate] channel order (channel 4u + g)."""
    B, _, T = v.shape
    return v.reshape(B, 4, 64, T).transpose(1, 2).reshape(B, 256, T)


def gate_major_order(v):
    B, _, T = v.shape
    return v.reshape(B, 64, 4, T).transpose(1, 2).reshape(B, 256, T)


def lstm_recurrence(P, xp_ug, variant, h_dev=None):
    """h for every step from the stored pre-activations (unit-gate order, scaled).  variant:
      "mma"  -- lstm_mmaw_kernel<4|8>: W_hh * sc and h fed back in fp16; teacher-forced: step t takes the device's h_{t-1}
                (`h_dev`, exactly what the kernel feeds back), so every step is checked on its own;
      "fp32" -- lstm_kernel<1, 8>: W_hh * sc and h in fp32; the fp32 h is not observable, so the recurrence runs freely.
    c is carried in fp32 (float64 without rounding); the clamps of `lstm_cell` are applied."""
    _, _, Whh = stereo_lstm_params(P)
    l2e = L2E32 if P.rounding else 1.0 / math.log(2.0)
    if variant == "mma" and P.rounding:
        Whh = r16(Whh)
    xg = gate_major_order(xp_ug)                      # [B, 256, T]
    B, _, T = xg.shape
    h = xg.new_zeros(B, 64)
    c = xg.new_zeros(B, 64)
    hs, mags = [], []
    def sig(p):
        return 1.0 / (1.0 + torch.exp2(-p))
    feed16 = variant == "mma" and P.rounding
    for t in range(T):
        if feed16 and h_dev is not None:
            hin = h_dev[:, :, t - 1] if t > 0 else xg.new_zeros(B, 64)
        else:
            hin = store16(h) if feed16 else h
        g = xg[:, :, t] + hin @ Whh.t()
        gm = (xg[:, :, t].abs() + hin.abs() @ Whh.abs().t()).reshape(B, 4, 64).amax(1)
        pi, pf, pg, po = g.reshape(B, 4, 64).unbind(1)
        if P.rounding:      # the clamps of lstm_cell (they move a gate by < 3e-9)
            pi, pf, po = (torch.clamp(p, min=-20.0 * l2e) for p in (pi, pf, po))
            pg = torch.clamp(pg, min=-40.0 * l2e)
        c_prev = c
        c = sig(pf) * c + sig(pi) * torch.tanh(pg / (2.0 * l2e))
        if P.rounding:
            c = c.float().double()
        h = sig(po) * torch.tanh(torch.clamp(c, min=-20.0) if P.rounding else c)
        hs.append(h)
        mags.append(gm + c_prev.abs() + 1.0)
    return torch.stack(hs, 2), torch.stack(mags, 2)


def stereo_layers(P, T, lstm_variant="fp32"):
    L = []

    def add(name, fn):
        L.append((name, fn))

    W0, b0 = P.fold("encoder.0.0", "encoder.0.1")
    add("stem", lambda S, x, o: conv(x, W0, b0, 3))
    prev = "stem"
    for i in range(1, 5):
        d = 1 << (i - 1)
        Wa, ba = P.engine_conv(f"encoder.{i}.0", f"encoder.{i}.1")
        Wb, bb = P.engine_conv(f"encoder.{i}.3", f"encoder.{i}.4")
        add(f"enc{i}a", lambda S, x, o, Wa=Wa, ba=ba, prev=prev, d=d: conv(S[prev], Wa, ba, d, d))
        add(f"enc{i}b", lambda S, x, o, Wb=Wb, bb=bb, i=i: conv(S[f"enc{i}a"], Wb, bb, 0))
        prev = f"enc{i}b"
    Wih, bih, _ = stereo_lstm_params(P)

    def xproj(S, x, o):
        v = conv(S["enc4b"], Wih[:, :, None], bih, 0, lrelu=False)
        return Val(unit_gate_order(v.v), unit_gate_order(v.mag))
    add("xproj", xproj)

    def lstm(S, x, o):
        h_dev = S.get("lstm") if (lstm_variant == "mma" and P.rounding) else None
        h, mag = lstm_recurrence(P, S["xproj"], lstm_variant, h_dev)
        return Val(h, mag)
    add("lstm", lstm)
    WL, bL = P.engine_conv("left_decoder.0", "left_decoder.1")
    WR, bR = P.engine_conv("right_decoder.0", "right_decoder.1")
    add("dec0", lambda S, x, o: conv(S["lstm"], torch.cat((WL, WR)), torch.cat((bL, bR)), 3))
    for side, tag, lo in (("left_decoder", "L", 0), ("right_decoder", "R", 128)):
        W1, b1 = P.engine_conv(f"{side}.3", f"{side}.4")
        W2, b2 = P.engine_conv(f"{side}.6", f"{side}.7")
        add(f"dec1{tag}", lambda S, x, o, W1=W1, b1=b1, lo=lo: conv(S["dec0"][:, lo:lo + 128], W1, b1, 3))
        add(f"dec2{tag}", lambda S, x, o, W2=W2, b2=b2, tag=tag: conv(S[f"dec1{tag}"], W2, b2, 3))
    heads = []
    for side, tag in (("left_decoder", "L"), ("right_decoder", "R")):
        WF, BF = P.raw(f"{side}.9.weight"), P.raw(f"{side}.9.bias")
        heads.append((tag, P.w16(WF) if P.engine == "umma" else WF, BF))

    def head(S, x, o):
        vs = [conv(S[f"dec2{tag}"], WF, BF, 3, lrelu=False) for tag, WF, BF in heads]
        return Val(torch.cat([v.v for v in vs], 1), torch.cat([v.mag for v in vs], 1), kind="fp32")
    add("y", head)
    return L


LAYERS = {"denoiser": denoiser_layers, "super_resolution": super_resolution_layers, "stereo": stereo_layers}


def layers(name, P, T, lstm_variant="fp32"):
    if name == "stereo":
        return stereo_layers(P, T, lstm_variant)
    return LAYERS[name](P, T)


def tapped_names(name, P, T):
    """Names of the stored tensors in launch order (the final output "y" excluded)."""
    return [n for n, _ in layers(name, P, T) if n != "y"]


def lstm_variant_for(B, sm_count):
    """The recurrence kernel a layer-by-layer stereo forward of B sequences runs (lstm.cu launch_lstm)."""
    return "mma" if B > 2 * sm_count else "fp32"


# ------------------------------------------------------------------------------------------------ chaining and checking
def store16(v):
    """What the device stores for a float64 value: fp32, then fp16 round-to-nearest-even with saturation."""
    return v.float().clamp(-HALF_MAX, HALF_MAX).half().double()


def run_layers(name, P, x, rounding=True, mutate=None, lstm_variant="fp32"):
    """Chain the restatement: every stored tensor from the stored tensors before it (rounded to fp16 when `rounding`).
    `mutate = (layer, fn(value) -> value, opts)` plants one mistake into one layer.  Returns ({name: tensor}, y)."""
    x = x.double()
    S = {}
    for n, fn in layers(name, P, x.shape[2], lstm_variant):
        opts = mutate[2] if (mutate and mutate[0] == n) else {}
        val = fn(S, x, opts)
        out = val.v
        if rounding and val.kind == "fp16":
            out = store16(out)
        elif rounding and val.kind == "fp32":
            out = out.float().double()
        if mutate and mutate[0] == n and mutate[1] is not None:
            out = mutate[1](out.clone())
        S[n] = out
    y = S.pop("y")
    return S, y


def compare(dev, val, slack):
    """Stats of one stored tensor against its float64 value: worst |dev - ref| / bound, the fraction of elements that
    differ from the correctly rounded reference, exact-position mismatches and non-finite values."""
    dev = dev.double()
    ref = val.v
    if val.kind == "exact":
        bad = int((dev != ref).sum())
        return {"kind": val.kind, "ratio": 0.0 if bad == 0 else float("inf"), "frac": bad / max(1, ref.numel()), "ndiff": bad, "n": ref.numel(),
                "exact_bad": bad, "nonfinite": int((~torch.isfinite(dev)).sum())}
    err = (dev - ref).abs()
    if val.kind == "fp16":
        bound = ulp16(ref) + slack * val.mag
        differ = dev != store16(ref)
    else:
        bound = slack * val.mag + 1e-30
        differ = dev != ref.float().double()
    ratio = err / bound
    exact_bad = 0
    if val.exact is not None:
        exact_bad = int(((dev != ref) & val.exact).sum())
        ratio = torch.where(val.exact, torch.zeros_like(ratio), ratio)
        differ = differ & ~val.exact
    ratio = torch.where(torch.isfinite(ratio), ratio, torch.full_like(ratio, float("inf")))
    return {"kind": val.kind, "ratio": float(ratio.max()) if ratio.numel() else 0.0,
            "frac": float(differ.double().mean()) if differ.numel() else 0.0, "ndiff": int(differ.sum()),
            "n": differ.numel(), "exact_bad": exact_bad, "nonfinite": int((~torch.isfinite(dev)).sum())}


def check_layers(name, P, x, S, y, lstm_variant="fp32", slack=SLACK, tail_slack=TAIL_SLACK, lstm_slack=None):
    """Every stored tensor of S (and the output y) against the restatement computed from S itself.
    Returns {layer: stats} in launch order; `failed(stats)` tells which fail."""
    x = x.double()
    out = {}
    for n, fn in layers(name, P, x.shape[2], lstm_variant):
        val = fn(S, x, {})
        dev = y if n == "y" else S[n]
        s = tail_slack if val.kind == "fp32" else (lstm_slack if (n == "lstm" and lstm_slack is not None) else slack)
        out[n] = compare(dev, val, s)
    return out


def failed(stats):
    """A stored fp16 tensor fails on one element outside its bound, or when more of its elements than MAX_DIFF_FRACTION
    (and more than MIN_DIFF_COUNT, so that one flip in a tiny tensor is not a failure) differ from the correctly rounded
    reference.  fp32 outputs are held to the bound only: their last bits depend on the summation order, so most differ
    from the correctly rounded value by an ulp."""
    if stats["ratio"] > 1.0 or stats["exact_bad"] > 0 or stats["nonfinite"] > 0:
        return True
    return stats["kind"] == "fp16" and stats["ndiff"] > max(MAX_DIFF_FRACTION * stats["n"], MIN_DIFF_COUNT)


def report(stats):
    return "\n".join(f"  {n:12s} worst |dev-ref|/bound {s['ratio']:.3g}  differing {100 * s['frac']:.3f} %"
                     + (" (fp32 output: last bits)" if s["kind"] == "fp32" else "")
                     + (f"  exact mismatches {s['exact_bad']}" if s["exact_bad"] else "")
                     + (f"  non-finite {s['nonfinite']}" if s["nonfinite"] else "")
                     + ("  FAIL" if failed(s) else "") for n, s in stats.items())


def tap_shapes(name, B, T):
    """{stored tensor: (channels, length)} of a forward on [B, 1, T] (the windows `ar_model_audit_tap` copies)."""
    if name == "denoiser":
        T1, T2, T3 = T // 2, T // 4, T // 8
        s = {"stem": (32, T), "enc0b": (32, T), "enc0b.pool": (32, T1), "enc1a": (64, T1), "enc1b": (64, T1),
             "enc1b.pool": (64, T2), "enc2a": (128, T2), "enc2b": (128, T2), "enc2b.pool": (128, T3), "bot_a": (256, T3),
             "bot_b": (256, T3), "up0": (128, T2), "dec0a": (128, T2), "dec0b": (128, T2), "up1": (64, T1), "dec1a": (64, T1),
             "dec1b": (64, T1), "up2": (32, T), "dec2a": (32, T), "dec2b": (32, T), "td0": (32, T)}
    elif name == "super_resolution":
        s = {"stem": (32, T)}
        for i in range(4):
            s[f"rb{i}a"] = s[f"rb{i}b"] = (32, T)
        s.update({"middle": (32, T), "up": (32, 2 * T), "hf": (32, 2 * T)})
    else:
        s = {"stem": (32, T)}
        for i, c in zip(range(1, 5), (64, 128, 128, 128)):
            s[f"enc{i}a"] = s[f"enc{i}b"] = (c, T)
        s.update({"xproj": (256, T), "lstm": (64, T), "dec0": (256, T), "dec1L": (64, T), "dec2L": (32, T),
                  "dec1R": (64, T), "dec2R": (32, T)})
    return s
