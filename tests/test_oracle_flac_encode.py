"""CPU: the exact-cost FLAC encoder reference (`encode_search` in tests/flac_encode_ref.py): round trips through the reference decoder
with the STREAMINFO MD5 over a sweep of contents, channel counts, depths, lengths and block sizes; known-answer streams
that force each choice (CONSTANT, a CONSTANT zero side channel, FIXED order 2, VERBATIM within the size bound, RICE2);
frame-header rate codes; and the host-side argument checks of the Python and C entry points."""
import ctypes as C

import numpy as np
import pytest

import flac_encode_ref as ref
from oracle import flac
from flac_encode_vectors import sweep

SWEEP = sweep()


def _bound(n: int, channels: int, bps: int, bs: int) -> int:
    """bytes of the file when every subframe is VERBATIM with the largest header (the encoder's size bound)"""
    frames = -(-n // bs)
    per = 16 + sum((8 + bs * (bps + (channels == 2 and c == 1)) + 7) // 8 for c in range(channels)) + 2
    return 4 + 4 + 34 + frames * per


def _frame0(data: bytes):
    """(channel assignment, [per coded channel: dict(type, wasted, method, porder, samples)]) of the first frame"""
    info, pos = flac.parse_container(data)
    h = flac.decode_header(data, pos, info)
    r = flac.BitReader(data, (pos + h["length"]) * 8)
    a, out = h["assign"], []
    for c in range(h["channels"]):
        depth = h["bps"] + ((a == 8 and c == 1) or (a == 9 and c == 0) or (a == 10 and c == 1))
        p = flac.BitReader(data, r.pos)
        p.bits(1)
        t = p.bits(6)
        w = p.unary() + 1 if p.bits(1) else 0
        d = dict(type=t, wasted=w)
        if 8 <= t <= 12:
            p.bits((t - 8) * (depth - w))
            d["method"], d["porder"] = p.bits(2), p.bits(4)
        d["samples"] = flac._subframe(r, h["block_size"], depth)
        out.append(d)
    return a, out


@pytest.mark.parametrize("case", SWEEP, ids=[c[0] for c in SWEEP])
def test_round_trip_and_md5(case):
    _, x, bps, bs = case
    data = ref.encode_search(x, bps, 44100, bs)
    info, got = flac.decode(data)
    assert np.array_equal(got, x)
    assert info["md5"] == flac.md5(x, bps)
    assert (info["channels"], info["bps"], info["sample_rate"], info["total_samples"]) == (x.shape[1], bps, 44100, len(x))
    assert info["min_block"] == info["max_block"] == bs
    assert len(data) <= _bound(len(x), x.shape[1], bps, bs)


def test_constant_block_is_constant():
    a, ch = _frame0(ref.encode_search(np.full((1000, 1), 1234), 16, 44100, 4096))
    assert ch[0]["type"] == 0 and ch[0]["wasted"] == 1 and ch[0]["samples"][0] == 1234


def test_equal_channels_code_a_constant_zero_side():
    x = np.random.default_rng(1).integers(-3000, 3000, (4096, 1))
    a, ch = _frame0(ref.encode_search(np.concatenate([x, x], axis=1), 16, 44100, 4096))
    assert a == 8                                                          # left/side: the lowest code of the tie
    assert ch[1]["type"] == 0 and ch[1]["samples"][0] == 0


def test_ramp_is_fixed_order_2_with_zero_residuals():
    x = (np.arange(4096) * 3 - 1000)[:, None]
    data = ref.encode_search(x, 16, 44100, 4096)
    _, ch = _frame0(data)
    assert ch[0]["type"] == 8 + 2 and ch[0]["wasted"] == 0
    assert np.array_equal(np.diff(np.array(ch[0]["samples"]), 2), np.zeros(4094))
    assert len(data) < 42 + 16 + 4 + 2 * 2 + 6 + 4096 // 8 + 64            # one bit per residual, and headers


def test_full_scale_noise_is_verbatim_within_the_bound():
    x = np.random.default_rng(2).integers(-32768, 32768, (3 * 4096 + 5, 2))
    data = ref.encode_search(x, 16, 44100, 4096)
    a, ch = _frame0(data)
    assert a == 1 and [c["type"] for c in ch] == [1, 1]
    assert len(data) <= _bound(len(x), 2, 16, 4096)
    assert np.array_equal(flac.decode(data)[1], x)


def test_loud_17_bit_side_channel_needs_rice2():
    rng = np.random.default_rng(3)
    noise, d = rng.integers(-(1 << 15), 1 << 15, 4096), rng.integers(0, 2, 4096)
    x = np.stack([100000 + noise, 100000 - noise + d], axis=1)              # M = 100000 exactly, S = 2 noise - d
    data = ref.encode_search(x, 24, 96000, 4096)
    a, ch = _frame0(data)
    assert a == 10 and ch[0]["type"] == 0
    assert 8 <= ch[1]["type"] <= 12 and ch[1]["method"] == 1
    assert np.array_equal(flac.decode(data)[1], x)


@pytest.mark.parametrize("rate,code", [(44100, 9), (11000, 12), (11025, 13), (100010, 14), (100001, 0), (655350, 14),
                                       (655349, 0)])
def test_rate_codes(rate, code):
    h = ref._frame_header(0, 4096, rate, 0, 16)
    assert h[2] & 15 == code
    x = np.arange(40)[:, None] * 5
    info, got = flac.decode(ref.encode_search(x, 16, rate, 16))
    assert info["sample_rate"] == rate and np.array_equal(got, x)


@pytest.mark.parametrize("kw", [dict(bps=20), dict(bps=8), dict(channels=9), dict(channels=0), dict(rate=0),
                                dict(rate=655351), dict(block=15), dict(block=4609), dict(n=0)])
def test_argument_errors(kw):
    a = {**dict(channels=2, n=100, bps=16, rate=44100, block=4096), **kw}
    x = np.zeros((a["n"], a["channels"]), np.int64)
    with pytest.raises(ValueError):
        ref.encode_search(x, a["bps"], a["rate"], a["block"])
    from ml_audio_restoration_b200 import _lib
    L = _lib.lib()
    ws, cap, total, mn, mx = C.c_size_t(), C.c_size_t(), C.c_int64(), C.c_int(), C.c_int()
    rc = L.ar_flac_encode(None, a["channels"], a["n"], a["bps"], a["rate"], a["block"], None, 0, None, C.byref(total),
                          C.byref(mn), C.byref(mx), None, 0, None)
    assert rc == _lib.AR_ERR_INVALID                                      # rejected on the host, before any launch
    if "rate" not in kw:
        assert L.ar_flac_encode_workspace_bytes(a["channels"], a["n"], a["block"], a["bps"], C.byref(ws),
                                                C.byref(cap)) == _lib.AR_ERR_INVALID


def test_out_of_range_samples_are_rejected():
    with pytest.raises(ValueError):
        ref.encode_search(np.array([[32768]]), 16, 44100, 4096)


def test_workspace_and_capacity_for_a_side():
    from ml_audio_restoration_b200 import _lib
    ws, cap = C.c_size_t(), C.c_size_t()
    n = 44100 * 180
    assert _lib.lib().ar_flac_encode_workspace_bytes(2, n, 4096, 16, C.byref(ws), C.byref(cap)) == _lib.AR_OK
    frames = -(-n // 4096)
    assert cap.value == frames * ((16 + 2 + (8 + 4096 * 16 + 7) // 8 + (8 + 4096 * 17 + 7) // 8 + 15) // 16 * 16)
    assert ws.value >= cap.value + 2 * n * 4


def test_save_audio_flac_rejects_float32(tmp_path):
    import torch
    from ml_audio_restoration_b200 import save_audio
    with pytest.raises(ValueError, match="FLAC stores integers"):
        save_audio(str(tmp_path / "x.FLAC"), torch.zeros(2, 10), 44100, encoding="float32")
    assert not (tmp_path / "x.FLAC").exists()


def test_quantise_matches_the_pcm16_wav_rounding():
    x = np.array([[0.5, -1.0, 1.5, -7.0, 1e-5, 0.99999, -0.499999 / 32767, 0.5 / 32767, 1.5 / 32767]], np.float32)
    assert np.array_equal(ref.quantise(x, 16)[:, 0], np.round(np.clip(x[0], -1, 1) * 32767.0).astype(np.int64))
    assert ref.quantise(np.array([[np.nan, np.inf, -np.inf]], np.float32), 24)[:, 0].tolist() == [0, 8388607, -8388607]
