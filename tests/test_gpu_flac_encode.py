"""GPU: the FLAC encoder (`ar_flac_encode` through `encode_flac_cuda`) byte-identical to `encode_search`
(tests/flac_encode_ref.py) over the sweep, bit-exact round trips through the device decoder, `save_audio` FLAC vs WAV at 16 and 24 bits, NaN / inf
input, the CLI writing FLAC, sides of realistic length, a 100 000-frame stream, and equal bytes from two streams."""
import hashlib

import numpy as np
import pytest
import torch

import oracle
import flac_encode_ref as ref
from oracle import flac
from flac_encode_vectors import sweep
from flac_vectors import signal
from ml_audio_restoration_b200.audio_processing import _read_wav, decode_flac_cuda, encode_flac_cuda, flac_info, save_audio
from ml_audio_restoration_b200.inference import main

pytestmark = pytest.mark.gpu
SWEEP = sweep()


def _unit(q: np.ndarray, bps: int) -> torch.Tensor:
    """[N, C] integers -> planar float32 [C, N] CUDA audio, q / 2^(bps-1) (what the readers of this package return)"""
    return torch.from_numpy(flac.to_float(q, bps)).cuda()


def _decode(tmp_path, data: bytes, name="e.flac"):
    p = tmp_path / name
    p.write_bytes(data)
    info = flac_info(str(p))
    raw = torch.frombuffer(bytearray(data[info["offset"]:]), dtype=torch.uint8).cuda()
    return decode_flac_cuda(raw, info).cpu().numpy(), info


@pytest.mark.parametrize("case", SWEEP, ids=[c[0] for c in SWEEP])
def test_bytes_equal_oracle_and_round_trip(case, tmp_path):
    _, x, bps, bs = case
    audio = _unit(x, bps)
    q = ref.quantise(audio.cpu().numpy(), bps)
    got = encode_flac_cuda(audio, 44100, bps=bps, block_size=bs)
    assert got == ref.encode_search(q, bps, 44100, bs)
    dec, info = _decode(tmp_path, got)
    assert np.array_equal(dec, flac.to_float(q, bps))
    assert info["total_samples"] == len(x)


def test_nan_and_inf_inputs(tmp_path):
    rng = np.random.default_rng(5)
    x = rng.uniform(-1.2, 1.2, (2, 9000)).astype(np.float32)
    x[0, ::97], x[1, ::89], x[0, 5::101], x[1, 7::103] = np.nan, np.inf, -np.inf, np.nan
    for bps in (16, 24):
        q = ref.quantise(x, bps)
        got = encode_flac_cuda(torch.from_numpy(x).cuda(), 48000, bps=bps)
        assert got == ref.encode_search(q, bps, 48000)
        dec, _ = _decode(tmp_path, got)
        assert np.array_equal(dec, flac.to_float(q, bps))


@pytest.mark.parametrize("encoding", ["pcm16", "pcm24"])
@pytest.mark.parametrize("channels", [1, 2])
def test_save_audio_flac_and_wav_load_identically(encoding, channels, tmp_path):
    a = torch.from_numpy(np.random.default_rng(channels).uniform(-1.1, 1.1, (channels, 30011)).astype(np.float32))
    for src in (a, a.cuda()):                                             # a host tensor goes to the current device
        fl, wav = tmp_path / "o.flac", tmp_path / "o.wav"
        save_audio(str(fl), src, 44100, encoding=encoding)
        save_audio(str(wav), src, 44100, encoding=encoding)
        assert fl.read_bytes()[:4] == b"fLaC" and wav.read_bytes()[:4] == b"RIFF"
        (f, sr_f), (w, sr_w) = _read_wav(str(fl)), _read_wav(str(wav))
        assert sr_f == sr_w == 44100 and torch.equal(f, w)
    default = tmp_path / "d.FLAC"
    save_audio(str(default), a.cuda(), 44100)                              # FLAC defaults to 24 bits
    assert flac_info(str(default))["bps"] == 24


def test_two_streams_give_identical_bytes():
    x = _unit(signal(44100 * 20, 2, 24, seed=11), 24)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        a = encode_flac_cuda(x, 44100, bps=16)
    with torch.cuda.stream(s2):
        b = encode_flac_cuda(x, 44100, bps=16)
    assert a == b == encode_flac_cuda(x, 44100, bps=16)


@pytest.mark.parametrize("bps", [16, 24])
def test_three_minute_side(bps, tmp_path):
    x = _unit(signal(44100 * 180, 2, 24, seed=bps), 24)
    data = encode_flac_cuda(x, 44100, bps=bps)
    q = ref.quantise(x.cpu().numpy(), bps)
    dec, info = _decode(tmp_path, data)
    assert np.array_equal(dec, flac.to_float(q, bps))
    info, _ = flac.parse_container(data)
    assert info["md5"] == flac.md5(q, bps)
    assert len(data) < q.size * bps // 8                                   # smaller than the PCM


def test_hundred_thousand_frames(tmp_path):
    x = _unit(signal(16 * 100_000 + 7, 1, 16, seed=4), 16)
    data = encode_flac_cuda(x, 22050, bps=16, block_size=16)
    q = ref.quantise(x.cpu().numpy(), 16)
    dec, info = _decode(tmp_path, data)
    assert np.array_equal(dec, flac.to_float(q, 16)) and info["min_block"] == 16
    width = q.astype("<i2").tobytes()
    assert flac.parse_container(data)[0]["md5"] == hashlib.md5(width).digest()


@pytest.fixture()
def checkpoints(state_dicts, tmp_path):
    paths = {}
    for name in oracle.MODEL_NAMES:
        p = tmp_path / f"{name}.pth"
        torch.save({"model_state_dict": state_dicts[name]}, p)
        paths[name] = str(p)
    return paths


def test_cli_flac_output_is_the_pcm24_quantisation_of_the_float_wav(checkpoints, tmp_path):
    src = tmp_path / "side.wav"
    save_audio(str(src), torch.from_numpy(flac.to_float(signal(2 * 9000, 2, 16, seed=8), 16)), 44100, encoding="pcm16")
    common = [str(src), "--denoiser", checkpoints["denoiser"], "--super-res", checkpoints["super_resolution"], "--stereo",
              checkpoints["stereo"], "--sample-rate", "22050", "--device", "cuda", "--mode", "chunked", "--chunk-size", "2048",
              "--overlap", "256"]
    wav, fl, fl16 = tmp_path / "out.wav", tmp_path / "out.flac", tmp_path / "out16.flac"
    main(common[:1] + [str(wav)] + common[1:])
    main(common[:1] + [str(fl)] + common[1:])
    main(common[:1] + [str(fl16)] + common[1:] + ["--output-encoding", "pcm16"])
    out, sr = _read_wav(str(wav))
    data = fl.read_bytes()
    info, ints = flac.decode(data)
    q = ref.quantise(out.numpy(), 24)
    assert sr == info["sample_rate"] == 44100 and info["bps"] == 24 and np.array_equal(ints, q)
    assert info["md5"] == flac.md5(ints, 24)
    got, _ = _read_wav(str(fl))                                           # the device decoder reads it back too
    assert np.array_equal(got.numpy(), flac.to_float(q, 24))
    assert np.array_equal(flac.decode(fl16.read_bytes())[1], ref.quantise(out.numpy(), 16))
    with pytest.raises(ValueError, match="FLAC stores integers"):
        main(common[:1] + [str(tmp_path / "f.flac")] + common[1:] + ["--output-encoding", "float32"])
