"""GPU: the frame-parallel FLAC decoder (`ar_flac_decode` through `decode_flac_cuda`) bit-exact against the encoded
integers and the reference decoder, FLAC and WAV loading identically, false sync codes, corrupt streams, sides of
realistic length, and FLAC through `restore_audio` / the CLI / `generate_test_output`."""
import numpy as np
import pytest
import torch

import oracle
from oracle import audio_io, flac
from flac_vectors import KATS, SYNC_FIXED, container, frame, signal, streaminfo, sweep, u
from ml_audio_restoration_b200.audio_processing import _read_wav, decode_flac_cuda, flac_info, load_audio_cuda
from ml_audio_restoration_b200.inference import generate_test_output, main

pytestmark = pytest.mark.gpu
SWEEP = sweep()


def _decode(tmp_path, data: bytes, name="s.flac"):
    p = tmp_path / name
    p.write_bytes(data)
    info = flac_info(str(p))
    raw = torch.frombuffer(bytearray(data[info["offset"]:]), dtype=torch.uint8).cuda()
    return decode_flac_cuda(raw, info).cpu().numpy(), info


def _scaled(x: np.ndarray, bps: int) -> np.ndarray:
    return flac.to_float(x, bps)


@pytest.mark.parametrize("case", SWEEP, ids=[c[0] for c in SWEEP])
def test_decode_bit_exact_sweep(case, tmp_path):
    _, x, bps, rate, kw = case
    got, info = _decode(tmp_path, flac.encode(x, bps, rate, **kw))
    assert got.dtype == np.float32 and np.array_equal(got, _scaled(x, bps))


@pytest.mark.parametrize("name", list(KATS))
def test_decode_known_answer_streams(name, tmp_path):
    data, expect = KATS[name]()
    info, ref = flac.decode(data)
    got, _ = _decode(tmp_path, data)
    assert np.array_equal(got, _scaled(ref, info["bps"]))
    assert np.array_equal(ref, np.array(expect))


@pytest.mark.parametrize("rate,bps,channels", [(44100, 16, 2), (48000, 16, 2), (22050, 16, 2), (44100, 24, 2),
                                               (48000, 24, 2), (22050, 24, 2), (44100, 16, 1), (48000, 24, 1),
                                               (22050, 16, 1)])
def test_flac_and_wav_load_identically(rate, bps, channels, tmp_path):
    x = signal(3 * rate // 2 + 17, channels, bps, seed=rate + bps)
    wav, fl = tmp_path / "a.wav", tmp_path / "a.flac"
    fmt = audio_io.PCM_S16 if bps == 16 else audio_io.PCM_S24
    audio_io.write_wav(str(wav), x.astype(np.int16) if bps == 16 else x.astype(np.int32), fmt, rate)
    fl.write_bytes(flac.encode(x, bps, rate, 4096))
    a, sr_a = load_audio_cuda(str(wav), 22050)
    b, sr_b = load_audio_cuda(str(fl), 22050)
    assert sr_a == sr_b == 22050 and torch.equal(a, b)
    host, sr = _read_wav(str(fl))                                        # the host reader decodes FLAC on the device too
    assert sr == rate and np.array_equal(host.numpy(), _scaled(x, bps))


def test_false_sync_inside_verbatim_subframe(tmp_path):
    """A VERBATIM subframe whose samples spell a sync code and a header with a valid CRC-8 that agrees with STREAMINFO (a
    copy of frame 0's own header) is not taken for a frame."""
    hdr = SYNC_FIXED + "0110" + "1001" + "0000" + "100" + "0" + "00000000" + u(7, 8)
    fake = frame(hdr, "0" + "000000" + "0" + u(1, 16))[:8]               # header bytes incl. a valid CRC-8
    fake_words = [int.from_bytes(fake[i:i + 2], "big") for i in range(0, 8, 2)]
    samples = [v - 65536 if v >= 32768 else v for v in fake_words] + [1, 2, 3, 4]
    f0 = frame(hdr, "0" + "000001" + "0" + "".join(u(v, 16) for v in samples))
    h1 = SYNC_FIXED + "0110" + "1001" + "0000" + "100" + "0" + "00000001" + u(7, 8)
    f1 = frame(h1, "0" + "000000" + "0" + u(-9, 16))
    data = container(streaminfo(8, 8, 44100, 1, 16, 16), [f0, f1])
    assert data.count(fake[:7]) == 2                                      # frame 0's header, and its copy in the samples
    got, _ = _decode(tmp_path, data)
    assert np.array_equal(got, _scaled(np.array(samples + [-9] * 8)[:, None], 16))


def test_corrupt_streams_raise_without_faulting(tmp_path):
    x = signal(20 * 1024, 2, 16, seed=3)
    data = flac.encode(x, 16, 44100, 1024)
    info, off = flac.parse_container(data)
    f7 = off
    for _ in range(7):
        f7 = flac.decode_frame(data, f7, info)[2]
    bad = bytearray(data)
    bad[f7 + 200] ^= 0x10                                                 # one bit in frame 7's residual
    with pytest.raises(RuntimeError, match=f"frame 7 at byte {f7 - off}"):
        _decode(tmp_path, bytes(bad), "flip.flac")
    with pytest.raises(RuntimeError, match="frame 19 at byte"):
        _decode(tmp_path, data[:-5], "trunc.flac")                       # truncated last frame
    reserved = bytearray(data)
    reserved[f7 + 2] = (reserved[f7 + 2] & 0xF0) | 0x0F                   # rate code 15
    with pytest.raises(RuntimeError, match="frame 7 .*sample-rate code"):
        _decode(tmp_path, bytes(reserved), "reserved.flac")
    got, _ = _decode(tmp_path, data, "ok.flac")                           # the device is still healthy
    assert np.array_equal(got, _scaled(x, 16))
    torch.cuda.synchronize()


def test_scale_sides_and_many_frames(tmp_path):
    cd = signal(44100 * 180, 2, 16, seed=1)
    got, _ = _decode(tmp_path, flac.encode(cd, 16, 44100, 4096, order=12), "cd.flac")
    assert np.array_equal(got, _scaled(cd, 16))
    del got
    hi = signal(96000 * 180, 2, 24, seed=2)
    got, _ = _decode(tmp_path, flac.encode(hi, 24, 96000, 4096, order=12), "hires.flac")
    assert np.array_equal(got, _scaled(hi, 24))
    del got
    many = signal(192 * 100_500, 1, 16, seed=4)
    got, _ = _decode(tmp_path, flac.encode(many, 16, 44100, 192, subframe="fixed", order=2), "many.flac")
    assert np.array_equal(got, _scaled(many, 16))


@pytest.fixture()
def checkpoints(state_dicts, tmp_path):
    paths = {}
    for name in oracle.MODEL_NAMES:
        p = tmp_path / f"{name}.pth"
        torch.save({"model_state_dict": state_dicts[name]}, p)
        paths[name] = str(p)
    return paths


def test_cli_flac_input_equals_wav_input(checkpoints, tmp_path):
    x = signal(2 * 9000, 2, 16, seed=8)
    wav, fl = tmp_path / "side.wav", tmp_path / "side.flac"
    audio_io.write_wav(str(wav), x.astype(np.int16), audio_io.PCM_S16, 44100)
    fl.write_bytes(flac.encode(x, 16, 44100, 4096))
    common = ["--denoiser", checkpoints["denoiser"], "--super-res", checkpoints["super_resolution"],
              "--stereo", checkpoints["stereo"], "--sample-rate", "22050", "--device", "cuda"]
    for mode, extra in (("whole", []), ("chunked", ["--chunk-size", "2048", "--overlap", "256"])):
        outs = []
        for src in (wav, fl):
            dst = tmp_path / f"{mode}_{src.suffix[1:]}.wav"
            main([str(src), str(dst), "--mode", mode] + extra + common)
            outs.append(dst.read_bytes())
        assert outs[0] == outs[1], mode


def test_generate_test_output_picks_up_flac(state_dicts, tmp_path):
    from gpu_util import make_model
    src, out = tmp_path / "in", tmp_path / "out"
    src.mkdir()
    (src / "side.flac").write_bytes(flac.encode(signal(30000, 2, 16, seed=9), 16, 44100, 4096))
    written = generate_test_output(make_model("denoiser", state_dicts["denoiser"]), str(src), str(out), "epoch_1")
    assert [p.split("/")[-1] for p in written] == ["side_restored_epoch_1.wav"]
    assert (out / "side_original.wav").exists() and (out / "side_degraded_epoch_1.wav").exists()
