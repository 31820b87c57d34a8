"""CPU: the FLAC reference decoder and test encoder (oracle/flac.py) against hand-written known-answer streams, encoder ->
decoder round trips with the STREAMINFO MD5, and the host container parse `flac_info` with its errors."""
import numpy as np
import pytest

from oracle import flac
from flac_vectors import KATS, container, crc16_bitwise, crc8_bitwise, frame, streaminfo, sweep, u, SYNC_FIXED
from ml_audio_restoration_b200.audio_processing import flac_info, is_flac

SWEEP = sweep()


@pytest.mark.parametrize("name", list(KATS))
def test_known_answer_streams(name):
    data, expect = KATS[name]()
    _, got = flac.decode(data)
    assert np.array_equal(got, np.array(expect, dtype=np.int64)), got.T.tolist()


def test_oracle_crc_tables_match_bitwise_crcs():
    data = bytes(range(256)) + b"FLAC frame"
    assert flac.crc8(data) == crc8_bitwise(data)
    assert flac.crc16(data) == crc16_bitwise(data)


@pytest.mark.parametrize("case", SWEEP, ids=[c[0] for c in SWEEP])
def test_encoder_round_trip_and_md5(case):
    _, x, bps, rate, kw = case
    data = flac.encode(x, bps, rate, **kw)
    info, got = flac.decode(data)
    assert np.array_equal(got, x)
    assert info["md5"] == flac.md5(got, bps) == flac.md5(x, bps)
    assert (info["channels"], info["bps"], info["sample_rate"]) == (x.shape[1], bps, rate)
    assert info["total_samples"] == kw.get("total_samples", len(x))


def test_flac_info_id3_and_every_skipped_block(tmp_path):
    x = np.arange(600, dtype=np.int64)[:, None] % 50
    blocks = [(1, b"\0" * 10), (2, b"abcd" + b"x" * 4), (3, (0).to_bytes(8, "big") * 2 + b"\0" * 2),
              (4, b"\x05\0\0\0vndr\0\0\0\0"), (5, b"\0" * 20), (6, b"\0" * 32)]
    data = flac.encode(x, 16, 44100, 256, subframe="fixed", order=1, metadata=blocks, id3=b"TIT2" + b"\0" * 30)
    p = tmp_path / "tagged.bin"                                       # the content decides, not the extension
    p.write_bytes(data)
    info = flac_info(str(p))
    ref, off = flac.parse_container(data)
    assert is_flac(str(p))
    assert info["offset"] == off and info["nbytes"] == len(data) - off
    assert (info["channels"], info["bps"], info["sample_rate"], info["total_samples"]) == (1, 16, 44100, 600)
    assert (info["min_block"], info["max_block"]) == (256, 256)
    assert data[off:off + 2] == b"\xff\xf8"


def _write(tmp_path, name, data):
    p = tmp_path / name
    p.write_bytes(data)
    return str(p)


def test_flac_info_errors(tmp_path):
    si = streaminfo(16, 16, 44100, 1, 16, 16)
    hdr = SYNC_FIXED + "0110" + "0000" + "0000" + "100" + "0" + "00000000" + u(15, 8)
    fr = frame(hdr, "0" + "000000" + "0" + u(3, 16))
    good = container(si, [fr])
    assert flac_info(_write(tmp_path, "good.flac", good))["total_samples"] == 16
    wav = b"RIFF\x24\0\0\0WAVEfmt "
    with pytest.raises(RuntimeError, match="not a FLAC"):
        flac_info(_write(tmp_path, "a.flac", wav))
    assert not is_flac(str(tmp_path / "a.flac"))
    no_si = b"fLaC" + bytes([0x81, 0, 0, 4]) + b"\0" * 4 + fr            # last block is PADDING, no STREAMINFO
    with pytest.raises(RuntimeError, match="STREAMINFO"):
        flac_info(_write(tmp_path, "b.flac", no_si))
    with pytest.raises(RuntimeError, match="truncated"):
        flac_info(_write(tmp_path, "c.flac", good[:20]))                  # STREAMINFO cut short
    with pytest.raises(RuntimeError, match="truncated"):
        flac_info(_write(tmp_path, "d.flac", b"fLaC\x00\x00"))
    with pytest.raises(RuntimeError, match="block type 127"):
        flac_info(_write(tmp_path, "e.flac", container(si, [fr], blocks=[(127, b"")])))
    bad_rate = container(streaminfo(16, 16, 0, 1, 16, 16), [fr])           # sample rate 0 is reserved
    with pytest.raises(RuntimeError, match="reserved"):
        flac_info(_write(tmp_path, "f.flac", bad_rate))
    bad_bs = container(streaminfo(0, 16, 44100, 1, 16, 16), [fr])          # block size 0
    with pytest.raises(RuntimeError, match="reserved"):
        flac_info(_write(tmp_path, "g.flac", bad_bs))


@pytest.mark.parametrize("field,bits", [("block size code 0", "0000" + "1001" + "0000" + "100" + "0"),
                                        ("rate code 15", "0110" + "1111" + "0000" + "100" + "0"),
                                        ("channel code 11", "0110" + "1001" + "1011" + "100" + "0"),
                                        ("bit-depth code 3", "0110" + "1001" + "0000" + "011" + "0"),
                                        ("reserved bit", "0110" + "1001" + "0000" + "100" + "1")])
def test_oracle_rejects_reserved_header_codes(field, bits):
    hdr = SYNC_FIXED + bits + "00000000" + u(15, 8)
    data = container(streaminfo(16, 16, 44100, 1, 16, 16), [frame(hdr, "0" + "000000" + "0" + u(3, 16))])
    with pytest.raises(ValueError):
        flac.decode(data)
