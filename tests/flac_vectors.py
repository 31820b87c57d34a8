"""FLAC test vectors shared by test_oracle_flac.py (CPU) and test_gpu_flac.py: hand-written known-answer streams, built
field by field from bit strings with bitwise CRCs (independent of oracle/flac.py), and the encoder sweep."""
import numpy as np

from oracle import flac


# ----------------------------------------------------------------------------- bit strings
def u(v: int, n: int) -> str:
    """n-bit field, two's complement for negative values"""
    return format(v & ((1 << n) - 1), f"0{n}b") if n else ""


def rice(v: int, k: int) -> str:
    """Rice code of a signed residual: zigzag u, then u >> k zeros, a 1 and the low k bits"""
    z = 2 * v if v >= 0 else -2 * v - 1
    return "0" * (z >> k) + "1" + u(z, k)


def to_bytes(bits: str) -> bytes:
    bits = "".join(bits.split())
    assert len(bits) % 8 == 0 and set(bits) <= {"0", "1"}, len(bits)
    return int(bits, 2).to_bytes(len(bits) // 8, "big") if bits else b""


def crc8_bitwise(data: bytes) -> int:
    c = 0
    for b in data:
        c ^= b
        for _ in range(8):
            c = ((c << 1) ^ 0x07) & 0xFF if c & 0x80 else (c << 1) & 0xFF
    return c


def crc16_bitwise(data: bytes) -> int:
    c = 0
    for b in data:
        c ^= b << 8
        for _ in range(8):
            c = ((c << 1) ^ 0x8005) & 0xFFFF if c & 0x8000 else (c << 1) & 0xFFFF
    return c


def frame(header: str, subframes: str) -> bytes:
    """header bits (sync .. optional rate, without CRC-8) + subframe bits -> frame bytes with both CRCs"""
    h = to_bytes(header)
    h += bytes([crc8_bitwise(h)])
    body = "".join(subframes.split())
    body += "0" * (-len(body) % 8)                                        # zero padding to a byte boundary
    f = h + to_bytes(body)
    return f + crc16_bitwise(f).to_bytes(2, "big")


def streaminfo(min_block, max_block, rate, channels, bps, total) -> str:
    return (u(min_block, 16) + u(max_block, 16) + u(0, 24) + u(0, 24)           # block sizes, frame sizes unknown
            + u(rate, 20) + u(channels - 1, 3) + u(bps - 1, 5) + u(total, 36)
            + u(0, 128))                                                   # MD5 not given


def container(si: str, frames, blocks=()) -> bytes:
    """`fLaC`, STREAMINFO (+ extra (type, body) blocks), frames"""
    md = [(0, to_bytes(si))] + list(blocks)
    out = b"fLaC"
    for i, (t, body) in enumerate(md):
        out += to_bytes(u(i == len(md) - 1, 1) + u(t, 7) + u(len(body), 24)) + body
    return out + b"".join(frames)


SYNC_FIXED, SYNC_VARIABLE = "11111111111110" + "0" + "0", "11111111111110" + "0" + "1"   # 14-bit sync, 0, strategy


# ----------------------------------------------------------------------------- known-answer streams
def kat_constant_bs192_rate0():
    """mono 8-bit, block-size code 1 (192), rate code 0 (from STREAMINFO), one CONSTANT subframe of -5"""
    hdr = (SYNC_FIXED + "0001" + "0000"          # block size 192, rate from STREAMINFO
           + "0000" + "001" + "0"                 # 1 channel, 8 bits, reserved
           + "00000000")                          # frame number 0
    sub = "0" + "000000" + "0" + u(-5, 8)         # pad, CONSTANT, no wasted bits, value
    return container(streaminfo(192, 192, 44100, 1, 8, 192), [frame(hdr, sub)]), [[-5]] * 192


def kat_verbatim_bs8bit_rate_khz():
    """mono 8-bit, block-size code 6 (8-bit value + 1 = 4), rate code 12 (8 kHz), VERBATIM"""
    hdr = (SYNC_FIXED + "0110" + "1100" + "0000" + "001" + "0" + "00000000"
           + u(3, 8)                               # block size - 1
           + u(8, 8))                              # kHz
    vals = [1, -2, 127, -128]
    sub = "0" + "000001" + "0" + "".join(u(v, 8) for v in vals)
    return container(streaminfo(4, 4, 8000, 1, 8, 4), [frame(hdr, sub)]), [[v] for v in vals]


def kat_fixed_orders_bs16bit_rate_hz():
    """5 independent 16-bit channels, block-size code 7 (16-bit value + 1 = 6), rate code 13 (11025 Hz), channel c is a
    FIXED subframe of order c with Rice parameter 1"""
    hdr = (SYNC_FIXED + "0111" + "1101" + "0100" + "100" + "0" + "00000000" + u(5, 16) + u(11025, 16))

    def fixed(order, warm, res):
        return ("0" + u(8 + order, 6) + "0" + "".join(u(v, 16) for v in warm)
                + "00" + "0000" + u(1, 4) + "".join(rice(r, 1) for r in res))

    subs = (fixed(0, [], [3, -1, 0, 2, -2, 1]) + fixed(1, [100], [1, 1, -1, 0, 2]) + fixed(2, [10, 12], [1, -1, 0, 0])
            + fixed(3, [1, 4, 9], [0, 0, 1]) + fixed(4, [0, 1, 8, 27], [0, -1]))
    expect = np.array([[3, -1, 0, 2, -2, 1], [100, 101, 102, 101, 101, 103], [10, 12, 15, 17, 19, 21],
                       [1, 4, 9, 16, 25, 37], [0, 1, 8, 27, 64, 124]]).T
    return container(streaminfo(6, 6, 11025, 5, 16, 6), [frame(hdr, subs)]), expect.tolist()


def kat_lpc_rice2_escape():
    """mono 16-bit, block size 8 (code 6), rate code 14 (2205 x 10 Hz), LPC order 2, precision 4, shift 1, coefficients
    (3, -1); Rice2 residual with partition order 2: partition 0 empty (2 - order), 1 a 5-bit parameter 16, 2 an escape
    with w = 0, 3 an escape with w = 5.  Predictions are negative: the shift is arithmetic."""
    hdr = SYNC_FIXED + "0110" + "1110" + "0000" + "100" + "0" + "00000000" + u(7, 8) + u(2205, 16)
    sub = ("0" + "100001" + "0"                     # LPC order 2
           + u(-20, 16) + u(-30, 16)                # warm-up
           + "0011" + "00001"                       # precision 4, shift 1
           + u(3, 4) + u(-1, 4)                     # coefficients
           + "01" + "0010"                          # Rice2, partition order 2
           + u(0, 5)                                # partition 0: parameter 0, no residuals
           + u(16, 5) + rice(-3, 16) + rice(5, 16)  # partition 1
           + "11111" + u(0, 5)                      # partition 2: escape, w = 0 (two zeros)
           + "11111" + u(5, 5) + u(-7, 5) + u(9, 5))  # partition 3: escape, w = 5
    return (container(streaminfo(8, 8, 22050, 1, 16, 8), [frame(hdr, sub)]),
            [[v] for v in [-20, -30, -38, -37, -37, -37, -44, -39]])


def kat_wasted_left_side():
    """stereo 16-bit left/side, block size 4; left VERBATIM with 2 wasted bits, side VERBATIM at 17 bits"""
    hdr = SYNC_FIXED + "0110" + "1001" + "1000" + "100" + "0" + "00000000" + u(3, 8)
    left = "0" + "000001" + "1" + "01" + "".join(u(v, 14) for v in [1, -2, 3, 100])
    side = "0" + "000001" + "0" + "".join(u(v, 17) for v in [1, -3, 5, -2])
    return (container(streaminfo(4, 4, 44100, 2, 16, 4), [frame(hdr, left + side)]),
            [[4, 3], [-8, -5], [12, 7], [400, 402]])


def kat_side_right():
    """stereo 16-bit side/right: side CONSTANT 7 (17 bits), right VERBATIM"""
    hdr = SYNC_FIXED + "0110" + "1001" + "1001" + "100" + "0" + "00000000" + u(3, 8)
    side = "0" + "000000" + "0" + u(7, 17)
    right = "0" + "000001" + "0" + "".join(u(v, 16) for v in [10, -10, 0, 5])
    return (container(streaminfo(4, 4, 44100, 2, 16, 4), [frame(hdr, side + right)]),
            [[17, 10], [-3, -10], [7, 0], [12, 5]])


def kat_mid_side_odd():
    """stereo 16-bit mid/side with odd side values"""
    hdr = SYNC_FIXED + "0110" + "1001" + "1010" + "100" + "0" + "00000000" + u(3, 8)
    mid = "0" + "000001" + "0" + "".join(u(v, 16) for v in [5, -3, 0, 7])
    side = "0" + "000001" + "0" + "".join(u(v, 17) for v in [3, -1, 2, 4])
    return (container(streaminfo(4, 4, 44100, 2, 16, 4), [frame(hdr, mid + side)]),
            [[7, 4], [-3, -2], [1, -1], [9, 5]])


def kat_variable_blocking():
    """variable blocking: frame 0 (sample 0, 200 samples, CONSTANT 1), frame 1 (sample 200 coded as the two-byte
    C3 88, 2 samples VERBATIM)"""
    h0 = SYNC_VARIABLE + "0110" + "1001" + "0000" + "100" + "0" + "00000000" + u(199, 8)
    h1 = SYNC_VARIABLE + "0110" + "1001" + "0000" + "100" + "0" + "11000011" + "10001000" + u(1, 8)
    f0 = frame(h0, "0" + "000000" + "0" + u(1, 16))
    f1 = frame(h1, "0" + "000001" + "0" + u(2, 16) + u(3, 16))
    return container(streaminfo(2, 200, 44100, 1, 16, 202), [f0, f1]), [[1]] * 200 + [[2], [3]]


KATS = {f.__name__[4:]: f for f in (kat_constant_bs192_rate0, kat_verbatim_bs8bit_rate_khz, kat_fixed_orders_bs16bit_rate_hz,
                                    kat_lpc_rice2_escape, kat_wasted_left_side, kat_side_right, kat_mid_side_odd,
                                    kat_variable_blocking)}


# ----------------------------------------------------------------------------- encoder sweep
def signal(n: int, channels: int, bps: int, seed: int = 0, shift: int = 0) -> np.ndarray:
    """[n, C] integers of a smooth signal plus noise within bps bits (lowest `shift` bits zero)"""
    rng = np.random.default_rng(seed)
    t = np.arange(n)[:, None]
    amp = 2.0 ** (bps - 3 - shift)
    x = amp * np.sin(t * (0.01 + 0.003 * np.arange(channels))[None, :]) + rng.normal(0, amp / 64 + 1, (n, channels))
    lim = 2 ** (bps - 1 - shift)
    return (np.clip(np.round(x), -lim, lim - 1).astype(np.int64)) << shift


def sweep():
    """(id, samples [N, C], bps, rate, encoder kwargs): every bit depth, 1..8 channels, every subframe type, LPC orders
    1..32 across precisions 1..15 and shifts 0..15, Rice / Rice2 at partition orders 0..8, wasted bits, the stereo modes,
    fixed and variable blocking with a short last frame, total samples 0."""
    cases = []
    for i, bps in enumerate((8, 12, 16, 20, 24, 32)):
        cases.append((f"bps{bps}", signal(1500, 1 + i % 3, bps, i), bps, 44100, dict(block_size=512)))
    for c in range(1, 9):
        cases.append((f"ch{c}", signal(1300, c, 16, 10 + c), 16, 48000, dict(block_size=576, stereo="independent")))
    cases.append(("constant", np.full((1024, 2), -77, np.int64), 16, 44100, dict(subframe="constant", block_size=256,
                                                                                  stereo="independent")))
    cases.append(("verbatim", signal(1000, 2, 24, 3), 24, 96000, dict(subframe="verbatim", block_size=300)))
    for o in range(5):
        cases.append((f"fixed{o}", signal(1200, 1, 16, 20 + o), 16, 44100, dict(subframe="fixed", order=o, block_size=400)))
    for o in range(1, 33):
        cases.append((f"lpc{o}", signal(1100, 1, 16, 40 + o), 16, 44100,
                      dict(order=o, precision=1 + (o - 1) % 15, shift=o % 16, block_size=512)))
    for p in range(9):
        cases.append((f"rice_p{p}", signal(1024, 1, 16, 80 + p), 16, 44100, dict(partition_order=p, block_size=512)))
        cases.append((f"rice2_p{p}", signal(1024, 1, 24, 90 + p), 24, 44100,
                      dict(partition_order=p, block_size=512, rice2=True)))
    cases.append(("escape", signal(1024, 2, 16, 5), 16, 44100, dict(escape=True, block_size=256, subframe="fixed", order=2)))
    cases.append(("escape_odd_zero", np.tile(np.arange(1024)[:, None] * 3, (1, 1)), 16, 44100,
                  dict(escape="odd", block_size=256, subframe="fixed", order=2, partition_order=2)))
    cases.append(("wasted", signal(1500, 2, 16, 6, shift=3), 16, 44100, dict(block_size=512)))
    for mode in ("left_side", "side_right", "mid_side"):
        cases.append((mode, signal(1500, 2, 16, 7), 16, 44100, dict(stereo=mode, block_size=512)))
        cases.append((mode + "_32", signal(900, 2, 32, 8), 32, 44100, dict(stereo=mode, block_size=300, subframe="fixed",
                                                                           order=2)))
    cases.append(("variable", signal(1500, 2, 16, 9), 16, 44100, dict(blocks=[100, 700, 16, 500, 184], partition_order=2)))
    cases.append(("unknown_total", signal(1500, 1, 16, 11), 16, 44100, dict(block_size=1024, total_samples=0)))
    cases.append(("rate_codes", signal(800, 1, 16, 12), 16, 37800, dict(block_size=200, rate_code=14, bs_code="16bit")))
    return cases
