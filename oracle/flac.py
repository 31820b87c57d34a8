"""TEST INFRASTRUCTURE ONLY -- FLAC (RFC 9639): a plain CPU reference decoder, written for reading rather than speed, and a
numpy-vectorised encoder for tests that can force every choice the format offers (subframe type, predictor order, LPC
precision and shift, Rice / Rice2 coding, partition order, escape partitions, wasted bits, stereo mode, block-size and
sample-rate codes, fixed or variable blocking, metadata blocks).  The reference reads FLAC through soundfile
(src/utils/audio_processing.py:24); neither soundfile nor libFLAC is installed here, so the device decoder is pinned to this
restatement and to hand-written bit strings in tests/test_oracle_flac.py.

Samples are `[N, C]` integer arrays (frames by channels), as `oracle.audio_io.write_wav` takes them.
Only tests/, __graft_entry__.smoke() and the measurement tools may import this package.
"""
import hashlib
import struct

import numpy as np


def _crc_table(poly: int, width: int):
    top, mask = 1 << (width - 1), (1 << width) - 1
    tab = []
    for v in range(256):
        c = v << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
        tab.append(c)
    return np.array(tab, dtype=np.int64)


CRC8_TABLE = _crc_table(0x07, 8)
CRC16_TABLE = _crc_table(0x8005, 16)


def crc8(data: bytes) -> int:
    c = 0
    for b in data:
        c = int(CRC8_TABLE[c ^ b])
    return c


def crc16(data: bytes) -> int:
    c = 0
    for b in data:
        c = ((c << 8) & 0xFFFF) ^ int(CRC16_TABLE[(c >> 8) ^ b])
    return c


BLOCK_SIZE_CODES = {192: 1, 576: 2, 1152: 3, 2304: 4, 4608: 5, 256: 8, 512: 9, 1024: 10, 2048: 11, 4096: 12, 8192: 13,
                    16384: 14, 32768: 15}
RATE_CODES = {88200: 1, 176400: 2, 192000: 3, 8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10, 96000: 11}
BPS_CODES = {8: 1, 12: 2, 16: 4, 20: 5, 24: 6, 32: 7}
STREAMINFO, PADDING, APPLICATION, SEEKTABLE, VORBIS_COMMENT, CUESHEET, PICTURE = range(7)


# ----------------------------------------------------------------------------- container
def parse_container(data: bytes):
    """(STREAMINFO dict, byte offset of the first frame): optional ID3v2 tag, `fLaC`, metadata blocks."""
    pos = 0
    if data[:3] == b"ID3":
        if len(data) < 10:
            raise ValueError("truncated ID3v2 header")
        size = (data[6] << 21) | (data[7] << 14) | (data[8] << 7) | data[9]
        pos = 10 + size + (10 if data[5] & 0x10 else 0)
    if data[pos:pos + 4] != b"fLaC":
        raise ValueError("not a FLAC stream")
    pos += 4
    info = None
    while True:
        if pos + 4 > len(data):
            raise ValueError("truncated metadata block header")
        last, btype, size = data[pos] >> 7, data[pos] & 0x7F, int.from_bytes(data[pos + 1:pos + 4], "big")
        pos += 4
        if pos + size > len(data):
            raise ValueError("truncated metadata block")
        body = data[pos:pos + size]
        if btype == STREAMINFO:
            if size != 34:
                raise ValueError("STREAMINFO must be 34 bytes")
            r = BitReader(body)
            info = {"min_block": r.bits(16), "max_block": r.bits(16), "min_frame": r.bits(24), "max_frame": r.bits(24),
                    "sample_rate": r.bits(20), "channels": r.bits(3) + 1, "bps": r.bits(5) + 1,
                    "total_samples": r.bits(36), "md5": body[18:34]}
        elif btype == 127:
            raise ValueError("invalid metadata block type 127")
        pos += size
        if last:
            break
    if info is None:
        raise ValueError("no STREAMINFO block")
    return info, pos


# ----------------------------------------------------------------------------- reference decoder
class BitReader:
    """MSB-first reader over `data` from bit `pos`."""

    def __init__(self, data: bytes, pos: int = 0):
        self.data, self.pos = data, pos

    def bits(self, n: int) -> int:
        if n == 0:
            return 0
        b0, off = self.pos >> 3, self.pos & 7
        nb = (off + n + 7) >> 3
        if b0 + nb > len(self.data):
            raise ValueError("read past the end of the data")
        v = int.from_bytes(self.data[b0:b0 + nb], "big")
        self.pos += n
        return (v >> (nb * 8 - off - n)) & ((1 << n) - 1)

    def sbits(self, n: int) -> int:
        v = self.bits(n)
        return v - (1 << n) if n and v >> (n - 1) else v

    def unary(self) -> int:
        q = 0
        while self.bits(1) == 0:
            q += 1
        return q

    def align(self):
        self.pos = (self.pos + 7) & ~7


def decode_header(data: bytes, pos: int, info: dict):
    """Frame header at byte `pos` -> dict (block_size, sample_rate, assign, channels, bps, variable, number, length)."""
    r = BitReader(data, pos * 8)
    if r.bits(15) != 0x7FFC:
        raise ValueError("no frame sync code")
    variable = r.bits(1)
    bs_code, rate_code, assign, bps_code = r.bits(4), r.bits(4), r.bits(4), r.bits(3)
    if r.bits(1):
        raise ValueError("reserved header bit set")
    if bs_code == 0 or rate_code == 15 or assign > 10 or bps_code == 3:
        raise ValueError("reserved code in the frame header")
    lead = r.bits(8)
    for n_extra, mask, tag in ((0, 0x80, 0x00), (1, 0xE0, 0xC0), (2, 0xF0, 0xE0), (3, 0xF8, 0xF0), (4, 0xFC, 0xF8),
                               (5, 0xFE, 0xFC), (6, 0xFF, 0xFE)):
        if lead & mask == tag:
            break
    else:
        raise ValueError("invalid coded number")
    if n_extra == 6 and not variable:
        raise ValueError("invalid coded number")
    number = lead & ~mask & 0xFF
    for _ in range(n_extra):
        c = r.bits(8)
        if c >> 6 != 2:
            raise ValueError("invalid coded number")
        number = (number << 6) | (c & 0x3F)
    if bs_code == 1:
        bs = 192
    elif bs_code <= 5:
        bs = 576 << (bs_code - 2)
    elif bs_code == 6:
        bs = r.bits(8) + 1
    elif bs_code == 7:
        bs = r.bits(16) + 1
    else:
        bs = 256 << (bs_code - 8)
    rates = {v: k for k, v in RATE_CODES.items()}
    if rate_code == 0:
        rate = info["sample_rate"]
    elif rate_code == 12:
        rate = r.bits(8) * 1000
    elif rate_code == 13:
        rate = r.bits(16)
    elif rate_code == 14:
        rate = r.bits(16) * 10
    else:
        rate = rates[rate_code]
    length = r.pos // 8 - pos
    if crc8(data[pos:pos + length]) != r.bits(8):
        raise ValueError("CRC-8 mismatch")
    bps = info["bps"] if bps_code == 0 else {v: k for k, v in BPS_CODES.items()}[bps_code]
    return {"block_size": bs, "sample_rate": rate, "assign": assign, "channels": assign + 1 if assign < 8 else 2,
            "bps": bps, "variable": variable, "number": number, "length": length + 1}


FIXED_COEFS = ((), (1,), (2, -1), (3, -3, 1), (4, -6, 4, -1))


def _residual(r: BitReader, bs: int, order: int):
    method = r.bits(2)
    if method > 1:
        raise ValueError("reserved residual coding method")
    pbits = 4 if method == 0 else 5
    porder = r.bits(4)
    parts = 1 << porder
    if bs % parts or (bs >> porder) < order:
        raise ValueError("invalid partition order")
    out = []
    for p in range(parts):
        count = (bs >> porder) - (order if p == 0 else 0)
        k = r.bits(pbits)
        if k == (1 << pbits) - 1:                                   # escape: w-bit signed values
            w = r.bits(5)
            out += [r.sbits(w) for _ in range(count)]
        else:
            for _ in range(count):
                u = (r.unary() << k) | r.bits(k)
                out.append((u >> 1) ^ -(u & 1))
    return out


def _subframe(r: BitReader, bs: int, depth: int):
    if r.bits(1):
        raise ValueError("subframe padding bit set")
    t = r.bits(6)
    wasted = r.unary() + 1 if r.bits(1) else 0
    depth -= wasted
    if t == 0:
        s = [r.sbits(depth)] * bs
    elif t == 1:
        s = [r.sbits(depth) for _ in range(bs)]
    elif 8 <= t <= 12:
        order = t - 8
        s = [r.sbits(depth) for _ in range(order)]
        for e in _residual(r, bs, order):
            s.append(e + sum(c * s[-1 - j] for j, c in enumerate(FIXED_COEFS[order])))
    elif t >= 32:
        order = t - 31
        s = [r.sbits(depth) for _ in range(order)]
        precision = r.bits(4) + 1
        if precision == 16:
            raise ValueError("invalid LPC precision")
        shift = r.sbits(5)
        if shift < 0:
            raise ValueError("negative LPC shift")
        coefs = [r.sbits(precision) for _ in range(order)]
        for e in _residual(r, bs, order):
            s.append(e + (sum(c * s[-1 - j] for j, c in enumerate(coefs)) >> shift))
    else:
        raise ValueError("reserved subframe type")
    return [v << wasted for v in s]


def decode_frame(data: bytes, pos: int, info: dict):
    """One frame at byte `pos` -> (samples [bs, C] int64, header dict, byte offset after the frame)."""
    h = decode_header(data, pos, info)
    if (h["channels"], h["bps"], h["sample_rate"]) != (info["channels"], info["bps"], info["sample_rate"]):
        raise ValueError("frame header disagrees with STREAMINFO")
    r = BitReader(data, (pos + h["length"]) * 8)
    bs, a = h["block_size"], h["assign"]
    chans = []
    for c in range(h["channels"]):
        side = (a == 8 and c == 1) or (a == 9 and c == 0) or (a == 10 and c == 1)
        chans.append(_subframe(r, bs, h["bps"] + side))
    r.align()
    end = r.pos // 8
    if crc16(data[pos:end]) != r.bits(16):
        raise ValueError("CRC-16 mismatch")
    x = np.array(chans, dtype=np.int64).T
    if a == 8:
        x[:, 1] = x[:, 0] - x[:, 1]
    elif a == 9:
        x[:, 0] = x[:, 0] + x[:, 1]
    elif a == 10:
        m = (x[:, 0] << 1) | (x[:, 1] & 1)
        x = np.stack([(m + x[:, 1]) >> 1, (m - x[:, 1]) >> 1], axis=1)
    return x, h, end + 2


def decode(data: bytes):
    """A whole .flac file -> (STREAMINFO dict, samples [N, C] int64)."""
    info, pos = parse_container(data)
    blocks, n = [], 0
    while pos < len(data) and not (info["total_samples"] and n >= info["total_samples"]):
        x, _, pos = decode_frame(data, pos, info)
        blocks.append(x)
        n += len(x)
    if info["total_samples"] and n != info["total_samples"]:
        raise ValueError("sample count disagrees with STREAMINFO")
    return info, np.concatenate(blocks) if blocks else np.zeros((0, info["channels"]), np.int64)


def md5(samples: np.ndarray, bps: int) -> bytes:
    """STREAMINFO MD5: interleaved signed little-endian samples in ceil(bps/8) bytes each."""
    width = (bps + 7) // 8
    v = np.ascontiguousarray(samples, dtype=np.int64).reshape(-1)
    b = np.stack([(v >> (8 * i)) & 0xFF for i in range(width)], axis=-1).astype(np.uint8)
    return hashlib.md5(b.tobytes()).digest()


def to_float(samples: np.ndarray, bps: int) -> np.ndarray:
    """[N, C] integers -> planar fp32 [C, N], x / 2^(bps-1) (soundfile's float32 read)."""
    return np.ascontiguousarray((samples.astype(np.int32).astype(np.float32) * np.float32(2.0 ** (1 - bps))).T)


# ----------------------------------------------------------------------------- encoder (tests)
def _utf8(v: int) -> bytes:
    if v < 0x80:
        return bytes([v])
    n = 2
    while v >= 1 << (5 * n + 1):
        n += 1
    out = [0x80 | ((v >> (6 * i)) & 0x3F) for i in range(n - 1)][::-1]
    return bytes([((0xFF00 >> n) & 0xFF) | (v >> (6 * (n - 1)))] + out)


def _signed_width(x: np.ndarray, axis) -> np.ndarray:
    """bits of the narrowest two's complement holding every value along `axis` (0 when all are zero)"""
    m = np.where(x < 0, ~x, x).max(axis=axis)
    nz = np.any(x != 0, axis=axis)
    return np.where(m > 0, np.frexp(np.maximum(m, 1).astype(np.float64))[1] + 1, np.where(nz, 1, 0)).astype(np.int64)


def _levinson(x: np.ndarray, order: int) -> np.ndarray:
    """LPC predictor coefficients [F, order] (c_j multiplies s[n-1-j]) of every row of x (Welch window, autocorrelation)."""
    F, n = x.shape
    w = 1.0 - ((np.arange(n) - (n - 1) / 2) / ((n + 1) / 2)) ** 2
    xw = x.astype(np.float64) * w
    R = np.stack([(xw[:, k:] * xw[:, :n - k]).sum(1) for k in range(order + 1)], axis=1)
    R[:, 0] *= 1.0 + 1e-9
    a = np.zeros((F, order))
    err = R[:, 0].copy()
    for i in range(order):
        acc = R[:, i + 1] - (a[:, :i] * R[:, i:0:-1]).sum(1)
        k = np.where(err > 0, acc / np.where(err > 0, err, 1.0), 0.0)
        prev = a[:, :i].copy()
        a[:, :i] = prev - k[:, None] * prev[:, ::-1]
        a[:, i] = k
        err = err * (1.0 - k * k)
    return a


def _subframe_fields(X: np.ndarray, depth: int, cfg: dict):
    """Fields (values, widths) [F, K] of one channel's subframes for a group of frames of equal block size."""
    F, bs = X.shape
    kind = cfg["subframe"]
    V, W = [], []

    def add(v, w):
        v = np.asarray(v, dtype=np.int64)
        if v.ndim == 0:
            v = np.full(F, int(v), np.int64)
        w = np.broadcast_to(np.asarray(w, dtype=np.int64), v.shape)
        V.append(v.reshape(F, -1))
        W.append(w.reshape(F, -1))

    # wasted bits: trailing zeros shared by every sample of the subframe
    if cfg["wasted"]:
        orr = np.bitwise_or.reduce(X, axis=1)
        low = orr & -orr
        k = np.where(orr != 0, np.log2(np.where(low > 0, low, 1).astype(np.float64)).astype(np.int64), 0)
        k = np.minimum(k, depth - 1)
    else:
        k = np.zeros(F, np.int64)
    Xs = X >> k[:, None]
    ed = depth - k
    if kind == "constant":
        if not np.all(Xs == Xs[:, :1]):
            raise ValueError("CONSTANT subframe of a non-constant block")
        t, order = np.zeros(F, np.int64), 0
    elif kind == "verbatim":
        t, order = np.ones(F, np.int64), 0
    elif kind == "fixed":
        order = cfg["order"]
        t = np.full(F, 8 + order)
    elif kind == "lpc":
        order = cfg["order"]
        t = np.full(F, 31 + order)
    else:
        raise ValueError(f"unknown subframe type {kind!r}")
    add((t << 1) | (k > 0), 8)
    add(np.where(k > 0, 1, 0), np.where(k > 0, k, 0))                     # k-1 zeros and a 1
    ew = ed[:, None]
    if kind == "constant":
        add(Xs[:, :1] & ((1 << ew) - 1), ew)
        return V, W
    if kind == "verbatim":
        add(Xs & ((1 << ew) - 1), ew)
        return V, W
    if order > bs:
        raise ValueError("predictor order larger than the block")
    add(Xs[:, :order] & ((1 << ew) - 1), ew)
    pred = np.zeros((F, bs - order), np.int64)
    if kind == "fixed":
        for j, c in enumerate(FIXED_COEFS[order]):
            pred += c * Xs[:, order - 1 - j:bs - 1 - j]
    else:
        prec = cfg["precision"]
        a = _levinson(Xs, order)
        if cfg["shift"] is None:
            cmax = np.maximum(np.abs(a).max(1), 1e-9)
            shift = np.clip(prec - 2 - np.floor(np.log2(cmax)).astype(np.int64), 0, 15)
        else:
            shift = np.full(F, cfg["shift"], np.int64)
        q = np.clip(np.round(a * (2.0 ** shift[:, None])), -(1 << (prec - 1)), (1 << (prec - 1)) - 1).astype(np.int64)
        add(prec - 1, 4)
        add(shift, 5)
        add(q & ((1 << prec) - 1), prec)
        acc = np.zeros((F, bs - order), np.int64)
        for j in range(order):
            acc += q[:, j:j + 1] * Xs[:, order - 1 - j:bs - 1 - j]
        pred = acc >> shift[:, None]
    res = Xs[:, order:] - pred
    if res.size and (res.min() < -(1 << 31) or res.max() >= (1 << 31)):
        raise ValueError("residual outside the 32-bit range: choose another predictor")
    _residual_fields(res, bs, order, cfg, add)
    return V, W


def _residual_fields(res, bs, order, cfg, add):
    F = res.shape[0]
    rice2 = cfg["rice2"]
    pbits, kmax = (5, 30) if rice2 else (4, 14)
    escape = (1 << pbits) - 1
    p = cfg["partition_order"]
    if p is None:
        p = 0
        while p < 8 and bs % (2 << p) == 0 and (bs >> (p + 1)) >= max(order, 64):
            p += 1
    while p > 0 and (bs % (1 << p) or (bs >> p) < order):               # a short last frame takes what fits
        p -= 1
    parts, ps = 1 << p, bs >> p
    full = np.concatenate([np.zeros((F, order), np.int64), res], axis=1).reshape(F, parts, ps)
    valid = np.ones((parts, ps), bool)
    valid[0, :order] = False
    u = ((full << 1) ^ (full >> 63)).astype(np.int64)
    cnt = valid.sum(1)
    mean = (u * valid).sum(2) / np.maximum(cnt, 1)
    k = np.clip(np.floor(np.log2(np.maximum(mean, 1.0))).astype(np.int64), 0, kmax)
    esc = np.zeros((F, parts), bool)
    if cfg["escape"] is True:
        esc[:] = True
    elif cfg["escape"] == "odd":
        esc[:, 1::2] = True
    ew = _signed_width(np.where(valid, full, 0), axis=2)                      # [F, parts]
    if np.any(esc & (ew > 31)):
        raise ValueError("escape partition wider than 31 bits")
    add(1 if rice2 else 0, 2)
    add(p, 4)
    V_part = np.where(esc, escape, k)
    kk = k[:, :, None]
    q = np.where(valid & ~esc[:, :, None], u >> kk, 0)
    code_v = np.where(esc[:, :, None], full & ((1 << ew[:, :, None]) - 1), (1 << kk) | (u & ((1 << kk) - 1)))
    code_w = np.where(esc[:, :, None], ew[:, :, None], kk + 1)
    code_v = np.where(valid, code_v, 0)
    code_w = np.where(valid, code_w, 0)
    # per partition: parameter, escape width, then (zero run, code) per residual
    head_v = np.stack([V_part, ew], axis=2)
    head_w = np.stack([np.full_like(V_part, pbits), np.where(esc, 5, 0)], axis=2)
    body_v = np.stack([np.zeros_like(q), code_v], axis=3).reshape(F, parts, 2 * ps)
    body_w = np.stack([q, code_w], axis=3).reshape(F, parts, 2 * ps)
    add(np.concatenate([head_v, body_v], axis=2).reshape(F, -1), np.concatenate([head_w, body_w], axis=2).reshape(F, -1))


def _pack(values: np.ndarray, widths: np.ndarray, starts: np.ndarray, nbytes: int) -> np.ndarray:
    """OR fields (value < 2^width, width <= 56 unless value == 0) into a byte array at bit positions `starts`."""
    nz = (values != 0) & (widths > 0)
    v, w, p = values[nz].astype(np.uint64), widths[nz], starts[nz]
    if np.any(w > 56):
        raise ValueError("field wider than 56 bits")
    shifted = v << (64 - (p & 7) - w).astype(np.uint64)
    b = (p >> 3).astype(np.int64)
    out = np.zeros(nbytes + 8, np.float64)
    for j in range(8):
        lane = ((shifted >> np.uint64(56 - 8 * j)) & np.uint64(0xFF)).astype(np.float64)
        out += np.bincount(b + j, weights=lane, minlength=nbytes + 8)[:nbytes + 8]
    return out[:nbytes].astype(np.uint8)


def _crc16_rows(buf: np.ndarray, starts: np.ndarray, lengths: np.ndarray) -> np.ndarray:
    crc = np.zeros(len(starts), np.int64)
    for j in range(int(lengths.max()) if len(lengths) else 0):
        live = j < lengths
        b = buf[np.minimum(starts + j, len(buf) - 1)].astype(np.int64)
        nxt = ((crc << 8) & 0xFFFF) ^ CRC16_TABLE[((crc >> 8) ^ b) & 0xFF]
        crc = np.where(live, nxt, crc)
    return crc


def encode(samples, bps: int, sample_rate: int, block_size: int = 4096, *, subframe: str = "lpc", order: int = 8,
           precision: int = 12, shift=None, rice2: bool = False, partition_order=None, escape=False, wasted: bool = True,
           stereo: str = "auto", blocks=None, bs_code=None, rate_code=None, metadata=(), total_samples=None,
           id3: bytes = None) -> bytes:
    """`samples` [N, C] integers in bps-bit range -> a .flac file.

    subframe "constant" / "verbatim" / "fixed" (order 0..4) / "lpc" (order 1..32, `precision` 1..15, `shift` 0..15 or
    None = chosen per frame from the coefficients); rice2 = 5-bit Rice parameters; partition_order None = chosen; escape
    False / True (every partition) / "odd" (odd partitions); wasted = detect wasted bits; stereo "independent" /
    "left_side" / "side_right" / "mid_side" ("auto" = mid_side for two channels); blocks = list of block sizes (variable
    blocking, coded sample numbers) instead of fixed `block_size` (coded frame numbers, short last frame); bs_code "8bit" /
    "16bit" forces the header's explicit block-size codes 6 / 7; rate_code forces 0 / 12 / 13 / 14; metadata = extra
    (type, body) blocks after STREAMINFO; total_samples overrides STREAMINFO's count (0 = unknown); id3 = an ID3v2 payload
    to put in front."""
    x = np.asarray(samples, dtype=np.int64)
    if x.ndim == 1:
        x = x[:, None]
    N, C = x.shape
    if not 1 <= C <= 8 or bps not in BPS_CODES and not 4 <= bps <= 32:
        raise ValueError("unsupported stream")
    if stereo == "auto":
        stereo = "mid_side" if C == 2 else "independent"
    assign = {"independent": C - 1, "left_side": 8, "side_right": 9, "mid_side": 10}[stereo]
    if assign >= 8 and C != 2:
        raise ValueError("stereo decorrelation needs two channels")
    variable = blocks is not None
    sizes = list(blocks) if variable else [block_size] * (N // block_size) + ([N % block_size] if N % block_size else [])
    if sum(sizes) != N or any(not 1 <= s <= 65535 for s in sizes):
        raise ValueError("block sizes must cover the samples")
    firsts = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64) if sizes else np.zeros(0, np.int64)
    cfg = dict(subframe=subframe, order=order, precision=precision, shift=shift, rice2=rice2, partition_order=partition_order,
               escape=escape, wasted=wasted)
    if subframe == "fixed" and not 0 <= order <= 4 or subframe == "lpc" and not (1 <= order <= 32 and 1 <= precision <= 15):
        raise ValueError("invalid predictor")

    # channels as coded
    if assign == 8:
        chans, depths = [x[:, 0], x[:, 0] - x[:, 1]], [bps, bps + 1]
    elif assign == 9:
        chans, depths = [x[:, 0] - x[:, 1], x[:, 1]], [bps + 1, bps]
    elif assign == 10:
        chans, depths = [(x[:, 0] + x[:, 1]) >> 1, x[:, 0] - x[:, 1]], [bps, bps + 1]
    else:
        chans, depths = [x[:, c] for c in range(C)], [bps] * C

    # frame headers
    headers = []
    for f, (first, bs) in enumerate(zip(firsts, sizes)):
        code, tail = BLOCK_SIZE_CODES.get(bs), b""
        if bs_code == "8bit" or (code is None and bs <= 256 and bs_code is None):
            code, tail = 6, bytes([bs - 1])
        elif bs_code == "16bit" or code is None:
            code, tail = 7, struct.pack(">H", bs - 1)
        rc = rate_code if rate_code is not None else RATE_CODES.get(sample_rate)
        if rc is None:
            rc = 12 if sample_rate % 1000 == 0 and sample_rate // 1000 < 256 else 13 if sample_rate < 65536 else 14
        rtail = {12: lambda: bytes([sample_rate // 1000]), 13: lambda: struct.pack(">H", sample_rate),
                 14: lambda: struct.pack(">H", sample_rate // 10)}.get(rc, lambda: b"")()
        h = bytes([0xFF, 0xF8 | variable, (code << 4) | rc, (assign << 4) | (BPS_CODES.get(bps, 0) << 1)])
        h += _utf8(int(first) if variable else f) + tail + rtail
        headers.append(h + bytes([crc8(h)]))

    # subframe fields, grouped by block size; every frame's bit length
    groups = {}
    for f, bs in enumerate(sizes):
        groups.setdefault(bs, []).append(f)
    frame_bits = np.zeros(len(sizes), np.int64)
    fields = []
    for bs, idx in groups.items():
        idx = np.array(idx)
        V, W = [], []
        gcfg = dict(cfg, subframe="verbatim") if subframe in ("fixed", "lpc") and bs <= order else cfg   # a short last frame
        for ch, depth in zip(chans, depths):
            X = ch[firsts[idx][:, None] + np.arange(bs)[None, :]]
            v, w = _subframe_fields(X, depth, gcfg)
            V += v
            W += w
        V, W = np.concatenate(V, axis=1), np.concatenate(W, axis=1)
        hl = np.array([len(headers[f]) for f in idx]) * 8
        frame_bits[idx] = hl + W.sum(1)
        fields.append((idx, hl, V, W))
    frame_bytes = (frame_bits + 7) // 8 + 2
    starts = np.concatenate([[0], np.cumsum(frame_bytes)[:-1]]).astype(np.int64) if len(sizes) else np.zeros(0, np.int64)
    total = int(frame_bytes.sum())
    vals, wids, poss = [], [], []
    for idx, hl, V, W in fields:
        pos = starts[idx][:, None] * 8 + hl[:, None] + np.cumsum(W, axis=1) - W
        vals.append(V.reshape(-1))
        wids.append(W.reshape(-1))
        poss.append(pos.reshape(-1))
    buf = _pack(np.concatenate(vals), np.concatenate(wids), np.concatenate(poss), total) if vals else np.zeros(0, np.uint8)
    for f, h in enumerate(headers):
        buf[starts[f]:starts[f] + len(h)] = np.frombuffer(h, np.uint8)
    crc = _crc16_rows(buf, starts, frame_bytes - 2)
    buf[starts + frame_bytes - 2] = (crc >> 8).astype(np.uint8)
    buf[starts + frame_bytes - 1] = (crc & 0xFF).astype(np.uint8)

    # STREAMINFO + metadata
    body_sizes = sizes[:-1] if len(sizes) > 1 else sizes
    si = (min(body_sizes) if variable else block_size) if sizes else block_size
    sx = (max(sizes) if variable else block_size) if sizes else block_size
    ts = N if total_samples is None else total_samples
    packed = struct.pack(">HH", si, sx) + int(frame_bytes.min() if len(sizes) else 0).to_bytes(3, "big")
    packed += int(frame_bytes.max() if len(sizes) else 0).to_bytes(3, "big")
    packed += ((sample_rate << 44) | ((C - 1) << 41) | ((bps - 1) << 36) | ts).to_bytes(8, "big") + md5(x, bps)
    blocks_md = [(STREAMINFO, packed)] + list(metadata)
    out = b"fLaC"
    for i, (t, body) in enumerate(blocks_md):
        out += bytes([(0x80 if i == len(blocks_md) - 1 else 0) | t]) + len(body).to_bytes(3, "big") + body
    if id3 is not None:
        n = len(id3)
        out = b"ID3\x04\x00\x00" + bytes([(n >> 21) & 0x7F, (n >> 14) & 0x7F, (n >> 7) & 0x7F, n & 0x7F]) + id3 + out
    return out + buf.tobytes()
