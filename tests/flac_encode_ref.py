"""TEST INFRASTRUCTURE ONLY -- the exact-cost FLAC encoder in numpy: the byte-for-byte reference of the device encoder
(`ar_flac_encode`, csrc/flac_encode.cu).  Every choice is defined and integer-only: fixed blocking, per channel the fewest
exact bits of CONSTANT / FIXED 0..4 (exact Rice / Rice2 and partition-order search) / VERBATIM with wasted bits, and for two
channels the cheapest stereo mode.  It packs frames with the bit packer, CRC-16 rows and MD5 of `oracle.flac` and decodes
through `oracle.flac.decode`.

The frame-header sample-rate code here falls back to 0 (rate from STREAMINFO) for a rate >= 65536 that is not a whole
number of tens of Hz; `oracle.flac.encode` writes code 14 there, which states a different rate (none of its vectors uses
such a rate).
"""
import struct

import numpy as np

from oracle.flac import BLOCK_SIZE_CODES, BPS_CODES, RATE_CODES, STREAMINFO, _crc16_rows, _pack, _utf8, crc8, md5


def _frame_header(number: int, bs: int, sample_rate: int, assign: int, bps: int) -> bytes:
    """Frame header (fixed blocking) with its CRC-8.  Block-size code from the table, else an explicit 8-bit (bs <= 256)
    or 16-bit field; sample-rate code from the table, else 12 / 13 / 14 when the rate is exact in that field, else 0
    (the rate comes from STREAMINFO)."""
    code, tail = BLOCK_SIZE_CODES.get(bs), b""
    if code is None:
        code, tail = (6, bytes([bs - 1])) if bs <= 256 else (7, struct.pack(">H", bs - 1))
    rc, rtail = RATE_CODES.get(sample_rate), b""
    if rc is None:
        if sample_rate % 1000 == 0 and sample_rate // 1000 < 256:
            rc, rtail = 12, bytes([sample_rate // 1000])
        elif sample_rate < 65536:
            rc, rtail = 13, struct.pack(">H", sample_rate)
        elif sample_rate % 10 == 0 and sample_rate // 10 < 65536:
            rc, rtail = 14, struct.pack(">H", sample_rate // 10)
        else:
            rc = 0
    h = bytes([0xFF, 0xF8, (code << 4) | rc, (assign << 4) | (BPS_CODES[bps] << 1)]) + _utf8(number) + tail + rtail
    return h + bytes([crc8(h)])


def _wasted_bits(X: np.ndarray, depth: int) -> np.ndarray:
    """[F] trailing zeros shared by every sample of each row, capped at depth - 1 (0 for an all-zero row)"""
    orr = np.bitwise_or.reduce(X, axis=1)
    low = orr & -orr
    k = np.where(orr != 0, np.log2(np.where(low > 0, low, 1).astype(np.float64)).astype(np.int64), 0)
    return np.minimum(k, depth - 1)


def _frames(headers: list, fields: list, frame_bits: np.ndarray):
    """(frame section uint8, bytes per frame): every frame's header, its subframe fields (frame indices, header bits,
    values [F, K], widths [F, K]) packed after it, zero padding to a byte boundary and the CRC-16."""
    frame_bytes = (frame_bits + 7) // 8 + 2
    starts = np.concatenate([[0], np.cumsum(frame_bytes)[:-1]]).astype(np.int64) if len(headers) else np.zeros(0, np.int64)
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
    return buf, frame_bytes


def _streaminfo(min_block, max_block, frame_bytes, sample_rate, C, bps, total_samples, md5sum) -> bytes:
    packed = struct.pack(">HH", min_block, max_block) + int(frame_bytes.min() if len(frame_bytes) else 0).to_bytes(3, "big")
    packed += int(frame_bytes.max() if len(frame_bytes) else 0).to_bytes(3, "big")
    return packed + ((sample_rate << 44) | ((C - 1) << 41) | ((bps - 1) << 36) | total_samples).to_bytes(8, "big") + md5sum


SEARCH_BPS = (16, 24)
SEARCH_MAX_BLOCK = 4608          # the largest block size the streamable subset allows at every sample rate
SEARCH_MAX_RATE = 655350         # the largest rate a frame header can state exactly (code 14: tens of Hz in 16 bits)
_RICE_METHODS = ((4, 14), (5, 30))   # (parameter bits, largest k) of RICE and RICE2; escape codes are never chosen


def check_search_args(channels: int, n: int, bps: int, sample_rate: int, block_size: int) -> None:
    """The streams encode_search (and ar_flac_encode) write: 1..8 channels, 16 or 24 bits, at least one sample."""
    if not 1 <= channels <= 8:
        raise ValueError(f"FLAC encoder: {channels} channels (1..8 supported)")
    if bps not in SEARCH_BPS:
        raise ValueError(f"FLAC encoder: {bps} bits per sample (16 or 24 supported)")
    if not 1 <= sample_rate <= SEARCH_MAX_RATE:
        raise ValueError(f"FLAC encoder: sample rate {sample_rate} Hz (1..{SEARCH_MAX_RATE} supported)")
    if not 16 <= block_size <= SEARCH_MAX_BLOCK:
        raise ValueError(f"FLAC encoder: block size {block_size} (16..{SEARCH_MAX_BLOCK} supported)")
    if n < 1:
        raise ValueError("FLAC encoder: no samples")


def _leaf_order(bs: int) -> int:
    """finest partition order: the largest p <= 8 with bs % 2^p == 0"""
    p = 0
    while p < 8 and bs % (2 << p) == 0:
        p += 1
    return p


def _rice_search(u: np.ndarray, order: int):
    """Exact Rice coding of zigzag residuals u [F, bs] (zeros at the `order` warm-up positions): (bits [F], method [F],
    partition order [F], k per partition [F, 2^P]).  Σ(u >> k) is summed once per finest leaf and k, then up the tree;
    ties go to the smaller method, then the smaller partition order, then the smaller k."""
    F, bs = u.shape
    P = _leaf_order(bs)
    S = np.stack([(u >> k).reshape(F, 1 << P, -1).sum(2) for k in range(31)], axis=2)      # [F, leaves, 31]
    n_leaf = (np.arange(bs) >= order).reshape(1 << P, -1).sum(1)
    bits = np.full(F, np.iinfo(np.int64).max, np.int64)
    method, porder = np.zeros(F, np.int64), np.zeros(F, np.int64)
    kk = np.zeros((F, 1 << P), np.int64)
    for m, (pbits, kmax) in enumerate(_RICE_METHODS):
        ks = np.arange(kmax + 1)
        for p in range(P + 1):
            if (bs >> p) < order:
                continue
            cost = S.reshape(F, 1 << p, -1, 31).sum(2)[:, :, :kmax + 1] + n_leaf.reshape(1 << p, -1).sum(1)[None, :, None] * (ks + 1)
            b = 6 + (pbits + cost.min(2)).sum(1)
            better = b < bits
            bits, method, porder = np.where(better, b, bits), np.where(better, m, method), np.where(better, p, porder)
            kk[better] = 0
            kk[better, :1 << p] = cost.argmin(2)[better]
    return bits, method, porder, kk


def _search_subframe(X: np.ndarray, depth: int):
    """The cheapest subframe of every row of X [F, bs] at `depth` bits: (bits [F], values [F, K], widths [F, K]).
    Candidates in tie-break order: CONSTANT (all samples equal), FIXED orders 0..4 (order <= bs), VERBATIM; wasted bits
    apply to each."""
    F, bs = X.shape
    w = _wasted_bits(X, depth)
    Xs = X >> w[:, None]
    ed = depth - w
    head = 8 + w
    big = np.iinfo(np.int64).max
    best = np.where(np.all(Xs == Xs[:, :1], axis=1), head + ed, big)
    typ = np.zeros(F, np.int64)                                        # 0 CONSTANT, 1 VERBATIM, 8 + o FIXED order o
    method, porder = np.zeros(F, np.int64), np.zeros(F, np.int64)
    kk = np.zeros((F, 1 << _leaf_order(bs)), np.int64)
    U = np.zeros((F, bs), np.int64)
    for o in range(min(4, bs) + 1):
        r = np.zeros((F, bs), np.int64)
        r[:, o:] = np.diff(Xs, n=o, axis=1)                           # FIXED order o predicts with the o-th difference
        if np.any(np.abs(r) >= 1 << 31):
            raise ValueError("residual outside the 32-bit range")
        u = (r << 1) ^ (r >> 63)
        rb, rm, rp, rk = _rice_search(u, o)
        b = head + o * ed + rb
        better = b < best
        best, typ = np.where(better, b, best), np.where(better, 8 + o, typ)
        method, porder = np.where(better, rm, method), np.where(better, rp, porder)
        kk[better], U[better] = rk[better], u[better]
    b = head + bs * ed
    better = b < best
    best, typ = np.where(better, b, best), np.where(better, 1, typ)

    mask = ((1 << ed) - 1)[:, None]
    fixed = typ >= 8
    order = np.where(fixed, typ - 8, 0)
    V, W = [], []

    def add(v, wid):
        wid = np.asarray(wid, np.int64)
        V.append(np.broadcast_to(np.asarray(v, np.int64), wid.shape))
        W.append(wid)

    add(((typ << 1) | (w > 0))[:, None], np.full((F, 1), 8))
    add(1, w[:, None])                                  # w - 1 zeros and a one
    add(Xs[:, :1] & mask, np.where(typ == 0, ed, 0)[:, None])
    add(Xs & mask, np.where(typ == 1, ed, 0)[:, None] * np.ones((1, bs), np.int64))
    warm = np.concatenate([Xs, np.zeros((F, 4), np.int64)], axis=1)[:, :4]
    add(warm & mask, np.where(fixed[:, None] & (np.arange(4)[None, :] < order[:, None]), ed[:, None], 0))
    add(method[:, None], np.where(fixed, 2, 0)[:, None])
    add(porder[:, None], np.where(fixed, 4, 0)[:, None])
    i = np.arange(bs)[None, :]
    ps = (bs >> porder)[:, None]
    k = np.take_along_axis(kk, i // ps, axis=1)
    live = fixed[:, None] & (i >= order[:, None])
    param_w = np.where(fixed[:, None] & (i % ps == 0), 4 + method[:, None], 0)
    zeros_w = np.where(live, U >> k, 0)
    code_v = np.where(live, (1 << k) | (U & ((1 << k) - 1)), 0)
    code_w = np.where(live, k + 1, 0)
    add(np.stack([k, np.zeros_like(k), code_v], axis=2).reshape(F, -1),
        np.stack([param_w, zeros_w, code_w], axis=2).reshape(F, -1))
    V, W = np.concatenate(V, axis=1), np.concatenate(W, axis=1)
    assert np.array_equal(W.sum(1), best)
    return best, V, W


def encode_search(samples, bps: int, sample_rate: int, block_size: int = 4096) -> bytes:
    """`samples` [N, C] integers in bps-bit range -> a .flac file, every choice defined and integer-only: fixed blocking
    (frame numbers, short last frame), per channel the cheapest of CONSTANT / FIXED 0..4 with an exact Rice / Rice2 and
    partition-order search / VERBATIM, and for two channels the cheapest of independent, left/side, side/right and
    mid/side (ties to the lower assignment code).  STREAMINFO (min = max block = block_size, min / max frame bytes, MD5)
    is the only metadata block.  Vectorised over frames; this is the byte-for-byte reference of ar_flac_encode."""
    x = np.asarray(samples, dtype=np.int64)
    if x.ndim == 1:
        x = x[:, None]
    N, C = x.shape
    check_search_args(C, N, bps, sample_rate, block_size)
    if x.min() < -(1 << (bps - 1)) or x.max() >= 1 << (bps - 1):
        raise ValueError(f"samples outside the {bps}-bit range")
    sizes = [block_size] * (N // block_size) + ([N % block_size] if N % block_size else [])
    firsts = np.arange(len(sizes), dtype=np.int64) * block_size
    assign = np.full(len(sizes), C - 1, np.int64)
    frame_bits = np.zeros(len(sizes), np.int64)
    fields = []
    for bs in sorted(set(sizes)):
        idx = np.array([f for f, s in enumerate(sizes) if s == bs])
        rows = firsts[idx][:, None] + np.arange(bs)[None, :]
        chans = [x[:, c][rows] for c in range(C)]
        if C == 2:
            L, R = chans
            (bl, vl, wl), (br, vr, wr) = _search_subframe(L, bps), _search_subframe(R, bps)
            (bsd, vs, ws), (bm, vm, wm) = _search_subframe(L - R, bps + 1), _search_subframe((L + R) >> 1, bps)
            pick = np.stack([bl + br, bl + bsd, bsd + br, bm + bsd], axis=1).argmin(1)    # 1, 8, 9, 10 in that order
            assign[idx] = np.array([1, 8, 9, 10])[pick]
            sel = lambda arrs: np.choose(pick[:, None], arrs)                           # noqa: E731
            V = np.concatenate([sel([vl, vl, vs, vm]), sel([vr, vs, vr, vs])], axis=1)
            W = np.concatenate([sel([wl, wl, ws, wm]), sel([wr, ws, wr, ws])], axis=1)
        else:
            parts = [_search_subframe(ch, bps) for ch in chans]
            V = np.concatenate([p[1] for p in parts], axis=1)
            W = np.concatenate([p[2] for p in parts], axis=1)
        fields.append((idx, V, W))
    headers = [_frame_header(f, bs, sample_rate, int(assign[f]), bps) for f, bs in enumerate(sizes)]
    packed_fields = []
    for idx, V, W in fields:
        hl = np.array([len(headers[f]) for f in idx]) * 8
        frame_bits[idx] = hl + W.sum(1)
        packed_fields.append((idx, hl, V, W))
    buf, frame_bytes = _frames(headers, packed_fields, frame_bits)
    si = _streaminfo(block_size, block_size, frame_bytes, sample_rate, C, bps, N, md5(x, bps))
    return b"fLaC" + bytes([0x80 | STREAMINFO]) + len(si).to_bytes(3, "big") + si + buf.tobytes()


def quantise(x: np.ndarray, bps: int) -> np.ndarray:
    """Planar float [C, N] -> [N, C] integers as the device encoder quantises: rint_even(clamp(x, -1, 1) * (2^(bps-1) - 1))
    with an fp32 multiply, NaN -> 0."""
    x = np.nan_to_num(np.asarray(x, np.float32), nan=0.0, posinf=np.inf, neginf=-np.inf)
    return np.round(np.clip(x, -1.0, 1.0) * np.float32((1 << (bps - 1)) - 1)).astype(np.int64).T
