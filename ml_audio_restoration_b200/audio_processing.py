"""Audio helpers on the restoration path (reference: src/utils/audio_processing.py).

What inference needs -- `normalize_audio` (device kernel, no host syncs), `chunk_audio` (the reference's chunk
vocabulary), small WAV load/save helpers and a GPU FLAC decoder and encoder so `restore_audio` works without `soundfile` --
plus the synthetic degradation generator `simulate_vinyl_artifacts` (SURVEY.md 8f n4) that produces the path's
78 rpm-like inputs, with its pops and zero-phase Butterworth filters on the GPU.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import wave

import numpy as np
import torch

from . import _lib


def normalize_audio(audio: torch.Tensor, target_db: float = -20.0) -> torch.Tensor:
    """RMS-normalise to `target_db`, then peak-limit to 1.0 (audio_processing.py:58-87).

    CUDA tensors only: two stream-ordered kernels (reduce, scale) with the gain computed on the
    device, instead of the reference's `if rms == 0` / `if max_val > 1.0` host round trips.
    Returns a new tensor; a silent input comes back unchanged.
    """
    if not audio.is_cuda:
        raise RuntimeError("normalize_audio: input must be a CUDA tensor -- this build has no CPU fallback")
    out = audio.to(torch.float32).contiguous().clone()
    if out.numel() == 0:
        raise RuntimeError("normalize_audio: empty audio")
    with torch.cuda.device(out.device):
        scratch = torch.empty(_lib.NORMALIZE_SCRATCH_BYTES, dtype=torch.uint8, device=out.device)
        _lib.check(_lib.lib().ar_normalize(out.data_ptr(), out.numel(), float(target_db), scratch.data_ptr(),
                                           torch.cuda.current_stream(out.device).cuda_stream))
    return out


def chunk_audio(audio: torch.Tensor, chunk_size: int, overlap: int = 0) -> list:
    """Views of `audio[..., N]` of length `chunk_size` every `chunk_size - overlap` samples.

    Mirrors the reference helper (audio_processing.py:229-253) including its tail rule: when
    N is not a multiple of the stride one extra chunk holding the LAST `chunk_size` samples is
    appended (so a few samples can be dropped when N % stride == 0 but (N - chunk_size) % stride != 0,
    and a single short chunk comes back when N < chunk_size).  The batched GPU pipeline does
    not use this function; it uses the gap-free plan of `inference.plan_chunks`.
    """
    n = audio.shape[-1]
    stride = chunk_size - overlap
    starts = list(range(0, n - chunk_size + 1, stride))
    pieces = [audio[..., s:s + chunk_size] for s in starts]
    if n % stride != 0:
        pieces.append(audio[..., -chunk_size:])
    return pieces


# ----------------------------------------------------------------------------- synthetic 78 rpm degradation
POP_DTYPE = np.dtype([("loc", "<i8"), ("length", "<i4"), ("has_resonance", "<i4"), ("amp_signed", "<f8"), ("amp", "<f8"),
                      ("tau", "<f8"), ("omega", "<f8")])      # == ar_pop_t (include/audiorestore.h)


def butter(order: int, wn: float, btype: str = "low"):
    """(b, a) float64 arrays -- `scipy.signal.butter(order, wn, btype)` for 'low' / 'high' (host design, `ar_butter`)."""
    if btype not in ("low", "high"):
        raise ValueError(f"butter: unsupported btype {btype!r}")
    b = (C.c_double * (order + 1))()
    a = (C.c_double * (order + 1))()
    _lib.check(_lib.lib().ar_butter(int(order), float(wn), int(btype == "high"), b, a))
    return np.array(b[:]), np.array(a[:])


def filtfilt(b, a, x: torch.Tensor, scale: float = 1.0, add1: torch.Tensor = None, add2: torch.Tensor = None) -> torch.Tensor:
    """float32 `scipy.signal.filtfilt(b, a, row)` of every row of `scale * x (+ add1) (+ add2)` ([rows, n] CUDA float32):
    the zero-phase forward/backward float64 IIR the reference runs per channel on the CPU (audio_processing.py:197-199,
    209-211, 221-223), as six block-parallel launches (`ar_filtfilt`).  Raises ValueError when n <= 3 * len(b) like scipy."""
    if not x.is_cuda or x.dim() != 2 or x.dtype != torch.float32:
        raise RuntimeError("filtfilt: expected a [rows, n] float32 CUDA tensor -- this build has no CPU fallback")
    b = np.ascontiguousarray(b, dtype=np.float64)
    a = np.ascontiguousarray(a, dtype=np.float64)
    if b.ndim != 1 or b.shape != a.shape or not 2 <= len(b) <= 5:
        raise ValueError("filtfilt: b and a must be 1-D, of equal length 2..5 (filter order 1..4)")
    x = x.contiguous()
    adds = []
    for t in (add1, add2):
        if t is not None:
            if t.shape != x.shape or t.dtype != torch.float32 or t.device != x.device:
                raise RuntimeError("filtfilt: addends must match x in shape, dtype and device")
            t = t.contiguous()
        adds.append(t)
    rows, n = x.shape
    L = _lib.lib()
    need = C.c_size_t()
    _lib.check(L.ar_filtfilt_workspace_bytes(rows, n, len(b) - 1, C.byref(need)))
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        ws = torch.empty(need.value, dtype=torch.uint8, device=x.device)
        _lib.check(L.ar_filtfilt(x.data_ptr(), float(scale), adds[0].data_ptr() if adds[0] is not None else None,
                                 adds[1].data_ptr() if adds[1] is not None else None, y.data_ptr(), rows, n,
                                 b.ctypes.data_as(C.POINTER(C.c_double)), a.ctypes.data_as(C.POINTER(C.c_double)),
                                 len(b) - 1, ws.data_ptr(), need.value, torch.cuda.current_stream(x.device).cuda_stream))
    return y


def plan_vinyl_artifacts(num_samples: int, sample_rate: int, impulse_rate: float = 10.0, impulse_amplitude=(0.1, 0.5),
                         surface_noise_level=(0.015, 0.03), crackle_level=(0.01, 0.02), add_rumble: bool = True,
                         add_rolloff: bool = True) -> dict:
    """Host half of `simulate_vinyl_artifacts`: draws every scalar the reference draws from the global `np.random`
    generator, in the reference's order (audio_processing.py:152, 158, 161-165, 171, 182, 191, 204, 219), so that
    `np.random.seed(s)` reproduces the reference's levels, pops and roll-off frequency.  Returns
    {surface_level, crackle_level, rumble_level | None, rolloff_hz | None, pops: structured array of POP_DTYPE}."""
    duration = num_samples / sample_rate
    surface = np.random.uniform(*surface_noise_level)
    num_pops = np.random.poisson(int(duration * impulse_rate))
    pops = np.zeros(num_pops, dtype=POP_DTYPE)
    kept = 0
    if num_pops > 0:
        locs = np.random.randint(0, num_samples, num_pops)
        amps = np.random.uniform(*impulse_amplitude, num_pops)
        pols = np.random.choice([-1, 1], num_pops, p=[0.45, 0.55])
        for loc, amp, pol in zip(locs, amps, pols):
            decay_time = np.random.uniform(0.001, 0.003) * (1 + amp)
            length = min(int(sample_rate * decay_time), num_samples - loc)
            if length <= 0:
                continue
            resonant = length > 10
            omega = 2 * np.pi * np.random.uniform(3000, 8000) if resonant else 0.0
            pops[kept] = (loc, length, int(resonant), amp * pol, amp, sample_rate * decay_time * 0.3, omega)
            kept += 1
    crackle = np.random.uniform(*crackle_level)
    rumble = np.random.uniform(0.005, 0.015) if add_rumble else None
    rolloff = np.random.uniform(6000, 8000) if add_rolloff else None
    return {"surface_level": surface, "crackle_level": crackle, "rumble_level": rumble, "rolloff_hz": rolloff,
            "pops": pops[:kept]}


def apply_vinyl_artifacts(audio: torch.Tensor, sample_rate: int, plan: dict, surface: torch.Tensor, crackle: torch.Tensor,
                          rumble: torch.Tensor = None) -> torch.Tensor:
    """Device half: `audio` [..., n] float32 CUDA, unit-variance noise tensors of the same shape and a plan ->
    degraded audio.  Launches: 1 mix (surface noise + pops), 6 per Butterworth filtfilt (crackle high-pass 2.5 kHz,
    rumble low-pass 100 Hz, roll-off low-pass) with the noise scaling and the `+ crackle + rumble` sums fused into the
    filters' loads."""
    if not audio.is_cuda:
        raise RuntimeError("simulate_vinyl_artifacts: input must be a CUDA tensor -- this build has no CPU fallback")
    shape = audio.shape
    n = shape[-1]
    x = audio.to(torch.float32).reshape(-1, n).contiguous()
    rows = x.shape[0]

    def flat(t):
        if t.shape != shape or not t.is_cuda:
            raise RuntimeError("simulate_vinyl_artifacts: noise tensors must match the audio tensor")
        return t.to(torch.float32).reshape(rows, n).contiguous()

    L = _lib.lib()
    pops = np.ascontiguousarray(plan["pops"], dtype=POP_DTYPE)
    mixed = torch.empty_like(x)
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream(x.device).cuda_stream
        pops_dev = None
        if len(pops):
            pops_dev = torch.from_numpy(pops.view(np.uint8).copy()).to(x.device)
        _lib.check(L.ar_vinyl_mix(x.data_ptr(), flat(surface).data_ptr(), float(plan["surface_level"]),
                                  pops_dev.data_ptr() if pops_dev is not None else None, len(pops), int(sample_rate),
                                  mixed.data_ptr(), rows, n, stream))
        nyquist = sample_rate / 2
        crk = filtfilt(*butter(4, 2500 / nyquist, "high"), flat(crackle), scale=float(plan["crackle_level"]))
        rmb = None
        if plan["rumble_level"] is not None:
            rmb = filtfilt(*butter(4, 100 / nyquist, "low"), flat(rumble), scale=float(plan["rumble_level"]))
        if plan["rolloff_hz"] is not None:
            out = filtfilt(*butter(3, plan["rolloff_hz"] / nyquist, "low"), mixed, add1=crk, add2=rmb)
        else:
            out = torch.empty_like(x)
            _lib.check(L.ar_vinyl_sum(mixed.data_ptr(), crk.data_ptr(), rmb.data_ptr() if rmb is not None else None,
                                      out.data_ptr(), out.numel(), stream))
    return out.reshape(shape)


def add_noise(audio: torch.Tensor, noise_level: float = 0.01) -> torch.Tensor:
    """`audio + randn_like(audio) * noise_level` (audio_processing.py:107-119) -- the pop-free case of `ar_vinyl_mix`."""
    if not audio.is_cuda:
        raise RuntimeError("add_noise: input must be a CUDA tensor -- this build has no CPU fallback")
    x = audio.to(torch.float32).contiguous()
    noise = torch.randn_like(x)
    y = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().ar_vinyl_mix(x.data_ptr(), noise.data_ptr(), float(noise_level), None, 0, 1, y.data_ptr(), 1,
                                           x.numel(), torch.cuda.current_stream(x.device).cuda_stream))
    return y


def simulate_vinyl_artifacts(audio: torch.Tensor, sample_rate: int, impulse_rate: float = 10.0,
                             impulse_amplitude=(0.1, 0.5), surface_noise_level=(0.015, 0.03),
                             crackle_level=(0.01, 0.02), add_rumble: bool = True, add_rolloff: bool = True) -> torch.Tensor:
    """Shellac-record artifacts for a clean `(channels, samples)` CUDA tensor -- same signature, same defaults and the
    same use of the two global generators as the reference (audio_processing.py:122-226): three `torch.randn_like`
    draws on the audio's device (surface, crackle, rumble) and the `np.random` plan of `plan_vinyl_artifacts`."""
    surface = torch.randn_like(audio)
    crackle = torch.randn_like(audio)
    rumble = torch.randn_like(audio) if add_rumble else None
    plan = plan_vinyl_artifacts(audio.shape[-1], sample_rate, impulse_rate, impulse_amplitude, surface_noise_level,
                                crackle_level, add_rumble, add_rolloff)
    return apply_vinyl_artifacts(audio, sample_rate, plan, surface, crackle, rumble)


# ----------------------------------------------------------------------------- minimal WAV I/O
def _read_wav(path: str):
    """Host read of an audio file as `[C, N]` float32 (the reference's `sf.read(..., dtype='float32')`,
    audio_processing.py:24): soundfile when it is installed, else FLAC through the device decoder (`decode_flac_cuda`,
    returned on the host) and WAV through the RIFF/WAVE reader of this module (8 / 16 / 24 / 32-bit integer PCM,
    32 / 64-bit IEEE float, plain or WAVE_FORMAT_EXTENSIBLE)."""
    try:
        import soundfile as sf  # optional
        data, sr = sf.read(path, always_2d=True, dtype="float32")
        return torch.from_numpy(np.ascontiguousarray(data.T)), sr
    except ImportError:
        pass
    if is_flac(path):                                             # decoded on the GPU (ar_flac_decode)
        info = flac_info(path)
        return decode_flac_cuda(_upload_frames(path, info, "cuda"), info).cpu(), info["sample_rate"]
    fmt, nch, sr, frames, offset = wav_info(path)
    width = _PCM_WIDTH[fmt]
    with open(path, "rb") as f:
        f.seek(offset)
        raw = f.read(frames * nch * width)
    if fmt == _PCM_S16:
        a = np.frombuffer(raw, dtype="<i2").astype(np.float32) / 32768.0
    elif fmt == _PCM_S32:
        a = np.frombuffer(raw, dtype="<i4").astype(np.float32) / 2147483648.0
    elif fmt == _PCM_S24:
        b = np.frombuffer(raw, dtype=np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        v = np.where(v & 0x800000, v - (1 << 24), v)
        a = v.astype(np.float32) / 8388608.0
    elif fmt == _PCM_U8:
        a = (np.frombuffer(raw, dtype=np.uint8).astype(np.float32) - 128.0) / 128.0
    elif fmt == _PCM_F32:
        a = np.frombuffer(raw, dtype="<f4").astype(np.float32)
    else:
        a = np.frombuffer(raw, dtype="<f8").astype(np.float32)
    return torch.from_numpy(np.ascontiguousarray(a.astype(np.float32).reshape(-1, nch).T)), sr


def load_audio(file_path: str, sample_rate: int = 22050, mono: bool = True):
    """(audio [C,N] float32, sample_rate) -- audio_processing.py:10-42 (host tensors, as the reference returns)."""
    audio, sr = _read_wav(file_path)
    if mono and audio.shape[0] > 1:
        audio = audio.mean(dim=0, keepdim=True)
    if sr != sample_rate:
        import torchaudio.functional as AF
        audio = AF.resample(audio, sr, sample_rate)
    return audio, sample_rate


def resample_mono_cuda(audio: torch.Tensor, sr: int, sample_rate: int = 22050) -> torch.Tensor:
    """`[C,N]` float32 CUDA -> `[1, ceil(sample_rate*N/sr)]`: the mono mix (`torch.mean(dim=0)`, audio_processing.py:33)
    fused with `torchaudio.transforms.Resample(sr, sample_rate)` (:38) in one kernel (`ar_resample_mono`)."""
    if not audio.is_cuda or audio.dim() != 2:
        raise RuntimeError("resample_mono_cuda: expected a [C,N] CUDA tensor -- this build has no CPU fallback")
    x = audio.to(torch.float32).contiguous()
    L = _lib.lib()
    n_out = C.c_int64()
    _lib.check(L.ar_resample_length(x.shape[1], int(sr), int(sample_rate), C.byref(n_out)))
    y = torch.empty((1, n_out.value), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(L.ar_resample_mono(x.data_ptr(), x.shape[0], x.shape[1], int(sr), int(sample_rate), y.data_ptr(),
                                      n_out.value, torch.cuda.current_stream(x.device).cuda_stream))
    return y


# sample encodings of `ar_pcm_to_float` (include/audiorestore.h AR_PCM_*)
_PCM_U8, _PCM_S16, _PCM_S24, _PCM_S32, _PCM_F32, _PCM_F64 = 1, 2, 3, 4, 5, 6
_PCM_WIDTH = {_PCM_U8: 1, _PCM_S16: 2, _PCM_S24: 3, _PCM_S32: 4, _PCM_F32: 4, _PCM_F64: 8}


def wav_info(path: str):
    """Header of a RIFF/WAVE file: (AR_PCM_* format, channels, sample rate, frames, byte offset of the samples).
    Handles format tags 1 (integer PCM), 3 (IEEE float) and 0xFFFE (WAVE_FORMAT_EXTENSIBLE wrapping either);
    raises RuntimeError for anything else (compressed WAVs, non-WAV containers)."""
    import struct
    with open(path, "rb") as f:
        head = f.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise RuntimeError(f"{path}: not a RIFF/WAVE file")
        fmt = None
        while True:
            hdr = f.read(8)
            if len(hdr) < 8:
                raise RuntimeError(f"{path}: no data chunk")
            cid, size = struct.unpack("<4sI", hdr)
            if cid == b"fmt ":
                body = f.read(size + (size & 1))
                tag, nch, sr, _, align, bits = struct.unpack_from("<HHIIHH", body, 0)
                if tag == 0xFFFE and size >= 26:
                    tag = struct.unpack_from("<H", body, 24)[0]          # first two bytes of the sub-format GUID
                fmt = (tag, nch, sr, align, bits)
            elif cid == b"data":
                if fmt is None:
                    raise RuntimeError(f"{path}: data chunk before fmt chunk")
                offset = f.tell()
                f.seek(0, 2)
                size = min(size, f.tell() - offset)                      # tolerate a truncated / streaming-length header
                break
            else:
                f.seek(size + (size & 1), 1)
    tag, nch, sr, align, bits = fmt
    code = {(1, 8): _PCM_U8, (1, 16): _PCM_S16, (1, 24): _PCM_S24, (1, 32): _PCM_S32, (3, 32): _PCM_F32, (3, 64): _PCM_F64}.get((tag, bits))
    if code is None or nch < 1 or align != nch * bits // 8:
        raise RuntimeError(f"{path}: unsupported WAV encoding (format tag {tag}, {bits} bits)")
    return code, nch, sr, size // align, offset


def decode_pcm_cuda(raw: torch.Tensor, fmt: int, channels: int, frames: int) -> torch.Tensor:
    """Raw interleaved sample bytes (uint8 CUDA tensor) -> planar `[channels, frames]` float32 (`ar_pcm_to_float`)."""
    if not raw.is_cuda or raw.dtype != torch.uint8:
        raise RuntimeError("decode_pcm_cuda: expected a uint8 CUDA tensor -- this build has no CPU fallback")
    planar = torch.empty((channels, frames), dtype=torch.float32, device=raw.device)
    with torch.cuda.device(raw.device):
        _lib.check(_lib.lib().ar_pcm_to_float(raw.data_ptr(), fmt, channels, frames, planar.data_ptr(),
                                              torch.cuda.current_stream(raw.device).cuda_stream))
    return planar


# ----------------------------------------------------------------------------- FLAC
_FLAC_SKIPPED_BLOCKS = (1, 2, 3, 4, 5, 6)     # PADDING, APPLICATION, SEEKTABLE, VORBIS_COMMENT, CUESHEET, PICTURE


def _flac_start(head: bytes) -> int:
    """Offset of the `fLaC` marker: 0, or past a leading ID3v2 tag (10-byte header, syncsafe size, optional footer)."""
    if head[:3] == b"ID3" and len(head) >= 10:
        size = (head[6] << 21) | (head[7] << 14) | (head[8] << 7) | head[9]
        return 10 + size + (10 if head[5] & 0x10 else 0)
    return 0


def is_flac(path: str) -> bool:
    """True when the file's content is a FLAC stream (optionally behind an ID3v2 tag), whatever its extension."""
    with open(path, "rb") as f:
        head = f.read(10)
        f.seek(_flac_start(head))
        return f.read(4) == b"fLaC"


def flac_info(path: str) -> dict:
    """Host parse of a FLAC container (RFC 9639): an optional leading ID3v2 tag, the `fLaC` marker, then the metadata
    blocks -- STREAMINFO required, PADDING / APPLICATION / SEEKTABLE / VORBIS_COMMENT / CUESHEET / PICTURE skipped.
    Returns {channels, bps, sample_rate, total_samples (0 = unknown), min_block, max_block, offset (byte offset of the
    first frame), nbytes (bytes of frame data)}; raises RuntimeError for anything that is not a well-formed FLAC header."""
    import os
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        pos = _flac_start(f.read(10))
        f.seek(pos)
        if f.read(4) != b"fLaC":
            raise RuntimeError(f"{path}: not a FLAC file")
        pos += 4
        info = None
        while True:
            hdr = f.read(4)
            if len(hdr) < 4:
                raise RuntimeError(f"{path}: truncated FLAC metadata block header")
            last, btype, length = hdr[0] >> 7, hdr[0] & 0x7F, int.from_bytes(hdr[1:4], "big")
            pos += 4
            if pos + length > size:
                raise RuntimeError(f"{path}: truncated FLAC metadata block (type {btype})")
            if btype == 0:
                if length != 34 or info is not None:
                    raise RuntimeError(f"{path}: malformed STREAMINFO block")
                b = f.read(34)
                v = int.from_bytes(b[10:18], "big")
                info = {"min_block": int.from_bytes(b[0:2], "big"), "max_block": int.from_bytes(b[2:4], "big"),
                        "sample_rate": v >> 44, "channels": ((v >> 41) & 7) + 1, "bps": ((v >> 36) & 31) + 1,
                        "total_samples": v & ((1 << 36) - 1)}
            elif btype in _FLAC_SKIPPED_BLOCKS or 7 <= btype < 127:
                f.seek(length, 1)
            else:
                raise RuntimeError(f"{path}: invalid FLAC metadata block type {btype}")
            pos += length
            if btype != 0 and info is None:
                raise RuntimeError(f"{path}: FLAC metadata does not start with STREAMINFO")
            if last:
                break
    if info["sample_rate"] == 0 or info["bps"] < 4 or info["min_block"] < 1 or info["max_block"] < info["min_block"]:
        raise RuntimeError(f"{path}: STREAMINFO holds a reserved value (rate {info['sample_rate']}, {info['bps']} bits, "
                           f"block sizes {info['min_block']}..{info['max_block']})")
    info["offset"] = pos
    info["nbytes"] = size - pos
    return info


def _upload_frames(path: str, info: dict, device) -> torch.Tensor:
    """The frame bytes of a FLAC file, read into pinned memory and copied to `device` (uint8)."""
    host = torch.empty(info["nbytes"], dtype=torch.uint8).pin_memory()
    with open(path, "rb") as f:
        f.seek(info["offset"])
        got = f.readinto(host.numpy())
    if got != host.numel():
        raise RuntimeError(f"{path}: file changed while reading")
    return host.to(torch.device(device), non_blocking=True)


def decode_flac_cuda(raw: torch.Tensor, info: dict) -> torch.Tensor:
    """The frame bytes of a FLAC stream (uint8 CUDA tensor, everything after the metadata blocks) and its `flac_info` ->
    planar `[channels, N]` float32, x / 2^(bps-1) as soundfile's float32 read (`ar_flac_decode`; bit-exact for
    bps <= 24).  Raises RuntimeError naming the frame and its byte offset in the file for a malformed stream."""
    if not raw.is_cuda or raw.dtype != torch.uint8 or raw.dim() != 1:
        raise RuntimeError("decode_flac_cuda: expected a 1-D uint8 CUDA tensor -- this build has no CPU fallback")
    raw = raw.contiguous()
    L = _lib.lib()
    need = C.c_size_t()
    _lib.check(L.ar_flac_workspace_bytes(raw.numel(), C.byref(need)))
    n_out = C.c_int64()
    with torch.cuda.device(raw.device):
        stream = torch.cuda.current_stream(raw.device).cuda_stream
        ws = torch.empty(need.value, dtype=torch.uint8, device=raw.device)
        args = (raw.data_ptr(), raw.numel(), info["channels"], info["bps"], info["sample_rate"], info["min_block"],
                info["max_block"], info["total_samples"])

        def run(y, n):
            try:
                _lib.check(L.ar_flac_decode(*args, y.data_ptr() if y is not None else None, n, C.byref(n_out),
                                            ws.data_ptr(), need.value, stream))
            except RuntimeError as e:
                off = info.get("offset")
                raise RuntimeError(str(e) + (f" (frame data starts at byte {off} of the file)" if off else "")) from None

        n = info["total_samples"]
        if n == 0:                                                # unknown length: count the samples first
            run(None, 0)
            n = n_out.value
        y = torch.empty((info["channels"], n), dtype=torch.float32, device=raw.device)
        run(y, n)
    return y


def load_audio_cuda(file_path: str, sample_rate: int = 22050, device="cuda"):
    """`load_audio(..., mono=True)` with the arithmetic on the GPU (SURVEY.md 8f n1): the `data` chunk of a WAV file --
    8 / 16 / 24 / 32-bit integer PCM, 32 / 64-bit IEEE float, plain or WAVE_FORMAT_EXTENSIBLE -- is uploaded as the raw
    bytes it is (a 16-bit file costs half the H2D bytes of float32) from pinned memory, then decoded, mixed to mono and
    resampled on the device.  A FLAC file (recognised by its content, not its extension) uploads its compressed frame
    bytes the same way and is decoded on the device (`decode_flac_cuda`).  Other containers go through `_read_wav`
    (soundfile, when installed) and only the mix and the resampling run on the GPU.  Returns (audio [1,N] float32 CUDA,
    sample_rate)."""
    dev = torch.device(device)
    if is_flac(file_path):
        info = flac_info(file_path)
        planar = decode_flac_cuda(_upload_frames(file_path, info, dev), info)
        if planar.shape[1] < 1:
            raise RuntimeError(f"{file_path}: no audio frames")
        return resample_mono_cuda(planar, info["sample_rate"], sample_rate), sample_rate
    try:
        fmt, nch, sr, frames, offset = wav_info(file_path)
    except RuntimeError:
        audio, sr = _read_wav(file_path)
        return resample_mono_cuda(audio.to(dev), sr, sample_rate), sample_rate
    if frames < 1:
        raise RuntimeError(f"{file_path}: no audio frames")
    width = _PCM_WIDTH[fmt]
    host = torch.empty(frames * nch * width, dtype=torch.uint8).pin_memory()
    with open(file_path, "rb") as f:
        f.seek(offset)
        got = f.readinto(host.numpy())
    if got != host.numel():
        raise RuntimeError(f"{file_path}: truncated data chunk")
    planar = decode_pcm_cuda(host.to(dev, non_blocking=True), fmt, nch, frames)
    return resample_mono_cuda(planar, sr, sample_rate), sample_rate


def encode_flac_cuda(audio: torch.Tensor, sample_rate: int, bps: int = 24, block_size: int = 4096) -> bytes:
    """Planar `[C, N]` (or `[N]`) float CUDA audio -> a complete .flac file (`fLaC`, STREAMINFO with the MD5, the frames),
    encoded on the audio's device and current stream (`ar_flac_encode`).  Samples are
    rint_even(clamp(x, -1, 1) * (2^(bps-1) - 1)), NaN -> 0, as `save_audio(..., encoding="pcm16")` rounds for WAV;
    bps 16 or 24, 1..8 channels, block_size 16..4608.  The PCM bytes come back in pinned memory first and are hashed while
    the frame bytes are still copying."""
    if not audio.is_cuda:
        raise RuntimeError("encode_flac_cuda: expected a CUDA tensor -- this build has no CPU fallback")
    x = audio.detach().to(torch.float32)
    x = (x[None] if x.dim() == 1 else x).contiguous()
    if x.dim() != 2:
        raise ValueError("encode_flac_cuda: expected [channels, samples] audio")
    channels, n = x.shape
    if not 1 <= int(sample_rate) <= 655350:
        raise ValueError(f"encode_flac_cuda: sample rate {sample_rate} Hz (1..655350 supported)")
    L = _lib.lib()
    ws, cap = C.c_size_t(), C.c_size_t()
    try:
        _lib.check(L.ar_flac_encode_workspace_bytes(channels, n, int(block_size), int(bps), C.byref(ws), C.byref(cap)))
    except RuntimeError as e:
        raise ValueError(str(e)) from None
    total, min_frame, max_frame = C.c_int64(), C.c_int(), C.c_int()
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream(x.device)
        work = torch.empty(ws.value, dtype=torch.uint8, device=x.device)
        frames = torch.empty(cap.value, dtype=torch.uint8, device=x.device)
        pcm = torch.empty(n * channels * (bps // 8), dtype=torch.uint8, device=x.device)
        _lib.check(L.ar_flac_encode(x.data_ptr(), channels, n, int(bps), int(sample_rate), int(block_size), frames.data_ptr(),
                                    cap.value, pcm.data_ptr(), C.byref(total), C.byref(min_frame), C.byref(max_frame),
                                    work.data_ptr(), ws.value, stream.cuda_stream))
        pcm_host = torch.empty(pcm.numel(), dtype=torch.uint8).pin_memory()
        frames_host = torch.empty(total.value, dtype=torch.uint8).pin_memory()
        pcm_host.copy_(pcm, non_blocking=True)
        pcm_done = torch.cuda.Event()
        pcm_done.record(stream)
        frames_host.copy_(frames[:total.value], non_blocking=True)
        pcm_done.synchronize()
        md5 = hashlib.md5(pcm_host.numpy()).digest()
        stream.synchronize()
    info = int(sample_rate) << 44 | (channels - 1) << 41 | (bps - 1) << 36 | n
    streaminfo = (int(block_size).to_bytes(2, "big") * 2 + min_frame.value.to_bytes(3, "big") + max_frame.value.to_bytes(3, "big")
                  + info.to_bytes(8, "big") + md5)
    return b"fLaC" + bytes([0x80]) + len(streaminfo).to_bytes(3, "big") + streaminfo + frames_host.numpy().tobytes()


def save_audio(file_path: str, audio: torch.Tensor, sample_rate: int = 22050, encoding: str = None) -> None:
    """Write `[C,N]` float audio (audio_processing.py:45-55), the container chosen by the extension as `torchaudio.save`
    chooses it.  A `.flac` path (any case) writes FLAC encoded on the GPU (`encode_flac_cuda`): `encoding` "pcm24" (the
    default) or "pcm16"; a CUDA tensor is encoded on its device, a host tensor on the current CUDA device.  Any other
    path writes WAV: `encoding` None / "float32" writes 32-bit IEEE-float samples (what the reference's `torchaudio.save`
    of a float tensor writes), "pcm16" / "pcm24" 16 / 24-bit PCM rounded as rint(clamp(x, -1, 1) * (2^(bits-1) - 1))."""
    import os
    import struct
    parent = os.path.dirname(os.path.abspath(file_path))
    if file_path.lower().endswith(".flac"):
        encoding = "pcm24" if encoding is None else encoding
        if encoding not in ("pcm16", "pcm24"):
            raise ValueError(f"unknown FLAC encoding {encoding!r}: FLAC stores integers, use 'pcm16' or 'pcm24'")
        x = audio.detach()
        data = encode_flac_cuda(x if x.is_cuda else x.to(torch.device("cuda", torch.cuda.current_device())), sample_rate,
                                bps=16 if encoding == "pcm16" else 24)
        os.makedirs(parent, exist_ok=True)
        with open(file_path, "wb") as f:
            f.write(data)
        return
    a = audio.detach().to("cpu", torch.float32).numpy()
    if a.ndim == 1:
        a = a[None]
    os.makedirs(parent, exist_ok=True)
    if encoding == "pcm16":
        pcm = np.round(np.clip(a, -1.0, 1.0).T * 32767.0).astype("<i2")
        with wave.open(file_path, "wb") as w:
            w.setnchannels(a.shape[0])
            w.setsampwidth(2)
            w.setframerate(int(sample_rate))
            w.writeframes(pcm.tobytes())
        return
    if encoding == "pcm24":
        v = np.ascontiguousarray(np.round(np.clip(np.nan_to_num(a, nan=0.0), -1.0, 1.0).T * np.float32(8388607.0)), "<i4")
        pcm = v.view(np.uint8).reshape(-1, 4)[:, :3]                   # 3-byte little-endian samples
        with wave.open(file_path, "wb") as w:
            w.setnchannels(a.shape[0])
            w.setsampwidth(3)
            w.setframerate(int(sample_rate))
            w.writeframes(pcm.tobytes())
        return
    if encoding not in (None, "float32"):
        raise ValueError(f"unknown WAV encoding {encoding!r}")
    data = np.ascontiguousarray(a.T).astype("<f4").tobytes()
    nch, sr = a.shape[0], int(sample_rate)
    fmt = struct.pack("<4sIHHIIHH", b"fmt ", 16, 3, nch, sr, sr * nch * 4, nch * 4, 32)      # format tag 3 = IEEE float
    fact = struct.pack("<4sII", b"fact", 4, a.shape[1])
    body = b"WAVE" + fmt + fact + struct.pack("<4sI", b"data", len(data)) + data
    with open(file_path, "wb") as f:
        f.write(struct.pack("<4sI", b"RIFF", len(body)) + body)
