"""Times the device FLAC encoder on many synthetic three-minute sides and prints one JSON line.

Device time: CUDA events around `ar_flac_encode` over 64 stereo 44.1 kHz sides (quantise, analyse, write, finish, gather,
and the one read-back of the frame totals per call), after a warm-up call, once at 16 and once at 24 bits.  Each side
reads its own device copy of the input (64 x 63.5 MB, far larger than the 126 MB L2); four distinct sides are generated
and copied.  Next to it: audio-seconds per second against the restoration chain's rate, the compression ratio against
the PCM samples, and the bytes a side sends to the host (frames + PCM for the MD5) against a float32 WAV.  End to end:
the wall clock of `encode_flac_cuda` (encode, pinned copies back, host MD5, container) per side, with the host MD5 of the
same PCM bytes timed on its own, so the split is measured.  The card's name and power limit are read in the same run.

    python tools/flac_encode_bench.py [--out profiles/flac_encode_bench.json]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import flac_encode_ref as ref  # noqa: E402
from oracle import flac  # noqa: E402
from flac_vectors import signal  # noqa: E402
from ml_audio_restoration_b200 import _lib  # noqa: E402
from ml_audio_restoration_b200.audio_processing import encode_flac_cuda  # noqa: E402

CHAIN_AUDIO_S_PER_S = 12843.8      # restoration chain, 1 B200: profiles/bench_r02_final_k20.json ("value")
RATE, SECONDS, SIDES, DISTINCT, BLOCK, E2E_SIDES = 44100, 180, 64, 4, 4096, 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, sm = (v.strip() for v in q.stdout.strip().split(","))
    return {"name": name, "power_limit_w": float(power), "sm_max_mhz": int(sm)}


def run(bps, sides):
    n = RATE * SECONDS
    L = _lib.lib()
    ws, cap = C.c_size_t(), C.c_size_t()
    _lib.check(L.ar_flac_encode_workspace_bytes(2, n, BLOCK, bps, C.byref(ws), C.byref(cap)))
    work = torch.empty(ws.value, dtype=torch.uint8, device="cuda")
    frames = torch.empty(cap.value, dtype=torch.uint8, device="cuda")
    pcm = torch.empty(n * 2 * (bps // 8), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    total, mn, mx = C.c_int64(), C.c_int(), C.c_int()

    def encode(x):
        _lib.check(L.ar_flac_encode(x.data_ptr(), 2, n, bps, RATE, BLOCK, frames.data_ptr(), cap.value, pcm.data_ptr(),
                                    C.byref(total), C.byref(mn), C.byref(mx), work.data_ptr(), ws.value, stream))
        return total.value

    encode(sides[0])                                                       # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    compressed = sum(encode(x) for x in sides)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    audio_s = len(sides) * SECONDS
    pcm_bytes = len(sides) * n * 2 * (bps // 8)
    wav_bytes = len(sides) * (n * 2 * 4 + 58)

    e2e, md5_s, files = [], [], []
    for x in sides[:E2E_SIDES]:
        torch.cuda.synchronize()
        t = time.perf_counter()
        data = encode_flac_cuda(x, RATE, bps=bps, block_size=BLOCK)
        e2e.append(time.perf_counter() - t)
        files.append(len(data))
        encode(x)
        host = pcm.cpu().numpy()                                           # the same side's PCM bytes
        t = time.perf_counter()
        digest = hashlib.md5(host).digest()
        md5_s.append(time.perf_counter() - t)
        assert flac.parse_container(data)[0]["md5"] == digest
    return {"bps": bps, "sides": len(sides), "distinct_sides": DISTINCT, "seconds_per_side": SECONDS, "sample_rate": RATE,
            "channels": 2, "block_size": BLOCK, "device_ms": ms, "device_ms_per_side": ms / len(sides),
            "audio_s_per_s": audio_s / (ms / 1e3), "x_chain_rate": audio_s / (ms / 1e3) / CHAIN_AUDIO_S_PER_S,
            "compressed_bytes": compressed, "compression_ratio_vs_pcm": compressed / pcm_bytes,
            "bytes_to_host_per_side": (compressed + pcm_bytes) / len(sides), "float32_wav_bytes_per_side": wav_bytes / len(sides),
            "bytes_to_host_vs_float32_wav": (compressed + pcm_bytes) / wav_bytes,
            "e2e_encode_flac_cuda_ms_per_side": 1e3 * float(np.median(e2e)), "host_md5_ms_per_side": 1e3 * float(np.median(md5_s)),
            "e2e_sides": len(e2e), "file_bytes_per_side": int(np.median(files))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flac_encode_bench: needs a CUDA device")
    base = [torch.from_numpy(flac.to_float(signal(RATE * SECONDS, 2, 24, seed=100 + k), 24)).cuda() for k in range(DISTINCT)]
    sides = [base[i % DISTINCT].clone() for i in range(SIDES)]
    res = {"metric": "FLAC encode on the GPU (ar_flac_encode per side: quantise + analyse + write + finish + gather + totals "
                     "read-back)", "unit": "audio-s/s", "card": card(), "chain_audio_s_per_s": CHAIN_AUDIO_S_PER_S,
           "timing": "CUDA events around the encode calls of all sides after one warm-up call; end to end: host clock "
                     "around encode_flac_cuda, median of the first sides",
           "workloads": [run(bps, sides) for bps in (16, 24)]}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
