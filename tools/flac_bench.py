"""Times the device FLAC decoder (`decode_flac_cuda` -> `ar_flac_decode`: index, walk, one copy of the frame table, chain,
decode) on many synthetic sides, with CUDA events around the decode calls after a warm-up pass, and prints one JSON line:
decoded audio-seconds per second and compressed GB/s per workload, next to the restoration chain's rate and the card's
name and power limit read in the same run.

Workloads: 64 three-minute stereo 44.1 kHz 16-bit sides (block size 4096, LPC order 12, mid/side) and 16 three-minute
stereo 96 kHz 24-bit sides.  Encoding in numpy takes seconds per side, so a few distinct sides are encoded and each is
uploaded several times: every decode reads its own device copy, and the compressed bytes of a workload (1.3 GB / 0.9 GB)
and its output (4 GB / 4.4 GB) are far larger than the 126 MB L2.

    python tools/flac_bench.py [--out profiles/flac_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import flac  # noqa: E402
from flac_vectors import signal  # noqa: E402
from ml_audio_restoration_b200.audio_processing import decode_flac_cuda  # noqa: E402

CHAIN_AUDIO_S_PER_S = 12843.8      # restoration chain, 1 B200: profiles/bench_r02_final_k20.json ("value")
WORKLOADS = [("cd_44k1_16bit", 44100, 16, 64, 2), ("hires_96k_24bit", 96000, 24, 16, 1)]   # name, rate, bps, sides, distinct
SECONDS = 180


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, sm = (v.strip() for v in q.stdout.strip().split(","))
    return {"name": name, "power_limit_w": float(power), "sm_max_mhz": int(sm)}


def run(name, rate, bps, sides, distinct):
    streams = []
    for k in range(distinct):
        x = signal(rate * SECONDS, 2, bps, seed=100 + k)
        data = flac.encode(x, bps, rate, 4096, order=12, stereo="mid_side")
        info, off = flac.parse_container(data)
        info = {**info, "offset": off}
        ref = flac.to_float(x, bps)
        streams.append((info, data[off:], ref))
    raws = [torch.frombuffer(bytearray(streams[i % distinct][1]), dtype=torch.uint8).cuda() for i in range(sides)]
    for i in range(distinct):                                            # warm-up, and a bit-exact check of each side
        got = decode_flac_cuda(raws[i], streams[i][0])
        assert np.array_equal(got.cpu().numpy(), streams[i][2]), f"{name}: decode differs from the encoded samples"
        del got
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    outs = [decode_flac_cuda(raws[i], streams[i % distinct][0]) for i in range(sides)]
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    nbytes = sum(r.numel() for r in raws)
    audio_s = sides * SECONDS
    del outs
    return {"workload": name, "sides": sides, "distinct_sides": distinct, "seconds_per_side": SECONDS, "sample_rate": rate,
            "bps": bps, "channels": 2, "block_size": 4096, "lpc_order": 12, "stereo": "mid_side",
            "compressed_bytes": nbytes, "ms": ms, "audio_s_per_s": audio_s / (ms / 1e3),
            "compressed_gb_per_s": nbytes / (ms / 1e3) / 1e9,
            "x_chain_rate": audio_s / (ms / 1e3) / CHAIN_AUDIO_S_PER_S}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flac_bench: needs a CUDA device")
    res = {"metric": "FLAC decode on the GPU (ar_flac_decode, per call: index + walk + frame-table copy + decode)",
           "unit": "audio-s/s", "card": card(), "chain_audio_s_per_s": CHAIN_AUDIO_S_PER_S,
           "timing": "CUDA events around the decode calls of all sides, after one warm-up decode per distinct side",
           "workloads": [run(*w) for w in WORKLOADS]}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
