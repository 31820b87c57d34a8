"""Catalog throughput: many 78 rpm sides through `restore_many` against a per-file `restore` loop, on one GPU.

Prints ONE JSON line.  The catalog is seeded and synthetic (bench.py's `synth_audio`): `--files` sides of 150-210 s at
22.05 kHz.  Reported:
  chunked   per-file `restore(mode="chunked")` loop vs `restore_many(mode="chunked")`, audio-s/s
  exact     `restore_many(mode="exact")` (lockstep windows, per-file LSTM state positions), audio-s/s, and the per-file
            `restore(mode="exact")` on `--exact-subset` files, extrapolated to the catalog at its measured rate (the
            per-file path runs one file after another, so its rate does not depend on the catalog size)
  passes    launches per group; time and bytes/s of the window gather / kept-range scatter of one lockstep step and of
            the per-file split / overlap-add / normalize passes of one chunked group (CUDA events, 20 repetitions)
  diff      largest per-file max |restore_many - per-file| of each mode
  gpu       card name, power limit and median SM clock, read in this run
Usage: python tools/catalog_bench.py [--files 256] [--exact-subset 4]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

from bench import SR, ClockSampler, synth_audio  # noqa: E402
from ml_audio_restoration_b200 import RestorationPipeline, _lib  # noqa: E402
from ml_audio_restoration_b200.inference import (DEFAULT_CHUNK, DEFAULT_OVERLAP, EXACT_STEREO_HALO,  # noqa: E402
                                                 plan_chunks)


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t


def event_ms(fn, reps=20):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def gpu_info(dev):
    info = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as e:  # NVML missing: say so
        info["nvml_error"] = repr(e)
    return info


def max_diff(a, b):
    return max(float((x - y).abs().max()) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=256)
    ap.add_argument("--min-s", type=float, default=150.0)
    ap.add_argument("--max-s", type=float, default=210.0)
    ap.add_argument("--exact-subset", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("catalog_bench needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    import oracle
    from oracle.weights import make_state_dict
    sds = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}
    pipe = RestorationPipeline.from_state_dicts(sds["denoiser"], sds["super_resolution"], sds["stereo"], dev)
    L = _lib.lib()
    g = torch.Generator().manual_seed(args.seed)
    lens = [int((args.min_s + (args.max_s - args.min_s) * float(torch.rand(1, generator=g))) * SR) for _ in range(args.files)]
    audios = [synth_audio(n, args.seed + i, dev) for i, n in enumerate(lens)]
    audio_s = sum(lens) / SR
    res = {"metric": "catalog_audio_s_per_s", "files": args.files, "audio_s": round(audio_s, 1),
           "side_s": [args.min_s, args.max_s], "seed": args.seed, "gpu": gpu_info(0)}

    # warm-up of every shape family (module loads, workspaces)
    pipe.restore_many(audios[:2], mode="chunked", return_device=True)
    pipe.restore(audios[0], mode="chunked", return_device=True)
    sampler = ClockSampler(0)
    sampler.start()

    # ---------------------------------------------------------------- chunked
    loop, t_loop = timed(lambda: [pipe.restore(a, mode="chunked", return_device=True) for a in audios])
    calls = {"chain": 0, "window": 0}
    fc, fw = pipe.forward_chunks, pipe.stereo.forward_window

    def count_chain(*a, **k):
        calls["chain"] += 1
        return fc(*a, **k)

    def count_window(*a, **k):
        calls["window"] += 1
        return fw(*a, **k)

    pipe.forward_chunks, pipe.stereo.forward_window = count_chain, count_window
    n0 = L.ar_launch_count()
    many, t_many = timed(lambda: pipe.restore_many(audios, mode="chunked", return_device=True))
    n_launch = L.ar_launch_count() - n0
    res["chunked"] = {"per_file_loop_audio_s_per_s": round(audio_s / t_loop, 1), "per_file_loop_s": round(t_loop, 3),
                      "restore_many_audio_s_per_s": round(audio_s / t_many, 1), "restore_many_s": round(t_many, 3),
                      "speedup": round(t_loop / t_many, 2), "groups": calls["chain"],
                      "native_launches_per_group": round(n_launch / max(1, calls["chain"]), 1),
                      "max_abs_diff_vs_per_file": max_diff(many, loop)}
    del loop, many

    # ---------------------------------------------------------------- exact
    pipe.restore_many(audios[:1], mode="exact", return_device=True)
    calls["window"] = 0
    n0 = L.ar_launch_count()
    many, t_many = timed(lambda: pipe.restore_many(audios, mode="exact", return_device=True))
    n_launch = L.ar_launch_count() - n0
    lock_steps = calls["window"]
    pipe.forward_chunks, pipe.stereo.forward_window = fc, fw
    sub = audios[:args.exact_subset]
    one, t_one = timed(lambda: [pipe.restore(a, mode="exact", return_device=True) for a in sub])
    sub_s = sum(lens[:args.exact_subset]) / SR
    res["exact"] = {"restore_many_audio_s_per_s": round(audio_s / t_many, 2), "restore_many_s": round(t_many, 3),
                    "lockstep_window_launches": lock_steps, "native_launches": n_launch,
                    "per_file_audio_s_per_s": round(sub_s / t_one, 2), "per_file_subset_files": len(sub),
                    "per_file_subset_s": round(t_one, 3),
                    "per_file_catalog_s_extrapolated": round(t_one / sub_s * audio_s, 1),
                    "extrapolation": "per-file restore(mode='exact') runs files one after another; its rate on the subset "
                                     "is applied to the whole catalog",
                    "speedup_extrapolated": round((t_one / sub_s * audio_s) / t_many, 2),
                    "max_abs_diff_vs_per_file": max_diff(many[:len(sub)], one)}
    del many, one

    # ---------------------------------------------------------------- host-issued passes
    stream = torch.cuda.current_stream(dev).cuda_stream
    r = pipe.rate
    S = (r * (DEFAULT_CHUNK - DEFAULT_CHUNK % 8) - 2 * EXACT_STEREO_HALO) // 16 * 16
    W = S + 2 * EXACT_STEREO_HALO
    B = len(audios)
    Ms = [r * n for n in lens]
    sig, offs = RestorationPipeline._packed(Ms, dev)
    sig.normal_()
    x = torch.empty((B, 1, W), device=dev)
    y = torch.randn((B, 2, W), device=dev)
    out, ooffs = RestorationPipeline._packed([2 * m for m in Ms], dev)
    ws = torch.empty(_lib.WINDOW_IO_BYTES_PER_ITEM * B, dtype=torch.uint8, device=dev)
    starts = (C.c_int64 * B)(*[o + m // 2 for o, m in zip(offs, Ms)])
    dst = (C.c_int64 * (2 * B))(*[v for o, m in zip(ooffs, Ms) for v in (o + m // 2, o + m + m // 2)])
    lo, ln = (C.c_int * B)(*[EXACT_STEREO_HALO] * B), (C.c_int * B)(*[S] * B)
    t_g = event_ms(lambda: _lib.check(L.ar_gather_windows(sig.data_ptr(), sig.numel(), starts, B, W, x.data_ptr(), ws.data_ptr(),
                                                          ws.numel(), stream)))
    t_s = event_ms(lambda: _lib.check(L.ar_scatter_kept(y.data_ptr(), B, W, dst, lo, ln, out.data_ptr(), out.numel(),
                                                        ws.data_ptr(), ws.numel(), stream)))
    g_bytes, s_bytes = 2 * 4 * B * W, 2 * 2 * 4 * B * S
    del sig, x, y, out
    # one chunked group: its files' split, overlap-add and normalize (in and out) passes, as restore_many issues them
    counts = [len(plan_chunks(n, DEFAULT_CHUNK, DEFAULT_OVERLAP)) for n in lens]
    grp, tot = [], 0
    for f, c in enumerate(counts):
        if tot + c > 16 * torch.cuda.get_device_properties(dev).multi_processor_count:
            break
        grp.append(f)
        tot += c
    buf = torch.empty((tot, 1, DEFAULT_CHUNK), device=dev)
    y_all = torch.randn((tot, 2, r * DEFAULT_CHUNK), device=dev)
    gout, goffs = RestorationPipeline._packed([2 * r * lens[f] for f in grp], dev)
    ins = [a.clone() for a in (audios[f] for f in grp)]

    def passes(which):
        first = 0
        for f, o, a in zip(grp, goffs, ins):
            n = lens[f]
            if which == "split":
                _lib.check(L.ar_split_chunks(a.data_ptr(), n, buf[first].data_ptr(), 0, counts[f], DEFAULT_CHUNK,
                                             DEFAULT_OVERLAP, stream))
            elif which == "ola":
                _lib.check(L.ar_overlap_add(y_all[first].data_ptr(), gout[o:].data_ptr(), n, counts[f], 2, DEFAULT_CHUNK,
                                            DEFAULT_OVERLAP, r, stream))
            else:
                pipe._normalize_(a)
                pipe._normalize_(gout[o:o + 2 * r * n])
            first += counts[f]

    n_in = sum(lens[f] for f in grp)
    t_split, t_ola, t_norm = (event_ms(lambda w=w: passes(w)) for w in ("split", "ola", "normalize"))
    hbm = 1e-9 / 1e-3
    res["passes"] = {
        "gather_windows": {"items": B, "W": W, "ms": round(t_g, 4), "bytes": g_bytes, "GB_s": round(g_bytes / t_g * hbm, 1)},
        "scatter_kept": {"items": B, "kept": S, "ms": round(t_s, 4), "bytes": s_bytes, "GB_s": round(s_bytes / t_s * hbm, 1)},
        "chunked_group": {"files": len(grp), "chunks": tot,
                          "split": {"launches": len(grp), "ms": round(t_split, 3), "bytes": 4 * (n_in + tot * DEFAULT_CHUNK)},
                          "overlap_add": {"launches": len(grp), "ms": round(t_ola, 3),
                                          "bytes": 4 * 2 * r * (tot * DEFAULT_CHUNK + n_in)},
                          "normalize": {"launches": 4 * len(grp), "ms": round(t_norm, 3),
                                        "bytes": 4 * 3 * (n_in + 2 * r * n_in)}},
        "hbm_datasheet_GB_s": 7700}
    for k in ("split", "overlap_add", "normalize"):
        p = res["passes"]["chunked_group"][k]
        p["GB_s"] = round(p["bytes"] / p["ms"] * hbm, 1)
    res["clocks"] = sampler.finish()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
