#!/usr/bin/env python
"""bench.py -- restored source audio-seconds per second through the full chain
(denoise -> super-res -> stereo, chunked with overlap-add, normalised) on N B200s.

  python bench.py [--gpus N --steps K --warmup W]            this repo's CUDA path
  python bench.py --impl reference [...]                     the reference's CPU path (oracle port)
  python bench.py [...] --dump-outputs DIR                   also write the last timed step's output to DIR/*.npy
  torchrun-style launch for N > 1 (one rank per GPU, RANK/LOCAL_RANK/WORLD_SIZE from env).

One "step" = one synthetic mono file of `--chunks-per-step` 2-second chunks per GPU pushed through
`RestorationPipeline.restore(mode="chunked")` (input normalise, chunk, chain, overlap-add, output
normalise).  It is a slice of BASELINE.json's 10-hour sweep: 2368 chunks = 4515.7 s, so 8 steps
are 10 h.  Files are independent => ranks share nothing (weak scaling, no collective on the data
path; NCCL is used only for the timing barrier / max-over-ranks).
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (no __pycache__ of its imports)

SR = 22050
CHUNK, OVERLAP = 44100, 2052
HOP = CHUNK - OVERLAP
# algorithmic FLOPs (2 x MAC of the reference's conv / convT / LSTM terms) per source audio-second,
# SURVEY.md 8(d) / BASELINE.md section 2
CHAIN_GFLOP_PER_AUDIO_S = 51.661
# of these, the share computed by the tcgen05 conv engine (every Conv1d / ConvTranspose1d with Cin >= 16 + the LSTM input
# projection): denoiser 147 968, super-res 41 984 MAC per input sample, stereo 473 088 MAC per 44.1 kHz sample (DESIGN.md 3)
CONV_GFLOP_PER_AUDIO_S = 2.0 * ((147968 + 41984) * SR + 473088 * 2 * SR) / 1e9          # 50.10
# beyond 8 sequences per SM the scan kernel computes the LSTM input projection itself (lstm_proj.cu): 32 768 MAC per 44.1 kHz
# sample leave the conv engine's account
CONV_GFLOP_PER_AUDIO_S_FUSED_SCAN = 2.0 * ((147968 + 41984) * SR + (473088 - 32768) * 2 * SR) / 1e9     # 47.21
# per-model algorithmic GFLOP per second of the model's OWN input signal (BASELINE.md section 2)
MODEL_GFLOP_PER_S = {"denoiser": 6.549, "super_resolution": 1.881, "stereo": 21.615}
METRIC = "restored audio-sec/sec (full chain)"
TRAFFIC_FILE = "conv_traffic_r02.json"


def conv_algorithmic_bytes_per_audio_s(fused_scan=False):
    """fp16 activation bytes (inputs read + outputs written, incl. pooled copies and residual operands) that the
    conv engine's launches of one chunk batch must move per source audio-second (DESIGN.md 3): entries are
    (bytes per row, rows per audio-second) per tensor stream of a launch.  Fused chains count their input and output only
    (U-Net double convs, super-resolution residual blocks -- whose skip operand is the block's own input --, the stereo
    dilated blocks, decoder layers 3 + 6 per side): their intermediates never reach HBM."""
    r = SR                                   # denoiser / SR input rate; stereo runs at 2r
    den = [(160, r),                                             # enc0b + pooled copy
           (256, r // 2), (512, r // 4),                         # fused enc1 / enc2 double convs + pooled copies
           (768, r // 8), (1024, r // 8),                        # bottleneck
           (512, r // 8), (256, r // 4), (768, r // 4), (512, r // 4),        # up0 (in, out), dec0a, dec0b
           (256, r // 4), (128, r // 2), (384, r // 2),          # up1 (in, out), fused dec1 double conv
           (128, r // 2), (64, r), (192, r),                     # up2 (in, out), fused dec2 double conv
           (128, r)]                                             # first transient-detector layer (32 -> 16 padded to 32 columns)
    sr = [(128, r)] * 4 + [(192, r)] + [(64, r), (64, 2 * r), (68, 2 * r)]   # 4 fused residual blocks, middle (+ skip), up (in, out), fused hf + head (fp32 out)
    st = [(192, 2 * r), (384, 2 * r), (512, 2 * r), (512 if fused_scan else 768, 2 * r),   # fused enc1, enc2, enc3, enc4 (+ xproj)
          (640, 2 * r), (320, 2 * r), (320, 2 * r)]                                    # dec0 (L+R), fused dec1 -> dec2 per side
    return float(sum(b * n for b, n in den + sr + st))


def elementwise_algorithmic_bytes(n_chunks, n):
    """Algorithmic HBM bytes per step of the CUDA-core (elementwise / Cin = 1 / Cout = 1) passes, per profile category
    (DESIGN.md 3): what each kernel must read and write once, counted over the samples it processes (chunk samples for
    the model stems / tails, file samples for normalize and overlap-add)."""
    c = n_chunks * CHUNK                    # 22.05 kHz chunk samples of the step (the stereo net runs on 2c)
    return {
        # fp32 sample in (4 B) + 32 fp16 channels out (64 B): denoiser k3 stem, super-resolution k7 stem, stereo k7 stem @ 2c
        "stem": 68.0 * (c + c + 2 * c),
        # denoiser tail: 32-channel features (64 B) + 16 transient-detector channels (32 B) + x (4 B) in, 4 B out;
        # stereo heads: 2 sides x 32 fp16 channels (128 B) in, L + R fp32 (8 B) out per 44.1 kHz sample
        "tail": 104.0 * c + 136.0 * 2 * c,
        # normalize_audio on the mono input (n) and the stereo output (2 x 2n): one reduction read + scale read + write
        "normalize": 12.0 * (n + 4 * n),
        # split: read + write every chunk sample; overlap-add: read both channels of every output-rate chunk, write 2 x 2n
        "chunk": 8.0 * c + 4.0 * (2 * 2 * c) + 4.0 * (2 * 2 * n),
    }


def load_conv_traffic(args):
    """DRAM bytes per conv-engine launch from the COMMITTED ncu capture (a static file, not measured in this run), if it
    was taken at this configuration and launch count; else None."""
    for name in (TRAFFIC_FILE, "conv_traffic_r01_final.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            c = t["config"]
            if c["chunks_per_step_per_gpu"] == args.chunks_per_step and c["batch_chunks"] == args.batch_chunks:
                return t["dram_bytes_per_launch_avg"], f"static ncu capture profiles/{name} ({t.get('launches_per_step', '?')} conv launches per step), not measured in this run"
        except Exception:
            pass
    return None, "no committed ncu capture for this configuration"


def synth_audio(n, seed, device):
    """Music proxy (sines + chirp) with hiss and pops, ~ -20 dBFS (BASELINE config 4 recipe)."""
    g = torch.Generator(device=device).manual_seed(seed)
    t = torch.arange(n, device=device, dtype=torch.float32) / SR
    x = 0.08 * torch.sin(2 * torch.pi * 220.0 * t) + 0.05 * torch.sin(2 * torch.pi * 554.4 * t + 0.3)
    x += 0.04 * torch.sin(2 * torch.pi * (300.0 + 40.0 * torch.sin(2 * torch.pi * 0.25 * t)) * t)
    x += 0.02 * torch.randn(n, device=device, generator=g)
    pops = torch.rand(n, device=device, generator=g) < 2e-4
    x += pops * (torch.rand(n, device=device, generator=g) - 0.5) * 1.2
    return x.unsqueeze(0).contiguous()


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.sm_max, self.ok = [], set(), None, False
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # NVML missing: report it rather than invent numbers
            self.err = repr(e)

    def run(self):
        while self.ok and not self._stop_evt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons), "samples": len(s)}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tflops": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "src": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback"}


def host_threads():
    """All host threads this process may use (torchrun pins OMP_NUM_THREADS=1, undo that for the CPU arm)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    torch.set_num_threads(n)
    return torch.get_num_threads()


def cpu_chain_rate(n_chunks):
    """Oracle port of the reference chain on the host cores: audio-s/s over `n_chunks` 2 s chunks."""
    import oracle
    from oracle.weights import make_state_dict
    sds = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}
    n = (n_chunks - 1) * HOP + CHUNK
    audio = synth_audio(n, 1, "cpu")
    with torch.no_grad():
        t0 = time.perf_counter()
        y = oracle.restore_chunked(sds, audio, CHUNK, OVERLAP, batch=min(n_chunks, 8))   # 8 chunks per forward: bounded host memory
        dt = time.perf_counter() - t0
    assert y.shape == (2, 2 * n)
    return (n / SR) / dt, dt, n / SR


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (oracle port: same ATen CPU kernels the
    reference modules dispatch to), all host threads, bounded sample per step."""
    if rank != 0:
        return
    cores = host_threads()
    nck = args.cpu_chunks
    for _ in range(args.warmup):
        cpu_chain_rate(1)
    tot_audio, tot_t = 0.0, 0.0
    for _ in range(args.steps):
        _, dt, secs = cpu_chain_rate(nck)
        tot_audio += secs
        tot_t += dt
    value = tot_audio / tot_t
    sample = f"{nck} chunks ({nck * HOP / SR + OVERLAP / SR:.1f} s of audio) per step, oracle port on torch CPU"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": "throughput sweep slice: synthetic 22.05 kHz mono, full chain denoise->super-res->stereo, "
                        "chunk 44100 / overlap 2052 overlap-add, input+output normalize",
            "chunks_per_step_per_gpu": args.chunks_per_step, "audio_s_per_step_per_gpu": round(step_samples(args) / SR, 2),
            "batch_chunks": args.batch_chunks, "streams": args.streams, "steps_for_10h": round(36000 / (step_samples(args) / SR), 1),
            "partition": f"by file, {world} rank(s), no collective", "l2": "inputs and activations far larger than L2 (no flush needed)"}


def step_samples(args):
    return (args.chunks_per_step - 1) * HOP + CHUNK


DUMP_MAX_BYTES = 64 << 20
DUMP_WINDOW = 4096                  # consecutive output samples per sampled window
DUMP_WINDOWS = 1024                 # windows per channel: 2 x 1024 x 4096 float32 = 32 MB


def dump_outputs(y, out_dir):
    """Write the restored stereo `[2, M]` of the last timed step under `out_dir`, so that two builds run with the same
    arguments (hence the same inputs) can be compared output for output.  Up to 64 MB it is written whole as
    `restored.npy`; a larger output as `restored_windows.npy` `[2, 1024, 4096]`: windows at the first and last sample and at
    1022 starts drawn from a fixed seed (the same positions for the same M), with the starts, as sample indices, in
    `restored_window_starts.npy` (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    if y.numel() * 4 <= DUMP_MAX_BYTES:
        np.save(os.path.join(out_dir, "restored.npy"), y.float().cpu().numpy())
        return
    m = y.shape[1]
    g = torch.Generator().manual_seed(0)
    drawn = torch.randint(0, m - DUMP_WINDOW + 1, (DUMP_WINDOWS - 2,), generator=g)
    starts = torch.cat([torch.tensor([0, m - DUMP_WINDOW]), drawn]).sort().values
    idx = (starts[:, None] + torch.arange(DUMP_WINDOW)).to(y.device)
    np.save(os.path.join(out_dir, "restored_windows.npy"), y[:, idx].float().cpu().numpy())
    np.save(os.path.join(out_dir, "restored_window_starts.npy"), starts.double().numpy())


def flush_l2(buf):
    buf.add_(1.0)     # read + write 512 MB: everything older leaves the 126 MB L2


def time_forward(fn, flush_buf, iters=7):
    """Median device time (ms) of `fn()`; L2 flushed before every timed call (the small configs fit in L2).  The GPU is
    first kept busy with `fn` for 0.3 s: these forwards follow CPU-only phases (the oracle timings) during which the idle GPU
    drops its clocks, and the latency-bound single-sequence LSTM scan scales 1:1 with the SM clock."""
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 0.3:
        fn()
        torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        flush_l2(flush_buf)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return sorted(times)[len(times) // 2]


def config_lines(pipe, sds, dev, cpu_cores):
    """BASELINE.json configs 1-4 (SURVEY.md 8d): per-model forwards at their stated batch (eager launch train and CUDA
    graph replay, next to the oracle port on the host cores) and config 4 as the latency of ONE 3-minute side."""
    import oracle
    from oracle.weights import make_input
    flush_buf = torch.zeros(128 * 1024 * 1024, dtype=torch.float32, device=dev)
    mods = {"denoiser": pipe.denoiser, "super_resolution": pipe.super_res, "stereo": pipe.stereo}
    fwd = {"denoiser": oracle.denoiser_forward, "super_resolution": oracle.super_resolution_forward, "stereo": oracle.stereo_forward}
    out = {}
    for cfg, name, B in (("cfg1", "denoiser", 2), ("cfg2", "stereo", 4), ("cfg3", "super_resolution", 16)):
        x = make_input(B, CHUNK)
        xd = x.to(dev)
        m = mods[name]
        with torch.no_grad():
            for _ in range(3):
                m(xd)
            eager_ms = time_forward(lambda: m(xd), flush_buf)
            g = m.capture(xd)
            for _ in range(3):
                g(xd)
            graph_ms = time_forward(lambda: g(xd), flush_buf)
            fwd[name](sds[name], x)
            t0 = time.perf_counter()
            for _ in range(3):
                fwd[name](sds[name], x)
            cpu_ms = (time.perf_counter() - t0) / 3 * 1e3
        secs = B * CHUNK / SR
        out[cfg] = {"model": name, "batch": B, "samples": CHUNK, "ms": graph_ms, "ms_eager_launches": eager_ms,
                    "audio_s_per_s": secs / (graph_ms / 1e3), "tflops": MODEL_GFLOP_PER_S[name] * secs / graph_ms,
                    "cpu": {"ms": cpu_ms, "audio_s_per_s": secs / (cpu_ms / 1e3), "cores": cpu_cores, "kind": "port"},
                    "timing": "median of 7, L2 flushed before each call, CUDA-graph replay of the forward"}
    n = 180 * SR
    side = synth_audio(n, 4, dev)
    with torch.no_grad():
        for _ in range(2):
            pipe.restore(side, mode="chunked", return_device=True)
        ms = time_forward(lambda: pipe.restore(side, mode="chunked", return_device=True), flush_buf, iters=5)
    out["cfg4"] = {"workload": "one synthetic 3-minute 22.05 kHz side, chunked chain (95 chunks, one batch), input+output normalize",
                   "ms": ms, "audio_s_per_s": 180.0 / (ms / 1e3), "chunks": 95,
                   "note": "single-file latency: 95 chunks under-fill the GPU (CUDA-core LSTM path, 1 sequence per CTA)"}
    del flush_buf
    return out


def library_bar(sds, dev, n_chunks=64, batch=16):
    """SECONDARY baseline (not the reference arm): the oracle-port modules -- the reference's op sequence, stock ATen /
    cuDNN kernels -- under torch eager on THIS GPU, fp32 and TF32-allowed, same 2 s chunks (batch bounded by the fp32
    activation memory of eager execution)."""
    import oracle
    import oracle.models as om
    from oracle.weights import make_input
    dsds = {k: {n: t.to(dev) for n, t in v.items()} for k, v in sds.items()}
    x = make_input(batch, CHUNK).to(dev)
    out = {}

    def timed(reps):
        with torch.no_grad():
            oracle.chain_forward(dsds, x)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                oracle.chain_forward(dsds, x)
            e1.record()
            e1.synchronize()
        return e0.elapsed_time(e1)

    for label, tf32 in (("fp32", False), ("tf32", True)):
        old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        try:
            reps, lstm = n_chunks // batch, "cuDNN RNN"
            try:
                ms = timed(reps)
            except RuntimeError as e:
                # cuDNN's RNN rejects the 88 200-step sequences of the chain (the reference's README.md:175 warns of
                # "cuDNN LSTM sequence length limits"): what a user of the reference can do is turn cuDNN off for the LSTM
                # (convs stay on cuDNN); ATen's native CUDA LSTM then launches a handful of kernels per time step
                lstm = f"ATen native CUDA LSTM (cuDNN RNN refused seq_len {2 * CHUNK}: {str(e)[:60]})"
                om.LSTM_WITHOUT_CUDNN = True
                reps = 1
                ms = timed(reps)
            out[label] = {"audio_s_per_s": (reps * batch * CHUNK / SR) / (ms / 1e3), "ms": ms, "chunks": reps * batch, "batch": batch,
                          "lstm": lstm}
        except Exception as e:
            out[label] = {"error": repr(e)[:200]}
        finally:
            om.LSTM_WITHOUT_CUDNN = False
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out["what"] = ("oracle-port modules (reference op sequence: F.conv1d / conv_transpose1d / batch_norm / max_pool1d / "
                   "torch.lstm ...) under stock torch eager + cuDNN on this GPU; chain on 2 s chunks, no stitching")
    return out


def parity_gate(pipe, sds, x_dev, args):
    """Outside the timed region: the chain on the step's OWN chunk batch (same batch size => same kernels, tile groups,
    fused chains, tensor-core LSTM) -- three of its chunks against the oracle.  Both tolerance clauses of north_star."""
    import ctypes as C
    import oracle
    from ml_audio_restoration_b200 import _lib, normalize_audio
    L = _lib.lib()
    n = x_dev.shape[1]
    a = normalize_audio(x_dev)
    B = min(args.batch_chunks, args.chunks_per_step)
    chunks = torch.empty((B, 1, CHUNK), dtype=torch.float32, device=x_dev.device)
    _lib.check(L.ar_split_chunks(a.data_ptr(), n, chunks.data_ptr(), 0, B, CHUNK, OVERLAP, torch.cuda.current_stream().cuda_stream))
    y = pipe.forward_chunks(chunks)
    picks = sorted({0, B // 2, B - 1})
    got = y[picks].cpu()
    with torch.no_grad():
        ref = oracle.chain_forward(sds, chunks[picks].cpu())
    err = float((ref - got).abs().max())
    snr = float(10 * torch.log10((ref.double() ** 2).sum() / ((ref - got).double() ** 2).sum()))
    ok = bool(torch.isfinite(got).all()) and err <= 1e-3 and snr >= 60.0
    return {"chunks": picks, "batch": B, "max_abs_err": err, "snr_db": snr, "tolerance": "max-abs <= 1e-3 AND snr >= 60 dB vs fp32 oracle",
            "pass": ok}


def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist
    from ml_audio_restoration_b200 import RestorationPipeline, _lib
    import oracle
    from oracle.weights import make_state_dict

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    sds = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}   # weights only: the oracle is not on the timed path
    pipe = RestorationPipeline.from_state_dicts(sds["denoiser"], sds["super_resolution"], sds["stereo"], dev)
    n = step_samples(args)
    audio_s = n / SR
    x_dev = synth_audio(n, 1000 + rank, dev)
    x_host = x_dev.cpu().pin_memory()

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def step_resident():
        return pipe.restore(x_dev, mode="chunked", chunk_size=CHUNK, overlap=OVERLAP, batch_chunks=args.batch_chunks,
                            return_device=True, streams=args.streams)

    for _ in range(args.warmup):
        step_resident()
    sync_all()

    # ---- timed region: K steps, inputs resident in HBM, CUDA events on the launching stream
    sampler = ClockSampler(local_rank)
    sampler.start()
    L.ar_profile_enable(1)
    launches0 = L.ar_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        y = step_resident()
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    launches = L.ar_launch_count() - launches0
    import ctypes as C
    ncat = len(_lib.PROFILE_CATEGORIES)
    p_ms, p_fl, p_ln = (C.c_double * ncat)(), (C.c_double * ncat)(), (C.c_longlong * ncat)()
    _lib.check(L.ar_profile_read(p_ms, p_fl, p_ln, ncat))
    L.ar_profile_enable(0)
    clocks = sampler.finish()
    assert y.shape == (2, 2 * n)
    if args.dump_outputs and rank == 0:
        dump_outputs(y, args.dump_outputs)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    t_s = float(ms.item()) / 1e3
    value = world * audio_s * args.steps / t_s

    # ---- end to end: host (pinned) input -> H2D -> chain -> D2H of the restored stereo, every step, through the serving
    # loop of the public API (`restore_stream`: the copies of neighbouring steps overlap the chain on their own streams;
    # all K uploads, K chain passes and K downloads happen inside the timed region)
    def e2e_loop(k):
        last = None
        for last in pipe.restore_stream((x_host for _ in range(k)), mode="chunked", chunk_size=CHUNK, overlap=OVERLAP,
                                        batch_chunks=args.batch_chunks, streams=args.streams):
            pass
        return last

    e2e_loop(2)
    sync_all()
    t0 = time.perf_counter()
    out = e2e_loop(args.steps)
    torch.cuda.synchronize(dev)
    te = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * audio_s * args.steps / float(te.item())
    assert out.shape == (2, 2 * n) and not out.is_cuda

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    cats = {name: {"ms": p_ms[i], "launches": int(p_ln[i]), "gflop": p_fl[i] / 1e9} for i, name in enumerate(_lib.PROFILE_CATEGORIES)}
    conv = cats["conv"]
    conv_s = conv["ms"] / 1e3
    # ALGORITHMIC FLOPs = SURVEY.md 8(d)'s per-SOURCE-second figure x the source seconds of the step: the 2 052-sample
    # chunk overlap that the chunked scheme recomputes is overhead, not work (it is in `achieved_incl_overlap` only)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    seq_in_flight = min(args.batch_chunks, args.chunks_per_step)
    fused_scan = seq_in_flight > 8 * sms
    conv_gflop = CONV_GFLOP_PER_AUDIO_S_FUSED_SCAN if fused_scan else CONV_GFLOP_PER_AUDIO_S
    achieved = (conv_gflop * audio_s * args.steps / 1e3) / conv_s if conv_s > 0 else 0.0
    achieved_incl = (conv["gflop"] / 1e3) / conv_s if conv_s > 0 else 0.0
    conv_bytes = conv_algorithmic_bytes_per_audio_s(fused_scan) * audio_s * args.steps      # algorithmic, this rank
    hbm_gbs = (conv_bytes / 1e9) / conv_s if conv_s > 0 else 0.0
    traffic, traffic_src = load_conv_traffic(args)
    lstm = cats["lstm"]
    lstm_steps = 2 * CHUNK                                                         # serial steps per launch (44.1 kHz, 2 s)
    lstm_ms_launch = lstm["ms"] / max(1, lstm["launches"])
    roofline = {
        "kernel": "tcgen05 conv engine: conv_umma2_kernel (2-CTA implicit-GEMM Conv1d / ConvT), conv_chain_kernel "
                  "(fused dilated blocks + LSTM input projection, U-Net 64 -> 128 -> 128 double conv), all template variants",
        "bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
        "frac": achieved / peaks["tflops"], "peak_source": f"{peaks['src']} bf16 dense sustained (fp16 operands run at the same rate)",
        "flops_per_unit": f"{conv_gflop:.2f} GFLOP per source audio-second (of the chain's {CHAIN_GFLOP_PER_AUDIO_S}"
                          + ("; the LSTM input projection, 2.89, runs inside the scan kernel" if fused_scan else "") + "), "
                          f"x {audio_s:.1f} source seconds per step; chunk-overlap recompute excluded",
        "achieved_incl_overlap": achieved_incl,
        "avg_launch_ms": conv["ms"] / max(1, conv["launches"]), "launches": conv["launches"],
        "launches_per_step": conv["launches"] // max(1, args.steps),
        "share_of_step": conv["ms"] / (1e3 * t_s), "traffic": traffic, "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": conv_bytes / max(1, conv["launches"]),
        "hbm": {"achieved": hbm_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_gbs / peaks["hbm_gbs"],
                "note": "same launches against the HBM roofline (algorithmic fp16 activation bytes per launch)"},
        "whole_chain": {"achieved": value / world * CHAIN_GFLOP_PER_AUDIO_S / 1e3, "unit": "TFLOP/s",
                        "frac": value / world * CHAIN_GFLOP_PER_AUDIO_S / 1e3 / peaks["tflops"],
                        "note": "all kernels of the step (convs, LSTM, stems, tails, normalize, split / overlap-add)"},
        "lstm": {"kernel": ("lstm_proj_kernel (tcgen05 input projection + mma.sync recurrence)" if fused_scan else "lstm_mmaw_kernel<4>" if seq_in_flight > 2 * sms else "lstm_kernel"),
                 "bound": "latency", "ms_per_launch": lstm_ms_launch, "serial_steps_per_launch": lstm_steps,
                 "ns_per_step": 1e6 * lstm_ms_launch / lstm_steps, "sequences_in_flight": seq_in_flight,
                 "sequences_per_sm": seq_in_flight / sms,
                 "sequence_steps_per_s": seq_in_flight * lstm_steps / (lstm_ms_launch / 1e3) if lstm_ms_launch > 0 else 0.0,
                 "share_of_step": lstm["ms"] / (1e3 * t_s)},
        "per_category_ms_per_step": {k: v["ms"] / args.steps for k, v in cats.items()},
    }
    # the elementwise / single-channel passes against the HBM roofline (north_star: "reported in achieved HBM GB/s")
    roofline["elementwise_hbm"] = {"unit": "GB/s", "peak": peaks["hbm_gbs"], "categories": {
        k: {"algorithmic_gb_per_step": b / 1e9, "ms_per_step": cats[k]["ms"] / args.steps,
            "achieved": (b / 1e9) / (cats[k]["ms"] / args.steps / 1e3) if cats[k]["ms"] > 0 else 0.0,
            "frac": (b / 1e9) / (cats[k]["ms"] / args.steps / 1e3) / peaks["hbm_gbs"] if cats[k]["ms"] > 0 else 0.0}
        for k, b in elementwise_algorithmic_bytes(args.chunks_per_step, n).items()}}
    line = {
        "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate", "data": "synthetic", "config": workload_config(args, world),
        "realtime_factor_per_gpu": value / world,
        "chain_tflops_per_gpu": value / world * CHAIN_GFLOP_PER_AUDIO_S / 1e3,
        "e2e": {"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 16 * n},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "lib": _lib.LIB_PATH,
    }
    cores = host_threads()
    line["parity"] = parity_gate(pipe, sds, x_dev, args)
    if world == 1 and not args.no_cpu_baseline:
        cpu_chain_rate(1)
        v, dt, secs = cpu_chain_rate(args.cpu_chunks)
        line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port",
                                "sample": f"{args.cpu_chunks} chunks ({secs:.1f} s of audio) in {dt:.1f} s, oracle port on torch CPU"}
    if world == 1 and not args.no_secondary:
        line["configs"] = config_lines(pipe, sds, dev, cores)
        line["secondary"] = {"torch_eager_same_gpu": library_bar(sds, dev)}
        for k in ("fp32", "tf32"):
            r = line["secondary"]["torch_eager_same_gpu"].get(k, {})
            if "audio_s_per_s" in r:
                r["this_repo_over_it"] = (value / world) / r["audio_s_per_s"]
    print(json.dumps(line), flush=True)
    if not line["parity"]["pass"]:
        raise SystemExit("bench.py: PARITY GATE FAILED -- the number above is not valid")
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--chunks-per-step", type=int, default=2368, help="2 s chunks per GPU per step (2368 = 16 per SM)")
    ap.add_argument("--batch-chunks", type=int, default=2368, help="chunks per chain launch (2368 = 16 per SM: one full-chip tensor-core LSTM "
                    "launch, 8 sequences per CTA x 2 CTAs per SM; the conv phases run on sub-batches around it)")
    ap.add_argument("--streams", type=int, default=1, help="chunk batches in flight (LSTM of one overlaps convs of the next)")
    ap.add_argument("--cpu-chunks", type=int, default=32, help="chunks in the bounded CPU sample (32 = 61 s of audio, about 11 s on 16 host cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the per-config lines (BASELINE configs 1-4) and the torch-eager same-GPU bar")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the restored stereo of the last one "
                    "(rank 0; whole up to 64 MB, else a fixed seeded sample of windows) to DIR as float32 .npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the CUDA path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N "
                         "--master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
