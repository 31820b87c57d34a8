"""CPU: C-ABI surface, host-side planning/sharding logic, drop-in API surface (no GPU compute)."""
import ctypes as C
import inspect
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from oracle import pipeline as opipe
from oracle.weights import make_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ml_audio_restoration_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "audiorestore.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(ar_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    lib = C.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported by {_lib.LIB_PATH}"
    assert _lib.lib().ar_version() >= 100


def test_library_is_sm100a_native_code():
    """The shipped library is sm_100a machine code with the Blackwell instructions the design rests on (DESIGN.md 3): tcgen05.mma
    (UTCHMMA, 1- and 2-CTA), TMEM loads (LDTM), bulk-async TMA copies and L2 prefetches (UBLKCP / UBLKPF), the LSTM's warp MMA
    (HMMA.16816), packed 2-wide fp32 (FFMA2) and the mixed-precision add (FHADD) -- no PTX-only / JIT path."""
    import shutil
    import subprocess
    from ml_audio_restoration_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not installed")
    elf = subprocess.run([cuobjdump, "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in elf and "sm_90" not in elf, elf
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for op in ("UTCHMMA.2CTA", "UTCHMMA", "LDTM", "UBLKCP", "UBLKPF", "HMMA.16816.F32", "FFMA2", "FHADD", "STG.E.EF"):
        assert op in sass, f"{op} missing from the SASS of {_lib.LIB_PATH}"


def test_num_chunks_matches_oracle_plan():
    from ml_audio_restoration_b200 import _lib, plan_chunks
    L = _lib.lib()
    for N, chunk, ov in [(9, 4, 1), (3, 4, 1), (4000, 1000, 100), (4000, 1000, 0), (1000, 1000, 100), (1001, 1000, 100),
                         (3969000, 44100, 2052), (793800000, 44100, 2052), (44100, 44100, 2052), (44101, 44100, 0)]:
        n = C.c_int()
        _lib.check(L.ar_num_chunks(N, chunk, ov, C.byref(n)))
        assert n.value == len(opipe.plan_chunks(N, chunk, ov)) == len(plan_chunks(N, chunk, ov))
    with pytest.raises(ValueError):
        _lib.check(L.ar_num_chunks(100, 10, 6, C.byref(C.c_int())))
    with pytest.raises(ValueError):
        _lib.check(L.ar_num_chunks(0, 10, 2, C.byref(C.c_int())))
    with pytest.raises(ValueError):
        plan_chunks(100, 10, 6)


def test_model_create_fails_loudly_without_gpu():
    """No CPU fallback: without an sm_100 device the native create call errors out."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from ml_audio_restoration_b200 import AudioSuperResolution, _lib
    m = AudioSuperResolution().eval()
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 1, 64))                       # CPU tensor
    h = C.c_void_p()
    rc = _lib.lib().ar_model_create(_lib.MODEL_SUPER_RES, None, 0, 0, C.byref(h))
    assert rc != 0 and _lib.lib().ar_last_error()


def test_drop_in_signatures_and_state_dict_keys():
    from ml_audio_restoration_b200 import AudioDenoiser, AudioSuperResolution, StereoSeparator, restore_audio
    sig = inspect.signature(AudioDenoiser.__init__)
    assert list(sig.parameters)[1:] == ["in_channels", "out_channels", "features"]
    sig = inspect.signature(AudioSuperResolution.__init__)
    assert [(p.name, p.default) for p in list(sig.parameters.values())[1:]] == [
        ("upscale_factor", 2), ("channels", 1), ("base_channels", 32), ("num_residual_blocks", 4)]
    sig = inspect.signature(StereoSeparator.__init__)
    assert [(p.name, p.default) for p in list(sig.parameters.values())[1:]] == [
        ("base_channels", 32), ("lstm_hidden", 64), ("num_lstm_layers", 1)]
    params = list(inspect.signature(restore_audio).parameters.values())
    assert [p.name for p in params[:8]] == ["input_path", "output_path", "denoiser_checkpoint", "super_res_checkpoint",
                                            "stereo_checkpoint", "sample_rate", "enable_super_resolution", "device"]
    assert params[2].default == "models/checkpoints/best_model.pth"       # inference.py:20, kept verbatim
    assert params[5].default == 22050 and params[6].default is True
    for cls, name in ((AudioDenoiser, "denoiser"), (AudioSuperResolution, "super_resolution"), (StereoSeparator, "stereo")):
        m = cls()
        sd = make_state_dict(name)
        assert sorted(m.state_dict().keys()) == sorted(sd.keys())
        for k, v in m.state_dict().items():
            assert v.shape == sd[k].shape and v.dtype == sd[k].dtype, k
    for bad in (lambda: AudioDenoiser(features=[64, 128, 256, 512]), lambda: AudioSuperResolution(upscale_factor=4),
                lambda: StereoSeparator(base_channels=64)):
        with pytest.raises(NotImplementedError):
            bad()


def test_src_import_paths_and_cli_flags():
    from src.models import AudioDenoiser  # noqa: F401
    from src.models.stereo_separator import StereoSeparator  # noqa: F401
    from src.inference import restore_audio  # noqa: F401
    out = subprocess.run([sys.executable, os.path.join(ROOT, "src", "inference.py"), "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--denoiser", "--super-res", "--stereo", "--sample-rate", "--no-super-res", "--device"):
        assert flag in out.stdout


def test_chunk_audio_reference_quirks():
    """chunk_audio mirrors audio_processing.py:229-253, including its documented tail behaviour (SURVEY 5b)."""
    from ml_audio_restoration_b200 import chunk_audio
    a = torch.arange(9.0)[None]
    c = chunk_audio(a, 4, 1)
    assert [x[0].tolist() for x in c] == [[0, 1, 2, 3], [3, 4, 5, 6]]       # samples 7-8 dropped
    c = chunk_audio(torch.arange(10.0)[None], 4, 0)
    assert [x[0].tolist() for x in c] == [[0, 1, 2, 3], [4, 5, 6, 7], [6, 7, 8, 9]]
    c = chunk_audio(torch.arange(3.0)[None], 4, 0)
    assert len(c) == 1 and c[0].shape[-1] == 3


def test_shard_range_partitions():
    from ml_audio_restoration_b200 import shard_range
    for n in (1, 7, 8, 95, 18000):
        for world in (1, 2, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_wav_round_trip(tmp_path):
    from ml_audio_restoration_b200 import load_audio, save_audio
    a = 0.5 * torch.sin(torch.arange(4410.0) * 0.05)[None].repeat(2, 1)
    p = str(tmp_path / "t.wav")
    save_audio(p, a, 44100)
    b, sr = load_audio(p, sample_rate=44100, mono=False)
    assert sr == 44100 and b.shape == a.shape and float((a - b).abs().max()) < 1e-4
    m, sr = load_audio(p, sample_rate=22050, mono=True)
    assert m.shape == (1, 2205)


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from ml_audio_restoration_b200 import shard_range, plan_chunks
from oracle import pipeline as opipe
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
N, chunk, ov = 50000, 4096, 512
starts = plan_chunks(N, chunk, ov)
lo, hi = shard_range(len(starts), rank, world)
# each rank stitches its own span from (recomputed-left-neighbour + own) chunks of a ramp signal
x = torch.arange(N, dtype=torch.float32)[None] / N
chunks = opipe.split_chunks(x, chunk, ov)
c0 = max(lo - 1, 0)
hop = chunk - ov
n_virtual = N - c0 * hop if hi == len(starts) else (hi - c0 - 1) * hop + chunk
part = opipe.stitch_chunks(chunks[c0:hi].repeat(1, 2, 1), n_virtual, chunk, ov, 1)
part = part[:, (lo - c0) * hop: (n_virtual if hi == len(starts) else (hi - c0) * hop)]
sizes = [torch.zeros(1, dtype=torch.long) for _ in range(world)]
dist.all_gather(sizes, torch.tensor([part.shape[1]]))
bufs = [torch.zeros(2, int(s)) for s in sizes]
dist.all_gather(bufs, part.contiguous()) if len(set(int(s) for s in sizes)) == 1 else None
if len(set(int(s) for s in sizes)) != 1:
    gathered = [None] * world
    dist.all_gather_object(gathered, part)
    bufs = gathered
full = torch.cat(bufs, dim=1)
assert full.shape == (2, N), full.shape
assert float((full[0] - x[0]).abs().max()) < 1e-6
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
"""


def test_two_rank_gloo_shards_cover_file(tmp_path):
    """world_size-2 CPU run of the sharding logic the multi-GPU bench uses (no data-path collective:
    the gather here is only the test's way of checking the concatenation)."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script), ROOT],
                         capture_output=True, text=True, env=env, timeout=240)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("ok") == 2


def test_bench_reference_arm_json_contract():
    """`bench.py --impl reference` (CPU oracle port) prints one JSON line with the contract's keys."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-chunks", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_bench_algorithmic_constants():
    sys.path.insert(0, ROOT)
    import bench
    # SURVEY.md 8(d): 51.661 GFLOP per source audio-second; unfused fp16 conv traffic ~354 MB per audio-second
    assert bench.CHAIN_GFLOP_PER_AUDIO_S == pytest.approx(2e-9 * (148504 * 22050 + 42656 * 22050 + 490144 * 44100), rel=1e-4)
    # 357.0 MB per audio-second layer by layer (incl. 2.8 MB for the first transient-detector layer, which runs in the conv
    # engine); the fused launches remove their intermediates: stereo dilated blocks [+ xproj] 101.6 MB, decoder layers 3 + 6
    # per side 22.6 MB, U-Net double convs 11.3 MB, super-resolution residual blocks 16.9 MB, hf_emphasis + output head 2.6 MB
    # -> 202.0 MB; with the LSTM input projection inside the scan kernel (batches beyond 8 per SM) its 256-channel output is
    # gone too -> 190.7 MB
    assert bench.conv_algorithmic_bytes_per_audio_s() == pytest.approx(202.0e6, rel=1e-3)
    assert bench.conv_algorithmic_bytes_per_audio_s(True) == pytest.approx(190.7e6, rel=1e-3)
    assert bench.CONV_GFLOP_PER_AUDIO_S - bench.CONV_GFLOP_PER_AUDIO_S_FUSED_SCAN == pytest.approx(2e-9 * 32768 * 44100, rel=1e-6)


def test_bench_dump_outputs_whole_or_fixed_sample(tmp_path):
    """`--dump-outputs`: an output up to 64 MB is written whole; a larger one as windows at fixed seeded positions (the first
    and last sample included) that hold exactly the output's samples, the same positions on every call, under 64 MB."""
    sys.path.insert(0, ROOT)
    import bench
    small = torch.randn(2, 1000)
    bench.dump_outputs(small, str(tmp_path / "small"))
    assert sorted(os.listdir(tmp_path / "small")) == ["restored.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "restored.npy"), small.numpy())
    m = bench.DUMP_MAX_BYTES // 8 + 1000                        # [2, m] float32 just over 64 MB
    big = torch.randn(2, m, generator=torch.Generator().manual_seed(5))
    for d in ("a", "b"):
        bench.dump_outputs(big, str(tmp_path / d))
    names = ["restored_window_starts.npy", "restored_windows.npy"]
    assert sorted(os.listdir(tmp_path / "a")) == names
    w, starts = np.load(tmp_path / "a" / names[1]), np.load(tmp_path / "a" / names[0])
    assert w.dtype == np.float32 and starts.dtype == np.float64
    assert w.shape == (2, bench.DUMP_WINDOWS, bench.DUMP_WINDOW) and w.nbytes + starts.nbytes <= bench.DUMP_MAX_BYTES
    assert starts[0] == 0 and starts[-1] == m - bench.DUMP_WINDOW and np.all(np.diff(starts) >= 0)
    for i in (0, 1, len(starts) // 2, len(starts) - 1):
        s = int(starts[i])
        assert np.array_equal(w[:, i], big[:, s:s + bench.DUMP_WINDOW].numpy())
    for name in names:
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(argv, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, cwd=tmp_path,
                         timeout=300)
    assert out.returncode == 2 and "error" in out.stderr, out.stderr[-2000:]
    assert not (tmp_path / "out").exists()


def test_butter_design_matches_scipy():
    """`ar_butter` (host function of the C-ABI) against scipy.signal.butter at the three designs the reference uses
    (audio_processing.py:196, 208, 220) and a few others."""
    from scipy import signal
    from ml_audio_restoration_b200 import audio_processing as ap
    for order, wn, btype in [(4, 2500 / 11025, "high"), (4, 100 / 11025, "low"), (3, 6000 / 11025, "low"),
                             (3, 8000 / 11025, "low"), (4, 2500 / 22050, "high"), (1, 0.3, "high"), (2, 0.5, "low")]:
        b, a = ap.butter(order, wn, btype)
        bs, as_ = signal.butter(order, wn, btype=btype)
        np.testing.assert_allclose(b, bs, rtol=1e-12, atol=0)
        np.testing.assert_allclose(a, as_, rtol=1e-12, atol=0)
    with pytest.raises(ValueError):
        ap.butter(4, 1.0, "low")           # scipy: "Digital filter critical frequencies must be 0 < Wn < 1"
    with pytest.raises(ValueError):
        ap.butter(4, 0.2, "band")


def test_vinyl_plan_consumes_numpy_generator_like_the_oracle():
    """The host half of simulate_vinyl_artifacts draws from np.random in the reference's order: with the same seed it
    yields the plan the (reference-pinned) oracle draws, and leaves the generator in the same state."""
    from oracle import degrade
    from ml_audio_restoration_b200 import audio_processing as ap
    for seed, n, sr, kw in [(3, 500, 22050, {"impulse_rate": 300.0}), (4, 44100, 22050, {}),
                            (5, 3000, 44100, {"add_rumble": False}), (6, 2205, 22050, {"add_rolloff": False}),
                            (7, 16, 22050, {"impulse_rate": 5000.0})]:
        np.random.seed(seed)
        mine = ap.plan_vinyl_artifacts(n, sr, **kw)
        after_mine = np.random.uniform()
        np.random.seed(seed)
        ref = degrade.draw_plan(n, sr, **kw)
        assert after_mine == np.random.uniform()
        for key in ("surface_level", "crackle_level", "rumble_level", "rolloff_hz"):
            assert mine[key] == ref[key]
        assert len(mine["pops"]) == len(ref["pops"])
        for p, q in zip(mine["pops"], ref["pops"]):
            assert (p["loc"], p["length"], bool(p["has_resonance"])) == (q["loc"], q["length"], q["resonance_freq"] is not None)
            assert p["amp_signed"] == q["amp"] * q["polarity"] and p["amp"] == q["amp"]
            assert p["tau"] == sr * q["decay_time"] * 0.3
            if q["resonance_freq"] is not None:
                assert p["omega"] == 2 * np.pi * q["resonance_freq"]
    assert ap.POP_DTYPE.itemsize == 48


def test_vinyl_artifacts_fail_loudly_on_cpu_tensors():
    from ml_audio_restoration_b200 import audio_processing as ap
    with pytest.raises(RuntimeError):
        ap.simulate_vinyl_artifacts(torch.zeros(1, 100), 22050)
    with pytest.raises(RuntimeError):
        ap.filtfilt([1.0, 0.0], [1.0, 0.0], torch.zeros(1, 100))
