"""GPU: normalize / split / overlap-add kernels and the chunked + whole-file pipelines vs the oracle."""
import numpy as np
import pytest
import torch

import oracle
from oracle import pipeline as opipe
from oracle.weights import make_input
from ml_audio_restoration_b200 import RestorationPipeline, normalize_audio
from gpu_util import assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pipe(state_dicts):
    return RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                state_dicts["stereo"], "cuda")


@pytest.fixture(scope="module")
def pipe_nosr(state_dicts):
    return RestorationPipeline.from_state_dicts(state_dicts["denoiser"], None, state_dicts["stereo"], "cuda")


def test_normalize_matches_reference_golden(golden):
    a = make_input(1, 4000)[0]
    assert_close(torch.from_numpy(golden["normalize_plain"]), normalize_audio(a.cuda()), "normalize", 1e-6, 120.0)
    z = torch.zeros(1, 100).cuda()
    assert torch.equal(normalize_audio(z).cpu(), torch.zeros(1, 100))          # rms == 0 branch
    spiky = a.clone() * 0.01
    spiky[0, 17] = 5.0
    assert_close(torch.from_numpy(golden["normalize_peak"]), normalize_audio(spiky.cuda()), "normalize peak-limit", 1e-6, 120.0)
    st = make_input(2, 3000)[:, 0]
    assert_close(torch.from_numpy(golden["normalize_stereo"]), normalize_audio(st.cuda()), "normalize stereo", 1e-6, 120.0)


@pytest.mark.parametrize("n", [1, 3, 5, 1023, 100003])
def test_normalize_odd_sizes(n):
    a = make_input(1, n, seed=n)[0]
    assert_close(opipe.normalize_audio(a), normalize_audio(a.cuda()), f"normalize n={n}", 1e-6, 110.0)


def test_whole_file_chain_matches_reference_golden(pipe, pipe_nosr, golden):
    audio = make_input(1, 3001, 1235, scale=0.3)[0]
    assert_close(torch.from_numpy(golden["chain_whole"]), pipe.restore(audio, mode="whole"), "whole-file chain")
    assert_close(torch.from_numpy(golden["chain_whole_nosr"]), pipe_nosr.restore(audio, mode="whole"), "whole-file chain (no SR)")


def test_chunked_overlap0_matches_trainer_loop_golden(pipe, golden):
    audio = make_input(1, 3001, 1235, scale=0.3)[0]
    y = pipe.restore(audio, mode="chunked", chunk_size=1000, overlap=0, normalize=False)
    assert_close(torch.from_numpy(golden["chain_trainer_chunks"]), y, "chunked overlap=0 vs trainer.py loop")


@pytest.mark.parametrize("N,chunk,ov,batch", [(9000, 2048, 256, 2), (2048, 2048, 256, 0), (2049, 2048, 256, 0),
                                              (7000, 2000, 1000, 3), (500, 2048, 0, 0)])
def test_chunked_restore_vs_oracle(pipe, state_dicts, N, chunk, ov, batch):
    audio = make_input(1, N, N, scale=0.2)[0]
    ref = opipe.restore_chunked(state_dicts, audio, chunk_size=chunk, overlap=ov)
    y = pipe.restore(audio, mode="chunked", chunk_size=chunk, overlap=ov, batch_chunks=batch)
    assert_close(ref, y, f"chunked N={N} chunk={chunk} ov={ov}")


def test_chunked_default_scheme_full_size_chunks(pipe, state_dicts):
    """Three real 2 s chunks (44100 / overlap 2052) with a ragged tail."""
    N = 2 * 42048 + 30000
    audio = make_input(1, N, 99, scale=0.2)[0]
    ref = opipe.restore_chunked(state_dicts, audio, batch=3)
    y = pipe.restore(audio, mode="chunked")
    assert y.shape == (2, 2 * N)
    assert_close(ref, y, "chunked default scheme")


def test_sharded_chunks_concatenate_to_unsharded(pipe):
    from ml_audio_restoration_b200 import plan_chunks, shard_range
    N, chunk, ov = 20000, 2048, 256
    audio = make_input(1, N, 3, scale=0.2)[0].cuda()
    full = pipe.restore(audio, mode="chunked", chunk_size=chunk, overlap=ov, normalize=False)
    n = len(plan_chunks(N, chunk, ov))
    for world in (2, 3):
        parts = [pipe.restore(audio, mode="chunked", chunk_size=chunk, overlap=ov, normalize=False,
                              chunk_range=shard_range(n, r, world)) for r in range(world)]
        got = torch.cat(parts, dim=1)
        assert got.shape == full.shape
        assert torch.equal(got, full), f"world={world}: sharded stitch differs"


def test_split_and_overlap_add_identities(pipe):
    """Size-independent properties at the BASELINE chunk geometry: stitching chunks of a constant
    signal gives the constant (windows sum to one); split then stitch at rate 1 is the identity."""
    import ctypes as C
    from ml_audio_restoration_b200 import _lib
    L = _lib.lib()
    N, chunk, ov = 10 * 42048 + 777, 44100, 2052
    n = C.c_int()
    _lib.check(L.ar_num_chunks(N, chunk, ov, C.byref(n)))
    n = n.value
    x = torch.randn(N, device="cuda")
    chunks = torch.empty(n, 1, chunk, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    _lib.check(L.ar_split_chunks(x.data_ptr(), N, chunks.data_ptr(), 0, n, chunk, ov, s))
    out = torch.empty(1, N, device="cuda")
    _lib.check(L.ar_overlap_add(chunks.data_ptr(), out.data_ptr(), N, n, 1, chunk, ov, 1, s))
    assert float((out[0] - x).abs().max()) <= 1e-6
    ref_chunks = opipe.split_chunks(x.cpu()[None], chunk, ov)
    assert torch.equal(ref_chunks, chunks.cpu())
    with pytest.raises(ValueError):
        _lib.check(L.ar_num_chunks(100, 10, 6, C.byref(C.c_int())))


@pytest.mark.parametrize("N,chunk,ov,rate,C_", [(5 * 42048 + 44100, 44100, 2052, 2, 2), (3 * 1000 + 1024, 1024, 24, 2, 2),
                                                 (7 * 96 + 128, 128, 32, 1, 1), (44100, 44100, 2052, 2, 2)])
def test_overlap_add_vector_path_equals_scalar_path_and_oracle(N, chunk, ov, rate, C_):
    """The four-samples-per-thread overlap-add (taken when chunk, hop, overlap at the output rate are multiples of 4 and the
    buffers are 16-byte aligned) against the one-sample-per-thread kernel (forced here by a 4-byte-offset output buffer):
    bit-identical; both against the oracle's stitch (oracle/pipeline.py:99)."""
    import ctypes as C
    from ml_audio_restoration_b200 import _lib
    L = _lib.lib()
    n = C.c_int()
    _lib.check(L.ar_num_chunks(N, chunk, ov, C.byref(n)))
    n = n.value
    g = torch.Generator().manual_seed(N % 977)
    y = torch.randn(n, C_, rate * chunk, generator=g)
    yd = y.cuda()
    s = torch.cuda.current_stream().cuda_stream
    out_v = torch.empty(C_, rate * N, device="cuda")
    _lib.check(L.ar_overlap_add(yd.data_ptr(), out_v.data_ptr(), N, n, C_, chunk, ov, rate, s))
    raw = torch.empty(C_ * rate * N + 1, device="cuda")
    out_s = raw[1:].view(C_, rate * N)                        # 4-byte offset: not 16-byte aligned -> scalar kernel
    assert out_s.data_ptr() % 16 != 0
    _lib.check(L.ar_overlap_add(yd.data_ptr(), out_s.data_ptr(), N, n, C_, chunk, ov, rate, s))
    assert torch.equal(out_v, out_s)
    ref = opipe.stitch_chunks(y, N, chunk, ov, rate)
    assert float((ref - out_v.cpu()).abs().max()) <= 2e-6


@pytest.mark.parametrize("name,N", [("denoiser", 5 * 44100 + 1234), ("stereo", 2 * 44100), ("super_resolution", 44100 + 17)])
def test_chunked_model_eval_matches_trainer_loop(state_dicts, name, N):
    """Drop-in of the reference's only chunked inference, Trainer.generate_test_output (trainer.py:652-681): 2 s chunks,
    zero-padded tail, per-chunk forward, `[:, :-padding]` strip, concat -- here as one batched forward."""
    from ml_audio_restoration_b200 import chunked_model_eval
    from gpu_util import make_model, assert_close
    fwd = {"denoiser": oracle.denoiser_forward, "super_resolution": oracle.super_resolution_forward, "stereo": oracle.stereo_forward}[name]
    x = make_input(1, N, seed=N % 101)[0]                      # [1, N]
    pieces = []
    for i in range(0, N, 44100):                                # the reference loop, on the oracle forward
        chunk = x[:, i:i + 44100]
        padding = 44100 - chunk.shape[1]
        if padding:
            chunk = torch.nn.functional.pad(chunk, (0, padding))
        y = fwd(state_dicts[name], chunk.unsqueeze(0)).squeeze(0)
        pieces.append(y[:, :-padding] if padding else y)
    ref = torch.cat(pieces, dim=1)
    got = chunked_model_eval(make_model(name, state_dicts[name]), x.cuda())
    assert_close(ref, got, f"chunked_model_eval {name} N={N}")


def test_generate_test_output_files(state_dicts, tmp_path):
    from ml_audio_restoration_b200 import generate_test_output, save_audio
    from ml_audio_restoration_b200.audio_processing import _read_wav
    from gpu_util import make_model
    src, dst = tmp_path / "in", tmp_path / "out"
    src.mkdir()
    save_audio(str(src / "side_a.wav"), make_input(1, 3 * 44100 + 5, seed=3)[0], 44100, encoding="pcm16")   # 44.1 kHz: resampled on the GPU
    model = make_model("stereo", state_dicts["stereo"])
    generate_test_output(model, str(src), str(dst), "epoch_1")
    out = generate_test_output(model, str(src), str(dst), "epoch_2")
    names = sorted(p.name for p in dst.iterdir())
    assert names == ["side_a_degraded_epoch_2.wav", "side_a_original.wav", "side_a_restored_epoch_2.wav"]   # epoch_1 cleaned up
    y, sr = _read_wav(out[0])
    d, _ = _read_wav(str(dst / "side_a_degraded_epoch_2.wav"))
    assert sr == 22050 and y.shape[0] == 2 and y.shape[1] == d.shape[1] == (3 * 44100 + 5 + 1) // 2


def test_config4_three_minute_side_properties_and_sampled_parity(pipe, state_dicts):
    """BASELINE config 4 at full size: a synthetic 3-minute 22.05 kHz side (95 chunks of 44100 / overlap 2052).
    Size-independent properties: the result does not depend on how the chunks are batched (one batch of 95 = tile
    groups + fused chains over many items, vs. batches of 40 with a ragged last one); sampled parity: the first two
    chunks against the oracle (normalisation off so a prefix of the file is comparable)."""
    sr, hop, chunk = 22050, 42048, 44100
    N = 180 * sr
    t = torch.arange(N, dtype=torch.float32) / sr
    g = torch.Generator().manual_seed(4)
    audio = (0.08 * torch.sin(2 * torch.pi * 220.0 * t) + 0.05 * torch.sin(2 * torch.pi * 554.4 * t + 0.3)
             + 0.02 * torch.randn(N, generator=g))
    audio[::7919] += 0.6                                   # pops
    audio = audio[None]
    dev = audio.cuda()
    y_all = pipe.restore(dev, mode="chunked", normalize=False)                       # one batch of 95 chunks
    y_b40 = pipe.restore(dev, mode="chunked", normalize=False, batch_chunks=40)      # 40 + 40 + 15
    assert y_all.shape == (2, 2 * N) and torch.isfinite(y_all).all()
    assert torch.equal(y_all, y_b40), "chunk results depend on the batch they were computed in"
    y_norm = pipe.restore(dev, mode="chunked")                                       # with input/output normalize_audio
    rms = float(y_norm.double().pow(2).mean().sqrt())
    assert abs(20 * np.log10(rms) + 20.0) < 0.05 or float(y_norm.abs().max()) <= 1.0 + 1e-6
    n_pre = hop + chunk                                                              # two chunks
    ref = opipe.restore_chunked(state_dicts, audio[:, :n_pre], normalize=False, batch=2)
    keep = 2 * hop                                                                   # output samples the 3rd chunk does not touch
    assert_close(ref[:, :keep], y_all[:, :keep], "config 4: first two chunks vs oracle")


def test_lstm_kernels_agree_at_full_length(state_dicts):
    """The tensor-core recurrence (batch > 2 sequences per SM) against the CUDA-core one (small batch) on full-length
    2 s chunks at the stereo stage's rate (88 200 steps): same chunks, different batch composition."""
    from gpu_util import make_model, assert_close as close
    m = make_model("stereo", state_dicts["stereo"])
    B = 2 * torch.cuda.get_device_properties(0).multi_processor_count + 8
    x = make_input(8, 88200, seed=21).cuda()
    xb = x.repeat((B + 7) // 8, 1, 1)[:B].contiguous()
    with torch.no_grad():
        y_small = m(x)                      # CUDA-core LSTM kernel
        y_big = m(xb)                       # tensor-core LSTM kernel
    assert torch.equal(y_big[:8], y_big[8:16]), "identical sequences in one batch must give identical outputs"
    close(y_small, y_big[:8], "stereo T=88200: tensor-core vs CUDA-core recurrence", max_abs=1e-3, min_snr=60.0)


def test_restore_stream_matches_per_file_restore(pipe):
    """The double-buffered serving loop (uploads / downloads of neighbouring files overlap the chain on their own
    streams) returns, file by file, exactly what a synchronous `restore` of each file returns -- ragged lengths, pinned
    and pageable inputs, buffers reused across files."""
    lengths = [30000, 9000, 47111, 2048, 30000, 64]
    files = [make_input(1, n, 40 + i, scale=0.2)[0] for i, n in enumerate(lengths)]
    files[2] = files[2].pin_memory()
    kw = dict(mode="chunked", chunk_size=4096, overlap=256, batch_chunks=3)
    want = [pipe.restore(f, **kw) for f in files]
    got = []
    for out in pipe.restore_stream(iter(files), **kw):
        assert not out.is_cuda and out.is_pinned()
        got.append(out.clone())             # a yielded view is only valid until the next item is requested
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == w.shape and torch.equal(g, w)
    assert list(pipe.restore_stream(iter([]))) == []
    with pytest.raises(ValueError):
        list(pipe.restore_stream(iter(files), return_device=True))


def test_bench_dump_outputs_is_the_timed_restore(tmp_path):
    """`bench.py --dump-outputs` at a small geometry, no warm-up: the JSON line reports the requested number of timed steps,
    and the dumped array is what `restore(mode="chunked")` returns for the bench's seeded input and weights."""
    import json
    import os
    import subprocess
    import sys
    from oracle.weights import make_state_dict
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    chunks = 4
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "0", "--chunks-per-step",
                          str(chunks), "--batch-chunks", str(chunks), "--no-cpu-baseline", "--no-secondary",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["warmup"] == 0 and line["parity"]["pass"]
    assert sorted(os.listdir(tmp_path)) == ["restored.npy"]
    dumped = np.load(tmp_path / "restored.npy")
    sds = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}
    p = RestorationPipeline.from_state_dicts(sds["denoiser"], sds["super_resolution"], sds["stereo"], "cuda")
    n = (chunks - 1) * bench.HOP + bench.CHUNK
    want = p.restore(bench.synth_audio(n, 1000, "cuda:0"), mode="chunked", chunk_size=bench.CHUNK, overlap=bench.OVERLAP,
                     batch_chunks=chunks)
    assert dumped.dtype == np.float32 and dumped.shape == (2, 2 * n)
    assert np.array_equal(dumped, want.cpu().numpy())
