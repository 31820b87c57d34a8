"""`RestorationPipeline.restore_many` (many files per chain launch), the per-sequence LSTM state capture under it
(`ar_stereo_forward_window_multi`), the window gather / kept-range scatter kernels and the CLI's directory mode."""
import ctypes as C
import os

import pytest
import torch

import oracle
from oracle.weights import make_input
from ml_audio_restoration_b200 import RestorationPipeline, _lib, save_audio
from ml_audio_restoration_b200.audio_processing import _read_wav
from ml_audio_restoration_b200.inference import EXACT_LSTM_LEAD, EXACT_STEREO_HALO, main, plan_exact_windows
from gpu_util import assert_close, make_model

E, P = EXACT_STEREO_HALO, EXACT_LSTM_LEAD


# ------------------------------------------------------------------------------------------------ planner (CPU)
def check_plan(M, S):
    W = S + 2 * E
    wins = plan_exact_windows(M, S)
    if M < W:
        assert wins is None
        return None
    assert len(wins) >= 2
    covered = []
    for j, (start, lstm_start, lo, hi, pos) in enumerate(wins):
        assert 0 <= start and start + W <= M                       # every window is W long and inside the file
        assert 0 <= lo < hi <= W
        covered.append((start + lo, start + hi))
        assert lstm_start == (0 if j == 0 else E - P)
        assert lstm_start < pos <= W - 18                         # capture where the LSTM inputs are exact
        if j + 1 < len(wins):
            nxt = wins[j + 1]
            assert nxt[0] + nxt[1] == start + pos                 # the next scan starts from this capture
    assert covered[0][0] == 0 and covered[-1][1] == M            # kept ranges tile [0, M) exactly once
    assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))
    k = wins[0][3]
    assert E <= k <= S + E
    assert wins[-1][0] == M - W and wins[-1][3] - wins[-1][2] == S + E
    return k


def test_exact_window_planner_invariants():
    for S in (16, 48, 1456, 88112):
        W = S + 2 * E
        ks = set()
        lengths = [W - 1, W, W + 1, W + 7, W + S - 1, W + S, W + S + 1, 2 * W + 3, 5 * W + 13, 17 * S + 2 * E + 5]
        lengths += list(range(W, W + 3 * S + 9))                 # every residue, so both bounds of k occur
        for M in lengths:
            k = check_plan(M, S)
            if k is not None:
                ks.add(k)
        assert min(ks) == E and max(ks) == S + E
    assert any(M % 8 for M in range(1536, 1545))


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def pipe(state_dicts):
    return RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                state_dicts["stereo"], "cuda")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["cuda_core", "mma4", "proj"])
def test_forward_window_per_item_state_pos_equals_scalar_calls(state_dicts, regime):
    """A list `state_pos` hands each item's state on at its own step in one scan; outputs and states are bitwise those of
    scalar calls on the same batch (same kernel instance), in each of the three scan-kernel regimes."""
    sms = _sms()
    B = {"cuda_core": 3, "mma4": 2 * sms + 8, "proj": 8 * sms + 13}[regime]
    T, ls = 200, 24
    m = make_model("stereo", state_dicts["stereo"])
    g = torch.Generator().manual_seed(B)
    x = (0.3 * torch.randn(B, 1, T, generator=g)).cuda()
    st = (0.5 * torch.randn(B, 2, 64, generator=g)).cuda()
    choices = [ls + 8, 96, 152, T]
    pos = [choices[(7 * b + 3) % len(choices)] for b in range(B)] if B > 3 else choices[1:]
    y, s = m.forward_window(x, st, lstm_start=ls, state_pos=pos)
    for p in choices:
        idx = torch.tensor([b for b in range(B) if pos[b] == p], dtype=torch.long, device="cuda")
        y1, s1 = m.forward_window(x, st, lstm_start=ls, state_pos=p)
        assert torch.equal(y[idx], y1[idx]) and torch.equal(s[idx], s1[idx]), f"state_pos {p}"
    for bad in ([ls] * B, [T + 1] * B, [96] * (B - 1)):
        with pytest.raises((ValueError, RuntimeError)):
            m.forward_window(x, st, lstm_start=ls, state_pos=bad)


@pytest.mark.gpu
def test_gather_windows_and_scatter_kept_equal_torch_slicing():
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(5)
    src = torch.randn(10007, generator=g).cuda()
    B, W = 7, 333
    offs = [0, 5, 17, 4000, 9674, 10007 - W, 1234]
    ws = torch.empty(_lib.WINDOW_IO_BYTES_PER_ITEM * B, dtype=torch.uint8, device="cuda")
    dst = torch.empty(B, 1, W, device="cuda")
    _lib.check(L.ar_gather_windows(src.data_ptr(), src.numel(), (C.c_int64 * B)(*offs), B, W, dst.data_ptr(), ws.data_ptr(),
                                   ws.numel(), stream))
    assert torch.equal(dst, torch.stack([src[o:o + W] for o in offs]).view(B, 1, W))
    y = torch.randn(B, 2, W, generator=g).cuda()
    out = torch.zeros(2 * 5000, device="cuda")
    lo = [0, 3, 100, 7, 0, 200, 50]
    ln = [W, 30, 233, 1, 0, 133, 17]
    dsto = [0, 2500, 400, 2900, 700, 3400, 1000, 4000, 1200, 4700, 1500, 4800, 1800, 4200]
    _lib.check(L.ar_scatter_kept(y.data_ptr(), B, W, (C.c_int64 * (2 * B))(*dsto), (C.c_int * B)(*lo), (C.c_int * B)(*ln),
                                 out.data_ptr(), out.numel(), ws.data_ptr(), ws.numel(), stream))
    ref = torch.zeros_like(out)
    for b in range(B):
        for c in range(2):
            ref[dsto[2 * b + c]:dsto[2 * b + c] + ln[b]] = y[b, c, lo[b]:lo[b] + ln[b]]
    assert torch.equal(out, ref)
    with pytest.raises(RuntimeError):                            # a window past the source end is refused on the host
        _lib.check(L.ar_gather_windows(src.data_ptr(), src.numel(), (C.c_int64 * 1)(10007 - W + 1), 1, W, dst.data_ptr(),
                                       ws.data_ptr(), ws.numel(), stream))


@pytest.mark.gpu
@pytest.mark.parametrize("normalize", [True, False])
def test_restore_many_chunked_equals_per_file_restore(pipe, normalize):
    """At most 2 chunks per SM: every file is bitwise what `restore(mode="chunked")` returns; ragged lengths, a file
    shorter than a chunk, one of exactly a chunk, host and device inputs, several groups and one file larger than a group."""
    lens = [5000, 1500, 2048, 9001, 3333, 2049, 700]
    audios = [make_input(1, n, 100 + n, scale=0.25)[0] for n in lens]
    audios = [a.cuda() if i % 2 else a for i, a in enumerate(audios)]
    outs = pipe.restore_many(audios, mode="chunked", chunk_size=2048, overlap=256, batch_chunks=4, normalize=normalize)
    assert len(outs) == len(audios)
    for a, y in zip(audios, outs):
        ref = pipe.restore(a, mode="chunked", chunk_size=2048, overlap=256, normalize=normalize)
        assert y.is_cuda == a.is_cuda and y.shape == ref.shape == (2, 2 * a.shape[-1])
        assert torch.equal(y.cpu(), ref.cpu())
    assert pipe.restore_many([]) == []
    for key in ("chunk_range", "reuse_output", "streams"):
        with pytest.raises(ValueError):
            pipe.restore_many(audios[:1], **{key: None})


@pytest.mark.gpu
def test_restore_many_exact_equals_whole_and_reference_golden(pipe, golden):
    """At most 2 files per SM: the lockstep path is within 1e-6 of `restore(mode="whole")` for every file (the bound of
    test_exact_mode_equals_whole_file_and_reference_golden), including that test's input against `chain_whole` and a
    file shorter than one window."""
    audios = [make_input(1, 3001, 1235, scale=0.3)[0], make_input(1, 2000, 3, scale=0.2)[0],
              make_input(1, 5003, 4, scale=0.2)[0].cuda(), make_input(1, 500, 5, scale=0.2)[0], make_input(1, 768, 6, scale=0.2)[0]]
    outs = pipe.restore_many(audios, mode="exact", chunk_size=768)
    for i, (a, y) in enumerate(zip(audios, outs)):
        whole = pipe.restore(a, mode="whole")
        diff = float((whole.cpu() - y.cpu()).abs().max())
        print(f"file {i} N={a.shape[-1]}: lockstep exact vs whole max|diff|={diff:.3e}")
        assert y.shape == whole.shape and diff <= 1e-6
    assert_close(torch.from_numpy(golden["chain_whole"]), outs[0], "restore_many exact vs reference golden chain_whole")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["chunked", "exact"])
def test_restore_many_tensor_core_regime(pipe, mode):
    """More than 2 chunks (windows) per SM: the tensor-core scan; within the kernel tolerance of per-file `restore`, and
    independent of the file order, bitwise."""
    n = 2 * _sms() + 4
    if mode == "chunked":
        lens = [2048 - (i % 5) * 111 for i in range(n)]
        kw = dict(chunk_size=2048, overlap=256)
    else:
        lens = [768 + (i % 4 == 3) * (1 + i % 37) for i in range(n)]
        kw = dict(chunk_size=768)
    audios = [make_input(1, m, 1000 + i, scale=0.25)[0].cuda() for i, m in enumerate(lens)]
    outs = pipe.restore_many(audios, mode=mode, **kw)
    for i in (0, 1, 2, 3, n - 1):
        assert_close(pipe.restore(audios[i], mode=mode, **kw), outs[i], f"{mode} file {i} vs per-file restore")
    perm = list(range(n))[::-1]
    outs_p = pipe.restore_many([audios[i] for i in perm], mode=mode, **kw)
    for j, i in enumerate(perm):
        assert torch.equal(outs_p[j], outs[i])


# ------------------------------------------------------------------------------------------------ CLI directory mode
@pytest.fixture()
def checkpoints(state_dicts, tmp_path):
    paths = {}
    for name in oracle.MODEL_NAMES:
        p = tmp_path / f"{name}.pth"
        torch.save({"model_state_dict": state_dicts[name]}, p)
        paths[name] = str(p)
    return paths


@pytest.mark.gpu
def test_cli_directory_mode(checkpoints, tmp_path, capsys):
    src = tmp_path / "in"
    src.mkdir()
    names = ["a.wav", "b.flac", "c.wav"]
    for i, (n, m) in enumerate(zip(names, (3001, 4100, 2500))):
        save_audio(str(src / n), make_input(1, m, 50 + i, scale=0.3)[0], 22050,
                   encoding="pcm16" if n.endswith(".flac") else None)
    (src / "notes.txt").write_text("not audio")
    ck = ["--denoiser", checkpoints["denoiser"], "--super-res", checkpoints["super_resolution"], "--stereo", checkpoints["stereo"]]
    main([str(src), str(tmp_path / "out_c"), "--mode", "chunked"] + ck)
    out = capsys.readouterr().out
    assert out.count("Saving to:") == 3 and "Dynamic-range audit:" in out and "Restoration complete!" in out
    assert sorted(os.listdir(tmp_path / "out_c")) == names
    for n in names:
        main([str(src / n), str(tmp_path / ("one_" + n)), "--mode", "chunked"] + ck)
        assert (tmp_path / "out_c" / n).read_bytes() == (tmp_path / ("one_" + n)).read_bytes(), n
    main([str(src), str(tmp_path / "out_w"), "--chunk-size", "768"] + ck)          # default mode 'whole': lockstep exact
    for n in names:
        main([str(src / n), str(tmp_path / ("whole_" + n)), "--mode", "whole"] + ck)
        y, _ = _read_wav(str(tmp_path / "out_w" / n))
        r, _ = _read_wav(str(tmp_path / ("whole_" + n)))
        tol = 1e-6 + (2.0 ** -22 if n.endswith(".flac") else 0.0)                   # one 24-bit step of the FLAC output
        assert y.shape == r.shape and float((y.cpu() - r.cpu()).abs().max()) <= tol, n
