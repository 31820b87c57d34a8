"""GPU: direct oracle parity ON THE GEOMETRY THE BENCH TIMES -- batches beyond two sequences per SM (tensor-core LSTM
`lstm_mmaw_kernel<4>`, tile groups, fused chains all active) and beyond eight per SM (`lstm_proj_kernel`: input projection
inside the scan; the chain's sub-batched conv phases around one scan), full-length 2 s chunks, BASELINE config 4 in full -- plus the LSTM carry
(`state_in`), the whole-file-exact chunked mode and the dynamic-range envelope of the fp16 storage."""
import numpy as np
import pytest
import torch

import oracle
from oracle import pipeline as opipe
from oracle.models import stereo_forward_window
from oracle.weights import calibrated_state_dicts, make_input, make_state_dict
from ml_audio_restoration_b200 import RestorationPipeline
from gpu_util import make_model, assert_close

pytestmark = pytest.mark.gpu


def big_batch():
    """Smallest batch that switches every bench-path kernel on: more than two sequences per SM."""
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count + 8      # 304 on a B200


def huge_batch():
    """Smallest convenient batch beyond eight sequences per SM: the eight-sequences-per-CTA LSTM kernel and the chain's
    sub-batched conv phases; not a multiple of 8 (a ragged last CTA)."""
    return 8 * torch.cuda.get_device_properties(0).multi_processor_count + 13     # 1197 on a B200


@pytest.fixture(scope="module")
def pipe(state_dicts):
    return RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                state_dicts["stereo"], "cuda")


def test_chain_at_bench_batch_vs_oracle(pipe, state_dicts):
    """Full chain on B >= 304 chunks of 44 100 samples (the bench's per-launch geometry scaled to the smallest batch that
    takes the same kernels); 8 of the chunks -- first, last and spread between -- meet `oracle.chain_forward` directly."""
    B, T = big_batch(), 44100
    x = make_input(B, T, seed=31)
    y = pipe.forward_chunks(x.cuda()).cpu()
    picks = sorted({0, 1, B // 5, B // 3, B // 2, 2 * B // 3, B - 2, B - 1})
    ref = opipe.chain_forward(state_dicts, x[picks])
    assert_close(ref, y[picks], f"chain B={B} T={T}: chunks {picks} vs oracle")


def test_chain_sixteen_chunks_per_sm_vs_oracle(pipe, state_dicts):
    """The bench's own launch: 16 chunks of 44 100 samples per SM (2368 on a B200) in ONE `ar_chain_forward` -- conv phases
    on sub-batches, one `lstm_proj_kernel` scan over all sequences; chunks from every sub-batch meet the oracle."""
    B, T = 16 * torch.cuda.get_device_properties(0).multi_processor_count, 44100
    free, _ = torch.cuda.mem_get_info()
    if pipe.workspace_bytes(B, T) > 0.9 * free:
        pytest.skip("not enough device memory for the 16-per-SM batch")
    x = make_input(B, T, seed=35)
    y = pipe.forward_chunks(x.cuda()).cpu()
    pipe._ws = None                                             # hand the 130 GB workspace back
    torch.cuda.empty_cache()
    picks = sorted({0, B // 4 - 1, B // 4, B // 2 + 3, 3 * B // 4, B - 1})
    ref = opipe.chain_forward(state_dicts, x[picks])
    assert_close(ref, y[picks], f"chain B={B} T={T}: chunks {picks} vs oracle")


def test_chain_sub_batched_equals_single_batches(pipe, state_dicts):
    """Beyond 8 chunks per SM the chain runs denoiser / super-resolution / encoder and the decoders on sub-batches around one
    scan: same kernels on the same operands per chunk, so the result equals the chain run on slices of at most 8 per SM
    (only the scan differs: it computes the same fp16 pre-activations itself and runs 16 sequences per CTA), and the oracle."""
    B, T = huge_batch(), 1037
    x = make_input(B, T, seed=36)
    xd = x.cuda()
    y = pipe.forward_chunks(xd)
    cut = 8 * torch.cuda.get_device_properties(0).multi_processor_count
    y_head = pipe.forward_chunks(xd[:cut].contiguous())         # tensor-core LSTM, 4 sequences per CTA: the same arithmetic
    diff = float((y[:cut] - y_head).abs().max())
    print(f"sub-batched chain vs single batch: max|diff|={diff:.3e}  bitwise equal: {torch.equal(y[:cut], y_head)}")
    assert diff <= 1e-6
    y_tail = pipe.forward_chunks(xd[cut:].contiguous())         # 13 chunks: the CUDA-core fp32 recurrence
    assert_close(y_tail, y[cut:], "last sub-batch vs its own small-batch run")
    picks = [0, cut // 2 - 1, cut // 2, cut - 1, cut, B - 1]
    assert_close(opipe.chain_forward(state_dicts, x[picks]), y[picks].cpu(), f"chain B={B} T={T}: chunks {picks} vs oracle")


@pytest.mark.parametrize("size", ["4-per-cta", "8-per-cta"])
def test_stereo_tensor_core_lstm_full_length_vs_oracle(state_dicts, size):
    """StereoSeparator alone at B >= 304 (`lstm_mmaw_kernel<4>`) and B >= 1197 (`lstm_proj_kernel`), T = 88 200 (the
    stage's length in the chain): 88 200 steps against the fp32 oracle DIRECTLY (not via the CUDA-core kernel) -- fp16
    W_hh and fp16 h feedback over the full scan is where drift would show.  Both tolerance clauses."""
    B, T = (big_batch() if size == "4-per-cta" else huge_batch()), 88200
    m = make_model("stereo", state_dicts["stereo"])
    x = make_input(B, T, seed=32)
    with torch.no_grad():
        y, st = m.forward_with_state(x.cuda())
    y, st = y.cpu(), st.cpu()
    picks = [0, B // 2 + 1, B - 5, B - 1]
    ref, (hn, cn) = oracle.stereo_forward(state_dicts["stereo"], x[picks], return_state=True)
    assert_close(ref, y[picks], f"stereo B={B} T={T}: sequences {picks} vs oracle")
    tail = slice(T - 4096, T)                                   # the end of the scan, where drift would have accumulated
    assert_close(ref[:, :, tail], y[picks][:, :, tail], "stereo: last 4096 samples of the scan")
    assert_close(hn[0], st[picks, 0], "final h after 88 200 steps", max_abs=1e-3, min_snr=50.0)
    assert_close(cn[0], st[picks, 1], "final c after 88 200 steps", max_abs=2e-3, min_snr=50.0)


def test_config4_full_side_vs_oracle(pipe, state_dicts):
    """BASELINE config 4 in full: a synthetic 3-minute 22.05 kHz side, ALL 95 chunks, input and output normalize_audio on,
    against `oracle.restore_chunked` (about half a minute of CPU)."""
    sr = 22050
    N = 180 * sr
    t = torch.arange(N, dtype=torch.float32) / sr
    g = torch.Generator().manual_seed(4)
    audio = (0.08 * torch.sin(2 * torch.pi * 220.0 * t) + 0.05 * torch.sin(2 * torch.pi * 554.4 * t + 0.3)
             + 0.02 * torch.randn(N, generator=g))
    audio[::7919] += 0.6                                        # pops
    audio = audio[None]
    y = pipe.restore(audio, mode="chunked")
    with torch.no_grad():
        ref = opipe.restore_chunked(state_dicts, audio, batch=8)
    assert y.shape == (2, 2 * N)
    assert_close(ref, y, "config 4: 180 s side, 95 chunks, normalize on, vs oracle")


@pytest.fixture(scope="module")
def calibrated():
    return calibrated_state_dicts()


@pytest.mark.parametrize("fusion,weights", [(1, "benign"), (0, "benign"), (1, "calibrated")],
                         ids=["projection-in-scan", "stored-pre-activations", "projection-in-scan-calibrated"])
def test_stereo_beyond_eight_per_sm_every_sequence_vs_oracle(state_dicts, calibrated, fusion, weights):
    """More than 8 sequences per SM: the scan kernel that computes the LSTM input projection itself (`lstm_proj_kernel`:
    tcgen05 GEMM per 8-step block + two 8-sequence recurrence groups per CTA; product path) and, layer by layer,
    `lstm_mmaw_kernel<8>` on stored pre-activations (cross-check path).  EVERY sequence of a ragged batch (1197 = 74 full
    CTAs of 16 + 13 sequences) and ragged length (203 = 25 blocks + 3 steps) against the oracle, outputs and final (h, c)
    (benign weights); the two paths against each other, bitwise (same fp16 pre-activations => the same recurrence), with
    both weight sets -- with calibrated ones the layer-by-layer path is pinned layer by layer (test_gpu_layers.py)."""
    sd = state_dicts["stereo"] if weights == "benign" else calibrated["stereo"]
    m = make_model("stereo", sd, fusion=fusion)
    B, T = huge_batch(), 203
    x = make_input(B, T, seed=37)
    with torch.no_grad():
        y, st = m.forward_with_state(x.cuda())
    if weights == "benign":
        ref, (hn, cn) = oracle.stereo_forward(sd, x, return_state=True)
        assert_close(ref, y, f"stereo B={B} T={T} (beyond 8 sequences per SM, fusion={fusion})")
        assert_close(hn[0], st[:, 0], "carried h", max_abs=1e-3, min_snr=50.0)
        assert_close(cn[0], st[:, 1], "carried c", max_abs=1e-3, min_snr=50.0)
    else:
        assert torch.isfinite(y).all() and torch.isfinite(st).all()
    if fusion == 1:
        other = make_model("stereo", sd, fusion=0)
        with torch.no_grad():
            y0, st0 = other.forward_with_state(x.cuda())
        print(f"[{weights}] projection inside the scan vs stored pre-activations: max|diff| {float((y0 - y).abs().max()):.3e}, "
              f"bitwise equal: outputs {torch.equal(y0, y)}, states {torch.equal(st0, st)}")
        assert torch.equal(y0, y), "projection inside the scan vs stored pre-activations: outputs differ"
        assert torch.equal(st0, st), "projection inside the scan vs stored pre-activations: final states differ"


@pytest.mark.parametrize("T", [1, 5, 8, 9, 16, 17, 24])
def test_scan_with_projection_short_sequences(state_dicts, T):
    """`lstm_proj_kernel` pipeline edges: one, two and three 8-step blocks, full and ragged (prologue-only GEMMs, first use of the
    second accumulator, first recycled staging slot), at a batch beyond 8 sequences per SM; every sequence vs the oracle."""
    m = make_model("stereo", state_dicts["stereo"])
    B = huge_batch()
    x = make_input(B, T, seed=40 + T)
    ref, (hn, cn) = oracle.stereo_forward(state_dicts["stereo"], x, return_state=True)
    with torch.no_grad():
        y, st = m.forward_with_state(x.cuda())
    assert_close(ref, y, f"stereo B={B} T={T}", min_snr=55.0 if T < 8 else 60.0)
    assert_close(hn[0], st[:, 0], "carried h", max_abs=1e-3, min_snr=50.0)
    assert_close(cn[0], st[:, 1], "carried c", max_abs=1e-3, min_snr=50.0)


@pytest.mark.parametrize("big", [0, 1, 2], ids=["cuda-core-lstm", "tensor-core-lstm-4", "tensor-core-lstm-8"])
def test_lstm_state_in_two_halves_equal_one_scan(state_dicts, big):
    """Feed the carried (h, c) back: forward(first half) -> state -> forward(second half, state) must reproduce the LSTM
    part of ONE scan over the whole sequence (stereo_separator.py:106-107).  The conv halves differ near the cut (each
    half zero-pads there), so outputs are compared where the cut is out of conv reach (30 samples), the states everywhere;
    both recurrence kernels; and against the oracle fed the same way."""
    m = make_model("stereo", state_dicts["stereo"])
    B, T = [(3, 3000), (big_batch(), 2048), (huge_batch(), 2048)][big]
    cut = T // 2 - (T // 2) % 8
    x = make_input(B, T, seed=33)
    xd = x.cuda()
    with torch.no_grad():
        y_full, st_full = m.forward_with_state(xd)
        y1, st1 = m.forward_with_state(xd[:, :, :cut].contiguous())
        y2, st2 = m.forward_with_state(xd[:, :, cut:].contiguous(), st1)
    picks = [0, B // 2, B - 1]
    r1, s1 = oracle.stereo_forward(state_dicts["stereo"], x[picks, :, :cut], return_state=True)
    r2, s2 = oracle.stereo_forward(state_dicts["stereo"], x[picks, :, cut:], state=s1, return_state=True)
    assert_close(r1, y1[picks], "first half vs oracle")
    assert_close(r2, y2[picks], "second half from the carried state vs oracle (state_in path)")
    assert_close(s2[0][0], st2[picks, 0], "h after both halves vs oracle", max_abs=1e-3, min_snr=50.0)
    assert_close(s2[1][0], st2[picks, 1], "c after both halves vs oracle", max_abs=1e-3, min_snr=50.0)
    # The split run differs from the single scan only through the LSTM INPUTS within encoder reach (18) of the cut,
    # which perturbs the state a little; far from the cut the outputs agree far inside the tolerance.
    assert_close(y_full[:, :, :cut - 32], y1[:, :, :cut - 32], "before the cut: identical inputs, identical scan", max_abs=1e-6, min_snr=120.0)
    assert_close(y_full[:, :, cut + 600:], y2[:, :, 600:], "after the cut: carried state == running state", max_abs=1e-3, min_snr=55.0)


@pytest.mark.parametrize("big", [False, True], ids=["cuda-core-lstm", "tensor-core-lstm"])
def test_forward_window_chain_equals_single_scan(state_dicts, big):
    """`ar_stereo_forward_window`: segments with conv halos, scan started inside the segment from the predecessor's state,
    state taken at an interior step -- chained over a sequence they reproduce the single forward EXACTLY (same kernels,
    same operands, same order), and one window call matches the oracle's restatement."""
    m = make_model("stereo", state_dicts["stereo"])
    B, T = (big_batch(), 1536) if big else (2, 5000)
    x = make_input(B, T, seed=34)
    xd = x.cuda()
    E, P, S = 40, 16, 512 if big else 1200
    with torch.no_grad():
        y_full, st_full = m.forward_with_state(xd)
        out = torch.empty_like(y_full)
        state, nseg = None, -(-T // S)
        for j in range(nseg):
            a0, a1 = j * S, min(T, (j + 1) * S)
            e0, e1 = max(0, a0 - E), min(T, a1 + E)
            y, state = m.forward_window(xd[:, :, e0:e1].contiguous(), state, lstm_start=0 if j == 0 else a0 - P - e0,
                                        state_pos=None if j == nseg - 1 else a1 - P - e0)
            out[:, :, a0:a1] = y[:, :, a0 - e0:a1 - e0]
            if j == 1:
                picks = [0, B - 1]
                ry, rs = stereo_forward_window(state_dicts["stereo"], x[picks, :, e0:e1],
                                               None if prev is None else (prev[picks, 0][None].cpu(), prev[picks, 1][None].cpu()),
                                               lstm_start=a0 - P - e0, state_pos=None if j == nseg - 1 else a1 - P - e0)
                assert_close(ry, y[picks], "one window call vs oracle restatement")
            prev = state
    diff = float((out - y_full).abs().max())
    print(f"windowed segments vs single scan: max|diff|={diff:.3e}  bitwise equal: {torch.equal(out, y_full)}")
    assert diff <= 1e-6
    assert float((state - st_full).abs().max()) <= 1e-6


def test_exact_mode_equals_whole_file_and_reference_golden(pipe, state_dicts, golden):
    """`restore(mode="exact")` -- chunk starts = 0 (mod 8), conv halos computed and discarded, LSTM (h, c) carried through
    the file -- equals `mode="whole"` (the reference's inference.py semantics) on a 6-chunk file, and the reference's own
    golden `chain_whole`.  This is the reference-PINNED stitching check (overlap-add mode is pinned by the oracle only)."""
    audio = make_input(1, 3001, 1235, scale=0.3)[0]
    whole = pipe.restore(audio, mode="whole")
    exact = pipe.restore(audio, mode="exact", chunk_size=768)            # hop 576 -> 6 chunks, ragged tail; 3 stereo segments
    diff = float((whole - exact).abs().max())
    print(f"exact vs whole: max|diff|={diff:.3e}  bitwise equal: {torch.equal(whole, exact)}")
    assert diff <= 1e-6
    assert_close(torch.from_numpy(golden["chain_whole"]), exact, "exact mode vs reference golden chain_whole")
    # longer file, default-size chunks (44 096 = 44 100 rounded down to a multiple of 8), batched stage 1
    N = 5 * 43904 + 12345
    long_audio = make_input(1, N, 77, scale=0.2)[0].cuda()
    whole = pipe.restore(long_audio, mode="whole")
    exact = pipe.restore(long_audio, mode="exact", batch_chunks=4)
    assert exact.shape == (2, 2 * N)
    diff = float((whole - exact).abs().max())
    print(f"exact vs whole, N={N}: max|diff|={diff:.3e}  bitwise equal: {torch.equal(whole, exact)}")
    assert diff <= 1e-6
    ref = opipe.restore_exact(state_dicts, make_input(1, 9000, 78, scale=0.2)[0], chunk_size=2048)
    assert_close(ref, pipe.restore(make_input(1, 9000, 78, scale=0.2)[0], mode="exact", chunk_size=2048), "exact mode vs oracle restatement")
    with pytest.raises(ValueError):
        pipe.restore(audio, mode="exact", chunk_size=256)


# ------------------------------------------------------------------------------------------------ dynamic range
def torch_eager_tf32_chain(sds, x):
    """The reference's op sequence under stock torch eager on the GPU with TF32 allowed -- PyTorch's DEFAULT for cuDNN
    convolutions (`torch.backends.cudnn.allow_tf32 = True`), i.e. what `python src/inference.py --device cuda` computes."""
    dsds = {k: {n: t.cuda() for n, t in v.items()} for k, v in sds.items()}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    import oracle.models as om
    try:
        with torch.no_grad():
            try:
                return opipe.chain_forward(dsds, x.cuda()).cpu()
            except RuntimeError:                                 # cuDNN's RNN refuses very long sequences (README.md:175)
                om.LSTM_WITHOUT_CUDNN = True
                return opipe.chain_forward(dsds, x.cuda()).cpu()
    finally:
        om.LSTM_WITHOUT_CUDNN = False
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def test_dynamic_range_full_scale_input_and_calibrated_batchnorm(calibrated):
    """The envelope of the 11-bit-significand operand path (fp16 storage == TF32 precision), with trained-like weights.

    Setting: (i) BatchNorm-calibrated checkpoints (folded gains up to ~100, activations at unit scale in every layer) and
    (ii) a full-scale input: pops that drive normalize_audio into its peak-limit branch (max |x| = 1.0).
    Range: finite output and an audited headroom of more than 30x below the fp16 limit in every one of the 49 stored tensors.
    Precision: with unit-scale activations in ~50 layers, 11-bit operands cost more than with the near-degenerate random-init
    weights of the parity tests (81 dB there): ~42 dB against the fp32 oracle (CPU emulation of operand rounding alone gives
    41-43 dB).  That is the precision class of the reference's OWN GPU path -- PyTorch runs cuDNN convolutions in TF32 by
    default -- so the assertion is: not worse than torch-eager-TF32 on the same GPU by more than 3 dB, and >= 38 dB."""
    sds = calibrated
    pipe = RestorationPipeline.from_state_dicts(sds["denoiser"], sds["super_resolution"], sds["stereo"], "cuda")
    N = 3 * 8192
    audio = make_input(1, N, 9, scale=0.02)[0]
    audio[0, 1000::4099] = 1.0                                   # pops: rms ~ 0.025 -> gain 4 -> peaks 4.0 -> peak-limited to 1.0
    a_norm = opipe.normalize_audio(audio)
    assert abs(float(a_norm.abs().max()) - 1.0) < 1e-6           # the peak-limit branch was taken
    x = a_norm.unsqueeze(0)
    with torch.no_grad():
        ref = opipe.chain_forward(sds, x)
    got = pipe.forward_chunks(x.cuda()).cpu()
    tf32 = torch_eager_tf32_chain(sds, x)
    from gpu_util import snr_db
    ours, theirs = snr_db(ref, got), snr_db(ref, tf32)
    print(f"calibrated BN, full-scale input: this repo {ours:.1f} dB, torch eager TF32 {theirs:.1f} dB vs the fp32 oracle "
          f"(max|err| {float((ref - got).abs().max()):.2e} / {float((ref - tf32).abs().max()):.2e}, max|ref| {float(ref.abs().max()):.2f})")
    assert torch.isfinite(got).all()
    assert ours >= 38.0 and ours >= theirs - 3.0
    report = pipe.check_dynamic_range(audio, chunk_size=8192)
    worst = max(report, key=report.get)
    print(f"dynamic range: {len(report)} audited tensors, largest |activation| = {report[worst]:.1f} in {worst}")
    assert len(report) >= 40 and all(np.isfinite(v) for v in report.values())
    assert report[worst] < 65504.0 / 30
    # plain synthetic weights at -20 dBFS for comparison: the audit sees every layer of the three models
    plain = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}
    p2 = RestorationPipeline.from_state_dicts(plain["denoiser"], plain["super_resolution"], plain["stereo"], "cuda")
    rep2 = p2.check_dynamic_range(audio, chunk_size=8192)
    assert set(rep2) == set(report)
    got2 = p2.restore(audio, mode="whole")
    assert_close(opipe.restore_whole(plain, audio), got2, "full-scale input (peak-limit branch), synthetic weights: whole chain vs oracle")


def test_dynamic_range_violations_are_reported_not_clamped():
    """A checkpoint outside the envelope fails loudly: (i) BN-folded weights beyond the fp16 range are refused when the
    model is packed (`ar_model_create` -> AR_ERR_WEIGHTS); (ii) activations that clip are caught by the audit that
    `restore_audio` runs first."""
    sds = {n: make_state_dict(n) for n in oracle.MODEL_NAMES}
    bad = dict(sds["stereo"])
    bad["encoder.2.1.running_var"] = torch.full_like(bad["encoder.2.1.running_var"], 1e-14)   # fold gain 3e4 * gamma ... eps floor
    bad["encoder.2.1.weight"] = bad["encoder.2.1.weight"] * 1e6
    with pytest.raises(RuntimeError, match="fp16 operand range"):
        make_model("stereo", bad)
    hot = dict(sds["super_resolution"])
    hot["initial.0.weight"] = hot["initial.0.weight"] * 1e7      # fp32 stem (not a tensor-core operand): its OUTPUT overflows fp16
    hot["initial.0.bias"] = hot["initial.0.bias"] * 1e7
    pipe = RestorationPipeline.from_state_dicts(sds["denoiser"], hot, sds["stereo"], "cuda")
    audio = make_input(1, 8192, 3, scale=0.5)[0]
    with pytest.raises(RuntimeError, match="clipped"):
        pipe.check_dynamic_range(audio, chunk_size=4096)


def test_batchnorm_eps_is_taken_from_the_module(state_dicts):
    """BatchNorm eps is a module attribute (not in the state_dict): a non-default eps reaches the fold."""
    m = make_model("stereo", state_dicts["stereo"])
    x = make_input(1, 1000, 2).cuda()
    with torch.no_grad():
        y0 = m(x)
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.eps = 0.5
        y1 = m(x)
    sd = {k: v.clone() for k, v in state_dicts["stereo"].items()}
    for k in list(sd):
        if k.endswith("running_var"):
            sd[k] = sd[k] + (0.5 - 1e-5)                         # the oracle's eps is fixed at 1e-5: shift var instead
    assert_close(oracle.stereo_forward(sd, x.cpu()), y1, "stereo with BatchNorm eps = 0.5")
    assert float((y0 - y1).abs().max()) > 1e-3


def test_two_devices_in_one_process(state_dicts):
    """One process, two GPUs: kernel attributes (opt-in shared memory) are per device -- a pipeline on cuda:1 created after
    one on cuda:0 must launch (and agree)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    audio = make_input(1, 9000, 12, scale=0.2)[0]
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        p = RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                 state_dicts["stereo"], dev)
        outs.append(p.restore(audio, mode="chunked", chunk_size=2048, overlap=256))
        xb = make_input(big_batch(), 256, 13).to(dev)            # tensor-core LSTM + every conv variant on this device too
        outs.append(p.forward_chunks(xb).cpu())
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])


def test_restore_sharded_on_one_device(pipe):
    """The sharded single-file entry point on ONE GPU (three "ranks" share cuda:0): equals the plain chunked restore."""
    from ml_audio_restoration_b200 import restore_sharded
    audio = make_input(1, 6 * 1792 + 999, 76, scale=0.2)[0]
    for normalize in (False, True):
        one = pipe.restore(audio, mode="chunked", chunk_size=2048, overlap=256, normalize=normalize)
        got = restore_sharded([pipe, pipe, pipe], audio, chunk_size=2048, overlap=256, normalize=normalize)
        assert torch.equal(one, got)
    with pytest.raises(ValueError):
        restore_sharded([], audio)


def test_one_file_sharded_over_two_gpus(state_dicts):
    """SURVEY.md 8e, by-chunk partition on REAL devices: one file split by chunk range over cuda:0 and cuda:1 (each shard
    recomputes the chunk left of its span, no exchange on the data path) equals the single-GPU chunked restore -- bit for bit
    without normalisation, and with the global input / output `normalize_audio` around it."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from ml_audio_restoration_b200 import restore_sharded
    pipes = [RestorationPipeline.from_state_dicts(state_dicts["denoiser"], state_dicts["super_resolution"],
                                                  state_dicts["stereo"], dev) for dev in ("cuda:0", "cuda:1")]
    audio = make_input(1, 7 * 1792 + 500, 77, scale=0.2)[0]            # 8 chunks of 2048 / overlap 256, ragged tail
    for normalize in (False, True):
        one = pipes[0].restore(audio, mode="chunked", chunk_size=2048, overlap=256, normalize=normalize)
        two = restore_sharded(pipes, audio, chunk_size=2048, overlap=256, normalize=normalize)
        assert two.shape == one.shape and not two.is_cuda
        if normalize:
            assert torch.allclose(one, two, rtol=0, atol=1e-6)
        else:
            assert torch.equal(one, two)
    dev_in = audio.to("cuda:0")
    assert restore_sharded(pipes, dev_in, chunk_size=2048, overlap=256).device == torch.device("cuda:0")
    # more pipelines than chunks: the surplus ones stay idle
    short = make_input(1, 1500, 78, scale=0.2)[0]
    assert torch.equal(restore_sharded(pipes, short, chunk_size=2048, overlap=256),
                       pipes[0].restore(short, mode="chunked", chunk_size=2048, overlap=256))


def test_forwards_on_two_streams_do_not_share_scratch(state_dicts):
    """Module forwards are stream-safe like the reference nn.Modules: concurrent forwards on two streams use separate
    workspaces and give the results of serial execution."""
    m = make_model("stereo", state_dicts["stereo"])
    xa, xb = make_input(6, 20000, 41).cuda(), make_input(6, 20000, 42).cuda()
    with torch.no_grad():
        ya, yb = m(xa), m(xb)
        torch.cuda.synchronize()
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        for _ in range(3):
            with torch.cuda.stream(s1):
                za = m(xa)
            with torch.cuda.stream(s2):
                zb = m(xb)
        torch.cuda.synchronize()
    assert torch.equal(ya, za) and torch.equal(yb, zb)
