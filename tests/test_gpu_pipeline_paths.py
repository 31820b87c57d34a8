"""One whole-file-exact path: `restore(mode="exact")` is the one-file case of `restore_many(mode="exact")`, around the
window boundaries of `plan_exact_windows`; and the one mono-input check of every entry point."""
import pytest
import torch

from oracle.weights import make_input
from ml_audio_restoration_b200 import RestorationPipeline, restore_sharded

pytestmark = pytest.mark.gpu

CHUNK = 768      # stage-1 chunks of 768 samples: S = 1456, W = 1536 with super-res (rate 2), S = 688, W = 768 without


@pytest.fixture(scope="module", params=[True, False], ids=["super-res", "no-super-res"])
def pipe(request, state_dicts):
    sr = state_dicts["super_resolution"] if request.param else None
    return RestorationPipeline.from_state_dicts(state_dicts["denoiser"], sr, state_dicts["stereo"], "cuda")


def lengths(rate):
    """Input lengths whose stage-1 signal (`rate * N` samples) lies around the window geometry of `CHUNK`: below one
    interior window's kept range S, between S and the window length W, at W, and just past W (W + 1, or W + 2 at rate 2),
    plus a file of several windows."""
    return [700, 750, 768, 769, 3001] if rate == 2 else [600, 720, 768, 769, 3001]


def test_exact_restore_equals_restore_many_and_whole(pipe):
    audios = [make_input(1, n, 400 + n, scale=0.25)[0] for n in lengths(pipe.rate)]
    many = pipe.restore_many(audios, mode="exact", chunk_size=CHUNK)
    for a, y_many in zip(audios, many):
        one = pipe.restore(a, mode="exact", chunk_size=CHUNK)
        whole = pipe.restore(a, mode="whole")
        diff = float((whole - one).abs().max())
        print(f"rate {pipe.rate}, N={a.shape[-1]}: exact vs whole max|diff|={diff:.3e}")
        assert one.shape == whole.shape == (2, pipe.rate * a.shape[-1])
        assert torch.equal(one, y_many), f"N={a.shape[-1]}: restore(mode='exact') differs from restore_many"
        assert diff <= 1e-6


@pytest.mark.parametrize("bad, exc", [(torch.zeros(2, 100), RuntimeError), (torch.zeros(1, 0), ValueError),
                                      (torch.zeros(1, 1, 100), RuntimeError)], ids=["stereo", "empty", "3d"])
def test_entry_points_refuse_non_mono_input(pipe, bad, exc):
    with pytest.raises(exc):
        pipe.restore(bad)
    with pytest.raises(exc):
        list(pipe.restore_stream([bad]))
    with pytest.raises(exc):
        pipe.restore_many([bad])
    with pytest.raises(exc):
        restore_sharded([pipe], bad)
    with pytest.raises(exc):
        pipe.check_dynamic_range(bad)
