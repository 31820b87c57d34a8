"""Drop-in `StereoSeparator` (reference: src/models/stereo_separator.py:5-122).

`forward(x[B,1,T]) -> [B,2,T]`.  Natively: k7 stem, four dilated (1,2,4,8) k3 + k1 conv pairs as
tcgen05 implicit GEMMs (dilation = a shift of the shared-memory descriptor), the LSTM input
projection as one more GEMM, a persistent register-resident LSTM recurrence kernel, the two
decoders with their first layers fused into one N=256 GEMM, and a tail kernel for the two
32->1 k7 convs that writes `[B,2,T]` directly (no permutes, no torch.cat).
`forward_with_state` exposes the LSTM carry for whole-file-exact chunking.
"""
import ctypes as C

import torch
import torch.nn as nn

from .. import _lib
from ._native import NativeModule, _Workspace, _stream_ptr


def _dilated(cin, cout, d):
    return nn.Sequential(
        nn.Conv1d(cin, cout, 3, dilation=d, padding=d), nn.BatchNorm1d(cout), nn.LeakyReLU(0.2, inplace=True),
        nn.Conv1d(cout, cout, 1), nn.BatchNorm1d(cout), nn.LeakyReLU(0.2, inplace=True))


def _decoder(hidden, b):
    layers = []
    for cin, cout in ((hidden, 4 * b), (4 * b, 2 * b), (2 * b, b)):
        layers += [nn.Conv1d(cin, cout, 7, padding=3), nn.BatchNorm1d(cout), nn.LeakyReLU(0.2, inplace=True)]
    layers.append(nn.Conv1d(b, 1, 7, padding=3))
    return nn.Sequential(*layers)


class StereoSeparator(NativeModule):
    KIND = _lib.MODEL_STEREO

    def __init__(self, base_channels: int = 32, lstm_hidden: int = 64, num_lstm_layers: int = 1):
        super().__init__()
        if (base_channels, lstm_hidden, num_lstm_layers) != (32, 64, 1):
            raise NotImplementedError(
                "the sm_100a kernels are specialised for StereoSeparator(base_channels=32, lstm_hidden=64, "
                "num_lstm_layers=1) (inference.py:85)")
        b = base_channels
        self.lstm_hidden = lstm_hidden
        stem = nn.Sequential(nn.Conv1d(1, b, 7, padding=3), nn.BatchNorm1d(b), nn.LeakyReLU(0.2, inplace=True))
        self.encoder = nn.ModuleList([stem, _dilated(b, 2 * b, 1), _dilated(2 * b, 4 * b, 2),
                                      _dilated(4 * b, 4 * b, 4), _dilated(4 * b, 4 * b, 8)])
        self.lstm = nn.LSTM(input_size=4 * b, hidden_size=lstm_hidden, num_layers=num_lstm_layers,
                            batch_first=True, bidirectional=False)
        self.left_decoder = _decoder(lstm_hidden, b)
        self.right_decoder = _decoder(lstm_hidden, b)

    def _out_shape(self, B, T):
        return (B, 2, T)

    def forward_with_state(self, x, state=None):
        """Like forward, but takes / returns the LSTM carry `[B,2,64]` (h, c)."""
        return self.forward_window(x, state, 0, None)

    def forward_window(self, x, state=None, lstm_start: int = 0, state_pos=None):
        """Forward on a window of a longer signal (`ar_stereo_forward_window`): convs over all of `x[B,1,T]`, the LSTM
        scan over steps `[lstm_start, T)` from `state` (None = zeros), returned state taken after step `state_pos - 1`
        (None = T).  `state_pos` may also be a sequence of B ints, `lstm_start < state_pos[b] <= T`: item b hands its
        state on at its own step, in the same scan (`ar_stereo_forward_window_multi`).  Building block of
        `RestorationPipeline.restore(mode="exact")` and `restore_many(mode="exact")`."""
        x = self._check_input(x)
        B, _, T = x.shape
        per_item = state_pos is not None and not isinstance(state_pos, int)
        if per_item:
            pos = [int(p) for p in state_pos]
            if len(pos) != B:
                raise ValueError(f"state_pos has {len(pos)} entries for a batch of {B}")
            pos = (C.c_int * B)(*pos)
        L = _lib.lib()
        with torch.cuda.device(x.device):
            h = self.native_handle(x.device)
            need = C.c_size_t()
            _lib.check(L.ar_model_workspace_bytes(h, B, T, C.byref(need)))
            ws = _Workspace.get(x.device, need.value)
            y = torch.empty((B, 2, T), dtype=torch.float32, device=x.device)
            new_state = torch.empty((B, 2, self.lstm_hidden), dtype=torch.float32, device=x.device)
            sin = None
            if state is not None:
                sin = state.to(device=x.device, dtype=torch.float32).contiguous()
                if sin.shape != new_state.shape:
                    raise RuntimeError(f"state must be {tuple(new_state.shape)}, got {tuple(sin.shape)}")
            sin_ptr = sin.data_ptr() if sin is not None else None
            if per_item:
                _lib.check(L.ar_stereo_forward_window_multi(h, x.data_ptr(), y.data_ptr(), B, T, int(lstm_start), pos, sin_ptr,
                                                            new_state.data_ptr(), ws.data_ptr(), ws.numel(),
                                                            _stream_ptr(x.device)))
            else:
                _lib.check(L.ar_stereo_forward_window(h, x.data_ptr(), y.data_ptr(), B, T, int(lstm_start),
                                                      T if state_pos is None else int(state_pos), sin_ptr,
                                                      new_state.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(x.device)))
        return y, new_state
