"""Restoration pipeline: drop-in `restore_audio` / CLI (reference: src/inference.py:17-143) plus
the batched, chunked GPU pipeline the reference does not have.

Two ways through the same three native models:

* whole-file (`mode="whole"`, what inference.py:59-95 does): normalise, run each model once on the
  whole `[1,1,N]` tensor, normalise.  Exact reference semantics; the stereo LSTM is one serial
  scan over the file, so this mode is latency-bound on long files.
* chunked (`mode="chunked"`, default for files longer than one chunk): split into equal chunks
  (`chunk_size`, `overlap` as in `chunk_audio`, tail zero-padded like trainer.py:660-665),
  run denoise -> super-res -> stereo on batches of chunks with the LSTM state reset per chunk
  (trainer.py:671), cross-fade overlap-add, normalise.  Chunks are independent, so batches
  shard across GPUs with no collective.
* exact (`mode="exact"`, SURVEY.md 8f n2): chunked, but equal to the whole-file result: chunk starts are multiples of 8
  (the U-Net's three pools), every chunk carries conv halos that are computed and discarded, and the stereo LSTM's
  (h, c) is carried from segment to segment of the file, so the scan is the reference's single scan
  (stereo_separator.py:106-107).  Bounded memory for files of any length; the scan of one file is serial.
"""
from __future__ import annotations

import argparse
import collections
import ctypes as C
import os
import math

import torch

from . import _lib
from .audio_processing import is_flac, load_audio, load_audio_cuda, save_audio
from .models import AudioDenoiser, AudioSuperResolution, StereoSeparator

DEFAULT_CHUNK = 44100     # 2.0 s at 22.05 kHz (trainer.py:652)
DEFAULT_OVERLAP = 2052    # hop 42048 = 0 (mod 8): chunk starts stay aligned to the U-Net's three pools
# mode="exact" (receptive fields: SURVEY.md App. E)
EXACT_HALO = 96           # input samples computed and discarded on each interior chunk edge of denoise -> super-res:
                          # denoiser reach 54 + super-res reach 15 = 69, rounded up to a multiple of 8 with margin
EXACT_STEREO_HALO = 40    # stereo stage, in ITS samples: encoder reach 18 (k7 stem 3 + dilated k3 1+2+4+8) on the side the
                          # scan enters, decoder reach 12 (four k7) on both
EXACT_LSTM_LEAD = 16      # a segment's scan starts (and its predecessor's state is taken) this many samples before the
                          # segment's kept range: >= decoder reach 12, and 40 - 16 = 24 >= encoder reach 18; multiples of 8


def plan_chunks(num_samples: int, chunk_size: int = DEFAULT_CHUNK, overlap: int = DEFAULT_OVERLAP):
    """Start offsets of the gap-free chunk plan (host mirror of `ar_num_chunks`)."""
    if not (0 <= overlap <= chunk_size // 2):
        raise ValueError("overlap must be in [0, chunk_size // 2]")
    if num_samples <= 0:
        raise ValueError("empty audio")
    hop = chunk_size - overlap
    n = 1 if num_samples <= chunk_size else math.ceil((num_samples - overlap) / hop)
    return [i * hop for i in range(n)]


def plan_exact_windows(M: int, S: int, E: int = EXACT_STEREO_HALO, P: int = EXACT_LSTM_LEAD):
    """Stereo-stage segmentation of one file of `M` samples for the lockstep whole-file-exact mode (`restore_many`):
    every window is `W = S + 2E` samples long and lies inside `[0, M)`, so the windows of many files form uniform
    launches.  Returns `[(start, lstm_start, keep_lo, keep_hi, state_pos)]` in window coordinates (the window is
    `[start, start + W)` of the file, it keeps `[start + keep_lo, start + keep_hi)`), or None when `M < W` (the file runs
    alone through `restore`).

    With `n >= 2` windows and `k = M - E - (n - 1) S`, `E <= k <= S + E`: the first window `[0, W)` keeps `[0, k)` and
    hands its state on at `k - P`, the only position that differs between files; interior windows start `E` before
    their kept range of `S` samples, scan from `E - P` and hand on at `S + E - P`; the last window `[M - W, M)` keeps its
    last `S + E` samples, so it ends at the file end without padding.  Each hand-on position is where the next window's
    scan starts, and at least `E + P` samples before its window's right edge: the LSTM inputs there are exact."""
    W = S + 2 * E
    if M < W:
        return None
    n1 = max(1, -(-(M - W) // S))                   # n - 1
    k = M - E - n1 * S
    wins = [(0, 0, 0, k, k - P)]
    for j in range(1, n1 + 1):
        a0 = k + (j - 1) * S
        last = j == n1
        start = M - W if last else a0 - E
        wins.append((start, E - P, E, E + S + (E if last else 0), S + E - P))
    return wins


def shard_range(n_items: int, rank: int, world: int):
    """Contiguous block partition `[lo, hi)` of chunk (or file) indices for one GPU (SURVEY.md 8e)."""
    lo = n_items * rank // world
    hi = n_items * (rank + 1) // world
    return lo, hi


def _load_checkpoint(module, path, device):
    ckpt = torch.load(path, map_location="cpu")
    module.load_state_dict(ckpt["model_state_dict"])
    return module.to(device).eval()


class RestorationPipeline:
    """denoise -> (super-res) -> stereo on one GPU, weights packed once (not per call)."""

    def __init__(self, denoiser: AudioDenoiser, super_res, stereo: StereoSeparator, device="cuda"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("RestorationPipeline needs a CUDA device -- this build has no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.denoiser = denoiser.to(self.device).eval()
        self.super_res = super_res.to(self.device).eval() if super_res is not None else None
        self.stereo = stereo.to(self.device).eval()
        self.rate = 2 if super_res is not None else 1
        self._chain = None
        self._chain_key = None
        self._ws = None
        self._streams = None
        self._host_out = None
        self._io_streams = None
        self._scratch = torch.empty(_lib.NORMALIZE_SCRATCH_BYTES, dtype=torch.uint8, device=self.device)

    @classmethod
    def from_state_dicts(cls, denoiser_sd, super_res_sd, stereo_sd, device="cuda"):
        den = AudioDenoiser()
        den.load_state_dict(denoiser_sd)
        sr = None
        if super_res_sd is not None:
            sr = AudioSuperResolution(upscale_factor=2)
            sr.load_state_dict(super_res_sd)
        st = StereoSeparator()
        st.load_state_dict(stereo_sd)
        return cls(den, sr, st, device)

    # ------------------------------------------------------------------ native plumbing
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def chain(self):
        hs = (self.denoiser.native_handle(self.device),
              self.super_res.native_handle(self.device) if self.super_res is not None else None,
              self.stereo.native_handle(self.device))
        key = tuple(h.value if h is not None else None for h in hs)
        if self._chain is None or key != self._chain_key:
            self.close()
            c = C.c_void_p()
            _lib.check(_lib.lib().ar_chain_create(hs[0], hs[1], hs[2], C.byref(c)))
            self._chain, self._chain_key = c, key
        return self._chain

    def close(self):
        if self._chain is not None:
            _lib.lib().ar_chain_destroy(self._chain)
            self._chain = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _workspace(self, nbytes, slot=0):
        if self._ws is None:
            self._ws = {}
        buf = self._ws.get(slot)
        if buf is None or buf.numel() < nbytes:
            self._ws[slot] = None
            buf = self._ws[slot] = torch.empty(nbytes + 4096, dtype=torch.uint8, device=self.device)
        return buf

    def _side_streams(self, n):
        if self._streams is None or len(self._streams) < n:
            self._streams = [torch.cuda.Stream(self.device) for _ in range(n)]
        return self._streams[:n]

    def _normalize_(self, t: torch.Tensor, target_db: float = -20.0):
        _lib.check(_lib.lib().ar_normalize(t.data_ptr(), t.numel(), target_db, self._scratch.data_ptr(), self._stream()))
        return t

    # ------------------------------------------------------------------ batched chain on chunks
    def forward_chunks(self, chunks: torch.Tensor, out: torch.Tensor = None, slot: int = 0) -> torch.Tensor:
        """`[B,1,T]` device chunks -> `[B,2,rate*T]` (one `ar_chain_forward` on the current stream)."""
        B, _, T = chunks.shape
        L = _lib.lib()
        with torch.cuda.device(self.device):
            c = self.chain()
            need = C.c_size_t()
            _lib.check(L.ar_chain_workspace_bytes(c, B, T, C.byref(need)))
            ws = self._workspace(need.value, slot)
            if out is None:
                out = torch.empty((B, 2, self.rate * T), dtype=torch.float32, device=self.device)
            _lib.check(L.ar_chain_forward(c, chunks.data_ptr(), out.data_ptr(), B, T, ws.data_ptr(), ws.numel(),
                                          self._stream()))
        return out

    def workspace_bytes(self, batch: int, chunk_size: int) -> int:
        """Chain workspace of one `forward_chunks` call on `batch` chunks (`ar_chain_workspace_bytes`)."""
        need = C.c_size_t()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ar_chain_workspace_bytes(self.chain(), batch, chunk_size, C.byref(need)))
        return need.value

    def max_batch(self, chunk_size: int, budget_bytes: int) -> int:
        """Largest chunk batch (up to 8 per SM) whose chain workspace fits in `budget_bytes`."""
        return max(1, int(budget_bytes // max(1, self.workspace_bytes(1, chunk_size))))

    def auto_batch(self, n_chunks: int, chunk_size: int, streams: int = 1) -> int:
        """Chunks per chain launch.  16 per SM when the workspace allows it (one tensor-core LSTM scan, 8 sequences per CTA,
        two CTAs per SM, fills the chip; the chain runs its conv phases on sub-batches around it), else 8 per SM (4 per
        CTA), else whatever fits."""
        free, _ = torch.cuda.mem_get_info(self.device)
        held = sum(b.numel() for b in (self._ws or {}).values() if b is not None)     # cached workspaces get reused
        budget = int((free + held) * 0.85) // max(1, streams)
        sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        for per_sm in (16, 8):
            if n_chunks > (per_sm // 2) * sms and self.workspace_bytes(min(n_chunks, per_sm * sms), chunk_size) <= budget:
                return min(n_chunks, per_sm * sms)
        return min(n_chunks, 8 * sms, self.max_batch(chunk_size, budget))

    # ------------------------------------------------------------------ public entry points
    @torch.no_grad()
    def restore(self, audio: torch.Tensor, mode: str = "auto", chunk_size: int = DEFAULT_CHUNK,
                overlap: int = DEFAULT_OVERLAP, batch_chunks: int = 0, normalize: bool = True,
                chunk_range=None, return_device: bool = False, reuse_output: bool = False,
                streams: int = 1) -> torch.Tensor:
        """Mono `[1,N]` (or `[N]`) float audio, host or device -> restored stereo `[2, rate*N]`.

        Host inputs are copied to the GPU (pinned memory makes the copy asynchronous) and the
        result is copied back unless `return_device`.  `chunk_range=(lo,hi)` restricts the
        chunked mode to a shard of the chunk plan and returns output samples
        `[rate*lo*hop, rate*hi*hop)` (to the file end for the last shard); shards concatenate to the
        unsharded result.  Sharded calls need `normalize=False`: `normalize_audio` is global, so the
        caller normalises the input first and the concatenated output afterwards.
        """
        if audio.dim() == 1:
            audio = audio.unsqueeze(0)
        if audio.dim() != 2 or audio.shape[0] != 1:
            raise RuntimeError(f"expected mono audio [1, N], got {tuple(audio.shape)}")
        N = audio.shape[1]
        if N == 0:
            raise ValueError("empty audio")
        if chunk_range is not None and normalize:
            raise ValueError("chunk_range needs normalize=False (normalisation is global over the file)")
        was_host = not audio.is_cuda
        with torch.cuda.device(self.device):
            a = audio.to(self.device, torch.float32, non_blocking=True).contiguous()
            if a.data_ptr() == audio.data_ptr():
                a = a.clone()
            if normalize:
                self._normalize_(a)
            if mode == "auto":
                mode = "whole" if N <= chunk_size else "chunked"
            if mode == "whole":
                y = self.forward_chunks(a.view(1, 1, N))[0]
            elif mode == "chunked":
                y = self._restore_chunked(a, N, chunk_size, overlap, batch_chunks, chunk_range, streams)
            elif mode == "exact":
                if chunk_range is not None:
                    raise ValueError("mode='exact' carries the LSTM state through the file: it cannot be sharded by chunk range")
                y = self._restore_exact(a, N, chunk_size, batch_chunks)
            else:
                raise ValueError(f"unknown mode {mode!r}")
            if normalize:
                self._normalize_(y)
            if was_host and not return_device:
                if not reuse_output:
                    return y.cpu()
                # serving loop: D2H into a cached pinned buffer (valid until the next reuse_output call)
                if self._host_out is None or self._host_out.numel() < y.numel():
                    self._host_out = torch.empty(y.numel(), dtype=torch.float32).pin_memory()
                host = self._host_out[:y.numel()].view(y.shape)
                host.copy_(y, non_blocking=True)
                torch.cuda.current_stream(self.device).synchronize()
                return host
        return y

    def restore_stream(self, audios, depth: int = 2, **restore_kwargs):
        """Serving loop over an iterable of mono host tensors (one per file): yields the restored stereo `[2, rate*N]`
        of each, in order, as a view of a pinned host buffer that stays valid until the next item is requested.

        The copies are double-buffered on their own streams (SURVEY.md 8f n1): while file i is in the chain, file i+1 is
        uploaded from pinned memory and file i-1 is downloaded, so `inference.py:47`'s H2D and `:102`'s D2H leave the
        critical path.  Inputs that are not pinned are staged through `pin_memory()` first.  `restore_kwargs` are those
        of `restore` (mode, chunk_size, overlap, batch_chunks, normalize, streams)."""
        if depth < 2:
            raise ValueError("restore_stream: depth must be >= 2")
        for key in ("return_device", "reuse_output", "chunk_range"):
            if key in restore_kwargs:
                raise ValueError(f"restore_stream does not take {key}")
        dev = self.device
        main = torch.cuda.current_stream(dev)
        if self._io_streams is None:
            self._io_streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        s_in, s_out = self._io_streams
        dev_in, in_free, host_out = [None] * depth, [None] * depth, [None] * depth
        pending = collections.deque()               # (device result kept alive, host view, D2H-done event)
        for i, audio in enumerate(audios):
            k = i % depth
            if audio.dim() == 1:
                audio = audio.unsqueeze(0)
            if audio.dim() != 2 or audio.shape[0] != 1:
                raise RuntimeError(f"expected mono audio [1, N], got {tuple(audio.shape)}")
            n = audio.shape[1]
            if n == 0:
                raise ValueError("empty audio")
            if audio.is_cuda:
                a = audio
            else:
                src = audio.to(torch.float32)
                if not src.is_pinned():
                    src = src.pin_memory()
                if dev_in[k] is None or dev_in[k].numel() < n:
                    dev_in[k] = torch.empty(n, dtype=torch.float32, device=dev)
                    s_in.wait_stream(main)          # a fresh block may still be read by kernels queued on `main`
                elif in_free[k] is not None:
                    s_in.wait_event(in_free[k])     # the chain call that read this slot `depth` files ago is done
                a = dev_in[k][:n].view(1, n)
                with torch.cuda.stream(s_in):
                    a.copy_(src, non_blocking=True)
                    uploaded = torch.cuda.Event()
                    uploaded.record(s_in)
                main.wait_event(uploaded)
            y = self.restore(a, return_device=True, **restore_kwargs)
            computed = torch.cuda.Event()
            computed.record(main)
            in_free[k] = computed
            if host_out[k] is None or host_out[k].numel() < y.numel():
                host_out[k] = torch.empty(y.numel(), dtype=torch.float32).pin_memory()
            host = host_out[k][:y.numel()].view(y.shape)
            s_out.wait_event(computed)
            with torch.cuda.stream(s_out):
                host.copy_(y, non_blocking=True)
                downloaded = torch.cuda.Event()
                downloaded.record(s_out)
            pending.append((y, host, downloaded, src if not audio.is_cuda else None))
            if len(pending) >= depth:
                _, h, ev, _ = pending.popleft()
                ev.synchronize()
                yield h
        while pending:
            _, h, ev, _ = pending.popleft()
            ev.synchronize()
            yield h

    @torch.no_grad()
    def restore_many(self, audios, mode: str = "chunked", chunk_size: int = DEFAULT_CHUNK, overlap: int = DEFAULT_OVERLAP,
                     batch_chunks: int = 0, normalize: bool = True, return_device: bool = False, **excluded) -> list:
        """Many mono files (`[1,N]` or `[N]`, host or device) -> their restored stereo `[2, rate*N]`, in input order.

        Each result is what `restore(audio, mode=mode, ...)` returns for that file (bitwise where the same kernel
        instances run, else within the tolerance between the LSTM kernels), but the files share chain launches, so a
        catalog of short sides fills the GPU like one long file does:

        * `mode="chunked"`: the chunks of a group of files form ONE `forward_chunks` batch (up to 16 per SM, the
          `auto_batch` rule); split, overlap-add and normalisation run per file on its own slice.  A file with more
          chunks than a group holds runs alone.
        * `mode="exact"`: stage 1 (denoise -> super-res) runs the full chunks of all files of a group in shared
          batches; the stereo stage runs the files in lockstep, window j of every file in ONE `forward_window` launch
          with per-file state positions (`plan_exact_windows`), the LSTM state passed from step to step.  Files
          shorter than one window run alone.

        `normalize` applies per file, as in `restore`."""
        for key in ("chunk_range", "reuse_output", "streams"):
            if key in excluded:
                raise ValueError(f"restore_many does not take {key}")
        if excluded:
            raise TypeError(f"restore_many got unexpected arguments {sorted(excluded)}")
        if mode not in ("chunked", "exact"):
            raise ValueError(f"restore_many: mode must be 'chunked' or 'exact', got {mode!r}")
        audios = list(audios)
        if not audios:
            return []
        was_host = []
        files = []
        with torch.cuda.device(self.device):
            for audio in audios:
                if audio.dim() == 1:
                    audio = audio.unsqueeze(0)
                if audio.dim() != 2 or audio.shape[0] != 1:
                    raise RuntimeError(f"expected mono audio [1, N], got {tuple(audio.shape)}")
                if audio.shape[1] == 0:
                    raise ValueError("empty audio")
                was_host.append(not audio.is_cuda)
                files.append(audio)
            run = self._many_chunked if mode == "chunked" else self._many_exact
            outs = run(files, chunk_size, overlap, batch_chunks, normalize)
        return [y.cpu() if h and not return_device else y for y, h in zip(outs, was_host)]

    def _prepared(self, audio, normalize):
        """Device copy of one mono file, normalised like `restore` normalises it."""
        a = audio.to(self.device, torch.float32, non_blocking=True).contiguous()
        if a.data_ptr() == audio.data_ptr():
            a = a.clone()
        if normalize:
            self._normalize_(a)
        return a

    def _budget(self):
        free, _ = torch.cuda.mem_get_info(self.device)
        held = sum(b.numel() for b in (self._ws or {}).values() if b is not None)
        return int((free + held) * 0.85)

    @staticmethod
    def _packed(sizes, device):
        """One buffer holding tensors of `sizes` floats, each starting on a 16-byte boundary (`ar_normalize` needs it)."""
        offs, total = [], 0
        for n in sizes:
            offs.append(total)
            total += -(-n // 4) * 4
        return torch.empty(max(total, 1), dtype=torch.float32, device=device), offs

    def _many_chunked(self, files, chunk_size, overlap, batch_chunks, normalize):
        r, L = self.rate, _lib.lib()
        counts = [len(plan_chunks(a.shape[1], chunk_size, overlap)) for a in files]
        if batch_chunks <= 0:
            batch_chunks = self.auto_batch(sum(counts), chunk_size)
        # the workspace of a full group up front: groups of slightly different sizes then share one buffer instead of
        # growing it while the previous one is still referenced
        self._workspace(self.workspace_bytes(min(batch_chunks, sum(counts)), chunk_size))
        outs = [None] * len(files)
        group = []

        def flush():
            if not group:
                return
            total = sum(counts[f] for f in group)
            buf = torch.empty((total, 1, chunk_size), dtype=torch.float32, device=self.device)
            first = 0
            for f in group:
                a = self._prepared(files[f], normalize)
                _lib.check(L.ar_split_chunks(a.data_ptr(), a.shape[1], buf[first].data_ptr(), 0, counts[f], chunk_size, overlap,
                                             self._stream()))
                first += counts[f]
            y_all = self.forward_chunks(buf)
            out, offs = self._packed([2 * r * files[f].shape[1] for f in group], self.device)
            first = 0
            for f, o in zip(group, offs):
                N = files[f].shape[1]
                y = out[o:o + 2 * r * N].view(2, r * N)
                _lib.check(L.ar_overlap_add(y_all[first].data_ptr(), y.data_ptr(), N, counts[f], 2, chunk_size, overlap, r,
                                            self._stream()))
                if normalize:
                    self._normalize_(y)
                outs[f] = y
                first += counts[f]
            group.clear()

        for f in range(len(files)):
            if counts[f] > batch_chunks:                     # larger than a group: alone, as `restore` runs it
                outs[f] = self.restore(files[f], mode="chunked", chunk_size=chunk_size, overlap=overlap,
                                       batch_chunks=batch_chunks, normalize=normalize, return_device=True)
                continue
            if sum(counts[g] for g in group) + counts[f] > batch_chunks:
                flush()
            group.append(f)
        flush()
        return outs

    def _many_exact(self, files, chunk_size, overlap, batch_chunks, normalize):
        r, E, P = self.rate, EXACT_STEREO_HALO, EXACT_LSTM_LEAD
        Lc = chunk_size - chunk_size % 8
        if Lc < 4 * EXACT_HALO:
            raise ValueError(f"mode='exact' needs chunk_size >= {4 * EXACT_HALO} (conv halos of {EXACT_HALO} samples per chunk edge)")
        S = (r * Lc - 2 * E) // 16 * 16
        W = S + 2 * E
        outs = [None] * len(files)
        plans = [plan_exact_windows(r * a.shape[1], S) for a in files]
        lock = []
        for f, plan in enumerate(plans):
            if plan is None:                                 # shorter than one window: alone
                outs[f] = self.restore(files[f], mode="exact", chunk_size=chunk_size, batch_chunks=batch_chunks,
                                       normalize=normalize, return_device=True)
            else:
                lock.append(f)
        if not lock:
            return outs
        # groups: up to 16 windows per SM (8, then whatever fits) beside the files' stage-1 signals and outputs
        sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        budget = self._budget()
        per_file = lambda f: 4 * 3 * r * files[f].shape[1]  # stage-1 signal + stereo output
        cap = 1
        for per_sm in (16, 8, 2):
            cap = min(len(lock), per_sm * sms)
            if self.stereo_workspace_bytes(cap, W) <= budget // 2:
                break
        groups, cur, used = [], [], 0
        for f in lock:
            if cur and (len(cur) == cap or used + per_file(f) > budget // 2):
                groups.append(cur)
                cur, used = [], 0
            cur.append(f)
            used += per_file(f)
        groups.append(cur)
        for grp in groups:
            self._exact_group([files[f] for f in grp], [plans[f] for f in grp], Lc, W, batch_chunks, normalize,
                              outs, grp)
        return outs

    def stereo_workspace_bytes(self, batch: int, T: int) -> int:
        need = C.c_size_t()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ar_model_workspace_bytes(self.stereo.native_handle(self.device), batch, T, C.byref(need)))
        return need.value

    def _exact_group(self, files, plans, Lc, W, batch_chunks, normalize, outs, idx):
        r, L = self.rate, _lib.lib()
        Ns = [a.shape[1] for a in files]
        Ms = [r * n for n in Ns]
        sig_all, sig_offs = self._packed(Ms, self.device)
        out_all, out_offs = self._packed([2 * m for m in Ms], self.device)
        ins = [self._prepared(a, normalize) for a in files]
        self._exact_stage1(ins, [sig_all[o:o + m].view(1, m) for o, m in zip(sig_offs, Ms)], Lc, batch_chunks)
        # lockstep over windows: files sorted by window count, so the files still running at step j are a prefix and
        # the state of step j + 1 is the first rows of the state step j returned
        order = sorted(range(len(files)), key=lambda i: -len(plans[i]))
        ws = torch.empty(_lib.WINDOW_IO_BYTES_PER_ITEM * len(files), dtype=torch.uint8, device=self.device)
        state = None
        for j in range(len(plans[order[0]])):
            act = [i for i in order if len(plans[i]) > j]
            B = len(act)
            wins = [plans[i][j] for i in act]
            x = torch.empty((B, 1, W), dtype=torch.float32, device=self.device)
            offs = (C.c_int64 * B)(*[sig_offs[i] + w[0] for i, w in zip(act, wins)])
            _lib.check(L.ar_gather_windows(sig_all.data_ptr(), sig_all.numel(), offs, B, W, x.data_ptr(), ws.data_ptr(),
                                           ws.numel(), self._stream()))
            y, state = self.stereo.forward_window(x, None if state is None else state[:B], lstm_start=wins[0][1],
                                                  state_pos=[w[4] for w in wins])
            dst = []
            for i, w in zip(act, wins):
                dst += [out_offs[i] + w[0] + w[2], out_offs[i] + Ms[i] + w[0] + w[2]]
            _lib.check(L.ar_scatter_kept(y.data_ptr(), B, W, (C.c_int64 * (2 * B))(*dst), (C.c_int * B)(*[w[2] for w in wins]),
                                         (C.c_int * B)(*[w[3] - w[2] for w in wins]), out_all.data_ptr(), out_all.numel(),
                                         ws.data_ptr(), ws.numel(), self._stream()))
        for i, (o, m) in enumerate(zip(out_offs, Ms)):
            y = out_all[o:o + 2 * m].view(2, m)
            if normalize:
                self._normalize_(y)
            outs[idx[i]] = y

    def _exact_stage1(self, ins, sigs, L, batch_chunks):
        """Stage 1 of the whole-file-exact mode (denoise -> super-res) for normalised mono `[1,N]` device signals `ins`
        into `sigs[f]` (`[1, rate*N]`).  Chunk i of a file covers input samples `[i*hop, i*hop + L)` with
        `hop = L - 2*EXACT_HALO`; the full chunks of all files run as shared batches, a ragged tail chunk runs alone at
        its true length (zero-padding it would move the file end), and only the samples further than EXACT_HALO from
        an interior chunk edge are kept.  Chunk starts are multiples of 8, so every chunk sees the pooling grid of the
        whole file (SURVEY.md App. E)."""
        r, H = self.rate, EXACT_HALO
        hop = L - 2 * H
        lib = _lib.lib()

        def stage1(x):                                  # [B,1,T] -> [B,1,r*T]
            y = self.denoiser(x)
            return self.super_res(y) if self.super_res is not None else y

        plans = []
        for a in ins:
            N = a.shape[1]
            n = 1 if N <= L else -(-(N - 2 * H) // hop)
            plans.append((N, n, n if (n - 1) * hop + L <= N else n - 1))
        full = [(f, i) for f, (_, _, n_full) in enumerate(plans) for i in range(n_full)]
        if batch_chunks <= 0:
            free, _ = torch.cuda.mem_get_info(self.device)
            sms = torch.cuda.get_device_properties(self.device).multi_processor_count
            batch_chunks = max(1, min(len(full), 8 * sms, self.max_batch(L, int(free * 0.5))))
        for b0 in range(0, len(full), batch_chunks):
            items = full[b0:b0 + batch_chunks]
            buf = torch.empty((len(items), 1, L), dtype=torch.float32, device=self.device)
            runs = []                                   # (file, first chunk, count, batch row) of each file in this batch
            for row, (f, i) in enumerate(items):
                if runs and runs[-1][0] == f:
                    runs[-1][2] += 1
                else:
                    runs.append([f, i, 1, row])
            for f, first, cnt, row in runs:
                a = ins[f]
                _lib.check(lib.ar_split_chunks(a.data_ptr(), a.shape[1], buf[row].data_ptr(), first, cnt, L, 2 * H, self._stream()))
            z_all = stage1(buf)
            for f, first, cnt, row in runs:
                N, n, _ = plans[f]
                sig, z = sigs[f], z_all[row:row + cnt]

                def keep(i):                            # kept input range of chunk i
                    return 0 if i == 0 else i * hop + H, N if i == n - 1 else (i + 1) * hop + H

                for i in range(first, first + cnt):
                    if i == 0 or i == n - 1:            # file edges keep their outer side
                        lo, hi = keep(i)
                        sig[:, r * lo:r * hi] = z[i - first, :, r * (lo - i * hop):r * (hi - i * hop)]
                i0, i1 = max(first, 1), min(first + cnt, n - 1)     # interior chunks: one strided copy
                if i1 > i0:
                    lo = i0 * hop + H
                    sig[0, r * lo:r * (lo + (i1 - i0) * hop)].view(i1 - i0, r * hop).copy_(
                        z[i0 - first:i1 - first, 0, r * H:r * (H + hop)])
        for f, (N, n, n_full) in enumerate(plans):
            if n_full < n:                              # ragged tail chunk at its true length
                start = (n - 1) * hop
                lo = 0 if n == 1 else (n - 1) * hop + H
                z = stage1(ins[f][:, start:N].reshape(1, 1, N - start).contiguous())
                sigs[f][:, r * lo:r * N] = z[0, :, r * (lo - start):r * (N - start)]

    def _restore_exact(self, a, N, chunk_size, batch_chunks):
        """Whole-file-exact chunked restoration of a normalised mono `[1,N]` device signal -> `[2, rate*N]`.

        Stage 1, denoise (-> super-res): `_exact_stage1` with `L = chunk_size` rounded down to a multiple of 8.
        Stage 2, stereo: segments of the stage-1 signal with EXACT_STEREO_HALO samples of context on both sides go
        through `forward_window` one after the other; the scan of segment j starts EXACT_LSTM_LEAD samples before the
        segment's kept range from the (h, c) its predecessor recorded at exactly that sample."""
        r, H = self.rate, EXACT_HALO
        L = chunk_size - chunk_size % 8
        if L < 4 * H:
            raise ValueError(f"mode='exact' needs chunk_size >= {4 * H} (conv halos of {H} samples per chunk edge)")
        sig = torch.empty((1, r * N), dtype=torch.float32, device=self.device)
        self._exact_stage1([a], [sig], L, batch_chunks)

        M, E, P = r * N, EXACT_STEREO_HALO, EXACT_LSTM_LEAD
        S2 = (r * L - 2 * E) // 16 * 16                 # kept samples per stereo segment
        out = torch.empty((2, M), dtype=torch.float32, device=self.device)
        state = None
        n_seg = -(-M // S2)
        for j in range(n_seg):
            a0, a1 = j * S2, min(M, (j + 1) * S2)
            e0, e1 = max(0, a0 - E), min(M, a1 + E)
            last = j == n_seg - 1
            y, state = self.stereo.forward_window(sig[:, e0:e1].reshape(1, 1, e1 - e0).contiguous(), state,
                                                  lstm_start=0 if j == 0 else a0 - P - e0,
                                                  state_pos=None if last else a1 - P - e0)
            out[:, a0:a1] = y[0, :, a0 - e0:a1 - e0]
        return out

    def check_dynamic_range(self, audio: torch.Tensor, chunk_size: int = DEFAULT_CHUNK, max_chunks: int = 8) -> dict:
        """Dynamic-range audit of this checkpoint set on `audio` (`[1,N]`, any device; normalised here like `restore`
        does): runs the three models layer by layer on up to `max_chunks` chunks -- evenly spread over the file plus the
        one holding the global peak -- and returns `{"<model>.<layer>": max |activation|}`.  Inter-layer activations
        are stored in fp16 and saturate at +-65504; raises RuntimeError naming the layer if one clipped
        (INTEGRATION.md, "dynamic range")."""
        if audio.dim() == 1:
            audio = audio.unsqueeze(0)
        N = audio.shape[1]
        with torch.cuda.device(self.device), torch.no_grad():
            a = audio.to(self.device, torch.float32).contiguous().clone()
            self._normalize_(a)
            T = min(chunk_size, N)
            n = max(1, N // T)
            picks = sorted(set([int(k * (n - 1) / max(1, max_chunks - 2)) for k in range(max_chunks - 1)] if n > 1 else [0])
                           | {min(n - 1, int(a.abs().argmax()) // T)})
            x = torch.stack([a[:, i * T:(i + 1) * T] for i in picks])          # [B,1,T]
            report = {}
            report.update({"denoiser." + k: v for k, v in self.denoiser.audit(x).items()})
            y = self.denoiser(x)
            if self.super_res is not None:
                report.update({"super_resolution." + k: v for k, v in self.super_res.audit(y).items()})
                y = self.super_res(y)
            report.update({"stereo." + k: v for k, v in self.stereo.audit(y).items()})
        clipped = [k for k, v in report.items() if not v < _lib.HALF_MAX]
        if clipped:
            raise RuntimeError("fp16 activation storage clipped (|x| >= 65504) in " + ", ".join(clipped) +
                               ": this checkpoint exceeds the dynamic-range envelope of the tensor-core path")
        return report

    def _restore_chunked(self, a, N, chunk_size, overlap, batch_chunks, chunk_range, streams=1):
        L = _lib.lib()
        n_chunks = C.c_int()
        _lib.check(L.ar_num_chunks(N, chunk_size, overlap, C.byref(n_chunks)))
        n_chunks = n_chunks.value
        lo, hi = (0, n_chunks) if chunk_range is None else chunk_range
        if not (0 <= lo < hi <= n_chunks):
            raise ValueError(f"chunk_range {chunk_range} outside [0, {n_chunks}]")
        r, hop = self.rate, chunk_size - overlap
        # a shard also recomputes the chunk before its first one, so the cross-fade at its left seam
        # is exact without any exchange between GPUs (SURVEY.md 8e)
        c0 = max(lo - 1, 0)
        cnt_all = hi - c0
        if batch_chunks <= 0:
            batch_chunks = self.auto_batch(cnt_all, chunk_size, streams)
        y_all = torch.empty((cnt_all, 2, r * chunk_size), dtype=torch.float32, device=self.device)
        firsts = list(range(c0, hi, batch_chunks))
        n_streams = max(1, min(streams, len(firsts)))
        main = torch.cuda.current_stream(self.device)
        if n_streams == 1:
            buf = torch.empty((min(batch_chunks, cnt_all), 1, chunk_size), dtype=torch.float32, device=self.device)
            for first in firsts:
                cnt = min(batch_chunks, hi - first)
                _lib.check(L.ar_split_chunks(a.data_ptr(), N, buf.data_ptr(), first, cnt, chunk_size, overlap, self._stream()))
                self.forward_chunks(buf[:cnt], y_all[first - c0:first - c0 + cnt])
        else:
            # Batches of chunks are independent: issue them round-robin on side streams (own workspace each)
            # so the latency-bound LSTM scan of one batch runs under the tensor-core convs of the next.
            side = self._side_streams(n_streams)
            ready = torch.cuda.Event()
            ready.record(main)
            bufs = [torch.empty((min(batch_chunks, cnt_all), 1, chunk_size), dtype=torch.float32, device=self.device)
                    for _ in range(n_streams)]
            for j, first in enumerate(firsts):
                k = j % n_streams
                cnt = min(batch_chunks, hi - first)
                if j < n_streams:
                    side[k].wait_event(ready)
                with torch.cuda.stream(side[k]):
                    _lib.check(L.ar_split_chunks(a.data_ptr(), N, bufs[k].data_ptr(), first, cnt, chunk_size, overlap,
                                                 side[k].cuda_stream))
                    self.forward_chunks(bufs[k][:cnt], y_all[first - c0:first - c0 + cnt], slot=k)
            for st in side:
                main.wait_stream(st)
            for t in bufs + [a, y_all]:
                for st in side:
                    t.record_stream(st)
        # stitch chunks [c0, hi) as a virtual file, then keep this shard's span [lo*hop, hi*hop) (or to N)
        n_virtual = N - c0 * hop if hi == n_chunks else (cnt_all - 1) * hop + chunk_size
        out = torch.empty((2, r * n_virtual), dtype=torch.float32, device=self.device)
        _lib.check(L.ar_overlap_add(y_all.data_ptr(), out.data_ptr(), n_virtual, cnt_all, 2, chunk_size, overlap, r,
                                    self._stream()))
        if chunk_range is None:
            return out
        begin = (lo - c0) * hop * r
        end = r * n_virtual if hi == n_chunks else (hi - c0) * hop * r
        return out[:, begin:end].contiguous()


@torch.no_grad()
def restore_sharded(pipes, audio: torch.Tensor, chunk_size: int = DEFAULT_CHUNK, overlap: int = DEFAULT_OVERLAP,
                    batch_chunks: int = 0, normalize: bool = True) -> torch.Tensor:
    """ONE file on several GPUs of this process (SURVEY.md 8e, the by-chunk partition): `pipes[r]` -- a
    `RestorationPipeline` per device, same weights -- restores the contiguous chunk range `shard_range(n_chunks, r, world)`.
    No exchange between the GPUs on the data path: every shard recomputes the one chunk left of its span, so its seam
    cross-fade is exact.  `normalize_audio` is global over the file: the input is normalised once on `pipes[0]`'s device
    and copied to the others, the shards come back to it and the concatenated output is normalised there.  The chain
    launches are asynchronous, so the shards run concurrently; the result (on `pipes[0]`'s device for device input, else
    on the host) equals `pipes[0].restore(audio, mode="chunked", ...)`."""
    if not pipes:
        raise ValueError("restore_sharded: no pipelines")
    if audio.dim() == 1:
        audio = audio.unsqueeze(0)
    if audio.dim() != 2 or audio.shape[0] != 1:
        raise RuntimeError(f"expected mono audio [1, N], got {tuple(audio.shape)}")
    N = audio.shape[1]
    n_chunks = len(plan_chunks(N, chunk_size, overlap))
    world = min(len(pipes), n_chunks)
    head = pipes[0]
    was_host = not audio.is_cuda
    with torch.cuda.device(head.device):
        a = audio.to(head.device, torch.float32).contiguous()
        if a.data_ptr() == audio.data_ptr():
            a = a.clone()
        if normalize:
            head._normalize_(a)
        torch.cuda.current_stream(head.device).synchronize()     # the peers read `a` on their own streams
    parts = []
    for r in range(world):
        p = pipes[r]
        a_r = a if p.device == head.device else a.to(p.device)
        parts.append(p.restore(a_r, mode="chunked", chunk_size=chunk_size, overlap=overlap, batch_chunks=batch_chunks,
                               normalize=False, chunk_range=shard_range(n_chunks, r, world), return_device=True))
    for r in range(world):
        torch.cuda.current_stream(pipes[r].device).synchronize()
    with torch.cuda.device(head.device):
        y = torch.cat([t.to(head.device) for t in parts], dim=1)
        if normalize:
            head._normalize_(y)
        return y.cpu() if was_host else y


def chunked_model_eval(model, waveform: torch.Tensor, chunk_size: int = 2 * 22050) -> torch.Tensor:
    """The tensor part of `Trainer.generate_test_output` (src/training/trainer.py:652-681) for ONE model: cut `[1,N]`
    into `chunk_size` pieces, zero-pad the last one, run the model per chunk (LSTM state reset per chunk), strip the
    padding and concatenate along time -> `[C_out, N_out]`.  The reference loops with batch 1 and a `.cpu()` per chunk;
    chunks are independent, so here they form ONE batch (`ar_split_chunks` with overlap 0 + one batched forward).
    As in the reference, exactly `padding` samples are stripped from the last chunk's output (`restored_chunk[:, :-padding]`,
    :674-675) whatever the model's rate, so a x2 model keeps `padding` samples computed from the zero-padded tail."""
    if waveform.dim() != 2 or waveform.shape[0] != 1 or not waveform.is_cuda:
        raise RuntimeError("chunked_model_eval: expected a mono [1,N] CUDA tensor -- this build has no CPU fallback")
    N = waveform.shape[1]
    n = (N + chunk_size - 1) // chunk_size
    a = waveform.to(torch.float32).contiguous()
    chunks = torch.empty((n, 1, chunk_size), dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().ar_split_chunks(a.data_ptr(), N, chunks.data_ptr(), 0, n, chunk_size, 0,
                                              torch.cuda.current_stream(a.device).cuda_stream))
    with torch.no_grad():
        y = model(chunks)                                   # [n, C, L]
    C_out, L = y.shape[1], y.shape[2]
    out = y.permute(1, 0, 2).reshape(C_out, n * L)
    padding = n * chunk_size - N
    return out[:, :n * L - padding].contiguous() if padding else out.contiguous()


def generate_test_output(model, test_audio_dir: str, test_output_dir: str, suffix: str, device: str = "cuda",
                         max_seconds: int = 30) -> list:
    """Drop-in for `Trainer.generate_test_output` (src/training/trainer.py:582-721) as a free function: for every
    `*.wav` and `*.flac` in `test_audio_dir` (root only) take the first `max_seconds` of the mono 22.05 kHz signal, restore
    it in 2 s chunks with `model`, and write `<stem>_original.wav` (once), `<stem>_degraded_<suffix>.wav` and
    `<stem>_restored_<suffix>.wav`; for `epoch_<k>` suffixes older epoch files of the same stem are deleted.
    Returns the restored file paths.  (mp3/ogg inputs of the reference need soundfile.)"""
    import glob
    import os
    os.makedirs(test_output_dir, exist_ok=True)
    written = []
    model.eval()
    for path in sorted(glob.glob(os.path.join(test_audio_dir, "*.wav")) + glob.glob(os.path.join(test_audio_dir, "*.flac"))):
        stem = os.path.splitext(os.path.basename(path))[0]
        original = os.path.join(test_output_dir, f"{stem}_original.wav")
        if not os.path.exists(original):
            host, sr_file = _read_original(path)
            save_audio(original, host[:, :sr_file * max_seconds], sr_file)
        wave_dev, sr = load_audio_cuda(path, sample_rate=22050, device=device)
        wave_dev = wave_dev[:, :22050 * max_seconds].contiguous()
        restored = chunked_model_eval(model, wave_dev)
        save_audio(os.path.join(test_output_dir, f"{stem}_degraded_{suffix}.wav"), wave_dev, sr)
        out_path = os.path.join(test_output_dir, f"{stem}_restored_{suffix}.wav")
        save_audio(out_path, restored, sr)
        written.append(out_path)
        if suffix.startswith("epoch_"):
            cur = int(suffix.split("_")[1])
            for pat in (f"{stem}_restored_epoch_*.wav", f"{stem}_degraded_epoch_*.wav"):
                for f in glob.glob(os.path.join(test_output_dir, pat)):
                    try:
                        if int(os.path.splitext(os.path.basename(f))[0].split("_epoch_")[1]) != cur:
                            os.remove(f)
                    except (ValueError, IndexError):
                        pass
    return written


def _read_original(path: str):
    """(mono [1,N] host float32 at the file's own rate, rate) -- the `_original.wav` copy of trainer.py:612-628."""
    from .audio_processing import _read_wav
    a, sr = _read_wav(path)
    if a.shape[0] > 1:
        a = a.mean(dim=0, keepdim=True)
    return a, sr


def restore_audio(
    input_path: str,
    output_path: str,
    denoiser_checkpoint: str = 'models/checkpoints/best_model.pth',
    super_res_checkpoint: str = 'models/checkpoints/super_resolution/best_model.pth',
    stereo_checkpoint: str = 'models/checkpoints/stereo/best_model.pth',
    sample_rate: int = 22050,
    enable_super_resolution: bool = True,
    device: str = 'cuda' if torch.cuda.is_available() else 'cpu',
    mode: str = 'whole',
    chunk_size: int = DEFAULT_CHUNK,
    overlap: int = DEFAULT_OVERLAP,
    output_encoding: str = None,
):
    """Drop-in for the reference `restore_audio` (inference.py:17-108): same positional/keyword
    arguments and progress prints; `mode`, `chunk_size`, `overlap`, `output_encoding` are additions (default
    `mode='whole'` keeps the reference's whole-file semantics; `'chunked'` is the fast path, `'exact'` the
    bounded-memory chunked form of `'whole'`).  Before restoring, the checkpoints' dynamic range is audited on a few
    chunks of the file (`RestorationPipeline.check_dynamic_range`).  The output container follows the extension of
    `output_path` (`save_audio`): a `.flac` path is encoded on the GPU straight from the restored device tensor;
    `output_encoding` ("float32" for WAV only, "pcm16", "pcm24") defaults to float32 WAV / 24-bit FLAC.
    """
    if torch.device(device).type != 'cuda':
        raise RuntimeError("restore_audio: device must be a CUDA device -- this build has no CPU fallback")
    if os.path.isdir(input_path):
        return _restore_directory(input_path, output_path, denoiser_checkpoint, super_res_checkpoint, stereo_checkpoint,
                                  sample_rate, enable_super_resolution, device, mode, chunk_size, overlap, output_encoding)
    print(f"Processing: {input_path}")
    print(f"Device: {device}")
    print("Loading audio...")
    if input_path.lower().endswith(".wav") or is_flac(input_path):
        audio, _ = load_audio_cuda(input_path, sample_rate=sample_rate, device=device)   # decode / mono mix / resample on the GPU
    else:
        audio, _ = load_audio(input_path, sample_rate=sample_rate, mono=True)
        audio = audio.pin_memory()
    print("Loading denoiser model...")
    den = _load_checkpoint(AudioDenoiser(), denoiser_checkpoint, device)
    sr = None
    if enable_super_resolution:
        print("Loading super-resolution model...")
        sr = _load_checkpoint(AudioSuperResolution(upscale_factor=2), super_res_checkpoint, device)
    print("Loading stereo separator model...")
    st = _load_checkpoint(StereoSeparator(), stereo_checkpoint, device)
    pipe = RestorationPipeline(den, sr, st, device)
    pipe.check_dynamic_range(audio, chunk_size)      # raises if this checkpoint clips the fp16 activation storage
    print("Applying denoising...")
    if enable_super_resolution:
        print("Applying bandwidth extension (22.05kHz -> 44.1kHz)...")
    print("Applying stereo separation...")
    stereo = pipe.restore(audio, mode=mode, chunk_size=chunk_size, overlap=overlap)
    out_rate = sample_rate * pipe.rate
    print(f"Saving to: {output_path}")
    save_audio(output_path, stereo, out_rate, encoding=output_encoding)
    print("Restoration complete!")
    suffix = " (bandwidth extended)" if enable_super_resolution else ""
    print(f"Output sample rate: {out_rate}Hz{suffix}")


def _restore_directory(input_dir, output_dir, denoiser_checkpoint, super_res_checkpoint, stereo_checkpoint, sample_rate,
                       enable_super_resolution, device, mode, chunk_size, overlap, output_encoding):
    """`restore_audio` on a directory: every `*.wav` / `*.flac` directly inside `input_dir`, in sorted order, into
    `output_dir` under the same file name and container.  Checkpoints load once and the files share chain launches
    (`restore_many`): `mode='chunked'` packs their chunks, `'whole'` and `'exact'` run the lockstep whole-file-exact path.
    Every file goes through the dynamic-range audit first; its share of the run time is printed."""
    import time
    names = sorted(n for n in os.listdir(input_dir)
                   if os.path.isfile(os.path.join(input_dir, n)) and os.path.splitext(n)[1].lower() in (".wav", ".flac"))
    print(f"Processing directory: {input_dir} ({len(names)} files)")
    print(f"Device: {device}")
    os.makedirs(output_dir, exist_ok=True)
    print("Loading denoiser model...")
    den = _load_checkpoint(AudioDenoiser(), denoiser_checkpoint, device)
    sr = None
    if enable_super_resolution:
        print("Loading super-resolution model...")
        sr = _load_checkpoint(AudioSuperResolution(upscale_factor=2), super_res_checkpoint, device)
    print("Loading stereo separator model...")
    st = _load_checkpoint(StereoSeparator(), stereo_checkpoint, device)
    pipe = RestorationPipeline(den, sr, st, device)
    t0 = time.perf_counter()
    audios, t_audit = [], 0.0
    for n in names:
        print(f"Loading audio: {os.path.join(input_dir, n)}")
        audio, _ = load_audio_cuda(os.path.join(input_dir, n), sample_rate=sample_rate, device=device)
        torch.cuda.synchronize(pipe.device)
        t = time.perf_counter()
        pipe.check_dynamic_range(audio, chunk_size)   # raises if this checkpoint clips the fp16 activation storage
        t_audit += time.perf_counter() - t
        audios.append(audio)
    print("Applying denoising, " + ("bandwidth extension (22.05kHz -> 44.1kHz), " if enable_super_resolution else "") +
          "stereo separation...")
    outs = pipe.restore_many(audios, mode="chunked" if mode == "chunked" else "exact", chunk_size=chunk_size,
                             overlap=overlap, return_device=True)
    out_rate = sample_rate * pipe.rate
    for n, stereo in zip(names, outs):
        print(f"Saving to: {os.path.join(output_dir, n)}")
        save_audio(os.path.join(output_dir, n), stereo, out_rate, encoding=output_encoding)
    torch.cuda.synchronize(pipe.device)
    total = time.perf_counter() - t0
    print(f"Dynamic-range audit: {t_audit:.2f} s of {total:.2f} s ({100 * t_audit / max(total, 1e-9):.0f} %)")
    print("Restoration complete!")
    suffix = " (bandwidth extended)" if enable_super_resolution else ""
    print(f"Output sample rate: {out_rate}Hz{suffix}")


def main(argv=None):
    ap = argparse.ArgumentParser(description='Restore 78rpm record audio')
    ap.add_argument('input', type=str, help='Input audio file path (a directory: every *.wav / *.flac directly inside it)')
    ap.add_argument('output', type=str, help='Output audio file path (a directory when the input is one)')
    ap.add_argument('--denoiser', type=str, default='models/checkpoints/best_model.pth', help='Path to denoiser checkpoint')
    ap.add_argument('--super-res', type=str, default='models/checkpoints/super_resolution/best_model.pth',
                    help='Path to super-resolution checkpoint')
    ap.add_argument('--stereo', type=str, default='models/checkpoints/stereo/best_model.pth',
                    help='Path to stereo separator checkpoint')
    ap.add_argument('--sample-rate', type=int, default=22050, help='Sample rate for processing')
    ap.add_argument('--no-super-res', action='store_true', help='Disable bandwidth extension (super-resolution)')
    ap.add_argument('--device', type=str, default='cuda' if torch.cuda.is_available() else 'cpu',
                    help='Device to use (cuda or cpu)')
    ap.add_argument('--mode', choices=('whole', 'chunked', 'exact'), default='whole',
                    help="'whole' = reference semantics; 'chunked' = batched 2 s chunks with overlap-add (fast path); "
                         "'exact' = chunked with conv halos and LSTM state carry, equal to 'whole' in bounded memory")
    ap.add_argument('--chunk-size', type=int, default=DEFAULT_CHUNK)
    ap.add_argument('--overlap', type=int, default=DEFAULT_OVERLAP)
    ap.add_argument('--output-encoding', choices=('float32', 'pcm16', 'pcm24'), default=None,
                    help="sample encoding of the output file (default: float32 for WAV, pcm24 for FLAC; FLAC stores integers)")
    a = ap.parse_args(argv)
    restore_audio(a.input, a.output, denoiser_checkpoint=a.denoiser, super_res_checkpoint=a.super_res,
                  stereo_checkpoint=a.stereo, sample_rate=a.sample_rate,
                  enable_super_resolution=not a.no_super_res, device=a.device, mode=a.mode,
                  chunk_size=a.chunk_size, overlap=a.overlap, output_encoding=a.output_encoding)


if __name__ == "__main__":
    main()
