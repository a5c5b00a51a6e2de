"""Live-video inference: per-chunk logits for many concurrent streams of one LFAN (optional, not in the reference).

:func:`windowing.infer_video` needs the whole video before it returns.  A :class:`StreamSession` serves up to
``max_streams`` live streams instead: ``push`` advances some of them by ``c`` frames and returns their
*provisional* logits, ``close`` ends one and returns the final logits of its last ``min(T, W)`` frames.  The
result is defined by the reference's windowed semantics (window_length W, hop_length H, trainer.py:832-913):

  * A stream has grid windows at its frames 0, H, 2H, ...  Every TemporalBlock is causal and fusion and the
    classifier are per frame, so a window's logit for frame t is fixed once frame t has arrived.
  * ``push`` returns for each frame the mean over every grid window started so far that covers it, and per
    stream ``final_upto = max(0, T_now - W)``: frames below it never change again.
  * Only the last ``min(T, W)`` frames depend on the length T: a grid window that does not complete does not
    exist, the tail window at T - W does, and a video shorter than W is one window padded by repeating its last
    frame.  ``close`` recomputes them from the retained inputs and logits.

The provisional logits of frames ``< T - min(T, W)`` followed by ``close``'s result equal
``infer_video(model, video, feats, W, H)`` bit for bit when the backbone embeddings are equal (always for
pre-extracted modalities; for 'video' / 'logmel' when the IR-50 / VGGish plan picks the same kernels at both
pass sizes, the dependence ``infer_videos`` documents).  The TCN and fusion kernels are the offline ones,
unchanged; csrc/stream.cu holds the per-stream state around them (DESIGN.md section 5.16).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import _capi
from .windowing import gather_windows, preprocess_frames, window_starts


# ----------------------------------------------------------------------------------------------
# Window bookkeeping (pure host logic)
# ----------------------------------------------------------------------------------------------
def n_window_slots(window_length: int, hop_length: int, max_chunk: int) -> int:
    """TCN state slots per stream: the most grid windows that can overlap one chunk of ``max_chunk`` frames,
    ceil((W + c - 1) / H) (2 = ceil(W / H) at W = 300, H = 200 for chunks up to 101 frames)."""
    return -(-(window_length + max_chunk - 1) // hop_length)


def n_logit_slots(window_length: int, hop_length: int, max_chunk: int) -> int:
    """Logit ring slots per stream: a completed window stays needed by ``close`` until the stream is 2W - 1
    frames past its start, so the ring holds every window started in 2W - 1 frames (and at least the active ones)."""
    return max(-(-(2 * window_length - 1) // hop_length), n_window_slots(window_length, hop_length, max_chunk))


def active_windows(t_now: int, chunk: int, window_length: int, hop_length: int) -> List[int]:
    """Indices k of the grid windows (start k * H) that cover a frame of [t_now, t_now + chunk)."""
    lo = max(0, (t_now - window_length) // hop_length + 1)
    hi = (t_now + chunk - 1) // hop_length
    return list(range(lo, hi + 1))


def final_upto(length: int, window_length: int) -> int:
    """Frames below this index of a stream of ``length`` frames so far never change again."""
    return max(0, length - window_length)


def close_range(length: int, window_length: int) -> Tuple[int, int]:
    """The frames [first, length) whose logits ``close`` returns."""
    return length - min(length, window_length), length


def close_windows(length: int, window_length: int, hop_length: int) -> List[Tuple[int, bool]]:
    """(start, recomputed) of the windows of ``window_starts(length)`` that cover a frame of ``close_range``, in
    start order; ``recomputed`` marks the tail window (and the single padded window of a short video), which
    ``close`` runs through the head again -- every other one is a completed grid window whose logits are kept."""
    starts = window_starts(length, window_length, hop_length)
    if length < window_length:
        return [(0, True)]
    first = length - window_length
    has_tail = first % hop_length != 0
    return [(s, has_tail and i == len(starts) - 1) for i, s in enumerate(starts) if s + window_length > first]


def step_table(streams: Sequence[Tuple[int, int, int]], chunk: int, window_length: int, hop_length: int,
               n_slots: int, n_lslots: int) -> np.ndarray:
    """The cer_stream_entry table of one step: streams = (sid, t_now, parity) per pushed stream ->
    int32 [len(streams) * n_slots, 8], each stream's active windows first, in start order."""
    tab = np.zeros((len(streams) * n_slots, len(_capi.STREAM_ENTRY_FIELDS)), dtype=np.int32)
    for i, (sid, t_now, parity) in enumerate(streams):
        ks = active_windows(t_now, chunk, window_length, hop_length)
        if len(ks) > n_slots:
            raise ValueError(f"{len(ks)} windows overlap the chunk but the session has {n_slots} slots")
        rows = tab[i * n_slots:(i + 1) * n_slots]
        rows[:, 0], rows[:, 4], rows[:, 5] = sid, t_now, parity
        for j, k in enumerate(ks):
            rows[j, 1], rows[j, 2], rows[j, 3], rows[j, 6] = k % n_slots, k % n_lslots, k * hop_length, 1
    return tab


# ----------------------------------------------------------------------------------------------
# Session
# ----------------------------------------------------------------------------------------------
class StreamSession:
    """Up to ``max_streams`` live streams of one eval-mode LFAN, pushed ``<= max_chunk`` frames at a time.

    Per push input (n streams, c frames each): 'video' as stored uint8 crops [n, c, H, W, 3] or fp32
    [n, c, 3, 40, 40]; 'logmel' as VGGish examples [n, c, 96, 64]; a pre-extracted modality as [n, c, D_m].
    One push is one backbone pass over the n * c frames and one fixed sequence of head launches (captured as a
    CUDA graph per (n, c), like LFAN.forward_features; eager when capture is off or fails)."""

    def __init__(self, model, max_streams: int = 256, max_chunk: int = 30, window_length: int = 300,
                 hop_length: int = 200):
        from .modules import LFAN
        if not isinstance(model, LFAN):
            raise TypeError("StreamSession streams LFAN only: the CAN / JMT / MT heads are not streamed (JMT / MT attend "
                            "over the whole window, so a frame's logits depend on later frames)")
        if not (1 <= hop_length <= window_length):
            raise ValueError(f"need 1 <= hop_length <= window_length, got {hop_length}, {window_length}")
        if max_streams < 1 or max_chunk < 1:
            raise ValueError("max_streams and max_chunk must be positive")
        _capi.require_gpu()
        self.model = model
        self._check_model()
        self.max_streams, self.max_chunk = int(max_streams), int(max_chunk)
        self.W, self.H = int(window_length), int(hop_length)
        self.n_slots = n_window_slots(self.W, self.H, self.max_chunk)
        self.n_lslots = n_logit_slots(self.W, self.H, self.max_chunk)
        self.modalities = list(model.modality)
        self.device = model.regressor.weight.device
        self._len: Dict[int, int] = {}
        self._parity: Dict[int, int] = {}
        self._free = list(range(self.max_streams - 1, -1, -1))
        self._eng = None
        self._pack()

    # -- state ------------------------------------------------------------------------------
    def _check_model(self):
        if self.model.training:
            raise RuntimeError("StreamSession runs the inference kernels: call model.eval() first")

    def _pack(self):
        """(Re)bind the model's packed head; allocate the rings and step buffers on first use."""
        tcn, fus = self.model._head_engines()
        self._eng, self._graphs = (tcn, fus), {}
        dev, S, ne, cm = self.device, self.max_streams, self.max_streams * self.n_slots, self.max_chunk
        f32 = dict(dtype=torch.float32, device=dev)
        self.n_out = fus.n_out
        fresh = not hasattr(self, "_tab")
        if fresh:
            self._tab = torch.zeros(ne, len(_capi.STREAM_ENTRY_FIELDS), dtype=torch.int32, device=dev)
            self._lring = torch.zeros(S, self.n_lslots, self.W, self.n_out, **f32)
            self._out = torch.empty(S * cm * self.n_out, **f32)
            self._in, self._inring, self._rings, self._staged, self._outs, self._ws, self._gath = {}, {}, {}, {}, {}, {}, {}
        self._blocks, self._rows = {}, {}
        for m in self.modalities:
            eng = tcn[m]
            if eng.precision != "tf32":      # LFAN packs its TCNs for the tensor-core kernel; the staging assumes its padding
                raise NotImplementedError(f"'{m}': StreamSession runs the tensor-core TCN kernel only")
            blocks = eng.blocks
            rows = [2 * (b.kernel_size - 1) * b.dilation for b in blocks]
            self._blocks[m], self._rows[m] = blocks, rows
            if not fresh:
                continue
            self._in[m] = torch.empty(S * cm * eng.c_in, **f32)
            self._inring[m] = torch.zeros(S, self.W, eng.c_in, **f32)
            self._rings[m] = [torch.zeros(S * self.n_slots * 2 * max(r, 1) * b.c_in, **f32) for b, r in zip(blocks, rows)]
            self._staged[m] = [torch.empty(ne * (r + cm) * b.c_in, **f32) for b, r in zip(blocks, rows)]
            self._outs[m] = [torch.empty(ne * (r + cm) * b.c_out, **f32) for b, r in zip(blocks, rows)]
            self._ws[m] = torch.empty(max(ne * (r + cm) * b.c_out for b, r in zip(blocks, rows)) * 4, dtype=torch.uint8,
                                      device=dev)
            self._gath[m] = torch.empty(ne * cm * eng.c_out, **f32)

    def _engines(self):
        eng = self.model._head_engines()
        if eng is not self._eng:                    # weights changed: the captured graphs hold the old packing
            self._pack()
        return self._eng

    def state_bytes(self) -> int:
        """Device memory one stream slot holds across steps (rings), in bytes."""
        n = self.n_lslots * self.W * self.n_out
        for m in self.modalities:
            n += self.W * self._inring[m].shape[-1]
            n += sum(self.n_slots * 2 * r * b.c_in for b, r in zip(self._blocks[m], self._rows[m]))
        return 4 * n

    def open(self) -> int:
        """A new stream at its frame 0; returns its id."""
        if not self._free:
            raise RuntimeError(f"all {self.max_streams} stream slots are open")
        sid = self._free.pop()
        self._len[sid], self._parity[sid] = 0, 0
        return sid

    def length(self, sid: int) -> int:
        return self._len[sid]

    # -- push -------------------------------------------------------------------------------
    def _chunk_features(self, inputs: Dict[str, torch.Tensor], n: int) -> Tuple[int, Dict[str, torch.Tensor]]:
        if "wave" in inputs:
            raise ValueError("'wave' cannot be streamed: the VGGish example of a frame needs 0.96 s of audio after it; "
                             "push 'logmel' examples [n, c, 96, 64] instead")
        chunk, out = None, {}
        for m in self.modalities:
            if m not in inputs:
                raise KeyError(f"push needs the '{m}' input")
            x = inputs[m]
            if x.dim() < 3 or x.shape[0] != n:
                raise ValueError(f"'{m}': expected [n={n}, c, ...], got {tuple(x.shape)}")
            c = int(x.shape[1])
            if chunk is None:
                chunk = c
            elif c != chunk:
                raise ValueError(f"every modality must carry the same number of frames ({chunk} != {c} for '{m}')")
            x = x.reshape(n * c, *x.shape[2:])
            if m == "video":
                if x.dtype == torch.uint8:
                    x = preprocess_frames(self.model, x)
                x = self.model.spatial["visual"](x.float())
            elif m == "logmel":
                x = self.model.spatial["audio"](x.float())
            elif x.dim() != 2:
                raise ValueError(f"'{m}': expected [n, c, D], got {tuple(inputs[m].shape)}")
            out[m] = x
        if not chunk or chunk > self.max_chunk:
            raise ValueError(f"chunk of {chunk} frames: need 1..{self.max_chunk}")
        return chunk, out

    def _run_head(self, n: int, c: int) -> None:
        """The fixed launch sequence of one step over the session's buffers (captured per (n, c))."""
        lib, chk = _capi.lib(), _capi.check
        st = _capi.current_stream_ptr(self.device)
        tcn, fus = self._eng
        ne, tab = n * self.n_slots, self._tab.data_ptr()
        feats = []
        for m in self.modalities:
            eng = tcn[m]
            d_in = eng.c_in
            chk(lib.cer_stream_retain(tab, n, self.n_slots, c, self._in[m].data_ptr(), d_in, self.W,
                                      self._inring[m].data_ptr(), st), "cer_stream_retain")
            src, src_dim, src_len, src_rows = self._in[m], d_in, 0, 0
            for b, (blk, rows) in enumerate(zip(self._blocks[m], self._rows[m])):
                L = rows + c
                staged, out = self._staged[m][b], self._outs[m][b]
                chk(lib.cer_stream_stage(tab, ne, self.n_slots, c, rows, blk.c_in, src.data_ptr(), src_dim, src_len,
                                         src_rows, self._rings[m][b].data_ptr(), staged.data_ptr(), st), "cer_stream_stage")
                chk(lib.cer_tcn_block_tc_forward(C.byref(blk), staged.data_ptr(), out.data_ptr(), ne, L,
                                                 self._ws[m].data_ptr(), self._ws[m].numel(), st),
                    "cer_tcn_block_tc_forward")
                src, src_dim, src_len, src_rows = out, blk.c_out, L, rows
            g = self._gath[m]
            chk(lib.cer_stream_gather(tab, ne, c, src.data_ptr(), src_rows, src_dim, g.data_ptr(), st), "cer_stream_gather")
            feats.append(g[:ne * c * src_dim].view(ne * c, src_dim))
        logits = fus.forward(feats)
        chk(lib.cer_stream_average(tab, n, self.n_slots, c, self.W, self.n_out, logits.data_ptr(), self._out.data_ptr(),
                                   self._lring.data_ptr(), self.n_lslots, st), "cer_stream_average")

    def _use_graph(self) -> bool:
        return (self.model.head_cuda_graph and os.environ.get("CER_HEAD_GRAPH", "1") != "0"
                and not torch.cuda.is_current_stream_capturing())

    @torch.no_grad()
    def push(self, ids: Sequence[int], inputs: Dict[str, torch.Tensor]) -> Tuple[torch.Tensor, List[int]]:
        """Advance streams ``ids`` by c frames -> (provisional logits [n, c, n_out], final_upto per stream)."""
        self._check_model()
        ids = [int(i) for i in ids]
        n = len(ids)
        if n == 0:
            raise ValueError("push needs at least one stream")
        if len(set(ids)) != n or any(i not in self._len for i in ids):
            raise ValueError(f"stream ids must be distinct open streams, got {ids}")
        self._engines()
        with torch.cuda.device(self.device):
            c, x = self._chunk_features(inputs, n)
            for m in self.modalities:
                d = self._inring[m].shape[-1]
                if x[m].shape[1] != d:
                    raise ValueError(f"'{m}': expected {d} features per frame, got {x[m].shape[1]}")
                self._in[m][:n * c * d].view(n * c, d).copy_(x[m])
            tab = step_table([(i, self._len[i], self._parity[i]) for i in ids], c, self.W, self.H, self.n_slots,
                             self.n_lslots)
            self._tab[:tab.shape[0]].copy_(torch.from_numpy(tab).pin_memory(), non_blocking=True)
            g = self._graphs.get((n, c)) if self._use_graph() else False
            if g:
                g.replay()
            else:
                # capture records the launches without running them: the eager run is this step's
                self._run_head(n, c)
                if g is None:
                    try:
                        graph = torch.cuda.CUDAGraph()
                        torch.cuda.synchronize(self.device)
                        with torch.cuda.graph(graph):
                            self._run_head(n, c)
                        self._graphs[(n, c)] = graph
                    except Exception:                     # capture not possible here: stay eager for this shape
                        self._graphs[(n, c)] = False
            out = self._out[:n * c * self.n_out].view(n, c, self.n_out).clone()
        for i in ids:
            self._len[i] += c
            self._parity[i] ^= 1
        return out, [final_upto(self._len[i], self.W) for i in ids]

    # -- close ------------------------------------------------------------------------------
    @torch.no_grad()
    def close(self, sid: int) -> torch.Tensor:
        """End stream ``sid`` -> the final logits [min(T, W), n_out] of its frames T - min(T, W) .. T - 1, and free
        its slot."""
        from .engine import stitch_windows
        if sid not in self._len:
            raise ValueError(f"stream {sid} is not open")
        self._check_model()
        self._engines()
        T, W = self._len.pop(sid), self.W
        del self._parity[sid]
        self._free.append(sid)
        if T == 0:
            return torch.empty(0, self.n_out, dtype=torch.float32, device=self.device)
        first, _ = close_range(T, W)
        wins = close_windows(T, W, self.H)
        with torch.cuda.device(self.device):
            rows = torch.arange(first, T, device=self.device) % W
            tail = None
            if any(rec for _, rec in wins):
                batch = {m: gather_windows(self._inring[m][sid][rows], [0], W).contiguous() for m in self.modalities}
                tail = self.model.forward_features(batch)[0]
            logits = torch.stack([tail if rec else self._lring[sid, (s // self.H) % self.n_lslots] for s, rec in wins])
            starts = torch.tensor([s - first for s, _ in wins], dtype=torch.int32).to(self.device, non_blocking=True)
            return stitch_windows(logits, starts, W)[:T - first]
