"""Live-video inference: per-chunk logits for many concurrent streams of one LFAN or CAN (optional, not in the reference).

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

A CAN has no windows: the reference runs it over the whole video, its TemporalBlocks are causal and its fusion and
tail are per frame, so a frame's logits are final as soon as it arrives.  Each stream is one TCN state slot that
starts at frame 0 and never ends, ``push`` returns final logits (``final_upto`` is the stream's length) and ``close``
returns only what was still held back.  The fusion head + tail run as one row-invariant kernel
(cer_can_head_forward), so a stream's logits do not depend on the other streams of a push or on its chunk sizes
(DESIGN.md section 5.18).

A JMT / MT (opened with ``max_frames``) attends over the whole sequence, so no logit is final before the stream ends.
Its backbones and causal TCN + BatchNorm1d still run as frames arrive, through CAN's continuous step, and each
stream keeps the TCN output rows on the device (its history).  ``push`` returns no logits; ``peek`` runs the fusion
over the history of the listed streams as if they ended now, and ``close`` does so for one stream and frees it
(DESIGN.md section 5.20).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from fractions import Fraction
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import _capi
from .packing import LOGMEL, logmel_tables
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


def continuous_step_table(streams: Sequence[Tuple[int, int, int]]) -> np.ndarray:
    """The cer_stream_entry table of one CAN step: streams = (sid, t_now, parity) per pushed stream -> int32
    [len(streams), 8], one active entry per stream whose single state slot starts at frame 0 and never ends."""
    tab = np.zeros((len(streams), len(_capi.STREAM_ENTRY_FIELDS)), dtype=np.int32)
    for i, (sid, t_now, parity) in enumerate(streams):
        tab[i, 0], tab[i, 4], tab[i, 5], tab[i, 6] = sid, t_now, parity, 1
    return tab


def history_overflow(lengths: Sequence[int], chunk: int, max_frames: int) -> List[int]:
    """Positions in ``lengths`` of the streams that a push of ``chunk`` frames would take past ``max_frames``."""
    return [i for i, t in enumerate(lengths) if int(t) + chunk > max_frames]


def history_row_index(sids: Sequence[int], lengths: Sequence[int], max_frames: int) -> torch.Tensor:
    """Rows of the [streams * max_frames] history view holding the first lengths[i] frames of stream sids[i], laid
    end to end in list order (stream sid, frame t -> sid * max_frames + t): int64 [sum(lengths)]."""
    idx = [int(s) * max_frames + torch.arange(int(t)) for s, t in zip(sids, lengths)]
    return torch.cat(idx) if idx else torch.empty(0, dtype=torch.int64)


def history_bytes(channels: Sequence[int], max_frames: int) -> int:
    """Device bytes of one JMT / MT stream's history: max_frames fp32 rows of each modality's last TCN channel count."""
    return 4 * max_frames * sum(int(c) for c in channels)


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
# Audio bookkeeping of a session opened with wave_fps (pure host logic; DESIGN.md section 5.17)
# ----------------------------------------------------------------------------------------------
def example_grid(fps: float) -> Tuple[int, float]:
    """(log-mel rows per VGGish example, rows between example starts) at ``fps``: the expressions of
    LogMelEngine.examples(wave, 0.96, 1 / fps), so that every start below is the offline one."""
    rate = 1.0 / (LOGMEL["hop"] / LOGMEL["sample_rate"])
    return int(round(0.96 * rate)), (1.0 / fps) * rate


def example_start(t: int, fps: float) -> int:
    """First log-mel row of frame t's example (Python round, as my_frame)."""
    return round(example_grid(fps)[1] * t)


def logmel_rows(n_samples: int) -> int:
    """Complete STFT rows of ``n_samples`` samples (cer_logmel_num_frames)."""
    win, hop = LOGMEL["win"], LOGMEL["hop"]
    return 0 if n_samples < win else 1 + (n_samples - win) // hop


def example_samples(t: int, fps: float) -> int:
    """Samples after which frame t's example is complete: its last row, s_t + 95, needs hop * (s_t + 95) + win."""
    rows = example_grid(fps)[0]
    return LOGMEL["hop"] * (example_start(t, fps) + rows - 1) + LOGMEL["win"]


def frames_ready(n_samples: int, fps: float) -> int:
    """Number of leading frames whose example is complete after ``n_samples`` samples."""
    rows, step = example_grid(fps)
    if n_samples < example_samples(0, fps):
        return 0
    t = int((logmel_rows(n_samples) - rows) / step) + 1            # estimate, then settle on the exact count
    while t > 0 and example_samples(t - 1, fps) > n_samples:
        t -= 1
    while example_samples(t, fps) <= n_samples:
        t += 1
    return t


def stream_lag(fps: float) -> int:
    """The fixed lag L of a wave stream: with audio in step with the video (floor(T * sr / fps) samples after T
    frames), frame T - L's example is complete.  Its last sample is hop * (s + rows - 1) + win with
    s <= hop_rows * (T - L) + 1/2, so L = ceil((hop * (rows - 1) + win + hop / 2 + 1) * fps / sr) suffices
    (the + 1 covers the floor)."""
    rows = example_grid(fps)[0]
    need = LOGMEL["hop"] * (rows - 1) + LOGMEL["win"] + Fraction(LOGMEL["hop"], 2) + 1
    return math.ceil(need * Fraction(fps) / LOGMEL["sample_rate"])


def synced_samples(frames: int, fps: float) -> int:
    """Samples of audio in step with ``frames`` video frames."""
    return math.floor(frames * LOGMEL["sample_rate"] / fps)


def released_upto(frames: int, n_samples: int, emitted: int, lag: int, fps: float) -> int:
    """Frames released once a stream has ``frames`` frames and ``n_samples`` samples and had released ``emitted``:
    frames [emitted, result) go through the head now."""
    return max(emitted, min(frames - lag, frames_ready(n_samples, fps)))


def n_examples_total(lm_rows: int, fps: float) -> int:
    """Examples of a log-mel of ``lm_rows`` rows (LogMelEngine.examples' count); frames at or above it reuse the last."""
    rows, step = example_grid(fps)
    return 1 + int(math.floor((lm_rows - rows) / step)) if lm_rows >= rows else 0


def flush_schedule(emitted: int, frames: int, max_chunk: int) -> List[Tuple[int, int]]:
    """(first frame, count) of the head steps that release frames [emitted, frames), at most max_chunk each."""
    return [(a, min(max_chunk, frames - a)) for a in range(emitted, frames, max_chunk)]


def hold_rows(lag: int, max_chunk: int) -> int:
    """Ring rows of held-back non-audio features: up to lag + 2 * max_chunk unreleased frames after a push, plus
    the chunk being pushed, which is stored before the frames it releases are gathered."""
    return lag + 3 * max_chunk


def logmel_ring_rows(lag: int, max_chunk: int, fps: float) -> int:
    """Log-mel ring rows per stream.  During a push the rows in use run from the example start of the oldest
    unreleased frame (>= T - lag - 3 * max_chunk) to the rows of audio at most lag + max_chunk frames ahead of T:
    fewer than (2 lag + 4 max_chunk) hop_rows rows.  close adds one second (100 rows) of padding and may reuse the
    example before the oldest unreleased frame (one more frame)."""
    step = example_grid(fps)[1]
    return math.ceil((2 * lag + 4 * max_chunk + 1) * step) + LOGMEL["sample_rate"] // LOGMEL["hop"] + 1


# ----------------------------------------------------------------------------------------------
# Session
# ----------------------------------------------------------------------------------------------
class StreamSession:
    """Up to ``max_streams`` live streams of one eval-mode LFAN or CAN, pushed ``<= max_chunk`` frames at a time.

    Per push input (n streams, c frames each): 'video' as stored uint8 crops [n, c, H, W, 3] or fp32
    [n, c, 3, 40, 40]; 'logmel' as VGGish examples [n, c, 96, 64]; a pre-extracted modality as [n, c, D_m].
    One push is one backbone pass over the n * c frames and one fixed sequence of head launches (captured as a
    CUDA graph per (n, c), like LFAN.forward_features; eager when capture is off or fails).

    With ``wave_fps`` set (a model with 'logmel' and at least one other modality), a push carries 'wave' instead
    of 'logmel': a sequence of n 1-D fp32 tensors on the session's device, each stream's next 16 kHz samples (any
    number, 0 included).  The session computes the log-mel rows as their samples arrive (cer_stream_logmel) and
    holds each frame back until its 0.96 s example is complete and it is ``lag`` frames old; ``push`` then returns
    one [r_i, n_out] tensor per stream for the frames it released, and ``close`` flushes the rest with the
    offline edge padding, so the examples are windowing.wave_to_examples' (DESIGN.md section 5.17).

    With a CAN the logits ``push`` returns are final; ``window_length`` / ``hop_length`` do not apply and must stay
    at their defaults (see the module docstring).

    A JMT / MT needs ``max_frames``, the most frames any stream of the session will carry: each stream keeps the
    [max_frames, C_m] TCN + BatchNorm1d output rows of every modality on the device (``state_bytes()`` counts them).
    Inputs are the model's modalities: 'video' as above and 'vggish' rows [n, c, 128] ('logmel' / ``wave_fps`` do
    not apply).  No frame is final before the stream ends, so ``push`` returns (logits [n, 0, n_out], [0] * n);
    ``peek(ids)`` returns per stream the whole-video logits [T_i, n_out] of the frames pushed so far, as if the
    stream ended now, from one fusion pass over all listed streams (JMT._fuse_videos, every attention inside its
    stream); ``close(sid)`` returns the same for one stream and frees it.  With equal backbone embeddings (always for
    'vggish' rows; for 'video' when the IR-50 plan picks the same kernels at both pass sizes, e.g. CER_RASTER=0),
    ``close`` and a one-stream ``peek`` equal ``windowing.infer_video`` on the same frames bit for bit: the
    continuous TCN rows are the offline rows, and the fusion on one stream of T rows is the launch sequence
    infer_videos runs for one video.  A peek of several streams agrees with per-stream peeks to fp32 reordering (the
    fusion's row GEMMs pick split-K from the total row count).  A push that would take a stream past ``max_frames``
    is refused before any state changes (DESIGN.md section 5.20)."""

    def __init__(self, model, max_streams: int = 256, max_chunk: int = 30, window_length: int = 300,
                 hop_length: int = 200, wave_fps: float = None, max_frames: int = None):
        from .heads import CAN, JMT
        from .modules import LFAN
        self.whole = isinstance(model, JMT)                # JMT / MT: TCN rows kept, fusion over them at peek / close
        if not (isinstance(model, (LFAN, CAN)) or (self.whole and max_frames is not None)):
            raise TypeError("StreamSession streams LFAN and CAN as they arrive, and JMT / MT only with max_frames (JMT / MT "
                            "attend over the whole window, so a frame's logits depend on later frames): open a JMT / MT "
                            "session as StreamSession(model, max_streams, max_chunk, max_frames=F), F the longest "
                            "stream, and read whole-stream logits with peek / close")
        if max_frames is not None and not self.whole:
            raise ValueError("max_frames applies to JMT / MT sessions only (an LFAN / CAN stream keeps no history)")
        if self.whole and int(max_frames) < 1:
            raise ValueError(f"max_frames must be positive, got {max_frames}")
        self.continuous = isinstance(model, (CAN, JMT))   # no windows: one never-ending TCN slot per stream
        if self.continuous and (window_length, hop_length) != (300, 200):
            name = getattr(model, "model_name", type(model).__name__)
            raise ValueError(f"a {name} stream has no windows: window_length / hop_length do not apply, got "
                             f"{window_length}, {hop_length}")
        if not (1 <= hop_length <= window_length):
            raise ValueError(f"need 1 <= hop_length <= window_length, got {hop_length}, {window_length}")
        if max_streams < 1 or max_chunk < 1:
            raise ValueError("max_streams and max_chunk must be positive")
        self.max_frames = int(max_frames) if self.whole else None
        _capi.require_gpu()
        self.model = model
        self._check_model()
        self.max_streams, self.max_chunk = int(max_streams), int(max_chunk)
        if self.continuous:
            self.W = self.H = None
            self.n_slots, self.n_lslots = 1, 0
            self._model_engines, mods, self.device = model._engines, model.modalities, model.fc2.weight.device
        else:
            self.W, self.H = int(window_length), int(hop_length)
            self.n_slots = n_window_slots(self.W, self.H, self.max_chunk)
            self.n_lslots = n_logit_slots(self.W, self.H, self.max_chunk)
            self._model_engines, mods, self.device = model._head_engines, model.modality, model.regressor.weight.device
        self.modalities = list(mods)
        self._len: Dict[int, int] = {}
        self._emitted: Dict[int, int] = {}
        self._parity: Dict[int, int] = {}
        self._free = list(range(self.max_streams - 1, -1, -1))
        self._eng = None
        self._pack()
        self.wave_fps = None if wave_fps is None else float(wave_fps)
        self.example_hook = None       # called as hook([(sid, first frame, count)], examples) before each VGGish pass
        if self.wave_fps is not None:
            self._init_wave()

    def _init_wave(self):
        if "logmel" not in self.modalities or len(self.modalities) < 2:
            raise ValueError("wave_fps needs a model with the 'logmel' modality and at least one other (which gives "
                             f"the frame count of a push), got {self.modalities}")
        if not self.wave_fps > 0:
            raise ValueError(f"wave_fps must be positive, got {self.wave_fps}")
        fps, S, dev = self.wave_fps, self.max_streams, self.device
        self.lag = stream_lag(fps)
        self.max_unreleased = self.lag + 2 * self.max_chunk
        self.max_ahead = self.lag + self.max_chunk
        self.example_rows = example_grid(fps)[0]
        self.n_lm_rows = logmel_ring_rows(self.lag, self.max_chunk, fps)
        self.n_hold = hold_rows(self.lag, self.max_chunk)
        self.tail_len = LOGMEL["win"] - 1
        self._samples: Dict[int, int] = {}
        self._lm_tables = logmel_tables(LOGMEL).to(dev)
        self._tails = torch.zeros(S, self.tail_len, dtype=torch.float32, device=dev)
        self._lmring = torch.zeros(S, self.n_lm_rows, LOGMEL["n_mel"], dtype=torch.float32, device=dev)
        self._atab = torch.zeros(S * np.dtype(list(_capi.STREAM_AUDIO_ENTRY_FIELDS)).itemsize, dtype=torch.uint8,
                                 device=dev)
        self._hold = {m: torch.zeros(S, self.n_hold, self._dims[m], dtype=torch.float32, device=dev)
                      for m in self.modalities if m != "logmel"}

    # -- state ------------------------------------------------------------------------------
    def _check_model(self):
        if self.model.training:
            raise RuntimeError("StreamSession runs the inference kernels: call model.eval() first")

    def _pack(self):
        """(Re)bind the model's packed head (LFAN: its FusionEngine; CAN: CAN.frame_head; JMT / MT: none, the fusion
        runs at peek / close); allocate the rings, histories and step buffers on first use."""
        self._eng, self._graphs = self._model_engines(), {}
        tcn = self._eng[0]
        self._head = None if self.whole else self.model.frame_head() if self.continuous else self._eng[1]
        self._tanh = self.continuous and self.model.task == "REGRESSION"
        dev, S, ne, cm = self.device, self.max_streams, self.max_streams * self.n_slots, self.max_chunk
        f32 = dict(dtype=torch.float32, device=dev)
        self.n_out = self.model.fc2.out_features if self.whole else self._head.n_out
        fresh = not hasattr(self, "_tab")
        if fresh:
            self._tab = torch.zeros(ne, len(_capi.STREAM_ENTRY_FIELDS), dtype=torch.int32, device=dev)
            if not self.continuous:
                self._lring = torch.zeros(S, self.n_lslots, self.W, self.n_out, **f32)
            self._out = torch.empty(0 if self.whole else S * cm * self.n_out, **f32)
            self._in, self._inring, self._rings, self._staged, self._outs, self._ws, self._gath = {}, {}, {}, {}, {}, {}, {}
            self._hist = {}
        self._blocks, self._rows, self._dims = {}, {}, {}
        for m in self.modalities:
            eng = tcn[m]
            self._dims[m] = eng.c_in
            if eng.precision != "tf32":      # LFAN packs its TCNs for the tensor-core kernel; the staging assumes its padding
                raise NotImplementedError(f"'{m}': StreamSession runs the tensor-core TCN kernel only")
            blocks = eng.blocks
            rows = [2 * (b.kernel_size - 1) * b.dilation for b in blocks]
            self._blocks[m], self._rows[m] = blocks, rows
            if not fresh:
                continue
            self._in[m] = torch.empty(S * cm * eng.c_in, **f32)
            if not self.continuous:
                self._inring[m] = torch.zeros(S, self.W, eng.c_in, **f32)
            self._rings[m] = [torch.zeros(S * self.n_slots * 2 * max(r, 1) * b.c_in, **f32) for b, r in zip(blocks, rows)]
            self._staged[m] = [torch.empty(ne * (r + cm) * b.c_in, **f32) for b, r in zip(blocks, rows)]
            self._outs[m] = [torch.empty(ne * (r + cm) * b.c_out, **f32) for b, r in zip(blocks, rows)]
            self._ws[m] = torch.empty(max(ne * (r + cm) * b.c_out for b, r in zip(blocks, rows)) * 4, dtype=torch.uint8,
                                      device=dev)
            self._gath[m] = torch.empty(ne * cm * eng.c_out, **f32)
            if self.whole:
                self._hist[m] = torch.zeros(S, self.max_frames, blocks[-1].c_out, **f32)

    def _engines(self):
        eng = self._model_engines()
        if eng is not self._eng:                    # weights changed: the captured graphs hold the old packing
            self._pack()
        return self._eng

    def _final_upto(self, emitted: int) -> int:
        if self.whole:
            return 0
        return emitted if self.continuous else final_upto(emitted, self.W)

    def state_bytes(self) -> int:
        """Device memory one stream slot holds across steps (rings), in bytes."""
        n = 0 if self.continuous else self.n_lslots * self.W * self.n_out
        for m in self.modalities:
            if not self.continuous:
                n += self.W * self._dims[m]
            n += sum(self.n_slots * 2 * r * b.c_in for b, r in zip(self._blocks[m], self._rows[m]))
        if self.wave_fps is not None:
            n += self.tail_len + self.n_lm_rows * LOGMEL["n_mel"] + sum(h.shape[1] * h.shape[2] for h in self._hold.values())
        if self.whole:
            return 4 * n + history_bytes([self._blocks[m][-1].c_out for m in self.modalities], self.max_frames)
        return 4 * n

    def open(self) -> int:
        """A new stream at its frame 0; returns its id."""
        if not self._free:
            raise RuntimeError(f"all {self.max_streams} stream slots are open")
        sid = self._free.pop()
        self._len[sid], self._emitted[sid], self._parity[sid] = 0, 0, 0
        if self.wave_fps is not None:
            self._samples[sid] = 0
        return sid

    def length(self, sid: int) -> int:
        """Frames pushed to stream ``sid``."""
        return self._len[sid]

    def emitted(self, sid: int) -> int:
        """Frames of stream ``sid`` whose logits were returned (== length without wave_fps)."""
        return self._emitted[sid]

    # -- push -------------------------------------------------------------------------------
    def _chunk_features(self, inputs: Dict[str, torch.Tensor], n: int, mods=None) -> Tuple[int, Dict[str, torch.Tensor]]:
        if "wave" in inputs:
            raise ValueError("'wave' cannot be streamed: the VGGish example of a frame needs 0.96 s of audio after it; "
                             "push 'logmel' examples [n, c, 96, 64] instead, or open the session with wave_fps")
        chunk, out = None, {}
        for m in mods or self.modalities:
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
        tcn = self._eng[0]
        ne, tab = n * self.n_slots, self._tab.data_ptr()
        feats = []
        for m in self.modalities:
            eng = tcn[m]
            d_in = eng.c_in
            if not self.continuous:
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
        if self.whole:                              # JMT / MT: the rows join each stream's history (peek / close fuse it)
            for m, f in zip(self.modalities, feats):
                chk(lib.cer_stream_append(tab, ne, c, f.data_ptr(), f.shape[1], self.max_streams, self.max_frames,
                                          self._hist[m].data_ptr(), st), "cer_stream_append")
            return
        if self.continuous:                         # per-frame and final: straight into the output buffer
            self._head.forward(feats, self._tanh, out=self._out[:n * c * self.n_out].view(n * c, self.n_out))
            return
        logits = self._head.forward(feats)
        chk(lib.cer_stream_average(tab, n, self.n_slots, c, self.W, self.n_out, logits.data_ptr(), self._out.data_ptr(),
                                   self._lring.data_ptr(), self.n_lslots, st), "cer_stream_average")

    def _use_graph(self) -> bool:
        return (getattr(self.model, "head_cuda_graph", True) and os.environ.get("CER_HEAD_GRAPH", "1") != "0"
                and not torch.cuda.is_current_stream_capturing())

    @torch.no_grad()
    def push(self, ids: Sequence[int], inputs: Dict[str, torch.Tensor]) -> Tuple[torch.Tensor, List[int]]:
        """Advance streams ``ids`` by c frames -> (provisional logits [n, c, n_out], final_upto per stream).

        With wave_fps: -> (a list of n tensors [r_i, n_out], the provisional logits of the frames this push
        released, continuing from emitted(i); final_upto = max(0, emitted(i) - W) per stream).

        With a CAN every returned logit is final: final_upto = emitted(i).

        With a JMT / MT no logit is final before close: -> (logits [n, 0, n_out], [0] * n); the frames' TCN rows join
        the streams' histories (read them through peek / close)."""
        self._check_model()
        ids = [int(i) for i in ids]
        n = len(ids)
        if n == 0:
            raise ValueError("push needs at least one stream")
        if len(set(ids)) != n or any(i not in self._len for i in ids):
            raise ValueError(f"stream ids must be distinct open streams, got {ids}")
        if self.whole:                              # every stream's bound, before any state changes
            x0 = inputs.get(self.modalities[0])
            c = int(x0.shape[1]) if isinstance(x0, torch.Tensor) and x0.dim() >= 2 else 0
            over = [ids[j] for j in history_overflow([self._len[i] for i in ids], c, self.max_frames)]
            if over:
                raise ValueError(f"streams {over}: a push of {c} frames would take them past max_frames = "
                                 f"{self.max_frames} (lengths {[self._len[i] for i in over]})")
        self._engines()
        if self.wave_fps is not None:
            return self._push_wave(ids, inputs)
        with torch.cuda.device(self.device):
            c, x = self._chunk_features(inputs, n)
            for m in self.modalities:
                d = self._dims[m]
                if x[m].shape[1] != d:
                    raise ValueError(f"'{m}': expected {d} features per frame, got {x[m].shape[1]}")
            out = self._head_step(ids, c, x)
        for i in ids:
            self._len[i] += c
        return out, [self._final_upto(self._len[i]) for i in ids]

    def _head_step(self, ids: List[int], c: int, x: Dict[str, torch.Tensor]) -> torch.Tensor:
        """Frames emitted(i) .. emitted(i) + c - 1 of streams ``ids`` (features x[m] [n * c, D_m]) through the head
        -> their provisional logits [n, c, n_out]; advances emitted and the TCN ring parity of those streams."""
        n = len(ids)
        for m in self.modalities:
            d = self._dims[m]
            self._in[m][:n * c * d].view(n * c, d).copy_(x[m])
        streams = [(i, self._emitted[i], self._parity[i]) for i in ids]
        tab = (continuous_step_table(streams) if self.continuous else
               step_table(streams, c, self.W, self.H, self.n_slots, self.n_lslots))
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
        out = (self._out.new_empty(n, 0, self.n_out) if self.whole else
               self._out[:n * c * self.n_out].view(n, c, self.n_out).clone())
        for i in ids:
            self._emitted[i] += c
            self._parity[i] ^= 1
        return out

    # -- wave streams -------------------------------------------------------------------------
    def _front_end(self, work: List[Tuple[int, int, torch.Tensor]]) -> None:
        """Append samples to streams: work = (sid, samples received before, new fp32 samples on the device).
        Computes every newly complete log-mel row into the ring and advances the tails (cer_stream_logmel)."""
        work = [w for w in work if w[2].numel() > 0]
        if not work:
            return
        tab = np.zeros(len(work), dtype=np.dtype(list(_capi.STREAM_AUDIO_ENTRY_FIELDS)))
        off = 0
        for k, (sid, a0, w) in enumerate(work):
            r0, r1 = logmel_rows(a0), logmel_rows(a0 + w.numel())
            tab[k] = (sid, r0, r1 - r0, 0, a0, off, w.numel())
            off += w.numel()
        samples = torch.cat([w for _, _, w in work]) if len(work) > 1 else work[0][2].contiguous()
        raw = torch.from_numpy(tab.view(np.uint8)).pin_memory()
        self._atab[:raw.numel()].copy_(raw, non_blocking=True)
        c = LOGMEL
        _capi.check(_capi.lib().cer_stream_logmel(
            self._atab.data_ptr(), len(work), int(tab["n_rows"].max()), samples.data_ptr(), self._lm_tables.data_ptr(),
            c["win"], c["hop"], c["fft"], c["n_mel"], c["log_offset"], self._tails.data_ptr(), self.tail_len,
            self._lmring.data_ptr(), self.n_lm_rows, _capi.current_stream_ptr(self.device)), "cer_stream_logmel")

    def _release(self, rel: List[Tuple[int, int, int, int]]) -> Dict[int, List[torch.Tensor]]:
        """Release frames through the head: rel = (sid, first frame == emitted(sid), count, examples available or 0
        for all).  One VGGish pass over every released example, then per group of streams with the same count one
        head step per max_chunk frames.  Returns sid -> the provisional logits of its steps, in frame order."""
        rel = [r for r in rel if r[2] > 0]
        outs: Dict[int, List[torch.Tensor]] = {}
        if not rel:
            return outs
        ex_rows, base, off = [], {}, 0
        for sid, e0, r, n_ex in rel:
            base[sid] = off
            for t in range(e0, e0 + r):
                ex_rows.append((sid, example_start(min(t, n_ex - 1) if n_ex else t, self.wave_fps), off))
                off += 1
        ent = torch.tensor(ex_rows, dtype=torch.int32).pin_memory().to(self.device, non_blocking=True)
        ex = torch.empty(off, self.example_rows, LOGMEL["n_mel"], dtype=torch.float32, device=self.device)
        _capi.check(_capi.lib().cer_stream_examples(self._lmring.data_ptr(), self.n_lm_rows, ent.data_ptr(), off,
                                                    self.example_rows, LOGMEL["n_mel"], ex.data_ptr(),
                                                    _capi.current_stream_ptr(self.device)), "cer_stream_examples")
        if self.example_hook is not None:
            self.example_hook([(sid, e0, r) for sid, e0, r, _ in rel], ex)
        emb = self.model.spatial["audio"](ex)
        groups: Dict[int, List[Tuple[int, int]]] = {}
        for sid, e0, r, _ in rel:
            groups.setdefault(r, []).append((sid, e0))
        for r, members in groups.items():
            ids = [sid for sid, _ in members]
            for a, cc in flush_schedule(0, r, self.max_chunk):
                rows = [(sid, e0 + a + k, base[sid] + a + k) for sid, e0 in members for k in range(cc)]
                idx = torch.tensor([[sid * self.n_hold + f % self.n_hold, j] for sid, f, j in rows],
                                   dtype=torch.int64).pin_memory().to(self.device, non_blocking=True)
                x = {m: (emb.index_select(0, idx[:, 1]) if m == "logmel" else
                         self._hold[m].view(-1, self._hold[m].shape[-1]).index_select(0, idx[:, 0]))
                     for m in self.modalities}
                out = self._head_step(ids, cc, x)
                for j, sid in enumerate(ids):
                    outs.setdefault(sid, []).append(out[j])
        return outs

    def _push_wave(self, ids: List[int], inputs) -> Tuple[List[torch.Tensor], List[int]]:
        n, others = len(ids), [m for m in self.modalities if m != "logmel"]
        if "logmel" in inputs:
            raise ValueError("a session opened with wave_fps takes 'wave', not 'logmel': push one or the other")
        if "wave" not in inputs:
            raise KeyError("push needs the 'wave' input: a sequence of one 1-D fp32 tensor of new samples per stream")
        waves = list(inputs["wave"])
        if len(waves) != n:
            raise ValueError(f"'wave': expected {n} tensors (one per stream), got {len(waves)}")
        for w in waves:
            if not isinstance(w, torch.Tensor) or w.dim() != 1 or w.dtype != torch.float32 or w.device != self.device:
                raise ValueError(f"'wave': every stream's samples must be a 1-D fp32 tensor on {self.device}")
        for m in others:
            if m not in inputs:
                raise KeyError(f"push needs the '{m}' input")
        x0 = inputs[others[0]]
        c = int(x0.shape[1]) if x0.dim() >= 2 else 0
        if not 1 <= c <= self.max_chunk:
            raise ValueError(f"chunk of {c} frames: need 1..{self.max_chunk}")
        plan = []
        for sid, w in zip(ids, waves):                    # the bounds, before any state changes
            T1, A1 = self._len[sid] + c, self._samples[sid] + w.numel()
            limit = synced_samples(T1 + self.max_ahead, self.wave_fps)
            if A1 > limit:
                raise ValueError(f"stream {sid}: audio may run ahead of the video by at most {self.max_ahead} frames "
                                 f"(lag + max_chunk): {A1} samples after {T1} frames, at most {limit}")
            E1 = released_upto(T1, A1, self._emitted[sid], self.lag, self.wave_fps)
            if T1 - E1 > self.max_unreleased:
                raise ValueError(f"stream {sid}: at most {self.max_unreleased} frames (lag + 2 * max_chunk) may wait "
                                 f"for their audio, {T1 - E1} would: push more audio")
            plan.append((sid, self._emitted[sid], E1 - self._emitted[sid]))
        with torch.cuda.device(self.device):
            _, x = self._chunk_features({m: inputs[m] for m in others}, n, others)
            for m in others:
                d = self._hold[m].shape[-1]
                if x[m].shape[1] != d:
                    raise ValueError(f"'{m}': expected {d} features per frame, got {x[m].shape[1]}")
            self._front_end([(sid, self._samples[sid], w) for sid, w in zip(ids, waves)])
            for sid, w in zip(ids, waves):
                self._samples[sid] += w.numel()
            idx = torch.tensor([sid * self.n_hold + (self._len[sid] + k) % self.n_hold for sid in ids for k in range(c)],
                               dtype=torch.int64).pin_memory().to(self.device, non_blocking=True)
            for m in others:
                self._hold[m].view(-1, self._hold[m].shape[-1]).index_copy_(0, idx, x[m])
            for sid in ids:
                self._len[sid] += c
            outs = self._release([(sid, e0, r, 0) for sid, e0, r in plan])
            empty = torch.empty(0, self.n_out, dtype=torch.float32, device=self.device)
            res = [torch.cat(outs[sid]) if sid in outs else empty for sid in ids]
        return res, [self._final_upto(self._emitted[i]) for i in ids]

    def _flush_wave(self, sid: int) -> List[torch.Tensor]:
        """close: one second of the last sample (wave_to_examples' edge padding), the remaining log-mel rows, and the
        held-back frames through the head; frames at or above the example count reuse the last example.  Returns the
        logits of those head steps, in frame order."""
        A, T, E = self._samples[sid], self._len[sid], self._emitted[sid]
        pad = self._tails[sid, -1:].expand(LOGMEL["sample_rate"]).contiguous()
        self._front_end([(sid, A, pad)])
        self._samples[sid] = A + pad.numel()
        n_ex = n_examples_total(logmel_rows(A + pad.numel()), self.wave_fps)
        return self._release([(sid, E, T - E, n_ex)]).get(sid, [])

    # -- JMT / MT: whole-stream logits -----------------------------------------------------------
    @torch.no_grad()
    def peek(self, ids: Sequence[int]) -> List[torch.Tensor]:
        """JMT / MT sessions: per listed open stream the whole-video logits [T_i, n_out] of the frames pushed so far,
        as if the stream ended now ([0, n_out] for a stream with no frames).  One fusion pass over all listed streams;
        the streams stay open."""
        if not self.whole:
            raise TypeError("peek reads the whole-stream logits of a JMT / MT session; an LFAN / CAN session returns "
                            "its logits from push and close")
        ids = [int(i) for i in ids]
        if len(set(ids)) != len(ids) or any(i not in self._len for i in ids):
            raise ValueError(f"stream ids must be distinct open streams, got {ids}")
        self._check_model()
        self._engines()
        return self._whole_logits(ids)

    def _whole_logits(self, ids: List[int]) -> List[torch.Tensor]:
        """The history rows of streams ``ids`` laid end to end through JMT._fuse_videos (the function infer_videos
        runs), so every attention stays inside its stream."""
        lengths = [self._len[i] for i in ids]
        live = [(i, t) for i, t in zip(ids, lengths) if t > 0]
        out = iter([])
        if live:
            sids, lens = [i for i, _ in live], [t for _, t in live]
            with torch.cuda.device(self.device):
                idx = history_row_index(sids, lens, self.max_frames).to(self.device, non_blocking=True)
                z = {m: self._hist[m].view(-1, self._hist[m].shape[-1]).index_select(0, idx) for m in self.modalities}
                out = iter(self.model._fuse_videos(z, lens).split(lens))
        return [next(out) if t > 0 else torch.empty(0, self.n_out, dtype=torch.float32, device=self.device)
                for t in lengths]

    # -- close ------------------------------------------------------------------------------
    @torch.no_grad()
    def close(self, sid: int) -> torch.Tensor:
        """End stream ``sid`` -> the final logits [min(T, W), n_out] of its frames T - min(T, W) .. T - 1, and free
        its slot.  With a CAN: the logits of the frames not returned yet ([0, n_out] without wave_fps; the
        held-back frames with it).  With a JMT / MT: the whole-video logits [T, n_out] of every frame, as
        ``peek([sid])`` computes them."""
        from .engine import stitch_windows
        if sid not in self._len:
            raise ValueError(f"stream {sid} is not open")
        self._check_model()
        self._engines()
        if self.whole:
            out = self._whole_logits([sid])[0]
            del self._len[sid], self._parity[sid], self._emitted[sid]
            self._free.append(sid)
            return out
        flushed = []
        if self.wave_fps is not None and self._len[sid] > 0:
            if self._samples[sid] == 0:
                raise ValueError(f"stream {sid} received no audio: its frames have no VGGish example (offline, "
                                 "wave_to_examples fails on an empty waveform the same way)")
            with torch.cuda.device(self.device):
                flushed = self._flush_wave(sid)
        T, W = self._len.pop(sid), self.W
        del self._parity[sid], self._emitted[sid]
        if self.wave_fps is not None:
            del self._samples[sid]
        self._free.append(sid)
        if self.continuous and flushed:
            return torch.cat(flushed)
        if T == 0 or self.continuous:
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
