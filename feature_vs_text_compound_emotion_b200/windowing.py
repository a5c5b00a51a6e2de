"""Long-video inference: windows of 300 frames every 200, overlap averaging -- on the device.

Restates the semantics of Trainer.windowing / window_input / inference_forward_windows
(trainer.py:788-913) around the CUDA path, with two exact savings the reference leaves on the
table (SURVEY.md section 8 f1):
  * IR-50 is per-frame in eval mode, so every *unique* frame is encoded once and the 512-d
    embeddings are windowed, instead of re-encoding the 100-frame overlaps (33-50 % less conv work);
  * all windows of a video go through the head as one batch (the reference loops with bsz 1).

The alternative heads CAN / JMT / MT have no windows: the reference runs them over the whole video with batch size
1 (trainer.py:480-485).  ``infer_video`` / ``infer_videos`` give them those semantics (see :func:`infer_videos`).
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import torch


def window_starts(length: int, window_length: int = 300, hop_length: int = 200) -> List[int]:
    """First frame of every window: a regular grid while a full window fits, plus one tail window
    flush with the end when the grid does not reach the last frame (trainer.py:894-913)."""
    if length < window_length:
        return [0]
    starts = list(range(0, length - window_length + 1, hop_length))
    if starts[-1] + window_length < length:
        starts.append(length - window_length)
    return starts


def gather_windows(feat: torch.Tensor, starts: Sequence[int], window_length: int) -> torch.Tensor:
    """feat [T, D] -> [n_windows, window_length, D].  A video shorter than the window is padded by
    repeating its last frame (the reference's training-time rule, base/dataset.py:570-582)."""
    T = feat.shape[0]
    if T < window_length:
        pad = feat[-1:].expand(window_length - T, *feat.shape[1:])
        feat = torch.cat([feat, pad], dim=0)
    idx = torch.as_tensor(starts, device=feat.device).view(-1, 1) + torch.arange(window_length, device=feat.device)
    return feat[idx]


def preprocess_frames(model, frames_u8: torch.Tensor, resize: int = 48, crop: int = 40) -> torch.Tensor:
    """uint8 [T,H,W,3] on the GPU -> fp32 [T,3,crop,crop]; the plan is cached on the model per input size."""
    from .engine import PreprocEngine
    cache = model.__dict__.setdefault("_preproc", {})
    key = (int(frames_u8.shape[1]), int(frames_u8.shape[2]), resize, crop, str(frames_u8.device))
    if key not in cache:
        cache[key] = PreprocEngine(key[0], key[1], frames_u8.device, resize, crop)
    return cache[key].forward(frames_u8)


def wave_to_examples(model, wave: torch.Tensor, n_frames: int, fps: float = 30.0) -> torch.Tensor:
    """Mono 16 kHz waveform on the GPU -> [n_frames, 96, 64] VGGish examples, one per video frame
    (0.96 s window, hop 1/fps; vggish_input.py:37-95 incl. the one second of edge padding :93; the
    last example is repeated if the audio track is shorter than the video)."""
    from .engine import LogMelEngine
    eng = model.__dict__.get("_logmel")
    if eng is None or eng.device != wave.device:
        eng = model.__dict__["_logmel"] = LogMelEngine(wave.device)
    sr = eng.cfg["sample_rate"]
    wave = torch.cat([wave.float(), wave[-1:].float().expand(sr)])
    ex = eng.examples(wave, 0.96, 1.0 / fps)
    if ex.shape[0] < n_frames:
        ex = torch.cat([ex, ex[-1:].expand(n_frames - ex.shape[0], -1, -1)])
    return ex[:n_frames].contiguous()


VOTE_KEYS = ("FRAMES_VOTE", "FRAMES_AVG_LOGITS", "FRAMES_AVG_PROBS")      # constants.py:136-142


def video_level_prediction(frame_logits: torch.Tensor, ignore_last_class: bool = False) -> Dict[str, int]:
    """The three video-level decision rules of metrics.py:88-145 (format_trg_pred_video) on the
    stitched per-frame logits [T, n_cls] of one video, on the device (cer_video_vote): FRAMES_VOTE
    (majority of per-frame argmax; ties go to the class that appears first, as Counter.most_common
    does), FRAMES_AVG_LOGITS, FRAMES_AVG_PROBS.  ``ignore_last_class`` drops the 'Other' class first
    (C-EXPR-DB, metrics.py:118-119)."""
    from . import _capi
    _capi.require_gpu()
    lg = frame_logits.float().contiguous()
    if lg.device.type != "cuda":
        raise _capi.CerError("video_level_prediction needs the logits on the CUDA device (no CPU fallback)")
    out = torch.empty(3, dtype=torch.int32, device=lg.device)
    with torch.cuda.device(lg.device):
        _capi.check(_capi.lib().cer_video_vote(lg.data_ptr(), lg.shape[0], lg.shape[1], int(ignore_last_class), out.data_ptr(),
                                               _capi.current_stream_ptr()), "cer_video_vote")
    return dict(zip(VOTE_KEYS, (int(v) for v in out.tolist())))


@torch.no_grad()
def infer_video(model, video: torch.Tensor, feats: Dict[str, torch.Tensor], window_length: int = 300,
                hop_length: int = 200, fps: float = 30.0) -> torch.Tensor:
    """One whole video through the LFAN mirror (or a CAN / JMT / MT: :func:`infer_videos` on this one video).

    video: [T,3,40,40] fp32 on the GPU (post eval-transform) or the stored uint8 [T,H,W,3] crops
    (then base/dataset.py:503-510 runs on the device, engine.PreprocEngine); feats[m]: [T, D_m] for
    the non-visual modalities ('logmel': [T,96,64] examples, encoded by the VGGish kernels; or
    'wave': the mono 16 kHz waveform, turned into one example per frame at ``fps`` on the device).  Returns per-frame logits [T, n_out] = the reference's stitched output.
    """
    from .engine import stitch_windows
    if _is_feature_head(model):
        return infer_videos(model, [video], [feats], window_length, hop_length, fps)[0]
    T = video.shape[0]
    if video.dtype == torch.uint8:                             # stored crops: the eval transform runs on the device
        video = preprocess_frames(model, video)
    emb = model.spatial["visual"](video)                       # every unique frame once
    starts = window_starts(T, window_length, hop_length)
    batch = {}
    for m in model.modality:
        if m == "video":
            src = emb
        elif m == "logmel":
            ex = feats[m] if m in feats else wave_to_examples(model, feats["wave"], T, fps)
            src = model.spatial["audio"](ex)                    # one example per frame (audio.py:126-127)
        else:
            src = feats[m]
        batch[m] = gather_windows(src, starts, window_length).contiguous()
    logits = model.forward_features(batch)                     # [n_windows, window_length, n_out]
    start_t = torch.as_tensor(starts, dtype=torch.int32, device=video.device)
    out = stitch_windows(logits, start_t, max(T, window_length))
    return out[:T]


def window_index_table(lengths: Sequence[int], window_length: int = 300, hop_length: int = 200):
    """Window grid of several videos laid end to end: (starts per video, int64 [n_windows_total, window_length]
    of row numbers into the concatenated frame axis).  A video shorter than the window repeats its last
    frame, as :func:`gather_windows` does."""
    starts = [window_starts(int(t), window_length, hop_length) for t in lengths]
    ar = torch.arange(window_length)
    rows, off = [], 0
    for t, st in zip(lengths, starts):
        rows.append(off + torch.clamp(torch.as_tensor(st).view(-1, 1) + ar, max=int(t) - 1))
        off += int(t)
    return starts, torch.cat(rows)


def padded_row_index(lengths: Sequence[int]):
    """Videos laid end to end -> (T_max, int64 [sum(lengths)]): the row of each frame in a right-padded
    [n_videos, T_max] batch (video i, frame t -> i * T_max + t), in concatenated order.  Scattering the concatenated
    rows through it fills the padded batch; gathering through it takes the valid rows back."""
    t_max = max((int(t) for t in lengths), default=0)
    idx = [i * t_max + torch.arange(int(t)) for i, t in enumerate(lengths)]
    return t_max, (torch.cat(idx) if idx else torch.empty(0, dtype=torch.int64))


def _is_feature_head(model) -> bool:
    from .heads import _FeatureHead
    return isinstance(model, _FeatureHead)


def _check_whole_videos(model, videos, feats, window_length: int, hop_length: int) -> List[int]:
    """The inputs of CAN / JMT / MT whole-video inference, checked before any device work -> the video lengths."""
    if (window_length, hop_length) != (300, 200):
        raise ValueError(f"{type(model).__name__} runs over the whole video, it has no windows: window_length / "
                         f"hop_length do not apply, got {window_length}, {hop_length}")
    lengths = []
    for i, (v, f) in enumerate(zip(videos, feats)):
        T = int(v.shape[0])
        if T == 0:
            raise ValueError(f"video {i} is empty")
        for m in model.modalities:
            if m == "video":
                continue
            key = "wave" if m == "logmel" and m not in f and "wave" in f else m
            if key not in f:
                raise ValueError(f"video {i}: the head needs modality '{m}'" + (" (or 'wave')" if m == "logmel" else ""))
            if key != "wave" and int(f[key].shape[0]) != T:
                raise ValueError(f"video {i}: '{key}' has {int(f[key].shape[0])} rows for {T} frames")
        lengths.append(T)
    return lengths


def _backbone_rows(model, videos, feats, lengths, modalities, fps: float) -> Dict[str, torch.Tensor]:
    """The frames of all videos through the eval transform and IR-50 / VGGish back to back in full passes ->
    src[m] [sum(lengths), D_m] in concatenated order (the non-visual feature rows concatenated as given)."""
    src = {}
    for m in modalities:
        if m == "video":
            frames = torch.cat([preprocess_frames(model, v) if v.dtype == torch.uint8 else v for v in videos])
            src[m] = model.spatial["visual"](frames)                # every unique frame of every video once
        elif m == "logmel":
            ex = torch.cat([f[m] if m in f else wave_to_examples(model, f["wave"], t, fps) for f, t in zip(feats, lengths)])
            src[m] = model.spatial["audio"](ex)
        else:
            src[m] = torch.cat([f[m] for f in feats])
    return src


@torch.no_grad()
def infer_videos(model, videos: Sequence[torch.Tensor], feats: Sequence[Dict[str, torch.Tensor]], window_length: int = 300,
                 hop_length: int = 200, fps: float = 30.0, windows_per_pass: int = 16) -> List[torch.Tensor]:
    """Several whole videos at once: the same result per video as :func:`infer_video` (the backbones are
    per-frame and the head is per-window in eval mode; values can differ by bf16 rounding only where the
    IR-50 plan picks another kernel for the larger pass -- the padded-raster stage needs >= 190 frames), but
    the frames of all videos go through IR-50 / VGGish back to back in full passes, the windows of all
    videos go through the head in groups of ``windows_per_pass`` (one CUDA graph, the last group padded by
    repeating its last window) and only the stitch is per video.  Short videos stop paying for
    partly-filled launches.  Returns one [T_i, n_out] tensor per video.

    A CAN / JMT / MT runs over each whole video as the reference does (batch 1, no windows; ``window_length`` /
    ``hop_length`` must stay at their defaults and ``windows_per_pass`` does not apply).  The backbone passes are
    shared as above, the TCN runs on one right-padded batch, and the fusion head on the frames of all videos laid end
    to end: CAN frame by frame, JMT / MT with every attention kept inside its video (engine.sdpa_segments).  A CAN's
    result per video does not depend on the other videos in the call; a JMT / MT's agrees to fp32 reordering (its
    row GEMMs pick split-K from the row count).  Every modality the head was built with is needed per video, with T
    rows ('logmel' may come as 'wave'); an empty video is refused."""
    from .engine import stitch_windows
    if len(videos) != len(feats):
        raise ValueError("one feature dict per video")
    whole = _is_feature_head(model)
    if whole:
        lengths = _check_whole_videos(model, videos, feats, window_length, hop_length)
    if not videos:
        return []
    dev = videos[0].device
    if whole:
        src = _backbone_rows(model, videos, feats, lengths, model.modalities, fps)
        return list(model.forward_videos(src, lengths).split(lengths))
    lengths = [int(v.shape[0]) for v in videos]
    src = _backbone_rows(model, videos, feats, lengths, model.modality, fps)
    starts, idx = window_index_table(lengths, window_length, hop_length)
    idx = idx.to(dev, non_blocking=True)                            # [n_windows_total, window_length]
    n_win = idx.shape[0]
    group = max(1, min(int(windows_per_pass), n_win))
    logits = None
    for a in range(0, n_win, group):
        sel = idx[a:a + group]
        if sel.shape[0] < group:
            sel = torch.cat([sel, sel[-1:].expand(group - sel.shape[0], -1)])
        out = model.forward_features({m: src[m][sel] for m in model.modality})
        if logits is None:
            logits = torch.empty(n_win, window_length, out.shape[-1], device=dev)
        logits[a:a + group] = out[:min(group, n_win - a)]
    start_all = torch.as_tensor([s0 for st in starts for s0 in st], dtype=torch.int32).to(dev, non_blocking=True)
    outs, w0 = [], 0
    for i, st in enumerate(starts):
        o = stitch_windows(logits[w0:w0 + len(st)], start_all[w0:w0 + len(st)], max(lengths[i], window_length))
        outs.append(o[:lengths[i]])
        w0 += len(st)
    return outs
