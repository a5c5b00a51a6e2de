"""Five-point face alignment on the device: full camera frames + a detector's landmarks -> the aligned uint8 face
crops that ``windowing.infer_video`` and ``StreamSession.push`` take as ``video``.

The reference's offline pipeline (abaw5_pre_processing/dlib, SURVEY §2.1 row 19) aligns each detected face with
face.evoLVe's ``warp_and_crop_face``: a five-point similarity fit (``get_similarity_transform_for_cv2`` with
``reflective=True``) and ``cv2.warpAffine`` with its defaults.  ``align`` does both on the B200 (csrc/align.cu): the fit
in fp64, the warp in OpenCV's fixed-point arithmetic, so a crop is bit for bit what ``cv2.warpAffine`` makes from the
same matrix.

    ref = faces.reference_points(crop_size=256)                       # [5, 2] fp64
    crops = faces.align(frames_u8, landmarks)                          # uint8 [N, 256, 256, 3] on the device
    logits = windowing.infer_video(model, crops, feats)

Landmarks are fp32 ``(x, y)`` pixel coordinates in the order left eye, right eye, nose, left mouth corner, right mouth
corner (MTCNN / RetinaFace / face.evoLVe).  Detection, and choosing which face of a frame to keep, stay with the
caller.  Channels are carried as given; the stored crops are RGB.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np
import torch

from . import _capi

# face.evoLVe align_trans.REFERENCE_FACIAL_POINTS: the five points in a 96 x 112 (width x height) crop
TEMPLATE_96x112 = np.array([[30.29459953, 51.69630051],
                            [65.53179932, 51.50139999],
                            [48.02519989, 71.73660278],
                            [33.54930115, 92.3655014],
                            [62.72990036, 92.20410156]])
MAX_CROP = 1024
MAX_SIDE = 32767         # OpenCV keeps the integer source pixel in int16


def reference_points(crop_size: int = 256, inner_padding_factor: float = 0.0, outer_padding=(0, 0),
                     default_square: bool = True) -> np.ndarray:
    """fp64 [5, 2]: where the five points land in a ``crop_size`` x ``crop_size`` crop.

    face.evoLVe's face_align.py recipe: ``get_reference_facial_points(default_square=True)`` (the 96 x 112 template
    with x shifted by 8 to make it 112 x 112) scaled by ``crop_size / 112``.  With padding, the template is padded by
    ``inner_padding_factor`` and resized into the crop inside ``outer_padding`` as ``get_reference_facial_points`` does
    for ``output_size = (crop_size, crop_size)``.

    Not checked: whether the reference's ``retinaface_align.py`` passes exactly these arguments for its 256 x 256
    crops (its source was not available).  Pass ``reference=`` to ``align`` to use other points."""
    pts = TEMPLATE_96x112.copy()
    size = np.array([96.0, 112.0])
    if default_square:
        pts += (size.max() - size) / 2
        size = np.full(2, size.max())
    pad = np.asarray(outer_padding, dtype=np.float64)
    if inner_padding_factor == 0 and not pad.any():
        return pts * (crop_size / 112.0)
    if not 0 <= inner_padding_factor <= 1.0:
        raise ValueError(f"reference_points: inner_padding_factor must be in [0, 1], got {inner_padding_factor}")
    if not (pad[0] < crop_size and pad[1] < crop_size):
        raise ValueError(f"reference_points: outer_padding {tuple(outer_padding)} does not fit a {crop_size} crop")
    if inner_padding_factor > 0:
        diff = size * inner_padding_factor * 2
        pts += diff / 2
        size = size + np.round(diff)
    inner = crop_size - pad * 2
    if inner[0] * size[1] != inner[1] * size[0]:
        raise ValueError("reference_points: the padded template is not square; use default_square=True or give "
                         "reference points directly")
    return pts * (inner[0] / size[0]) + pad


def _reference(reference) -> np.ndarray:
    ref = np.asarray(reference, dtype=np.float64)
    if ref.shape != (5, 2) or not np.isfinite(ref).all():
        raise ValueError(f"reference must be 5 finite (x, y) points, got shape {ref.shape}")
    if not ((ref - ref.mean(0)) ** 2).sum() > 0:
        raise ValueError("reference points must not all coincide")
    return np.ascontiguousarray(ref)


def _landmarks(landmarks) -> torch.Tensor:
    if not isinstance(landmarks, torch.Tensor) or landmarks.dtype != torch.float32 or landmarks.dim() != 3 \
            or tuple(landmarks.shape[1:]) != (5, 2):
        raise ValueError(f"landmarks must be an fp32 tensor [N, 5, 2], got "
                         f"{getattr(landmarks, 'dtype', type(landmarks))} {tuple(getattr(landmarks, 'shape', ()))}")
    return landmarks


def _fit(lm: torch.Tensor, ref: np.ndarray):
    n = lm.shape[0]
    fwd = torch.empty(n, 2, 3, dtype=torch.float64, device=lm.device)
    inv = torch.empty_like(fwd)
    with torch.cuda.device(lm.device):
        _capi.check(_capi.lib().cer_face_fit(lm.data_ptr(), n, ref.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                             fwd.data_ptr(), inv.data_ptr(), _capi.current_stream_ptr(lm.device)),
                    "cer_face_fit")
    return fwd, inv


def similarity_transforms(landmarks: torch.Tensor, reference=None) -> torch.Tensor:
    """fp64 [N, 2, 3] on the landmarks' device: per face the source -> crop matrix ``cv2.warpAffine`` would be given
    by face.evoLVe's ``get_similarity_transform_for_cv2(landmarks[i], reference, reflective=True)``, computed in fp64
    on the device (no host synchronisation).  ``reference`` defaults to ``reference_points(256)``."""
    ref = _reference(reference_points() if reference is None else reference)
    lm = _landmarks(landmarks)
    if lm.device.type != "cuda":
        raise ValueError(f"landmarks must be on a CUDA device, got {lm.device}")
    _capi.require_gpu()
    return _fit(lm.contiguous(), ref)[0]


def _frame_index(frame_index, n: int, n_frames: int) -> np.ndarray:
    if frame_index is None:
        if n != n_frames:
            raise ValueError(f"align: {n} landmark sets for {n_frames} frames; give frame_index when a frame holds "
                             "other than exactly one face")
        return np.arange(n, dtype=np.int64)
    if isinstance(frame_index, torch.Tensor):
        if frame_index.device.type != "cpu" or frame_index.dtype != torch.int64:
            raise ValueError(f"frame_index must be a host-side int64 sequence, got a {frame_index.dtype} tensor on "
                             f"{frame_index.device}")
        idx = frame_index.numpy()
    elif isinstance(frame_index, np.ndarray):
        if frame_index.dtype != np.int64:
            raise ValueError(f"frame_index must be a host-side int64 sequence, got dtype {frame_index.dtype}")
        idx = frame_index
    elif isinstance(frame_index, (list, tuple)):
        if not all(isinstance(i, (int, np.integer)) and not isinstance(i, (bool, np.bool_)) for i in frame_index):
            raise ValueError("frame_index must be a host-side int64 sequence of integers")
        idx = np.array(frame_index, dtype=np.int64).reshape(-1)
    else:
        raise ValueError(f"frame_index must be a host-side int64 sequence, got {type(frame_index).__name__}")
    if idx.ndim != 1 or idx.shape[0] != n:
        raise ValueError(f"frame_index must hold one frame per face ({n}), got shape {idx.shape}")
    if n and (idx.min() < 0 or idx.max() >= n_frames):
        raise ValueError(f"frame_index holds {idx.min() if idx.min() < 0 else idx.max()}, outside [0, {n_frames})")
    return np.ascontiguousarray(idx)


def align(frames: torch.Tensor, landmarks: torch.Tensor, frame_index: Optional[Sequence[int]] = None,
          crop_size: int = 256, reference=None) -> torch.Tensor:
    """uint8 [N, crop_size, crop_size, 3] on the frames' device: face i warped out of ``frames[frame_index[i]]``.

    ``frames``: uint8 [F, H, W, 3] on a CUDA device, H and W at most 32767.  ``landmarks``: fp32 [N, 5, 2] on the same
    device.  ``frame_index``: host-side int64 sequence of N indices into ``frames`` (several faces may share a frame);
    ``None`` means face i comes from frame i and needs N == F.  ``reference``: the five points in the crop, default
    ``reference_points(crop_size)``.  Every check runs on the host before any device work and raises ``ValueError``.

    Face i is ``cv2.warpAffine(frames[frame_index[i]], M_i, (crop_size, crop_size))`` bit for bit, where M_i is
    ``similarity_transforms(landmarks, reference)[i]``: face.evoLVe's ``warp_and_crop_face`` with its matrix fitted
    in fp64 (face.evoLVe fits float32-rounded points, which moves M by about 1e-7 relative)."""
    if not isinstance(frames, torch.Tensor) or frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[3] != 3:
        raise ValueError(f"frames must be a uint8 [F, H, W, 3] tensor, got "
                         f"{getattr(frames, 'dtype', type(frames))} {tuple(getattr(frames, 'shape', ()))}")
    lm = _landmarks(landmarks)
    F_, H, W = (int(s) for s in frames.shape[:3])
    n = lm.shape[0]
    idx = _frame_index(frame_index, n, F_)
    if isinstance(crop_size, bool) or not isinstance(crop_size, (int, np.integer)) or not 1 <= crop_size <= MAX_CROP:
        raise ValueError(f"crop_size must be an integer in 1..{MAX_CROP}, got {crop_size!r}")
    if H > MAX_SIDE or W > MAX_SIDE:
        raise ValueError(f"frames of {H} x {W}: at most {MAX_SIDE} pixels per side")
    ref = _reference(reference_points(int(crop_size)) if reference is None else reference)
    if lm.device != frames.device:
        raise ValueError(f"landmarks must be on the frames' device ({frames.device}), got {lm.device}")
    if frames.device.type != "cuda":
        raise ValueError(f"frames must be on a CUDA device, got {frames.device}")
    S = int(crop_size)
    dev = frames.device
    out = torch.empty(n, S, S, 3, dtype=torch.uint8, device=dev)
    if n == 0:
        return out
    _capi.require_gpu()
    frames = frames.contiguous()
    _, inv = _fit(lm.contiguous(), ref)
    idx_dev = torch.from_numpy(idx).to(dev)
    with torch.cuda.device(dev):
        _capi.check(_capi.lib().cer_face_warp(frames.data_ptr(), F_, H, W, idx_dev.data_ptr(), inv.data_ptr(), n, S,
                                              out.data_ptr(), _capi.current_stream_ptr(dev)), "cer_face_warp")
    return out
