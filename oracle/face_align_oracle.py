"""numpy restatement of five-point face alignment, independent of the kernels and of OpenCV:

  * ``reference_points``: face.evoLVe's ``get_reference_facial_points`` (align_trans.py) on the 96 x 112 template,
    scaled by ``crop_size / 112`` as face.evoLVe's face_align.py does;
  * ``similarity_fit``: face.evoLVe's ``matlab_cp2tform.get_similarity_transform_for_cv2(src, ref, reflective=True)``:
    the non-reflective least-squares similarity (``np.linalg.lstsq``), again with the reference's x negated and
    composed with the reflection, keeping the smaller residual (the non-reflective one on a tie);
    ``recipe=True`` casts landmarks and reference to float32 first, as ``warp_and_crop_face`` does;
  * ``invert``: the 2 x 3 inversion ``cv::warpAffine`` applies to the matrix it is given;
  * ``warp``: ``cv2.warpAffine(img, M, (S, S))`` with its defaults (INTER_LINEAR, BORDER_CONSTANT 0) in OpenCV's
    fixed-point arithmetic: 10-bit coordinate steps, 1/32-px taps, 15-bit bilinear weights.
"""
from __future__ import annotations

import numpy as np

TEMPLATE_96x112 = np.array([[30.29459953, 51.69630051],
                            [65.53179932, 51.50139999],
                            [48.02519989, 71.73660278],
                            [33.54930115, 92.3655014],
                            [62.72990036, 92.20410156]])


def get_reference_facial_points(output_size=None, inner_padding_factor=0.0, outer_padding=(0, 0),
                                default_square=False):
    """face.evoLVe align_trans.get_reference_facial_points, line for line (exceptions become ValueError)."""
    tmp_5pts = TEMPLATE_96x112.copy()
    tmp_crop_size = np.array((96, 112))
    if default_square:
        size_diff = max(tmp_crop_size) - tmp_crop_size
        tmp_5pts += size_diff / 2
        tmp_crop_size += size_diff
    if output_size and output_size[0] == tmp_crop_size[0] and output_size[1] == tmp_crop_size[1]:
        return tmp_5pts
    if inner_padding_factor == 0 and tuple(outer_padding) == (0, 0):
        if output_size is None:
            return tmp_5pts
        raise ValueError(f"No paddings to do, output_size must be None or {tmp_crop_size}")
    if not 0 <= inner_padding_factor <= 1.0:
        raise ValueError("Not (0 <= inner_padding_factor <= 1.0)")
    if (inner_padding_factor > 0 or outer_padding[0] > 0 or outer_padding[1] > 0) and output_size is None:
        output_size = tmp_crop_size * (1 + inner_padding_factor * 2)
        output_size = output_size.astype(np.int32) + np.array(outer_padding)
    if not (outer_padding[0] < output_size[0] and outer_padding[1] < output_size[1]):
        raise ValueError("Not (outer_padding[0] < output_size[0] and outer_padding[1] < output_size[1])")
    if inner_padding_factor > 0:
        size_diff = tmp_crop_size * inner_padding_factor * 2
        tmp_5pts += size_diff / 2
        tmp_crop_size += np.round(size_diff).astype(np.int32)
    size_bf_outer_pad = np.array(output_size) - np.array(outer_padding) * 2
    if size_bf_outer_pad[0] * tmp_crop_size[1] != size_bf_outer_pad[1] * tmp_crop_size[0]:
        raise ValueError("Must have (output_size - outer_padding) = some_scale * (crop_size * (1.0 + inner_padding_factor)")
    scale_factor = size_bf_outer_pad[0].astype(np.float32) / tmp_crop_size[0]
    tmp_5pts = tmp_5pts * scale_factor
    return tmp_5pts + np.array(outer_padding)


def reference_points(crop_size=256, inner_padding_factor=0.0, outer_padding=(0, 0), default_square=True):
    """face_align.py's recipe: ``get_reference_facial_points(default_square=True) * (crop_size / 112)``; with padding,
    the template is padded and resized to a crop_size x crop_size output by the function itself."""
    if inner_padding_factor == 0 and tuple(outer_padding) == (0, 0):
        return get_reference_facial_points(default_square=default_square) * (crop_size / 112.0)
    return get_reference_facial_points((crop_size, crop_size), inner_padding_factor, outer_padding, default_square)


def _nonreflective(uv, xy):
    """findNonreflectiveSimilarity(uv, xy): T (3 x 3, row-vector convention) maps uv onto xy."""
    x, y = xy[:, :1], xy[:, 1:]
    M = xy.shape[0]
    X = np.vstack((np.hstack((x, y, np.ones((M, 1)), np.zeros((M, 1)))),
                   np.hstack((y, -x, np.zeros((M, 1)), np.ones((M, 1))))))
    U = np.vstack((uv[:, :1], uv[:, 1:]))
    if np.linalg.matrix_rank(X) < 4:
        raise ValueError("cp2tform: two unique points required")
    sc, ss, tx, ty = np.squeeze(np.linalg.lstsq(X, U, rcond=None)[0])
    Tinv = np.array([[sc, -ss, 0], [ss, sc, 0], [tx, ty, 1]])
    T = np.linalg.inv(Tinv)
    T[:, 2] = np.array([0, 0, 1])
    return T


def _nonreflective_centred(uv, xy):
    """The same least squares in the centred closed form (the one csrc/align.cu uses), in long double."""
    uv, xy = uv.astype(np.longdouble), xy.astype(np.longdouble)
    xc, yc = xy[:, 0] - xy[:, 0].mean(), xy[:, 1] - xy[:, 1].mean()
    uc, vc = uv[:, 0] - uv[:, 0].mean(), uv[:, 1] - uv[:, 1].mean()
    n = (xc * xc + yc * yc).sum()
    sc, ss = (xc * uc + yc * vc).sum() / n, (yc * uc - xc * vc).sum() / n
    tx = uv[:, 0].mean() - sc * xy[:, 0].mean() - ss * xy[:, 1].mean()
    ty = uv[:, 1].mean() + ss * xy[:, 0].mean() - sc * xy[:, 1].mean()
    d = sc * sc + ss * ss
    return np.array([[sc / d, ss / d, 0], [-ss / d, sc / d, 0], [-(sc * tx - ss * ty) / d, -(ss * tx + sc * ty) / d, 1]])


def _fwd(T, uv):
    return np.dot(np.hstack((uv, np.ones((uv.shape[0], 1)))), T)[:, :2]


def similarity_fit(src, ref, recipe=False, exact=False):
    """The 2 x 3 forward matrix (source -> crop) that ``cv2.warpAffine`` is given, float64.  ``src`` [5, 2] landmarks,
    ``ref`` [5, 2] reference points.  ``recipe``: cast both to float32 first (warp_and_crop_face).  ``exact``: solve
    in the centred closed form in long double instead of ``lstsq`` (whose float64 result on these uncentred systems
    is off by up to ~2e-11 relative), rounded to float64 at the end."""
    dt = np.float32 if recipe else np.float64
    uv, xy = np.asarray(src, dtype=dt), np.asarray(ref, dtype=dt)
    solve = _nonreflective_centred if exact else _nonreflective
    T1 = solve(uv, xy)
    xyR = xy.copy()
    xyR[:, 0] = -1 * xyR[:, 0]
    T2 = np.dot(solve(uv, xyR), np.array([[-1, 0, 0], [0, 1, 0], [0, 0, 1]]))
    n1 = np.linalg.norm(_fwd(T1, uv) - xy)
    n2 = np.linalg.norm(_fwd(T2, uv) - xy)
    T = T1 if n1 <= n2 else T2
    return np.ascontiguousarray(T[:, 0:2].T).astype(np.float64)


def invert(M):
    """cv::warpAffine's own inversion of the forward matrix (imgwarp.cpp), same operation order, float64."""
    M = np.asarray(M, dtype=np.float64).reshape(6).tolist()
    D = M[0] * M[4] - M[1] * M[3]
    D = 1.0 / D if D != 0 else 0.0
    A11, A22 = M[4] * D, M[0] * D
    A12, A21 = M[1] * -D, M[3] * -D
    b1 = -A11 * M[2] - A12 * M[5]
    b2 = -A21 * M[2] - A22 * M[5]
    return np.array([[A11, A12, b1], [A21, A22, b2]])


def _taps(A, S):
    """Per output pixel of an S x S crop: the top-left source tap (sx, sy) and its 1/32-px fractions (fx, fy)."""
    r = np.arange(S, dtype=np.float64)
    adelta = np.rint(A[0, 0] * r * 1024).astype(np.int64)
    bdelta = np.rint(A[1, 0] * r * 1024).astype(np.int64)
    X0 = np.rint((A[0, 1] * r + A[0, 2]) * 1024).astype(np.int64) + 16
    Y0 = np.rint((A[1, 1] * r + A[1, 2]) * 1024).astype(np.int64) + 16
    X = (X0[:, None] + adelta[None, :]) >> 5
    Y = (Y0[:, None] + bdelta[None, :]) >> 5
    return np.clip(X >> 5, -32768, 32767), np.clip(Y >> 5, -32768, 32767), X & 31, Y & 31


def warp(img, M, S, inverse=None):
    """``cv2.warpAffine(img, M, (S, S))`` for uint8 [H, W, C]: OpenCV's fixed-point INTER_LINEAR, BORDER_CONSTANT 0.
    ``inverse`` skips the inversion (the matrices a device fit produced)."""
    img = np.asarray(img)
    H, W = img.shape[:2]
    A = invert(M) if inverse is None else np.asarray(inverse, dtype=np.float64).reshape(2, 3)
    sx, sy, fx, fy = _taps(A, S)
    acc = np.zeros((S, S) + img.shape[2:], dtype=np.int64)
    for dy, wy in ((0, 32 - fy), (1, fy)):
        for dx, wx in ((0, 32 - fx), (1, fx)):
            ty, tx = sy + dy, sx + dx
            ok = (ty >= 0) & (ty < H) & (tx >= 0) & (tx < W)
            v = img[np.where(ok, ty, 0), np.where(ok, tx, 0)].astype(np.int64)
            w = (wy * wx * 32) * ok
            acc += v * (w[..., None] if img.ndim == 3 else w)
    return np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)


def interior(M, S, H, W):
    """bool [S, S]: the crop pixels of ``warp(img, M, S)`` (img H x W) whose four taps all lie inside the frame."""
    sx, sy, _, _ = _taps(invert(M), S)
    return (sx >= 0) & (sx + 1 < W) & (sy >= 0) & (sy + 1 < H)


def align(frames, landmarks, frame_index, S, ref, recipe=False):
    """Per face i: ``warp(frames[frame_index[i]], similarity_fit(landmarks[i], ref), S)`` -> uint8 [N, S, S, C]."""
    return np.stack([warp(frames[f], similarity_fit(lm, ref, recipe), S) for lm, f in zip(landmarks, frame_index)])
