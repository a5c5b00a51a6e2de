"""Generate tests/golden/face_align.pt from OpenCV's own cv2.warpAffine.

    python oracle/gen_align_golden.py

Needs `cv2` (opencv-python); the tests read the file and never import it.
  * frames: seeded uint8 noise (``frame(h, w, seed)``, numpy PCG64) at 640x480, 1280x720, 300x500 (tall) and 7x5;
    each frame's byte sum is stored so that a change of the generator is caught as such;
  * landmark sets (``LANDMARK_SETS``): the reference points under a seeded similarity plus 0.75 px noise: upright,
    rotated +40 and -40 degrees, mirrored (the reflective branch), small (the warp up-scales), large (down-scales),
    partly outside the frame and wholly outside it (the constant border); frame-relative so every frame size has all;
  * crops at 256 and 112;
  * per case: the fp32 landmarks, the matrix cv2 received (face.evoLVe's float32 recipe, ``similarity_fit(..,
    recipe=True)``), the sha256 of cv2's whole crop and every 8th row of it (the file stays near 1 MB);
  * the OpenCV version.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import face_align_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "face_align.pt")
FRAMES = ((480, 640, 11), (720, 1280, 12), (500, 300, 13), (5, 7, 14))      # (h, w, seed)
CROPS = (256, 112)
ROW_STRIDE = 8
# name: (rotation deg, face size as a fraction of min(h, w), centre (x, y) as fractions of (w, h), mirrored)
LANDMARK_SETS = {
    "upright": (0.0, 0.35, (0.5, 0.45), False),
    "rot_p40": (40.0, 0.35, (0.45, 0.5), False),
    "rot_m40": (-40.0, 0.35, (0.55, 0.5), False),
    "mirrored": (10.0, 0.35, (0.5, 0.5), True),
    "small": (5.0, 0.08, (0.3, 0.6), False),
    "large": (-8.0, 0.9, (0.5, 0.5), False),
    "partly_outside": (15.0, 0.4, (0.97, 0.1), False),
    "outside": (0.0, 0.3, (-1.5, 2.0), False),
}


def frame(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def landmarks(h, w, rot_deg, size, centre, mirrored, seed, noise=0.75):
    """fp32 [5, 2]: the 112-crop reference points, centred, scaled to ``size * min(h, w)`` across, rotated, moved to
    ``centre`` and jittered by ``noise`` px (seeded), so the fit is never exact."""
    ref = O.reference_points(112)
    p = (ref - ref.mean(0)) / 112.0 * size * min(h, w)
    if mirrored:
        p[:, 0] = -p[:, 0]
    t = np.deg2rad(rot_deg)
    R = np.array([[np.cos(t), -np.sin(t)], [np.sin(t), np.cos(t)]])
    p = p @ R.T + np.array([centre[0] * w, centre[1] * h])
    p += np.random.default_rng(seed).normal(0, noise, p.shape)
    return p.astype(np.float32)


# The realistic workload of the GPU tests and tools/align_bench.py: smooth frames (a shifted low-frequency pattern, so
# neighbouring pixels differ by a few levels as in camera frames) and one face per frame, or four on some frames.
def smooth_frames(n, h=720, w=1280):
    """n uint8 [h, w, 3] frames (views of one pattern): frame k is a sum of low-frequency waves shifted by (7k, 13k)."""
    y = np.arange(h + 7 * (n - 1), dtype=np.float64)[:, None, None]
    x = np.arange(w + 13 * (n - 1), dtype=np.float64)[None, :, None]
    c = np.arange(3, dtype=np.float64)[None, None, :]
    v = 128 + 55 * np.sin(x / 23.0 + 1.3 * c) + 45 * np.cos(y / 17.0 + 0.7 * c) + 20 * np.sin((x + y) / 41.0 + c)
    base = np.clip(np.rint(v), 0, 255).astype(np.uint8)
    return [base[7 * k:7 * k + h, 13 * k:13 * k + w] for k in range(n)]


def workload_faces(faces_per_frame, h=720, w=1280, seed=0):
    """(fp32 landmarks [N, 5, 2], int64 frame_index [N]) for frames with the given face counts: per face a seeded
    rotation in +-40 degrees, a size of 0.12 - 0.45 of min(h, w), a centre anywhere in the middle 80 % and 1 px of
    landmark noise."""
    rng = np.random.default_rng(seed)
    lms, idx = [], []
    for f, k in enumerate(faces_per_frame):
        for _ in range(k):
            spec = (rng.uniform(-40, 40), rng.uniform(0.12, 0.45), (rng.uniform(0.1, 0.9), rng.uniform(0.1, 0.9)), False)
            lms.append(landmarks(h, w, *spec, seed=int(rng.integers(1 << 31)), noise=1.0))
            idx.append(f)
    return np.stack(lms), np.array(idx, dtype=np.int64)


def main():
    import cv2
    cases = []
    for fi, (h, w, seed) in enumerate(FRAMES):
        img = frame(h, w, seed)
        for li, (name, spec) in enumerate(LANDMARK_SETS.items()):
            lm = landmarks(h, w, *spec, seed=1000 + 10 * fi + li)
            for S in CROPS:
                M = O.similarity_fit(lm, O.reference_points(S), recipe=True)
                crop = cv2.warpAffine(img, M, (S, S))
                cases.append({"frame": fi, "set": name, "crop": S, "landmarks": torch.from_numpy(lm),
                              "M": torch.from_numpy(M), "sha256": hashlib.sha256(crop.tobytes()).hexdigest(),
                              "rows": torch.from_numpy(np.ascontiguousarray(crop[::ROW_STRIDE]))})
    torch.save({"frames": [{"h": h, "w": w, "seed": s, "byte_sum": int(frame(h, w, s).sum(dtype=np.int64))}
                           for h, w, s in FRAMES],
                "row_stride": ROW_STRIDE, "cases": cases, "opencv": cv2.__version__}, OUT)
    print(f"{OUT}: {len(cases)} cases, {os.path.getsize(OUT) / 1e6:.2f} MB, OpenCV {cv2.__version__}")


if __name__ == "__main__":
    main()
