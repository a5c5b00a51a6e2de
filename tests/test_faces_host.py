"""Face alignment's host side, without a GPU: the numpy oracle against OpenCV's warpAffine outputs pinned in
tests/golden/face_align.pt (and against cv2 itself where it is installed), the similarity fit, the reference points,
every refusal of ``faces.align`` (all raised before any device work) and the new C-ABI symbols."""
import hashlib
import os

import numpy as np
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import faces
from oracle import face_align_oracle as O
from oracle import gen_align_golden as G


@pytest.fixture(scope="module")
def golden(golden_dir):
    return torch.load(os.path.join(golden_dir, "face_align.pt"))


def _frames(golden):
    out = []
    for f in golden["frames"]:
        img = G.frame(f["h"], f["w"], f["seed"])
        assert int(img.sum(dtype=np.int64)) == f["byte_sum"], "the seeded frame generator changed"
        out.append(img)
    return out


def test_golden_covers_the_cases(golden):
    cases = golden["cases"]
    assert len(cases) == 4 * 8 * 2
    assert {c["set"] for c in cases} == set(G.LANDMARK_SETS) and {c["crop"] for c in cases} == {256, 112}
    assert {(f["h"], f["w"]) for f in golden["frames"]} == {(480, 640), (720, 1280), (500, 300), (5, 7)}
    dets = [np.linalg.det(c["M"].numpy()[:, :2]) for c in cases if c["set"] == "mirrored" and c["frame"] < 3]
    assert all(d < 0 for d in dets), "the mirrored faces take the reflective branch"


def test_oracle_warp_equals_golden_cv2_bit_for_bit(golden):
    frames = _frames(golden)
    stride = golden["row_stride"]
    for c in golden["cases"]:
        got = O.warp(frames[c["frame"]], c["M"].numpy(), c["crop"])
        assert torch.equal(torch.from_numpy(np.ascontiguousarray(got[::stride])), c["rows"]), (c["frame"], c["set"])
        assert hashlib.sha256(got.tobytes()).hexdigest() == c["sha256"], (c["frame"], c["set"], c["crop"])


def test_golden_matrices_are_the_float32_recipe(golden):
    for c in golden["cases"]:
        want = O.similarity_fit(c["landmarks"].numpy(), O.reference_points(c["crop"]), recipe=True)
        assert np.array_equal(want, c["M"].numpy())


def test_oracle_warp_equals_cv2_on_fresh_cases():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2024)
    for t in range(40):
        H, W = [(480, 640), (720, 1280), (37, 53), (3, 2), (301, 199)][t % 5]
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        S = [256, 112, 31, 1][t % 4]
        ang, sc = rng.uniform(-np.pi, np.pi), np.exp(rng.uniform(-2, 2))
        M = np.array([[np.cos(ang) * sc, -np.sin(ang) * sc, rng.uniform(-W, W)],
                      [np.sin(ang) * sc, np.cos(ang) * sc, rng.uniform(-H, H)]])
        if t % 3 == 0:
            M[0] *= -1
        assert np.array_equal(O.warp(img, M, S), cv2.warpAffine(img, M, (S, S))), t


def _similarity(theta, s, t, reflect=False):
    c, si = np.cos(theta) * s, np.sin(theta) * s
    M = np.array([[c, -si, t[0]], [si, c, t[1]]])
    if reflect:
        M[0, :2] *= -1
    return M


@pytest.mark.parametrize("reflect", [False, True])
def test_fit_recovers_a_known_transform(reflect):
    ref = O.reference_points(256)
    for k, (theta, s, t) in enumerate([(0.0, 1.0, (0, 0)), (0.7, 2.3, (-40.0, 310.0)), (-0.69, 0.4, (12.5, -3.0))]):
        M = _similarity(theta, s, t, reflect)                   # crop -> source; the fit returns source -> crop
        src = ref @ M[:, :2].T + M[:, 2]
        fwd = O.similarity_fit(src, ref)
        assert (np.linalg.det(fwd[:, :2]) < 0) == reflect
        back = src @ fwd[:, :2].T + fwd[:, 2]
        assert np.abs(back - ref).max() <= 1e-12 * 256, k
        want = O.invert(M)
        assert np.abs(O.similarity_fit(src, ref, exact=True) - want).max() <= 1e-13 * np.abs(want).max(), k
        assert np.abs(fwd - want).max() <= 1e-10 * np.abs(want).max(), k     # lstsq's own float64 accuracy


def test_fit_on_noisy_landmarks():
    """Against the least-squares solution in long double (the centred closed form csrc/align.cu uses): the same
    closed form in float64 to 1e-14 relative, face.evoLVe's ``lstsq`` in float64 to 1e-10 (its own accuracy on these
    uncentred systems, measured up to 1.6e-11) and the float32 recipe to float32 precision."""
    lms, _ = G.workload_faces([1] * 64, seed=5)
    ref = O.reference_points(256)
    xm, ym = ref[:, 0].mean(), ref[:, 1].mean()
    xc, yc = ref[:, 0] - xm, ref[:, 1] - ym
    for lm in lms.astype(np.float64):
        want = O.similarity_fit(lm, ref, exact=True)
        scale = np.abs(want).max()
        uc, vc = lm[:, 0] - lm[:, 0].mean(), lm[:, 1] - lm[:, 1].mean()
        n = (xc * xc + yc * yc).sum()
        a, b = (xc * uc + yc * vc).sum() / n, (yc * uc - xc * vc).sum() / n
        tx, ty = lm[:, 0].mean() - a * xm - b * ym, lm[:, 1].mean() + b * xm - a * ym
        d = a * a + b * b
        f64 = np.array([[a / d, -b / d, -(a * tx - b * ty) / d], [b / d, a / d, -(b * tx + a * ty) / d]])
        assert np.abs(f64 - want).max() <= 1e-14 * scale
        assert np.abs(O.similarity_fit(lm, ref) - want).max() <= 1e-10 * scale
        f32 = O.similarity_fit(lm.astype(np.float32), ref, recipe=True)
        assert np.abs(f32 - want).max() <= 4 * np.finfo(np.float32).eps * scale


@pytest.mark.parametrize("crop", [112, 256, 96])
def test_reference_points_restate_face_evolve(crop):
    want = O.get_reference_facial_points(default_square=True) * (crop / 112.0)
    assert np.array_equal(faces.reference_points(crop), want)
    assert np.array_equal(O.reference_points(crop), want)
    if crop == 112:
        assert np.array_equal(want[:, 0], O.TEMPLATE_96x112[:, 0] + 8)


def test_reference_points_with_padding():
    for pad, outer in [(0.25, (0, 0)), (0.0, (16, 16)), (0.1, (8, 8))]:
        assert np.array_equal(faces.reference_points(256, pad, outer), O.reference_points(256, pad, outer))
    with pytest.raises(ValueError):
        faces.reference_points(256, 1.5)


def _u8(*shape):
    return torch.zeros(*shape, dtype=torch.uint8)


def _lm(n):
    return torch.zeros(n, 5, 2)


@pytest.mark.parametrize("bad", ["dtype", "rank", "channels", "device"])
def test_align_refuses_frames(bad):
    frames = {"dtype": torch.zeros(2, 8, 8, 3), "rank": _u8(8, 8, 3), "channels": _u8(2, 8, 8, 4),
              "device": _u8(2, 8, 8, 3)}[bad]
    with pytest.raises(ValueError, match="frames"):
        faces.align(frames, _lm(2))


@pytest.mark.parametrize("bad", ["dtype", "shape", "points", "type"])
def test_align_refuses_landmarks(bad):
    lm = {"dtype": _lm(2).double(), "shape": torch.zeros(2, 10), "points": torch.zeros(2, 4, 2),
          "type": np.zeros((2, 5, 2), np.float32)}[bad]
    with pytest.raises(ValueError, match="landmarks"):
        faces.align(_u8(2, 8, 8, 3), lm)


def test_align_refuses_landmarks_on_another_device():
    with pytest.raises(ValueError, match="landmarks must be on the frames' device"):
        faces.align(_u8(2, 8, 8, 3), _lm(2).to("meta"))


@pytest.mark.parametrize("idx", [[0, 2], [-1, 0], [0], [0, 1, 1], [0.0, 1.0], [True, False], "01",
                                 np.array([0, 1], np.int32), torch.tensor([0, 1], dtype=torch.int32),
                                 torch.tensor([[0, 1]]), np.array([[0], [1]])])
def test_align_refuses_frame_index(idx):
    with pytest.raises(ValueError, match="frame_index"):
        faces.align(_u8(2, 8, 8, 3), _lm(2), frame_index=idx)


def test_align_refuses_a_device_frame_index():
    with pytest.raises(ValueError, match="frame_index"):
        faces.align(_u8(2, 8, 8, 3), _lm(2), frame_index=torch.tensor([0, 1]).to("meta"))


def test_align_needs_one_face_per_frame_without_frame_index():
    with pytest.raises(ValueError, match="frame_index"):
        faces.align(_u8(2, 8, 8, 3), _lm(3))


@pytest.mark.parametrize("crop", [0, 1025, -3, 2.5, True])
def test_align_refuses_crop_size(crop):
    with pytest.raises(ValueError, match="crop_size"):
        faces.align(_u8(2, 8, 8, 3), _lm(2), crop_size=crop)


@pytest.mark.parametrize("hw", [(32768, 4), (4, 32768)])
def test_align_refuses_frames_over_32767_px(hw):
    frames = _u8(1, 1, 1, 3).expand(1, *hw, 3)                   # a stride-0 view: no memory behind it
    with pytest.raises(ValueError, match="32767"):
        faces.align(frames, _lm(1))


@pytest.mark.parametrize("ref", [np.zeros((5, 2)), np.ones((4, 2)), np.full((5, 2), np.nan)])
def test_align_refuses_reference(ref):
    with pytest.raises(ValueError, match="reference"):
        faces.align(_u8(2, 8, 8, 3), _lm(2), reference=ref)


def test_valid_arguments_reach_the_device_check():
    """Everything above passes with these arguments: only the frames' device is left to refuse."""
    with pytest.raises(ValueError, match="CUDA"):
        faces.align(_u8(4, 8, 8, 3), _lm(5), frame_index=[0, 1, 1, 3, 3], crop_size=1024)
    with pytest.raises(ValueError, match="CUDA"):
        faces.similarity_transforms(_lm(2))


def test_capi_declares_the_face_symbols():
    from feature_vs_text_compound_emotion_b200 import _capi
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cer_b200.h")).read()
    for name in ("cer_face_fit", "cer_face_warp"):
        assert name in _capi.SIGNATURES and f"int {name}(" in hdr
