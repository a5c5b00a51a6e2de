"""Face alignment on the device (csrc/align.cu, faces.align): the warp reproduces OpenCV's crops pinned in
tests/golden/face_align.pt bit for bit, the fit agrees with the fp64 least squares, fit + warp equal the numpy oracle
bit for bit at a realistic size, and the crops drive infer_video and StreamSession as the oracle's crops do."""
import hashlib
import os
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import _capi, faces, streaming, synthetic, windowing
from oracle import face_align_oracle as O
from oracle import gen_align_golden as G

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
# fp64 fit vs face.evoLVe's float32 recipe on the realistic workload, measured with the numpy oracle (DESIGN §5.22):
# 2,550 of 109,314,048 channel values differ (2.33e-5), by at most 1 level where all four taps are inside the frame
# and by at most 6 at the frame's edge (the constant border makes steps of up to 255 / 32 levels per 1/32 px).
MAX_DIFF_FRACTION = 1e-4


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def golden(golden_dir):
    return torch.load(os.path.join(golden_dir, "face_align.pt"))


def _warp(frames, idx, inv, S):
    n = idx.shape[0]
    out = torch.empty(n, S, S, 3, dtype=torch.uint8, device=frames.device)
    _capi.check(_capi.lib().cer_face_warp(frames.data_ptr(), frames.shape[0], frames.shape[1], frames.shape[2],
                                          idx.data_ptr(), inv.data_ptr(), n, S, out.data_ptr(),
                                          _capi.current_stream_ptr()), "cer_face_warp")
    return out


def test_warp_reproduces_every_golden_crop(golden):
    dev = _dev()
    stride = golden["row_stride"]
    for fi, f in enumerate(golden["frames"]):
        img = G.frame(f["h"], f["w"], f["seed"])
        assert int(img.sum(dtype=np.int64)) == f["byte_sum"]
        frames = torch.from_numpy(img)[None].to(dev)
        for S in (256, 112):
            cases = [c for c in golden["cases"] if c["frame"] == fi and c["crop"] == S]
            inv = torch.tensor(np.stack([O.invert(c["M"].numpy()) for c in cases])).to(dev)
            out = _warp(frames, torch.zeros(len(cases), dtype=torch.int64, device=dev), inv, S).cpu()
            for c, crop in zip(cases, out):
                assert torch.equal(crop[::stride], c["rows"]), (fi, c["set"], S)
                assert hashlib.sha256(crop.numpy().tobytes()).hexdigest() == c["sha256"], (fi, c["set"], S)


def test_out_of_range_frame_index_gives_a_zero_crop_and_unaligned_output():
    """The C-ABI reads nothing for an index outside [0, n_frames); an output at an odd address and an odd crop take
    the byte head / tail of the store path."""
    dev = _dev()
    img = G.frame(480, 640, 11)
    frames = torch.from_numpy(img)[None].to(dev)
    M = O.similarity_fit(G.landmarks(480, 640, 10.0, 0.4, (0.5, 0.5), False, seed=1), O.reference_points(37))
    inv = torch.tensor(np.stack([O.invert(M)] * 3)).to(dev)
    idx = torch.tensor([0, 5, -1], dtype=torch.int64, device=dev)
    buf = torch.full((3 * 37 * 37 * 3 + 1,), 7, dtype=torch.uint8, device=dev)
    out = buf[1:].view(3, 37, 37, 3)
    _capi.check(_capi.lib().cer_face_warp(frames.data_ptr(), 1, 480, 640, idx.data_ptr(), inv.data_ptr(), 3, 37,
                                          out.data_ptr(), _capi.current_stream_ptr()), "cer_face_warp")
    assert np.array_equal(out[0].cpu().numpy(), O.warp(img, M, 37))
    assert int(out[1:].count_nonzero()) == 0 and int(buf[0]) == 7


def test_fit_agrees_with_the_fp64_least_squares(golden):
    dev = _dev()
    lms, _ = G.workload_faces([1] * 200, seed=9)
    lms = np.concatenate([lms, np.stack([c["landmarks"].numpy() for c in golden["cases"] if c["crop"] == 256])])
    ref = faces.reference_points(256)
    fwd = faces.similarity_transforms(torch.from_numpy(lms).to(dev), ref).cpu().numpy()
    for lm, got in zip(lms, fwd):
        want = O.similarity_fit(lm, ref, exact=True)
        assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
        assert np.abs(got - O.similarity_fit(lm, ref)).max() <= 1e-10 * np.abs(want).max()   # lstsq's accuracy


@pytest.fixture(scope="module")
def realistic():
    """300 frames of 1280x720 with one face each and 64 with four: (frames on the device, host frames, landmarks,
    frame_index)."""
    dev = _dev()
    counts = [1] * 300 + [4] * 64
    host = G.smooth_frames(len(counts))
    frames = torch.empty(len(counts), 720, 1280, 3, dtype=torch.uint8, device=dev)
    for k, f in enumerate(host):
        frames[k].copy_(torch.from_numpy(np.ascontiguousarray(f)))
    lm, idx = G.workload_faces(counts)
    return frames, host, lm, idx


def test_fit_and_warp_equal_the_oracle_at_a_realistic_size(realistic):
    frames, host, lm, idx = realistic
    dev = frames.device
    ref = faces.reference_points(256)
    lm_dev = torch.from_numpy(lm).to(dev)
    crops = faces.align(frames, lm_dev, idx).cpu().numpy()
    fwd = faces.similarity_transforms(lm_dev, ref).cpu().numpy()
    assert crops.shape == (len(idx), 256, 256, 3)
    n_diff = n_tot = 0
    for i, f in enumerate(idx):
        assert np.array_equal(crops[i], O.warp(host[f], fwd[i], 256)), i     # cv2.warpAffine(frame, fwd[i])
        M32 = O.similarity_fit(lm[i], ref, recipe=True)
        d = np.abs(crops[i].astype(np.int16) - O.warp(host[f], M32, 256).astype(np.int16))
        inside = O.interior(fwd[i], 256, 720, 1280) & O.interior(M32, 256, 720, 1280)
        assert d[inside].max(initial=0) <= 1 and d.max() <= 8, i
        n_diff += int((d > 0).sum())
        n_tot += d.size
    assert n_diff / n_tot <= MAX_DIFF_FRACTION, n_diff / n_tot


def _lfan(mods, dev, seed=0):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=mods, kernel_size=5, example_length=300,
             tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(seed))
    m.load_state_dict(synthetic.lfan_state_dict(seed, mods), strict=True)
    return m.to(dev).eval()


def test_aligned_crops_through_infer_video_and_a_stream(realistic):
    frames, host, lm, idx = realistic
    dev = frames.device
    T = 96
    sel = np.arange(T)                              # the first 96 one-face frames
    lm_dev = torch.from_numpy(lm[sel]).to(dev)
    crops = faces.align(frames[:T], lm_dev)
    fwd = faces.similarity_transforms(lm_dev).cpu().numpy()
    ref = faces.reference_points(256)
    oracle = torch.from_numpy(np.stack([O.warp(host[i], fwd[i], 256) for i in sel])).to(dev)
    recipe = torch.from_numpy(np.stack([O.warp(host[i], O.similarity_fit(lm[i], ref, recipe=True), 256)
                                        for i in sel])).to(dev)
    assert torch.equal(crops, oracle)
    mods = ["video", "vggish", "bert"]
    m = _lfan(mods, dev, seed=3)
    g = torch.Generator().manual_seed(4)
    feats = {"vggish": torch.randn(T, 128, generator=g).to(dev), "bert": torch.randn(T, 768, generator=g).to(dev)}
    got = windowing.infer_video(m, crops, feats)
    assert torch.equal(got, windowing.infer_video(m, oracle, feats))
    # against the crops face.evoLVe + cv2 make (float32 recipe): same embeddings and decisions
    emb = m.spatial["visual"](windowing.preprocess_frames(m, crops))
    emb_cv2 = m.spatial["visual"](windowing.preprocess_frames(m, recipe))
    assert F.cosine_similarity(emb, emb_cv2, dim=1).min().item() >= 0.9999
    want = windowing.infer_video(m, recipe, feats)
    assert torch.equal(got.argmax(-1), want.argmax(-1))
    # one StreamSession push of the aligned crops equals pushing the oracle's crops
    outs = []
    for video in (crops, oracle):
        sess = streaming.StreamSession(m, max_streams=1, max_chunk=T)
        sid = sess.open()
        logits, _ = sess.push([sid], {"video": video[None], **{k: v[None] for k, v in feats.items()}})
        outs.append((logits, sess.close(sid)))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
