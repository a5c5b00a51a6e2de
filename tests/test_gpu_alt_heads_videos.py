"""Whole-video inference of CAN / JMT / MT over many videos per call (windowing.infer_videos) and the segmented
tensor-core attention under it (cer_sdpa_tc_seg_forward): the kernel against an fp64 attention and bit for bit against
batch-1 launches, CAN equal to per-video inference and to a StreamSession, JMT / MT against per-video forward and the
CPU oracle."""
import warnings

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, engine as E, streaming, synthetic, windowing
from oracle import lfan_oracle as O

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
SEG_LENGTHS = [1, 7, 63, 64, 65, 300, 1000, 3001]


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _fp64_attention(q, k, v):
    q, k, v = (t.double() for t in (q, k, v))
    return torch.softmax(q @ k.t() / q.shape[1] ** 0.5, dim=-1) @ v


@pytest.mark.parametrize("e", [128, 64])
def test_segmented_kernel_against_fp64_and_batch1(e):
    """Self-attention on column slices of a packed [rows, 3E] projection, and cross-attention with q from that buffer
    and k / v from another; segments in two orders (so each length sits at different offsets)."""
    dev = _dev()
    g = torch.Generator().manual_seed(e)
    for lengths in (SEG_LENGTHS, SEG_LENGTHS[::-1]):
        seg = E.Segments(lengths, dev)
        qkv = torch.randn(seg.rows, 3 * e, generator=g).to(dev)
        kv = torch.randn(seg.rows, 2 * e, generator=g).to(dev)
        for name, (q, k, v) in {"self": (qkv[:, :e], qkv[:, e:2 * e], qkv[:, 2 * e:]),
                                "cross": (qkv[:, :e], kv[:, :e], kv[:, e:])}.items():
            got = E.sdpa_segments(q, k, v, seg)
            assert got.shape == (seg.rows, e)
            for a, b in zip(seg.offsets[:-1], seg.offsets[1:]):
                err = (got[a:b].double() - _fp64_attention(q[a:b], k[a:b], v[a:b])).abs().max().item()
                assert err <= 5e-3, (name, e, b - a, err)
                alone = E.sdpa(q[a:b], k[a:b], v[a:b], 1, b - a, b - a)          # cer_sdpa_tc_forward, batch 1
                assert torch.equal(got[a:b], alone), (name, e, b - a)


def test_segmented_kernel_refusals():
    dev = _dev()
    seg = E.Segments([3, 5], dev)
    x = torch.randn(8, 3 * 128, device=dev)
    with pytest.raises(ValueError, match="E 64 or 128"):
        E.sdpa_segments(x[:, :96], x[:, 96:192], x[:, 192:288], seg)
    with pytest.raises(ValueError, match="16-byte aligned"):
        E.sdpa_segments(x[:, 1:129], x[:, 128:256], x[:, 256:], seg)
    with pytest.raises(ValueError, match=r"\[8, E\]"):
        E.sdpa_segments(x[:7, :128], x[:7, 128:256], x[:7, 256:], seg)
    many = E.Segments([1] * 65536, dev)
    y = torch.randn(65536, 64, device=dev)
    with pytest.raises(_capi.CerError, match="65535"):
        E.sdpa_segments(y, y, y, many)
    out = torch.full((8, 128), 7.0, device=dev)
    lib = _capi.lib()
    assert lib.cer_sdpa_tc_seg_forward(x.data_ptr(), 384, x.data_ptr(), 384, x.data_ptr(), 384, seg.off.data_ptr(), 0, 0, 128,
                                       out.data_ptr(), 128, _capi.current_stream_ptr()) == 0
    torch.cuda.synchronize()
    assert (out == 7.0).all()                                             # n_seg == 0: nothing launched


def _can(mods, dev, seed=0, task="CLASSIFICATION"):
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    m = CAN(task=task, modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
            root_dir="", device=dev,
            visual_state_dict=synthetic.visual_backbone_state_dict(seed) if "video" in mods else None,
            audio_state_dict=synthetic.vggish_state_dict(seed) if "logmel" in mods else None)
    m.load_state_dict(synthetic.can_state_dict(seed, mods), strict=True)
    return m.to(dev).eval()


def _jmt(name, dev, seed=0):
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    mods = ["video", "vggish"]
    m = JMT(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
            root_dir="", device=dev, model_name=name, visual_state_dict=synthetic.visual_backbone_state_dict(seed))
    m.load_state_dict(synthetic.jmt_state_dict(seed, mods, model_name=name), strict=True)
    return m.to(dev).eval()


def _videos(lengths, dev, seed):
    """uint8 256x256 crops, log-mel examples, vggish / bert rows per video (slices of shared seeded buffers)."""
    n = max(lengths)
    raw = synthetic.raw_frames_u8(64, seed=seed).repeat((n + 64 * len(lengths)) // 64 + 1, 1, 1, 1).to(dev)
    lm = synthetic.logmel_patches(n, seed=seed + 1).to(dev)
    g = torch.Generator().manual_seed(seed + 2)
    bert, vgg = torch.randn(n, 768, generator=g).to(dev), torch.randn(n, 128, generator=g).to(dev)
    vids = [raw[11 * i:11 * i + t] for i, t in enumerate(lengths)]
    feats = [{"logmel": lm[:t], "bert": bert[n - t:], "vggish": vgg[:t]} for t in lengths]
    return vids, feats


CAN_LENGTHS = [1, 37, 300, 1201]


def test_can_videos_equal_per_video_inference_and_forward(monkeypatch):
    """infer_videos over several videos is infer_video per video bit for bit (one IR-50 plan for every pass size,
    CER_RASTER=0, so the embeddings agree), within 1e-5 relative of CAN.forward(X) in the reference layout (the
    offline chain of linear launches), and a 'wave' run equals the same run on wave_to_examples' examples."""
    dev = _dev()
    monkeypatch.setenv("CER_RASTER", "0")
    for task in ("CLASSIFICATION", "REGRESSION"):
        mods = ["video", "logmel", "bert"]
        m = _can(mods, dev, seed=3, task=task)
        vids, feats = _videos(CAN_LENGTHS, dev, seed=40)
        feats = [{k: f[k] for k in ("logmel", "bert")} for f in feats]
        batch = windowing.infer_videos(m, vids, feats)
        assert [tuple(o.shape) for o in batch] == [(t, 7) for t in CAN_LENGTHS]
        for v, f, got in zip(vids, feats, batch):
            assert torch.equal(windowing.infer_video(m, v, dict(f)), got), v.shape[0]
            T = v.shape[0]
            if T == 1:
                continue                  # the reference layout cannot carry T = 1: _backbones squeezes dim 1 (model.py)
            X = {"video": windowing.preprocess_frames(m, v)[None],
                 "logmel": f["logmel"].view(1, T, 96, 64).permute(0, 3, 1, 2).contiguous(), "bert": f["bert"][None]}
            want = m(X)[0]
            err = (got - want).abs().max().item()
            assert err <= 1e-5 * max(1.0, want.abs().max().item()), (task, T, err)
        if task == "REGRESSION":
            assert max(o.abs().max().item() for o in batch) <= 1.0
    fps = 30.0
    waves = [(torch.randn(streaming.synced_samples(t, fps) - 700 * i, generator=torch.Generator().manual_seed(i)) * 0.3).to(dev)
             for i, t in enumerate(CAN_LENGTHS)]
    with_wave = windowing.infer_videos(m, vids, [{"wave": w, "bert": f["bert"]} for w, f in zip(waves, feats)], fps=fps)
    with_ex = windowing.infer_videos(m, vids, [{"logmel": windowing.wave_to_examples(m, w, v.shape[0], fps), "bert": f["bert"]}
                                               for w, v, f in zip(waves, vids, feats)], fps=fps)
    for a, b in zip(with_wave, with_ex):
        assert torch.equal(a, b)


def test_can_videos_equal_stream_session():
    """With the same feature rows, a video's logits from infer_videos equal the concatenated push + close results of a
    StreamSession bit for bit, whatever the other videos in the call: both run the row-invariant head kernel on the
    causal TCN's rows."""
    dev = _dev()
    mods = ["cnn_res50", "vggish", "bert"]
    m = _can(mods, dev, seed=5)
    lengths = CAN_LENGTHS + [64]
    g = torch.Generator().manual_seed(9)
    rows = [{k: torch.randn(t, synthetic.EMBEDDING_DIM[k], generator=g).to(dev) for k in mods} for t in lengths]
    dummy = [torch.empty(t, 1, device=dev) for t in lengths]               # no 'video' modality: only the length is read
    batch = windowing.infer_videos(m, dummy, rows)
    pair = windowing.infer_videos(m, dummy[1:3], rows[1:3])
    assert torch.equal(pair[0], batch[1]) and torch.equal(pair[1], batch[2])
    sess = streaming.StreamSession(m, max_streams=len(lengths), max_chunk=30)
    for t, x, want in zip(lengths, rows, batch):
        sid = sess.open()
        got = [sess.push([sid], {k: v[None, a:a + 30] for k, v in x.items()})[0][0] for a in range(0, t, 30)]
        got.append(sess.close(sid))
        got = torch.cat(got)
        assert got.shape == (t, 7) and torch.equal(got, want), (t, (got - want).abs().max().item())


@pytest.mark.parametrize("name", ["JMT", "MT"])
def test_jmt_videos_against_per_video_forward(name, monkeypatch):
    """Against per-video JMT.forward(X) with B = 1 (its final encoder attends over the same T rows): the row GEMMs
    pick split-K from the row count, so the bits differ; max-abs <= 1e-4 x the logits' scale, argmax >= 99.5 %.  The
    same video alone and inside a batch of others agrees to the same bar."""
    dev = _dev()
    monkeypatch.setenv("CER_RASTER", "0")
    m = _jmt(name, dev, seed=2)
    lengths = [1, 37, 300, 1201]
    vids, feats = _videos(lengths, dev, seed=50)
    feats = [{"vggish": f["vggish"]} for f in feats]
    batch = windowing.infer_videos(m, vids, feats)
    agree, n = 0, 0
    for v, f, got in zip(vids, feats, batch):
        T = v.shape[0]
        alone = windowing.infer_video(m, v, dict(f))
        assert got.shape == (T, 7) and (alone - got).abs().max().item() <= 1e-4 * max(1.0, alone.abs().max().item()), T
        if T == 1:
            continue                      # the reference layout cannot carry T = 1: _backbones squeezes dim 1 (model.py)
        want = m({"video": windowing.preprocess_frames(m, v)[None], "vggish": f["vggish"][None]})[0]
        scale = max(1.0, want.abs().max().item())
        assert (got - want).abs().max().item() <= 1e-4 * scale, (T, (got - want).abs().max().item())
        agree += (got.argmax(-1) == want.argmax(-1)).sum().item()
        n += T
    assert agree / n >= 0.995, agree / n


@pytest.mark.parametrize("name", ["JMT", "MT"])
def test_jmt_whole_video_against_oracle(name):
    """One 700-frame video, longer than a window, as one sequence: the TCN + fusion head against the CPU oracle's
    jmt_fuse on the same embeddings (the oracle is pinned to the reference's goldens by heads_t300.pt; IR-50 is
    checked against it elsewhere) with BASELINE.json's bars."""
    dev = _dev()
    m = _jmt(name, dev, seed=0)
    T = 700
    frames = synthetic.frames(T, seed=77).to(dev)
    vgg = torch.randn(T, 128, generator=torch.Generator().manual_seed(78)).to(dev)
    got = windowing.infer_video(m, frames, {"vggish": vgg}).cpu()
    emb = m.spatial["visual"](frames)
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    x = {}
    for k, f in (("video", emb), ("vggish", vgg)):
        h = O.tcn_forward(sd, f"temporal.{k}.", f.double().cpu().t()[None], O._tcn_levels(sd, f"temporal.{k}."))
        x[k] = O._bn_eval(sd, f"bn.{k}", h)
    want = O.jmt_fuse(sd, x, name)[0].float()
    assert got.shape == want.shape == (T, 7)
    err = (got - want).abs().max().item()
    agree = (got.argmax(-1) == want.argmax(-1)).float().mean().item()
    print(f"{name} T={T}: max-abs {err:.3g}, argmax agreement {agree:.4f}")
    assert err <= 2e-2 * max(1.0, want.abs().max().item()) and agree >= 0.995, (err, agree)
