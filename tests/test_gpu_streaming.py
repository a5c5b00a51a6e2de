"""streaming.StreamSession on the device: provisional logits of frames below T - min(T, W) followed by close's
result equal windowed inference bit for bit (the TCN and fusion kernels are the offline ones, fed identical rows)."""
import warnings
from contextlib import contextmanager

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, streaming, synthetic, windowing
from feature_vs_text_compound_emotion_b200.engine import stitch_windows

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _lfan(mods, dev, seed=0, task="CLASSIFICATION", num_heads=2):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings=BS, output_dim=7, task=task, modality=mods, kernel_size=5, example_length=300,
             tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=num_heads, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(seed) if "video" in mods else None,
           audio_state_dict=synthetic.vggish_state_dict(seed) if "logmel" in mods else None)
    m.load_state_dict(synthetic.lfan_state_dict(seed, mods), strict=True)
    return m.to(dev).eval()


def _offline(m, feats, W=300, H=200):
    """windowing.infer_video on pre-extracted features (its own steps: the video argument only feeds IR-50)."""
    T = next(iter(feats.values())).shape[0]
    starts = windowing.window_starts(T, W, H)
    logits = m.forward_features({k: windowing.gather_windows(v, starts, W).contiguous() for k, v in feats.items()})
    st = torch.as_tensor(starts, dtype=torch.int32, device=logits.device)
    return stitch_windows(logits, st, max(T, W))[:T]


TCN_VARIANTS = {"tcn_igemm_kernel<64,8>", "tcn_igemm_kernel<32,8>"}
FUSION_VARIANTS = {f"fusion_head_kernel<{k}>" for k in range(4, 9)}


@contextmanager
def _variants():
    """The TCN and fusion instantiations (cer_head_last_variant) of every host-side launch inside the block.  A CUDA
    graph replay launches nothing from the host, so only a shape's first (eager + capture) call adds names."""
    lib = _capi.lib()
    seen = {"tcn": set(), "fusion": set()}
    orig = {}
    for name, key in (("cer_tcn_block_tc_forward", "tcn"), ("cer_fusion_head_forward", "fusion")):
        orig[name] = fn = getattr(lib, name)

        def wrap(*a, _fn=fn, _key=key):
            r = _fn(*a)
            seen[_key].add(lib.cer_head_last_variant().decode())
            return r
        setattr(lib, name, wrap)
    try:
        yield seen
    finally:
        for name, fn in orig.items():
            setattr(lib, name, fn)


def _pin_variants(m, online, offline):
    """The streaming path runs the TCN instantiations the offline path runs: the N tile follows C_out only.  The
    fusion kFR follows the row count (n * n_slots * c rows against n_windows * W), so it may differ; each row is
    computed the same way for every kFR, which the torch.equal checks confirm."""
    want = {"tcn_igemm_kernel<64,8>" if c % 64 == 0 else "tcn_igemm_kernel<32,8>"
            for mod in m.modality for c in m.tcn_channel[mod]}
    assert online["tcn"] == offline["tcn"] == want, (online, offline)
    assert online["fusion"] and offline["fusion"], (online, offline)
    assert online["fusion"] <= FUSION_VARIANTS and offline["fusion"] <= FUSION_VARIANTS, (online, offline)


def _feats(mods, T, seed, dev):
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k in mods:
        x = torch.randn(T, synthetic.EMBEDDING_DIM[k], generator=g)
        out[k] = (torch.nn.functional.normalize(x, dim=-1) if k == "cnn_res50" else x).to(dev)
    return out


def _stream(sess, plan, inputs, W=300):
    """plan: per stream (length, chunk, step it opens at).  Every step pushes each open stream's next chunk, one
    push per chunk size (a stream's last chunk may be partial).  Returns per stream provisional + close logits and
    checks that frames below final_upto are already final when reported."""
    sids, prov, done, step = {}, {}, {}, 0
    while len(done) < len(plan):
        for i, (T, c, at) in enumerate(plan):
            if at == step and i not in sids:
                sids[i], prov[i] = sess.open(), []
        groups = {}
        for i, sid in sids.items():
            if i in done:
                continue
            t = sess.length(sid)
            groups.setdefault(min(plan[i][1], plan[i][0] - t), []).append(i)
        for c, idx in groups.items():
            ids = [sids[i] for i in idx]
            x = {k: torch.stack([inputs[i][k][sess.length(sids[i]):sess.length(sids[i]) + c] for i in idx])
                 for k in inputs[idx[0]]}
            out, fin = sess.push(ids, x)
            assert out.shape == (len(idx), c, sess.n_out)
            for j, i in enumerate(idx):
                prov[i].append(out[j])
                assert fin[j] == max(0, sess.length(sids[i]) - W)
                if sess.length(sids[i]) == plan[i][0]:
                    done[i] = sess.close(sids[i])
        step += 1
    res = []
    for i, (T, _, _) in enumerate(plan):
        p = torch.cat(prov[i])
        assert p.shape[0] == T and done[i].shape[0] == min(T, W)
        res.append((p, torch.cat([p[:T - min(T, W)], done[i]])))
    return res


def test_many_streams_equal_windowed_inference():
    dev = _dev()
    mods = ["cnn_res50", "vggish", "bert"]
    m = _lfan(mods, dev, seed=1)
    lengths = [1, 199, 200, 299, 300, 301, 499, 500, 501, 777, 1234]
    chunks = [1, 8, 30, 1, 8, 30, 1, 8, 30, 8, 30]
    plan = [(T, c, 3 * i) for i, (T, c) in enumerate(zip(lengths, chunks))]
    inputs = [_feats(mods, T, 100 + i, dev) for i, T in enumerate(lengths)]
    sess = streaming.StreamSession(m, max_streams=16, max_chunk=30)
    assert sess.n_slots == 2 and sess.n_lslots == 3
    with _variants() as online:
        res = _stream(sess, plan, inputs)
    with _variants() as offline:
        wants = [_offline(m, x) for x in inputs]
    _pin_variants(m, online, offline)
    for (p, got), want, T in zip(res, wants, lengths):
        assert torch.equal(got, want), (T, (got - want).abs().max().item())
        assert torch.equal(p[:max(0, T - 300)], want[:max(0, T - 300)])


def test_reused_slot_is_a_fresh_stream():
    dev = _dev()
    mods = ["cnn_res50", "vggish", "bert"]
    m = _lfan(mods, dev, seed=2)
    x = _feats(mods, 437, 7, dev)
    fresh = _stream(streaming.StreamSession(m, max_streams=1, max_chunk=30), [(437, 30, 0)], [x])[0]
    sess = streaming.StreamSession(m, max_streams=1, max_chunk=30)
    _stream(sess, [(613, 8, 0)], [_feats(mods, 613, 8, dev)])
    again = _stream(sess, [(437, 30, 0)], [x])[0]
    assert torch.equal(fresh[1], again[1]) and torch.equal(fresh[0], again[0])
    assert torch.equal(fresh[1], _offline(m, x))


@pytest.mark.parametrize("mods", [["mfcc", "egemaps", "bert"], ["bert", "mfcc"]])
def test_padded_channel_modalities(mods):
    dev = _dev()
    m = _lfan(mods, dev, seed=3)
    lengths = [123, 350, 640]
    inputs = [_feats(mods, T, 30 + T, dev) for T in lengths]
    sess = streaming.StreamSession(m, max_streams=4, max_chunk=16)
    with _variants() as online:
        res = _stream(sess, [(T, 16, i) for i, T in enumerate(lengths)], inputs)
    with _variants() as offline:
        wants = [_offline(m, x) for x in inputs]
    _pin_variants(m, online, offline)
    for (_, got), want in zip(res, wants):
        assert torch.equal(got, want)


def test_two_modalities_four_heads_regression_and_other_window():
    dev = _dev()
    mods = ["cnn_res50", "vggish"]
    m = _lfan(mods, dev, seed=4, task="REGRESSION", num_heads=4)
    lengths = [90, 260, 333]
    inputs = [_feats(mods, T, 40 + T, dev) for T in lengths]
    for W, H, c in ((300, 200, 30), (100, 50, 7)):
        sess = streaming.StreamSession(m, max_streams=3, max_chunk=c, window_length=W, hop_length=H)
        with _variants() as online:
            res = _stream(sess, [(T, c, 2 * i) for i, T in enumerate(lengths)], inputs, W=W)
        with _variants() as offline:
            wants = [_offline(m, x, W, H) for x in inputs]
        _pin_variants(m, online, offline)
        for (_, got), want in zip(res, wants):
            assert torch.equal(got, want)


def test_chunks_longer_than_the_window():
    """A chunk of more frames than the window (W / H = 100 / 50, 128 frames per push): the input ring keeps the
    chunk's last W rows, so close rebuilds the tail window from the right frames."""
    dev = _dev()
    mods = ["cnn_res50", "vggish"]
    m = _lfan(mods, dev, seed=7)
    lengths = [90, 128, 300, 333, 517]
    inputs = [_feats(mods, T, 70 + T, dev) for T in lengths]
    sess = streaming.StreamSession(m, max_streams=5, max_chunk=128, window_length=100, hop_length=50)
    assert sess.n_slots == 5
    res = _stream(sess, [(T, 128, i) for i, T in enumerate(lengths)], inputs, W=100)
    for (_, got), x, T in zip(res, inputs, lengths):
        want = _offline(m, x, 100, 50)
        assert torch.equal(got, want), (T, (got - want).abs().max().item())


def test_pixels_and_logmel_bit_equal_at_the_offline_pass_size():
    """'video' (stored uint8 crops) and 'logmel' (examples) run IR-50 / VGGish on the n * c chunk frames of a push.
    Three 330-frame streams pushed 110 frames at a time give 330-frame backbone passes, the pass infer_video runs per
    video, so the plans pick the same kernels and the result is infer_video's, bit for bit."""
    dev = _dev()
    mods = ["video", "logmel", "bert"]
    m = _lfan(mods, dev, seed=6)
    T, c, n = 330, 110, 3
    inputs = [{"video": synthetic.raw_frames_u8(T, seed=61 + i).to(dev),
               "logmel": synthetic.logmel_patches(T, seed=62 + i).to(dev),
               "bert": torch.randn(T, 768, generator=torch.Generator().manual_seed(63 + i)).to(dev)} for i in range(n)]
    with _variants() as offline:
        wants = [windowing.infer_video(m, x["video"], {"logmel": x["logmel"], "bert": x["bert"]}) for x in inputs]
    sess = streaming.StreamSession(m, max_streams=n, max_chunk=c)
    with _variants() as online:
        res = _stream(sess, [(T, c, 0)] * n, inputs)
    _pin_variants(m, online, offline)
    for (_, got), want in zip(res, wants):
        assert torch.equal(got, want), (got - want).abs().max().item()


def test_pixels_and_logmel_at_a_smaller_pass_size():
    """One stream pushed 30 frames at a time: IR-50 / VGGish passes of 30 frames against infer_video's 330.  The
    embeddings are compared directly: where they are equal the logits must be too, otherwise (a plan that picks
    another kernel for the smaller pass, e.g. IR-50 stage 2 below 190 frames) BASELINE's tolerances hold."""
    dev = _dev()
    mods = ["video", "logmel", "bert"]
    m = _lfan(mods, dev, seed=6)
    T, c = 330, 30
    raw = synthetic.raw_frames_u8(T, seed=61).to(dev)
    lm = synthetic.logmel_patches(T, seed=62).to(dev)
    bert = torch.randn(T, 768, generator=torch.Generator().manual_seed(63)).to(dev)
    want = windowing.infer_video(m, raw, {"logmel": lm, "bert": bert})
    sess = streaming.StreamSession(m, max_streams=1, max_chunk=c)
    got = _stream(sess, [(T, c, 0)], [{"video": raw, "logmel": lm, "bert": bert}])[0][1]
    frames = windowing.preprocess_frames(m, raw)
    emb_equal = (torch.equal(torch.cat([m.spatial["visual"](frames[a:a + c]) for a in range(0, T, c)]),
                             m.spatial["visual"](frames))
                 and torch.equal(torch.cat([m.spatial["audio"](lm[a:a + c]) for a in range(0, T, c)]),
                                 m.spatial["audio"](lm)))
    ir = m.spatial["visual"].backbone.engine()
    same_plan = all(ir.op_variant(i, c) == ir.op_variant(i, T) for i in range(ir.n_conv_ops))
    print(f"IR-50 plan equal at {c} and {T} frames: {same_plan}; embeddings equal: {emb_equal}")
    if emb_equal:
        assert torch.equal(got, want)
    cos = torch.nn.functional.cosine_similarity(got, want, dim=1).min().item()
    assert cos >= 0.999 and (got - want).abs().max().item() <= 2e-2
    assert (got.argmax(-1) == want.argmax(-1)).float().mean().item() >= 0.995


def test_refused_inputs():
    dev = _dev()
    mods = ["cnn_res50", "vggish"]
    m = _lfan(mods, dev, seed=5)
    sess = streaming.StreamSession(m, max_streams=1, max_chunk=8)
    sid = sess.open()
    with pytest.raises(RuntimeError, match="stream slots are open"):
        sess.open()
    x = _feats(mods, 8, 1, dev)
    with pytest.raises(ValueError, match="'wave' cannot be streamed"):
        sess.push([sid], {"wave": torch.zeros(16000, device=dev), **{k: v[None] for k, v in x.items()}})
    with pytest.raises(ValueError, match="chunk of 16 frames"):
        sess.push([sid], {k: torch.cat([v, v])[None] for k, v in x.items()})
    with pytest.raises(ValueError, match="distinct open streams"):
        sess.push([sid + 1], {k: v[None] for k, v in x.items()})
    m.train()
    with pytest.raises(RuntimeError, match="model.eval"):
        sess.push([sid], {k: v[None] for k, v in x.items()})
    with pytest.raises(RuntimeError, match="model.eval"):
        streaming.StreamSession(m)
    m.eval()
    assert sess.length(sid) == 0
    with pytest.raises(ValueError, match="hop_length"):
        streaming.StreamSession(m, window_length=100, hop_length=200)
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    with pytest.raises(TypeError, match="JMT / MT attend over the whole window"):
        streaming.StreamSession(JMT.__new__(JMT))
