"""JMT / MT on live streams (streaming.StreamSession with max_frames): cer_stream_append against a torch reference, and
whole-stream logits from peek / close that equal windowing.infer_video on the same frames bit for bit (one IR-50 plan
for every pass size, CER_RASTER=0), whatever the push composition, plus the refusal and repacking rules."""
import warnings

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, streaming, synthetic, windowing

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
CHUNKS = (1, 7, 30)


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _jmt(name, dev, seed=0, task="CLASSIFICATION"):
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    mods = ["video", "vggish"]
    m = JMT(task=task, modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
            root_dir="", device=dev, model_name=name, visual_state_dict=synthetic.visual_backbone_state_dict(seed))
    m.load_state_dict(synthetic.jmt_state_dict(seed, mods, model_name=name), strict=True)
    return m.to(dev).eval()


def _streams(lengths, dev, seed, pixels):
    """Per stream {'video': uint8 256x256 crops or fp32 [T, 3, 40, 40] pixels, 'vggish': [T, 128]}."""
    n = sum(lengths) + 11 * len(lengths)
    if pixels == "u8":
        video = synthetic.raw_frames_u8(64, seed=seed).repeat(n // 64 + 1, 1, 1, 1).to(dev)
    else:
        video = synthetic.frames(n, seed=seed).to(dev)
    g = torch.Generator().manual_seed(seed + 1)
    out, off = [], 0
    for t in lengths:
        out.append({"video": video[off:off + t], "vggish": torch.randn(t, 128, generator=g).to(dev)})
        off += t + 11
    return out


def _push(sess, sids, inputs, c):
    x = {k: torch.stack([x[k][sess.length(s):sess.length(s) + c] for s, x in zip(sids, inputs)]) for k in inputs[0]}
    logits, fin = sess.push(sids, x)
    assert logits.shape == (len(sids), 0, sess.n_out) and fin == [0] * len(sids)


def _infer(m, x, T=None):
    T = x["video"].shape[0] if T is None else T
    return windowing.infer_video(m, x["video"][:T], {"vggish": x["vggish"][:T]})


@pytest.mark.parametrize("dim", [32, 64, 128, 256])
def test_append_kernel_against_torch(dim):
    """Random tables (distinct sids, ragged t_now, inactive entries, one entry whose chunk runs past max_frames) into a
    sentinel-filled history: exactly the rows [t_now, t_now + chunk) of each active entry's sid change."""
    dev = _dev()
    g = torch.Generator().manual_seed(dim)
    S, F, fields = 13, 97, len(_capi.STREAM_ENTRY_FIELDS)
    for chunk, ne in ((1, 1), (7, 5), (30, 9), (30, 13)):
        tab = torch.zeros(ne, fields, dtype=torch.int32)
        tab[:, 0] = torch.randperm(S, generator=g)[:ne].int()
        tab[:, 4] = torch.randint(0, F - chunk + 1, (ne,), generator=g).int()
        tab[:, 5] = torch.randint(0, 2, (ne,), generator=g).int()
        tab[:, 6] = 1
        if ne > 2:
            tab[1, 6] = 0                                          # padding entry: writes nothing
            tab[2, 4] = F - chunk // 2                             # rows past max_frames are dropped
        src = torch.randn(ne, chunk, dim, generator=g)
        hist = torch.full((S, F, dim), -7.25)
        want = hist.clone()
        for e in range(ne):
            sid, t0, active = int(tab[e, 0]), int(tab[e, 4]), int(tab[e, 6])
            if active:
                r = min(chunk, F - t0)
                want[sid, t0:t0 + r] = src[e, :r]
        hd, sd, td = hist.to(dev), src.to(dev), tab.to(dev)
        _capi.check(_capi.lib().cer_stream_append(td.data_ptr(), ne, chunk, sd.data_ptr(), dim, S, F, hd.data_ptr(),
                                                  _capi.current_stream_ptr()), "cer_stream_append")
        assert torch.equal(hd.cpu(), want), (dim, chunk, ne)
    bad = _capi.lib().cer_stream_append(td.data_ptr(), ne, 0, sd.data_ptr(), dim, S, F, hd.data_ptr(),
                                        _capi.current_stream_ptr())
    assert bad < 0


LENGTHS = [1, 29, 331, 7, 30, 31, 64, 200, 45, 13, 90]          # 331 > 10 x max_chunk


def _drive(sess, inputs, watch):
    """Stream i opens at step 2 i once a slot is free; its k-th push carries CHUNKS[(i + k) % 3] frames (the last one
    ragged), and streams with i % 4 == 1 skip every other step.  Each step groups the pushing streams by chunk size,
    one push per group.  Every third step peeks all open streams at once and each alone; stream ``watch`` is also
    peeked alone after its pushes 3, 7 and 11.  Returns close's logits per stream, the sids in open order, the
    (all-streams, alone) peek pairs and the watched peeks as (length, logits)."""
    sids, pushes, done, res, used, pairs, watched, step = {}, {}, set(), {}, [], [], [], 0
    while len(done) < len(LENGTHS):
        for i in range(len(LENGTHS)):
            if 2 * i <= step and i not in sids and len(sids) - len(done) < sess.max_streams:
                sids[i], pushes[i] = sess.open(), 0
                used.append(sids[i])
        groups = {}
        for i, sid in sids.items():
            if i in done or (i % 4 == 1 and step % 2):
                continue
            c = min(CHUNKS[(i + pushes[i]) % 3], LENGTHS[i] - sess.length(sid))
            groups.setdefault(c, []).append(i)
        for c, idx in groups.items():
            _push(sess, [sids[i] for i in idx], [inputs[i] for i in idx], c)
            for i in idx:
                pushes[i] += 1
                if i == watch and pushes[i] in (3, 7, 11):
                    watched.append((sess.length(sids[i]), sess.peek([sids[i]])[0]))
                if sess.length(sids[i]) == LENGTHS[i]:
                    res[i] = sess.close(sids[i])
                    done.add(i)
        if step % 3 == 2:
            live = [i for i in sids if i not in done]
            for i, p in zip(live, sess.peek([sids[i] for i in live])):
                assert p.shape == (sess.length(sids[i]), 7)
                pairs.append((p, sess.peek([sids[i]])[0]))
        step += 1
    return [res[i] for i in range(len(LENGTHS))], used, pairs, watched


@pytest.mark.parametrize("name,pixels", [("JMT", "u8"), ("MT", "f32")])
def test_streams_equal_infer_video(name, pixels, monkeypatch):
    dev = _dev()
    monkeypatch.setenv("CER_RASTER", "0")
    m = _jmt(name, dev, seed=3)
    inputs = _streams(LENGTHS, dev, seed=60, pixels=pixels)
    sess = streaming.StreamSession(m, max_streams=6, max_chunk=30, max_frames=max(LENGTHS))
    assert sess.n_slots == 1 and sess.n_out == 7
    watch = LENGTHS.index(331)
    res, used, pairs, watched = _drive(sess, inputs, watch)
    assert len(set(used)) < len(used)                                      # a slot was reused after close
    for got, x, T in zip(res, inputs, LENGTHS):
        want = _infer(m, x)
        assert got.shape == (T, 7) and torch.equal(got, want), (name, T, (got - want).abs().max().item())
    assert [L for L, _ in watched] == [sum(CHUNKS[(watch + k) % 3] for k in range(p)) for p in (3, 7, 11)]
    for L, p in watched:
        want = _infer(m, inputs[watch], L)
        assert torch.equal(p, want), (name, L, (p - want).abs().max().item())
    agree = n = 0
    for together, alone in pairs:
        if alone.shape[0] == 0:
            assert together.shape == (0, 7)
            continue
        scale = max(1.0, alone.abs().max().item())
        assert (together - alone).abs().max().item() <= 1e-4 * scale
        agree += (together.argmax(-1) == alone.argmax(-1)).sum().item()
        n += alone.shape[0]
    assert n > 500 and agree / n >= 0.995, (n, agree / n)


def test_regression_and_graph_switch(monkeypatch):
    dev = _dev()
    monkeypatch.setenv("CER_RASTER", "0")
    m = _jmt("JMT", dev, seed=4, task="REGRESSION")
    x = _streams([95], dev, seed=70, pixels="f32")[0]
    want = _infer(m, x)
    assert want.abs().max().item() <= 1.0

    def run():
        sess = streaming.StreamSession(m, max_streams=2, max_chunk=30, max_frames=95)
        sid, k = sess.open(), 0
        while sess.length(sid) < 95:                     # 30, 7, 30, 7, 21: the (1, 30) and (1, 7) graphs replay
            _push(sess, [sid], [x], min((30, 7)[k % 2], 95 - sess.length(sid)))
            k += 1
        return sess.close(sid)

    graphed = run()
    monkeypatch.setenv("CER_HEAD_GRAPH", "0")
    eager = run()
    assert torch.equal(graphed, want) and torch.equal(eager, want)


def test_refusals():
    dev = _dev()
    m = _jmt("MT", dev, seed=5)
    x = _streams([60, 60], dev, seed=80, pixels="f32")
    with pytest.raises(ValueError, match="'logmel'"):
        streaming.StreamSession(m, max_frames=100, wave_fps=30.0)
    sess = streaming.StreamSession(m, max_streams=3, max_chunk=30, max_frames=40)
    a, b = sess.open(), sess.open()
    assert [t.shape for t in sess.peek([a, b])] == [(0, 7), (0, 7)]
    _push(sess, [a, b], x, 20)
    _push(sess, [a], x[:1], 15)
    with pytest.raises(ValueError, match=rf"streams \[{a}\].*max_frames = 40"):
        _push(sess, [a, b], x, 10)                                           # only a would overflow
    assert (sess.length(a), sess.length(b)) == (35, 20)
    _push(sess, [a, b], x, 5)
    _push(sess, [b], x[1:], 15)
    with pytest.raises(ValueError, match="max_frames"):
        sess.push([a], {k: v[None, 40:41] for k, v in x[0].items()})
    for sid, xi in zip((a, b), x):
        assert torch.equal(sess.close(sid), _infer(m, xi, 40))
    with pytest.raises(ValueError, match="distinct open streams"):
        sess.peek([a])
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    can = CAN(task="CLASSIFICATION", modalities=["vggish", "bert"], tcn_settings=synthetic.TCN_SETTINGS,
              backbone_settings=BS, output_dim=7, root_dir="", device=dev)
    can.load_state_dict(synthetic.can_state_dict(0, ["vggish", "bert"]), strict=True)
    can_sess = streaming.StreamSession(can.to(dev).eval(), max_streams=1, max_chunk=8)
    with pytest.raises(TypeError, match="peek reads the whole-stream logits of a JMT / MT session"):
        can_sess.peek([can_sess.open()])
    m.train()
    with pytest.raises(RuntimeError, match="model.eval"):
        sess.peek([sess.open()])


def test_repacking_and_state_bytes(monkeypatch):
    """History rows computed before a weight change are kept and fused with the new weights; frames pushed after it
    run the new backbones and TCN.  state_bytes() is the TCN rings plus the history the session allocated."""
    dev = _dev()
    monkeypatch.setenv("CER_RASTER", "0")
    m = _jmt("JMT", dev, seed=6)
    x = _streams([50], dev, seed=90, pixels="f32")[0]
    sess = streaming.StreamSession(m, max_streams=3, max_chunk=30, max_frames=60)
    rings = sum(t.numel() for k in sess.modalities for t in sess._rings[k])
    hist = sum(t.numel() for t in sess._hist.values())
    assert sess.state_bytes() * sess.max_streams == 4 * (rings + hist)
    assert sess._hist["video"].shape == (3, 60, 128) and sess._hist["vggish"].shape == (3, 60, 64)
    sid = sess.open()
    _push(sess, [sid], [x], 30)
    _push(sess, [sid], [x], 20)
    old = sess.peek([sid])[0]
    assert torch.equal(old, _infer(m, x))
    tcn = m._engines()[0]
    z = {"video": tcn["video"].forward(m.spatial["visual"](x["video"])[None])[0],
         "vggish": tcn["vggish"].forward(x["vggish"][None].contiguous())[0]}
    m.load_state_dict(synthetic.jmt_state_dict(9, ["video", "vggish"], model_name="JMT"), strict=True)
    new = sess.peek([sid])[0]
    assert not torch.equal(new, old)
    assert torch.equal(new, m._fuse_videos(z, [50]))
    sid2 = sess.open()
    _push(sess, [sid2], [x], 30)
    _push(sess, [sid2], [x], 20)
    assert torch.equal(sess.close(sid2), _infer(m, x))
    assert torch.equal(sess.close(sid), new)
