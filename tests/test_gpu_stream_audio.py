"""streaming.StreamSession with wave_fps on the device: the incremental log-mel rows equal the offline front end bit for
bit, the session's examples equal windowing.wave_to_examples, and provisional + close logits equal windowed inference
on the same embeddings."""
import warnings

import numpy as np
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, streaming, synthetic, windowing
from feature_vs_text_compound_emotion_b200.engine import LogMelEngine
from feature_vs_text_compound_emotion_b200.packing import LOGMEL
from tests.test_gpu_streaming import _dev, _feats, _lfan, _offline

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")


def test_stream_logmel_rows_equal_the_offline_front_end():
    """Five streams, every call carrying ragged pieces of all of them (1 sample, odd sizes, more rows than the ring):
    each ring row equals cer_logmel_forward on the whole wave."""
    dev = _dev()
    eng = LogMelEngine(dev)
    rng = np.random.default_rng(5)
    n, R, tail = 5, 128, LOGMEL["win"] - 1
    waves = [torch.from_numpy(rng.standard_normal(int(s)).astype(np.float32) * 0.2).to(dev)
             for s in (31_000, 47_123, 80_000, 12_345, 64_001)]
    ref = [eng.log_mel(w) for w in waves]
    tails = torch.zeros(n, tail, device=dev)
    ring = torch.full((n, R, 64), float("nan"), device=dev)
    tables = eng._tables
    sizes = [1, 1, 533, 534, 7919, 30_000, 1, 399, 400, 160, 161, 20_000]
    pos, call = [0] * n, 0
    dtype = np.dtype(list(_capi.STREAM_AUDIO_ENTRY_FIELDS))
    while any(p < w.numel() for p, w in zip(pos, waves)):
        work, off = [], 0
        for i, w in enumerate(waves):
            k = min(sizes[(call + 3 * i) % len(sizes)], w.numel() - pos[i])
            if k > 0:
                work.append((i, pos[i], w[pos[i]:pos[i] + k]))
        tab = np.zeros(len(work), dtype=dtype)
        for j, (i, a0, piece) in enumerate(work):
            r0, r1 = streaming.logmel_rows(a0), streaming.logmel_rows(a0 + piece.numel())
            tab[j] = (i, r0, r1 - r0, 0, a0, off, piece.numel())
            off += piece.numel()
        samples = torch.cat([p for _, _, p in work])
        tdev = torch.from_numpy(tab.view(np.uint8).copy()).to(dev)
        _capi.check(_capi.lib().cer_stream_logmel(tdev.data_ptr(), len(work), int(tab["n_rows"].max()), samples.data_ptr(),
                                                  tables.data_ptr(), 400, 160, 512, 64, LOGMEL["log_offset"],
                                                  tails.data_ptr(), tail, ring.data_ptr(), R,
                                                  torch.cuda.current_stream().cuda_stream), "cer_stream_logmel")
        for i, a0, piece in work:
            pos[i] += piece.numel()
            done = streaming.logmel_rows(pos[i])
            rows = torch.arange(max(0, done - R), done, device=dev)
            assert torch.equal(ring[i][rows % R], ref[i][rows]), (call, i)
        call += 1
    assert call > 10


def _run(sess, plan, inputs, fps, audio, owner, visual_out=None):
    """plan: per stream (T, chunk, step it opens at); audio(i, T_after_push) -> samples delivered so far; owner: sid ->
    the stream open on it.  Returns per stream (provisional, provisional + close) logits and the sids in open order;
    checks emitted and final_upto on every push."""
    sids, prov, done, A, step, used = {}, {}, {}, {}, 0, []
    W = sess.W
    while len(done) < len(plan):
        for i, (T, c, at) in enumerate(plan):
            if at <= step and i not in sids:
                sids[i], prov[i], A[i] = sess.open(), [], 0
                owner[sids[i]] = i
                used.append(sids[i])
        groups = {}
        for i, sid in sids.items():
            if i not in done:
                groups.setdefault(min(plan[i][1], plan[i][0] - sess.length(sid)), []).append(i)
        for c, idx in groups.items():
            ids = [sids[i] for i in idx]
            x = {k: torch.stack([inputs[i][k][sess.length(sids[i]):sess.length(sids[i]) + c] for i in idx])
                 for k in inputs[idx[0]] if k != "wave" and not k.startswith("_")}
            waves = []
            for i in idx:
                a1 = audio(i, sess.length(sids[i]) + c)
                waves.append(inputs[i]["wave"][A[i]:a1])
                A[i] = a1
            out, fin = sess.push(ids, {**x, "wave": waves})
            if visual_out is not None:
                emb = visual_out.pop().view(len(idx), c, -1)
                for j, i in enumerate(idx):
                    inputs[i].setdefault("_vis", []).append(emb[j])
            for j, i in enumerate(idx):
                prov[i].append(out[j])
                assert sum(p.shape[0] for p in prov[i]) == sess.emitted(sids[i])
                assert fin[j] == max(0, sess.emitted(sids[i]) - W)
                if sess.length(sids[i]) == plan[i][0]:
                    done[i] = sess.close(sids[i])
        step += 1
    res = []
    for i, (T, _, _) in enumerate(plan):
        p = torch.cat(prov[i])
        assert done[i].shape[0] == min(T, W)
        res.append((p, torch.cat([p[:T - min(T, W)], done[i]])))
    return res, used


def _hooks(sess):
    """Records every VGGish pass of the session: its layout [(stream, first frame, count)] and its examples."""
    passes, owner = [], {}
    sess.example_hook = lambda layout, ex: passes.append(([(owner[sid], e0, r) for sid, e0, r in layout], ex.clone()))
    return passes, owner


@pytest.mark.parametrize("fps", [30, 25])
def test_session_examples_equal_wave_to_examples(fps):
    dev = _dev()
    mods = ["cnn_res50", "logmel", "bert"]
    m = _lfan(mods, dev, seed=11)
    Ts = [1, 17, 29, 30, 31, 299, 300, 777]
    plan, inputs, totals = [], [], []
    for k, kind in enumerate(("short", "equal", "long")):
        for j, T in enumerate(Ts):
            syn = streaming.synced_samples(T, fps)
            total = {"short": max(1, syn - streaming.synced_samples(min(T, 20), fps)), "equal": syn,
                     "long": syn + 8000}[kind]
            g = torch.Generator().manual_seed(1000 * k + j)
            x = _feats(["cnn_res50", "bert"], T, 7 * k + j, dev)
            x["wave"] = (torch.randn(total, generator=g) * 0.3).to(dev)
            plan.append((T, 30, j))
            inputs.append(x)
            totals.append(total)
    sess = streaming.StreamSession(m, max_streams=len(plan), max_chunk=30, wave_fps=fps)
    passes, owner = _hooks(sess)

    def audio(i, t):
        T = plan[i][0]
        return totals[i] if t == T else min(totals[i], streaming.synced_samples(t, fps))
    _run(sess, plan, inputs, fps, audio, owner)
    got = {}
    for layout, ex in passes:
        o = 0
        for i, e0, r in layout:
            got.setdefault(i, {}).update({e0 + k: ex[o + k] for k in range(r)})
            o += r
    for i, (T, _, _) in enumerate(plan):
        want = windowing.wave_to_examples(m, inputs[i]["wave"], T, fps)
        have = torch.stack([got[i][t] for t in range(T)])
        assert torch.equal(have, want), (plan[i], totals[i])


@pytest.mark.parametrize("mods", [["cnn_res50", "logmel", "bert"], ["video", "logmel", "bert"]])
def test_wave_streams_equal_windowed_inference(mods):
    dev = _dev()
    fps = 30.0
    m = _lfan(mods, dev, seed=12)
    lengths = [1, 17, 199, 300, 301, 500, 777, 1234]
    chunks = [1, 8, 1, 30, 8, 30, 8, 30]
    plan = [(T, c, 3 * i) for i, (T, c) in enumerate(zip(lengths, chunks))]
    inputs, totals = [], []
    for i, T in enumerate(lengths):
        syn = streaming.synced_samples(T, fps)
        total = syn + (8000 if i == 6 else -streaming.synced_samples(10, fps) if i == 7 else 0)
        g = torch.Generator().manual_seed(500 + i)
        x = _feats([k for k in mods if k not in ("video", "logmel")], T, 60 + i, dev)
        if "video" in mods:
            x["video"] = synthetic.raw_frames_u8(T, seed=70 + i).to(dev)
        x["wave"] = (torch.randn(max(total, 1), generator=g) * 0.3).to(dev)
        inputs.append(x)
        totals.append(max(total, 1))

    def audio(i, t):                       # odd streams' audio one push behind the video; the rest in step
        T, c, _ = plan[i]
        if t == T:
            return totals[i]
        return min(totals[i], streaming.synced_samples(max(0, t - c) if i % 2 else t, fps))
    sess = streaming.StreamSession(m, max_streams=7, max_chunk=30, wave_fps=fps)
    passes, owner = _hooks(sess)
    vis_out = None
    if "video" in mods:
        vis_out, vis = [], m.spatial["visual"]
        vis_fwd = vis.forward
        vis.forward = lambda x, *a, **k: vis_out.append(vis_fwd(x, *a, **k)) or vis_out[-1]
    aud = m.spatial["audio"]
    aud_fwd, aud_sizes = aud.forward, []
    aud.forward = lambda x, *a, **k: aud_sizes.append(x.shape[0]) or aud_fwd(x, *a, **k)
    try:
        res, used = _run(sess, plan, inputs, fps, audio, owner, vis_out)
    finally:
        del aud.forward
        if vis_out is not None:
            del m.spatial["visual"].forward
    assert [sum(r for _, _, r in layout) for layout, _ in passes] == aud_sizes
    assert len(set(used)) < len(used)                                 # a slot was reused
    # the session's examples are the offline ones; VGGish on them at the session's pass sizes
    offline_ex = [windowing.wave_to_examples(m, x["wave"][:totals[i]], lengths[i], fps) for i, x in enumerate(inputs)]
    emb = [torch.empty(T, 128, device=dev) for T in lengths]
    for layout, ex in passes:
        batch = torch.cat([offline_ex[i][e0:e0 + r] for i, e0, r in layout])
        assert torch.equal(batch, ex)
        e, o = m.spatial["audio"](batch), 0
        for i, e0, r in layout:
            emb[i][e0:e0 + r] = e[o:o + r]
            o += r
    for i, ((p, got), T) in enumerate(zip(res, lengths)):
        feats = {k: v for k, v in inputs[i].items() if k in mods and k != "video"}
        feats["logmel"] = emb[i]
        if "video" in mods:
            feats["video"] = torch.cat(inputs[i]["_vis"])
        want = _offline(m, {k: feats[k] for k in mods})
        assert torch.equal(got, want), (T, (got - want).abs().max().item())
        assert torch.equal(p[:max(0, T - 300)], want[:max(0, T - 300)])
        if "video" in mods:                                           # against infer_video on the whole wave
            off = windowing.infer_video(m, inputs[i]["video"], {"wave": inputs[i]["wave"][:totals[i]],
                                                                "bert": inputs[i]["bert"]}, fps=fps)
            full_a = m.spatial["audio"](offline_ex[i])
            full_v = m.spatial["visual"](windowing.preprocess_frames(m, inputs[i]["video"]))
            if torch.equal(full_a, emb[i]) and torch.equal(full_v, feats["video"]):
                assert torch.equal(got, off)
            cos = torch.nn.functional.cosine_similarity(got, off, dim=1).min().item()
            assert cos >= 0.999 and (got - off).abs().max().item() <= 2e-2
            assert (got.argmax(-1) == off.argmax(-1)).float().mean().item() >= 0.995


def test_wave_refusals():
    dev = _dev()
    mods = ["cnn_res50", "logmel", "bert"]
    m = _lfan(mods, dev, seed=13)
    with pytest.raises(ValueError, match="'logmel' modality and at least one other"):
        streaming.StreamSession(_lfan(["cnn_res50", "bert"], dev), wave_fps=30)
    with pytest.raises(ValueError, match="'logmel' modality and at least one other"):
        streaming.StreamSession(_lfan(["logmel"], dev), wave_fps=30)
    sess = streaming.StreamSession(m, max_streams=2, max_chunk=8, wave_fps=30)
    sid = sess.open()
    x = {k: v[None] for k, v in _feats(["cnn_res50", "bert"], 8, 3, dev).items()}
    ok = torch.zeros(100, device=dev)
    with pytest.raises(ValueError, match="not 'logmel'"):
        sess.push([sid], {**x, "wave": [ok], "logmel": torch.zeros(1, 8, 96, 64, device=dev)})
    for bad in (torch.zeros(2, 50, device=dev), torch.zeros(100, dtype=torch.float64, device=dev), torch.zeros(100)):
        with pytest.raises(ValueError, match="1-D fp32"):
            sess.push([sid], {**x, "wave": [bad]})
    with pytest.raises(ValueError, match="one per stream"):
        sess.push([sid], {**x, "wave": [ok, ok]})
    limit = streaming.synced_samples(8 + sess.lag + 8, 30)
    with pytest.raises(ValueError, match="run ahead"):
        sess.push([sid], {**x, "wave": [torch.zeros(limit + 1, device=dev)]})
    assert sess.length(sid) == 0 and sess.emitted(sid) == 0
    for _ in range(5):                                                # 40 frames, no audio: all held back
        out, fin = sess.push([sid], {**x, "wave": [torch.zeros(0, device=dev)]})
        assert out[0].shape == (0, sess.n_out) and fin == [0]
    with pytest.raises(ValueError, match="may wait for their audio"):
        sess.push([sid], {**x, "wave": [torch.zeros(0, device=dev)]})
    assert sess.length(sid) == 40 and sess.emitted(sid) == 0
    with pytest.raises(ValueError, match="received no audio"):
        sess.close(sid)
    sess.push([sid], {k: v[:, :1] for k, v in x.items()} | {"wave": [torch.ones(streaming.synced_samples(41, 30),
                                                                                 device=dev)]})
    assert sess.emitted(sid) == 41 - sess.lag
    assert sess.close(sid).shape == (41, sess.n_out)
    assert sess.state_bytes() > streaming.StreamSession(m, max_streams=1, max_chunk=8).state_bytes()
