"""CAN on the device: the row-invariant fusion head + tail kernel (cer_can_head_forward) against an fp64 reference and
against offline CAN, and streaming.StreamSession with a CAN: final per-frame logits that equal the kernel on the
offline TCN output of the whole stream, bit for bit, whatever the other streams and chunk sizes."""
import warnings

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, streaming, synthetic, windowing
from oracle import lfan_oracle as O

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
FEATS = ["cnn_res50", "vggish", "bert"]


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _can(mods, dev, seed=0, task="CLASSIFICATION"):
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    m = CAN(task=task, modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
            root_dir="", device=dev,
            visual_state_dict=synthetic.visual_backbone_state_dict(seed) if "video" in mods else None,
            audio_state_dict=synthetic.vggish_state_dict(seed) if "logmel" in mods else None)
    m.load_state_dict(synthetic.can_state_dict(seed, mods), strict=True)
    return m.to(dev).eval()


def _feats(mods, T, seed, dev):
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(T, synthetic.EMBEDDING_DIM[k], generator=g).to(dev) for k in mods}


def _kernel_on_tcn(m, feats):
    """The head kernel on the offline TcnEngine output of a whole stream: feats[k] [T, D_k] -> [T, n_out]."""
    tcn = m._engines()[0]
    z = [tcn[k].forward(feats[k][None].contiguous())[0] for k in m.modalities]
    return m.frame_head().forward(z, m.task == "REGRESSION")


@pytest.mark.parametrize("task", ["CLASSIFICATION", "REGRESSION"])
@pytest.mark.parametrize("mods", [["bert"], ["vggish", "bert"], FEATS])
def test_kernel_against_fp64(mods, task):
    dev = _dev()
    m = _can(mods, dev, seed=len(mods), task=task)
    head = m.frame_head()
    sd = {k: v.detach().double().cpu() for k, v in m.state_dict().items()}
    dims = [synthetic.TCN_SETTINGS[k]["channel"][-1] for k in mods]
    for rows in (1, 7, 30, 7680):
        g = torch.Generator().manual_seed(rows)
        z = [torch.randn(rows, d, generator=g) for d in dims]
        wide = torch.randn(rows, dims[0] + 5, generator=g)            # modality 0 read through a wider row pitch
        wide[:, :dims[0]] = z[0]
        zd = [wide.to(dev)[:, :dims[0]]] + [t.to(dev) for t in z[1:]]
        got = head.forward(zd, task == "REGRESSION")
        assert _capi.lib().cer_head_last_variant() == b"can_head_kernel"
        ref = O.can_fuse(sd, {k: t.double().t()[None] for k, t in zip(mods, z)}, mods)[0]
        if task == "REGRESSION":
            ref = torch.tanh(ref)
        err = (got.double().cpu() - ref).abs().max().item()
        assert got.shape == (rows, 7) and err <= 1e-5 * max(1.0, ref.abs().max().item()), (rows, err)


def test_rows_do_not_depend_on_the_call():
    """A row alone, inside a batch of 7 and inside 7 680 rows (at every tile position) gives the same bits."""
    dev = _dev()
    m = _can(FEATS, dev, seed=3)
    head = m.frame_head()
    g = torch.Generator().manual_seed(0)
    z = [torch.randn(7680, synthetic.TCN_SETTINGS[k]["channel"][-1], generator=g).to(dev) for k in FEATS]
    big = head.forward(z, False)
    assert torch.equal(head.forward([t[100:107] for t in z], False), big[100:107])
    for r in (0, 31, 32, 103, 7679):
        assert torch.equal(head.forward([t[r:r + 1] for t in z], False), big[r:r + 1]), r
    for shift in (1, 5, 17):
        rolled = head.forward([torch.roll(t, shift, 0) for t in z], False)
        assert torch.equal(rolled, torch.roll(big, shift, 0)), shift


def test_kernel_on_tcn_outputs_matches_offline_can():
    dev = _dev()
    m = _can(FEATS, dev, seed=4)
    feats = _feats(FEATS, 1001, 9, dev)
    want = m.forward_features({k: v[None] for k, v in feats.items()})[0]
    got = _kernel_on_tcn(m, feats)
    err = (got - want).abs().max().item()
    assert err <= 1e-5 * max(1.0, want.abs().max().item()), err
    top = want.topk(2, dim=-1).values
    sure = (top[:, 0] - top[:, 1]) > 1e-4
    assert torch.equal(got.argmax(-1)[sure], want.argmax(-1)[sure])


def _drive(sess, plan, inputs, chunks):
    """plan: per stream (length, step it opens at); a stream's k-th push carries chunks[(i + k) % len(chunks)] frames
    (its last one partial); each step groups the open streams by chunk size, one push per group, and a stream opens
    once a slot is free.  Returns per stream its pushed logits followed by close's, and the sids in open order."""
    sids, got, done, pushes, step, used = {}, {}, set(), {}, 0, []
    while len(done) < len(plan):
        for i, (T, at) in enumerate(plan):
            if at <= step and i not in sids and len(sids) - len(done) < sess.max_streams:
                sids[i], got[i], pushes[i] = sess.open(), [], 0
                used.append(sids[i])
        groups = {}
        for i, sid in sids.items():
            if i not in done:
                c = min(chunks[(i + pushes[i]) % len(chunks)], plan[i][0] - sess.length(sid))
                groups.setdefault(c, []).append(i)
        for c, idx in groups.items():
            ids = [sids[i] for i in idx]
            x = {k: torch.stack([inputs[i][k][sess.length(sids[i]):sess.length(sids[i]) + c] for i in idx])
                 for k in inputs[idx[0]]}
            out, fin = sess.push(ids, x)
            assert out.shape == (len(idx), c, sess.n_out)
            for j, i in enumerate(idx):
                got[i].append(out[j])
                pushes[i] += 1
                assert fin[j] == sess.length(sids[i]) == sess.emitted(sids[i])
                if sess.length(sids[i]) == plan[i][0]:
                    tail = sess.close(sids[i])
                    assert tail.shape == (0, sess.n_out)
                    got[i].append(tail)
                    done.add(i)
        step += 1
    return [torch.cat(got[i]) for i in range(len(plan))], used


def test_streams_equal_the_kernel_on_offline_tcn_outputs():
    dev = _dev()
    m = _can(FEATS, dev, seed=5)
    lengths = [1, 29, 300, 1001, 7, 30, 31, 64, 200, 450, 613]
    inputs = [_feats(FEATS, T, 200 + i, dev) for i, T in enumerate(lengths)]
    sess = streaming.StreamSession(m, max_streams=6, max_chunk=30)
    assert sess.n_slots == 1
    res, used = _drive(sess, [(T, 2 * i) for i, T in enumerate(lengths)], inputs, (1, 7, 30))
    assert len(set(used)) < len(used)                                 # a slot was reused
    for got, x, T in zip(res, inputs, lengths):
        want = _kernel_on_tcn(m, x)
        assert got.shape == (T, 7) and torch.equal(got, want), (T, (got - want).abs().max().item())
    alone = streaming.StreamSession(m, max_streams=1, max_chunk=13)
    for i in (1, 3, 10):
        again = _drive(alone, [(lengths[i], 0)], [inputs[i]], (13, 2))[0][0]
        assert torch.equal(again, res[i]), lengths[i]
    blocks = sess._blocks
    assert sess.state_bytes() == 4 * sum(2 * 2 * (b.kernel_size - 1) * b.dilation * b.c_in
                                         for k in FEATS for b in blocks[k])


def test_regression_stream_and_graph_switch(monkeypatch):
    dev = _dev()
    m = _can(["vggish", "bert"], dev, seed=6, task="REGRESSION")
    x = _feats(["vggish", "bert"], 95, 1, dev)
    want = _kernel_on_tcn(m, x)
    assert want.abs().max().item() <= 1.0
    graphed = _drive(streaming.StreamSession(m, max_streams=2, max_chunk=30), [(95, 0)], [x], (30, 7))[0][0]
    monkeypatch.setenv("CER_HEAD_GRAPH", "0")
    eager = _drive(streaming.StreamSession(m, max_streams=2, max_chunk=30), [(95, 0)], [x], (30, 7))[0][0]
    assert torch.equal(graphed, want) and torch.equal(eager, want)


def test_pixels_and_wave():
    """uint8 crops + raw audio: after close every frame's logit was returned exactly once; equal bit for bit to the
    kernel on the TCN output of the embeddings the session computed, and close to CAN.forward_features on the
    whole-video embeddings (backbone passes of other sizes)."""
    dev = _dev()
    fps = 30.0
    mods = ["video", "logmel", "bert"]
    m = _can(mods, dev, seed=7)
    T, c, n = 330, 110, 3
    inputs = []
    for i in range(n):
        total = streaming.synced_samples(T, fps) - (4000 if i == 1 else 0)
        inputs.append({"video": synthetic.raw_frames_u8(T, seed=71 + i).to(dev),
                       "bert": torch.randn(T, 768, generator=torch.Generator().manual_seed(72 + i)).to(dev),
                       "wave": (torch.randn(total, generator=torch.Generator().manual_seed(73 + i)) * 0.3).to(dev)})
    sess = streaming.StreamSession(m, max_streams=n, max_chunk=c, wave_fps=fps)
    passes = []
    sess.example_hook = lambda layout, ex: passes.append((list(layout), ex.clone()))
    vis_out, vis = [], m.spatial["visual"]
    vis_fwd = vis.forward
    vis.forward = lambda t, *a, **k: vis_out.append(vis_fwd(t, *a, **k)) or vis_out[-1]
    ids = [sess.open() for _ in range(n)]
    got = {sid: [] for sid in ids}
    try:
        for t0 in range(0, T, c):
            waves = [x["wave"][streaming.synced_samples(t0, fps):streaming.synced_samples(t0 + c, fps)] for x in inputs]
            out, fin = sess.push(ids, {"video": torch.stack([x["video"][t0:t0 + c] for x in inputs]),
                                       "bert": torch.stack([x["bert"][t0:t0 + c] for x in inputs]), "wave": waves})
            for sid, o, f in zip(ids, out, fin):
                got[sid].append(o)
                assert f == sess.emitted(sid)
        for sid in ids:
            got[sid].append(sess.close(sid))
    finally:
        del vis.forward
    vis_emb = torch.cat(vis_out).view(T // c, n, c, -1).permute(1, 0, 2, 3).reshape(n, T, -1)
    aud_emb = torch.empty(n, T, 128, device=dev)
    for layout, ex in passes:
        e, o = m.spatial["audio"](ex), 0
        for sid, e0, r in layout:
            aud_emb[ids.index(sid), e0:e0 + r] = e[o:o + r]
            o += r
    for i, sid in enumerate(ids):
        logits = torch.cat(got[sid])
        assert logits.shape == (T, 7)
        same = _kernel_on_tcn(m, {"video": vis_emb[i], "logmel": aud_emb[i], "bert": inputs[i]["bert"]})
        assert torch.equal(logits, same), (logits - same).abs().max().item()
        frames = windowing.preprocess_frames(m, inputs[i]["video"])
        full = {"video": m.spatial["visual"](frames),
                "logmel": m.spatial["audio"](windowing.wave_to_examples(m, inputs[i]["wave"], T, fps)),
                "bert": inputs[i]["bert"]}
        want = m.forward_features({k: v[None] for k, v in full.items()})[0]
        err = (logits - want).abs().max().item()
        print(f"stream {i}: max |stream - forward_features| = {err:.3g}; embeddings equal: video "
              f"{torch.equal(full['video'], vis_emb[i])}, logmel {torch.equal(full['logmel'], aud_emb[i])}")
        assert err <= 1e-4 * max(1.0, want.abs().max().item())


def test_refusals_and_repacking():
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    with pytest.raises(TypeError, match="JMT / MT attend over the whole window"):
        streaming.StreamSession(JMT.__new__(JMT))
    mods = ["vggish", "bert"]
    m = _can(mods, dev, seed=8)
    with pytest.raises(ValueError, match="no windows"):
        streaming.StreamSession(m, window_length=100, hop_length=50)
    sess = streaming.StreamSession(m, max_streams=2, max_chunk=8)
    sid = sess.open()
    x = _feats(mods, 16, 2, dev)
    with pytest.raises(ValueError, match="'wave' cannot be streamed"):
        sess.push([sid], {"wave": torch.zeros(16000, device=dev), **{k: v[None, :8] for k, v in x.items()}})
    m.train()
    with pytest.raises(RuntimeError, match="model.eval"):
        sess.push([sid], {k: v[None, :8] for k, v in x.items()})
    with pytest.raises(RuntimeError, match="model.eval"):
        streaming.StreamSession(m)
    m.eval()
    tcn = m._engines()[0]["bert"]
    tcn.precision = "fp32"
    try:
        with pytest.raises(NotImplementedError, match="tensor-core TCN"):
            streaming.StreamSession(m)
    finally:
        tcn.precision = "tf32"
    old = _kernel_on_tcn(m, x)
    assert torch.equal(sess.push([sid], {k: v[None, :8] for k, v in x.items()})[0][0], old[:8])
    m.load_state_dict(synthetic.can_state_dict(9, mods), strict=True)
    new = _kernel_on_tcn(m, x)
    assert not torch.equal(new, old)
    sid2 = sess.open()
    out = torch.cat([sess.push([sid2], {k: v[None, a:a + 8] for k, v in x.items()})[0][0] for a in (0, 8)])
    assert torch.equal(out, new)
