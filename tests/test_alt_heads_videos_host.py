"""Whole-video inference of CAN / JMT / MT (windowing.infer_videos) on the host, no GPU: the segment offsets and the
padded-batch row tables built from video lengths, every refusal made before device work, and the dispatch between
the windowed LFAN path and the whole-video path."""
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import engine, synthetic, windowing

BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}


@pytest.mark.parametrize("lengths", [[1], [1, 1, 1], [5, 5, 5], [3000], [7, 1, 300, 1201, 2], [150, 3000, 37]])
def test_segments_and_padded_rows_from_lengths(lengths):
    seg = engine.Segments(lengths, "cpu")
    want = [0]
    for t in lengths:
        want.append(want[-1] + t)
    assert seg.offsets == want and seg.off.dtype == torch.int32 and seg.off.tolist() == want
    assert seg.n_seg == len(lengths) and seg.max_len == max(lengths) and seg.rows == sum(lengths)

    t_max, idx = windowing.padded_row_index(lengths)
    assert t_max == max(lengths) and idx.dtype == torch.int64 and idx.shape == (sum(lengths),)
    rows = torch.arange(sum(lengths)) + 1
    pad = torch.zeros(len(lengths) * t_max, dtype=torch.int64)
    pad[idx] = rows                                               # scatter the concatenated rows into the padded batch
    pad = pad.view(len(lengths), t_max)
    for i, t in enumerate(lengths):
        assert torch.equal(pad[i, :t], rows[want[i]:want[i + 1]])
        assert (pad[i, t:] == 0).all()                            # padding only past a video's end
    assert torch.equal(pad.view(-1)[idx], rows)                   # and gathered back in concatenated order


def test_empty_tables():
    seg = engine.Segments([], "cpu")
    assert seg.n_seg == 0 and seg.max_len == 0 and seg.rows == 0 and seg.off.tolist() == [0]
    t_max, idx = windowing.padded_row_index([])
    assert t_max == 0 and idx.numel() == 0
    with pytest.raises(ValueError, match="positive lengths"):
        engine.Segments([3, 0, 2], "cpu")


def _can(mods):
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    return CAN(task="CLASSIFICATION", modalities=list(mods), tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
               output_dim=7, root_dir="", device="cpu",
               audio_state_dict=synthetic.vggish_state_dict(0) if "logmel" in mods else None).eval()


def _jmt(name="JMT"):
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    return JMT(task="CLASSIFICATION", modalities=["video", "vggish"], tcn_settings=synthetic.TCN_SETTINGS,
               backbone_settings=BS, output_dim=7, root_dir="", device="cpu", model_name=name,
               visual_state_dict=synthetic.visual_backbone_state_dict(0)).eval()


def _video(T):
    return torch.zeros(T, 256, 256, 3, dtype=torch.uint8)


def test_refusals():
    can = _can(["vggish", "logmel", "bert"])
    ok = {"vggish": torch.zeros(4, 128), "logmel": torch.zeros(4, 96, 64), "bert": torch.zeros(4, 768)}
    for kw in ({"window_length": 100}, {"hop_length": 100}, {"window_length": 600, "hop_length": 300}):
        with pytest.raises(ValueError, match="has no windows"):
            windowing.infer_videos(can, [_video(4)], [dict(ok)], **kw)
        with pytest.raises(ValueError, match="has no windows"):
            windowing.infer_video(can, _video(4), dict(ok), **kw)
    for drop in ("vggish", "bert"):
        with pytest.raises(ValueError, match=f"video 1: the head needs modality '{drop}'"):
            windowing.infer_videos(can, [_video(4), _video(4)], [dict(ok), {k: v for k, v in ok.items() if k != drop}])
    with pytest.raises(ValueError, match=r"needs modality 'logmel' \(or 'wave'\)"):
        windowing.infer_videos(can, [_video(4)], [{k: v for k, v in ok.items() if k != "logmel"}])
    for key, bad in (("bert", torch.zeros(5, 768)), ("logmel", torch.zeros(3, 96, 64)), ("vggish", torch.zeros(1, 128))):
        with pytest.raises(ValueError, match=f"'{key}' has {bad.shape[0]} rows for 4 frames"):
            windowing.infer_videos(can, [_video(4)], [{**ok, key: bad}])
    with pytest.raises(ValueError, match="video 0 is empty"):
        windowing.infer_videos(can, [_video(0)], [{k: v[:0] for k, v in ok.items()}])
    with pytest.raises(ValueError, match="one feature dict per video"):
        windowing.infer_videos(can, [_video(4)], [])
    assert windowing.infer_videos(can, [], []) == []
    jmt = _jmt()
    with pytest.raises(ValueError, match="JMT runs over the whole video"):
        windowing.infer_videos(jmt, [_video(4)], [{"vggish": torch.zeros(4, 128)}], hop_length=150)
    with pytest.raises(ValueError, match="needs modality 'vggish'"):
        windowing.infer_videos(jmt, [_video(4)], [{"bert": torch.zeros(4, 768)}])
    with pytest.raises(ValueError, match="video 0 is empty"):
        windowing.infer_video(jmt, _video(0), {"vggish": torch.zeros(0, 128)})


class _Stop(Exception):
    pass


def test_dispatch(monkeypatch):
    """An LFAN goes through the window grid; a CAN / JMT / MT through forward_videos with the video lengths, and
    infer_video of a head is infer_videos on that one video.  The backbones are stubbed (no device work)."""
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    calls = []

    def rows(model, videos, feats, lengths, mods, fps):
        calls.append(("rows", list(mods), list(lengths)))
        return {m: torch.zeros(sum(lengths), 1) for m in mods}

    def grid(lengths, W, H):
        calls.append(("windows", list(lengths), W, H))
        raise _Stop

    monkeypatch.setattr(windowing, "_backbone_rows", rows)
    monkeypatch.setattr(windowing, "window_index_table", grid)
    lfan = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=["vggish", "bert"], kernel_size=5,
                example_length=300, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2, root_dir="", device="cpu")
    with pytest.raises(_Stop):
        windowing.infer_videos(lfan, [_video(3), _video(5)], [{}, {}], window_length=100, hop_length=50)
    assert calls == [("rows", ["vggish", "bert"], [3, 5]), ("windows", [3, 5], 100, 50)]

    for model in (_can(["vggish", "bert"]), _jmt("MT")):
        calls.clear()
        feats = {m: torch.zeros(0, 1) for m in model.modalities if m != "video"}
        monkeypatch.setattr(type(model), "forward_videos",
                            lambda self, src, lengths: calls.append(("head", sorted(src), list(lengths)))
                            or torch.arange(sum(lengths)).view(-1, 1))
        per = [{m: torch.zeros(t, 1) for m in feats} for t in (3, 1, 4)]
        out = windowing.infer_videos(model, [_video(3), _video(1), _video(4)], per)
        assert calls == [("rows", model.modalities, [3, 1, 4]), ("head", sorted(model.modalities), [3, 1, 4])]
        assert [o.view(-1).tolist() for o in out] == [[0, 1, 2], [3], [4, 5, 6, 7]]
        seen = []
        monkeypatch.setattr(windowing, "infer_videos", lambda *a: seen.append(a) or [torch.ones(2, 7)])
        assert torch.equal(windowing.infer_video(model, _video(2), per[0], 300, 200, 25.0), torch.ones(2, 7))
        assert seen[0][0] is model and len(seen[0][1]) == 1 and seen[0][3:] == (300, 200, 25.0)
        monkeypatch.undo()
        monkeypatch.setattr(windowing, "_backbone_rows", rows)
        monkeypatch.setattr(windowing, "window_index_table", grid)
