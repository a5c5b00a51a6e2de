"""JMT / MT streaming bookkeeping of streaming.StreamSession on the host, no GPU: the history rows a peek gathers, the
max_frames bound of a push, the history's share of state_bytes, and the argument checks made before any device work."""
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import streaming, synthetic

BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}


def _naive_rows(sids, lengths, max_frames):
    rows = []
    for s, t in zip(sids, lengths):
        for f in range(t):
            rows.append(s * max_frames + f)
    return rows


@pytest.mark.parametrize("sids,lengths,max_frames", [
    ([0], [1], 1),
    ([0], [0], 5),
    ([3, 0, 7], [5, 0, 9], 9),                       # a 0-length stream, and one at full max_frames
    ([7, 2, 5, 1], [18000, 1, 0, 17999], 18000),
    ([4, 1], [30, 30], 30),
    ([], [], 10),
])
def test_history_row_index_against_a_loop(sids, lengths, max_frames):
    idx = streaming.history_row_index(sids, lengths, max_frames)
    assert idx.dtype == torch.int64 and idx.shape == (sum(lengths),)
    assert idx.tolist() == _naive_rows(sids, lengths, max_frames)
    assert idx.numel() == 0 or int(idx.max()) < (max(sids) + 1) * max_frames


def test_history_row_index_gathers_each_stream_in_order():
    S, F, C = 4, 6, 3
    hist = torch.arange(S * F * C, dtype=torch.float32).view(S, F, C)
    sids, lengths = [2, 0, 3], [4, 6, 1]
    got = hist.view(-1, C).index_select(0, streaming.history_row_index(sids, lengths, F))
    want = torch.cat([hist[s, :t] for s, t in zip(sids, lengths)])
    assert torch.equal(got, want)


def test_max_frames_bound():
    F = 100
    assert streaming.history_overflow([70], 30, F) == []             # exactly max_frames
    assert streaming.history_overflow([71], 30, F) == [0]            # one frame past it
    assert streaming.history_overflow([0], F, F) == []
    assert streaming.history_overflow([0], F + 1, F) == [0]
    assert streaming.history_overflow([F], 1, F) == [0]              # a full stream takes no more frames
    assert streaming.history_overflow([10, 99, 70, 0], 1, F) == []
    assert streaming.history_overflow([10, 99, 70, 0], 2, F) == [1]  # only one of several streams overflows
    assert streaming.history_overflow([10, 99, 70, 0], 31, F) == [1, 2]


def test_history_bytes_formula():
    chans = [synthetic.TCN_SETTINGS[m]["channel"][-1] for m in ("video", "vggish")]
    assert chans == [128, 64]
    assert streaming.history_bytes(chans, 1) == 768                  # fp32 video 128 + vggish 64 per frame
    assert streaming.history_bytes(chans, 18000) == 18000 * 768      # 10 min at 30 fps: 13.8 MB per stream
    assert streaming.history_bytes([32], 7) == 4 * 7 * 32
    assert streaming.history_bytes(chans, 0) == 0


def _jmt(name="JMT"):
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    return JMT(task="CLASSIFICATION", modalities=["video", "vggish"], tcn_settings=synthetic.TCN_SETTINGS,
               backbone_settings=BS, output_dim=7, root_dir="", device="cpu", model_name=name,
               visual_state_dict=synthetic.visual_backbone_state_dict(0)).eval()


@pytest.mark.parametrize("name", ["JMT", "MT"])
def test_refusals_before_the_device(name):
    from feature_vs_text_compound_emotion_b200.models.model import CAN, LFAN
    m = _jmt(name)
    with pytest.raises(TypeError, match="JMT / MT attend over the whole window") as e:
        streaming.StreamSession(m)
    assert "max_frames" in str(e.value)
    for bad in (0, -5):
        with pytest.raises(ValueError, match="max_frames must be positive"):
            streaming.StreamSession(m, max_frames=bad)
    for W, H in ((100, 50), (300, 100)):
        with pytest.raises(ValueError, match=f"a {name} stream has no windows"):
            streaming.StreamSession(m, max_frames=100, window_length=W, hop_length=H)
    with pytest.raises(ValueError, match="must be positive"):
        streaming.StreamSession(m, max_frames=100, max_streams=0)
    for other in (LFAN.__new__(LFAN), CAN.__new__(CAN)):
        with pytest.raises(ValueError, match="max_frames applies to JMT / MT sessions only"):
            streaming.StreamSession(other, max_frames=100)
