"""Continuous-stream bookkeeping of streaming.StreamSession with a CAN (host logic, no GPU), and the argument checks
that are made before any device work."""
import numpy as np
import pytest

from feature_vs_text_compound_emotion_b200 import _capi, streaming, synthetic

BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
FIELDS = {name: i for i, name in enumerate(_capi.STREAM_ENTRY_FIELDS)}


def test_continuous_step_table_one_never_ending_slot_per_stream():
    parity = {3: 0, 9: 0}
    t = {3: 0, 9: 0}
    for step in range(40):
        c = (1, 7, 30)[step % 3]
        streams = [(sid, t[sid], parity[sid]) for sid in (3, 9)]
        tab = streaming.continuous_step_table(streams)
        assert tab.dtype == np.int32 and tab.shape == (2, len(_capi.STREAM_ENTRY_FIELDS))
        for row, (sid, t_now, p) in zip(tab, streams):
            assert row[FIELDS["sid"]] == sid and row[FIELDS["t_now"]] == t_now and row[FIELDS["parity"]] == p
            assert row[FIELDS["start"]] == 0 and row[FIELDS["slot"]] == 0 and row[FIELDS["active"]] == 1
            assert row[FIELDS["lslot"]] == 0 and row[FIELDS["reserved"]] == 0
        for sid in t:
            t[sid] += c
            parity[sid] ^= 1
        assert parity[3] == (step + 1) % 2
    far = streaming.continuous_step_table([(0, 10 ** 8, 1)])
    assert far.tolist() == [[0, 0, 0, 0, 10 ** 8, 1, 1, 0]]
    assert streaming.continuous_step_table([]).shape == (0, len(_capi.STREAM_ENTRY_FIELDS))


def _can(mods=("cnn_res50", "vggish")):
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    return CAN(task="CLASSIFICATION", modalities=list(mods), tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
               output_dim=7, root_dir="", device="cpu").eval()


@pytest.mark.parametrize("W,H", [(100, 50), (300, 100), (200, 200)])
def test_can_refuses_window_arguments(W, H):
    with pytest.raises(ValueError, match="no windows"):
        streaming.StreamSession(_can(), window_length=W, hop_length=H)


def test_jmt_mt_and_other_objects_refused():
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    for obj in (JMT.__new__(JMT), object()):
        with pytest.raises(TypeError, match="JMT / MT attend over the whole window"):
            streaming.StreamSession(obj)


def test_can_refuses_empty_sessions():
    with pytest.raises(ValueError, match="must be positive"):
        streaming.StreamSession(_can(), max_streams=0)
    with pytest.raises(ValueError, match="must be positive"):
        streaming.StreamSession(_can(), max_chunk=0)
