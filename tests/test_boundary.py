"""Drop-in boundary on the CPU: constructors, state_dict layout, strict loading, C-ABI symbols.
No compute calls (those need a GPU and live in test_gpu_*.py)."""
import ctypes
import json
import os
import re
import warnings

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import _capi, synthetic

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}


def _lfan(mods):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=mods, kernel_size=5,
             example_length=300, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2, root_dir="",
             device="cpu")
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(0) if "video" in mods else None,
           audio_state_dict=synthetic.vggish_state_dict(0) if "logmel" in mods else None)
    return m


def test_lfan_state_dict_layout_equals_reference(golden_dir):
    keys = json.load(open(os.path.join(golden_dir, "state_keys.json")))
    m = _lfan(["video", "vggish", "bert"])
    sd = m.state_dict()
    assert list(sd) == list(keys)
    for k, v in sd.items():
        assert list(v.shape) == keys[k], k
    m.load_state_dict(synthetic.lfan_state_dict(0, ["video", "vggish", "bert"]), strict=True)
    trainable = sum(p.numel() for p in m.parameters() if p.requires_grad)
    assert trainable == 5002503          # SURVEY.md section 9
    assert sum(p.numel() for p in m.parameters()) == 42290127


def test_logmel_lfan_and_vggish_layouts_equal_reference(golden_dir, tmp_path):
    g = torch.load(os.path.join(golden_dir, "lfan_logmel_b1.pt"))
    m = _lfan(g["modalities"])
    assert {k: list(v.shape) for k, v in m.state_dict().items()} == g["keys"]
    assert list(m.state_dict()) == list(g["keys"])
    m.load_state_dict(synthetic.lfan_state_dict(0, g["modalities"]), strict=True)
    assert not any(p.requires_grad for p in m.spatial["audio"].parameters())
    # vggish.pth layout through root_dir, as models/model.py:437-449 loads it
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    torch.save(synthetic.vggish_state_dict(0), tmp_path / "vggish.pth")
    m2 = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=["logmel"], root_dir=str(tmp_path),
              tcn_channel=synthetic.TCN_CHANNELS, device="cpu")
    m2.init()
    v = torch.load(os.path.join(golden_dir, "vggish_n6.pt"))
    assert {k: list(t.shape) for k, t in m2.spatial["audio"].backbone.state_dict().items()} == v["keys"]


def test_feature_only_modalities():
    m = _lfan(["cnn_res50", "vggish", "bert"])
    assert "spatial.visual.backbone.input_layer.0.weight" not in m.state_dict()
    m.load_state_dict(synthetic.lfan_state_dict(0, ["cnn_res50", "vggish", "bert"]), strict=True)
    assert m.final_dim == 224


def test_visual_backbone_loads_checkpoint_layout(tmp_path):
    from feature_vs_text_compound_emotion_b200.models.backbone import VisualBackbone
    p = tmp_path / "res50_ir_0.887.pth"
    torch.save(synthetic.visual_backbone_state_dict(0), p)
    vb = VisualBackbone(use_pretrained=True, state_dict_path=str(p))
    assert len(vb.state_dict()) == 351
    assert vb.backbone.output_layer[3].in_features == 12800


def test_forward_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    m = _lfan(["cnn_res50", "vggish", "bert"]).eval()
    X = synthetic.feature_windows(1, 300)
    with pytest.raises(_capi.CerError):
        with torch.no_grad():
            m(X)


def test_training_mode_never_falls_back():
    """LFAN in training mode goes to the CUDA training plan (CerError without a GPU); the
    inference-only sub-modules refuse a training-mode forward instead of computing something else."""
    m = _lfan(["cnn_res50", "vggish", "bert"]).train()
    if not torch.cuda.is_available():
        with pytest.raises(_capi.CerError), torch.enable_grad():
            m(synthetic.feature_windows(1, 300))
    with pytest.raises(NotImplementedError), torch.enable_grad():
        m.temporal["vggish"](torch.randn(1, 128, 300))


def test_head_parameter_order_matches_oracle_and_flat_layout():
    from feature_vs_text_compound_emotion_b200 import training
    from oracle import lfan_oracle as O
    mods = ["cnn_res50", "vggish", "bert"]
    m = _lfan(mods)
    names = [k for k, _ in training.head_parameters(m)]
    assert names == O.trainable_names(synthetic.lfan_state_dict(0, mods))
    assert sum(p.numel() for _, p in training.head_parameters(m)) == 5002503
    assert ctypes.sizeof(_capi.TrainConv) == 48 and ctypes.sizeof(_capi.TrainBlock) == 16 + 2 * 48 + 32


def test_capi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "cer_b200.h")).read()
    declared = set(re.findall(r"\b(cer_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_capi.SIGNATURES), declared ^ set(_capi.SIGNATURES)
    lib = _capi.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.cer_version() >= 100


def test_struct_sizes_match_header_layout():
    # 64-bit: int32 x4 + 5 pointers; guards against silent ctypes/header drift
    assert ctypes.sizeof(_capi.IrUnit) == 16 + 5 * 8
    assert ctypes.sizeof(_capi.TcnBlock) == 16 + 8 * 8
    assert ctypes.sizeof(_capi.Ir50Weights) == 8 + 3 * 8 + 8 + 8 + 8 + 2 * 8
    assert ctypes.sizeof(_capi.VggishStep) == 7 * 4


def test_alternative_head_layouts_equal_reference(golden_dir):
    from feature_vs_text_compound_emotion_b200.models.model import CAN, JMT
    g = torch.load(os.path.join(golden_dir, "heads.pt"))
    vsd = synthetic.visual_backbone_state_dict(0)
    can = CAN(task="CLASSIFICATION", modalities=g["CAN"]["modalities"], tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
              output_dim=7, root_dir="", device="cpu", visual_state_dict=vsd)
    assert {k: list(v.shape) for k, v in can.state_dict().items()} == g["CAN"]["keys"]
    assert list(can.state_dict()) == list(g["CAN"]["keys"])
    can.load_state_dict(synthetic.can_state_dict(0, g["CAN"]["modalities"]), strict=True)
    for name in ("JMT", "MT"):
        jm = JMT(task="CLASSIFICATION", modalities=g[name]["modalities"], tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
                 output_dim=7, root_dir="", device="cpu", model_name=name, visual_state_dict=vsd)
        assert list(jm.state_dict()) == list(g[name]["keys"]), name
        assert {k: list(v.shape) for k, v in jm.state_dict().items()} == g[name]["keys"], name
        jm.load_state_dict(synthetic.jmt_state_dict(0, g[name]["modalities"], model_name=name), strict=True)
