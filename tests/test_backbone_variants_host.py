"""Host side of the six reference backbones Backbone(num_layers in {50, 100, 152}, mode in {'ir', 'ir_se'}):
module key layout, the packed SE / identity-column algebra against the oracle, and IR-50 packing unchanged."""
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from feature_vs_text_compound_emotion_b200.modules import Backbone, VisualBackbone
from tests import oracle_se
from tests import emulate, emulate_se

torch.set_grad_enabled(False)

CONFIGS = [(50, "ir"), (50, "ir_se"), (100, "ir"), (100, "ir_se"), (152, "ir"), (152, "ir_se")]
KEYS = {(50, "ir"): 349, (50, "ir_se"): 397, (100, "ir"): 674, (100, "ir_se"): 772, (152, "ir"): 687, (152, "ir_se"): 787}


def backbone_state_dict(num_layers, mode, seed=0, spatial=7):
    """Backbone.state_dict() layout (no prefix) of synthetic weights."""
    units = synthetic.ir_units(num_layers)
    sd = synthetic.visual_backbone_state_dict(seed, units=units, spatial=spatial, se=mode == "ir_se")
    return {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}


def packed_forward(pk, x):
    """Packed-weight forward without activation rounding (fp32 algebra check)."""
    w = pk["stem_w"].view(3, 3, 3, 64).permute(3, 2, 0, 1)
    h = torch.nn.functional.conv2d(x, w, pk["stem_bias"], 1, 1)
    h = torch.where(h >= 0, h, h * pk["stem_alpha"].view(1, -1, 1, 1))
    for u in pk["units"]:
        h = (emulate_se.se_unit(u, h, round_act=False) if "se" in u else emulate.ir50_unit(u, h, round_t=False))[0]
    e = torch.nn.functional.linear(h.permute(0, 2, 3, 1).reshape(x.shape[0], -1), pk["fc_w"].float(), pk["fc_bias"])
    return e / e.norm(dim=1, keepdim=True)


@pytest.mark.parametrize("num_layers,mode", CONFIGS, ids=[f"{n}_{m}" for n, m in CONFIGS])
def test_module_keys_and_strict_load(num_layers, mode):
    m = Backbone(num_layers, 0.4, 3, mode)
    assert len(m.state_dict()) == KEYS[(num_layers, mode)]
    m.load_state_dict(backbone_state_dict(num_layers, mode), strict=True)
    if mode == "ir_se":
        d = m.body[-1].res_layer[5]
        assert d.fc1.weight.shape == (32, 512, 1, 1) and d.fc2.weight.shape == (512, 32, 1, 1)


def test_visual_backbone_ir_se_keys():
    vb = VisualBackbone(use_pretrained=False, mode="ir_se")
    sd = synthetic.visual_backbone_state_dict(0, se=True)
    assert len(vb.state_dict()) == 399 and list(vb.state_dict()) == list(sd)
    vb.load_state_dict(sd, strict=True)


@pytest.mark.parametrize("num_layers,mode", CONFIGS, ids=[f"{n}_{m}" for n, m in CONFIGS])
def test_packed_algebra_exact_in_fp32(num_layers, mode):
    """fp32 operands, no activation rounding: the SE tail, the split projection (bias2 [2][depth]) and the
    identity columns of a MaxPool(1, 2) shortcut reproduce the oracle to fp32 round-off.  Small inputs (the units
    run at any size): 40 px for IR-50 (5x5 head), 32 px for IR-100 / IR-152 (2x2 head)."""
    hw, spatial = (40, 5) if num_layers == 50 else (32, 2)
    units = synthetic.ir_units(num_layers)
    sd = synthetic.visual_backbone_state_dict(1, units=units, spatial=spatial, se=mode == "ir_se")
    pk = packing.pack_ir50(sd, "backbone.", in_hw=hw, operand_dtype=torch.float32, strides=[s for _, _, s in units])
    x = synthetic.frames(2, seed=6, size=hw)
    ref = oracle_se.ir_forward(sd, x, "backbone.", units=units, se=mode == "ir_se")
    err = (packed_forward(pk, x) - ref).abs().max().item()
    assert err < 2e-5, err
    u0 = pk["units"][0]
    if num_layers != 50 and mode == "ir":
        assert u0["has_proj"] == 1 and u0.get("identity_sc") == 1 and u0["w2"].shape == (64, 9 * 64 + 64)
        assert torch.equal(u0["w2"][:, 9 * 64:], torch.eye(64))
    if num_layers != 50 and mode == "ir_se":
        assert u0["has_proj"] == 0 and u0["stride"] == 2 and u0["w2"].shape == (64, 9 * 64)
    if mode == "ir_se":
        t = next(u for u in pk["units"] if u["has_proj"])
        assert t["bias2"].shape == (2, t["depth"]) and t["se"]["fc1"].shape == (t["depth"] // 16, t["depth"])


def test_ir50_packing_without_strides_unchanged():
    """pack_ir50 without strides infers IR-50's strides as before; passing them gives the same tensors, and no
    IR-50 unit gains identity columns or SE weights."""
    sd = synthetic.visual_backbone_state_dict(0)
    a = packing.pack_ir50(sd, "backbone.")
    b = packing.pack_ir50(sd, "backbone.", strides=[s for _, _, s in synthetic.IR50_UNITS])
    assert [u["stride"] for u in a["units"]] == [s for _, _, s in synthetic.IR50_UNITS]
    for ua, ub in zip(a["units"], b["units"]):
        assert set(ua) == set(ub) == {"cin", "depth", "stride", "has_proj", "w1", "bias1", "alpha", "w2", "bias2"}
        for k, v in ua.items():
            assert torch.equal(v, ub[k]) if torch.is_tensor(v) else v == ub[k]
        assert ua["bias2"].shape == (ua["depth"],)


@pytest.mark.parametrize("num_layers,mode", CONFIGS, ids=[f"{n}_{m}" for n, m in CONFIGS])
def test_oracle_matches_staged_reference_backbone(num_layers, mode):
    """Where oracle/_ref is staged: the oracle equals the reference's own Backbone (arcface_model.py) in eval mode."""
    import importlib
    from oracle import build_ref
    build_ref.stage()
    if not build_ref.available():
        pytest.skip("oracle/_ref not staged (no /root/reference here)")
    build_ref.load()
    am = importlib.import_module("models.arcface_model")
    ref = am.Backbone(num_layers=num_layers, drop_ratio=0.4, input_channels=3, mode=mode)
    sd = backbone_state_dict(num_layers, mode, seed=4)
    ref.load_state_dict(sd, strict=True)
    ref.eval()
    hw = 56 if num_layers == 50 else 112
    x = synthetic.frames(1, seed=3, size=hw)
    want = ref(x)
    got = oracle_se.ir_forward(sd, x, "", units=synthetic.ir_units(num_layers), se=mode == "ir_se")
    assert (got - want).abs().max().item() < 2e-5
