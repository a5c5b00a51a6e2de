"""CPU checks that keep the IR-SE per-unit bound (tests/emulate_se.py) honest, on a stage-1 unit (stride 1 and the
stride-2 identity unit of IR-SE-100), a transition unit (projection shortcut) and a stage-3 unit:

1. an fp32 stand-in for a correct plan (fp32 convs and gate, bf16 stores where the plan stores) stays under it;
2. each SE-tail fault a kernel could make exceeds it by more than 4x.

The synthetic gates must be spread out, neither saturated (a dropped gate would pass) nor all alike (a gate
from the neighbouring frame would pass); their spread is printed and checked.
"""
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate, emulate_se

torch.set_grad_enabled(False)


def _bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def _chain(num_layers, in_hw, upto, n=3):
    """Packed IR-SE weights and the bf16 input of every unit up to `upto` (fp32 chain, bf16 stores)."""
    units = synthetic.ir_units(num_layers)
    sd = synthetic.visual_backbone_state_dict(0, units=units, spatial=in_hw // (8 if num_layers == 50 else 16), se=True)
    pk = packing.pack_ir50(sd, "backbone.", in_hw=in_hw, strides=[s for _, _, s in units])
    x = emulate_se.spread_frames(synthetic.frames(n, seed=21, size=in_hw), seed=3)
    h = emulate_se.stem(pk, x)
    # deep in the synthetic network the frames' channel means converge; per-frame scales of each unit's input keep
    # the frames' gates apart (the chain itself runs unscaled)
    scale = torch.linspace(0.4, 1.8, n).view(n, 1, 1, 1)
    ins = {}
    for i in range(upto + 1):
        ins[i] = _bf(h * scale)
        y, _, _ = emulate_se.se_unit(pk["units"][i], h)
        h = _bf(y)
    return pk, ins


@pytest.fixture(scope="module")
def se50():
    return _chain(50, 40, 10)


@pytest.fixture(scope="module")
def se100():
    return _chain(100, 112, 0, n=2)


CASES = [("se50", 1, "stage 1"), ("se50", 3, "transition 64->128"), ("se50", 10, "stage 3"),
         ("se100", 0, "stage 1, stride-2 identity")]


@pytest.mark.parametrize("net,unit,what", CASES, ids=[f"{c[0]}_u{c[1]}" for c in CASES])
def test_se_unit_bound_passes_fp32_and_fails_each_fault(request, net, unit, what):
    pk, ins = request.getfixturevalue(net)
    u = pk["units"][unit]
    h = ins[unit].double()
    ref, B, gate = emulate_se.se_unit(u, h, envelope=True)
    standin = _bf(emulate_se.se_unit(u, h.float())[0])
    worst = emulate.bound_ratio(standin, ref, B).max().item()
    sat = ((gate < 0.02) | (gate > 0.98)).double().mean().item()
    nb = (gate - gate.roll(1, 0)).abs().mean().item()
    print(f"\n[{net} unit {unit}, {what}] fp32 stand-in worst ratio {worst:.3f}; gate min/std/max "
          f"{gate.min():.3f}/{gate.std():.3f}/{gate.max():.3f}, {100 * sat:.1f} % outside [0.02, 0.98], "
          f"mean |gate - neighbour frame's| {nb:.3f}")
    assert worst <= 1.0, f"fp32 stand-in exceeds the bound: {worst}"
    assert sat < 0.1 and gate.std() > 0.1 and nb > 0.02, "synthetic gates saturated or alike"
    ratios = {}
    for fault in emulate_se.FAULTS:
        if fault == "unstrided_shortcut" and (u["stride"] == 1 or u["has_proj"]):
            continue
        got = _bf(emulate_se.se_unit(u, h, fault=fault)[0])
        ratios[fault] = emulate.bound_ratio(got, ref, B).max().item()
    print("  fault ratios: " + " ".join(f"{k}:{v:.1f}" for k, v in ratios.items()))
    weak = {k: v for k, v in ratios.items() if not v > 4.0}
    assert not weak, f"unit {unit}: faults pass the bound: {weak}"
