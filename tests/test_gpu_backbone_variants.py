"""IR-SE-50, IR-100, IR-SE-100 and IR-SE-152 plans, unit by unit, against an fp64 reference of each unit; and the
six Backbone(num_layers, mode) modules end to end against the fp32 oracle.

Same design as tests/test_gpu_ir50_layers.py: the plan's own bf16 output of unit i-1 (debug_activation) is the
input of an fp64 reference of unit i on the device, and the plan's output of unit i must satisfy
emulate.bound_ratio <= 1.  Plain IR units use emulate.ir50_unit (a MaxPool(1, 2) shortcut is packed as identity
columns, which the reference runs as a 1x1 stride-2 conv with the identity matrix); IR-SE units use
emulate_se.se_unit, whose bound adds the envelope of r's bf16 rounding scaled by the gate and the gate error that
envelope implies.  Each case pins the set of kernels its conv ops launch (op_variant, projection convs included):
all of them are instantiations that tests/test_gpu_ir50_layers.py and tests/test_gpu_kernels.py already pin; the
SE kernels (se.cu) are not conv instantiations.  Inputs are synthetic frames with per-frame contrast and
brightness (emulate_se.spread_frames) so that the frames' gates differ.
"""
import time

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import oracle_se
from tests import emulate, emulate_se
from tests.test_backbone_variants_host import CONFIGS, backbone_state_dict
from tests.test_gpu_ir50_layers import (HALO128, IGEMM128, IGEMM128_ALIGNED, IGEMM256, IGEMM256_ALIGNED, PAIR256,
                                        PAIR_BRES18, PAIR_BRES19, STRIP, _chunks, _stem_worst)

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

IGEMM64 = "conv_igemm_kernel<64,8,0,0>"
IGEMM64_BRES9 = "conv_igemm_kernel<64,9,1,1>"
IGEMM128_BRES = "conv_igemm_kernel<128,4,1,0>"

_SE50 = frozenset({STRIP, HALO128, PAIR_BRES18, PAIR256, IGEMM128_BRES, IGEMM256, IGEMM256_ALIGNED, IGEMM128})
_SE50_SMALL = frozenset({STRIP, HALO128, IGEMM128, IGEMM128_ALIGNED, IGEMM256, IGEMM256_ALIGNED})
# 112 px: the stride-2 64 -> 64 conv2 of unit 0 on igemm<64> (10 k-steps with the identity columns, 9 without),
# stage 2 (28 x 28, too wide for the raster kernel) on the pair kernels
_DEEP_IR = frozenset({STRIP, IGEMM64, HALO128, PAIR_BRES19, PAIR_BRES18, PAIR256, IGEMM256, IGEMM256_ALIGNED, IGEMM128})
_DEEP_SE = frozenset({STRIP, IGEMM64_BRES9, HALO128, PAIR_BRES18, IGEMM128_BRES, PAIR256, IGEMM256, IGEMM256_ALIGNED,
                      IGEMM128})

PLAN_CASES = [
    # IR-SE-50 at 40 px: the benchmarked pass size, a ragged count, and a pass below the pair-kernel threshold
    dict(id="se50_p2400_n2400", layers=50, se=True, in_hw=40, fpp=2400, n=2400, variants=_SE50),
    dict(id="se50_p2400_n1999", layers=50, se=True, in_hw=40, fpp=2400, n=1999, variants=_SE50),
    dict(id="se50_p2400_n189", layers=50, se=True, in_hw=40, fpp=2400, n=189, variants=_SE50_SMALL),
    # IR-100 at 112 px (Backbone.deep_frames_per_pass = 512): stage 1 starts with the identity-column unit
    dict(id="ir100_p512_n512", layers=100, se=False, in_hw=112, fpp=512, n=512, variants=_DEEP_IR),
    dict(id="ir100_p512_n333", layers=100, se=False, in_hw=112, fpp=512, n=333, variants=_DEEP_IR),
    # IR-SE-100 / IR-SE-152: stride-2 identity shortcut read by the SE tail
    dict(id="se100_p512_n512", layers=100, se=True, in_hw=112, fpp=512, n=512, variants=_DEEP_SE),
    dict(id="se152_p512_n512", layers=152, se=True, in_hw=112, fpp=512, n=512, variants=_DEEP_SE),
]

FC_ATOL = 1e-5


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _unit_worst(u, h, got):
    n, H, W, _ = h.shape
    worst = 0.0
    for f0, f1 in _chunks(n, H * W * max(u["cin"], u["depth"])):
        hh = h[f0:f1].permute(0, 3, 1, 2).double()
        if "se" in u:
            ref, B, _ = emulate_se.se_unit(u, hh, envelope=True)
        else:
            ref, B = emulate.ir50_unit(u, hh, envelope=True)
        worst = max(worst, emulate.bound_ratio(got[f0:f1].permute(0, 3, 1, 2), ref, B).max().item())
    return worst


def _to(u, dev):
    out = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in u.items()}
    if "se" in u:
        out["se"] = {k: v.to(dev) for k, v in u["se"].items()}
    return out


@pytest.mark.parametrize("case", PLAN_CASES, ids=lambda c: c["id"])
def test_variant_plan_units_vs_fp64_reference(case):
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    t0 = time.time()
    hw, n = case["in_hw"], case["n"]
    units = synthetic.ir_units(case["layers"])
    sd = synthetic.visual_backbone_state_dict(0, units=units, spatial=7 if hw == 112 else hw // 8, se=case["se"])
    pk = packing.pack_ir50(sd, "backbone.", in_hw=hw, strides=[s for _, _, s in units])
    eng = Ir50Engine(pk, dev, frames_per_pass=case["fpp"])
    assert eng.n_conv_ops == 2 * len(units) + 1 + (3 if case["se"] else 0)
    ran = {eng.op_variant(op, n) for op in range(eng.n_conv_ops)}
    assert ran == case["variants"], f"extra {sorted(ran - case['variants'])}, missing {sorted(case['variants'] - ran)}"

    x = emulate_se.spread_frames(synthetic.frames(n, seed=41, size=hw), seed=5).to(dev)
    dunits = [_to(u, dev) for u in pk["units"]]
    prev = eng.debug_activation(x, -1)
    worst = {-1: _stem_worst(pk, x, prev)}
    for i, u in enumerate(dunits):
        got = eng.debug_activation(x, i)
        worst[i] = _unit_worst(u, prev, got)
        prev = got
    e = prev.reshape(n, -1).double() @ pk["fc_w"].to(dev, torch.float64).t() + pk["fc_bias"].to(dev, torch.float64)
    emb = eng.forward(x)
    fc_err = (emb.double() - e / e.norm(dim=1, keepdim=True)).abs().max().item()
    torch.cuda.synchronize()
    print(f"\n[{case['id']}] {time.time() - t0:.1f} s; worst bound ratio min/max over units "
          f"{min(worst.values()):.3f}/{max(worst.values()):.3f}: " + " ".join(f"{i}:{r:.3f}" for i, r in worst.items())
          + f"; FC + l2norm max abs err {fc_err:.2e}")
    over = {i: r for i, r in worst.items() if not r <= 1.0}
    assert not over, f"units over the bound (-1 = stem): {over}"
    assert fc_err <= FC_ATOL


@pytest.mark.parametrize("num_layers,mode", CONFIGS, ids=[f"{n}_{m}" for n, m in CONFIGS])
def test_backbone_module_vs_oracle(num_layers, mode):
    """Backbone(num_layers, 0.4, 3, mode) with its 7x7 head (56 px for IR-50, 112 px for IR-100 / IR-152)."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.modules import Backbone
    units = synthetic.ir_units(num_layers)
    hw = 56 if num_layers == 50 else 112
    m = Backbone(num_layers, 0.4, 3, mode)
    sd = backbone_state_dict(num_layers, mode)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval()
    x = emulate_se.spread_frames(synthetic.frames(4, seed=9, size=hw), seed=2)
    ref = oracle_se.ir_forward(sd, x, "", units=units, se=mode == "ir_se")
    got = m(x.to(dev)).cpu()
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=1).min().item()
    print(f"\n[Backbone({num_layers}, mode={mode!r})] min embedding cosine vs fp32 oracle {cos:.6f}")
    assert cos >= 0.999


def test_visual_backbone_ir_se_vs_oracle():
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.modules import VisualBackbone
    vb = VisualBackbone(use_pretrained=False, mode="ir_se")
    sd = synthetic.visual_backbone_state_dict(3, se=True)
    vb.load_state_dict(sd, strict=True)
    vb = vb.to(dev).eval()
    x = emulate_se.spread_frames(synthetic.frames(6, seed=8), seed=1)
    ref = oracle_se.ir_forward(sd, x, "backbone.", se=True)
    cos = torch.nn.functional.cosine_similarity(vb(x.to(dev)).cpu(), ref, dim=1).min().item()
    print(f"\n[VisualBackbone(mode='ir_se')] min embedding cosine vs fp32 oracle {cos:.6f}")
    assert cos >= 0.999
