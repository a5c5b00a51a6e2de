"""CPU checks that keep the conv parity tests honest.

1. The per-element bound of tests/emulate.py (bound_ratio over ir50_unit) passes a correct kernel and fails
   each kernel-style fault: fp32 F.conv2d, which sums in another order than the fp64 reference, stands in
   for a correct kernel; the faults are the kinds a tiled conv kernel makes at borders, in its K loop,
   per N chunk, at the ragged tail and in the residual epilogue.
2. Every kernel instantiation that csrc/ir50.cu can select has a GPU parity case that pins it by name
   (tests/test_gpu_kernels.py CONV_CASES, tests/test_gpu_ir50_layers.py PLAN_CASES).
"""
import copy
import os
import re

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate

torch.set_grad_enabled(False)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


@pytest.fixture(scope="module")
def unit_inputs():
    pk = packing.pack_ir50(synthetic.visual_backbone_state_dict(0), "backbone.")
    _, taps = emulate.ir50_packed(pk, synthetic.frames(3, seed=21), round_act=True, upto=21)
    return pk, taps


def _drop_k_chunk(u):
    d = u["depth"]
    u["w2"][:, 4 * d:4 * d + 64] = 0               # centre tap of conv2, first 64 input channels


def _corner_takes_edge_bias(u):
    u["bias1"][0] = u["bias1"][1]                   # top-left corner class gets the top-edge bias


def _prelu_skipped_on_last_n_chunk(u):
    u["alpha"][-64:] = 1.0


WEIGHT_FAULTS = {"corner_bias": _corner_takes_edge_bias, "k_chunk": _drop_k_chunk, "prelu_n_chunk": _prelu_skipped_on_last_n_chunk}


@pytest.mark.parametrize("unit", [3, 5, 10, 21])
def test_unit_bound_passes_fp32_and_fails_each_fault(unit_inputs, unit):
    pk, taps = unit_inputs
    u = pk["units"][unit]
    h = taps[unit - 1].permute(0, 3, 1, 2).double()
    ref, E = emulate.ir50_unit(u, h, envelope=True)
    standin = _bf(emulate.ir50_unit(u, h.float())[0])
    worst = emulate.bound_ratio(standin, ref, E).max().item()
    assert worst <= 1.0, f"fp32 stand-in exceeds the bound: {worst}"
    faulty = {}
    for name, fault in WEIGHT_FAULTS.items():
        m = copy.deepcopy(u)
        fault(m)
        faulty[name] = _bf(emulate.ir50_unit(m, h)[0])
    tail = _bf(ref).clone()
    tail[-1, :, -1, -3:] = 0                        # the last three pixels of the last frame never stored
    faulty["tail_unstored"] = tail
    if not u["has_proj"]:
        faulty["residual_shifted"] = _bf(ref - h + h.roll(1, dims=3))    # residual read one pixel off
    for name, got in faulty.items():
        r = emulate.bound_ratio(got, ref, E).max().item()
        assert r > 4.0, f"unit {unit}: fault {name} passes the bound (worst ratio {r})"


def _selectable_variants():
    src = open(os.path.join(ROOT, "feature_vs_text_compound_emotion_b200", "csrc", "ir50.cu")).read()
    table = re.search(r"kVariantNames\[\]\s*=\s*\{(.*?)\};", src, re.S)
    assert table, "kVariantNames not found in ir50.cu"
    names = set(re.findall(r'"([^"]+)"', table.group(1))) - {"none"}
    raster = re.findall(r'kRasterName\w*\s*=\s*"([^"]+)"', src)
    assert raster, "raster kernel name not found in ir50.cu"
    return names | set(raster)


def test_every_conv_variant_has_a_parity_case():
    from tests.test_gpu_ir50_layers import PLAN_CASES
    from tests.test_gpu_kernels import CONV_CASES, PADDED_CASES
    from tests import test_gpu_vggish_layers as vgg
    pinned = {c[-1] for c in CONV_CASES} | {c[-1] for _, c in PADDED_CASES}
    for case in PLAN_CASES:
        pinned |= case["variants"]
    for case in vgg.PLAN_CASES:
        pinned |= {v for _, v, _ in case["variants"]} - {vgg.STEM, vgg.POOL}
    selectable = _selectable_variants()
    assert selectable == pinned, (f"without a parity case: {sorted(selectable - pinned)}; "
                                  f"not a kernel of ir50.cu: {sorted(pinned - selectable)}")
