"""CPU checks that keep the VGGish per-step parity tests (tests/test_gpu_vggish_layers.py) honest.

1. Through the emulated stack (three patches, the fused plan's steps), the per-element bounds of tests/emulate.py pass an
   fp32 stand-in for a correct kernel (F.conv2d / F.linear in fp32, bf16-rounded where the plan stores) on every step,
   and fail each kernel-style fault on the step it targets by more than 4x: pooling faults of the fused epilogue, a
   dropped K chunk, a shifted bias read, a skipped ReLU on one N chunk, the wrong flatten order, an unstored ragged tail,
   the wrong stem padding.
2. Every kernel instantiation that can take a pooled layer runs pooled in some VGGish plan case, and every VGGish pin
   names a kernel the sources define.
"""
import copy
import os
import re

import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate
from tests.test_conv_parity_guards import ROOT, _selectable_variants

torch.set_grad_enabled(False)

# conv_can_pool + select_conv_variant: the Cin = 64 conv (conv2) always pools on the halo kernel; the im2col convs
# (W = 16: conv4, W = 8: conv6) on the pair kernel or the one-CTA kernels at N tiles of 256 / 128 / 64
POOLED_VARIANTS = {"conv_halo_kernel<128>", "conv_igemm2_kernel<256,6>", "conv_igemm_kernel<256,4,0,1>",
                   "conv_igemm_kernel<128,6,0,1>", "conv_igemm_kernel<64,8,0,0>"}
CONV2, CONV3, CONV4, CONV5, CONV6 = range(5)      # packed["convs"] indices
FC1, FC2, FC3 = range(3)


def _bf(t):
    return t.to(torch.bfloat16).to(t.dtype)


def _nchw_flat(h):
    return h.permute(0, 2, 3, 1).reshape(h.shape[0], -1)         # the plan's NHWC flatten


@pytest.fixture(scope="module")
def stack():
    """Inputs (the stand-in's stored values, fp64) and fp64 references of every step."""
    pk = packing.pack_vggish(synthetic.vggish_state_dict(0))
    x = synthetic.logmel_patches(3, seed=31).double()
    ref = {"stem": emulate.vggish_stem(pk, x)}
    got = {"stem": _bf(emulate.vggish_stem(pk, x.float())).double()}
    inp = {}
    h = got["stem"]
    for i, c in enumerate(pk["convs"]):
        inp[("conv", i)] = h
        ref[("conv", i)] = emulate.vggish_conv(c, h, c["pool_after"])
        got[("conv", i)] = _bf(emulate.vggish_conv(c, h.float(), c["pool_after"])).double()
        h = got[("conv", i)]
    a = _nchw_flat(h)
    for i, f in enumerate(pk["fcs"]):
        inp[("fc", i)] = a
        ref[("fc", i)] = emulate.vggish_fc(f, a)
        y = emulate.vggish_fc(f, a.float()).double()
        got[("fc", i)] = y if i == len(pk["fcs"]) - 1 else _bf(y)
        a = got[("fc", i)]
    return pk, x, inp, ref, got


def _ratio(pk, key, got, ref, inp):
    if key == ("fc", FC3):
        return emulate.fc_dot_ratio(got, inp[key], pk["fcs"][FC3]).max().item()
    return emulate.bound_ratio(got, ref[key]).max().item()


def test_bounds_pass_the_fp32_standin(stack):
    pk, _, inp, ref, got = stack
    worst = {k: _ratio(pk, k, got[k], ref, inp) for k in ref}
    print("\nfp32 stand-in, worst bound ratio per step: " + " ".join(f"{k}:{r:.4f}" for k, r in worst.items()))
    assert all(r <= 1.0 for r in worst.values()), worst
    # FC_DOT_C keeps an 8x margin over the stand-in's fp32 reordering of the 4096-long dot products
    assert worst[("fc", FC3)] <= 1 / 8, worst[("fc", FC3)]


def _pool_shifted(y):
    return F.max_pool2d(y.roll(-1, dims=3), 2)                   # window one column to the right


def _pool_horizontal_only(y):
    return F.max_pool2d(y, (1, 2))[:, :, ::2]


def _pool_top_left(y):
    return y[:, :, ::2, ::2]


def _conv_faults(pk, inp):
    """(name, step key, faulty output) for the conv steps."""
    out = []
    for i, pool in ((CONV4, _pool_shifted), (CONV6, _pool_shifted), (CONV4, _pool_horizontal_only),
                    (CONV4, _pool_top_left), (CONV6, _pool_top_left)):
        y = emulate.vggish_conv(pk["convs"][i], inp[("conv", i)], False)
        out.append((pool.__name__, ("conv", i), _bf(pool(y))))
    c = copy.deepcopy(pk["convs"][CONV4])
    c["w"][:, 4 * c["cin"]:4 * c["cin"] + 64] = 0                # centre tap, first 64 input channels
    out.append(("k_chunk_dropped", ("conv", CONV4), _bf(emulate.vggish_conv(c, inp[("conv", CONV4)], True))))
    c = copy.deepcopy(pk["convs"][CONV5])
    c["bias"] = c["bias"].roll(128)
    out.append(("bias_off_by_128", ("conv", CONV5), _bf(emulate.vggish_conv(c, inp[("conv", CONV5)], False))))
    return out


def test_bounds_fail_each_fault(stack):
    pk, x, inp, ref, _ = stack
    faults = _conv_faults(pk, inp)
    f = pk["fcs"][FC2]
    y = F.linear(inp[("fc", FC2)], f["w"].double(), f["bias"].double())
    y[:, :-64] = torch.relu(y[:, :-64])                           # ReLU skipped on the last 64 outputs
    faults.append(("relu_skipped_last_n_chunk", ("fc", FC2), _bf(y)))
    h6 = _bf(ref[("conv", CONV6)])
    faults.append(("fc1_reads_chw_flatten", ("fc", FC1), _bf(emulate.vggish_fc(pk["fcs"][FC1], h6.reshape(3, -1)))))
    for key in (("conv", CONV2), ("conv", CONV6), ("fc", FC3)):
        tail = (_bf(ref[key]) if key != ("fc", FC3) else ref[key]).clone()
        tail[-1] = 0                                              # the last patch of the pass never stored
        faults.append(("last_patch_unstored", key, tail))
    f3 = copy.deepcopy(pk["fcs"][FC3])
    f3["w"][:, 1024:1088] = 0
    faults.append(("k_chunk_dropped", ("fc", FC3), emulate.vggish_fc(f3, inp[("fc", FC3)])))
    w = pk["conv1_w"].double().view(3, 3, -1).permute(2, 0, 1).unsqueeze(1)
    z = F.conv2d(F.pad(x.unsqueeze(1), (1, 1, 1, 1), mode="replicate"), w, pk["conv1_bias"].double())
    faults.append(("stem_edge_replicated", "stem", _bf(F.max_pool2d(torch.relu(z), 2))))
    ratios = {(name, key): _ratio(pk, key, got, ref, inp) for name, key, got in faults}
    print("\nfaults, worst bound ratio: " + " ".join(f"{n}@{k}:{r:.1f}" for (n, k), r in ratios.items()))
    passing = {k: r for k, r in ratios.items() if not r > 4.0}
    assert not passing, f"faults within 4x of the bound: {passing}"


def test_every_pooled_variant_has_a_vggish_case():
    from tests.test_gpu_vggish_layers import PLAN_CASES, POOL, STEM
    pooled = {v for case in PLAN_CASES for (_, v, p) in case["variants"] if p}
    assert POOLED_VARIANTS <= pooled, f"never run pooled: {sorted(POOLED_VARIANTS - pooled)}"
    conv_pins = {v for case in PLAN_CASES for (_, v, _) in case["variants"]} - {STEM, POOL}
    assert conv_pins <= _selectable_variants(), f"not a kernel of ir50.cu: {sorted(conv_pins - _selectable_variants())}"
    src = open(os.path.join(ROOT, "feature_vs_text_compound_emotion_b200", "csrc", "vggish.cu")).read()
    for name in (STEM, POOL):
        assert re.search(r"__global__ void\b[^;{]*?\b" + name + r"\(", src), f"{name} is not a kernel of vggish.cu"
