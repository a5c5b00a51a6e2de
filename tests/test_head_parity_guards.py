"""CPU checks that keep the head parity tests (tests/test_gpu_head_launches.py) honest.

1. The per-element bounds of tests/emulate_head.py pass a correct kernel and fail kernel-style faults by more
   than 4x.  A correct TCN launch is stood in for by TF32-converted operands with fp32 matmuls, a correct
   fusion head by the plain fp32 emulate.fusion_packed; both sum in other orders than the fp64 references.
   The faults are the kinds the tiled kernels make: in the causal padding and tap offsets, in the K loop, per
   N tile, at the ragged M tile, in the epilogue, in the per-warp frame groups and in the reductions.
2. Every instantiation in the name tables of csrc/tcn_tc.cu, csrc/tcn.cu and csrc/fusion.cu (kHeadVariantNames,
   what cer_head_last_variant reports) is pinned by a GPU parity case.
"""
import copy
import os
import re

import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate, emulate_head as EH

torch.set_grad_enabled(False)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, T = 2, 100                       # M = 200 rows: the last 128-row M tile is ragged (72 rows)
FAULT_MIN = 4.0


def _stack(mods, channels=None, bn=True, seed=0):
    sd = synthetic.head_state_dict(seed, mods, tcn_channels=channels)
    out = {}
    for m in mods:
        blocks = packing.pack_tcn(sd, f"temporal.{m}.", f"bn.{m}" if bn else None)
        out[m] = [packing.tcn_block_to_kmajor(b) for b in blocks]
    return out


def _worst(got, ref, bound):
    return EH.ratio(got, ref, bound).max().item()


def _unstore_ragged_tile(t):
    t = t.clone().view(-1, t.shape[-1])
    t[(t.shape[0] // 128) * 128:] = 0
    return t.view(B, T, -1)


def _tcn_faults(blk, x, h1, ref1, ref2):
    """{(launch, fault name): faulty output} for one block; x, h1 the launch inputs."""
    k, d, cin, cout = blk["kernel_size"], blk["dilation"], blk["c_in"], blk["c_out"]
    out = {}
    if d >= 2 and k >= 2:
        shifts = [(k - 1 - j) * d for j in range(k)]
        shifts[0] = (k - 1) * (d // 2)                                        # the widest tap at dilation d/2
        out[1, "tap_half_dilation"] = EH.tcn_tc_launch1(blk, x, torch.float32, shifts=shifts)[0]
    leak = EH.tcn_tc_launch1(blk, x.reshape(1, B * T, cin), torch.float32)[0]  # padding reads the previous window
    out[1, "causal_padding_leak"] = leak.view(B, T, cout)
    m = copy.copy(blk)
    w1 = blk["w1"].clone()
    w1.view(cout, k, cin)[:, k - 1, :32] = 0                                   # last tap, first 32-channel K chunk
    m["w1"] = w1
    out[1, "k_chunk_dropped"] = EH.tcn_tc_launch1(m, x, torch.float32)[0]
    out[1, "ragged_tile_unstored"] = _unstore_ragged_tile(ref1)
    out[2, "ragged_tile_unstored"] = _unstore_ragged_tile(ref2)
    if blk["wd"] is not None:
        m = dict(blk, bd=torch.zeros_like(blk["bd"]))
        out[2, "ds_bias_dropped"] = EH.tcn_tc_launch2(m, x, h1, torch.float32)[0]
    if blk["post_scale"] is not None:
        s, t = blk["post_scale"].clone(), blk["post_shift"].clone()
        s[:32], t[:32] = 1, 0
        out[2, "post_skipped_on_n_tile"] = EH.tcn_tc_launch2(dict(blk, post_scale=s, post_shift=t), x, h1, torch.float32)[0]
    x_late = F.pad(x, (0, 0, 1, 0))[:, :T]                                     # residual read one step off
    out[2, "residual_shifted"] = EH.tcn_tc_launch2(blk, x_late, h1, torch.float32)[0]
    if cout == 96:
        for launch, ref in ((1, ref1), (2, ref2)):
            t = ref.clone()
            t[..., 64:96] = 0
            out[launch, "cols_64_95_unwritten"] = t
    return out


def test_tcn_bounds_pass_standin_and_fail_each_fault():
    stacks = _stack(["video", "vggish", "bert"])
    stacks.update({"c96": _stack(["vggish"], {"vggish": [96, 96]}, bn=False)["vggish"]})
    g = torch.Generator().manual_seed(3)
    worst_standin, least_fault = 0.0, float("inf")
    seen = set()
    for name, blocks in stacks.items():
        x = torch.randn(B, T, blocks[0]["c_in"], generator=g)
        for i, blk in enumerate(blocks):
            h1, _ = EH.tcn_tc_launch1(blk, x, torch.float32)
            y, _ = EH.tcn_tc_launch2(blk, x, h1, torch.float32)
            ref1, b1 = EH.tcn_tc_launch1(blk, x)
            ref2, b2 = EH.tcn_tc_launch2(blk, x, h1)
            r1, r2 = _worst(h1, ref1, b1), _worst(y, ref2, b2)
            assert max(r1, r2) <= 1.0, f"{name} block {i}: stand-in exceeds the bound ({r1:.3f}, {r2:.3f})"
            worst_standin = max(worst_standin, r1, r2)
            for (launch, fault), got in _tcn_faults(blk, x, h1, ref1.float(), ref2.float()).items():
                r = _worst(got, *((ref1, b1) if launch == 1 else (ref2, b2)))
                assert r > FAULT_MIN, f"{name} block {i} launch {launch}: fault {fault} passes (worst ratio {r:.3g})"
                least_fault = min(least_fault, r)
                seen.add(fault)
            x = y
    assert seen == {"tap_half_dilation", "causal_padding_leak", "k_chunk_dropped", "ragged_tile_unstored",
                    "ds_bias_dropped", "post_skipped_on_n_tile", "residual_shifted", "cols_64_95_unwritten"}
    print(f"TCN tensor-core bound: worst stand-in ratio {worst_standin:.4f}, smallest fault ratio {least_fault:.3g}")


def _fusion_standin(fw, feats, fault=None):
    """emulate.fusion_packed in fp32 with one injected fault."""
    if fault is None:
        return emulate.fusion_packed(fw, feats)
    M, md, H = fw["n_modals"], fw["modal_dim"], fw["num_heads"]
    hd = md // H
    R = feats[0].shape[0]
    qkv = [f @ w + b for f, w, b in zip(feats, fw["wqkv"], fw["bqkv"])]
    q = torch.stack([t.view(R, H, 3, hd)[:, :, 0] for t in qkv], dim=2)
    k = torch.stack([t.view(R, H, 3, hd)[:, :, 1] for t in qkv], dim=2)
    v = torch.stack([t.view(R, H, 3, hd)[:, :, 2] for t in qkv], dim=2)
    if fault == "head1_reads_head0_k":
        k = k.clone()
        k[:, 1] = k[:, 0]
    s = q @ k.transpose(-1, -2) / hd ** 0.5
    if fault == "softmax_over_m_minus_1_keys":
        s = s.clone()
        s[..., -1] = -float("inf")
    att = torch.softmax(s, dim=-1)
    vals = att @ v if fault == "v_residual_dropped" else att @ v + v
    o = vals.reshape(R, -1) @ fw["wo"] + fw["bo"]
    if fault == "layernorm_unbiased_var":
        mu = o.mean(-1, keepdim=True)
        fused = (o - mu) / (o.var(-1, unbiased=True, keepdim=True) + 1e-5).sqrt() * fw["ln_g"] + fw["ln_b"]
    else:
        fused = F.layer_norm(o, (o.shape[-1],), fw["ln_g"], fw["ln_b"], 1e-5)
    return None, fused


FUSION_CONFIGS = {
    "reference": dict(mods=["video", "vggish", "bert"], n_out=7, heads=2),
    "four_32d_nout16": dict(mods=["vggish", "mfcc", "egemaps", "logmel"], n_out=16, heads=2),
}


@pytest.mark.parametrize("cfg", list(FUSION_CONFIGS))
def test_fusion_bounds_pass_standin_and_fail_each_fault(cfg):
    c = FUSION_CONFIGS[cfg]
    sd = synthetic.head_state_dict(1, c["mods"], output_dim=c["n_out"])
    fw = packing.pack_fusion(sd, c["mods"], 32, c["heads"])
    R, fr = 203, 5                                     # 40 full 5-frame groups and a partial one of 3
    g = torch.Generator().manual_seed(7)
    feats = [torch.randn(R, d, generator=g) for d in fw["dim"]]
    ref_f, bnd_f = EH.fusion_fused(fw, feats)
    logits, fused = _fusion_standin(fw, feats)
    ref_l, bnd_l = EH.fusion_logits(fw, feats[0], fused)
    worst = max(_worst(fused, ref_f, bnd_f), _worst(logits, ref_l, bnd_l))
    assert worst <= 1.0, f"fp32 stand-in exceeds the fusion bound: {worst}"

    faults = {f: _fusion_standin(fw, feats, f)[1] for f in
              ("v_residual_dropped", "softmax_over_m_minus_1_keys", "head1_reads_head0_k", "layernorm_unbiased_var")}
    lagged = [t.clone() for t in feats]
    for t in lagged:
        t[fr - 1::fr] = t[0::fr][:t[fr - 1::fr].shape[0]]          # the last frame of each group reads frame 0's inputs
    faults["frame_reads_frame0_inputs"] = emulate.fusion_packed(fw, lagged)[1]
    tail = fused.clone()
    tail[(R // fr) * fr:] = 0
    faults["partial_group_unstored"] = tail
    least = float("inf")
    for name, got in faults.items():
        r = _worst(got, ref_f, bnd_f)
        assert r > FAULT_MIN, f"{cfg}: fault {name} passes the fused bound (worst ratio {r:.3g})"
        least = min(least, r)
    logit_faults = {}
    if fw["dim"][1] == fw["dim"][0]:
        logit_faults["leader_from_modality_1"] = torch.cat([feats[1], fused], -1) @ fw["wr"] + fw["br"]
    br = fw["br"].clone()
    br[0] = 0
    logit_faults["classifier_bias_dropped"] = torch.cat([feats[0], fused], -1) @ fw["wr"] + br
    for name, got in logit_faults.items():
        r = _worst(got, ref_l, bnd_l)
        assert r > FAULT_MIN, f"{cfg}: fault {name} passes the logit bound (worst ratio {r:.3g})"
        least = min(least, r)
    print(f"fusion bound ({cfg}): worst stand-in ratio {worst:.4f}, smallest fault ratio {least:.3g}")


def _names(fname):
    src = open(os.path.join(ROOT, "feature_vs_text_compound_emotion_b200", "csrc", fname)).read()
    table = re.search(r"kHeadVariantNames\[\]\s*=\s*\{(.*?)\};", src, re.S)
    assert table, f"kHeadVariantNames not found in {fname}"
    return set(re.findall(r'"([^"]+)"', table.group(1)))


def test_every_head_variant_has_a_parity_case():
    from tests.test_gpu_head_launches import FP32_CASES, FUSION_CASES, TC_CASES
    selectable = _names("tcn_tc.cu") | _names("tcn.cu") | _names("fusion.cu")
    pinned = set()
    for case in list(TC_CASES) + list(FP32_CASES) + list(FUSION_CASES):
        pinned |= case["variants"]
    assert selectable == pinned, (f"without a parity case: {sorted(selectable - pinned)}; "
                                  f"not a kernel of the head sources: {sorted(pinned - selectable)}")
