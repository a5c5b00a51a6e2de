"""The head kernels launch by launch against fp64 references on the device (tests/emulate_head.py).

  * TCN on the tensor cores (cer_tcn_block_tc_forward): every block of a stack is driven on its own with the
    TcnEngine's packed blocks; both launches of the block are checked, launch 2 from the h1 the kernel stored
    in the workspace, so errors do not compound across launches or blocks.
  * TCN on the CUDA cores (cer_tcn_block_forward): each block against an fp64 block.
  * Fusion head (cer_fusion_head_forward, and the composed path FusionEngine uses when the weights do not fit
    in shared memory): fused features against the fp64 fusion path, logits against an fp64 classifier on
    cat(leader features, the kernel's fused features).
Every case pins the exact set of kernel instantiations it launches (cer_head_last_variant);
tests/test_head_parity_guards.py checks that together they cover every instantiation of the head sources.
Run with -s to see the worst ratio to the bound per case and launch.
"""
import ctypes as C

import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate_head as EH

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

TC64, TC32 = "tcn_igemm_kernel<64,8>", "tcn_igemm_kernel<32,8>"


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _lib():
    from feature_vs_text_compound_emotion_b200 import _capi
    return _capi


def _variant():
    return _lib().lib().cer_head_last_variant().decode()


def _on(packed, dev):
    """A packed block / fusion dict with its tensors (and lists of tensors) on `dev`."""
    def mv(v):
        return v.to(dev) if torch.is_tensor(v) else [mv(t) for t in v] if isinstance(v, list) else v
    return {k: mv(v) for k, v in packed.items()}


def _blocks(mod, channels, k, bn, seed=0):
    sd = synthetic.head_state_dict(seed, [mod], kernel_size=k, tcn_channels={mod: channels or synthetic.TCN_CHANNELS[mod]})
    return packing.pack_tcn(sd, f"temporal.{mod}.", f"bn.{mod}" if bn else None)


# name, modality (input width), channels (None: the reference's), kernel size, B, T, BN post, variants
TC_CASES = [
    dict(name="bench_video", mod="video", ch=None, k=5, B=8, T=300, bn=True, variants={TC64}),
    dict(name="bench_vggish", mod="vggish", ch=None, k=5, B=8, T=300, bn=True, variants={TC64, TC32}),
    dict(name="bench_bert", mod="bert", ch=None, k=5, B=8, T=300, bn=True, variants={TC64}),
    dict(name="tiles_b3_t77", mod="vggish", ch=None, k=5, B=3, T=77, bn=True, variants={TC64, TC32}),
    dict(name="tiles_window_aligned", mod="vggish", ch=None, k=5, B=2, T=128, bn=True, variants={TC64, TC32}),
    dict(name="halo_exceeds_T", mod="vggish", ch=None, k=5, B=1, T=5, bn=True, variants={TC64, TC32}),
    dict(name="single_step", mod="vggish", ch=None, k=5, B=1, T=1, bn=True, variants={TC64, TC32}),
    dict(name="padded_mfcc_39", mod="mfcc", ch=None, k=5, B=3, T=100, bn=True, variants={TC32}),
    dict(name="padded_egemaps_88", mod="egemaps", ch=None, k=5, B=3, T=100, bn=True, variants={TC32}),
    dict(name="cout_96_160_512", mod="vggish", ch=[96, 96, 160, 160, 512], k=5, B=3, T=300, bn=True, variants={TC64, TC32}),
    dict(name="k1", mod="vggish", ch=None, k=1, B=2, T=300, bn=True, variants={TC64, TC32}),
    dict(name="k3", mod="vggish", ch=None, k=3, B=2, T=300, bn=True, variants={TC64, TC32}),
    dict(name="k8", mod="vggish", ch=None, k=8, B=2, T=300, bn=True, variants={TC64, TC32}),
    dict(name="five_blocks_video", mod="video", ch=synthetic.TCN_SETTINGS["video"]["channel"], k=5, B=8, T=300, bn=True,
         variants={TC64}),
    dict(name="five_blocks_logmel", mod="logmel", ch=synthetic.TCN_SETTINGS["logmel"]["channel"], k=5, B=8, T=300, bn=True,
         variants={TC64}),
    dict(name="largest_halo_128", mod="vggish", ch=[64, 32, 32, 32, 32, 32], k=5, B=2, T=300, bn=True,
         variants={TC64, TC32}),
]


def _run_tc(case, dev, tf32=None):
    """-> (kernel names, [(block, worst launch-1 ratio, worst launch-2 ratio)])."""
    from feature_vs_text_compound_emotion_b200.engine import TcnEngine
    _capi = _lib()
    blocks = _blocks(case["mod"], case["ch"], case["k"], case["bn"])
    eng = TcnEngine(blocks, dev)
    kms = [_on(packing.tcn_block_to_kmajor(b), dev) for b in blocks]
    B, T = case["B"], case["T"]
    g = torch.Generator().manual_seed(17)
    x = torch.randn(B, T, blocks[0]["c_in"], generator=g).to(dev)
    x = torch.nn.functional.pad(x, (0, kms[0]["c_in"] - blocks[0]["c_in"])).contiguous()
    ws = torch.empty(max(B * T * b["c_out"] for b in kms) * 4, dtype=torch.uint8, device=dev)
    stream = _capi.current_stream_ptr(dev)
    ran, worst = set(), []
    for i, (blk, kb) in enumerate(zip(eng.blocks, kms)):
        y = torch.full((B, T, kb["c_out"]), float("nan"), device=dev)
        ws.view(torch.float32).fill_(float("nan"))
        _capi.check(_capi.lib().cer_tcn_block_tc_forward(C.byref(blk), x.data_ptr(), y.data_ptr(), B, T, ws.data_ptr(),
                                                         ws.numel(), stream), "cer_tcn_block_tc_forward")
        ran.add(_variant())
        h1 = ws[:B * T * kb["c_out"] * 4].view(torch.float32).view(B, T, kb["c_out"]).clone()
        ref1, bnd1 = EH.tcn_tc_launch1(kb, x, tf32=tf32)
        ref2, bnd2 = EH.tcn_tc_launch2(kb, x, h1, tf32=tf32)
        worst.append((i, EH.ratio(h1, ref1, bnd1).max().item(), EH.ratio(y, ref2, bnd2).max().item()))
        x = y
    return ran, worst


@pytest.mark.parametrize("case", TC_CASES, ids=[c["name"] for c in TC_CASES])
def test_tcn_tc_launches(case):
    dev = _dev()
    ran, worst = _run_tc(case, dev)
    print(f"\n{case['name']}: " + "  ".join(f"b{i} L1 {a:.3f} L2 {b:.3f}" for i, a, b in worst))
    assert ran == case["variants"]
    for i, a, b in worst:
        assert a <= 1.0 and b <= 1.0, f"block {i}: worst ratio to the bound launch 1 {a:.4g}, launch 2 {b:.4g}"


def test_tf32_operand_convention():
    """The pinned TF32 conversion (EH.TF32_OPERAND) bounds the kernel on the benchmark's video stack; the other
    convention does not, so the pin is a measurement and not a choice."""
    dev = _dev()
    case = dict(TC_CASES[0])
    _, pinned = _run_tc(case, dev)
    _, other = _run_tc(case, dev, tf32=EH.TF32_OTHER)
    worst_pinned = max(max(a, b) for _, a, b in pinned)
    worst_other = max(max(a, b) for _, a, b in other)
    print(f"\nTF32 convention: pinned {worst_pinned:.3f}, other {worst_other:.3f}")
    assert worst_pinned <= 1.0 < worst_other


def test_tcn_tc_refuses_halo_above_128_before_launching():
    """(k-1) d = 129: one past the rank-4 im2col corner range.  Refused with CerError; no kernel is launched."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import TcnEngine
    _capi = _lib()
    eng = TcnEngine(_blocks("vggish", [64], 2, False), dev)
    x = torch.randn(1, 300, 128, device=dev)
    eng.forward(x)
    torch.cuda.synchronize()
    before = _variant()
    blk = eng.blocks[0]
    blk.dilation = 129
    y = torch.empty(1, 300, 64, device=dev)
    ws = torch.empty(300 * 64 * 4, dtype=torch.uint8, device=dev)
    with pytest.raises(_capi.CerError, match="at most 128"):
        _capi.check(_capi.lib().cer_tcn_block_tc_forward(C.byref(blk), x.data_ptr(), y.data_ptr(), 1, 300, ws.data_ptr(),
                                                         ws.numel(), _capi.current_stream_ptr(dev)), "cer_tcn_block_tc_forward")
    torch.cuda.synchronize()
    assert _variant() == before == TC64


def _fp32_names(c):
    return {f"tcn_block_kernel<{c},{d},5>" for d in (1, 2, 4, 8)}


FP32_CASES = [dict(name=f"c{c}_b8_t300", ch=[c] * 4, B=8, T=300, variants=_fp32_names(c)) for c in (32, 64, 128, 256)]
FP32_CASES.append(dict(name="c128_b3_t77", ch=[128] * 4, B=3, T=77, variants=_fp32_names(128)))


@pytest.mark.parametrize("case", FP32_CASES, ids=[c["name"] for c in FP32_CASES])
def test_tcn_fp32_launches(case):
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import TcnEngine
    _capi = _lib()
    blocks = _blocks("vggish", case["ch"], 5, True)
    eng = TcnEngine(blocks, dev, precision="fp32")
    B, T = case["B"], case["T"]
    x = torch.randn(B, T, 128, generator=torch.Generator().manual_seed(19)).to(dev)
    ran, worst = set(), []
    for blk, tb in zip(eng.blocks, blocks):
        y = torch.full((B, T, tb["c_out"]), float("nan"), device=dev)
        _capi.check(_capi.lib().cer_tcn_block_forward(C.byref(blk), x.data_ptr(), y.data_ptr(), B, T, None, 0,
                                                      _capi.current_stream_ptr(dev)), "cer_tcn_block_forward")
        ran.add(_variant())
        ref, bnd = EH.tcn_fp32_block(_on(tb, dev), x)
        worst.append(EH.ratio(y, ref, bnd).max().item())
        x = y
    print(f"\n{case['name']}: " + "  ".join(f"b{i} {r:.3f}" for i, r in enumerate(worst)))
    assert ran == case["variants"]
    assert max(worst) <= 1.0, worst


FUSION_CONFIGS = {
    "reference": dict(mods=["video", "vggish", "bert"], md=32, heads=2, n_out=7),
    "four_32d_e128_nout16": dict(mods=["vggish", "mfcc", "egemaps", "logmel"], md=32, heads=2, n_out=16),
    "one_modality": dict(mods=["video"], md=32, heads=2, n_out=7),
    "heads1": dict(mods=["video", "vggish", "bert"], md=32, heads=1, n_out=7),
    "heads4": dict(mods=["video", "vggish", "bert"], md=32, heads=4, n_out=7),
    "composed_md64": dict(mods=["video", "vggish", "bert"], md=64, heads=2, n_out=7),
}


def _rows_for_fr(fr, sms):
    """A row count that selects kFR = fr (rows in (4 sms (fr-1), 4 sms fr]) and is not a multiple of fr."""
    r = 4 * sms * (fr - 1) + 2 * sms + 1
    while r % fr == 0:
        r += 1
    return r


# rows: an int, or ("fr", n) for the count that selects kFR = n on this device; variants: the fused kernel
# instantiation it launches (2400 rows select kFR = 5 on the B200's 148 SMs), empty for the composed path
FUSION_CASES = [dict(name=f"reference_fr{fr}", cfg="reference", rows=("fr", fr), variants={f"fusion_head_kernel<{fr}>"})
                for fr in (4, 5, 6, 7)]
FUSION_CASES += [
    dict(name="four_32d_fr8", cfg="four_32d_e128_nout16", rows=("fr", 8), variants={"fusion_head_kernel<8>"}),
    dict(name="reference_2400", cfg="reference", rows=2400, variants={"fusion_head_kernel<5>"}),
    dict(name="reference_1", cfg="reference", rows=1, variants={"fusion_head_kernel<4>"}),
    dict(name="reference_3", cfg="reference", rows=3, variants={"fusion_head_kernel<4>"}),
    dict(name="one_modality_2400", cfg="one_modality", rows=2400, variants={"fusion_head_kernel<5>"}),
    dict(name="heads1_603", cfg="heads1", rows=603, variants={"fusion_head_kernel<4>"}),
    dict(name="heads4_603", cfg="heads4", rows=603, variants={"fusion_head_kernel<4>"}),
    dict(name="composed_md64_2400", cfg="composed_md64", rows=2400, variants=set()),
]


@pytest.mark.parametrize("case", FUSION_CASES, ids=[c["name"] for c in FUSION_CASES])
def test_fusion_launches(case):
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import FusionEngine
    c = FUSION_CONFIGS[case["cfg"]]
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    rows = _rows_for_fr(case["rows"][1], sms) if isinstance(case["rows"], tuple) else case["rows"]
    sd = synthetic.head_state_dict(2, c["mods"], output_dim=c["n_out"], modal_dim=c["md"])
    fw = packing.pack_fusion(sd, c["mods"], c["md"], c["heads"])
    eng = FusionEngine(fw, dev)
    assert eng.composed == (not case["variants"])
    g = torch.Generator().manual_seed(23)
    feats = [torch.randn(rows, d, generator=g).to(dev) for d in fw["dim"]]
    before = _variant()
    logits, fused = eng.forward(feats, want_fused=True)
    after = _variant()
    if case["variants"]:
        assert {after} == case["variants"]
    else:
        assert after == before                      # the fused kernel did not run
    fwd = _on(fw, dev)
    ref_f, bnd_f = EH.fusion_fused(fwd, feats)
    ref_l, bnd_l = EH.fusion_logits(fwd, feats[0], fused)
    rf, rl = EH.ratio(fused, ref_f, bnd_f).max().item(), EH.ratio(logits, ref_l, bnd_l).max().item()
    print(f"\n{case['name']} ({rows} rows, {after if case['variants'] else 'composed'}): fused {rf:.3f} logits {rl:.3f}")
    assert rf <= 1.0 and rl <= 1.0, (rf, rl)
