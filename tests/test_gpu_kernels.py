"""GPU parity tests, kernel by kernel, through the C-ABI (libcer_b200.so).

Each CUDA kernel is compared with a plain PyTorch computation of the same op (F.conv2d etc. on the
bf16-rounded operands the kernel sees), so a failure points at one kernel.  Single convolutions: fp64
reference on the device, the kernel instantiation that ran pinned by name (cer_conv_last_variant), and
the per-element bound of tests/emulate.py (bound_ratio: one bf16 rounding plus 1e-4 of the rms) for bf16
outputs, 1e-4 of the rms for fp32 outputs.  Other kernels: fp32 references, 1e-4 absolute for fp32 heads.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from oracle import lfan_oracle as O
from tests import emulate

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _rel_err(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-6)).item()


def _conv_case(dev, n, H, W, cin, cout, ksize, stride, classes, prelu, residual, fp32, seed, n_alloc=None):
    """Runs one conv through cer_conv_forward -> (output, fp64 reference NHWC, name of the kernel that ran)."""
    from feature_vs_text_compound_emotion_b200 import _capi
    from feature_vs_text_compound_emotion_b200.engine import conv_forward
    g = torch.Generator().manual_seed(seed)
    pad = 1 if ksize == 3 else 0
    n_alloc = n_alloc or n
    x = torch.randn(n_alloc, H, W, cin, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(cout, ksize, ksize, cin, generator=g) * (ksize * ksize * cin) ** -0.5).to(torch.bfloat16).to(dev)
    bias = (0.5 * torch.randn(classes, cout, generator=g)).to(dev)
    alpha = (0.25 + 0.1 * torch.randn(cout, generator=g)).to(dev) if prelu else None
    Ho, Wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    res = torch.randn(n, Ho, Wo, cout, generator=g).to(torch.bfloat16).to(dev) if residual else None
    # fp64 reference on the same bf16-rounded operands
    y = F.conv2d(x[:n].double().permute(0, 3, 1, 2), w.double().permute(0, 3, 1, 2), None, stride, pad)
    if classes == 9:
        y = y + bias.double()[emulate.border_class_map(Ho, Wo).to(dev)].permute(2, 0, 1).unsqueeze(0)
    else:
        y = y + bias.double().view(1, -1, 1, 1)
    if prelu:
        y = torch.where(y >= 0, y, y * alpha.double().view(1, -1, 1, 1))
    y = y.permute(0, 2, 3, 1)
    if residual:
        y = y + res.double()
    out = conv_forward(x, w.reshape(cout, -1), bias, ksize, stride, pad, alpha=alpha, res=res, out_fp32=fp32, n_frames=n)
    torch.cuda.synchronize()
    return out, y, _capi.lib().cer_conv_last_variant().decode()


def _assert_conv_within_bound(out, ref, fp32):
    if fp32:
        err = (out.double() - ref).abs().max().item()
        assert err <= emulate.C_RMS * ref.pow(2).mean().sqrt().item(), f"max abs error {err}"
    else:
        worst = emulate.bound_ratio(out, ref).max().item()
        assert worst <= 1.0, f"worst ratio to the bound {worst}"


# (n, H, W, cin, cout, ksize, stride, classes, prelu, residual, fp32, kernel instantiation it selects)
CONV_CASES = [
    (3, 10, 10, 256, 256, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,1>"),     # stage-3 conv1, ragged M = 300
    (3, 10, 10, 256, 256, 3, 1, 1, False, True, False, "conv_igemm_kernel<64,8,0,0>"),      # stage-3 conv2 + residual, BN narrowed
    (2, 40, 40, 64, 64, 3, 1, 9, True, False, False, "conv_igemm_kernel<64,8,0,0>"),        # stage-1 conv1, too few tiles for halo
    (2, 40, 40, 64, 128, 3, 1, 9, True, False, False, "conv_igemm_kernel<128,6,0,0>"),      # widening conv1
    (2, 40, 40, 128, 128, 3, 2, 1, False, False, False, "conv_igemm_kernel<64,8,0,0>"),     # stride-2 conv2
    (5, 20, 20, 128, 128, 3, 1, 1, False, True, False, "conv_igemm_kernel<64,8,0,0>"),      # stage 2
    (7, 5, 5, 512, 512, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,1>"),       # stage 4: 25 px/frame, tiles span frames, 2 n-tiles
    (4, 10, 10, 256, 512, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,1>"),     # widening to 512
    (4, 10, 10, 512, 512, 3, 2, 1, False, False, False, "conv_igemm_kernel<128,6,0,1>"),    # stride-2 at 10x10 -> 5x5
    (3, 40, 40, 64, 128, 1, 2, 1, False, False, False, "conv_igemm_kernel<64,8,0,0>"),      # 1x1 stride-2 projection alone
    (130, 1, 1, 12800, 512, 1, 1, 1, False, False, True, "conv_igemm_kernel<128,6,0,0>"),   # the FC head as a 1x1 conv, fp32 out, 2 m-tiles
    (1, 5, 5, 512, 512, 3, 1, 9, True, True, False, "conv_igemm_kernel<256,4,0,1>"),        # a single frame (tiny tensor: driver-quirk path)
    (48, 40, 40, 64, 64, 3, 1, 9, True, False, False, "conv_strip_kernel"),                 # 600 tiles >= 2 waves
    (48, 40, 40, 64, 64, 3, 1, 1, False, True, False, "conv_strip_kernel"),                 # same with residual epilogue
    (48, 40, 40, 64, 128, 3, 1, 9, True, False, False, "conv_halo_kernel<128>"),            # Cout = 128
    (49, 40, 40, 64, 64, 3, 1, 9, True, False, False, "conv_strip_kernel"),                 # odd frame count: the last tile is half empty
    (49, 40, 40, 64, 64, 3, 1, 1, False, True, False, "conv_strip_kernel"),                 # same with residual
    (21, 56, 56, 64, 64, 3, 1, 9, True, False, False, "conv_strip_kernel"),                 # 56-row map: tiles cross strips and frames mid-tile
    (800, 10, 10, 256, 256, 3, 1, 9, True, False, False, "conv_igemm2_kernel<256,6>"),      # 625 tiles (odd): ragged last CTA pair
    (800, 10, 10, 256, 256, 3, 1, 1, False, True, False, "conv_igemm2_kernel<256,6>"),      # CTA pair with residual epilogue
    (200, 20, 20, 128, 128, 3, 1, 9, True, False, False, "conv_igemm2_bres_kernel<128,4,18>"),  # CTA pair, weights resident
    (1530, 5, 5, 512, 512, 3, 1, 9, True, False, False, "conv_igemm2_kernel<256,6>"),       # CTA pair, two n-tiles, tiles span frames
    (198, 12, 16, 64, 64, 3, 1, 9, True, False, False, "conv_halo_kernel<64>"),             # H % 8 != 0: no strip; ragged 16-row band
    (190, 20, 20, 64, 64, 3, 1, 9, True, False, False, "conv_igemm_kernel<64,9,1,1>"),      # W % 8 != 0: no halo; weights resident
    (190, 20, 20, 64, 128, 3, 1, 9, True, False, False, "conv_igemm_kernel<128,4,1,0>"),    # same, Cout = 128
    (95, 10, 10, 64, 256, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,0>"),     # 9 k-steps: not a multiple of 4
    (3, 5, 5, 512, 64, 3, 1, 9, True, False, False, "conv_igemm_kernel<64,8,0,1>"),         # 72 k-steps, BN = 64
    (758, 10, 10, 256, 128, 3, 1, 9, True, False, False, "conv_igemm2_kernel<128,6>"),      # CTA pair, 36 k-steps, BN = 128
    (7, 6, 10, 256, 256, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,1>"),      # non-square map, 9-class bias
]


def _conv_id(c):
    hw = "h%d" % c[1] if c[1] == c[2] else "h%dw%d" % (c[1], c[2])
    return "n%d_%s_%dto%d_k%ds%d_c%d%s%s%s" % (c[0], hw, c[3], c[4], c[5], c[6], c[7], "_prelu" if c[8] else "",
                                              "_res" if c[9] else "", "_f32" if c[10] else "")


@pytest.mark.parametrize("case", CONV_CASES, ids=_conv_id)
def test_conv_igemm_matches_conv2d(case):
    dev = _dev()
    *shape, variant = case
    out, ref, ran = _conv_case(dev, *shape, seed=11)
    assert ran == variant
    _assert_conv_within_bound(out, ref, shape[-1])


# (n_alloc, case): the tensor-map extent holds more frames than the pass computes (the plan's layout)
PADDED_CASES = [
    (11, (3, 10, 10, 256, 256, 3, 1, 9, True, False, False, "conv_igemm_kernel<256,4,0,1>")),
    (806, (799, 10, 10, 256, 256, 3, 1, 9, True, False, False, "conv_igemm2_kernel<256,6>")),    # ragged last CTA pair
]


def test_conv_igemm_padded_allocation_matches():
    """Same layers with the tensor-map extent larger than the valid frames (the plan's layout)."""
    dev = _dev()
    for n_alloc, (*shape, variant) in PADDED_CASES:
        out, ref, ran = _conv_case(dev, *shape, seed=12, n_alloc=n_alloc)
        assert ran == variant
        _assert_conv_within_bound(out, ref, shape[-1])


def test_stem_and_units_progressively():
    """Stem, then the output of selected residual units, against the packed-weight emulation
    (which tests/test_packing.py ties to the oracle)."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    sd = synthetic.visual_backbone_state_dict(0)
    pk = packing.pack_ir50(sd, "backbone.")
    x = synthetic.frames(5, seed=21)
    _, taps = emulate.ir50_packed(pk, x, round_act=True)
    eng = Ir50Engine(pk, dev, frames_per_pass=16)
    for unit in (-1, 0, 2, 3, 6, 7, 8, 20, 21, 23):
        got = eng.debug_activation(x.to(dev), unit)
        torch.cuda.synchronize()
        err = _rel_err(got, taps[unit])
        assert err < 3e-2, f"unit {unit}: relative error {err}"


def test_raster_stage_matches_im2col_plan(monkeypatch):
    """IR-50 stage 2 on the padded-raster kernel (passes with enough frames; conv_raster.cuh) against the same
    plan with CER_RASTER=0 (im2col pair kernel): the unit in front of the stage (stores the padded raster), the
    stage's units (the last one stores dense NHWC again), the unit behind it and the embeddings.  The two
    differ only in the order the 1152 products of an output are accumulated in fp32."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    sd = synthetic.visual_backbone_state_dict(0)
    pk = packing.pack_ir50(sd, "backbone.")
    n = 199                                   # odd count: the last pair tile is ragged, frames end mid-tile
    x = synthetic.frames(8, seed=23).repeat(25, 1, 1, 1)[:n].contiguous()
    x = (x + 0.05 * torch.randn(x.shape, generator=torch.Generator().manual_seed(24))).to(dev)
    monkeypatch.setenv("CER_RASTER", "0")
    ref = Ir50Engine(pk, dev, frames_per_pass=256)
    monkeypatch.delenv("CER_RASTER")
    eng = Ir50Engine(pk, dev, frames_per_pass=256)
    assert ref.op_variant(2 * 4, n).startswith("conv_igemm2_bres_kernel")
    assert eng.op_variant(0, n) == ref.op_variant(0, n) == "conv_strip_kernel"          # 64 -> 64 stays on the strip kernel
    assert [eng.op_variant(op, n) for op in range(2 * 4, 2 * 7)] == ["conv_raster2_kernel<128,3,18,176>"] * 6
    assert not eng.op_variant(2 * 4, 64).startswith("conv_raster2")          # small passes keep the im2col plan
    assert eng.launches(n) == ref.launches(n) + 1                               # + raster_zero_pads_kernel
    for unit in (2, 3, 4, 5, 6, 7):
        a = ref.debug_activation(x, unit).float()
        b = eng.debug_activation(x, unit).float()
        torch.cuda.synchronize()
        assert a.shape == b.shape
        scale = a.abs().max().item()
        assert (a - b).abs().max().item() <= 0.02 * scale, f"unit {unit}"
        assert (a - b).abs().mean().item() <= 2e-3 * a.abs().mean().item(), f"unit {unit}"
    ea, eb = ref.forward(x), eng.forward(x)
    assert F.cosine_similarity(ea, eb, dim=1).min().item() >= 0.9999
    # a second, smaller pass through the same plan leaves no stale pad data behind
    small = eng.forward(x[:7])
    assert F.cosine_similarity(small, ea[:7], dim=1).min().item() >= 0.9999
    again = eng.forward(x)
    assert torch.equal(again, eb)


def test_ir50_embedding_vs_golden(golden_dir):
    import os
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    g = torch.load(os.path.join(golden_dir, "ir50_n4.pt"))
    sd = synthetic.visual_backbone_state_dict(g["weights_seed"])
    eng = Ir50Engine(packing.pack_ir50(sd, "backbone."), dev, frames_per_pass=8)
    emb = eng.forward(synthetic.frames(g["n"], seed=g["x_seed"]).to(dev)).cpu()
    cos = F.cosine_similarity(emb, g["emb"], dim=1)
    assert cos.min().item() >= 0.999, cos          # BASELINE.json tolerance
    assert torch.allclose(emb.norm(dim=1), torch.ones(4), atol=1e-4)


@pytest.mark.parametrize("n,fpp", [(1, 8), (13, 8), (37, 16), (64, 64)])
def test_ir50_passes_and_ragged_counts(n, fpp):
    """n not a multiple of the pass size / tile size gives the same rows as one big pass."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    sd = synthetic.visual_backbone_state_dict(0)
    pk = packing.pack_ir50(sd, "backbone.")
    x = synthetic.frames(n, seed=31).to(dev)
    a = Ir50Engine(pk, dev, frames_per_pass=fpp).forward(x)
    b = Ir50Engine(pk, dev, frames_per_pass=128).forward(x)
    torch.cuda.synchronize()
    # frames are independent: identical arithmetic per frame regardless of batching
    assert torch.equal(a, b)
    ref = O.ir50_forward(sd, x[: min(n, 4)].cpu(), "backbone.")
    assert F.cosine_similarity(a[: min(n, 4)].cpu(), ref, dim=1).min().item() >= 0.999


@pytest.mark.parametrize("precision,tol", [("tf32", 5e-3), ("fp32", 1e-4)])
@pytest.mark.parametrize("modal,B,T", [("vggish", 2, 300), ("cnn_res50", 1, 300), ("bert", 3, 77), ("vggish", 1, 5)])
def test_tcn_stack_vs_oracle(modal, B, T, precision, tol):
    """4 TemporalBlocks + folded BatchNorm1d.  tf32 = tcgen05 kind::tf32 kernel (10-bit mantissa
    products, fp32 accumulate: tolerance 5e-3 on O(1) activations); fp32 = CUDA-core kernel."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import TcnEngine
    sd = synthetic.head_state_dict(2, [modal])
    x = torch.randn(B, T, synthetic.EMBEDDING_DIM[modal], generator=torch.Generator().manual_seed(5))
    want = O._bn_eval(sd, f"bn.{modal}", O.tcn_forward(sd, f"temporal.{modal}.", x.transpose(1, 2))).transpose(1, 2)
    eng = TcnEngine(packing.pack_tcn(sd, f"temporal.{modal}.", f"bn.{modal}"), dev, precision=precision)
    got = eng.forward(x.to(dev)).cpu()
    assert (got - want).abs().max().item() < tol * max(1.0, want.abs().max().item())


def test_fusion_head_vs_oracle():
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import FusionEngine
    mods = ["cnn_res50", "vggish", "bert"]
    sd = synthetic.lfan_state_dict(4, mods)
    g = torch.Generator().manual_seed(9)
    rows = 603                                  # not a multiple of the 4-frame warp group
    feats = [torch.randn(rows, d, generator=g) for d in (128, 32, 128)]
    enc = {m: f.view(1, rows, -1) for m, f in zip(mods, feats)}
    fused = O.fusion_forward(sd, "fusion.", enc, mods)
    want = F.linear(torch.cat((enc[mods[0]], fused), -1), sd["regressor.weight"], sd["regressor.bias"])[0]
    eng = FusionEngine(packing.pack_fusion(sd, mods, 32, 2), dev)
    logits, fz = eng.forward([f.to(dev) for f in feats], want_fused=True)
    assert (fz.cpu() - fused[0]).abs().max().item() < 1e-4
    assert (logits.cpu() - want).abs().max().item() < 1e-4


def test_stitch_windows_vs_oracle():
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import stitch_windows
    L = 701
    wins = O.windowing(L, 300, 200)
    g = torch.Generator().manual_seed(3)
    wl = torch.randn(len(wins), 300, 7, generator=g)
    out = torch.zeros(L, 7)
    cnt = torch.zeros(L)
    for i, w in enumerate(wins):
        out[w] += wl[i]
        cnt[w] += 1
    want = out / cnt.view(-1, 1)
    starts = torch.tensor([int(w[0]) for w in wins], dtype=torch.int32)
    got = stitch_windows(wl.to(dev), starts.to(dev), L).cpu()
    assert (got - want).abs().max().item() < 1e-6


def test_preprocess_bit_exact_vs_reference_golden(golden_dir):
    """uint8 stored crops -> fp32 NCHW through cer_preproc_forward: integer pipeline, so the bar is
    bit-exact against the reference transform (real Pillow) for square, non-square and up-scaled inputs."""
    import os
    from feature_vs_text_compound_emotion_b200.engine import PreprocEngine
    dev = _dev()
    g = torch.load(os.path.join(golden_dir, "eval_transform.pt"))
    for name, c in g["cases"].items():
        raw = synthetic.raw_frames_u8(c["n"], seed=c["seed"], h=c["h"], w=c["w"])
        eng = PreprocEngine(c["h"], c["w"], dev)
        out = eng.forward(raw.to(dev)).cpu()
        assert torch.equal(out, c["out"]), (name, (out - c["out"]).abs().max().item())


def test_preprocess_many_frames_vs_oracle():
    from feature_vs_text_compound_emotion_b200.engine import PreprocEngine
    dev = _dev()
    raw = synthetic.raw_frames_u8(37, seed=77)
    raw[0] = 0
    raw[1] = 255
    out = PreprocEngine(256, 256, dev).forward(raw.to(dev)).cpu()
    assert torch.equal(out, O.eval_transform(raw.numpy()))
    assert out[0].eq(-1).all() and out[1].eq(1).all()


def test_logmel_front_end_vs_reference_golden(golden_dir):
    """Waveform -> log-mel -> VGGish examples on the device (fp64 DFT) against the reference's
    numpy code: 2e-5 absolute on log-mel values (fp32 output, fp32 fixture)."""
    import os
    from feature_vs_text_compound_emotion_b200.engine import LogMelEngine
    dev = _dev()
    g = torch.load(os.path.join(golden_dir, "logmel.pt"))
    wave = synthetic.waveform(g["seconds"], seed=g["seed"])
    eng = LogMelEngine(dev)
    lm = eng.log_mel(wave.to(dev)).cpu()
    assert lm.shape == g["log_mel"].shape
    assert (lm - g["log_mel"]).abs().max().item() < 2e-5
    ex = eng.examples(wave.to(dev), 0.96, g["hop_sec"]).cpu()
    assert ex.shape == (g["n_examples"], 96, 64)
    assert (ex[7] - g["example_7"]).abs().max().item() < 2e-5
    assert (ex[-1] - g["example_last"]).abs().max().item() < 2e-5
    assert (ex.double().sum(dim=(1, 2)) - g["example_sum"]).abs().max().item() < 5e-2
    # the examples feed VGGish directly
    want = torch.from_numpy(O.waveform_to_examples(wave.double().numpy(), 0.96, g["hop_sec"])).float()
    assert (ex - want).abs().max().item() < 2e-5


def test_c_abi_error_paths_report_status_and_message():
    """Bad arguments come back as negative cer_status + cer_last_error(), never as a crash or a silent
    fallback (include/cer_b200.h conventions)."""
    import ctypes as C
    from feature_vs_text_compound_emotion_b200 import _capi
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine, conv_forward
    dev = _dev()
    lib = _capi.lib()
    x = torch.zeros(2, 8, 8, 32, dtype=torch.bfloat16, device=dev)            # Cin = 32: not a multiple of 64
    w = torch.zeros(64, 9 * 32, dtype=torch.bfloat16, device=dev)
    with pytest.raises(_capi.CerError, match="multiples of 64"):
        conv_forward(x, w, torch.zeros(1, 64, device=dev), 3, 1, 1)
    assert lib.cer_ce_loss(None, None, 10, 7, None, None, None) == -1 and b"cer_ce_loss" in lib.cer_last_error()
    assert lib.cer_optimizer_step(5, None, None, None, None, 0, 0.1, 0.0, 0.9, 0.0, 1e-8, 0, 1, 1.0, None) == -1
    # workspace too small
    pk = packing.pack_ir50(synthetic.visual_backbone_state_dict(0))
    eng = Ir50Engine(pk, dev, frames_per_pass=8)
    h = C.c_void_p()
    ws = torch.empty(1024, dtype=torch.uint8, device=dev)
    rc = lib.cer_ir50_create(C.byref(h), C.byref(eng._w), 8, ws.data_ptr(), 1024)
    assert rc == -4 and b"workspace" in lib.cer_last_error()
    # shape checks of the Python mirrors
    with pytest.raises(ValueError):
        eng.forward(torch.zeros(2, 3, 32, 32, device=dev))
    with pytest.raises(ValueError):
        eng.forward(torch.zeros(2, 3, 40, 40))                               # CPU tensor


def test_head_building_blocks_vs_torch():
    """cer_linear_forward / cer_softmax_gate / cer_add_layernorm (exact fp32) and both attention kernels --
    cer_sdpa_forward (fp32 CUDA cores) and cer_sdpa_tc_forward (TF32 tensor-core flash attention) --
    against plain PyTorch fp32 on the CPU: ragged lengths, several batches, operands that are column slices
    of a packed projection (row pitch 3E), E = 128 and 64."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200 import engine as E
    g = torch.Generator().manual_seed(31)
    x = torch.randn(333, 200, generator=g)
    w, b = torch.randn(96, 200, generator=g) * 0.1, torch.randn(96, generator=g)
    for act, f in ((None, lambda t: t), ("leaky_relu", F.leaky_relu), ("relu", F.relu)):
        got = E.linear(x.to(dev), w.to(dev), b.to(dev), act).cpu()
        assert (got - f(x @ w.t() + b)).abs().max().item() < 1e-4, act
    wide = torch.zeros(333, 256, device=dev)
    E.linear(x.to(dev), w.to(dev), b.to(dev), out=wide[:, 128:224])                    # concat without a copy
    assert (wide[:, 128:224].cpu() - (x @ w.t() + b)).abs().max().item() < 1e-4 and float(wide[:, :128].abs().max()) == 0.0
    gate, feat = torch.randn(77, 384, generator=g), torch.randn(77, 384, generator=g)
    assert (E.softmax_gate(gate.to(dev), feat.to(dev)).cpu() - torch.softmax(gate, -1) * feat).abs().max().item() < 1e-6
    res = torch.randn(333, 96, generator=g)
    gam, bet = torch.rand(96, generator=g) + 0.5, torch.randn(96, generator=g)
    want = F.layer_norm(x @ w.t() + res, (96,), gam, bet, 1e-5)
    got = E.add_layernorm((x @ w.t()).to(dev), res.to(dev), gam.to(dev), bet.to(dev)).cpu()
    assert (got - want).abs().max().item() < 1e-4
    for (e, batch, lq, lk) in ((128, 2, 300, 300), (128, 1, 600, 600), (128, 3, 37, 91), (64, 2, 65, 130), (128, 1, 1, 1)):
        qkv = torch.randn(batch * max(lq, lk), 3 * e, generator=g)
        q, k, v = qkv[:batch * lq, :e], qkv[:batch * lk, e:2 * e], qkv[:batch * lk, 2 * e:]
        want = F.scaled_dot_product_attention(q.reshape(batch, lq, e), k.reshape(batch, lk, e), v.reshape(batch, lk, e)).reshape(-1, e)
        qd = qkv.to(dev)
        qs, ks, vs = qd[:batch * lq, :e], qd[:batch * lk, e:2 * e], qd[:batch * lk, 2 * e:]
        exact = E.sdpa(qs, ks, vs, batch, lq, lk, precision="fp32").cpu()
        assert (exact - want).abs().max().item() < 2e-5, (e, batch, lq, lk)
        tc = E.sdpa(qs, ks, vs, batch, lq, lk, precision="tf32").cpu()
        assert (tc - want).abs().max().item() < 5e-3, (e, batch, lq, lk, (tc - want).abs().max().item())
        assert not torch.equal(tc, exact) or lk == 1                                    # the tensor-core kernel did run
