"""Every unit of the IR-50 plan, isolated, against an fp64 reference of that one unit.

For each pass size, the plan's own bf16 output of unit i-1 (debug_activation) is the input of an fp64
reference of unit i (tests/emulate.py ir50_unit), and the plan's output of unit i must lie within the
per-element bound of emulate.bound_ratio:

    |got - ref| <= (1 + 2^-5) 2^-8 |ref| + E + 1e-4 rms(ref)

with E the envelope of conv1's intermediate bf16 rounding.  Isolating a unit keeps the budget at one rounding;
through 24 units it would compound, and a plan-level check (embedding cosine >= 0.999) lets a border-class,
K-loop or ragged-tile bug in one layer pass.  The stem is checked the same way (E = 0) against an fp64 conv of
TF32-rounded operands (cvt.rna, as stem_tc.cuh rounds them), the FC + L2 norm against an fp64 GEMM of the
plan's last unit output.

The pass sizes and plans are chosen so that each kernel the plan can select runs: the set of kernels each
case launches is pinned (PLAN_CASES[..]["variants"], read back through op_variant), and
tests/test_conv_parity_guards.py checks that these sets and tests/test_gpu_kernels.py together cover every
instantiation of csrc/ir50.cu.  At n == frames_per_pass, debug_activation runs exactly the forward's pass.
"""
import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from oracle.lfan_oracle import tf32_round
from tests import emulate

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

STRIP = "conv_strip_kernel"
HALO128 = "conv_halo_kernel<128>"
PAIR_BRES18 = "conv_igemm2_bres_kernel<128,4,18>"
PAIR_BRES19 = "conv_igemm2_bres_kernel<128,4,19>"
PAIR256 = "conv_igemm2_kernel<256,6>"
IGEMM256 = "conv_igemm_kernel<256,4,0,0>"
IGEMM256_ALIGNED = "conv_igemm_kernel<256,4,0,1>"
IGEMM128 = "conv_igemm_kernel<128,6,0,0>"
IGEMM128_ALIGNED = "conv_igemm_kernel<128,6,0,1>"
RASTER = "conv_raster2_kernel<128,3,18,176>"

# the benchmarked 40 px plan at >= 190 frames: stage 1 on the strip kernel, the widening conv1 on halo<128>,
# the stride-2 conv with fused projection on the pair kernel, stage 2 on the raster kernel, stage 3 and the
# widening into stage 4 on pair<256>, the rest on the one-CTA kernels, the FC (M = frames) on igemm<128,6>
_BENCH = frozenset({STRIP, HALO128, PAIR_BRES19, RASTER, PAIR256, IGEMM256, IGEMM256_ALIGNED, IGEMM128})
_NO_RASTER = (_BENCH - {RASTER}) | {PAIR_BRES18}

PLAN_CASES = [
    # the benchmarked pass (bench.py: frames_per_pass = 2400)
    dict(id="p2400_n2400", in_hw=40, fpp=2400, n=2400, env={}, variants=_BENCH),
    # odd count: frames end mid-tile, the last CTA pair is ragged
    dict(id="p2400_n1999", in_hw=40, fpp=2400, n=1999, env={}, variants=_BENCH),
    # the smallest pass on the raster / pair kernels (raster_pass: 190 x 400 px >= 4 x 148 tiles of 128 px) ...
    dict(id="p2400_n190", in_hw=40, fpp=2400, n=190, env={}, variants=_BENCH),
    # ... and the largest below: stage 2 and 3 on the one-CTA kernels
    dict(id="p2400_n189", in_hw=40, fpp=2400, n=189, env={},
         variants=frozenset({STRIP, HALO128, IGEMM128, IGEMM128_ALIGNED, IGEMM256, IGEMM256_ALIGNED})),
    # stage 2 on the im2col pair kernel with resident weights
    dict(id="p2400_n2400_raster0", in_hw=40, fpp=2400, n=2400, env={"CER_RASTER": "0"}, variants=_NO_RASTER),
    # epilogue constants in shared-memory tables instead of kernel parameters
    dict(id="p2400_n2400_ctab0", in_hw=40, fpp=2400, n=2400, env={"CER_CTAB": "0"}, variants=_BENCH),
    # 56 px input (7 x 7 stage 4: 49 px per frame); stage 2 at 28 x 28 is too wide for the raster kernel
    dict(id="p300_n300_56px", in_hw=56, fpp=300, n=300, env={}, variants=_NO_RASTER),
]

FC_ATOL = 1e-5          # unit-norm fp32 embedding against fp64


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _chunks(n, pixels_per_frame):
    """Frame ranges whose fp64 tensors stay at about 256 MB each."""
    step = max(1, 2 ** 25 // pixels_per_frame)
    return [(f0, min(n, f0 + step)) for f0 in range(0, n, step)]


def _stem_worst(pk, x, got):
    dev = x.device
    w = tf32_round(pk["stem_w"]).view(3, 3, 3, 64).permute(3, 2, 0, 1).to(dev, torch.float64)
    b = pk["stem_bias"].to(dev, torch.float64)
    al = pk["stem_alpha"].to(dev, torch.float64).view(1, -1, 1, 1)
    n, _, H, W = x.shape
    worst = 0.0
    for f0, f1 in _chunks(n, H * W * 64):
        z = F.conv2d(tf32_round(x[f0:f1]).double(), w, b, 1, 1)
        ref = torch.where(z >= 0, z, z * al)
        worst = max(worst, emulate.bound_ratio(got[f0:f1].permute(0, 3, 1, 2), ref).max().item())
    return worst


def _unit_worst(u, h, got):
    """h, got: the plan's bf16 NHWC input and output of unit u (weights on the device)."""
    n, H, W, _ = h.shape
    worst = 0.0
    for f0, f1 in _chunks(n, H * W * max(u["cin"], u["depth"])):
        ref, E = emulate.ir50_unit(u, h[f0:f1].permute(0, 3, 1, 2).double(), envelope=True)
        worst = max(worst, emulate.bound_ratio(got[f0:f1].permute(0, 3, 1, 2), ref, E).max().item())
    return worst


@pytest.mark.parametrize("case", PLAN_CASES, ids=lambda c: c["id"])
def test_plan_units_vs_fp64_reference(case, monkeypatch):
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import Ir50Engine
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)                    # read when the plan is created
    hw, n = case["in_hw"], case["n"]
    sd = synthetic.visual_backbone_state_dict(0, spatial=hw // 8)          # stage 4 map: in_hw / 8
    pk = packing.pack_ir50(sd, "backbone.", in_hw=hw)
    eng = Ir50Engine(pk, dev, frames_per_pass=case["fpp"])
    ran = {eng.op_variant(op, n) for op in range(eng.n_conv_ops)}
    assert ran == case["variants"], f"extra {sorted(ran - case['variants'])}, missing {sorted(case['variants'] - ran)}"

    x = synthetic.frames(n, seed=41, size=hw).to(dev)
    units = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in u.items()} for u in pk["units"]]
    prev = eng.debug_activation(x, -1)
    worst = {-1: _stem_worst(pk, x, prev)}
    for i, u in enumerate(units):
        got = eng.debug_activation(x, i)
        worst[i] = _unit_worst(u, prev, got)
        prev = got
    e = prev.reshape(n, -1).double() @ pk["fc_w"].to(dev, torch.float64).t() + pk["fc_bias"].to(dev, torch.float64)
    emb = eng.forward(x)
    fc_err = (emb.double() - e / e.norm(dim=1, keepdim=True)).abs().max().item()
    print(f"\n[{case['id']}] worst bound ratio: " + " ".join(f"{i}:{r:.3f}" for i, r in worst.items())
          + f"; FC + l2norm max abs err {fc_err:.2e}")
    over = {i: r for i, r in worst.items() if not r <= 1.0}
    assert not over, f"units over the bound (-1 = stem): {over}"
    assert fc_err <= FC_ATOL
