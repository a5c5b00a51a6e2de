"""Every step of the VGGish plan, isolated, against an fp64 reference of that one step.

For each pass size, the plan's own output of step s-1 (VggishEngine.debug_activation) is the input of an fp64
reference of step s (tests/emulate.py vggish_stem / vggish_conv / vggish_fc), and the plan's output of step s must lie
within the per-element bound of emulate.bound_ratio:

    |got - ref| <= (1 + 2^-5) 2^-8 |ref| + 1e-4 rms(ref)

One bf16 rounding follows each fp32 accumulation, so there is no envelope term.  A conv whose epilogue applies the
following MaxPool2d(2,2) (the two shfl.xor rounds of conv_epilogue_tile / conv_halo_kernel) is checked against the
fp64 pool of the fp64 conv: a wrong pool partner, a window that straddles a warp or a ragged-tile store moves single
values far outside the bound, where an embedding cosine of 0.999 lets them pass.  The last FC stores fp32 and is held
to emulate.fc_dot_ratio (FC_DOT_C (|a| |w|^T + |b|)).

Each case pins the set of (step, kernel, pooled) the plan reports through op_variant; tests/test_vggish_parity_guards.py
checks that every instantiation that can take a pooled layer runs pooled in some case.  Only variables a plan reads when
it is created can differ per case (CER_NO_POOL_FUSION); the ones cached on first use (CER_NO_PAIR, CER_HALO, CER_STRIP,
CER_PAIR_BRES) cannot be switched within one process.  There is no CER_CTAB case: the VGGish plan builds its convs
without host tables, so its epilogue constants always come from shared memory and CER_CTAB=0 would repeat p1200_n1200.
"""
import pytest
import torch
import torch.nn.functional as F

from feature_vs_text_compound_emotion_b200 import packing, synthetic
from tests import emulate

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

STEM = "vgg_stem_pool_kernel"
POOL = "maxpool2x2_kernel"
HALO128 = "conv_halo_kernel<128>"
PAIR256 = "conv_igemm2_kernel<256,6>"
IGEMM256 = "conv_igemm_kernel<256,4,0,0>"
IGEMM256_ALIGNED = "conv_igemm_kernel<256,4,0,1>"
IGEMM128_ALIGNED = "conv_igemm_kernel<128,6,0,1>"
IGEMM64 = "conv_igemm_kernel<64,8,0,0>"
IGEMM64_ALIGNED = "conv_igemm_kernel<64,8,0,1>"

# steps of the fused plan: conv2+pool, conv3, conv4+pool, conv5, conv6+pool, FC 12288->4096, FC 4096->4096, FC 4096->128
_FUSED_POOLED = (True, False, True, False, True, False, False, False)


def _fused(conv3, conv4, conv5, conv6, fc12=IGEMM256_ALIGNED, fc3=IGEMM64_ALIGNED):
    kernels = (HALO128, conv3, conv4, conv5, conv6, fc12, fc12, fc3)
    return frozenset({(-1, STEM, False)} | {(s, k, p) for s, (k, p) in enumerate(zip(kernels, _FUSED_POOLED))})


PLAN_CASES = [
    # the `full` workload's pass (VGGish.patches_per_pass = 1200): convs 3-6 on the CTA pair, the two wide FCs on
    # igemm<256,4,0,1> with a 2 x 4096-float epilogue table, the 128-wide FC on a 64-wide N tile
    dict(id="p1200_n1200", fpp=1200, n=1200, env={}, variants=_fused(PAIR256, PAIR256, PAIR256, PAIR256)),
    # the last M tile and the last CTA pair are ragged
    dict(id="p1200_n1199", fpp=1200, n=1199, env={}, variants=_fused(PAIR256, PAIR256, PAIR256, PAIR256)),
    # conv3/4 on the pair kernel, conv5/6 below four waves of pair tiles (test_infer_video_from_stored_uint8_crops_and_logmel)
    dict(id="p1200_n330", fpp=1200, n=330, env={},
         variants=_fused(PAIR256, PAIR256, IGEMM256_ALIGNED, IGEMM256_ALIGNED)),
    # one patch: every tile ragged, conv3's 18 k-steps on the unaligned 256 kernel
    dict(id="p1200_n1", fpp=1200, n=1, env={},
         variants=_fused(IGEMM256, IGEMM256_ALIGNED, IGEMM256_ALIGNED, IGEMM256_ALIGNED)),
    # 48 patches of allocation narrow conv5/6 to a 128-wide N tile
    dict(id="p40_n17", fpp=40, n=17, env={},
         variants=_fused(IGEMM256, IGEMM256_ALIGNED, IGEMM128_ALIGNED, IGEMM128_ALIGNED)),
    # 9 patches of allocation narrow conv3/4 to a 64-wide N tile
    dict(id="p1_n1", fpp=1, n=1, env={},
         variants=_fused(IGEMM64, IGEMM64, IGEMM128_ALIGNED, IGEMM128_ALIGNED)),
    # every pool as its own kernel after an unpooled conv
    dict(id="p1200_n1200_nofuse", fpp=1200, n=1200, env={"CER_NO_POOL_FUSION": "1"},
         variants=frozenset({(-1, STEM, False), (0, HALO128, False), (1, POOL, False), (2, PAIR256, False),
                             (3, PAIR256, False), (4, POOL, False), (5, PAIR256, False), (6, PAIR256, False),
                             (7, POOL, False), (8, IGEMM256_ALIGNED, False), (9, IGEMM256_ALIGNED, False),
                             (10, IGEMM64_ALIGNED, False)})),
]


def _dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _chunks(n, elems_per_patch):
    """Patch ranges whose fp64 tensors stay at about 256 MB each."""
    step = max(1, 2 ** 25 // elems_per_patch)
    return [(f0, min(n, f0 + step)) for f0 in range(0, n, step)]


def _on(pk, dev):
    return {"conv1_w": pk["conv1_w"].to(dev), "conv1_bias": pk["conv1_bias"].to(dev),
            "convs": [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in c.items()} for c in pk["convs"]],
            "fcs": [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in f.items()} for f in pk["fcs"]]}


def _stem_worst(pk, x, got):
    n, H, W = x.shape
    worst = 0.0
    for f0, f1 in _chunks(n, H * W * 64):
        ref = emulate.vggish_stem(pk, x[f0:f1].double())
        worst = max(worst, emulate.bound_ratio(got[f0:f1].permute(0, 3, 1, 2), ref).max().item())
    return worst


def _step_worst(pk, d, h, got):
    """h, got: the plan's input and output of step d (NHWC, or [n,1,1,dim] for an FC)."""
    n = h.shape[0]
    worst = 0.0
    if d["kind"] == "fc":
        f = pk["fcs"][d["layer"]]
        a = h.reshape(n, -1)
        for f0, f1 in _chunks(n, max(f["in_dim"], f["out_dim"])):
            g = got[f0:f1].reshape(f1 - f0, -1)
            ad = a[f0:f1].double()
            r = emulate.fc_dot_ratio(g, ad, f) if d["dtype"] == torch.float32 else emulate.bound_ratio(g, emulate.vggish_fc(f, ad))
            worst = max(worst, r.max().item())
        return worst
    _, H, W, C = h.shape
    c = pk["convs"][d["layer"]]
    for f0, f1 in _chunks(n, H * W * max(C, c["cout"])):
        hd = h[f0:f1].permute(0, 3, 1, 2).double()
        ref = F.max_pool2d(hd, 2) if d["kind"] == "pool" else emulate.vggish_conv(c, hd, d["pool_fused"])
        worst = max(worst, emulate.bound_ratio(got[f0:f1].permute(0, 3, 1, 2), ref).max().item())
    return worst


@pytest.fixture(scope="module")
def packed():
    return packing.pack_vggish(synthetic.vggish_state_dict(0))


@pytest.mark.parametrize("case", PLAN_CASES, ids=lambda c: c["id"])
def test_plan_steps_vs_fp64_reference(case, packed, monkeypatch):
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import VggishEngine
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)                    # read when the plan is created
    n = case["n"]
    eng = VggishEngine(packed, dev, patches_per_pass=case["fpp"])
    ran = {(s, eng.op_variant(s, n), s >= 0 and eng.step_shapes[s]["pool_fused"]) for s in range(-1, len(eng.step_shapes))}
    assert ran == case["variants"], f"extra {sorted(ran - case['variants'])}, missing {sorted(case['variants'] - ran)}"

    pk = _on(packed, dev)
    x = synthetic.logmel_patches(n, seed=51 + n).to(dev)
    prev = eng.debug_activation(x, -1)
    worst = {-1: _stem_worst(pk, x, prev)}
    for s, d in enumerate(eng.step_shapes):
        got = eng.debug_activation(x, s)
        worst[s] = _step_worst(pk, d, prev, got)
        prev = got
    names = {s: ("P" if d["pool_fused"] else "") + d["kind"] + str(d["layer"]) for s, d in enumerate(eng.step_shapes)}
    print(f"\n[{case['id']}] worst bound ratio: stem:{worst[-1]:.3f} "
          + " ".join(f"{names[s]}:{worst[s]:.3f}" for s in names))
    over = {s: r for s, r in worst.items() if not r <= 1.0}
    assert not over, f"steps over the bound (-1 = stem): {over}"
    if n == case["fpp"]:
        assert torch.equal(eng.forward(x), prev.reshape(n, -1)), "the forward pass differs from the debug pass"


def test_multi_pass_rows_equal_single_passes(packed):
    """2401 patches at 1200 per pass: every pass reads its own input rows and writes its own output rows."""
    dev = _dev()
    from feature_vs_text_compound_emotion_b200.engine import VggishEngine
    eng = VggishEngine(packed, dev, patches_per_pass=1200)
    x = synthetic.logmel_patches(2401, seed=77).to(dev)
    full = eng.forward(x)
    for a, b in ((0, 1200), (1200, 2400), (2400, 2401)):
        assert torch.equal(full[a:b], eng.forward(x[a:b])), f"rows [{a}, {b})"
