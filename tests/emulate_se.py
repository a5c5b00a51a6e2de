"""Reference of one IR-SE unit from its PACKED weights (tests only), with the acceptance envelope of its bf16
stores.  The SE plan stores conv1's output t, the pre-gate residual r and (transition units) the projection p in
bf16; the gate is computed in fp32 from the stored r.  se_unit rounds where the plan stores and returns the extra
bound term B for emulate.bound_ratio(got, y, B):

    |got - y| <= (1 + 2^-5) 2^-8 |y| + B + 1e-4 rms(y),   B = g A_r + |r| dg + A_p

* A_r = |bf16(rr + d) - bf16(rr - d)|, d = E_t + 2^-14 |rr| + 1e-6 rms(rr): the rounding-ambiguity envelope of
  r (rr = r before rounding; E_t = conv2(A_t, |w2|) is emulate.ir50_unit's envelope of t), scaled by the gate g.
* dg: the gate error that A_r implies.  The mean moves by at most mean_hw(A_r) (+ fp32 summation), the hidden
  layer by |fc1| of that, the logit by |fc2| of that, the gate by max sigmoid' over the logit's interval times it.
* A_p: the envelope of the projection's bf16 rounding (d = 2^-14 |p| + 1e-6 rms(p)).
"""
import torch
import torch.nn.functional as F

from tests import emulate

FAULTS = ("no_gate", "neighbour_gate", "no_sigmoid", "sum_not_mean", "unstrided_shortcut", "shortcut_before_gate")


def _r(x, on=True):
    return x.to(torch.bfloat16).to(x.dtype) if on else x


def _amb(v, d):
    return (_r(v + d) - _r(v - d)).abs()


def _rms(v):
    return v.pow(2).mean().sqrt()


def spread_frames(x, seed=0):
    """Per-frame contrast and brightness (x * a + b, a in [0.2, 1], b in [-0.4, 0.4], clamped to [-1, 1]): frames of
    synthetic.frames share their statistics, so their SE gates would be alike and a gate taken from the
    neighbouring frame would go unnoticed."""
    g = torch.Generator().manual_seed(seed)
    a = 0.2 + 0.8 * torch.rand(x.shape[0], 1, 1, 1, generator=g)
    b = 0.8 * torch.rand(x.shape[0], 1, 1, 1, generator=g) - 0.4
    return (x * a + b).clamp(-1, 1)


def stem(pk, x):
    """The stem's bf16 output [N, 64, H, W] (fp32 conv, as emulate.ir50_packed computes it)."""
    w = pk["stem_w"].view(3, 3, 3, 64).permute(3, 2, 0, 1)
    h = F.conv2d(x, w, pk["stem_bias"], 1, 1)
    return _r(torch.where(h >= 0, h, h * pk["stem_alpha"].view(1, -1, 1, 1)))


def se_unit(u, h, round_act=True, envelope=False, fault=None):
    """One IR-SE unit (u["se"] present) in h's dtype and on h's device.  h: the unit's input [N, cin, H, W] (NCHW).
    Returns (y, B, gate): y before the final bf16 rounding, B the extra bound term (None without envelope),
    gate [N, depth].  ``fault`` injects one of FAULTS (CPU guards of the bound)."""
    cin, depth, stride = u["cin"], u["depth"], u["stride"]
    dt = h.dtype
    w1 = u["w1"].to(dt).view(depth, 3, 3, cin).permute(0, 3, 1, 2)
    cls = emulate.border_class_map(h.shape[2], h.shape[3]).to(h.device)
    z = F.conv2d(h, w1, None, 1, 1) + u["bias1"].to(dt)[cls].permute(2, 0, 1).unsqueeze(0)
    al = u["alpha"].to(dt).view(1, -1, 1, 1)

    def prelu(v):
        return torch.where(v >= 0, v, v * al)

    t = _r(prelu(z), round_act)
    w2 = u["w2"].to(dt)
    w2m = w2[:, :9 * depth].view(depth, 3, 3, depth).permute(0, 3, 1, 2)
    bias2 = u["bias2"].to(dt).view(-1, depth)
    rr = F.conv2d(t, w2m, None, stride, 1) + bias2[0].view(1, -1, 1, 1)
    r = _r(rr, round_act)
    Ho, Wo = r.shape[2], r.shape[3]
    if u["has_proj"]:
        pp = F.conv2d(h, w2[:, 9 * depth:].reshape(depth, cin, 1, 1), None, stride) + bias2[1].view(1, -1, 1, 1)
        sc = _r(pp, round_act)
    elif fault == "unstrided_shortcut":
        sc = h[:, :, :Ho, :Wo]
    else:
        sc = h[:, :, ::stride, ::stride]
    fc1, fc2 = u["se"]["fc1"].to(dt), u["se"]["fc2"].to(dt)
    m = r.sum(dim=(2, 3)) if fault == "sum_not_mean" else r.mean(dim=(2, 3))
    hid = torch.relu(m @ fc1.t())
    logit = hid @ fc2.t()
    g = logit if fault == "no_sigmoid" else torch.sigmoid(logit)
    if fault == "neighbour_gate":
        g = g.roll(1, dims=0)
    g4 = g.view(g.shape[0], depth, 1, 1)
    if fault == "no_gate":
        y = r + sc
    elif fault == "shortcut_before_gate":
        y = (r + sc) * g4
    else:
        y = r * g4 + sc
    B = None
    if envelope:
        d_z = 2.0 ** -14 * z.abs() + 1e-6 * _rms(z)
        E_t = F.conv2d((_r(prelu(z + d_z)) - _r(prelu(z - d_z))).abs(), w2m.abs(), None, stride, 1)
        A_r = _amb(rr, E_t + 2.0 ** -14 * rr.abs() + 1e-6 * _rms(rr))
        dm = A_r.mean(dim=(2, 3)) + 2.0 ** -20 * r.abs().mean(dim=(2, 3))
        dhid = dm @ fc1.abs().t() + 2.0 ** -20 * (m.abs() @ fc1.abs().t())
        dlogit = dhid @ fc2.abs().t() + 2.0 ** -20 * (hid.abs() @ fc2.abs().t())
        nearest0 = torch.minimum(torch.maximum(torch.zeros_like(logit), logit - dlogit), logit + dlogit)
        sp = torch.sigmoid(nearest0)
        dg = sp * (1 - sp) * dlogit + 2.0 ** -22
        B = g4 * A_r + r.abs() * dg.view_as(g4)
        if u["has_proj"]:
            B = B + _amb(pp, 2.0 ** -14 * pp.abs() + 1e-6 * _rms(pp))
    return y, B, g
