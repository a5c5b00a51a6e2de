"""Pure-torch emulation of what the CUDA kernels compute from the PACKED weights (tests only).

Used on the CPU to prove the packing algebra (BN folding, border-class bias table, fused
projection shortcut, NHWC FC permutation, weight-norm, tap-major TCN weights) before any GPU
time is spent, and to predict the bf16 error budget.  `round_act=True` rounds every stored
activation to bf16 exactly where the kernels do.
"""
import torch
import torch.nn.functional as F


def _r(x, on):
    return x.to(torch.bfloat16).to(x.dtype) if on else x


def border_class_map(H, W):
    r = torch.ones(H, dtype=torch.long); r[0] = 0; r[-1] = 2
    c = torch.ones(W, dtype=torch.long); c[0] = 0; c[-1] = 2
    return r.view(-1, 1) * 3 + c.view(1, -1)          # [H, W]


def ir50_unit(u, h, round_t=True, envelope=False):
    """One IR-50 residual unit from its packed weights, computed in h's dtype and on h's device.

    h: the unit's input [N, cin, H, W] (NCHW; bf16 values as the previous unit stored them).  Returns (y, E):
    y is the unit's output before its final bf16 rounding.  conv1's output t is rounded to bf16 where the
    kernels round it (round_t).  E (envelope=True) is a rounding-ambiguity envelope: conv2(A, |w2|) with
    A = |bf16(prelu(z + d)) - bf16(prelu(z - d))|, d = 2^-14 |z| + 1e-6 rms(z), z = conv1's pre-activation.
    It bounds how far a correct kernel's output can move because its fp32 z (summed in another order)
    rounds t to the other neighbouring bf16 value.  E is None without envelope."""
    cin, depth, stride = u["cin"], u["depth"], u["stride"]
    w1 = u["w1"].to(h.dtype).view(depth, 3, 3, cin).permute(0, 3, 1, 2)
    cls = border_class_map(h.shape[2], h.shape[3]).to(h.device)
    z = F.conv2d(h, w1, None, 1, 1) + u["bias1"].to(h.dtype)[cls].permute(2, 0, 1).unsqueeze(0)   # [9,depth] by class
    al = u["alpha"].to(h.dtype).view(1, -1, 1, 1)

    def prelu(v):
        return torch.where(v >= 0, v, v * al)

    t = _r(prelu(z), round_t)
    w2 = u["w2"].to(h.dtype)
    w2m = w2[:, :9 * depth].view(depth, 3, 3, depth).permute(0, 3, 1, 2)
    y = F.conv2d(t, w2m, None, stride, 1)
    if u["has_proj"]:
        y = y + F.conv2d(h, w2[:, 9 * depth:].view(depth, cin, 1, 1), None, stride)
    else:
        y = y + h
    y = y + u["bias2"].to(h.dtype).view(1, -1, 1, 1)
    E = None
    if envelope:
        d = 2.0 ** -14 * z.abs() + 1e-6 * z.pow(2).mean().sqrt()
        A = (_r(prelu(z + d), True) - _r(prelu(z - d), True)).abs()
        E = F.conv2d(A, w2m.abs(), None, stride, 1)
    return y, E


# Per-element acceptance bound of a bf16 kernel output against a high-precision reference of the same op:
#   |got - ref| <= (1 + BF16_SLACK) 2^-8 |ref| + E + C_RMS rms(ref)
# 2^-8 |ref| is the round-to-nearest step to bf16 (pack_bf16x2); E covers intermediate roundings (ir50_unit),
# C_RMS rms(ref) the fp32 accumulation of a different summation order.
C_RMS = 1e-4
BF16_SLACK = 2.0 ** -5


def bound_ratio(got, ref, E=None, c=C_RMS):
    """Elementwise |got - ref| / bound (<= 1 passes), computed in ref's dtype; a NaN in got counts as inf."""
    got = got.to(ref.dtype)
    bound = (1 + BF16_SLACK) * 2.0 ** -8 * ref.abs() + c * ref.pow(2).mean().sqrt()
    if E is not None:
        bound = bound + E
    return torch.nan_to_num((got - ref).abs() / bound, nan=float("inf"))


def vggish_stem(pk, x):
    """VGGish features.0-2 from the packed fp32 weights, in x's dtype: x [N,H,W] -> maxpool2(relu(conv3x3(x) + b))
    [N,64,H/2,W/2] (NCHW).  The fp32 weights and inputs are exact in fp64."""
    w = pk["conv1_w"].to(x.device, x.dtype).view(3, 3, -1).permute(2, 0, 1).unsqueeze(1)     # [(r,s)][co] -> [co,1,r,s]
    z = F.conv2d(x.unsqueeze(1), w, pk["conv1_bias"].to(x.device, x.dtype), 1, 1)
    return F.max_pool2d(torch.relu(z), 2)


def vggish_conv(c, h, pool):
    """One packed VGGish conv in h's dtype: h [N,cin,H,W] (the bf16 values the previous step stored) ->
    relu(conv3x3(h, w) + b), max-pooled 2x2 if `pool`.  One rounding (to bf16) follows the fp32 accumulation, so
    the bound needs no envelope (E = 0); max commutes with that monotone rounding, and with ReLU every pooled value
    bounds the other three of its window, so the pooled output keeps the same bound."""
    cin, cout = c["cin"], c["cout"]
    w = c["w"].to(h.device, h.dtype).view(cout, 3, 3, cin).permute(0, 3, 1, 2)
    y = torch.relu(F.conv2d(h, w, c["bias"].to(h.device, h.dtype), 1, 1))
    return F.max_pool2d(y, 2) if pool else y


def vggish_fc(f, a):
    """One packed VGGish FC in a's dtype: a [N,in_dim] (the NHWC flatten of the previous step) -> a w^T + b, ReLU if
    f["relu"]."""
    y = F.linear(a, f["w"].to(a.device, a.dtype), f["bias"].to(a.device, a.dtype))
    return torch.relu(y) if f["relu"] else y


# The last FC stores fp32: |got - ref| <= FC_DOT_C (|a| |w|^T + |b|), a bound on reordering an fp32 dot product.
# 2^-14 is the ceiling at which one dropped 64-wide K chunk of a 4096-long dot product still fails it
# (tests/test_vggish_parity_guards.py keeps both sides of that honest).
FC_DOT_C = 2.0 ** -14


def fc_dot_ratio(got, a, f, c=FC_DOT_C):
    """Elementwise |got - vggish_fc(f, a)| / (c (|a| |w|^T + |b|)), computed in a's dtype; NaN counts as inf."""
    w = f["w"].to(a.device, a.dtype)
    b = f["bias"].to(a.device, a.dtype)
    ref = vggish_fc(f, a)
    bound = c * (a.abs() @ w.abs().t() + b.abs())
    return torch.nan_to_num((got.to(a.dtype) - ref).abs() / bound, nan=float("inf"))


def ir50_packed(pk, x, round_act=True, upto=None):
    """x: [N,3,H,W] fp32 -> (emb [N,512], dict of unit outputs NHWC)."""
    N, _, H, W = x.shape
    w = pk["stem_w"].view(3, 3, 3, 64).permute(3, 2, 0, 1)           # [(r,s,ci)][co] -> [co,ci,r,s]
    h = F.conv2d(x, w, pk["stem_bias"], 1, 1)
    a = pk["stem_alpha"].view(1, -1, 1, 1)
    h = _r(torch.where(h >= 0, h, h * a), round_act)
    taps = {-1: h.permute(0, 2, 3, 1).contiguous()}
    for i, u in enumerate(pk["units"]):
        y, _ = ir50_unit(u, h, round_t=round_act)
        h = _r(y, round_act)
        taps[i] = h.permute(0, 2, 3, 1).contiguous()
        if upto is not None and i == upto:
            return None, taps
    flat = h.permute(0, 2, 3, 1).reshape(N, -1)
    e = F.linear(flat, pk["fc_w"].float(), pk["fc_bias"])
    return e / e.norm(dim=1, keepdim=True), taps


def tcn_packed(blocks, x):
    """x: [B,T,Cin] -> [B,T,Cout], from tap-major packed weights."""
    for blk in blocks:
        k, d = blk["kernel_size"], blk["dilation"]
        def cconv(inp, w, b):
            B, T, _ = inp.shape
            out = b.view(1, 1, -1).expand(B, T, -1).clone()
            for j in range(k):
                sh = (k - 1 - j) * d
                shifted = F.pad(inp, (0, 0, sh, 0))[:, :T]
                out = out + shifted @ w[j]
            return out
        h = F.leaky_relu(cconv(x, blk["w1"], blk["b1"]), 0.01)
        h = F.leaky_relu(cconv(h, blk["w2"], blk["b2"]), 0.01)
        res = x if blk["wd"] is None else x @ blk["wd"] + blk["bd"]
        x = F.leaky_relu(h + res, 0.01)
        if blk["post_scale"] is not None:
            x = x * blk["post_scale"] + blk["post_shift"]
    return x


def fusion_packed(fw, feats):
    """feats: list of [R, D_m] -> (logits [R,n_out], fused [R,E])."""
    M, md, H = fw["n_modals"], fw["modal_dim"], fw["num_heads"]
    hd = md // H
    qkv = [f @ w + b for f, w, b in zip(feats, fw["wqkv"], fw["bqkv"])]          # [R, 3*md]
    R = feats[0].shape[0]
    q = torch.stack([t.view(R, H, 3, hd)[:, :, 0] for t in qkv], dim=2)           # [R,H,M,hd]
    k = torch.stack([t.view(R, H, 3, hd)[:, :, 1] for t in qkv], dim=2)
    v = torch.stack([t.view(R, H, 3, hd)[:, :, 2] for t in qkv], dim=2)
    att = torch.softmax(q @ k.transpose(-1, -2) / hd ** 0.5, dim=-1)
    vals = (att @ v + v).reshape(R, H * M * hd)
    o = vals @ fw["wo"] + fw["bo"]
    fused = F.layer_norm(o, (o.shape[-1],), fw["ln_g"], fw["ln_b"], 1e-5)
    logits = torch.cat([feats[0], fused], dim=-1) @ fw["wr"] + fw["br"]
    return logits, fused
