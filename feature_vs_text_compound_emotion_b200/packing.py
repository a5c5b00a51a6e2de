"""One-time weight packing: reference-layout state_dict -> the layouts the CUDA kernels read
(include/cer_b200.h).  Runs on the CPU in fp64 so that folding adds no rounding of its own; the
results are cast to bf16 (tensor-core operands) / fp32 (biases, head weights) at the end.

Algebra (eval mode; reference lines in brackets):

* BatchNorm as affine: y = s*x + t with s = w/sqrt(var+eps), t = b - mean*s.
* Post-conv BN (stem [arcface_model.py:130-131], res_layer.4 [:55], shortcut BN [:50-51]):
  scale the conv's output channel -> W'[co] = s[co]*W[co], bias = t[co].
* Pre-conv BN (res_layer.0 -> zero-padded 3x3 conv [:53-54]): the conv pads with zeros AFTER the
  BN, so the shift t cannot become a plain bias: on the 1-pixel border some taps see padding,
  not t.  By linearity conv(pad(s*x+t)) = conv_{W*s}(pad(x)) + conv_W(pad(t*1)), and the second
  term takes only 9 values per output channel (3 row classes x 3 column classes: first / inner /
  last).  We fold s into the weights' input channel and ship that [9][Cout] table; the kernel
  epilogue indexes it with the border class of each output pixel.  Exact, no extra activation.
* The 1x1/stride-2 projection shortcut of the first unit of stages 2-4 is appended to conv2's K
  axis (its own BN scale folded in), so `res + shortcut` [:57-60] is one accumulation.
* The MaxPool2d(1, 2) shortcut of a stride-2 unit with cin == depth (stage 1 of IR-100 / IR-152) is
  packed the same way with identity columns, w2 = [w2 | I]: products by 1.0 are exact.
* IR-SE units (bottleneck_IR_SE [:63-84], SEModule [:23-41]): the gate scales the residual branch
  only, so the plan keeps the shortcut out of conv2 -- a projection keeps its columns in w2 but runs
  as its own 1x1 conv, with its BN shift as a second bias row (bias2 [2][depth]); a stride-2
  identity shortcut stays an identity (has_proj = 0).  fc1 / fc2 ship as fp32 matrices.
* output_layer [backbone.py:99-103]: BN2d and BN1d are folded into the Linear, whose K axis is
  permuted from NCHW-flatten (c,h,w) [arcface_model.py:12-14] to the NHWC order the conv stack
  produces.
* weight_norm [temporal_convolutional_model.py:24,30]: w = g*v/||v|| per output channel.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import torch

BN_EPS = 1e-5


def _bn_affine(sd, p):
    w = sd[p + ".weight"].double()
    s = w / torch.sqrt(sd[p + ".running_var"].double() + BN_EPS)
    t = sd[p + ".bias"].double() - sd[p + ".running_mean"].double() * s
    return s, t


def infer_units(sd: Dict[str, torch.Tensor], prefix: str, strides: Sequence[int] = None):
    """(cin, depth, stride, proj) per unit, recovered from the state_dict itself: a unit has a projection
    shortcut iff shortcut_layer.0.weight exists.  Without ``strides``, stride 2 is inferred from a projection
    (IR-50, arcface_model.py:87-102); the MaxPool2d(1, 2) shortcut of IR-100 / IR-152 stage 1 leaves no key,
    so those strides come from the modules (``strides``, one per unit)."""
    units = []
    i = 0
    while f"{prefix}body.{i}.res_layer.1.weight" in sd:
        w1 = sd[f"{prefix}body.{i}.res_layer.1.weight"]
        depth, cin = int(w1.shape[0]), int(w1.shape[1])
        proj = f"{prefix}body.{i}.shortcut_layer.0.weight" in sd
        units.append((cin, depth, (2 if proj else 1) if strides is None else int(strides[i]), proj))
        i += 1
    if strides is not None and len(strides) != len(units):
        raise ValueError(f"{len(strides)} strides for {len(units)} units")
    return units


def pack_ir50(sd: Dict[str, torch.Tensor], prefix: str = "backbone.", in_hw: int = 40,
              operand_dtype: torch.dtype = torch.bfloat16, strides: Sequence[int] = None) -> dict:
    """Returns {'stem_w','stem_bias','stem_alpha', 'units': [ {cin,depth,stride,has_proj,w1,bias1,alpha,w2,bias2} ],
    'fc_w','fc_bias','fc_in','emb_dim'} as CPU tensors (``operand_dtype`` for w1/w2/fc_w -- bf16 for the
    kernels, fp32 only in tests of the algebra -- fp32 otherwise).  ``strides``: the units' strides (see
    infer_units).  A unit whose MaxPool2d(1, 2) shortcut became identity columns also has 'identity_sc': 1; an
    IR-SE unit has 'se': {'fc1' [hidden][depth], 'fc2' [depth][hidden]} (fp32)."""
    p = prefix
    out = {}
    W = sd[p + "input_layer.0.weight"].double()                      # [64, 3, 3, 3] (co, ci, r, s)
    s, t = _bn_affine(sd, p + "input_layer.1")
    Ws = W * s.view(-1, 1, 1, 1)
    out["stem_w"] = Ws.permute(2, 3, 1, 0).reshape(27, W.shape[0]).float().contiguous()   # [(r,s,ci)][co]
    out["stem_bias"] = t.float().contiguous()
    out["stem_alpha"] = sd[p + "input_layer.2.weight"].float().contiguous()

    units = []
    hw = in_hw
    for i, (cin, depth, stride, proj) in enumerate(infer_units(sd, p, strides)):
        u = f"{p}body.{i}."
        se = u + "res_layer.5.fc1.weight" in sd
        s1, t1 = _bn_affine(sd, u + "res_layer.0")
        W1 = sd[u + "res_layer.1.weight"].double()                   # [depth, cin, 3, 3]
        w1 = (W1 * s1.view(1, -1, 1, 1)).permute(0, 2, 3, 1).reshape(depth, 9 * cin)     # K = (r, s, ci)
        T = torch.einsum("ocrs,c->ors", W1, t1)                      # shift pushed through each tap
        bias1 = torch.empty(9, depth, dtype=torch.float64)
        valid = {0: (1, 2), 1: (0, 1, 2), 2: (0, 1)}                 # class 0: first row/col (tap 0 pads); 2: last
        for rc in range(3):
            for cc in range(3):
                bias1[rc * 3 + cc] = T[:, list(valid[rc])][:, :, list(valid[cc])].sum(dim=(1, 2))
        s2, t2 = _bn_affine(sd, u + "res_layer.4")
        W2 = sd[u + "res_layer.3.weight"].double()                   # [depth, depth, 3, 3]
        w2 = (W2 * s2.view(-1, 1, 1, 1)).permute(0, 2, 3, 1).reshape(depth, 9 * depth)
        bias2 = t2.clone()
        identity_sc = not proj and not se and stride != 1
        if proj:
            ss, ts = _bn_affine(sd, u + "shortcut_layer.1")
            Wsc = sd[u + "shortcut_layer.0.weight"].double().reshape(depth, cin)
            w2 = torch.cat([w2, Wsc * ss.view(-1, 1)], dim=1)
            bias2 = torch.stack([bias2, ts]) if se else bias2 + ts
        elif identity_sc:
            if cin != depth:
                raise ValueError(f"unit {i}: an identity shortcut needs cin == depth")
            w2 = torch.cat([w2, torch.eye(depth, dtype=torch.float64)], dim=1)
        unit = {
            "cin": cin, "depth": depth, "stride": stride, "has_proj": int(proj or identity_sc),
            "w1": w1.to(operand_dtype).contiguous(), "bias1": bias1.float().contiguous(),
            "alpha": sd[u + "res_layer.2.weight"].float().contiguous(),
            "w2": w2.to(operand_dtype).contiguous(), "bias2": bias2.float().contiguous(),
        }
        if identity_sc:
            unit["identity_sc"] = 1
        if se:
            fc1 = sd[u + "res_layer.5.fc1.weight"]
            unit["se"] = {"fc1": fc1.reshape(fc1.shape[0], depth).float().contiguous(),
                          "fc2": sd[u + "res_layer.5.fc2.weight"].reshape(depth, fc1.shape[0]).float().contiguous()}
        units.append(unit)
        hw = (hw - 1) // stride + 1
    out["units"] = units

    c = units[-1]["depth"]
    s0, t0 = _bn_affine(sd, p + "output_layer.0")
    Wl = sd[p + "output_layer.3.weight"].double()                    # [emb, c*hw*hw], K = (c, h, w)
    bl = sd[p + "output_layer.3.bias"].double()
    s4, t4 = _bn_affine(sd, p + "output_layer.4")
    emb = Wl.shape[0]
    if Wl.shape[1] != c * hw * hw:
        raise ValueError(f"output_layer.3 expects {Wl.shape[1]} inputs but the body yields {c}x{hw}x{hw}")
    Wl4 = Wl.view(emb, c, hw, hw)
    fc_w = (Wl4 * s0.view(1, -1, 1, 1)).permute(0, 2, 3, 1).reshape(emb, hw * hw * c) * s4.view(-1, 1)
    fc_b = s4 * (bl + torch.einsum("ochw,c->o", Wl4, t0)) + t4
    out["fc_w"] = fc_w.to(operand_dtype).contiguous()
    out["fc_bias"] = fc_b.float().contiguous()
    out["fc_in"] = hw * hw * c
    out["emb_dim"] = emb
    out["in_hw"] = in_hw
    return out


def weight_norm_effective(g: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    v = v.double()
    return g.double() * v / v.reshape(v.shape[0], -1).norm(dim=1).view(-1, 1, 1)


def tcn_block_to_kmajor(blk: dict) -> dict:
    """Tap-major fp32-kernel layout -> the K-major layout of the tensor-core kernel:
    w1 [cout][k*cin] with K = (tap, ci); w2 [cout][k*cout (+ cin)] with the downsample appended."""
    out = dict(blk)
    k, cin, cout = blk["w1"].shape
    w1, wd = blk["w1"], blk["wd"]
    if cin % 32:
        # the tensor-core kernel moves 32-channel chunks: pad the input channels with zero weights
        # (mfcc: 39 -> 64, egemaps: 88 -> 96); TcnEngine zero-pads the features to match
        pad = 32 - cin % 32
        w1 = torch.nn.functional.pad(w1, (0, 0, 0, pad))                     # [k][cin+pad][cout]
        if wd is not None:
            wd = torch.nn.functional.pad(wd, (0, 0, 0, pad))                 # [cin+pad][cout]
        cin += pad
        out["c_in"] = cin
    if cout % 32:
        raise ValueError("TemporalBlock output channels must be multiples of 32 for the tensor-core kernel")
    out["w1"] = w1.permute(2, 0, 1).reshape(cout, k * cin).contiguous()
    w2 = blk["w2"].permute(2, 0, 1).reshape(cout, k * cout)
    if wd is not None:
        w2 = torch.cat([w2, wd.t()], dim=1)
    out["w2"] = w2.contiguous()
    out["layout"] = "k_major"
    return out


def pack_tcn(sd: Dict[str, torch.Tensor], prefix: str, bn_prefix: str = None) -> List[dict]:
    """prefix = 'temporal.<m>.'; bn_prefix = 'bn.<m>' folds the trailing BatchNorm1d
    (models/model.py:515) into the last block's output affine.  Returns the tap-major layout
    ([k][cin][cout]); engine.TcnEngine converts to K-major for the tensor-core kernel."""
    blocks = []
    i = 0
    while f"{prefix}network.{i}.conv1.weight_v" in sd:
        b = f"{prefix}network.{i}."
        w1 = weight_norm_effective(sd[b + "conv1.weight_g"], sd[b + "conv1.weight_v"])    # [cout, cin, k]
        w2 = weight_norm_effective(sd[b + "conv2.weight_g"], sd[b + "conv2.weight_v"])
        blk = {
            "c_in": int(w1.shape[1]), "c_out": int(w1.shape[0]), "kernel_size": int(w1.shape[2]), "dilation": 2 ** i,
            "w1": w1.permute(2, 1, 0).float().contiguous(),          # [k][cin][cout]
            "b1": sd[b + "conv1.bias"].float().contiguous(),
            "w2": w2.permute(2, 1, 0).float().contiguous(),
            "b2": sd[b + "conv2.bias"].float().contiguous(),
            "wd": None, "bd": None, "post_scale": None, "post_shift": None,
        }
        if b + "downsample.weight" in sd:
            blk["wd"] = sd[b + "downsample.weight"][:, :, 0].t().float().contiguous()       # [cin][cout]
            blk["bd"] = sd[b + "downsample.bias"].float().contiguous()
        blocks.append(blk)
        i += 1
    if bn_prefix is not None and blocks:
        s, t = _bn_affine(sd, bn_prefix)
        blocks[-1]["post_scale"] = s.float().contiguous()
        blocks[-1]["post_shift"] = t.float().contiguous()
    return blocks


def pack_fusion(sd: Dict[str, torch.Tensor], modalities: Sequence[str], modal_dim: int, num_heads: int,
                prefix: str = "fusion.", regressor: str = "regressor") -> dict:
    a = prefix + "layers.self_attn."
    out = {"modal_dim": modal_dim, "num_heads": num_heads, "n_modals": len(modalities),
           "dim": [int(sd[f"{a}qkv_proj.{m}.weight"].shape[1]) for m in modalities],
           "wqkv": [sd[f"{a}qkv_proj.{m}.weight"].t().float().contiguous() for m in modalities],
           "bqkv": [sd[f"{a}qkv_proj.{m}.bias"].float().contiguous() for m in modalities],
           "wo": sd[a + "o_proj.weight"].t().float().contiguous(),
           "bo": sd[a + "o_proj.bias"].float().contiguous(),
           "ln_g": sd[prefix + "layers.norm1.weight"].float().contiguous(),
           "ln_b": sd[prefix + "layers.norm1.bias"].float().contiguous(),
           "wr": sd[regressor + ".weight"].t().float().contiguous(),
           "br": sd[regressor + ".bias"].float().contiguous(),
           # nn.Linear layout [out][in] for the composed path (cer_linear_forward) used when the fused
           # kernel's shared-memory weight staging does not fit (large modal_dim)
           "wqkv_oi": [sd[f"{a}qkv_proj.{m}.weight"].float().contiguous() for m in modalities],
           "wo_oi": sd[a + "o_proj.weight"].float().contiguous(),
           "wr_oi": sd[regressor + ".weight"].float().contiguous()}
    out["n_out"] = int(out["br"].shape[0])
    return out


def pack_bert(sd: Dict[str, torch.Tensor], n_layers: int = None) -> dict:
    """HF BertModel state_dict -> the cer_bert_weights layout (include/cer_b200.h): fp32, nn.Linear / nn.Embedding
    layouts as they are, except that each layer's query / key / value weights and biases are stacked into one [3H, H]
    projection (wqkv) and one [3H] bias (bqkv).  The pooler is not used."""
    if n_layers is None:
        n_layers = 0
        while f"encoder.layer.{n_layers}.attention.self.query.weight" in sd:
            n_layers += 1
    f = lambda k: sd[k].detach().float().contiguous()
    e = "embeddings."
    out = {"word_emb": f(e + "word_embeddings.weight"), "pos_emb": f(e + "position_embeddings.weight"),
           "type_emb": f(e + "token_type_embeddings.weight"), "emb_ln_g": f(e + "LayerNorm.weight"),
           "emb_ln_b": f(e + "LayerNorm.bias"), "layers": []}
    for i in range(n_layers):
        p = f"encoder.layer.{i}."
        a = p + "attention.self."
        out["layers"].append({
            "wqkv": torch.cat([f(a + n + ".weight") for n in ("query", "key", "value")]).contiguous(),
            "bqkv": torch.cat([f(a + n + ".bias") for n in ("query", "key", "value")]).contiguous(),
            "wo": f(p + "attention.output.dense.weight"), "bo": f(p + "attention.output.dense.bias"),
            "ln1_g": f(p + "attention.output.LayerNorm.weight"), "ln1_b": f(p + "attention.output.LayerNorm.bias"),
            "w1": f(p + "intermediate.dense.weight"), "b1": f(p + "intermediate.dense.bias"),
            "w2": f(p + "output.dense.weight"), "b2": f(p + "output.dense.bias"),
            "ln2_g": f(p + "output.LayerNorm.weight"), "ln2_b": f(p + "output.LayerNorm.bias")})
    return out


VGGISH_CFG = (64, "M", 128, "M", 256, 256, "M", 512, 512, "M")     # make_layers(), models/backbone.py:43-53


def pack_vggish(sd: Dict[str, torch.Tensor], prefix: str = "", in_hw=(96, 64),
                operand_dtype: torch.dtype = torch.bfloat16) -> dict:
    """vggish.pth layout (features.{0,3,6,8,11,13}, embeddings.{0,2,4}; models/backbone.py:16-66)
    -> {'conv1_w' [9][64] fp32, 'conv1_bias', 'convs': [{cin,cout,pool_after,w [cout][9*cin],bias}],
    'fcs': [{in_dim,out_dim,relu,w [out][in],bias}], 'zeros'}.  Conv weights go to K = (r,s,ci);
    the first FC's K axis is already the (h,w,c) flatten the reference builds with its two
    transposes (:34-37), which is the NHWC order the kernels produce, so it is used as is."""
    idx, cin, convs = 0, 1, []
    for j, v in enumerate(VGGISH_CFG):
        if v == "M":
            idx += 1
            continue
        W = sd[f"{prefix}features.{idx}.weight"].double()             # [cout, cin, 3, 3]
        b = sd[f"{prefix}features.{idx}.bias"].float().contiguous()
        pool = int(j + 1 < len(VGGISH_CFG) and VGGISH_CFG[j + 1] == "M")
        if cin == 1:
            if not pool:
                raise ValueError("the first conv must be followed by a pool")
            conv1 = (W.permute(2, 3, 1, 0).reshape(9, v).float().contiguous(), b)
        else:
            convs.append({"cin": cin, "cout": v, "pool_after": pool,
                          "w": W.permute(0, 2, 3, 1).reshape(v, 9 * cin).to(operand_dtype).contiguous(), "bias": b})
        idx += 2
        cin = v
    fcs = []
    for i in (0, 2, 4):
        W = sd[f"{prefix}embeddings.{i}.weight"]
        fcs.append({"in_dim": int(W.shape[1]), "out_dim": int(W.shape[0]), "relu": int(i != 4),
                    "w": W.to(operand_dtype).contiguous(), "bias": sd[f"{prefix}embeddings.{i}.bias"].float().contiguous()})
    width = max([c["cout"] for c in convs] + [f["out_dim"] for f in fcs])
    return {"in_h": in_hw[0], "in_w": in_hw[1], "c1": int(conv1[0].shape[1]), "conv1_w": conv1[0], "conv1_bias": conv1[1],
            "convs": convs, "fcs": fcs, "zeros": torch.zeros(width), "emb_dim": fcs[-1]["out_dim"]}


# VGGish front-end parameters (abaw5_pre_processing/base/vggish/vggish_params.py)
LOGMEL = {"sample_rate": 16000, "win": 400, "hop": 160, "fft": 512, "n_mel": 64, "mel_lo": 125.0, "mel_hi": 7500.0,
          "log_offset": 0.01}


def logmel_tables(cfg: dict = None) -> torch.Tensor:
    """fp64 [win | fft | fft | (fft/2+1)*n_mel]: periodic Hann window, cos/sin twiddles and the HTK
    mel matrix (mel_features.py:66-90, :129-204) for cer_logmel_forward."""
    import numpy as np
    c = cfg or LOGMEL
    win, fft, n_mel = c["win"], c["fft"], c["n_mel"]
    hann = 0.5 - 0.5 * np.cos(2 * np.pi / win * np.arange(win))
    ang = 2 * np.pi * np.arange(fft) / fft
    bins = fft // 2 + 1
    mel = lambda f: 1127.0 * np.log(1.0 + f / 700.0)
    bins_mel = mel(np.linspace(0.0, c["sample_rate"] / 2.0, bins))
    edges = np.linspace(mel(c["mel_lo"]), mel(c["mel_hi"]), n_mel + 2)
    m = np.empty((bins, n_mel))
    for i in range(n_mel):
        lo, ce, up = edges[i:i + 3]
        m[:, i] = np.maximum(0.0, np.minimum((bins_mel - lo) / (ce - lo), (up - bins_mel) / (up - ce)))
    m[0, :] = 0.0
    return torch.from_numpy(np.concatenate([hann, np.cos(ang), np.sin(ang), m.reshape(-1)]))
