"""Seeded synthetic weights and inputs in the reference's state_dict layout.

Checkpoints (res50_ir_0.887.pth, vggish.pth, best-models/*/model.pt) are not available
offline, so benches, tests and golden fixtures use randomly initialised weights whose *key
layout and shapes* are exactly those the reference's strict ``load_state_dict`` calls pin
(models/model.py:430, experiment.py:245-246; SURVEY.md section 8b).  BatchNorm running
statistics and affines are randomised too -- the default identity BN would hide every
BN-folding bug (SURVEY.md section 7.0).

Everything is generated on the CPU with an explicit ``torch.Generator`` so the same seed
gives the same tensors in the build container and on the GPU box.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, List, Sequence

import torch

from .modules import get_blocks

# (in_channel, depth, stride) per residual unit of IR-50 as configured by the reference
# (models/arcface_model.py:95-102: unit counts 3/4/14/3, first stage stride 1).
IR50_UNITS = ([(64, 64, 1)] * 3
              + [(64, 128, 2)] + [(128, 128, 1)] * 3
              + [(128, 256, 2)] + [(256, 256, 1)] * 13
              + [(256, 512, 2)] + [(512, 512, 1)] * 2)


def ir_units(num_layers: int):
    """(in_channel, depth, stride) per unit of IR-50 / IR-100 / IR-152 (modules.get_blocks)."""
    return get_blocks(num_layers)


# SE weight gains: fc1 ~ U(+-SE_GAIN1 / sqrt(depth)), fc2 ~ U(+-SE_GAIN2 / sqrt(hidden)).  Larger than a default
# init so that the gates differ across channels AND frames (a gate stuck near one value would hide a gate
# applied to the wrong frame), without saturating them (which would hide a dropped gate).
SE_GAIN1, SE_GAIN2 = 8.0, 4.0

# configs.py:61-73 (tcn.channels) and models/model.py:388-393 (embedding_dim / encoder_dim)
TCN_CHANNELS = {
    "video": [256, 256, 128, 128], "cnn_res50": [256, 256, 128, 128],
    "vggish": [64, 64, 32, 32], "logmel": [64, 64, 32, 32],
    "bert": [256, 256, 128, 128], "mfcc": [32, 32, 32, 32], "egemaps": [32, 32, 32, 32],
}
EMBEDDING_DIM = {"video": 512, "bert": 768, "cnn_res50": 512, "mfcc": 39, "vggish": 128,
                 "logmel": 128, "egemaps": 88}
ENCODER_DIM = {"video": 128, "bert": 128, "cnn_res50": 128, "mfcc": 32, "vggish": 32,
               "logmel": 32, "egemaps": 32}


def _uniform(g, shape, bound):
    return (torch.rand(shape, generator=g) * 2 - 1) * bound


def _bn(sd, p, c, g):
    """Randomised eval-mode BatchNorm (SURVEY.md section 8d, cfg 2)."""
    sd[p + ".weight"] = torch.rand(c, generator=g) + 0.5
    sd[p + ".bias"] = 0.1 * torch.randn(c, generator=g)
    sd[p + ".running_mean"] = 0.1 * torch.randn(c, generator=g)
    sd[p + ".running_var"] = torch.rand(c, generator=g) + 0.5
    sd[p + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)


def _conv(sd, key, cout, cin, k, g):
    fan_in = cin * k * k
    sd[key] = _uniform(g, (cout, cin, k, k), fan_in ** -0.5)


def visual_backbone_state_dict(seed: int = 0, units=IR50_UNITS, num_classes: int = 8,
                               spatial: int = 5, se: bool = False) -> "OrderedDict[str, torch.Tensor]":
    """``VisualBackbone.state_dict()`` layout (models/backbone.py:69-130): prefix ``backbone.``
    for the IR-50 and the unused ``logits.*`` head that strict loading still requires.  ``units``: any
    get_blocks table (ir_units(100) ...); ``se``: IR-SE units (res_layer.5.fc{1,2}.weight, drawn from their own
    generator, so every other tensor equals the se=False one)."""
    g = torch.Generator().manual_seed(seed)
    gse = torch.Generator().manual_seed(seed + 104729)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    b = "backbone."
    _conv(sd, b + "input_layer.0.weight", 64, 3, 3, g)
    _bn(sd, b + "input_layer.1", 64, g)
    sd[b + "input_layer.2.weight"] = 0.25 + 0.1 * torch.randn(64, generator=g)
    for i, (cin, depth, stride) in enumerate(units):
        u = f"{b}body.{i}."
        if cin != depth:
            _conv(sd, u + "shortcut_layer.0.weight", depth, cin, 1, g)
            _bn(sd, u + "shortcut_layer.1", depth, g)
        _bn(sd, u + "res_layer.0", cin, g)
        _conv(sd, u + "res_layer.1.weight", depth, cin, 3, g)
        sd[u + "res_layer.2.weight"] = 0.25 + 0.1 * torch.randn(depth, generator=g)
        _conv(sd, u + "res_layer.3.weight", depth, depth, 3, g)
        _bn(sd, u + "res_layer.4", depth, g)
        if se:
            hid = depth // 16
            sd[u + "res_layer.5.fc1.weight"] = _uniform(gse, (hid, depth, 1, 1), SE_GAIN1 * depth ** -0.5)
            sd[u + "res_layer.5.fc2.weight"] = _uniform(gse, (depth, hid, 1, 1), SE_GAIN2 * hid ** -0.5)
    c = units[-1][1]
    _bn(sd, b + "output_layer.0", c, g)
    fin = c * spatial * spatial
    sd[b + "output_layer.3.weight"] = _uniform(g, (512, fin), fin ** -0.5)
    sd[b + "output_layer.3.bias"] = 0.1 * torch.randn(512, generator=g)
    _bn(sd, b + "output_layer.4", 512, g)
    sd["logits.weight"] = _uniform(g, (num_classes, 512), 512 ** -0.5)
    sd["logits.bias"] = torch.zeros(num_classes)
    # registration order in Backbone.__init__ is input_layer, output_layer, body (arcface_model.py:130-146)
    order = [k for k in sd if ".input_layer." in k] + [k for k in sd if ".output_layer." in k] \
        + [k for k in sd if ".body." in k] + [k for k in sd if k.startswith("logits.")]
    return OrderedDict((k, sd[k]) for k in order)


VGGISH_CFG = (64, "M", 128, "M", 256, 256, "M", 512, 512, "M")     # models/backbone.py:43-53
VGGISH_FC = ((512 * 4 * 6, 4096), (4096, 4096), (4096, 128))        # models/backbone.py:20-27


def vggish_state_dict(seed: int = 0) -> "OrderedDict[str, torch.Tensor]":
    """``VGGish.state_dict()`` layout = vggish.pth (models/backbone.py:16-66): 18 keys
    ``features.{0,3,6,8,11,13}.{weight,bias}``, ``embeddings.{0,2,4}.{weight,bias}``.
    He-uniform weights keep the ReLU activations O(1) through the stack."""
    g = torch.Generator().manual_seed(seed + 7919)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    idx, cin = 0, 1
    for v in VGGISH_CFG:
        if v == "M":
            idx += 1
            continue
        sd[f"features.{idx}.weight"] = _uniform(g, (v, cin, 3, 3), (6.0 / (cin * 9)) ** 0.5)
        sd[f"features.{idx}.bias"] = 0.05 * torch.randn(v, generator=g)
        idx += 2
        cin = v
    for i, (fin, fout) in zip((0, 2, 4), VGGISH_FC):
        sd[f"embeddings.{i}.weight"] = _uniform(g, (fout, fin), (6.0 / fin) ** 0.5)
        sd[f"embeddings.{i}.bias"] = 0.05 * torch.randn(fout, generator=g)
    return sd


def logmel_patches(n: int, seed: int = 1234, frames: int = 96, bands: int = 64) -> torch.Tensor:
    """VGGish input examples [n, 96, 64]: log(mel + 0.01) values (vggish_input.py:37-82 /
    mel_features.py:207-236) lie in about [-4.6, 3]; here N(-1.5, 1.2)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, frames, bands, generator=g) * 1.2 - 1.5


def head_state_dict(seed: int = 0, modalities: Sequence[str] = ("video", "vggish", "bert"),
                    output_dim: int = 7, kernel_size: int = 5, modal_dim: int = 32,
                    tcn_channels: Dict[str, List[int]] = None,
                    embedding_dim: Dict[str, int] = None,
                    encoder_dim: Dict[str, int] = None) -> "OrderedDict[str, torch.Tensor]":
    """Everything of ``LFAN.state_dict()`` except ``spatial.*``: ``temporal.<m>.network.<i>.*``
    (with the reference's duplicated ``conv1``/``net.0`` and ``conv2``/``net.4`` keys,
    temporal_convolutional_model.py:24-37), ``bn.<m>.*``, ``fusion.layers.*``,
    ``regressor.*`` (models/model.py:451-485)."""
    tcn_channels = tcn_channels or TCN_CHANNELS
    embedding_dim = embedding_dim or EMBEDDING_DIM
    encoder_dim = encoder_dim or ENCODER_DIM
    g = torch.Generator().manual_seed(seed)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    for m in modalities:
        cin = embedding_dim[m]
        for i, cout in enumerate(tcn_channels[m]):
            p = f"temporal.{m}.network.{i}."
            made = {}
            for name, ci in (("conv1", cin), ("conv2", cout)):
                v = _uniform(g, (cout, ci, kernel_size), (ci * kernel_size) ** -0.5)
                gn = v.reshape(cout, -1).norm(dim=1).view(cout, 1, 1) * (torch.rand(cout, 1, 1, generator=g) + 0.5)
                bias = _uniform(g, (cout,), (ci * kernel_size) ** -0.5)
                made[name] = (bias, gn, v)
            # module registration order: conv1, conv2, then net (net.0 is conv1, net.4 is conv2)
            for nm, src in (("conv1", "conv1"), ("conv2", "conv2"), ("net.0", "conv1"), ("net.4", "conv2")):
                sd[p + nm + ".bias"], sd[p + nm + ".weight_g"], sd[p + nm + ".weight_v"] = made[src]
            if cin != cout:
                sd[p + "downsample.weight"] = _uniform(g, (cout, cin, 1), cin ** -0.5)
                sd[p + "downsample.bias"] = _uniform(g, (cout,), cin ** -0.5)
            cin = cout
    for m in modalities:
        _bn(sd, f"bn.{m}", tcn_channels[m][-1], g)
    a = "fusion.layers.self_attn."
    for m in modalities:
        d = encoder_dim[m]
        sd[f"{a}qkv_proj.{m}.weight"] = _uniform(g, (3 * modal_dim, d), (6.0 / (d + 3 * modal_dim)) ** 0.5)
        sd[f"{a}qkv_proj.{m}.bias"] = 0.05 * torch.randn(3 * modal_dim, generator=g)
    e = modal_dim * len(modalities)
    sd[a + "o_proj.weight"] = _uniform(g, (e, e), (3.0 / e) ** 0.5)
    sd[a + "o_proj.bias"] = 0.05 * torch.randn(e, generator=g)
    sd["fusion.layers.norm1.weight"] = torch.rand(e, generator=g) + 0.5
    sd["fusion.layers.norm1.bias"] = 0.1 * torch.randn(e, generator=g)
    fd = encoder_dim[modalities[0]] + e
    sd["regressor.weight"] = _uniform(g, (output_dim, fd), fd ** -0.5)
    sd["regressor.bias"] = _uniform(g, (output_dim,), fd ** -0.5)
    return sd


def lfan_state_dict(seed: int = 0, modalities: Sequence[str] = ("video", "vggish", "bert"),
                    **kw) -> "OrderedDict[str, torch.Tensor]":
    """Full ``LFAN.state_dict()`` layout; ``spatial.visual.*`` only when 'video' is a
    modality (models/model.py:455-458).  Key order follows module registration order."""
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    head = head_state_dict(seed + 1, modalities, **kw)
    for k, v in head.items():
        if k.startswith("temporal."):
            sd[k] = v
    if "video" in modalities:
        for k, v in visual_backbone_state_dict(seed).items():
            sd["spatial.visual." + k] = v
    if "logmel" in modalities:                      # models/model.py:460-463, AudioBackbone.backbone = VGGish
        for k, v in vggish_state_dict(seed).items():
            sd["spatial.audio.backbone." + k] = v
    for k, v in head.items():
        if not k.startswith("temporal."):
            sd[k] = v
    return sd


def frames(n: int, seed: int = 1234, size: int = 40) -> torch.Tensor:
    """Aligned face crops after the reference eval transform, i.e. uniform in [-1, 1]
    (base/dataset.py:503-510): [n, 3, size, size] fp32 NCHW."""
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 3, size, size, generator=g) * 2 - 1


def feature_windows(batch: int, length: int = 300, seed: int = 1234,
                    modalities: Sequence[str] = ("cnn_res50", "vggish", "bert"),
                    embedding_dim: Dict[str, int] = None) -> Dict[str, torch.Tensor]:
    """Pre-extracted feature windows [B,1,T,D_m] (shapes documented at trainer.py:461-465).
    Visual embeddings are unit-norm (arcface_model.py:151); audio/text are z-scored
    (base/dataset.py:529-536) => standard normal."""
    embedding_dim = embedding_dim or EMBEDDING_DIM
    g = torch.Generator().manual_seed(seed)
    out = {}
    for m in modalities:
        x = torch.randn(batch, 1, length, embedding_dim[m], generator=g)
        if m in ("video", "cnn_res50"):
            x = torch.nn.functional.normalize(x, dim=-1)
        out[m] = x
    return out


def raw_frames_u8(n: int, seed: int = 1234, h: int = 256, w: int = 256) -> torch.Tensor:
    """Stored aligned face crops as the reference keeps them on disk: uint8 [n, h, w, 3]
    (video.npy, abaw5_pre_processing/project/abaw5/configs.py:20,236).  Low-frequency content plus
    noise, so that the antialiased resize has structure to preserve."""
    g = torch.Generator().manual_seed(seed)
    yy = torch.arange(h, dtype=torch.float32).view(1, h, 1, 1)
    xx = torch.arange(w, dtype=torch.float32).view(1, 1, w, 1)
    ph = torch.rand(n, 1, 1, 3, generator=g) * 6.28
    fy = (torch.rand(n, 1, 1, 3, generator=g) * 3 + 1) * 6.28 / h
    fx = (torch.rand(n, 1, 1, 3, generator=g) * 3 + 1) * 6.28 / w
    base = 127.5 + 80 * torch.sin(yy * fy + xx * fx + ph)
    noise = torch.randint(-40, 41, (n, h, w, 3), generator=g).float()
    return (base + noise).clamp(0, 255).to(torch.uint8)


def waveform(seconds: float, seed: int = 1234, sample_rate: int = 16000) -> torch.Tensor:
    """Mono speech-like test signal in [-1, 1]: a few drifting harmonics, an amplitude envelope with
    pauses, and noise.  fp32 [seconds * sample_rate]."""
    g = torch.Generator().manual_seed(seed)
    n = int(round(seconds * sample_rate))
    t = torch.arange(n, dtype=torch.float64) / sample_rate
    f0 = 120.0 + 40.0 * torch.sin(2 * torch.pi * 0.7 * t)
    phase = 2 * torch.pi * torch.cumsum(f0, 0) / sample_rate
    sig = sum(a * torch.sin(h * phase) for h, a in ((1, 0.35), (2, 0.2), (3, 0.12), (5, 0.06), (9, 0.03)))
    env = (torch.sin(2 * torch.pi * 1.3 * t) > -0.3).double() * (0.6 + 0.4 * torch.sin(2 * torch.pi * 0.21 * t))
    noise = 0.02 * torch.randn(n, generator=g, dtype=torch.float64)
    return (sig * env + noise).clamp(-1, 1).float()


# configs.py:79-126 (tcn_settings used by CAN / JMT / MT)
TCN_SETTINGS = {
    "video": {"input_dim": 512, "channel": [256, 256, 128, 128, 128], "kernel_size": 5},
    "cnn_res50": {"input_dim": 512, "channel": [256, 256, 128, 128], "kernel_size": 5},
    "vggish": {"input_dim": 128, "channel": [128, 128, 64, 64], "kernel_size": 5},
    "logmel": {"input_dim": 128, "channel": [128, 128, 64, 64, 64], "kernel_size": 5},
    "bert": {"input_dim": 768, "channel": [256, 256, 128, 128], "kernel_size": 5},
}


def _tcn(sd, prefix, cin, channels, k, g):
    """``TemporalConvNet.state_dict()`` keys under ``prefix`` (temporal_convolutional_model.py:21-75)."""
    for i, cout in enumerate(channels):
        p = f"{prefix}network.{i}."
        made = {}
        for name, ci in (("conv1", cin), ("conv2", cout)):
            v = _uniform(g, (cout, ci, k), (ci * k) ** -0.5)
            gn = v.reshape(cout, -1).norm(dim=1).view(cout, 1, 1) * (torch.rand(cout, 1, 1, generator=g) + 0.5)
            made[name] = (_uniform(g, (cout,), (ci * k) ** -0.5), gn, v)
        for nm, src in (("conv1", "conv1"), ("conv2", "conv2"), ("net.0", "conv1"), ("net.4", "conv2")):
            sd[p + nm + ".bias"], sd[p + nm + ".weight_g"], sd[p + nm + ".weight_v"] = made[src]
        if cin != cout:
            sd[p + "downsample.weight"] = _uniform(g, (cout, cin, 1), cin ** -0.5)
            sd[p + "downsample.bias"] = _uniform(g, (cout,), cin ** -0.5)
        cin = cout


def _linear(sd, p, fout, fin, g):
    sd[p + ".weight"] = _uniform(g, (fout, fin), (3.0 / fin) ** 0.5)
    sd[p + ".bias"] = 0.1 * torch.randn(fout, generator=g)


def _mha(sd, p, e, g):
    """nn.MultiheadAttention(e, 1): in_proj_weight [3e, e], in_proj_bias, out_proj.{weight,bias}."""
    sd[p + ".in_proj_weight"] = _uniform(g, (3 * e, e), (3.0 / e) ** 0.5)
    sd[p + ".in_proj_bias"] = 0.1 * torch.randn(3 * e, generator=g)
    _linear(sd, p + ".out_proj", e, e, g)


def _encoder_block(sd, p, e, hidden, g):
    """TransformerEncoderBlock(e, 1, hidden, 1) (models/model.py:716-750)."""
    q = p + ".layers.0"
    _mha(sd, q + ".attention", e, g)
    _linear(sd, q + ".feed_forward.0", hidden, e, g)
    _linear(sd, q + ".feed_forward.2", e, hidden, g)
    for n in ("layer_norm1", "layer_norm2"):
        sd[f"{q}.{n}.weight"] = torch.rand(e, generator=g) + 0.5
        sd[f"{q}.{n}.bias"] = 0.1 * torch.randn(e, generator=g)


def _head_common(sd, modalities, settings, g):
    for m in modalities:
        _tcn(sd, f"temporal.{m}.", settings[m]["input_dim"], settings[m]["channel"], settings[m]["kernel_size"], g)
    for m in modalities:
        _bn(sd, f"bn.{m}", settings[m]["channel"][-1], g)


def _spatial(sd, modalities, seed):
    if "video" in modalities:
        for k, v in visual_backbone_state_dict(seed).items():
            sd["spatial.visual." + k] = v
    if "logmel" in modalities:
        for k, v in vggish_state_dict(seed).items():
            sd["spatial.audio.backbone." + k] = v


def can_state_dict(seed: int = 0, modalities: Sequence[str] = ("video", "vggish", "bert"), output_dim: int = 7,
                   settings: Dict[str, dict] = None) -> "OrderedDict[str, torch.Tensor]":
    """``CAN.state_dict()`` layout (models/model.py:571-622): temporal, bn, spatial, fuse.attn.<i>,
    fuse.weights, conv_c (unused by forward), bn1, fc1, fc2."""
    settings = settings or TCN_SETTINGS
    g = torch.Generator().manual_seed(seed + 104729)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    _head_common(sd, modalities, settings, g)
    _spatial(sd, modalities, seed)
    n = len(modalities)
    for i, m in enumerate(modalities):
        _linear(sd, f"fuse.attn.{i}", 128, settings[m]["channel"][-1], g)
    _linear(sd, "fuse.weights", 128 * n, 128 * n, g)
    sd["conv_c.weight"] = _uniform(g, (128, 128 * n, 1), (128 * n) ** -0.5)
    sd["conv_c.bias"] = 0.1 * torch.randn(128, generator=g)
    _bn(sd, "bn1", 128 * n, g)
    _linear(sd, "fc1", 128 * n, 128 * n, g)
    _linear(sd, "fc2", output_dim, 128 * n, g)
    return sd


def jmt_state_dict(seed: int = 0, modalities: Sequence[str] = ("video", "vggish"), output_dim: int = 7,
                   model_name: str = "JMT", settings: Dict[str, dict] = None) -> "OrderedDict[str, torch.Tensor]":
    """``JMT.state_dict()`` layout for model_name 'JMT' or 'MT' (models/model.py:895-1105)."""
    settings = settings or TCN_SETTINGS
    g = torch.Generator().manual_seed(seed + 1299709)
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    _head_common(sd, modalities, settings, g)
    _spatial(sd, modalities, seed)
    f = "fuse."
    encs = ("visual_encoder", "audio_encoder", "jr_encoder", "final_encoder") if model_name == "JMT" else \
        ("visual_encoder", "audio_encoder", "final_encoder")
    for e in encs:
        _encoder_block(sd, f + e, 128, 128, g)
    cas = ("CA_va", "CA_av", "CA_jra", "CA_ajr", "CA_vjr", "CA_jrv") if model_name == "JMT" else ("CA_va", "CA_av")
    for c in cas:
        _mha(sd, f + c, 128, g)
    _linear(sd, f + "reduce_feats_dim", 128, 256, g)
    _linear(sd, f + "augment_audio_feats_dim", 128, 64, g)
    _mha(sd, f + "final_self_attention", 128, g)
    _bn(sd, "bn1", 128, g)
    _linear(sd, "fc1", 128, 128, g)
    _linear(sd, "fc2", output_dim, 128, g)
    return sd
