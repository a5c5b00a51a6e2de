"""Host-side mirrors of the reference's nn.Modules for the LFAN hot path.

Same constructor signatures, forward signatures and ``state_dict()`` key layout as
/root/reference/models/{arcface_model,backbone,temporal_convolutional_model,transformer,model}.py
(SURVEY.md section 8b), so ``load_state_dict(strict=True)`` of a reference checkpoint works and
the modules drop in under experiment.py:298-315 / trainer.py:368,485,852.

The torch sub-modules declared here are PARAMETER CONTAINERS ONLY (they pin names and shapes);
none of their ``forward`` methods is ever called.  ``forward`` of the mirrors packs the weights
once (packing.py), keeps them resident on the GPU and calls the sm_100a kernels through the
C-ABI (engine.py).  The sub-modules are inference-only (a forward in training mode with grad
enabled raises instead of silently running something else); LFAN.forward in training mode runs
the head's training plan (training.py, csrc/train.cu) and is attached to autograd.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch
from torch import nn
from torch.nn.utils import weight_norm

from . import packing
from .engine import FusionEngine, Ir50Engine, TcnEngine, VggishEngine

TASKS = ("CLASSIFICATION", "REGRESSION")          # constants.py:17-20


class _PackedModule(nn.Module):
    """Caches a device engine built from the current parameters; dropped whenever the
    parameters may have changed: load_state_dict, .to()/.cuda()/.half(), explicit repack(), a
    training-mode forward (``_mark_dirty``), or any in-place update of a parameter or buffer since
    the engine was packed (``optimizer.step()`` of a torch optimizer bumps the tensors' version
    counters; ``_fresh_engine`` compares their sum with the stamp taken at packing time)."""

    def __init__(self):
        super().__init__()
        self.__dict__["_engine"] = None
        self.__dict__["_stamp"] = None
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.repack())

    def repack(self):
        self.__dict__["_engine"] = None
        self.__dict__["_stamp"] = None
        self.__dict__.pop("_ptensors", None)
        for m in self.children():
            if isinstance(m, _PackedModule):
                m.repack()

    def _stamp_tensors(self):
        """Tensors whose in-place modification invalidates this module's packed engine."""
        return list(self.parameters()) + list(self.buffers())

    def _version_stamp(self) -> int:
        ts = self.__dict__.get("_ptensors")
        if ts is None:
            ts = self.__dict__["_ptensors"] = self._stamp_tensors()
        return sum(t._version for t in ts)

    def _fresh_engine(self):
        """The cached engine, or None if there is none or the weights changed since it was packed."""
        eng = self.__dict__["_engine"]
        if eng is not None and self.__dict__["_stamp"] != self._version_stamp():
            self.repack()                                      # weights were updated in place: re-pack
            eng = None
        return eng

    def _set_engine(self, eng):
        self.__dict__["_engine"] = eng
        self.__dict__["_stamp"] = self._version_stamp()
        return eng

    def _apply(self, fn, *a, **kw):
        self.__dict__["_engine"] = None
        self.__dict__["_stamp"] = None
        self.__dict__.pop("_ptensors", None)
        self.__dict__.pop("_trainer", None)      # a training plan holds raw pointers into the old parameter storage
        self.__dict__.pop("_preproc", None)
        self.__dict__.pop("_logmel", None)
        self.__dict__.pop("_head_graphs", None)
        self.__dict__.pop("_head_streams", None)
        return super()._apply(fn, *a, **kw)

    def _device(self) -> torch.device:
        return next(self.parameters()).device

    def _check_inference(self):
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            raise NotImplementedError(
                "this sub-module's B200 kernels are forward-only: call .eval() or run under torch.no_grad() "
                "(training runs through LFAN.forward in train mode / training.HeadTrainer)")


class Flatten(nn.Module):                      # models/arcface_model.py:12-14 (container only)
    pass


class bottleneck_IR(nn.Module):
    """Parameter layout of models/arcface_model.py:44-60: shortcut_layer.{0,1} (projection units
    only) and res_layer.{0: BN, 1: conv3x3, 2: PReLU, 3: conv3x3/stride, 4: BN}."""

    def __init__(self, in_channel: int, depth: int, stride: int):
        super().__init__()
        if in_channel == depth:
            self.shortcut_layer = nn.MaxPool2d(1, stride)
        else:
            self.shortcut_layer = nn.Sequential(nn.Conv2d(in_channel, depth, (1, 1), stride, bias=False),
                                                nn.BatchNorm2d(depth))
        self.res_layer = nn.Sequential(nn.BatchNorm2d(in_channel),
                                       nn.Conv2d(in_channel, depth, (3, 3), (1, 1), 1, bias=False),
                                       nn.PReLU(depth),
                                       nn.Conv2d(depth, depth, (3, 3), stride, 1, bias=False),
                                       nn.BatchNorm2d(depth))


class SEModule(nn.Module):
    """Parameter layout of models/arcface_model.py:23-41: fc1 / fc2 1x1 convs without bias (the gate
    sigmoid(fc2(relu(fc1(mean_hw(x))))) runs in se.cu)."""

    def __init__(self, channels: int, reduction: int):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc1 = nn.Conv2d(channels, channels // reduction, kernel_size=1, padding=0, bias=False)
        self.relu = nn.ReLU(inplace=True)
        self.fc2 = nn.Conv2d(channels // reduction, channels, kernel_size=1, padding=0, bias=False)
        self.sigmoid = nn.Sigmoid()


class bottleneck_IR_SE(bottleneck_IR):
    """Parameter layout of models/arcface_model.py:63-84: bottleneck_IR plus res_layer.5 = SEModule(depth, 16)."""

    def __init__(self, in_channel: int, depth: int, stride: int):
        super().__init__(in_channel, depth, stride)
        self.res_layer.append(SEModule(depth, 16))


def get_blocks(num_layers: int):
    """Unit table of models/arcface_model.py:95-117 as (in_channel, depth, stride) triples."""
    def stage(cin, depth, n, stride=2):
        return [(cin, depth, stride)] + [(depth, depth, 1)] * (n - 1)
    if num_layers == 50:
        return stage(64, 64, 3, 1) + stage(64, 128, 4) + stage(128, 256, 14) + stage(256, 512, 3)
    if num_layers == 100:
        return stage(64, 64, 3) + stage(64, 128, 13) + stage(128, 256, 30) + stage(256, 512, 3)
    if num_layers == 152:
        return stage(64, 64, 3) + stage(64, 128, 8) + stage(128, 256, 36) + stage(256, 512, 3)
    raise AssertionError("num_layers should be 50,100, or 152")


def _output_layer(channels: int, spatial: int, drop_ratio: float, emb: int = 512) -> nn.Sequential:
    return nn.Sequential(nn.BatchNorm2d(channels), nn.Dropout(drop_ratio), Flatten(),
                         nn.Linear(channels * spatial * spatial, emb), nn.BatchNorm1d(emb))


class Backbone(_PackedModule):
    """models/arcface_model.py:120-151.  ``forward(x[N,3,H,W]) -> [N,512]`` unit-norm embeddings.
    The CUDA plan is built for the spatial size the output_layer expects (H = 8*sqrt(fc_in/512));
    as in the reference, a mismatching input size is an error."""

    frames_per_pass = 2400      # frames per pass of IR-50 / IR-SE-50 plans (workspace ~1.25 MB per 40 px frame)
    # IR-100 / IR-152 (total stride 16, 112 px inputs for the 7x7 head): ~4.8 MB of workspace per frame; 512 frames
    # give stage 4 (7 x 7 px per frame) about 200 output tiles of 128 px x 256 channels, more than the 148 SMs
    deep_frames_per_pass = 512

    def __init__(self, num_layers, drop_ratio, input_channels=3, mode='ir'):
        super().__init__()
        assert num_layers in [50, 100, 152], 'num_layers should be 50,100, or 152'
        assert mode in ['ir', 'ir_se'], 'mode should be ir or ir_se'
        if input_channels != 3:
            raise NotImplementedError("the stem kernel is built for 3 input channels (RGB face crops)")
        unit_module = bottleneck_IR if mode == 'ir' else bottleneck_IR_SE
        self.input_layer = nn.Sequential(nn.Conv2d(input_channels, 64, (3, 3), 1, 1, bias=False),
                                         nn.BatchNorm2d(64), nn.PReLU(64))
        self.output_layer = _output_layer(512, 7, drop_ratio)
        self.body = nn.Sequential(*[unit_module(c, d, s) for c, d, s in get_blocks(num_layers)])
        self._strides = [s for _, _, s in get_blocks(num_layers)]
        self._num_layers = num_layers

    def _build_engine(self) -> Ir50Engine:
        sd = {k: v.detach().cpu() for k, v in self.state_dict().items()}
        total_stride = 1
        for s in self._strides:
            total_stride *= s
        fc_in = sd["output_layer.3.weight"].shape[1]
        spatial = int(round((fc_in / 512) ** 0.5))
        # the reference's strides are carried by the modules, not the state_dict
        pk = packing.pack_ir50(sd, prefix="", in_hw=spatial * total_stride, strides=self._strides)
        fpp = self.frames_per_pass if self._num_layers == 50 else self.deep_frames_per_pass
        return Ir50Engine(pk, self._device(), fpp)

    def engine(self) -> Ir50Engine:
        eng = self._fresh_engine()
        return eng if eng is not None else self._set_engine(self._build_engine())

    def forward(self, x):
        if self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            self._check_inference()
        return self.engine().forward(x.float())


class VisualBackbone(_PackedModule):
    """models/backbone.py:69-130: IR-50 (mode='ir') or IR-SE-50 (mode='ir_se') with the 5x5 head (40x40
    inputs) plus the unused ``logits`` Linear that strict state_dict loading requires."""

    def __init__(self, input_channels=3, num_classes=8, use_pretrained=True, state_dict_path="", mode="ir",
                 embedding_dim=512):
        super().__init__()
        self.backbone = Backbone(input_channels=input_channels, num_layers=50, drop_ratio=0.4, mode=mode)
        if use_pretrained:
            state_dict = torch.load(state_dict_path, map_location='cpu')
            if "backbone" in list(state_dict.keys())[0]:
                self.backbone.output_layer = _output_layer(embedding_dim, 5, 0.4, embedding_dim)
                self.backbone.load_state_dict({k[9:]: v for k, v in state_dict.items() if "logits" not in k})
            else:
                self.backbone.load_state_dict(state_dict)
            for param in self.backbone.parameters():
                param.requires_grad = False
        # the reference re-creates (and re-initialises) the head after loading (backbone.py:99-121)
        self.backbone.output_layer = _output_layer(embedding_dim, 5, 0.4, embedding_dim)
        self.logits = nn.Linear(in_features=embedding_dim, out_features=num_classes)
        for m in self.backbone.output_layer.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                nn.init.constant_(m.bias, 0)
        nn.init.xavier_uniform_(self.logits.weight)
        nn.init.constant_(self.logits.bias, 0)
        self.backbone.repack()

    def forward(self, x):
        return self.backbone(x)

    def extract(self, x):
        return self.backbone(x)


# ----------------------------------------------------------------------------------------------
# VGGish (models/backbone.py:16-66, :133-145)
# ----------------------------------------------------------------------------------------------
def make_layers() -> nn.Sequential:
    """Parameter layout of models/backbone.py:43-53 (features.{0,3,6,8,11,13})."""
    layers, in_channels = [], 1
    for v in packing.VGGISH_CFG:
        if v == "M":
            layers += [nn.MaxPool2d(kernel_size=2, stride=2)]
        else:
            layers += [nn.Conv2d(in_channels, v, kernel_size=3, padding=1), nn.ReLU(inplace=True)]
            in_channels = v
    return nn.Sequential(*layers)


class VGG(_PackedModule):
    """models/backbone.py:16-40.  ``forward(x[N,1,96,64]) -> [N,128]``."""

    patches_per_pass = 1200     # patches per pass of the plan (workspace ~0.8 MB per patch)

    def __init__(self, features):
        super().__init__()
        self.features = features
        self.embeddings = nn.Sequential(nn.Linear(512 * 4 * 6, 4096), nn.ReLU(True), nn.Linear(4096, 4096),
                                        nn.ReLU(True), nn.Linear(4096, 128))

    def engine(self) -> VggishEngine:
        eng = self._fresh_engine()
        if eng is None:
            sd = {k: v.detach().cpu() for k, v in self.state_dict().items()}
            eng = self._set_engine(VggishEngine(packing.pack_vggish(sd), self._device(), self.patches_per_pass))
        return eng

    def forward(self, x):
        self._check_inference()
        if x.dim() != 4 or x.shape[1] != 1:
            raise ValueError(f"expected [N,1,96,64], got {tuple(x.shape)}")
        return self.engine().forward(x[:, 0].float())


def _vgg():
    return VGG(make_layers())


class VGGish(VGG):
    """models/backbone.py:59-66: takes [N,96,64] examples (adds the channel axis itself)."""

    def __init__(self):
        super().__init__(make_layers())

    def forward(self, x, fs=None):
        x = torch.as_tensor(x, device=self._device())[:, None, :, :].float()
        return VGG.forward(self, x)


class AudioBackbone(_PackedModule):
    """models/backbone.py:133-145: frozen VGGish; ``forward(x[N,96,64]) -> [N,128]``."""

    def __init__(self):
        super().__init__()
        self.backbone = VGGish()
        for param in self.backbone.parameters():
            param.requires_grad = False

    def forward(self, x, extract_vggish=False):
        return self.backbone(x)


# ----------------------------------------------------------------------------------------------
# TCN (models/temporal_convolutional_model.py)
# ----------------------------------------------------------------------------------------------
class Chomp1d(nn.Module):                       # :12-18 (container only; the kernel is causal by construction)
    def __init__(self, chomp_size):
        super().__init__()
        self.chomp_size = chomp_size


class TemporalBlock(_PackedModule):
    """:21-54.  ``forward(x[B,C_in,T]) -> [B,C_out,T]``.  conv1/conv2 are registered twice (attribute
    and inside ``net``) exactly like the reference, which is what gives the duplicated
    ``conv1.*`` / ``net.0.*`` state_dict keys."""

    def __init__(self, n_inputs, n_outputs, kernel_size, stride, dilation, padding, dropout=0.2):
        super().__init__()
        if stride != 1 or padding != (kernel_size - 1) * dilation:
            raise NotImplementedError("the kernel implements the causal configuration stride=1, padding=(k-1)*dilation")
        self.conv1 = weight_norm(nn.Conv1d(n_inputs, n_outputs, kernel_size, stride=stride, padding=padding,
                                           dilation=dilation))
        self.chomp1 = Chomp1d(padding)
        self.relu1 = nn.LeakyReLU()
        self.dropout1 = nn.Dropout(dropout)
        self.conv2 = weight_norm(nn.Conv1d(n_outputs, n_outputs, kernel_size, stride=stride, padding=padding,
                                           dilation=dilation))
        self.chomp2 = Chomp1d(padding)
        self.relu2 = nn.LeakyReLU()
        self.dropout2 = nn.Dropout(dropout)
        self.net = nn.Sequential(self.conv1, self.chomp1, self.relu1, self.dropout1,
                                 self.conv2, self.chomp2, self.relu2, self.dropout2)
        self.downsample = nn.Conv1d(n_inputs, n_outputs, 1) if n_inputs != n_outputs else None
        self.relu = nn.LeakyReLU()
        self.dilation = dilation
        if self.downsample is not None:
            nn.init.xavier_uniform_(self.downsample.weight, gain=2 ** 0.5)

    def packed(self, sd=None, prefix="") -> dict:
        sd = sd if sd is not None else {k: v.detach().cpu() for k, v in self.state_dict().items()}
        w1 = packing.weight_norm_effective(sd[prefix + "conv1.weight_g"], sd[prefix + "conv1.weight_v"])
        w2 = packing.weight_norm_effective(sd[prefix + "conv2.weight_g"], sd[prefix + "conv2.weight_v"])
        blk = {"c_in": int(w1.shape[1]), "c_out": int(w1.shape[0]), "kernel_size": int(w1.shape[2]),
               "dilation": int(self.dilation),
               "w1": w1.permute(2, 1, 0).float().contiguous(), "b1": sd[prefix + "conv1.bias"].float().contiguous(),
               "w2": w2.permute(2, 1, 0).float().contiguous(), "b2": sd[prefix + "conv2.bias"].float().contiguous(),
               "wd": None, "bd": None, "post_scale": None, "post_shift": None}
        if self.downsample is not None:
            blk["wd"] = sd[prefix + "downsample.weight"][:, :, 0].t().float().contiguous()
            blk["bd"] = sd[prefix + "downsample.bias"].float().contiguous()
        return blk

    def forward(self, x):
        self._check_inference()
        eng = self._fresh_engine()
        if eng is None:
            eng = self._set_engine(TcnEngine([self.packed()], self._device()))
        return eng.forward(x.float().transpose(1, 2)).transpose(1, 2)


class TemporalConvNet(_PackedModule):
    """:57-75.  ``forward(x[B,C,T]) -> [B,C',T]``; level i has dilation 2**i."""

    def __init__(self, num_inputs, num_channels, kernel_size=2, dropout=0.2, max_length=200, attention=0):
        super().__init__()
        if attention:
            raise NotImplementedError("AttentionBlock is dead code in the reference (attention=0 always; it calls .cuda())")
        layers = []
        for i, out_channels in enumerate(num_channels):
            d = 2 ** i
            in_channels = num_inputs if i == 0 else num_channels[i - 1]
            layers.append(TemporalBlock(in_channels, out_channels, kernel_size, stride=1, dilation=d,
                                        padding=(kernel_size - 1) * d, dropout=dropout))
        self.network = nn.Sequential(*layers)

    def packed_blocks(self, post_scale=None, post_shift=None) -> List[dict]:
        blocks = [b.packed() for b in self.network]
        if post_scale is not None:
            blocks[-1]["post_scale"], blocks[-1]["post_shift"] = post_scale, post_shift
        return blocks

    def forward_time_major(self, x):
        """x [B,T,C] -> [B,T,C'] without the reference's transposes."""
        eng = self._fresh_engine()
        if eng is None:
            eng = self._set_engine(TcnEngine(self.packed_blocks(), self._device()))
        return eng.forward(x)

    def forward(self, x):
        self._check_inference()
        return self.forward_time_major(x.float().transpose(1, 2)).transpose(1, 2)


# ----------------------------------------------------------------------------------------------
# Cross-modal attention (models/transformer.py)
# ----------------------------------------------------------------------------------------------
class MultimodalMultiheadAttention(nn.Module):
    """Parameter layout of :102-131 (qkv_proj.<modal>, o_proj)."""

    def __init__(self, modalities, input_dim, modal_dim, num_heads):
        super().__init__()
        assert modal_dim % num_heads == 0, "Embedding dimension must be 0 modulo number of heads."
        self.modalities = modalities
        self.embed_dim = modal_dim
        self.num_heads = num_heads
        self.head_dim = modal_dim // num_heads
        self.qkv_proj = nn.ModuleDict({m: nn.Linear(input_dim[m], 3 * modal_dim) for m in modalities})
        e = modal_dim * len(modalities)
        self.o_proj = nn.Linear(e, e)
        for m in modalities:
            nn.init.xavier_uniform_(self.qkv_proj[m].weight)
            self.qkv_proj[m].bias.data.fill_(0)
        nn.init.xavier_uniform_(self.o_proj.weight)
        self.o_proj.bias.data.fill_(0)


class MultiModalEncoderBlock(nn.Module):
    """Parameter layout of :168-190 (self_attn, norm1; dropout is inert in eval)."""

    def __init__(self, modalities, input_dim, modal_dim, num_heads, dropout=0.0):
        super().__init__()
        self.self_attn = MultimodalMultiheadAttention(modalities, input_dim, modal_dim, num_heads)
        self.norm1 = nn.LayerNorm(modal_dim * len(modalities))
        self.dropout = nn.Dropout(dropout)


class MultimodalTransformerEncoder(_PackedModule):
    """:200-215.  ``forward(x: dict[modal -> [B,T,D_m]]) -> [B,T,modal_dim*M]``."""

    def __init__(self, modalities, input_dim, modal_dim, num_heads, dropout=0.0):
        super().__init__()
        self.layers = MultiModalEncoderBlock(modalities, input_dim, modal_dim, num_heads, dropout)
        self.modalities = list(modalities)
        self.modal_dim = modal_dim
        self.num_heads = num_heads

    def packed(self, regressor: Optional[nn.Linear] = None) -> dict:
        sd = {"fusion." + k: v.detach().cpu() for k, v in self.state_dict().items()}
        e = self.modal_dim * len(self.modalities)
        d0 = self.layers.self_attn.qkv_proj[self.modalities[0]].in_features
        if regressor is None:          # stand-alone use: a 1-output zero classifier that is ignored
            sd["regressor.weight"], sd["regressor.bias"] = torch.zeros(1, d0 + e), torch.zeros(1)
        else:
            sd["regressor.weight"], sd["regressor.bias"] = regressor.weight.detach().cpu(), regressor.bias.detach().cpu()
        return packing.pack_fusion(sd, self.modalities, self.modal_dim, self.num_heads)

    def forward(self, x, mask=None):
        self._check_inference()
        if mask is not None:
            raise NotImplementedError("mask is never passed on the LFAN path (model.py:517)")
        eng = self._fresh_engine()
        if eng is None:
            eng = self._set_engine(FusionEngine(self.packed(), self._device()))
        B, T, _ = x[self.modalities[0]].shape
        feats = [x[m].float().reshape(B * T, -1) for m in self.modalities]
        _, fused = eng.forward(feats, want_fused=True)
        return fused.view(B, T, -1)

    def get_attention_maps(self, x, mask=None):
        """transformer.py:211-215: ``[attention]`` with attention [B, num_heads, T, M, M] (the softmax
        of the modality-by-modality scores, one 3x3 map per frame and head)."""
        import ctypes as C
        from . import _capi, engine as E
        if mask is not None:
            raise NotImplementedError("mask is never passed on the LFAN path (model.py:517)")
        B, T, _ = x[self.modalities[0]].shape
        rows = B * T
        attn = self.layers.self_attn
        qkv = [E.linear(x[m].float().reshape(rows, -1).contiguous(), attn.qkv_proj[m].weight, attn.qkv_proj[m].bias)
               for m in self.modalities]
        ptrs = (C.c_void_p * len(qkv))(*[t.data_ptr() for t in qkv])
        M, H = len(self.modalities), self.num_heads
        maps = torch.empty(rows, H, M, M, dtype=torch.float32, device=qkv[0].device)
        with torch.cuda.device(maps.device):
            _capi.check(_capi.lib().cer_modal_attention_maps(ptrs, rows, M, H, self.modal_dim // H, maps.data_ptr(),
                                                             _capi.current_stream_ptr()), "cer_modal_attention_maps")
        return [maps.view(B, T, H, M, M).permute(0, 2, 1, 3, 4)]


# ----------------------------------------------------------------------------------------------
# LFAN (models/model.py:375-526)
# ----------------------------------------------------------------------------------------------
class LFAN(_PackedModule):
    """Drop-in for models/model.py:375-526.  After construction call ``init()`` (as
    experiment.py:298-315 does); ``forward(X: dict) -> [B, example_length, output_dim]``.
    Like the reference, forward re-binds the entries of ``X`` (to the [B,T,C] encoded features).
    """

    def __init__(self, backbone_settings, output_dim: int, task: str, modality=['frame'], kernel_size=5,
                 example_length=300, tcn_attention=0,
                 tcn_channel={'video': [512, 256, 256, 128], 'cnn_res50': [512, 256, 256, 128],
                              'mfcc': [32, 32, 32, 32], 'vggish': [32, 32, 32, 32], 'logmel': [32, 32, 32, 32]},
                 embedding_dim={'video': 512, 'bert': 768, 'cnn_res50': 512, 'mfcc': 39, 'vggish': 128,
                                'logmel': 128, 'egemaps': 88},
                 encoder_dim={'video': 128, 'bert': 128, 'cnn_res50': 128, 'mfcc': 32, 'vggish': 32, 'logmel': 32,
                              'egemaps': 32},
                 modal_dim=32, num_heads=2, root_dir='', device='cuda'):
        super().__init__()
        assert task in TASKS, task
        self.task = task
        self.output_dim = output_dim
        self.backbone_settings = backbone_settings
        self.root_dir = root_dir
        self.device = device
        self.modality = modality
        self.kernel_size = kernel_size
        self.example_length = example_length
        self.tcn_channel = tcn_channel
        self.tcn_attention = tcn_attention
        self.embedding_dim = embedding_dim
        self.encoder_dim = encoder_dim
        self.outputs = {}
        self.temporal, self.fusion = nn.ModuleDict(), None
        self.num_heads = num_heads
        self.modal_dim = modal_dim
        self.final_dim = self.encoder_dim[self.modality[0]] + self.modal_dim * len(self.modality)
        self.spatial = nn.ModuleDict()
        self.bn = nn.ModuleDict()

    def load_visual_backbone(self, backbone_settings, state_dict=None):
        resnet = VisualBackbone(mode='ir', use_pretrained=False)
        if state_dict is None:
            state_dict = torch.load(os.path.join(self.root_dir, backbone_settings['visual_state_dict'] + ".pth"),
                                    map_location='cpu')
        resnet.load_state_dict(state_dict)
        for param in resnet.parameters():
            param.requires_grad = False
        return resnet

    def load_audio_backbone(self, backbone_settings, state_dict=None):
        """models/model.py:437-449: vggish.pth is the VGGish (not AudioBackbone) state_dict."""
        vggish = AudioBackbone()
        if state_dict is None:
            state_dict = torch.load(os.path.join(self.root_dir, backbone_settings['audio_state_dict'] + ".pth"),
                                    map_location='cpu')
        vggish.backbone.load_state_dict(state_dict)
        for param in vggish.parameters():
            param.requires_grad = False
        return vggish

    def init(self, visual_state_dict=None, audio_state_dict=None):
        """models/model.py:451-485.  ``visual_state_dict`` / ``audio_state_dict`` (optional, not in
        the reference) let a caller hand over the backbone weights directly instead of through
        root_dir/<name>.pth."""
        if 'video' in self.modality:
            self.spatial["visual"] = self.load_visual_backbone(self.backbone_settings, visual_state_dict)
        if 'logmel' in self.modality:
            self.spatial["audio"] = self.load_audio_backbone(self.backbone_settings, audio_state_dict)
        for modal in self.modality:
            self.temporal[modal] = TemporalConvNet(num_inputs=self.embedding_dim[modal], max_length=self.example_length,
                                                   num_channels=self.tcn_channel[modal], attention=self.tcn_attention,
                                                   kernel_size=self.kernel_size, dropout=0.1).to(self.device)
            self.bn[modal] = nn.BatchNorm1d(self.tcn_channel[modal][-1])
        self.fusion = MultimodalTransformerEncoder(modalities=self.modality, input_dim=self.encoder_dim,
                                                   modal_dim=self.modal_dim, num_heads=self.num_heads, dropout=0.1)
        self.regressor = nn.Linear(self.final_dim, self.output_dim)
        self.repack()

    # -- engines ------------------------------------------------------------------------------
    def _stamp_tensors(self):
        # the head's engines depend on everything but the (frozen) backbones, which track themselves
        return ([p for k, p in self.named_parameters() if not k.startswith("spatial.")]
                + [b for k, b in self.named_buffers() if not k.startswith("spatial.")])

    def _mark_dirty(self):
        """A training-mode forward ran: BatchNorm1d statistics moved (and an optimizer step usually
        follows).  The next inference forward re-packs the head."""
        self.__dict__["_dirty"] = True

    def _head_engines(self):
        if self.__dict__.pop("_dirty", False):
            self.repack()
        eng = self._fresh_engine()
        if eng is None:
            dev = self.regressor.weight.device
            tcn = {}
            for m in self.modality:
                s, t = packing._bn_affine({f"bn.{k}": v.detach().cpu() for k, v in self.bn[m].state_dict().items()}, "bn")
                tcn[m] = TcnEngine(self.temporal[m].packed_blocks(s.float(), t.float()), dev)
            fus = FusionEngine(self.fusion.packed(self.regressor), dev)
            eng = self._set_engine((tcn, fus))
        return eng

    def encode_frames(self, video: torch.Tensor) -> torch.Tensor:
        """[B,T,3,H,W] -> [B,T,512] through the IR-50 kernels (model.py:489-497)."""
        B, T = video.shape[:2]
        emb = self.spatial["visual"](video.reshape(B * T, *video.shape[2:]))
        return emb.view(B, T, -1)

    def encode_logmel(self, logmel: torch.Tensor) -> torch.Tensor:
        """[B,64,T,96] -> [B,T,128] through the VGGish kernels (model.py:499-509: one [96,64]
        example per frame, laid out as [batch, bands, length, frames])."""
        B, hh, T, ww = logmel.shape
        patches = logmel.permute(0, 2, 3, 1).contiguous().view(-1, ww, hh)
        return self.spatial["audio"](patches).view(B, T, -1)

    # The head is 25 launches of 20-80 CTAs each: a launch-latency-bound chain.  With
    # ``head_cuda_graph`` (default on) it is captured once per input shape into a CUDA graph over
    # static buffers and replayed; CER_HEAD_GRAPH=0 or any capture failure keeps the eager launches.
    head_cuda_graph = True

    # The three TCN stacks are independent chains of 8 small launches (19-76 CTAs each, latency bound): they
    # run on parallel streams (fork / join with events; inside the CUDA graph these become parallel branches)
    # and only the fusion kernel waits for all of them.  CER_HEAD_STREAMS=0 serialises them (A/B timing).
    head_parallel_streams = True

    def _forward_features_eager(self, feats: Dict[str, torch.Tensor]) -> torch.Tensor:
        tcn, fus = self._head_engines()
        mods = list(self.modality)
        dev = feats[mods[0]].device
        enc = [None] * len(mods)
        parallel = (self.head_parallel_streams and len(mods) > 1 and dev.type == "cuda"
                    and os.environ.get("CER_HEAD_STREAMS", "1") != "0")
        if not parallel:
            for i, m in enumerate(mods):
                enc[i] = tcn[m].forward(feats[m].float())
        else:
            main = torch.cuda.current_stream(dev)
            side = self.__dict__.setdefault("_head_streams", {})
            key = str(dev)
            if key not in side:
                side[key] = [torch.cuda.Stream(device=dev) for _ in range(len(mods) - 1)]
            capturing = torch.cuda.is_current_stream_capturing()
            fork = torch.cuda.Event()
            fork.record(main)
            joins = []
            for i, m in enumerate(mods):
                x = feats[m].float()
                if i == 0:
                    enc[0] = tcn[m].forward(x)
                    continue
                st = side[key][i - 1]
                st.wait_event(fork)
                with torch.cuda.stream(st):
                    enc[i] = tcn[m].forward(x)
                    ev = torch.cuda.Event()
                    ev.record(st)
                    joins.append(ev)
                if not capturing:                     # a graph's private pool keeps its blocks; eager mode must tell the allocator
                    x.record_stream(st)
                    enc[i].record_stream(main)        # allocated on the side stream, consumed on the caller's
            for ev in joins:
                main.wait_event(ev)
        for m, e in zip(mods, enc):
            feats[m] = e
        B, T, _ = enc[0].shape
        logits = fus.forward([e.view(B * T, -1) for e in enc])
        return logits.view(B, T, -1)

    def forward_features(self, feats: Dict[str, torch.Tensor]) -> torch.Tensor:
        """feats[m]: [B,T,D_m] fp32 (visual = IR-50 embeddings) -> logits [B,T,output_dim].
        As in the reference, ``feats[m]`` is re-bound to the modality's encoded [B,T,C] features."""
        from . import _capi
        _capi.require_gpu()                                        # CerError without a B200: no fallback of any kind
        if not self.head_cuda_graph or os.environ.get("CER_HEAD_GRAPH", "1") == "0" or torch.cuda.is_current_stream_capturing():
            return self._forward_features_eager(feats)
        self._head_engines()
        x0 = feats[self.modality[0]]
        key = (tuple(x0.shape[:2]), str(x0.device))
        graphs = self.__dict__.setdefault("_head_graphs", {})
        g = graphs.get(key)
        if g is None:
            ins = {m: feats[m].float().contiguous() for m in self.modality}
            out = self._forward_features_eager(dict(ins))          # warm-up: one-time kernel attribute setup, workspaces
            try:
                static_in = {m: v.clone() for m, v in ins.items()}
                graph = torch.cuda.CUDAGraph()
                torch.cuda.synchronize(x0.device)
                with torch.cuda.graph(graph):
                    static_feats = dict(static_in)
                    static_out = self._forward_features_eager(static_feats)
                g = graphs[key] = (graph, static_in, static_feats, static_out)
            except Exception:                                       # capture not possible here: stay eager for this shape
                graphs[key] = False
                g = False
            if g is False:
                return self._forward_features_eager(feats)
        if g is False:
            return self._forward_features_eager(feats)
        graph, static_in, static_feats, static_out = g
        for m in self.modality:
            static_in[m].copy_(feats[m])
        graph.replay()
        for m in self.modality:
            feats[m] = static_feats[m].clone()
        return static_out.clone()

    def repack(self):
        self.__dict__.pop("_head_graphs", None)                     # graphs hold the old packed weights' pointers
        super().repack()

    def _training_forward(self, X):
        """model.train() + grad enabled (trainer.py:365-391): the frozen backbones run their
        inference kernels under no_grad (the CUDA kernels fold BatchNorm, i.e. the backbones stay in
        eval mode -- the reference would switch IR-50's BatchNorms to batch statistics under
        model.train(); train from pre-extracted features for step-for-step parity), the head runs
        the training plan and is attached to autograd."""
        from . import training
        with torch.no_grad():
            if 'video' in X:
                X['video'] = self.encode_frames(X['video']).unsqueeze(1)
            if 'logmel' in X:
                X['logmel'] = self.encode_logmel(X['logmel']).unsqueeze(1)
        feats = {m: X[m].squeeze(1) for m in self.modality}
        self._mark_dirty()
        out = training.forward_with_grad(self, feats)
        for m in X:
            X[m] = feats.get(m, X[m])
        if self.task == "REGRESSION":
            out = torch.tanh(out)
        return out

    def forward(self, X):
        if self.training and torch.is_grad_enabled():
            return self._training_forward(X)
        if 'video' in X:
            X['video'] = self.encode_frames(X['video']).unsqueeze(1)
        if 'logmel' in X:
            X['logmel'] = self.encode_logmel(X['logmel']).unsqueeze(1)
        for modal in X:
            X[modal] = X[modal].squeeze(1)
        batch_size = X[self.modality[0]].shape[0]
        out = self.forward_features(X)
        out = out.reshape(batch_size, self.example_length, -1)
        if self.task == "REGRESSION":
            from .engine import tanh_
            out = tanh_(out.contiguous())
        return out
