"""Host-side mirrors of the reference's alternative fusion heads: CAN (models/model.py:529-684)
and JMT / MT (:709-750, :895-1167), selected by ``--model_name`` (experiment.py:317-347).

Same constructors, ``forward`` signatures and ``state_dict()`` layouts as the reference (checked
key by key against listings produced by the reference: tests/golden/heads.pt).  The torch
sub-modules are parameter containers; forward runs the shared backbones / TCN engines and the fp32
building blocks of csrc/heads.cu through the C-ABI.  Training (model.train() with grad enabled, or
heads_training.AltHeadTrainer.step) runs the hand-written backward of the same blocks.

Two exact savings over the reference's arithmetic (JMT / MT):
  * only the LAST slot of the stacked cross-attention outputs is returned (``out_feats[:, :, -1, :]``,
    model.py:975) and nn.MultiheadAttention treats the stack slots as independent batch entries, so
    the other slots -- and, for JMT, the visual encoder that only feeds them -- are never computed;
  * the final encoder / self-attention attend over all L*B positions (the reference views the
    [L, B, S, E] stack as [L*B, S, E] and feeds sequence-first modules); attention over a set is
    permutation-equivariant, so it is run batch-major as one sequence of B*L rows.
"""
from __future__ import annotations

import os
from typing import Dict

import torch
from torch import nn

from . import engine as E
from . import packing
from .engine import TcnEngine
from .modules import AudioBackbone, TemporalConvNet, VisualBackbone, _PackedModule, TASKS


class AttentionFusion(nn.Module):
    """Parameter layout of models/model.py:529-550 (attn.<i>: Linear(C_i, 128); weights)."""

    def __init__(self, num_feats_modality: list, num_out_feats: int = 256):
        super().__init__()
        self.attn = nn.ModuleList([nn.Linear(n, num_out_feats) for n in num_feats_modality])
        self.weights = nn.Linear(num_out_feats * len(num_feats_modality), num_out_feats * len(num_feats_modality))
        self.num_features = num_out_feats * len(num_feats_modality)


class SequentialEncoder(nn.Sequential):                     # models/model.py:709-713 (container)
    pass


class TransformerEncoderLayer(nn.Module):
    """Parameter layout of models/model.py:728-738."""

    def __init__(self, input_dim, num_heads, hidden_dim):
        super().__init__()
        if num_heads != 1:
            raise NotImplementedError("the reference only instantiates single-head attention (model.py:910-931)")
        self.attention = nn.MultiheadAttention(input_dim, num_heads)
        self.feed_forward = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, input_dim))
        self.layer_norm1 = nn.LayerNorm(input_dim)
        self.layer_norm2 = nn.LayerNorm(input_dim)


class TransformerEncoderBlock(nn.Module):
    def __init__(self, input_dim, num_heads, hidden_dim, num_layers):
        super().__init__()
        self.layers = SequentialEncoder(*[TransformerEncoderLayer(input_dim, num_heads, hidden_dim) for _ in range(num_layers)])


def _mha(mod: nn.MultiheadAttention, q_in, kv_in, layout):
    """nn.MultiheadAttention(E, 1)(q_in, kv_in, kv_in) on rows [R, E].  ``layout``: (batch, len_q, len_k) for batch-major
    sequences of equal length, or an engine.Segments (one sequence per video, queries and keys segmented alike)."""
    e = mod.embed_dim
    W, b = mod.in_proj_weight, mod.in_proj_bias
    if q_in is kv_in:
        qkv = E.linear(q_in, W, b)
        q, k, v = qkv[:, :e], qkv[:, e:2 * e], qkv[:, 2 * e:]
    else:
        q = E.linear(q_in, W[:e], b[:e])
        kv = E.linear(kv_in, W[e:], b[e:])
        k, v = kv[:, :e], kv[:, e:]
    att = E.sdpa_segments(q, k, v, layout) if isinstance(layout, E.Segments) else E.sdpa(q, k, v, *layout)
    return E.linear(att, mod.out_proj.weight, mod.out_proj.bias)


def _encoder(block: TransformerEncoderBlock, x, layout):
    """TransformerEncoderBlock.forward (model.py:723-750) on rows; ``layout`` as for _mha."""
    for layer in block.layers:
        a = _mha(layer.attention, x, x, layout)
        x = E.add_layernorm(x, a, layer.layer_norm1.weight, layer.layer_norm1.bias, layer.layer_norm1.eps)
        ff = E.linear(E.linear(x, layer.feed_forward[0].weight, layer.feed_forward[0].bias, "relu"),
                      layer.feed_forward[2].weight, layer.feed_forward[2].bias)
        x = E.add_layernorm(x, ff, layer.layer_norm2.weight, layer.layer_norm2.bias, layer.layer_norm2.eps)
    return x


class JMTFusion(nn.Module):
    """Parameter layout of models/model.py:895-931."""

    def __init__(self, num_feats_modality: list, num_out_feats: int = 256):
        super().__init__()
        self.visual_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.audio_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.jr_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.final_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        for n in ("CA_va", "CA_av", "CA_jra", "CA_ajr", "CA_vjr", "CA_jrv"):
            setattr(self, n, nn.MultiheadAttention(128, 1))
        self.reduce_feats_dim = nn.Linear(128 * 2, 128)
        self.augment_audio_feats_dim = nn.Linear(64, 128)
        self.final_self_attention = nn.MultiheadAttention(128, 1)


class MTFusion(nn.Module):
    """Parameter layout of models/model.py:982-1012."""

    def __init__(self, num_feats_modality: list, num_out_feats: int = 256):
        super().__init__()
        self.visual_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.audio_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.final_encoder = TransformerEncoderBlock(128, 1, 128, 1)
        self.CA_va = nn.MultiheadAttention(128, 1)
        self.CA_av = nn.MultiheadAttention(128, 1)
        self.reduce_feats_dim = nn.Linear(128 * 2, 128)
        self.augment_audio_feats_dim = nn.Linear(64, 128)
        self.final_self_attention = nn.MultiheadAttention(128, 1)


class _FeatureHead(_PackedModule):
    """What CAN and JMT share (model.py:592-649, :1079-1132): TemporalConvNet + BatchNorm1d per
    modality, the frozen backbones, and the fc1 -> bn1 -> leaky_relu -> fc2 tail."""

    def _init_common(self, task, modalities, tcn_settings, backbone_settings, root_dir, device, with_up_sample):
        assert task in TASKS, task
        self.task = task
        self.device = device
        self.modalities = list(modalities)
        # registration order of the reference decides the state_dict key order
        self.temporal = nn.ModuleDict()
        if with_up_sample:
            self.up_sample = nn.ModuleDict()          # declared and left empty by CAN (model.py:587)
        self.bn = nn.ModuleDict()
        self.spatial = nn.ModuleDict()
        for modal in modalities:
            self.temporal[modal] = TemporalConvNet(num_inputs=tcn_settings[modal]['input_dim'],
                                                   num_channels=tcn_settings[modal]['channel'],
                                                   kernel_size=tcn_settings[modal]['kernel_size'])
            self.bn[modal] = nn.BatchNorm1d(tcn_settings[modal]['channel'][-1])
        self.root_dir = root_dir
        self.backbone_settings = backbone_settings

    def _load_backbones(self, modalities, visual_state_dict=None, audio_state_dict=None):
        if 'video' in modalities:
            resnet = VisualBackbone(mode='ir', use_pretrained=False)
            sd = visual_state_dict if visual_state_dict is not None else torch.load(
                os.path.join(self.root_dir, self.backbone_settings['visual_state_dict'] + ".pth"), map_location='cpu')
            resnet.load_state_dict(sd)
            for p in resnet.parameters():
                p.requires_grad = False
            self.spatial["visual"] = resnet
        if 'logmel' in modalities:
            vggish = AudioBackbone()
            sd = audio_state_dict if audio_state_dict is not None else torch.load(
                os.path.join(self.root_dir, self.backbone_settings['audio_state_dict'] + ".pth"), map_location='cpu')
            vggish.backbone.load_state_dict(sd)
            for p in vggish.parameters():
                p.requires_grad = False
            self.spatial["audio"] = vggish

    def _engines(self):
        if self.__dict__.pop("_dirty", False):
            self.repack()                      # a training forward moved the BatchNorm statistics (and weights usually follow)
        eng = self._fresh_engine()
        if eng is None:
            dev = self.fc2.weight.device
            tcn = {}
            for m in self.modalities:
                s, t = packing._bn_affine({f"bn.{k}": v.detach().cpu() for k, v in self.bn[m].state_dict().items()}, "bn")
                tcn[m] = TcnEngine(self.temporal[m].packed_blocks(s.float(), t.float()), dev)
            # fc1 followed by the eval BatchNorm1d over its output features: fold the affine into fc1
            s1, t1 = packing._bn_affine({f"bn1.{k}": v.detach().cpu() for k, v in self.bn1.state_dict().items()}, "bn1")
            w = (self.fc1.weight.detach().cpu().double() * s1.view(-1, 1)).float().contiguous().to(dev)
            b = (self.fc1.bias.detach().cpu().double() * s1 + t1).float().contiguous().to(dev)
            eng = self._set_engine((tcn, w, b))
        return eng

    def _backbones(self, X) -> Dict[str, torch.Tensor]:
        """X as the reference receives it -> feats[m] [B, T, D_m]: the frozen backbones' inference kernels."""
        if 'video' in X:
            B, T = X['video'].shape[:2]
            X['video'] = self.spatial["visual"](X['video'].reshape(B * T, *X['video'].shape[2:])).view(B, T, -1).unsqueeze(1)
        if 'logmel' in X:
            B, hh, T, ww = X['logmel'].shape
            patches = X['logmel'].permute(0, 2, 3, 1).contiguous().view(-1, ww, hh)
            X['logmel'] = self.spatial["audio"](patches).view(B, T, -1).unsqueeze(1)
        return {m: X[m].squeeze(1) for m in X}

    def _encode(self, X) -> Dict[str, torch.Tensor]:
        """X as the reference receives it -> z[m] [B, T, C_m] (TCN + BatchNorm1d), time-major."""
        return self._encode_features(self._backbones(X))

    def _training_forward(self, X):
        """model.train() + grad enabled (trainer.py:365-391): the frozen backbones run their inference kernels under
        no_grad (i.e. stay in eval mode, see INTEGRATION.md), the head runs heads_training.AltHeadTrainer and is attached
        to autograd."""
        from . import heads_training
        with torch.no_grad():
            feats = self._backbones(X)
        self.__dict__["_dirty"] = True
        out = heads_training.forward_with_grad(self, feats)
        return torch.tanh(out) if self.task == "REGRESSION" else out

    def _is_training_call(self) -> bool:
        return self.training and torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())

    def _encode_features(self, feats) -> Dict[str, torch.Tensor]:
        """feats[m] [B, T, D_m] (visual = 512-d IR-50 embeddings) -> z[m] [B, T, C_m]."""
        tcn, _, _ = self._engines()
        return {m: tcn[m].forward(feats[m].float().contiguous()) for m in feats}

    def forward_features(self, feats) -> torch.Tensor:
        """The head alone on pre-encoded features (like LFAN.forward_features): feats[m] [B, T, D_m]."""
        from . import _capi
        _capi.require_gpu()
        return self._fuse(self._encode_features(feats))

    def forward_videos(self, feats, lengths) -> torch.Tensor:
        """Whole videos laid end to end, each run as the reference runs these heads (batch 1, the whole video):
        feats[m] [sum(lengths), D_m] (visual = 512-d IR-50 embeddings) -> per-frame logits [sum(lengths), n_out].

        The TCN runs on one right-padded [n_videos, T_max, D_m] batch: its blocks are causal, so rows past a video's
        end never reach the video's frames, and the tensor-core kernel's per-row arithmetic does not depend on B or
        T, so each video's rows are those of a TCN run on that video alone.  The valid rows are then gathered back
        into the concatenated layout for the fusion head (see _fuse_videos)."""
        from . import _capi, windowing
        _capi.require_gpu()
        tcn, _, _ = self._engines()
        dev = self.fc2.weight.device
        n = len(lengths)
        t_max, idx = windowing.padded_row_index(lengths)
        idx = idx.to(dev, non_blocking=True)
        z = {}
        for m in self.modalities:
            x = feats[m].float()
            pad = torch.zeros(n * t_max, x.shape[1], dtype=torch.float32, device=dev)
            pad[idx] = x
            z[m] = tcn[m].forward(pad.view(n, t_max, -1)).view(n * t_max, -1)[idx]
        return self._fuse_videos(z, lengths)

    def _tail(self, c2d: torch.Tensor, B: int, T: int) -> torch.Tensor:
        _, w1, b1 = self._engines()
        h = E.linear(c2d, w1, b1, "leaky_relu")
        out = E.linear(h, self.fc2.weight, self.fc2.bias).view(B, T, -1)
        return E.tanh_(out.contiguous()) if self.task == "REGRESSION" else out


class CAN(_FeatureHead):
    """Drop-in for models/model.py:571-684.  ``forward(X: dict) -> [B, T, output_dim]``.
    ``visual_state_dict`` / ``audio_state_dict`` (optional, not in the reference) hand the backbone
    weights over directly instead of through root_dir/<name>.pth."""

    def __init__(self, task: str, modalities, tcn_settings, backbone_settings, output_dim, root_dir, device,
                 visual_state_dict=None, audio_state_dict=None):
        super().__init__()
        self._init_common(task, modalities, tcn_settings, backbone_settings, root_dir, device, with_up_sample=True)
        feas = [tcn_settings[m]['channel'][-1] for m in modalities]
        self.fuse = AttentionFusion(num_feats_modality=feas, num_out_feats=128)
        self.conv_c = nn.Conv1d(128 * len(modalities), 128, 1)            # declared, never used by forward (model.py:607)
        self.bn1 = nn.BatchNorm1d(128 * len(modalities))
        self.fc1 = nn.Linear(128 * len(modalities), 128 * len(modalities))
        self.fc2 = nn.Linear(128 * len(modalities), output_dim)
        self._load_backbones(modalities, visual_state_dict, audio_state_dict)

    def forward(self, X):
        if self._is_training_call():
            return self._training_forward(X)
        return self._fuse(self._encode(X))

    def _fuse(self, z):
        order = list(z)                                   # AttentionFusion walks x.values() (model.py:560-561)
        B, T, _ = z[order[0]].shape
        n = len(order)
        cat = torch.empty(B * T, 128 * n, dtype=torch.float32, device=z[order[0]].device)
        for i, m in enumerate(order):
            E.linear(z[m].view(B * T, -1), self.fuse.attn[i].weight, self.fuse.attn[i].bias, out=cat[:, 128 * i:128 * (i + 1)])
        gate = E.linear(cat, self.fuse.weights.weight, self.fuse.weights.bias)
        return self._tail(E.softmax_gate(gate, cat), B, T)

    def _fuse_videos(self, z, lengths):
        """AttentionFusion + tail row by row (frame_head(): one result per frame whatever else is in the call, so a
        video's logits equal a StreamSession's for the same frames)."""
        return self.frame_head().forward([z[m] for m in self.modalities], self.task == "REGRESSION")

    def frame_head(self) -> E.CanHeadEngine:
        """AttentionFusion + tail as one row-invariant launch over the current weights (what streaming.StreamSession
        runs; _fuse keeps its own launches).  A new engine whenever _engines() repacks."""
        eng = self._engines()
        cached = self.__dict__.get("_frame_head")
        if cached is None or cached[0] is not eng:
            _, w1, b1 = eng
            f = self.fuse
            head = E.CanHeadEngine([(a.weight, a.bias) for a in f.attn], (f.weights.weight, f.weights.bias), (w1, b1),
                                   (self.fc2.weight, self.fc2.bias), w1.device)
            cached = self.__dict__["_frame_head"] = (eng, head)
        return cached[1]


class JMT(_FeatureHead):
    """Drop-in for models/model.py:1051-1167 (``model_name`` 'JMT' or 'MT'); needs the 'video' and
    'vggish' modalities like the reference's fusion modules (:940-941, :1022-1023)."""

    def __init__(self, task: str, modalities, tcn_settings, backbone_settings, output_dim, root_dir, device, model_name,
                 visual_state_dict=None, audio_state_dict=None):
        super().__init__()
        self._init_common(task, modalities, tcn_settings, backbone_settings, root_dir, device, with_up_sample=False)
        feas = [tcn_settings[m]['channel'][-1] for m in modalities]
        if model_name == "JMT":
            self.fuse = JMTFusion(num_feats_modality=feas, num_out_feats=128)
        elif model_name == "MT":
            self.fuse = MTFusion(num_feats_modality=feas, num_out_feats=128)
        else:
            raise NotImplementedError(model_name)
        self.model_name = model_name
        self.bn1 = nn.BatchNorm1d(128)
        self.fc1 = nn.Linear(128, 128)
        self.fc2 = nn.Linear(128, output_dim)
        self._load_backbones(modalities, visual_state_dict, audio_state_dict)

    def forward(self, X):
        if self._is_training_call():
            return self._training_forward(X)
        return self._fuse(self._encode(X))

    def _fuse(self, z):
        B, T, _ = z['video'].shape
        R = B * T
        # the final encoder attends over all L*B positions (see module docstring)
        out = self._fuse_rows(z['video'].view(R, -1), z['vggish'].view(R, -1), (B, T, T), (1, R, R))
        return self._tail(out, B, T)

    def _fuse_videos(self, z, lengths):
        """With batch 1 per video, the reference's "all L*B positions" are the video's own frames: every attention
        runs inside each video's segment of the concatenated rows."""
        seg = E.Segments(lengths, z['video'].device)
        return self._tail(self._fuse_rows(z['video'], z['vggish'], seg, seg), 1, seg.rows)[0]

    def _fuse_rows(self, vis, vggish, seq, final):
        """JMTFusion / MTFusion on rows [R, C]: ``seq`` lays out the sequences of the modality encoders and the
        cross-attention, ``final`` those of the final encoder and self-attention (each as _mha's layout)."""
        f = self.fuse
        aud = E.linear(vggish, f.augment_audio_feats_dim.weight, f.augment_audio_feats_dim.bias)
        ea = _encoder(f.audio_encoder, aud, seq)
        if self.model_name == "JMT":
            jr = E.linear(torch.cat((vis, aud), dim=1), f.reduce_feats_dim.weight, f.reduce_feats_dim.bias)
            ej = _encoder(f.jr_encoder, jr, seq)
            last = _mha(f.CA_ajr, ea, ej, seq)                # the only stack slot the output reads
        else:
            ev = _encoder(f.visual_encoder, vis, seq)
            last = _mha(f.CA_av, ea, ev, seq)
        enc = _encoder(f.final_encoder, last, final)
        return _mha(f.final_self_attention, enc, enc, final)
