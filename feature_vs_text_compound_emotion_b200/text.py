"""The `bert` feature stream from transcripts, on the device.

The reference makes bert.npy with HF ``BertModel.from_pretrained('bert-base-uncased')`` (speech.py:185-250): each
token's vector is the sum of the last four hidden states (speech.py:617-626), ``align_word_embedding_new``
(speech.py:690-740) copies token i's vector to every frame of the i-th contiguous block of the video's frames, and the
dataset z-scores each dimension (base/dataset.py:516-539).  ``BertTextEncoder`` does all of it on the B200:

    enc = text.BertTextEncoder(); enc.load_state_dict(torch.load("bert-base-uncased.pt"), strict=True); enc.cuda().eval()
    rows = enc.frame_rows(ids, [len(v) for v in videos], mean, std)    # one [T_v, 768] tensor per video

``ids`` are WordPiece ids exactly as the caller's tokenizer returned them, [CLS] and [SEP] included; tokenization is
string processing against the user's vocab.txt and stays on the host, outside this module.  All transcripts of a call
share every launch (csrc/bert.cu) and a token's row does not depend on the other transcripts of the call.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch
from torch import nn

from . import packing
from .engine import BertEngine, Segments, text_frames
from .modules import _PackedModule


def token_blocks(n_tokens: int, T: int) -> List[np.ndarray]:
    """The frames of token i: the i-th piece of ``numpy.array_split(numpy.arange(T), n_tokens)``.  The first
    ``T mod n`` blocks get one frame more; when T < n frame t takes token t and the later tokens get no frames.

    This is SURVEY.md's statement of ``align_word_embedding_new`` (speech.py:690-740, SURVEY §8d config 3:
    block-constant rows, speech.py:718-735).  It was not checked against the reference's source.  It is the one place
    the alignment rule lives: if the source differs, change this function."""
    if n_tokens <= 0 or T <= 0:
        raise ValueError(f"token_blocks: n_tokens and T must be positive, got {n_tokens}, {T}")
    # array_split's pieces, cut by slicing (array_split itself costs ~1 us per piece)
    q, r = divmod(T, n_tokens)
    ends = (np.arange(1, n_tokens + 1) * q + np.minimum(np.arange(1, n_tokens + 1), r)).tolist()
    frames = np.arange(T)
    return [frames[e - q - (i < r):e] for i, e in enumerate(ends)]


def frame_tokens(n_tokens: int, T: int) -> np.ndarray:
    """int64 [T]: the token each frame takes, from :func:`token_blocks`."""
    return np.repeat(np.arange(n_tokens), [len(b) for b in token_blocks(n_tokens, T)])


class _Container(nn.Module):
    """Parameter container (pins HF BertModel's state_dict names); its forward is never called."""

    def __init__(container, /, **children):             # positional-only: HF names one child "self"
        super().__init__()
        for name, m in children.items():
            container.add_module(name, m)


class BertTextEncoder(_PackedModule):
    """HF ``BertModel`` in eval mode, without the pooler's use, on the sm_100a kernels (csrc/bert.cu).

    Constructor arguments are the ``BertConfig`` fields this encoder uses, with bert-base-uncased's values as defaults.
    Parameters have exactly the keys and shapes of ``transformers.BertModel(BertConfig(...)).state_dict()``, ``pooler.*``
    included, so a bert-base-uncased state_dict loads with ``strict=True``.  Supported: head_dim 64, hidden and
    intermediate sizes multiples of 64, at most 512 positions, ``hidden_act="gelu"`` (exact erf-GELU); anything else
    raises ``ValueError`` here."""

    def __init__(self, vocab_size: int = 30522, hidden_size: int = 768, num_hidden_layers: int = 12,
                 num_attention_heads: int = 12, intermediate_size: int = 3072, hidden_act: str = "gelu",
                 max_position_embeddings: int = 512, type_vocab_size: int = 2, layer_norm_eps: float = 1e-12):
        super().__init__()
        if num_attention_heads <= 0 or hidden_size != 64 * num_attention_heads:
            raise ValueError(f"BertTextEncoder: head_dim must be 64 (hidden_size {hidden_size}, "
                             f"{num_attention_heads} heads)")
        if intermediate_size <= 0 or intermediate_size % 64:
            raise ValueError(f"BertTextEncoder: intermediate_size must be a positive multiple of 64, got {intermediate_size}")
        if not 0 < max_position_embeddings <= 512:
            raise ValueError(f"BertTextEncoder: at most 512 positions, got {max_position_embeddings}")
        if hidden_act != "gelu":
            raise ValueError(f"BertTextEncoder: only hidden_act='gelu' (exact erf-GELU) is supported, got {hidden_act!r}")
        if vocab_size <= 0 or type_vocab_size <= 0 or num_hidden_layers <= 0:
            raise ValueError("BertTextEncoder: vocab_size, type_vocab_size and num_hidden_layers must be positive")
        H, I = hidden_size, intermediate_size
        self.config = {"hidden": H, "intermediate": I, "n_heads": num_attention_heads, "vocab": vocab_size,
                       "max_pos": max_position_embeddings, "type_vocab": type_vocab_size, "ln_eps": float(layer_norm_eps)}
        self.embeddings = _Container(word_embeddings=nn.Embedding(vocab_size, H),
                                     position_embeddings=nn.Embedding(max_position_embeddings, H),
                                     token_type_embeddings=nn.Embedding(type_vocab_size, H),
                                     LayerNorm=nn.LayerNorm(H, eps=layer_norm_eps))
        layers = []
        for _ in range(num_hidden_layers):
            attn = _Container(self=_Container(query=nn.Linear(H, H), key=nn.Linear(H, H), value=nn.Linear(H, H)),
                              output=_Container(dense=nn.Linear(H, H), LayerNorm=nn.LayerNorm(H, eps=layer_norm_eps)))
            layers.append(_Container(attention=attn, intermediate=_Container(dense=nn.Linear(H, I)),
                                     output=_Container(dense=nn.Linear(I, H), LayerNorm=nn.LayerNorm(H, eps=layer_norm_eps))))
        self.encoder = _Container(layer=nn.ModuleList(layers))
        self.pooler = _Container(dense=nn.Linear(H, H))

    @property
    def hidden_size(self) -> int:
        return self.config["hidden"]

    def engine(self) -> BertEngine:
        eng = self._fresh_engine()
        if eng is None:
            sd = {k: v.detach().cpu() for k, v in self.state_dict().items()}
            eng = self._set_engine(BertEngine(packing.pack_bert(sd), self.config, self._device()))
        return eng

    def _host_ids(self, ids_list: Sequence) -> List[torch.Tensor]:
        """Every refusal about the ids, on the host, before any device work."""
        if len(ids_list) == 0:
            raise ValueError("BertTextEncoder: no transcripts")
        out = []
        for i, ids in enumerate(ids_list):
            t = torch.as_tensor(ids)
            if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
                raise ValueError(f"transcript {i}: expected a 1-D integer tensor of WordPiece ids, got {t.dtype} "
                                 f"{tuple(t.shape)}")
            t = t.to(device="cpu", dtype=torch.int64)
            if t.numel() == 0:
                raise ValueError(f"transcript {i}: empty id list ([CLS] and [SEP] are part of the ids)")
            if t.numel() > self.config["max_pos"]:
                raise ValueError(f"transcript {i}: {t.numel()} ids, more than max_position_embeddings "
                                 f"({self.config['max_pos']})")
            lo, hi = int(t.min()), int(t.max())
            if lo < 0 or hi >= self.config["vocab"]:
                raise ValueError(f"transcript {i}: id {lo if lo < 0 else hi} outside the vocabulary "
                                 f"[0, {self.config['vocab']})")
            out.append(t)
        return out

    def _encode(self, host: List[torch.Tensor]) -> torch.Tensor:
        self._check_inference()
        dev = self._device()
        if dev.type != "cuda":
            raise ValueError("BertTextEncoder runs on the GPU: move it with .cuda() first")
        seg = Segments([t.numel() for t in host], dev)
        ids = torch.cat(host).to(dev)
        return self.engine().forward(ids, seg)

    def encode(self, ids_list: Sequence) -> List[torch.Tensor]:
        """Per transcript the sum of the last four hidden states, [n_i, hidden] fp32 (views into one buffer)."""
        host = self._host_ids(ids_list)
        return list(self._encode(host).split([t.numel() for t in host]))

    forward = encode

    def frame_rows(self, ids_list: Sequence, frames_list: Sequence[int], mean: Optional[torch.Tensor] = None,
                   std: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """One [T_i, hidden] fp32 tensor per video: token j's summed hidden states on every frame of
        ``token_blocks(n_i, T_i)[j]``, z-scored per dimension as ``(x - mean) / std`` when ``mean`` / ``std`` (each
        [hidden]) are given.  The tensors are views into one buffer, ready as ``feats["bert"]`` of
        ``windowing.infer_video(s)`` or ``LFAN.forward``."""
        host = self._host_ids(ids_list)
        frames = [int(T) for T in frames_list]
        if len(frames) != len(host):
            raise ValueError(f"frame_rows: {len(host)} transcripts but {len(frames)} frame counts")
        if any(T <= 0 for T in frames):
            raise ValueError(f"frame_rows: every video needs T > 0 frames, got {frames}")
        H = self.hidden_size
        if (mean is None) != (std is None):
            raise ValueError("frame_rows: give both mean and std, or neither")
        if mean is not None and (tuple(mean.shape) != (H,) or tuple(std.shape) != (H,)):
            raise ValueError(f"frame_rows: mean and std must have shape ({H},), got {tuple(mean.shape)}, {tuple(std.shape)}")
        tok, base = [], 0
        for t, T in zip(host, frames):
            tok.append(frame_tokens(t.numel(), T) + base)
            base += t.numel()
        rows = self._encode(host)
        dev = rows.device
        tok_dev = torch.from_numpy(np.concatenate(tok).astype(np.int32)).to(dev)
        if mean is not None:
            mean = mean.to(device=dev, dtype=torch.float32).contiguous()
            std = std.to(device=dev, dtype=torch.float32).contiguous()
        return list(text_frames(rows, tok_dev, mean, std).split(frames))
