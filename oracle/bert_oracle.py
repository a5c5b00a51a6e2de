"""fp64 torch restatement of the `bert` stream's contract (HF BertModel in eval mode, one unpadded transcript at a
time), independent of the kernels and of transformers:

  * embeddings: LayerNorm(word[ids] + token_type[0] + position[0..n-1]);
  * per layer: q / k / v projections, softmax(q k^T / sqrt(64)) v per 64-wide head, output projection, residual +
    LayerNorm, 768 -> 3072 with exact erf-GELU, 3072 -> 768, residual + LayerNorm;
  * per token the sum of the last four hidden states (hidden_states[-4:], the embeddings counting as hidden state 0);
  * frame rows: token i's row on every frame of numpy.array_split(numpy.arange(T), n)[i], then (x - mean) / std.

Runs on whichever device the state_dict's tensors are moved to (``device``); the GPU tests use it on the GPU for speed.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch


def _ln(x, g, b, eps):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * g + b


def encode(sd: Dict[str, torch.Tensor], ids_list: Sequence[torch.Tensor], n_heads: int = 12, eps: float = 1e-12,
           device=None) -> List[torch.Tensor]:
    """Per transcript [n, H] fp64: the sum of the last four hidden states."""
    dev = torch.device(device) if device is not None else torch.device("cpu")
    P = {k: v.to(device=dev, dtype=torch.float64) for k, v in sd.items() if not k.startswith("pooler.")}
    n_layers = 0
    while f"encoder.layer.{n_layers}.attention.self.query.weight" in P:
        n_layers += 1
    lin = lambda x, p: x @ P[p + ".weight"].T + P[p + ".bias"]
    e = "embeddings."
    out = []
    for ids in ids_list:
        ids = torch.as_tensor(ids, dtype=torch.int64).to(dev)
        n = ids.numel()
        x = P[e + "word_embeddings.weight"][ids] + P[e + "token_type_embeddings.weight"][0] + P[e + "position_embeddings.weight"][:n]
        h = _ln(x, P[e + "LayerNorm.weight"], P[e + "LayerNorm.bias"], eps)
        hs = [h]
        for i in range(n_layers):
            p = f"encoder.layer.{i}."
            H = h.shape[1]
            d = H // n_heads
            q, k, v = (lin(h, p + "attention.self." + s).view(n, n_heads, d).transpose(0, 1) for s in ("query", "key", "value"))
            a = torch.softmax(q @ k.transpose(1, 2) / d ** 0.5, dim=-1) @ v
            ctx = a.transpose(0, 1).reshape(n, H)
            a1 = _ln(lin(ctx, p + "attention.output.dense") + h, P[p + "attention.output.LayerNorm.weight"],
                     P[p + "attention.output.LayerNorm.bias"], eps)
            inter = torch.nn.functional.gelu(lin(a1, p + "intermediate.dense"))
            h = _ln(lin(inter, p + "output.dense") + a1, P[p + "output.LayerNorm.weight"], P[p + "output.LayerNorm.bias"], eps)
            hs.append(h)
        out.append(sum(hs[-4:]))
    return out


def frame_rows(token_rows: torch.Tensor, T: int, mean: Optional[torch.Tensor] = None,
               std: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[n, H] token rows -> [T, H] frame rows by numpy.array_split blocks, optionally z-scored."""
    n = token_rows.shape[0]
    idx = np.concatenate([np.full(len(b), i) for i, b in enumerate(np.array_split(np.arange(T), n))])
    rows = token_rows[torch.from_numpy(idx).to(token_rows.device)]
    if mean is not None:
        rows = (rows - mean.to(rows)) / std.to(rows)
    return rows
