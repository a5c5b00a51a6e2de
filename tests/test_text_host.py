"""The `bert` stream's host side, without a GPU: the fp64 oracle against HF BertModel's output pinned in
tests/golden/bert_text.pt, the frame alignment rule, the drop-in state_dict layout, the weight packing, the refusals
(all raised before any device work) and the new C-ABI symbols."""
import json
import os

import numpy as np
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import packing, synthetic, text
from oracle import bert_oracle as O

torch.set_grad_enabled(False)


@pytest.fixture(scope="module")
def golden(golden_dir):
    return torch.load(os.path.join(golden_dir, "bert_text.pt"))


@pytest.fixture(scope="module")
def sd():
    return synthetic.bert_state_dict(0)


def test_golden_ids_are_the_seeded_transcripts(golden):
    assert golden["lengths"] == [1, 2, 63, 64, 65, 512]
    for a, b in zip(golden["ids"], synthetic.transcript_ids(golden["lengths"], seed=golden["ids_seed"])):
        assert torch.equal(a, b)


def test_fp64_oracle_matches_hf_bert(golden, sd):
    """The oracle restates HF BertModel: within 1e-4 x row scale (max-abs) of its fp32 output, on the golden's
    column sample; the scale is the oracle's whole row."""
    ref = O.encode(sd, golden["ids"])
    cols = golden["columns"]
    assert cols.numel() == 64
    for want, have in zip(golden["sums"], ref):
        assert have.shape == (want.shape[0], 768)
        scale = have.abs().max(dim=1).values
        err = (want.double() - have[:, cols]).abs().max(dim=1).values
        assert bool((err <= 1e-4 * scale).all()), float((err / scale).max())


def test_golden_aligned_rows_follow_token_blocks(golden):
    """The golden's rows were written out with numpy.array_split blocks; token_blocks / frame_tokens give the same
    rows, and the oracle's expansion too."""
    sums = golden["sums"][golden["aligned_index"]]
    n = sums.shape[0]
    assert set(golden["aligned"]) == {100, 63, 20}
    for T, rows in golden["aligned"].items():
        assert rows.shape == (T, sums.shape[1])
        assert torch.equal(sums[torch.from_numpy(text.frame_tokens(n, T))], rows)
        assert torch.equal(O.frame_rows(sums, T), rows)


def test_token_blocks_is_numpy_array_split():
    """Every n, T in 1..600 against numpy's rule for array_split (T mod n pieces of T // n + 1 frames, then pieces of
    T // n, in order), and against numpy.array_split itself for every T at a set of n."""
    for n in range(1, 601):
        for T in range(1, 601):
            blocks = text.token_blocks(n, T)
            q, r = divmod(T, n)
            assert [len(b) for b in blocks] == [q + 1] * r + [q] * (n - r), (n, T)
            assert np.array_equal(np.concatenate(blocks), np.arange(T)), (n, T)
            if T < n:                                      # frame t takes token t, later tokens get no frames
                assert np.array_equal(text.frame_tokens(n, T), np.arange(T))
    for n in (1, 2, 3, 7, 63, 64, 65, 300, 511, 512, 599, 600):
        for T in range(1, 601):
            want = np.array_split(np.arange(T), n)
            have = text.token_blocks(n, T)
            assert len(have) == n and all(np.array_equal(a, b) for a, b in zip(have, want)), (n, T)
    with pytest.raises(ValueError):
        text.token_blocks(0, 5)
    with pytest.raises(ValueError):
        text.token_blocks(5, 0)


def test_state_dict_layout_is_hf_bert_model(golden_dir, sd):
    keys = json.load(open(os.path.join(golden_dir, "bert_state_keys.json")))
    with torch.device("meta"):
        enc = text.BertTextEncoder()
    assert {k: list(v.shape) for k, v in enc.state_dict().items()} == keys
    assert list(keys) == list(sd)
    assert len(keys) == 199 and "pooler.dense.weight" in keys
    enc = text.BertTextEncoder()
    enc.load_state_dict(sd, strict=True)
    assert torch.equal(enc.encoder.layer[3].attention.self.value.weight, sd["encoder.layer.3.attention.self.value.weight"])


def test_pack_bert_layout(sd):
    pk = packing.pack_bert(sd)
    assert len(pk["layers"]) == 12
    L = pk["layers"][5]
    p = "encoder.layer.5."
    assert L["wqkv"].shape == (2304, 768) and L["bqkv"].shape == (2304,)
    for i, n in enumerate(("query", "key", "value")):
        assert torch.equal(L["wqkv"][768 * i:768 * (i + 1)], sd[f"{p}attention.self.{n}.weight"])
        assert torch.equal(L["bqkv"][768 * i:768 * (i + 1)], sd[f"{p}attention.self.{n}.bias"])
    assert torch.equal(L["w1"], sd[p + "intermediate.dense.weight"]) and L["w1"].shape == (3072, 768)
    assert torch.equal(L["w2"], sd[p + "output.dense.weight"]) and L["w2"].shape == (768, 3072)
    assert torch.equal(pk["type_emb"], sd["embeddings.token_type_embeddings.weight"])


SMALL = dict(vocab_size=100, hidden_size=64, num_hidden_layers=1, num_attention_heads=1, intermediate_size=128,
             max_position_embeddings=16)


@pytest.mark.parametrize("bad, match", [
    (dict(num_attention_heads=2), "head_dim must be 64"),
    (dict(hidden_size=96, num_attention_heads=1), "head_dim must be 64"),
    (dict(intermediate_size=100), "multiple of 64"),
    (dict(max_position_embeddings=513), "at most 512"),
    (dict(hidden_act="gelu_new"), "hidden_act"),
    (dict(hidden_act="relu"), "hidden_act"),
])
def test_unsupported_configurations_are_refused(bad, match):
    with pytest.raises(ValueError, match=match):
        text.BertTextEncoder(**{**SMALL, **bad})


def test_refusals_come_before_any_device_work():
    """The module lives on the CPU here: each bad input must raise its own ValueError, not the "runs on the GPU" one
    that valid input reaches."""
    enc = text.BertTextEncoder(**SMALL).eval()
    ok = torch.tensor([1, 5, 2])
    with pytest.raises(ValueError, match="runs on the GPU"):
        enc.frame_rows([ok], [10])
    with pytest.raises(ValueError, match="runs on the GPU"):
        enc.encode([ok])
    cases = [
        (([torch.tensor([], dtype=torch.int64)], [10]), {}, "empty id list"),
        (([ok, torch.arange(17) % 100], [10, 10]), {}, "more than max_position_embeddings"),
        (([torch.tensor([1, 100])], [10]), {}, "outside the vocabulary"),
        (([torch.tensor([-1, 3])], [10]), {}, "outside the vocabulary"),
        (([torch.tensor([[1, 2]])], [10]), {}, "1-D integer"),
        (([torch.tensor([1.0, 2.0])], [10]), {}, "1-D integer"),
        (([], []), {}, "no transcripts"),
        (([ok], [0]), {}, "T > 0"),
        (([ok], [-3]), {}, "T > 0"),
        (([ok, ok], [5]), {}, "frame counts"),
        (([ok], [10]), {"mean": torch.zeros(63), "std": torch.ones(64)}, "shape"),
        (([ok], [10]), {"mean": torch.zeros(64), "std": torch.ones(64, 1)}, "shape"),
        (([ok], [10]), {"mean": torch.zeros(64)}, "both mean and std"),
    ]
    for args, kw, match in cases:
        with pytest.raises(ValueError, match=match):
            enc.frame_rows(*args, **kw)
    with pytest.raises(ValueError, match="empty id list"):
        enc.encode([ok, torch.tensor([], dtype=torch.int64)])


def test_workspace_covers_the_plan_buffers():
    """cer_bert_workspace_bytes is a host call: h, qkv (3H), ctx, t, a and inter (I) per token, fp32."""
    import ctypes as C
    from feature_vs_text_compound_emotion_b200 import _capi
    w = _capi.BertWeights()
    w.hidden, w.intermediate = 768, 3072
    for n in (1, 707, 16015):
        assert _capi.lib().cer_bert_workspace_bytes(C.byref(w), n) == n * (7 * 768 + 3072) * 4


def test_new_c_abi_symbols_are_exported():
    from feature_vs_text_compound_emotion_b200 import _capi
    lib = _capi.lib()
    for name in ("cer_bert_workspace_bytes", "cer_bert_create", "cer_bert_forward", "cer_bert_destroy", "cer_bert_embed",
                 "cer_bert_linear", "cer_text_frames", "cer_sdpa_tc_seg_heads_forward"):
        assert name in _capi.SIGNATURES and hasattr(lib, name), name
    assert lib.cer_version() == 109
