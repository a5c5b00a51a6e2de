"""The `bert` stream on the device (csrc/bert.cu): the tcgen05 TF32 linear kernel against fp64 at the encoder's shapes,
head-batched attention against single-head launches bit for bit, the embedding and frame kernels against torch bit for
bit, the whole encoder against the fp64 oracle and HF's golden output, row invariance across calls, LFAN end to end on
frame_rows, and repacking after an in-place weight update."""
import os
import warnings

import numpy as np
import pytest
import torch

from feature_vs_text_compound_emotion_b200 import engine, synthetic, text, windowing
from oracle import bert_oracle as O
from tests.test_gpu_streaming import _dev, _lfan

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
warnings.filterwarnings("ignore")

BATCH_LENGTHS = [int(n) for n in np.random.default_rng(7).integers(16, 513, 56)]      # U{16..512}, seed 7


@pytest.fixture(scope="module")
def golden(golden_dir):
    return torch.load(os.path.join(golden_dir, "bert_text.pt"))


_ENC = {}


def _encoder(std):
    if std not in _ENC:
        sd = synthetic.bert_state_dict(0, std=std)
        enc = text.BertTextEncoder()
        enc.load_state_dict(sd, strict=True)
        _ENC[std] = (enc.to(_dev()).eval(), sd)
    return _ENC[std]


@pytest.mark.parametrize("K, N, epi", [(768, 2304, "bias"), (768, 768, "residual"), (768, 3072, "gelu"),
                                       (3072, 768, "residual"), (3072, 768, "bias")])
@pytest.mark.parametrize("M", [1, 127, 129, 5000])
def test_linear_epilogues_against_fp64(K, N, epi, M):
    """|err| <= 2.5e-3 * (|x| @ |w|^T) + 1e-5: TF32 keeps 10 mantissa bits of each operand (2^-9 relative per product)
    with margin for the fp32 accumulation; erf-GELU's slope is below 1.13."""
    dev = _dev()
    g = torch.Generator().manual_seed(M * 7 + N)
    x = torch.randn(M, K, generator=g).to(dev)
    w = (0.02 * torch.randn(N, K, generator=g)).to(dev)
    b = (0.02 * torch.randn(N, generator=g)).to(dev)
    res = torch.randn(M, N, generator=g).to(dev) if epi == "residual" else None
    y = engine.bert_linear(x, w, b, epi, res)
    ref = x.double() @ w.double().T + b.double()
    if epi == "gelu":
        ref = torch.nn.functional.gelu(ref)
    elif epi == "residual":
        ref = ref + res.double()
    bound = 2.5e-3 * (x.double().abs() @ w.double().abs().T) * (1.13 if epi == "gelu" else 1.0) + 1e-5
    err = (y.double() - ref).abs()
    assert bool((err <= bound).all()), float((err / bound).max())


def test_head_batched_attention_equals_single_head_launches():
    dev = _dev()
    lengths = [1, 512, 37, 64, 65, 300, 2, 129, 1, 511]
    seg = engine.Segments(lengths, dev)
    g = torch.Generator().manual_seed(11)
    qkv = (2.0 * torch.randn(seg.rows, 3 * 768, generator=g)).to(dev)
    out = engine.sdpa_segments_heads(qkv, seg, 12)
    for h in range(12):
        c = 64 * h
        one = engine.sdpa_segments(qkv[:, c:c + 64], qkv[:, 768 + c:768 + c + 64], qkv[:, 1536 + c:1536 + c + 64], seg)
        assert torch.equal(out[:, c:c + 64], one), h


def _embed_torch(sd, ids, lengths, eps, dev):
    """The embedding kernel's fp32 operation sequence: lane-strided sums over 32 lanes, an xor butterfly, separate
    (unfused) products and sums."""
    P = {k: sd["embeddings." + k].to(dev) for k in ("word_embeddings.weight", "position_embeddings.weight",
                                                    "token_type_embeddings.weight", "LayerNorm.weight", "LayerNorm.bias")}
    pos = torch.cat([torch.arange(n) for n in lengths]).to(dev)
    x = (P["word_embeddings.weight"][ids] + P["token_type_embeddings.weight"][0]) + P["position_embeddings.weight"][pos]
    n, H = x.shape
    lanes = torch.arange(32, device=dev)

    def warp_sum(v):
        v = v.view(n, H // 32, 32)
        s = torch.zeros(n, 32, device=dev)
        for j in range(H // 32):
            s = s + v[:, j]
        for o in (16, 8, 4, 2, 1):
            s = s + s[:, lanes ^ o]
        return s[:, :1]

    Hs = torch.full((n, 1), float(H), device=dev)
    mean = warp_sum(x) / Hs
    d = x - mean
    rstd = torch.ones_like(mean) / torch.sqrt(warp_sum(d * d) / Hs + eps)
    return (d * rstd) * P["LayerNorm.weight"] + P["LayerNorm.bias"]


def test_embedding_kernel_equals_torch(golden):
    enc, sd = _encoder(0.02)
    dev = _dev()
    ids_list = golden["ids"] + synthetic.transcript_ids(BATCH_LENGTHS[:8], seed=7)
    lengths = [t.numel() for t in ids_list]
    seg = engine.Segments(lengths, dev)
    ids = torch.cat(ids_list).to(dev)
    have = enc.engine().embed(ids, seg)
    assert torch.equal(have, _embed_torch(sd, ids, lengths, 1e-12, dev))


def test_frame_kernel_equals_torch():
    dev = _dev()
    g = torch.Generator().manual_seed(3)
    rows = torch.randn(700, 768, generator=g).to(dev)
    tok = torch.randint(0, 700, (5000,), generator=g, dtype=torch.int32).to(dev)
    mean = torch.randn(768, generator=g).to(dev)
    std = (0.5 + torch.rand(768, generator=g)).to(dev)
    assert torch.equal(engine.text_frames(rows, tok), rows[tok.long()])
    assert torch.equal(engine.text_frames(rows, tok, mean, std), (rows[tok.long()] - mean) / std)


def _check_rows(have, want, what):
    """Per row: cosine >= 0.9999 and max-abs error <= 1e-2 x the row's max-abs."""
    have, want = have.double(), want.double()
    cos = torch.nn.functional.cosine_similarity(have, want, dim=1)
    rel = (have - want).abs().max(dim=1).values / want.abs().max(dim=1).values
    print(f"{what}: min cosine {float(cos.min()):.7f}, max-abs / row scale {float(rel.max()):.2e}")
    assert float(cos.min()) >= 0.9999 and float(rel.max()) <= 1e-2, (what, float(cos.min()), float(rel.max()))
    return float(cos.min()), float(rel.max())


@pytest.mark.parametrize("std", [0.02, 0.1])
def test_encoder_against_fp64_oracle(std, golden):
    enc, sd = _encoder(std)
    dev = _dev()
    batch = synthetic.transcript_ids(BATCH_LENGTHS, seed=7)
    for name, ids_list in (("golden transcripts", golden["ids"]), ("56 transcripts", batch)):
        have = enc.encode(ids_list)
        want = O.encode(sd, ids_list, device=dev)
        _check_rows(torch.cat(have), torch.cat(want), f"std {std}, {name}")
    if std == 0.02:                                              # HF BertModel's own fp32 output, on its column sample
        cols = golden["columns"].to(dev)
        _check_rows(torch.cat(enc.encode(golden["ids"]))[:, cols], torch.cat(golden["sums"]).to(dev), "against HF")
        i = golden["aligned_index"]
        Ts = sorted(golden["aligned"])
        rows = enc.frame_rows([golden["ids"][i]] * len(Ts), Ts)
        for T, r in zip(Ts, rows):
            _check_rows(r[:, cols], golden["aligned"][T].to(dev), f"frame rows T={T}")


def test_rows_do_not_depend_on_the_rest_of_the_call():
    enc, _ = _encoder(0.02)
    batch = synthetic.transcript_ids(BATCH_LENGTHS, seed=7)
    together = enc.encode(batch)
    for i in (0, 17, 55, int(np.argmax(BATCH_LENGTHS)), int(np.argmin(BATCH_LENGTHS))):
        assert torch.equal(enc.encode([batch[i]])[0], together[i]), i
    pair = enc.encode([batch[3], batch[40]])
    assert torch.equal(pair[0], together[3]) and torch.equal(pair[1], together[40])


def test_lfan_end_to_end_on_frame_rows():
    """windowing.infer_video of an LFAN(video, logmel, bert) fed raw audio, with `bert` rows from frame_rows against the
    same call with the oracle's rows: logits within the head tolerance, argmax agreement >= 99.5 %."""
    enc, sd = _encoder(0.02)
    dev = _dev()
    m = _lfan(["video", "logmel", "bert"], dev)
    Ts = [450, 233]
    ids = synthetic.transcript_ids([40, 300], seed=21)
    g = torch.Generator().manual_seed(22)
    mean = (0.1 * torch.randn(768, generator=g)).to(dev)
    std = (0.5 + torch.rand(768, generator=g)).to(dev)
    rows = enc.frame_rows(ids, Ts, mean, std)
    ref_tok = O.encode(sd, ids, device=dev)
    for j, T in enumerate(Ts):
        ref_rows = O.frame_rows(ref_tok[j], T, mean, std).float()
        _check_rows(rows[j], ref_rows, f"z-scored rows T={T}")
        video = synthetic.frames(T, seed=23 + j).to(dev)
        wave = synthetic.waveform(T / 30.0 + 1.0, seed=25 + j).to(dev)
        got = windowing.infer_video(m, video, {"wave": wave, "bert": rows[j]})
        want = windowing.infer_video(m, video, {"wave": wave, "bert": ref_rows})
        err = float((got - want).abs().max())
        agree = float((got.argmax(-1) == want.argmax(-1)).float().mean())
        print(f"LFAN T={T}: logits max-abs {err:.2e}, argmax agreement {agree:.4f}")
        assert err <= 2e-2 and agree >= 0.995, (err, agree)


def test_repacks_after_an_in_place_weight_update():
    sd = synthetic.bert_state_dict(1)
    enc = text.BertTextEncoder()
    enc.load_state_dict(sd, strict=True)
    enc = enc.to(_dev()).eval()
    ids = synthetic.transcript_ids([50, 9], seed=5)
    before = enc.encode(ids)
    with torch.no_grad():
        enc.encoder.layer[11].output.dense.weight.mul_(3.0)
        enc.embeddings.word_embeddings.weight.add_(0.01)
    after = enc.encode(ids)
    assert not torch.equal(torch.cat(before), torch.cat(after))
    sd2 = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
    _check_rows(torch.cat(after), torch.cat(O.encode(sd2, ids, device=_dev())), "after the update")
