"""Throughput of the `bert` stream (text.BertTextEncoder on csrc/bert.cu), with the card's name, power limit and max SM
clock in the record.

    python tools/text_bench.py --out profiles/r08_text.json

Workloads (synthetic seeded transcripts, ids as synthetic.transcript_ids; weights synthetic.bert_state_dict(0), which
has bert-base-uncased's sizes):
  * "56": 56 transcripts with lengths U{16..512} (numpy seed 7), the batch of tests/test_gpu_text.py;
  * "1000": 1000 transcripts with lengths U{16..512} (numpy seed 8).
1. encode(): tokens/s from CUDA events around `reps` calls after `warmup` calls, ending in a device synchronise, and
   TFLOP/s from the counted work: 2 * 84.9 M FLOP per token for the encoder's weights (one multiply-add each) plus
   4 * n * 768 FLOP per token per layer for attention over a transcript of n tokens.  Weights (340 MB) and
   activations of the 56-transcript batch fit the 126 MB L2 only in part; nothing is flushed between calls.
2. Library bar: the same transcripts through HF transformers.BertModel on the same GPU (padded batches of 56 with an
   attention mask, the padding not counted as tokens), eager fp32 and bf16 autocast, if transformers imports;
   otherwise "not measured".
3. Share of the full path: frame_rows() of the 56 transcripts onto 56 videos with T_v ~ U[150, 3000] (the lengths of
   bench.py's full workload), against windowing.infer_videos of an LFAN(video, logmel, bert) on those videos (8 per
   call, stored uint8 crops + log-mel examples + the bert rows), measured in the same process.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from feature_vs_text_compound_emotion_b200 import synthetic, text, windowing  # noqa: E402

WEIGHT_FLOP_PER_TOKEN = 2 * 84.9e6
TF32_DENSE_TFLOPS = 1125.0          # HGX B200 data sheet, one GPU, dense, at up to 1000 W
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}


def card():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in q.split(",")]
        info.update({"card": name, "power_limit": power, "max_sm_clock": clk})
    except Exception as e:
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def lengths(n, seed):
    return [int(x) for x in np.random.default_rng(seed).integers(16, 513, n)]


def flop(lens, layers=12, hidden=768):
    return sum(n * WEIGHT_FLOP_PER_TOKEN + layers * 4.0 * n * n * hidden for n in lens)


def timed_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def hf_bar(sd, ids, dev, reps):
    try:
        import transformers
        from transformers import BertConfig, BertModel
    except Exception as e:                                   # noqa: BLE001
        return {"status": f"not measured: transformers does not import ({type(e).__name__})"}
    m = BertModel(BertConfig()).eval()
    m.load_state_dict(sd, strict=True)
    m = m.to(dev)
    batches = []
    for a in range(0, len(ids), 56):
        grp = ids[a:a + 56]
        L = max(t.numel() for t in grp)
        x = torch.zeros(len(grp), L, dtype=torch.int64)
        mask = torch.zeros(len(grp), L, dtype=torch.int64)
        for i, t in enumerate(grp):
            x[i, :t.numel()] = t
            mask[i, :t.numel()] = 1
        batches.append((x.to(dev), mask.to(dev)))

    def run():
        for x, mask in batches:
            hs = m(input_ids=x, attention_mask=mask, output_hidden_states=True).hidden_states
            sum(hs[-4:])

    out = {"transformers": transformers.__version__, "padding": "batches of 56 padded to their longest transcript"}
    tokens = sum(t.numel() for t in ids)
    with torch.no_grad():
        ms = timed_ms(run, reps, 1)
        out["fp32_eager"] = {"ms": ms, "tokens_per_s": tokens / (ms / 1e3)}
        with torch.autocast("cuda", dtype=torch.bfloat16):
            ms = timed_ms(run, reps, 1)
        out["bf16_autocast"] = {"ms": ms, "tokens_per_s": tokens / (ms / 1e3)}
    del m
    torch.cuda.empty_cache()
    return out


def full_path_share(enc, ids56, dev, reps):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    mods = ["video", "logmel", "bert"]
    m = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=mods, kernel_size=5, example_length=300,
             tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(0), audio_state_dict=synthetic.vggish_state_dict(0))
    m.load_state_dict(synthetic.lfan_state_dict(0, mods), strict=True)
    m = m.to(dev).eval()
    g = torch.Generator().manual_seed(7)
    vlens = torch.randint(150, 3001, (56,), generator=g).tolist()          # bench.video_lengths(56)
    tmax = max(vlens)
    raw = synthetic.raw_frames_u8(64, seed=11).repeat((tmax + 63) // 64, 1, 1, 1)[:tmax].contiguous().to(dev)
    lm = synthetic.logmel_patches(tmax, seed=12).to(dev)
    rows = enc.frame_rows(ids56, vlens)

    def text_branch():
        enc.frame_rows(ids56, vlens)

    def rest():
        for a in range(0, 56, 8):
            windowing.infer_videos(m, [raw[:t] for t in vlens[a:a + 8]],
                                   [{"logmel": lm[:t], "bert": rows[a + j]} for j, t in enumerate(vlens[a:a + 8])])

    t_text = timed_ms(text_branch, reps, 1)
    t_rest = timed_ms(rest, reps, 1)
    return {"videos": 56, "frames": sum(vlens), "video_lengths_seed": 7, "text_ms": t_text, "infer_videos_ms": t_rest,
            "text_share": t_text / (t_text + t_rest),
            "note": "text_ms: frame_rows (encode + frame expansion) of the 56 transcripts; infer_videos_ms: the rest of "
                    "the full call (eval transform, IR-50, VGGish, TCN, fusion, stitching) with the rows as input"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r08_text.json")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    torch.set_grad_enabled(False)
    dev = torch.device("cuda:0")
    rec = {"card": card(), "weight_flop_per_token": WEIGHT_FLOP_PER_TOKEN, "tf32_dense_peak_tflops": TF32_DENSE_TFLOPS,
           "workloads": {}}
    sd = synthetic.bert_state_dict(0)
    enc = text.BertTextEncoder()
    enc.load_state_dict(sd, strict=True)
    enc = enc.to(dev).eval()
    ids = {}
    for name, n, seed in (("56", 56, 7), ("1000", 1000, 8)):
        lens = lengths(n, seed)
        ids[name] = synthetic.transcript_ids(lens, seed=seed)
        host = enc._host_ids(ids[name])
        ms = timed_ms(lambda: enc._encode(host), args.reps, args.warmup)
        tokens, f = sum(lens), flop(lens)
        w = {"transcripts": n, "lengths": f"U{{16..512}}, numpy seed {seed}", "tokens": tokens, "ms_per_call": ms,
             "tokens_per_s": tokens / (ms / 1e3), "flop": f, "tflops": f / (ms / 1e3) / 1e12,
             "share_of_tf32_dense_peak": f / (ms / 1e3) / 1e12 / TF32_DENSE_TFLOPS,
             "timing": f"CUDA events around {args.reps} encode calls after {args.warmup} warm-up calls, ids already on the host"}
        w["library_bar"] = hf_bar(sd, ids[name], dev, max(2, args.reps // 5))
        rec["workloads"][name] = w
        print(name, json.dumps({k: v for k, v in w.items() if k != "library_bar"}), flush=True)
        print(" library", json.dumps(w["library_bar"]), flush=True)
    rec["full_path_share"] = full_path_share(enc, ids["56"], dev, max(2, args.reps // 5))
    print("share", json.dumps(rec["full_path_share"]), flush=True)
    rec["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(rec, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
