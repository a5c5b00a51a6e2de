"""Whole-video inference with the alternative heads CAN / JMT / MT (windowing.infer_videos), with the card's name and
power limit in the record.

    python tools/alt_heads_bench.py --out profiles/r06_alt_heads_videos.json

Workload: BASELINE config 3 for each head -- n videos (default 56) with T_v ~ U[150, 3000], the seeded lengths of
bench.video_lengths; stored uint8 256x256 crops (every video a prefix of one synthetic video, as bench.py does), plus
per-frame log-mel examples and BERT rows for CAN ('video', 'logmel', 'bert') and VGGish feature rows for JMT / MT
('video', 'vggish').
1. Throughput in unique frames/s, two arms measured in the same process and alternated round by round:
   - loop: the status quo before infer_videos took these heads -- one model.forward(X) per video in the reference
     layout (fp32 [1,T,3,40,40] pixels from the device eval transform, log-mel examples as [1,64,T,96]), the caller
     doing the transform and the layout;
   - infer_videos: 8 videos per call.
   Each arm is one pass over all n videos between CUDA events, ending in a device synchronise.
2. A torch.profiler run of its own (one infer_videos pass): CUDA kernel time split into backbone (eval transform,
   IR-50, VGGish), head (TCN, linear / LayerNorm / gate, attention, CAN head kernel) and the rest (PyTorch's copies,
   gathers and fills that lay the rows out).
3. JMT only: the segmented attention alone (cer_sdpa_tc_seg_forward, E = 128) on q / k / v slices of one packed
   projection of all n videos' frames, CUDA events over repeated launches; achieved TFLOP/s from 4 * sum(T_v^2) * E
   against the data-sheet dense TF32 rate and the minimal HBM traffic against 7.7 TB/s.
Weights and inputs are synthetic and seeded; timing only (the numerics are tests/test_gpu_alt_heads_videos.py's).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from feature_vs_text_compound_emotion_b200 import engine as E, synthetic, windowing  # noqa: E402

BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
HEAD_KERNELS = ("tcn_", "sdpa", "row_gemm", "add_layernorm", "softmax_gate", "can_head", "tanh_inplace")
TF32_DENSE_TFLOPS = 1125.0          # HGX B200 data sheet, one GPU, dense, at up to 1000 W
HBM_TBPS = 7.7
PER_CALL = 8


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


def video_lengths(n, seed=7):
    """bench.video_lengths: T_v ~ U{150..3000}, seeded."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(150, 3001, (n,), generator=g).tolist()


def build(name, dev):
    from feature_vs_text_compound_emotion_b200.models.model import CAN, JMT
    if name == "CAN":
        mods = ["video", "logmel", "bert"]
        m = CAN(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
                output_dim=7, root_dir="", device=dev, visual_state_dict=synthetic.visual_backbone_state_dict(0),
                audio_state_dict=synthetic.vggish_state_dict(0))
        m.load_state_dict(synthetic.can_state_dict(0, mods), strict=True)
    else:
        mods = ["video", "vggish"]
        m = JMT(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS,
                output_dim=7, root_dir="", device=dev, model_name=name, visual_state_dict=synthetic.visual_backbone_state_dict(0))
        m.load_state_dict(synthetic.jmt_state_dict(0, mods, model_name=name), strict=True)
    return m.to(dev).eval(), mods


def timed_ms(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def time_seg_attention(lengths, dev, reps):
    seg = E.Segments(lengths, dev)
    qkv = torch.randn(seg.rows, 3 * 128, generator=torch.Generator().manual_seed(1)).to(dev)
    q, k, v = qkv[:, :128], qkv[:, 128:256], qkv[:, 256:]
    for _ in range(3):
        E.sdpa_segments(q, k, v, seg)
    ms = timed_ms(lambda: [E.sdpa_segments(q, k, v, seg) for _ in range(reps)]) / reps
    flop = 4.0 * sum(t * t for t in lengths) * 128
    nbytes = 4.0 * seg.rows * 128 * 4                        # q, k, v read once and out written once: the least traffic
    t_compute, t_mem = flop / (TF32_DENSE_TFLOPS * 1e12), nbytes / (HBM_TBPS * 1e12)
    return {"n_seg": seg.n_seg, "rows": seg.rows, "max_len": seg.max_len, "launches_timed": reps, "ms_per_launch": ms,
            "flop": flop, "achieved_tflops": flop / (ms * 1e-3) / 1e12,
            "bound": "compute (TF32 dense)" if t_compute >= t_mem else "memory (HBM)",
            "share_of_bound": max(t_compute, t_mem) / (ms * 1e-3), "tf32_dense_peak_tflops": TF32_DENSE_TFLOPS,
            "min_bytes": nbytes, "note": "warp-level mma.sync TF32 (HMMA), not tcgen05: the data-sheet rate is out of its reach; "
                                         "inputs (~{:.0f} MB) are L2-resident across repeated launches".format(nbytes * 0.75 / 1e6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06_alt_heads_videos.json")
    ap.add_argument("--videos", type=int, default=56)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--heads", default="CAN,JMT,MT")
    ap.add_argument("--attn-reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("alt_heads_bench.py measures on the GPU: no CUDA device")
    torch.set_grad_enabled(False)
    dev = torch.device("cuda:0")
    lengths = video_lengths(args.videos)
    tmax, total = max(lengths), sum(lengths)
    raw = synthetic.raw_frames_u8(64, seed=11).repeat((tmax + 63) // 64, 1, 1, 1)[:tmax].contiguous().to(dev)
    lm = synthetic.logmel_patches(tmax, seed=12).to(dev)
    g = torch.Generator().manual_seed(13)
    rows = {"bert": torch.randn(tmax, 768, generator=g).to(dev), "vggish": torch.randn(tmax, 128, generator=g).to(dev)}
    rec = {"card": card(), "videos": args.videos, "lengths_seed": 7, "unique_frames": total, "videos_per_call": PER_CALL,
           "rounds": args.rounds, "heads": {}}
    print(json.dumps(rec["card"]), flush=True)

    for name in args.heads.split(","):
        m, mods = build(name, dev)
        feats = [{k: (lm if k == "logmel" else rows[k])[:t] for k in mods if k != "video"} for t in lengths]

        def loop():
            for t, f in zip(lengths, feats):
                X = {"video": windowing.preprocess_frames(m, raw[:t])[None]}
                for k, v in f.items():
                    X[k] = v.view(1, t, 96, 64).permute(0, 3, 1, 2).contiguous() if k == "logmel" else v[None]
                m(X)

        def batched():
            for a in range(0, len(lengths), PER_CALL):
                windowing.infer_videos(m, [raw[:t] for t in lengths[a:a + PER_CALL]], feats[a:a + PER_CALL])

        arms = {"loop": loop, "infer_videos": batched}
        for fn in arms.values():                                   # warm-up: plans, engines, allocator
            fn()
        times = {k: [] for k in arms}
        for r in range(args.rounds):
            order = list(arms) if r % 2 == 0 else list(arms)[::-1]
            for k in order:
                times[k].append(timed_ms(arms[k]))
        h = {"modalities": mods}
        for k, ts in times.items():
            best = min(ts)
            h[k] = {"ms_per_pass": ts, "unique_frames_per_s_best": total / (best / 1e3),
                    "unique_frames_per_s_mean": total / (sum(ts) / len(ts) / 1e3)}
        h["speedup_best"] = h["infer_videos"]["unique_frames_per_s_best"] / h["loop"]["unique_frames_per_s_best"]

        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batched()
            torch.cuda.synchronize()
        head = back = rest = 0.0
        for ev in prof.key_averages():
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            if ev.device_type is None or "Memcpy" in ev.key or "Memset" in ev.key:
                continue
            if "cer::" not in ev.key:
                rest += t
            elif any(("cer::" + p) in ev.key for p in HEAD_KERNELS):
                head += t
            else:
                back += t
        tot = max(head + back + rest, 1e-9)
        h["profiled_kernel_ms_per_pass"] = {"backbone": back / 1e3, "head": head / 1e3, "other": rest / 1e3,
                                            "head_share": head / tot, "backbone_share": back / tot, "other_share": rest / tot}
        if name == "JMT":
            rec["segmented_attention"] = time_seg_attention(lengths, dev, args.attn_reps)
            print(json.dumps(rec["segmented_attention"]), flush=True)
        rec["heads"][name] = h
        print(json.dumps({name: h}), flush=True)
        del m
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
