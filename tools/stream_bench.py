"""Step latency and throughput of streaming.StreamSession, with the card's name and power limit in the record.

    python tools/stream_bench.py --out profiles/r04_streaming.json

LFAN with 'video' (fp32 40 px crops through IR-50) + 'vggish' + 'bert', W = 300, H = 200, one session of 256
stream slots and chunks up to 30 frames.
1. For n in {1, 32, 256} streams and c in {1, 8, 30} frames per push: every push of a window of >= --window seconds
   timed with CUDA events (backbone pass + head graph + the host work of a push); median and p99 step latency,
   frames/s from the median and from the mean step time, and for every step slower than 3x the median the time
   its push call spent on the host and whether a garbage collection ran inside it.
2. A torch.profiler run of its own at each (n, c): CUDA kernel time split into backbone (IR-50 / VGGish /
   preprocessing kernels) and head (TCN, fusion, stream.cu kernels), so the cost of the recomputed TCN history is
   measured; the rows recomputed per output row, from the shapes, are recorded beside it.
3. windowing.infer_videos on the same frames (n = 32 videos of the frames one stream would see), measured in the
   same run.
Weights and inputs are synthetic and seeded; timing only (the numerics are tests/test_gpu_streaming.py's).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from feature_vs_text_compound_emotion_b200 import streaming, synthetic, windowing  # noqa: E402

HEAD_KERNELS = ("tcn_", "fusion_", "stream_")
GC_RUNS = [0]
gc.callbacks.append(lambda phase, info: GC_RUNS.__setitem__(0, GC_RUNS[0] + (phase == "start")))
MODS = ["video", "vggish", "bert"]


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


def lfan(dev):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings={"visual_state_dict": "", "audio_state_dict": ""}, output_dim=7, task="CLASSIFICATION",
             modality=MODS, kernel_size=5, example_length=300, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32,
             num_heads=2, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(0))
    m.load_state_dict(synthetic.lfan_state_dict(0, MODS), strict=True)
    return m.to(dev).eval()


def chunk_inputs(n, c, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return {"video": torch.rand(n, c, 3, 40, 40, device=dev, generator=g) * 2 - 1,
            "vggish": torch.randn(n, c, 128, device=dev, generator=g),
            "bert": torch.randn(n, c, 768, device=dev, generator=g)}


def recompute_rows(sess, c):
    """Rows the staged TCN launches compute per output row (per modality: mean over blocks of (R_b + c) / c)."""
    return {m: [round((r + c) / c, 2) for r in sess._rows[m]] for m in sess.modalities}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_streaming.json")
    ap.add_argument("--window", type=float, default=2.0)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    rec = {"card": card(), "modalities": MODS, "window_length": 300, "hop_length": 200, "configs": []}
    m = lfan(dev)
    sess = streaming.StreamSession(m, max_streams=256, max_chunk=30)
    rec["state_bytes_per_stream"] = sess.state_bytes()
    rec["n_slots"], rec["n_logit_slots"] = sess.n_slots, sess.n_lslots
    for n in (1, 32, 256):
        ids = [sess.open() for _ in range(n)]
        for c in (1, 8, 30):
            pool = [chunk_inputs(n, c, dev, 10 * n + c + k) for k in range(4)]
            for k in range(6):                                    # warm-up: every phase's first graph and plan setup
                sess.push(ids, pool[k % 4])
            torch.cuda.synchronize()
            times, host, gcs, t0, k = [], [], [], time.perf_counter(), 0
            while time.perf_counter() - t0 < args.window or len(times) < 20:
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0 = GC_RUNS[0]
                s.record()
                h0 = time.perf_counter()
                sess.push(ids, pool[k % 4])
                host.append((time.perf_counter() - h0) * 1e3)     # the push call alone: enqueue + host work
                e.record()
                e.synchronize()
                times.append(s.elapsed_time(e))
                gcs.append(GC_RUNS[0] - g0)
                k += 1
            ts = sorted(times)
            mean, med = sum(ts) / len(ts), ts[len(ts) // 2]
            slow = [j for j, t in enumerate(times) if t > 3 * med]
            cfg = {"streams": n, "chunk": c, "steps": len(ts), "median_ms": med,
                   "p99_ms": ts[min(len(ts) - 1, int(0.99 * len(ts)))],
                   "frames_per_s_median": n * c / (med / 1e3), "frames_per_s_mean": n * c / (mean / 1e3),
                   "median_host_ms": sorted(host)[len(host) // 2],
                   # steps slower than 3x the median: where their time went (host call vs device) and whether a
                   # garbage collection ran inside them
                   "slow_steps": [{"step": j, "ms": round(times[j], 3), "host_ms": round(host[j], 3), "gc_runs": gcs[j]}
                                  for j in slow],
                   "recompute_rows_per_output_row": recompute_rows(sess, c)}
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for j in range(10):
                    sess.push(ids, pool[j % 4])
                torch.cuda.synchronize()
            head = back = 0.0
            for ev in prof.key_averages():
                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if ev.device_type is None or "Memcpy" in ev.key or "Memset" in ev.key:
                    continue
                if any(ev.key.startswith("void cer::" + h) or ev.key.startswith(h) or ("cer::" + h) in ev.key
                       for h in HEAD_KERNELS):
                    head += t
                else:
                    back += t
            cfg["profiled_kernel_us_per_step"] = {"backbone": back / 10, "head": head / 10,
                                                  "head_share": head / max(head + back, 1e-9)}
            rec["configs"].append(cfg)
            print(json.dumps(cfg), flush=True)
        for i in ids:
            sess.close(i)
    # offline reference on the same kind of frames: 32 videos of 900 frames through infer_videos
    L, nv = 900, 32
    vids = [torch.rand(L, 3, 40, 40, device=dev, generator=torch.Generator(device=dev).manual_seed(i)) * 2 - 1
            for i in range(nv)]
    feats = [{"vggish": torch.randn(L, 128, device=dev), "bert": torch.randn(L, 768, device=dev)} for _ in range(nv)]
    windowing.infer_videos(m, vids, [dict(f) for f in feats])
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, t0 = 0, time.perf_counter()
    s.record()
    while time.perf_counter() - t0 < args.window or reps < 2:
        windowing.infer_videos(m, vids, [dict(f) for f in feats])
        reps += 1
    e.record()
    e.synchronize()
    rec["infer_videos"] = {"videos": nv, "frames_per_video": L, "reps": reps,
                           "frames_per_s": reps * nv * L / (s.elapsed_time(e) / 1e3)}
    print(json.dumps(rec["infer_videos"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
