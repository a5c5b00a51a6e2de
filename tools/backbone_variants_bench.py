"""Throughput of the IR-SE and IR-100 / IR-152 backbone plans (Ir50Engine), measured with CUDA events and
torch.profiler, with the card's name and power limit in every record.

    python tools/backbone_variants_bench.py --out profiles/backbone_variants.json

1. IR-50 against IR-SE-50 at 40 px, 2400 frames per call (the benchmarked pass size), alternated in one process,
   each timed over a window of >= --window seconds: frames/s.  Then, in a profiled run of its own, the SE kernels'
   time and achieved GB/s against their algorithmic bytes (the squeeze reads r; the scale reads r and the shortcut
   and writes the output: 4 x the unit output's bytes per unit).
2. IR-100, IR-SE-100, IR-152 and IR-SE-152 at 112 px (7 x 7 head), Backbone.deep_frames_per_pass frames per pass:
   frames/s and TFLOP/s of the conv work computed from the shapes (Ir50Engine.conv_ops; identity columns of the
   MaxPool(1, 2) shortcut are not counted).

Weights are synthetic and seeded; timing only (the numerics are tests/test_gpu_backbone_variants.py's).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from feature_vs_text_compound_emotion_b200 import packing, synthetic  # noqa: E402
from feature_vs_text_compound_emotion_b200.engine import Ir50Engine  # noqa: E402
from feature_vs_text_compound_emotion_b200.modules import Backbone  # noqa: E402

SE_KERNELS = ("se_squeeze_excite_kernel", "se_scale_shortcut_kernel")


def card():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in q.split(",")]
        info.update({"card": name, "power_limit": power, "max_sm_clock": clk})
    except Exception as e:                     # a record without the power limit says so
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def engine(layers, se, in_hw, fpp, dev):
    units = synthetic.ir_units(layers)
    sd = synthetic.visual_backbone_state_dict(0, units=units, spatial=7 if in_hw == 112 else in_hw // 8, se=se)
    pk = packing.pack_ir50(sd, "backbone.", in_hw=in_hw, strides=[s for _, _, s in units])
    return Ir50Engine(pk, dev, frames_per_pass=fpp)


def timed_window(eng, x, out, window_s):
    """frames/s of eng.forward(x) over >= window_s seconds (CUDA events around the whole window)."""
    for _ in range(2):
        eng.forward(x, out)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    eng.forward(x, out)
    e.record()
    e.synchronize()
    reps = max(1, int(window_s * 1000.0 / s.elapsed_time(e)) + 1)
    s.record()
    for _ in range(reps):
        eng.forward(x, out)
    e.record()
    e.synchronize()
    ms = s.elapsed_time(e)
    return {"reps": reps, "window_s": round(ms / 1000.0, 3), "ms_per_call": round(ms / reps, 4),
            "frames_per_s": round(x.shape[0] * reps * 1000.0 / ms, 1)}


def se_unit_bytes(eng, frames):
    """Algorithmic bytes of the SE tail per forward: 4 x the bf16 unit output per unit (+ gates, negligible)."""
    return sum(4 * frames * h * w * c * 2 + 2 * frames * c * 4 for h, w, c in eng.unit_shapes)


def profile_se(eng, x, out, calls):
    from torch.profiler import ProfilerActivity, profile
    eng.forward(x, out)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            eng.forward(x, out)
        torch.cuda.synchronize()
    per = {}
    total = 0.0
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        total += t
        for k in SE_KERNELS:
            if k in ev.key:
                per[k] = per.get(k, 0.0) + t
    se_ms = sum(per.values()) / 1000.0 / calls
    nbytes = se_unit_bytes(eng, x.shape[0])
    return {"se_kernel_ms_per_call": round(se_ms, 4),
            "per_kernel_ms_per_call": {k: round(v / 1000.0 / calls, 4) for k, v in per.items()},
            "all_kernels_ms_per_call": round(total / 1000.0 / calls, 4),
            "se_share_of_kernel_time": round(sum(per.values()) / total, 4) if total else None,
            "se_algorithmic_bytes_per_call": nbytes,
            "se_achieved_GB_per_s": round(nbytes / (se_ms * 1e6), 1) if se_ms else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--window", type=float, default=2.0, help="seconds per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternations of IR-50 / IR-SE-50")
    ap.add_argument("--deep-frames", type=int, default=2048, help="frames per call of the 112 px plans")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    rec = {"card": card(), "window_s_min": args.window}

    n = 2400
    x = synthetic.frames(n, seed=11).to(dev)
    out = torch.empty(n, 512, device=dev)
    engs = {"IR-50": engine(50, False, 40, Backbone.frames_per_pass, dev),
            "IR-SE-50": engine(50, True, 40, Backbone.frames_per_pass, dev)}
    runs = {k: [] for k in engs}
    for _ in range(args.rounds):
        for k, eng in engs.items():
            runs[k].append(timed_window(eng, x, out, args.window))
    pair = {}
    for k, eng in engs.items():
        fps = sorted(r["frames_per_s"] for r in runs[k])
        gflop = sum(op["flop"] for op in eng.conv_ops) * n / 1e9
        pair[k] = {"frames": n, "frames_per_pass": eng.frames_per_pass, "launches_per_call": eng.launches(n),
                   "frames_per_s_median": fps[len(fps) // 2], "runs": runs[k],
                   "conv_tflop_per_s_median": round(gflop / (n / fps[len(fps) // 2]) / 1000.0, 1)}
    pair["IR-SE-50"]["slowdown_vs_IR-50"] = round(pair["IR-50"]["frames_per_s_median"] / pair["IR-SE-50"]["frames_per_s_median"] - 1, 4)
    pair["IR-SE-50"]["profile"] = profile_se(engs["IR-SE-50"], x, out, calls=5)
    rec["40px_2400"] = pair
    del engs, x, out
    torch.cuda.empty_cache()

    nd = args.deep_frames
    x = synthetic.frames(nd, seed=12, size=112).to(dev)
    out = torch.empty(nd, 512, device=dev)
    deep = {}
    for layers in (100, 152):
        for se in (False, True):
            name = f"IR-{'SE-' if se else ''}{layers}"
            eng = engine(layers, se, 112, Backbone.deep_frames_per_pass, dev)
            r = timed_window(eng, x, out, args.window)
            gflop = sum(op["flop"] for op in eng.conv_ops) * nd / 1e9
            deep[name] = dict(r, frames=nd, frames_per_pass=eng.frames_per_pass, launches_per_call=eng.launches(nd),
                              conv_gflop_per_frame=round(gflop / nd, 2),
                              conv_tflop_per_s=round(gflop / r["ms_per_call"], 1))
            if se:
                deep[name]["profile"] = profile_se(eng, x, out, calls=2)
            del eng
            torch.cuda.empty_cache()
    rec["112px"] = deep
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
