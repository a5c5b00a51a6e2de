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

    python tools/stream_bench.py --audio wave --out profiles/r05_stream_audio.json

streams raw audio instead (DESIGN.md section 5.17): 'video' + 'logmel' computed from the waveform + 'bert', a session
with wave_fps = 30 and every push carrying the samples in step with its frames, so each push releases c frames once
warmed up.  The profiled run splits kernel time into IR-50 and preprocessing / VGGish / log-mel front end
(cer_stream_logmel, cer_stream_examples) / head; VGGish is timed with CUDA events around its calls in that run (its
convolutions are the IR-50 kernels, so kernel names cannot tell them apart) and IR-50 and preprocessing are the rest of
the backbone kernel time.  infer_videos is not run in this mode.

    python tools/stream_bench.py --head can --out profiles/r06_stream_can.json

streams a CAN instead (DESIGN.md section 5.18): 'video' + 'vggish' + 'bert' with synthetic.TCN_SETTINGS, final per-frame
logits, at (n, c) in {1x1, 1x30, 32x8, 32x30, 256x1, 256x8, 256x30}; head kernels are the TCN, stream.cu and
can_head_kernel.  The same run times can_head_kernel alone at 7 680 rows (CUDA events over repeated launches on one
set of inputs, so its 1.4 MB of weights are L2-resident as in a step) and reports GFLOP/s from the shape-derived
FLOP count.  infer_videos is not run in this mode.

    python tools/stream_bench.py --head jmt --out profiles/r07_stream_jmt.json

streams a JMT (or MT, --head mt) instead (DESIGN.md section 5.20): 'video' (fp32 40 px crops) + 'vggish' rows with
synthetic.TCN_SETTINGS, one session of 256 slots, chunks up to 30 and max_frames 6000.
1. The push step (backbones + continuous TCN + cer_stream_append) at 1x1, 32x8 and 256x30, timed as above.
2. peek over all open streams at 300, 1000 and 3000 frames per stream, for 1, 32 and 256 streams (host clock around
   the call, which ends in a device synchronise: its logits are read); the attention FLOPs of one peek (5 attentions
   per stream, 4 T^2 E each, E = 128) beside it.
3. close of one 3000-frame stream against windowing.infer_video on the same whole video started at end of stream,
   alternated, with the largest difference between their logits.
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

HEAD_KERNELS = ("tcn_", "fusion_", "stream_", "can_head")
FRONT_END_KERNELS = ("stream_logmel", "stream_tail", "stream_examples")
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


def lfan(dev, mods=MODS):
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings={"visual_state_dict": "", "audio_state_dict": ""}, output_dim=7, task="CLASSIFICATION",
             modality=mods, kernel_size=5, example_length=300, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32,
             num_heads=2, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(0),
           audio_state_dict=synthetic.vggish_state_dict(0) if "logmel" in mods else None)
    m.load_state_dict(synthetic.lfan_state_dict(0, mods), strict=True)
    return m.to(dev).eval()


def can(dev, mods=MODS):
    from feature_vs_text_compound_emotion_b200.models.model import CAN
    m = CAN(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS,
            backbone_settings={"visual_state_dict": "", "audio_state_dict": ""}, output_dim=7, root_dir="", device=dev,
            visual_state_dict=synthetic.visual_backbone_state_dict(0))
    m.load_state_dict(synthetic.can_state_dict(0, mods), strict=True)
    return m.to(dev).eval()


def jmt(dev, name):
    from feature_vs_text_compound_emotion_b200.models.model import JMT
    mods = ["video", "vggish"]
    m = JMT(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS,
            backbone_settings={"visual_state_dict": "", "audio_state_dict": ""}, output_dim=7, root_dir="", device=dev,
            model_name=name, visual_state_dict=synthetic.visual_backbone_state_dict(0))
    m.load_state_dict(synthetic.jmt_state_dict(0, mods, model_name=name), strict=True)
    return m.to(dev).eval()


def timed_call(fn, reps):
    """Median and all wall times (ms) of fn() over reps calls, each ending in a device synchronise."""
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2], ts


def whole_stream_bench(args, m, dev, rec):
    """--head jmt / mt: push step, peek and close against infer_video (see the module docstring)."""
    max_frames, E = 6000, 128
    sess = streaming.StreamSession(m, max_streams=256, max_chunk=30, max_frames=max_frames)
    rec.update({"max_frames": max_frames, "state_bytes_per_stream": sess.state_bytes(),
                "tcn_settings": {k: synthetic.TCN_SETTINGS[k] for k in m.modalities}, "configs": [], "peek": [],
                "close_vs_infer_video": {}})
    for n, c in ((1, 1), (32, 8), (256, 30)):
        ids = [sess.open() for _ in range(n)]
        pool = [chunk_inputs(n, c, dev, 10 * n + c + k, bert=False) for k in range(4)]
        for k in range(6):
            sess.push(ids, pool[k % 4])
        torch.cuda.synchronize()
        times, t0, k = [], time.perf_counter(), 0
        while ((time.perf_counter() - t0 < args.window or len(times) < 20)
               and sess.length(ids[0]) + c <= max_frames):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            sess.push(ids, pool[k % 4])
            e.record()
            e.synchronize()
            times.append(s.elapsed_time(e))
            k += 1
        ts = sorted(times)
        mean, med = sum(ts) / len(ts), ts[len(ts) // 2]
        cfg = {"streams": n, "chunk": c, "steps": len(ts), "median_ms": med,
               "p99_ms": ts[min(len(ts) - 1, int(0.99 * len(ts)))],
               "frames_per_s_median": n * c / (med / 1e3), "frames_per_s_mean": n * c / (mean / 1e3)}
        rec["configs"].append(cfg)
        print(json.dumps(cfg), flush=True)
        for i in ids:
            sess.close(i)
    for n in (1, 32, 256):
        ids = [sess.open() for _ in range(n)]
        pool = [chunk_inputs(n, 30, dev, 1000 + n + k, bert=False) for k in range(4)]
        k = 0
        for T in (300, 1000, 3000):
            while sess.length(ids[0]) < T:
                sess.push(ids, pool[k % 4])
                k += 1
            sess.peek(ids)                                        # warm-up at this shape
            med, ts = timed_call(lambda: sess.peek(ids), 5 if n * T < 100000 else 3)
            flop = 5 * 4 * n * T * T * E
            cfg = {"streams": n, "frames_per_stream": T, "median_ms": med, "times_ms": [round(t, 3) for t in ts],
                   "attention_gflop": flop / 1e9, "attention_tflop_per_s": flop / (med / 1e3) / 1e12}
            rec["peek"].append(cfg)
            print(json.dumps(cfg), flush=True)
        for i in ids:
            sess.close(i)
    T = 3000
    g = torch.Generator(device=dev).manual_seed(5)
    video = torch.rand(T, 3, 40, 40, device=dev, generator=g) * 2 - 1
    vgg = torch.randn(T, 128, device=dev, generator=g)
    windowing.infer_video(m, video, {"vggish": vgg})              # warm-up: plans for the 3000-frame passes
    close_ms, infer_ms, diff = [], [], 0.0
    for _ in range(4):
        sid = sess.open()
        for a in range(0, T, 30):
            sess.push([sid], {"video": video[None, a:a + 30], "vggish": vgg[None, a:a + 30]})
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = sess.close(sid)
        torch.cuda.synchronize()
        close_ms.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        want = windowing.infer_video(m, video, {"vggish": vgg})
        torch.cuda.synchronize()
        infer_ms.append((time.perf_counter() - t0) * 1e3)
        diff = max(diff, (got - want).abs().max().item())
    rec["close_vs_infer_video"] = {
        "frames": T, "reps": len(close_ms), "close_ms": [round(t, 3) for t in close_ms],
        "infer_video_ms": [round(t, 3) for t in infer_ms], "close_median_ms": sorted(close_ms)[len(close_ms) // 2],
        "infer_video_median_ms": sorted(infer_ms)[len(infer_ms) // 2], "max_abs_diff": diff,
        "note": "default IR-50 plan (CER_RASTER unset): the push passes and the 3000-frame pass may pick other kernels"}
    print(json.dumps(rec["close_vs_infer_video"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)


def can_head_flop(m) -> int:
    """FLOPs of one frame through cer_can_head_forward: the four GEMVs (softmax, activation and bias not counted)."""
    D = 128 * len(m.modalities)
    cs = sum(synthetic.TCN_SETTINGS[k]["channel"][-1] for k in m.modalities)
    return 2 * 128 * cs + 2 * 2 * D * D + 2 * D * m.fc2.weight.shape[0]


def time_can_head(m, dev, rows=7680, reps=200):
    head = m.frame_head()
    g = torch.Generator(device=dev).manual_seed(7)
    z = [torch.randn(rows, synthetic.TCN_SETTINGS[k]["channel"][-1], device=dev, generator=g) for k in m.modalities]
    out = torch.empty(rows, head.n_out, device=dev)
    for _ in range(10):
        head.forward(z, False, out=out)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        head.forward(z, False, out=out)
    e.record()
    e.synchronize()
    us = s.elapsed_time(e) * 1e3 / reps
    flop = can_head_flop(m) * rows
    return {"rows": rows, "reps": reps, "us_per_launch": us, "flop_per_frame": can_head_flop(m),
            "gflop_per_s": flop / (us * 1e-6) / 1e9}


def chunk_inputs(n, c, dev, seed, wave=False, bert=True):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = {"video": torch.rand(n, c, 3, 40, 40, device=dev, generator=g) * 2 - 1}
    if bert:
        x["bert"] = torch.randn(n, c, 768, device=dev, generator=g)
    if wave:      # one 30-frame second of samples per stream; each push slices what is in step with its frames
        x["_wave"] = torch.randn(n, 16000, device=dev, generator=g) * 0.3
    else:
        x["vggish"] = torch.randn(n, c, 128, device=dev, generator=g)
    return x


class Synced:
    """Per push, the samples of every stream that keep its audio in step with its video (all streams of a config
    are pushed together, so one count serves all)."""

    def __init__(self, sess, fps):
        self.sess, self.fps = sess, fps

    def __call__(self, ids, x):
        if "_wave" not in x:
            return x
        c = x["video"].shape[1]
        t = self.sess.length(ids[0])
        k = streaming.synced_samples(t + c, self.fps) - streaming.synced_samples(t, self.fps)
        return {"video": x["video"], "bert": x["bert"], "wave": [w[:k] for w in x["_wave"]]}


def recompute_rows(sess, c):
    """Rows the staged TCN launches compute per output row (per modality: mean over blocks of (R_b + c) / c)."""
    return {m: [round((r + c) / c, 2) for r in sess._rows[m]] for m in sess.modalities}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_streaming.json")
    ap.add_argument("--window", type=float, default=2.0)
    ap.add_argument("--audio", choices=("vggish", "wave"), default="vggish",
                    help="wave: stream raw audio (logmel from the waveform) instead of pre-extracted vggish features")
    ap.add_argument("--head", choices=("lfan", "can", "jmt", "mt"), default="lfan")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench measures the B200 kernels: no CUDA device")
    dev = torch.device("cuda:0")
    torch.set_grad_enabled(False)
    wave = args.audio == "wave"
    if args.head in ("jmt", "mt"):
        if wave:
            raise SystemExit("--head jmt / mt streams pre-extracted vggish features")
        m = jmt(dev, args.head.upper())
        whole_stream_bench(args, m, dev, {"card": card(), "head": args.head, "modalities": m.modalities})
        return
    is_can = args.head == "can"
    if wave and is_can:
        raise SystemExit("--head can streams pre-extracted vggish features")
    mods = ["video", "logmel", "bert"] if wave else MODS
    fps = 30.0
    rec = {"card": card(), "head": args.head, "modalities": mods, "configs": []}
    if is_can:
        rec["tcn_settings"] = {k: synthetic.TCN_SETTINGS[k] for k in mods}
    else:
        rec.update({"window_length": 300, "hop_length": 200})
    m = can(dev, mods) if is_can else lfan(dev, mods)
    sess = streaming.StreamSession(m, max_streams=256, max_chunk=30, wave_fps=fps if wave else None)
    rec["state_bytes_per_stream"] = sess.state_bytes()
    rec["n_slots"], rec["n_logit_slots"] = sess.n_slots, sess.n_lslots
    if wave:
        rec.update({"wave_fps": fps, "lag_frames": sess.lag, "logmel_ring_rows": sess.n_lm_rows,
                    "hold_rows": sess.n_hold})
    synced = Synced(sess, fps)
    vgg_ms = []
    if wave:                            # device time of every VGGish call, read after the profiled run
        aud = m.spatial["audio"]
        aud_fwd = aud.forward

        def timed(x, *a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            y = aud_fwd(x, *a, **k)
            e.record()
            vgg_ms.append((s, e))
            return y
    grid = {1: (1, 30), 32: (8, 30), 256: (1, 8, 30)} if is_can else {n: (1, 8, 30) for n in (1, 32, 256)}
    for n, chunks in grid.items():
        ids = [sess.open() for _ in range(n)]
        for c in chunks:
            pool = [chunk_inputs(n, c, dev, 10 * n + c + k, wave) for k in range(4)]
            for k in range(6 + (-(-sess.lag // c) if wave else 0)):   # warm-up: past the lag, every graph and plan
                sess.push(ids, synced(ids, pool[k % 4]))
            torch.cuda.synchronize()
            times, host, gcs, t0, k = [], [], [], time.perf_counter(), 0
            while time.perf_counter() - t0 < args.window or len(times) < 20:
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0 = GC_RUNS[0]
                s.record()
                h0 = time.perf_counter()
                sess.push(ids, synced(ids, pool[k % 4]))
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
            if wave:
                vgg_ms.clear()
                aud.forward = timed
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for j in range(10):
                    sess.push(ids, synced(ids, pool[j % 4]))
                torch.cuda.synchronize()
            if wave:
                del aud.forward
            head = back = front = 0.0
            for ev in prof.key_averages():
                t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if ev.device_type is None or "Memcpy" in ev.key or "Memset" in ev.key:
                    continue
                if any(("cer::" + h) in ev.key or ev.key.startswith(h) for h in FRONT_END_KERNELS):
                    front += t
                elif any(ev.key.startswith("void cer::" + h) or ev.key.startswith(h) or ("cer::" + h) in ev.key
                         for h in HEAD_KERNELS):
                    head += t
                else:
                    back += t
            cfg["profiled_kernel_us_per_step"] = {"backbone": back / 10, "head": head / 10,
                                                  "head_share": head / max(head + back + front, 1e-9)}
            if wave:
                vgg = sum(s.elapsed_time(e) for s, e in vgg_ms) * 1e3
                total = head + back + front
                cfg["profiled_kernel_us_per_step"].update({
                    "vggish_event_us": vgg / 10, "ir50_preproc": (back - vgg) / 10, "logmel_front_end": front / 10,
                    "shares": {"ir50_preproc": (back - vgg) / total, "vggish": vgg / total,
                               "logmel_front_end": front / total, "head": head / total}})
            rec["configs"].append(cfg)
            print(json.dumps(cfg), flush=True)
        for i in ids:
            sess.close(i)
    if is_can:
        rec["can_head_kernel"] = time_can_head(m, dev)
        print(json.dumps(rec["can_head_kernel"]), flush=True)
    if wave or is_can:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)
        return
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
