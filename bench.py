#!/usr/bin/env python
"""bench.py -- end-to-end frames/s of the LFAN inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's own modules on host cores

Workload (config.workload): BASELINE.json configs[1] shape -- 8 windows x 300 aligned 40x40 face
crops per GPU -- run through the WHOLE path the metric names (IR-50 -> TCN x3 -> cross-modal
attention -> classifier) with synthetic VGGish/BERT feature windows beside the frames.
One step = one forward over that batch (2400 frames per GPU).  Weak scaling: every rank runs its
own 8 windows; the only collective is ONE final all_gather of the per-frame logits of all K steps,
inside the timed region, after the last step.

Prints ONE JSON line (rank 0):
  value        frames/s over exactly K steps, inputs resident in HBM (CUDA events, max over ranks)
  long_run     the same loop repeated until >= 2 s of device time (the power-capped steady state)
  e2e          through the public nn.Module API with pinned-host inputs, H2D and D2H inside the timed region
  roofline     the dominant kernel (256->256 3x3 @10x10 conv, 50.7 % of the FLOPs) timed alone; its name
               is the variant the C-ABI reports it launched
  roofline_hbm the memory-/latency-bound kernels (stem, TCN stacks, fusion head, eval transform): GB/s of
               algorithmic bytes against the measured HBM peak
  ir50 / ir50_layers   the whole backbone and every layer class timed in place (cer_ir50_run_ops)
  head_only / train / full / sweep / alt_heads   compact records of BASELINE configs[0] / [3] / [2] / [4] and of the
               CAN / JMT / MT heads on the same box
  library_bar  the reference's own IR-50 through cuDNN (channels_last, cudnn.benchmark, bf16/fp16 autocast)
  cpu_baseline the reference's own LFAN.forward (oracle/_ref) on this box's host cores, bounded sample
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import tempfile
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

import torch  # noqa: E402

WINDOWS, LENGTH = 8, 300
MODS = ["video", "vggish", "bert"]
IR50_GFLOP_PER_FRAME = 6.0545            # SURVEY.md section 8d / BASELINE.md section 2
HEAD_MFLOP_PER_FRAME = 9.988
VGGISH_GFLOP_PER_EXAMPLE = 1.7278
DOM = dict(h=10, cin=256, cout=256, ksize=3)   # dominant conv class (SURVEY.md appendix A)
BS = {"visual_state_dict": "res50_ir_0.887", "audio_state_dict": "vggish"}
ROT = 4   # rotating input sets: 4 x 54.7 MB > L2, and each step streams > 1 GB of activations


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def build_model(dev, mods=MODS, seed=0):
    from feature_vs_text_compound_emotion_b200 import synthetic
    from feature_vs_text_compound_emotion_b200.models.model import LFAN
    m = LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=mods, kernel_size=5,
             example_length=LENGTH, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2, root_dir="", device=dev)
    m.init(visual_state_dict=synthetic.visual_backbone_state_dict(seed) if "video" in mods else None,
           audio_state_dict=synthetic.vggish_state_dict(seed) if "logmel" in mods else None)
    m.load_state_dict(synthetic.lfan_state_dict(seed, mods), strict=True)
    return m.to(dev).eval()


def host_batch(seed, windows=WINDOWS):
    from feature_vs_text_compound_emotion_b200 import synthetic
    f = synthetic.feature_windows(windows, LENGTH, seed=seed, modalities=["vggish", "bert"])
    return {"video": synthetic.frames(windows * LENGTH, seed=seed + 1).view(windows, LENGTH, 3, 40, 40),
            "vggish": f["vggish"], "bert": f["bert"]}


def batch_seed(i, rank):
    return 100 + 10 * i + 1000 * rank


def _events_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def time_dominant_conv(dev, frames, iters=20):
    """The 256->256 3x3 @10x10 conv (PReLU epilogue), alone, back to back: average launch time and the
    kernel variant the C-ABI says it launched."""
    from feature_vs_text_compound_emotion_b200 import _capi
    from feature_vs_text_compound_emotion_b200.engine import conv_forward
    g = torch.Generator().manual_seed(0)
    h, cin, cout = DOM["h"], DOM["cin"], DOM["cout"]
    x = torch.randn(frames + 8, h, h, cin, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(cout, 9 * cin, generator=g) * (9 * cin) ** -0.5).to(torch.bfloat16).to(dev)
    bias = torch.randn(9, cout, generator=g).to(dev)
    alpha = torch.full((cout,), 0.25).to(dev)
    ms = _events_ms(lambda i: conv_forward(x, w, bias, 3, 1, 1, alpha=alpha, n_frames=frames), iters, warm=3)
    variant = (_capi.lib().cer_conv_last_variant() or b"?").decode()
    flops = 2.0 * frames * h * h * cout * 9 * cin
    return ms, flops, variant


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's own modules (oracle/_ref, staged by oracle/build_ref.py) on host cores
# ----------------------------------------------------------------------------------------------
_REF_CACHE = {}


def reference_lfan(device="cpu"):
    """The UNMODIFIED reference LFAN(video, vggish, bert) with the synthetic weights this repo's model
    uses (models/model.py:375-526, models/backbone.py:69-130), or None when oracle/_ref is not staged."""
    key = str(device)
    if key in _REF_CACHE:
        return _REF_CACHE[key]
    from feature_vs_text_compound_emotion_b200 import synthetic
    from oracle import build_ref
    model = None
    if build_ref.available():
        ref = build_ref.load()
        tmp = tempfile.mkdtemp(prefix="cer_ref_")
        torch.save(synthetic.visual_backbone_state_dict(0), os.path.join(tmp, BS["visual_state_dict"] + ".pth"))
        model = ref.LFAN(backbone_settings=BS, output_dim=7, task="CLASSIFICATION", modality=list(MODS), kernel_size=5,
                         example_length=LENGTH, tcn_channel=synthetic.TCN_CHANNELS, modal_dim=32, num_heads=2,
                         root_dir=tmp, device=device)
        model.init()
        model.load_state_dict(synthetic.lfan_state_dict(0, MODS), strict=True)
        model = model.to(device).eval()
    _REF_CACHE[key] = model
    return model


def cpu_reference_step(windows, threads, seed=5):
    """One bounded step on host cores: `windows` x 300 frames from pixels through the reference's own
    LFAN.forward (kind "reference"), or through the oracle port when oracle/_ref is absent ("port")."""
    torch.set_num_threads(threads)
    X = host_batch(seed, windows)
    model = reference_lfan("cpu")
    with torch.no_grad():
        t0 = time.perf_counter()
        if model is not None:
            out = model({k: v.clone() for k, v in X.items()})
            kind = "reference"
        else:
            from feature_vs_text_compound_emotion_b200 import synthetic
            from oracle import lfan_oracle as O
            out = O.lfan_forward(synthetic.lfan_state_dict(0, MODS), X, MODS)
            kind = "port"
        dt = time.perf_counter() - t0
    assert out.shape == (windows, LENGTH, 7)
    return dt, kind


def cpu_baseline_record(budget_s, threads):
    t1, kind = cpu_reference_step(1, threads)                     # calibration = warm-up (one window)
    windows = int(max(1, min(WINDOWS, budget_s / max(t1, 1e-3))))
    dt, kind = cpu_reference_step(windows, threads, seed=7)
    what = "the reference's own LFAN.forward (oracle/_ref: unmodified models/*.py)" if kind == "reference" else "oracle port"
    return {"value": windows * LENGTH / dt, "unit": "frames/s", "cores": threads, "kind": kind,
            "sample": f"{windows} windows x {LENGTH} frames from pixels through {what}, fp32, torch CPU on all host threads"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on all host cores; each step is a
    bounded sample (as many of the 8 windows as the time budget allows)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    t1, kind = cpu_reference_step(1, threads)
    budget = 200.0 / max(1, args.steps + args.warmup)
    windows = int(max(1, min(WINDOWS, budget / max(t1, 1e-3))))
    for _ in range(args.warmup):
        cpu_reference_step(windows, threads)
    t0 = time.perf_counter()
    for i in range(args.steps):
        cpu_reference_step(windows, threads, seed=5 + i)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    fps = windows * LENGTH / dt
    what = "the reference's own LFAN.forward (oracle/_ref: unmodified models/*.py)" if kind == "reference" else "oracle port"
    sample = f"{windows} of the {WINDOWS} windows x {LENGTH} frames per step, from pixels, through {what}, fp32, torch CPU"
    print(json.dumps({
        "impl": "reference", "metric": "frames_per_s", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"LFAN inference (IR-50+TCN+fusion), {WINDOWS} windows x {LENGTH} frames of 40x40 crops per GPU",
                   "sample": sample},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def library_bar(dev, frames):
    """The reference's own IR-50 (oracle/_ref VisualBackbone) through eager PyTorch + cuDNN on this B200:
    channels_last, cudnn.benchmark, TF32 / bf16 / fp16 autocast (the reference's --amp True is fp16).
    A baseline for the record, not a product path."""
    from feature_vs_text_compound_emotion_b200 import synthetic
    model = reference_lfan("cpu")
    if model is None:
        return {"unavailable": "oracle/_ref not staged"}
    import copy
    ref_vb = copy.deepcopy(model.spatial["visual"]).to(dev).eval().to(memory_format=torch.channels_last)
    l2_norm = sys.modules["models.arcface_model"].l2_norm

    def vb(t):
        # Backbone.forward (models/arcface_model.py:147-151) module by module: the reference's Flatten is a
        # .view, which needs an NCHW-contiguous tensor, so the 5x5x512 map is made contiguous before output_layer
        bb = ref_vb.backbone
        h = bb.body(bb.input_layer(t))
        return l2_norm(bb.output_layer(h.contiguous()))

    x = synthetic.frames(frames, seed=9).to(dev).contiguous(memory_format=torch.channels_last)
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    res = {"frames": frames, "what": "reference VisualBackbone.forward (oracle/_ref), eager, channels_last, cudnn.benchmark"}
    try:
        torch.backends.cudnn.benchmark = True
        torch.backends.cudnn.allow_tf32 = True
        torch.backends.cuda.matmul.allow_tf32 = True
        with torch.no_grad():
            res["tf32_ms"] = _events_ms(lambda i: vb(x), 3, warm=2)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                res["bf16_autocast_ms"] = _events_ms(lambda i: vb(x), 3, warm=2)
            with torch.autocast("cuda", dtype=torch.float16):
                res["fp16_autocast_ms"] = _events_ms(lambda i: vb(x), 3, warm=2)
    except Exception as e:        # an out-of-memory or cuDNN failure must not lose the bench line
        res["error"] = f"{type(e).__name__}: {e}"[:200]
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        del ref_vb, x
        torch.cuda.empty_cache()
    best = min([v for k, v in res.items() if k.endswith("_ms")], default=None)
    if best:
        res["best_frames_per_s"] = frames / best * 1e3
    return res


# ----------------------------------------------------------------------------------------------
def dump_outputs(directory, arrays):
    """--dump-outputs: every array as <directory>/<name>.npy in float32, so that two builds can be compared
    output for output (the inputs and weights are seeded: the same arguments give the same inputs)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


def _timed(fn, steps, warmup, world, dist, dev, local, after=None):
    """warm-up, barrier, CUDA-event timing of `steps` calls (+ `after()` once, inside the timed region),
    max over ranks -> (total ms, clocks)."""
    for i in range(warmup):
        fn(i)
    if after is not None and warmup:
        after()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    if after is not None:
        after()
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return ms.item(), clocks


def video_lengths(n, seed=7):
    """SURVEY.md section 8d cfg 3/5: T_v ~ U{150..3000}, seeded."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(150, 3001, (n,), generator=g).tolist()


def measure_videos(dev, world, rank, local, dist, n_videos, steps, warmup, with_e2e=True, model=None):
    """configs[2] / configs[4]: whole videos from stored uint8 256x256 crops + per-frame log-mel examples +
    BERT features -> device eval transform -> IR-50 / VGGish -> TCN -> fusion -> window stitching ->
    video-level vote.  Videos are sharded over the ranks (longest first); the only collective is the final
    gather of per-frame logits."""
    from feature_vs_text_compound_emotion_b200 import sharding, synthetic, windowing
    mods = ["video", "logmel", "bert"]
    m = model if model is not None else build_model(dev, mods)
    lengths = video_lengths(n_videos)
    mine = sharding.shard_videos(lengths, world)[rank]
    tmax = max(lengths)
    # one synthetic video of the maximum length; every video is a prefix of it (synthetic data, real sizes)
    raw_host = synthetic.raw_frames_u8(64, seed=11 + rank).repeat((tmax + 63) // 64, 1, 1, 1)[:tmax].contiguous().pin_memory()
    lm_host = synthetic.logmel_patches(tmax, seed=12 + rank).pin_memory()
    bert_host = torch.randn(tmax, 768, generator=torch.Generator().manual_seed(13 + rank)).pin_memory()
    raw, lm, bert = raw_host.to(dev), lm_host.to(dev), bert_host.to(dev)
    votes = {}

    group = max(1, int(os.environ.get("CER_VIDEOS_PER_CALL", "8")))

    def run_shard(_):
        local_out = {}
        for a in range(0, len(mine), group):
            ids = mine[a:a + group]
            if group == 1:
                T = lengths[ids[0]]
                outs = [windowing.infer_video(m, raw[:T], {"logmel": lm[:T], "bert": bert[:T]})]
            else:                                          # frames of `group` videos share the backbone passes
                outs = windowing.infer_videos(m, [raw[:lengths[i]] for i in ids],
                                              [{"logmel": lm[:lengths[i]], "bert": bert[:lengths[i]]} for i in ids])
            for i, o in zip(ids, outs):
                local_out[i] = votes[i] = o
        return sharding.gather_predictions(local_out, lengths, 7, dev)

    total_ms, clocks = _timed(run_shard, steps, warmup, world, dist, dev, local)
    frames_total = sum(lengths)
    rec = {"value": frames_total * steps / (total_ms / 1e3), "ms_per_step": total_ms / steps, "clocks": clocks,
           "frames_total": frames_total, "n_videos": n_videos, "videos_per_call": group,
           "windows": sum(len(windowing.window_starts(t)) for t in lengths), "n_mine": sum(lengths[i] for i in mine)}
    if mine:
        rec["example_vote"] = windowing.video_level_prediction(votes[mine[0]])
    if with_e2e:
        # end to end: every video's crops / log-mel / BERT rows come from pinned host memory; the copy of
        # video i+1 overlaps the compute of video i (pipeline.HostPrefetcher), logits go back to the host
        from feature_vs_text_compound_emotion_b200.pipeline import HostPrefetcher
        out_host = torch.empty(max(1, rec["n_mine"]), 7).pin_memory()
        pf = HostPrefetcher(dev)
        offs, o = {}, 0
        for k in mine:
            offs[k] = o
            o += lengths[k]

        def e2e(_):
            local_out = {}

            def one(b):
                return windowing.infer_video(m, b["raw"], {"logmel": b["logmel"], "bert": b["bert"]})

            def sink(j, out):
                k = mine[j]
                local_out[k] = out
                out_host[offs[k]:offs[k] + lengths[k]].copy_(out, non_blocking=True)

            pf.run(({"raw": raw_host[:lengths[k]], "logmel": lm_host[:lengths[k]], "bert": bert_host[:lengths[k]]} for k in mine), one, sink)
            sharding.gather_predictions(local_out, lengths, 7, dev)

        n_e2e = max(1, steps // 2)
        e2e_ms, _ = _timed(e2e, n_e2e, 1, world, dist, dev, local)
        rec["e2e_value"] = frames_total * n_e2e / (e2e_ms / 1e3)
    del raw, lm, bert
    return rec


def run_videos(args, dev, world, rank, local, dist):
    n_videos = args.videos or (56 if args.workload == "full" else 1000)
    rec = measure_videos(dev, world, rank, local, dist, n_videos, args.steps, args.warmup)
    if rank == 0:
        burst, sustained, hbm, src = _peaks()
        flops = (IR50_GFLOP_PER_FRAME + VGGISH_GFLOP_PER_EXAMPLE + HEAD_MFLOP_PER_FRAME * 1e-3) * 1e9
        value = rec["value"]
        line = {
            "metric": "frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {n_videos} videos, T_v~U[150,3000] (seed 7), {rec['frames_total']} unique frames, "
                                   f"{rec['windows']} windows of 300/hop 200; stored uint8 256x256 crops -> device eval transform -> IR-50; "
                                   "log-mel 96x64 -> VGGish; BERT 768-d; TCN; fusion; stitch; video vote",
                       "sharding": "videos, longest first", "l2": "each video streams >100 MB of crops and >1 GB of activations",
                       "collective": "all_gather of per-frame logits" if world > 1 else "none",
                       "example_vote": rec.get("example_vote")},
            "clocks": rec["clocks"],
            "e2e": {"value": rec["e2e_value"], "unit": "frames/s",
                    "h2d_bytes_per_step": rec["n_mine"] * (256 * 256 * 3 + 96 * 64 * 4 + 768 * 4), "d2h_bytes_per_step": rec["n_mine"] * 28},
            "gpu_launches": None,
            "roofline": {"bound": "tensor", "achieved": value / world * flops / 1e12, "peak": sustained, "unit": "TFLOP/s",
                         "frac": value / world * flops / 1e12 / sustained, "traffic": None,
                         "kernel": "whole pipeline, algorithmic 7.792 GFLOP per unique frame (IR-50 6.0545 + VGGish 1.7278 + head 0.010)",
                         "peak_source": f"{src} sustained"},
        }
        print(json.dumps(line))


def measure_train(dev, world, rank, local, dist, B, steps, warmup, with_e2e=True):
    """configs[3]: fusion-head training step on feature windows (frozen backbones => pre-extracted
    512/128/768-d features), AdamW(lr 1e-4, wd 1e-4), gradients summed with ONE NCCL all-reduce of the flat
    20 MB bucket; weak scaling (B windows per rank)."""
    from feature_vs_text_compound_emotion_b200 import synthetic
    from feature_vs_text_compound_emotion_b200.training import HeadTrainer
    mods = ["cnn_res50", "vggish", "bert"]
    with torch.enable_grad():
        m = build_model(dev, mods).train()
        tr = HeadTrainer(m, B, LENGTH, optimizer={"name": "adamw", "lr": 1e-4, "weight_decay": 1e-4}, seed=rank)
        host = [synthetic.feature_windows(B, LENGTH, seed=200 + i + 100 * rank, modalities=mods) for i in range(2)]
        labs = [torch.randint(0, 7, (B, LENGTH, 1), generator=torch.Generator().manual_seed(300 + i + 100 * rank)) for i in range(2)]
        devb = [{k: v.to(dev) for k, v in h.items()} for h in host]
        devl = [l.to(dev) for l in labs]
        losses = []
        total_ms, clocks = _timed(lambda i: losses.append(tr.step(devb[i % 2], devl[i % 2])), steps, warmup, world, dist, dev, local)
        frames = B * LENGTH
        rec = {"value": world * frames * steps / (total_ms / 1e3), "ms_per_step": total_ms / steps, "clocks": clocks,
               "frames_per_step_per_gpu": frames, "loss_first_last": [float(losses[0]), float(losses[-1])],
               "precision": getattr(tr, "precision", "fp32")}
        if with_e2e:
            pinned = [{k: v.pin_memory() for k, v in h.items()} for h in host]
            pl = [l.pin_memory() for l in labs]
            loss_host = torch.empty(1).pin_memory()
            # features + labels of step i+1 are staged on a side stream while step i computes
            from feature_vs_text_compound_emotion_b200.pipeline import HostPrefetcher
            pf = HostPrefetcher(dev)

            def e2e_run(n):
                batches = ({**pinned[i % 2], "labels": pl[i % 2]} for i in range(n))
                pf.run(batches, lambda b: tr.step({k: v for k, v in b.items() if k != "labels"}, b["labels"]),
                       lambda i, loss: loss_host.copy_(loss, non_blocking=True))

            e2e_run(2)
            e2e_ms, _ = _timed(lambda i: e2e_run(steps) if i == 0 else None, 1, 0, world, dist, dev, local)
            rec["e2e_value"] = world * frames * steps / (e2e_ms / 1e3)
            rec["h2d"] = sum(v.numel() * v.element_size() for v in pinned[0].values()) + pl[0].numel() * 8
    return rec


def run_train(args, dev, world, rank, local, dist):
    rec = measure_train(dev, world, rank, local, dist, args.train_batch, args.steps, args.warmup)
    if rank == 0:
        burst, sustained, hbm, src = _peaks()
        B = args.train_batch
        tf = 3 * HEAD_MFLOP_PER_FRAME * 1e6 * B * LENGTH / (rec["ms_per_step"] * 1e-3) / 1e12
        line = {
            "metric": "frames_per_s", "value": rec["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": rec["precision"], "data": "synthetic",
            "config": {"workload": f"train: fusion-head step (fwd+CE+bwd+AdamW), {B} windows x {LENGTH} frames per GPU, "
                                   "features 512/128/768-d, dropout 0.1, BatchNorm1d batch stats",
                       "l2": "two rotating batches; 20 MB weights + ~120 MB of saved activations per step",
                       "collective": "one all_reduce(SUM) of the flat 5,002,503-float gradient bucket" if world > 1 else "none",
                       "loss_first_last": rec["loss_first_last"]},
            "clocks": rec["clocks"],
            "e2e": {"value": rec["e2e_value"], "unit": "frames/s", "h2d_bytes_per_step": rec["h2d"], "d2h_bytes_per_step": 4},
            "gpu_launches": None,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": burst, "unit": "TFLOP/s", "frac": tf / burst, "traffic": None,
                         "kernel": "whole training step, algorithmic 3 x 9.988 MFLOP per frame (launch/latency bound at this size)",
                         "peak_source": f"{src} burst bf16 (tf32 tensor peak is half of it)"},
        }
        print(json.dumps(line))


def measure_head_only(dev, reps=50):
    """configs[0]: the fusion model forward alone (TCN per modality + attention fusion + classifier) on
    pre-extracted features, batch 2 x 300 frames: latency per forward on the GPU."""
    from feature_vs_text_compound_emotion_b200 import synthetic
    mods = ["cnn_res50", "vggish", "bert"]
    m = build_model(dev, mods)
    X = [{k: v.to(dev) for k, v in synthetic.feature_windows(2, LENGTH, seed=1234 + i, modalities=mods).items()} for i in range(2)]
    ms = _events_ms(lambda i: m(dict(X[i % 2])), reps, warm=3)
    hbm = _peaks()[2]
    by = 20.01e6 + 600 * (5632 + 28)             # SURVEY 8d: fp32 weights + in/out rows
    return {"workload": "configs[0]: fusion head forward only, batch 2 x 300 feature windows (512/128/768-d)",
            "ms_per_forward": ms, "frames_per_s": 600 / ms * 1e3, "algorithmic_bytes": by,
            "hbm_frac": by / (ms * 1e-3) / 1e9 / hbm, "bound": "launch latency (9 kernels in one CUDA graph)"}


def measure_alt_heads(dev, reps=10):
    """SURVEY 8(f4): the alternative heads CAN / JMT / MT (models/model.py:529-684, :895-1167) alone, on
    pre-encoded features for 8 windows x 300 frames: TCN stacks + fusion (JMT / MT: single-head attention over
    T = 300 and over all 2400 positions, TF32 tensor-core flash attention) + the fc tail."""
    from feature_vs_text_compound_emotion_b200 import synthetic
    from feature_vs_text_compound_emotion_b200.models.model import CAN, JMT
    out = {}
    for name in ("CAN", "JMT", "MT"):
        mods = ["video", "vggish", "bert"] if name == "CAN" else ["video", "vggish"]
        if name == "CAN":
            m = CAN(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
                    root_dir="", device=dev, visual_state_dict=synthetic.visual_backbone_state_dict(0))
            m.load_state_dict(synthetic.can_state_dict(0, mods), strict=True)
        else:
            m = JMT(task="CLASSIFICATION", modalities=mods, tcn_settings=synthetic.TCN_SETTINGS, backbone_settings=BS, output_dim=7,
                    root_dir="", device=dev, model_name=name, visual_state_dict=synthetic.visual_backbone_state_dict(0))
            m.load_state_dict(synthetic.jmt_state_dict(0, mods, model_name=name), strict=True)
        m = m.to(dev).eval()
        dims = {"video": 512, "vggish": 128, "bert": 768}
        feats = {k: torch.randn(WINDOWS, LENGTH, dims[k], device=dev) for k in mods}
        ms = _events_ms(lambda i: m.forward_features(dict(feats)), reps, warm=2)
        out[name] = {"ms_per_forward": ms, "frames_per_s": WINDOWS * LENGTH / ms * 1e3}
        # one optimisation step of the same head (forward in training mode, CE, hand-written backward, AdamW)
        from feature_vs_text_compound_emotion_b200.heads_training import AltHeadTrainer
        with torch.enable_grad():
            tr = AltHeadTrainer(m.train(), WINDOWS, LENGTH, optimizer={"name": "adamw", "lr": 1e-4, "weight_decay": 1e-4})
            labels = torch.randint(0, 7, (WINDOWS, LENGTH, 1), device=dev)
            tms = _events_ms(lambda i: tr.step(feats, labels, sync_grads=False), 5, warm=2)   # rank 0 only: no collective
        out[name]["train_ms_per_step"] = tms
        out[name]["train_frames_per_s"] = WINDOWS * LENGTH / tms * 1e3
        del m, tr
    out["workload"] = ("alternative heads on pre-encoded features, 8 windows x 300 frames: head-only forward (TCN + fusion + fc tail) "
                       "and one training step (TF32 TCN GEMMs, fp32 fusion; AdamW)")
    return out


def hbm_rooflines(dev, model, devb, frames):
    """Memory-/latency-bound kernels of the path, each timed alone over rotating inputs: algorithmic bytes
    (DESIGN.md section 5) / time against the measured HBM copy bandwidth."""
    from feature_vs_text_compound_emotion_b200 import synthetic
    from feature_vs_text_compound_emotion_b200.engine import PreprocEngine
    hbm = _peaks()[2]
    out = []

    def add(name, ms, nbytes, note):
        out.append({"kernel": name, "ms": ms, "bytes": nbytes, "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": nbytes / (ms * 1e-3) / 1e9 / hbm, "note": note})

    eng = model.spatial["visual"].backbone.engine()
    vids = [b["video"].view(frames, 3, 40, 40) for b in devb]
    eng.forward(vids[0])
    ms = _events_ms(lambda i: eng.run_ops(vids[i % len(vids)], frames, 0, 0), 12)
    add("stem_kernel (conv3x3 3->64 + BN + PReLU, fp32 NCHW -> bf16 NHWC)", ms, frames * (3 * 1600 * 4 + 1600 * 64 * 2),
        "19.2 KB in + 204.8 KB out per frame; K = 27 on CUDA cores: FP32-FMA bound, not HBM bound")
    tcn, fus = model._head_engines()
    dims = {"video": 512, "vggish": 128, "bert": 768}
    wbytes = {"video": 4.424e6 / 2 * 4 / 1.0, "vggish": 0.276e6 / 2 * 4, "bert": 5.210e6 / 2 * 4}   # params = MFLOP/frame / 2
    for mname in model.modality:
        xs = [torch.randn(WINDOWS, LENGTH, dims[mname], device=dev) for _ in range(2)]
        ms = _events_ms(lambda i: tcn[mname].forward(xs[i % 2]), 20)
        nb = wbytes[mname] + frames * 4 * (dims[mname] + tcn[mname].c_out)
        add(f"TCN stack '{mname}' ({tcn[mname].launches} launches, tcgen05 kind::tf32)", ms, nb,
            "weights + first input + last output; launch/latency bound at 2400 rows")
    enc = [[torch.randn(frames, d, device=dev) for d in (128, 32, 128)] for _ in range(2)]
    ms = _events_ms(lambda i: fus.forward(enc[i % 2]), 20)
    add("fusion_head_kernel (3-token attention + LayerNorm + classifier)", ms, frames * 1180 + 150e3,
        "1180 B per frame + 150 KB of weights; latency bound")
    pre = PreprocEngine(256, 256, dev)
    n_pre = 1200
    raws = [synthetic.raw_frames_u8(64, seed=21 + i).repeat((n_pre + 63) // 64, 1, 1, 1)[:n_pre].contiguous().to(dev) for i in range(2)]
    ms = _events_ms(lambda i: pre.forward(raws[i % 2]), 6)
    add("preprocess_kernel (Pillow-exact resize 48 + crop 40 + normalise)", ms, n_pre * (219 * 219 * 3 + 19200),
        "reads the 219x219 footprint of each stored 256x256 crop; byte-gather bound")
    return out


def ir50_layer_table(eng, frames, reps=5):
    """Every conv op of the plan launched alone through the plan's own descriptors (cer_ir50_run_ops), grouped
    by layer class.  The three rotating activation buffers hold finite bf16 activations of the last forward
    (not necessarily this layer's own input): a timing run, not a numerics run."""
    burst = _peaks()[0]
    groups = {}
    for op, meta in enumerate(eng.conv_ops):
        ms = _events_ms(lambda i: eng.run_ops(None, frames, op + 1, op + 1), reps, warm=1)
        name = (f"fc {meta['cin']}->{meta['cout']}" if meta["h_in"] == 1 else
                f"{meta['cin']}->{meta['cout']} @{meta['h_in']}x{meta['h_in']}"
                + (f" s{meta['stride']}" if meta["stride"] > 1 else "") + (f" +1x1 proj {meta['proj_cin']}" if meta["proj_cin"] else ""))
        var = eng.op_variant(op, frames)
        g = groups.setdefault((name, var), {"class": name, "variant": var, "launches": 0, "ms": 0.0, "gflop": 0.0})
        g["launches"] += 1
        g["ms"] += ms
        g["gflop"] += meta["flop"] * frames / 1e9
    rows = []
    for g in groups.values():
        g["tflops"] = g["gflop"] / g["ms"]
        g["frac_of_burst"] = g["tflops"] / burst
        g["ms"] = round(g["ms"], 4)
        g["gflop"] = round(g["gflop"], 1)
        rows.append(g)
    return rows


def run_infer(args, dev, world, rank, local, dist):
    from feature_vs_text_compound_emotion_b200 import modules
    model = build_model(dev)
    frames = WINDOWS * LENGTH
    K = args.steps
    host = [host_batch(batch_seed(i, rank)) for i in range(ROT)]
    devb = [{k: v.to(dev) for k, v in h.items()} for h in host]
    # per-frame logits of the last K steps stay on the device; ONE all_gather at the end ships them
    outs = torch.zeros(K, frames, 7, device=dev)
    gathered = torch.zeros(world, K, frames, 7, device=dev) if world > 1 else None

    def step(i, batch=None):
        out = model(dict(devb[i % ROT] if batch is None else batch))
        outs[i % K].copy_(out.view(frames, 7))
        return out

    def final_gather():
        if world > 1:
            dist.all_gather_into_tensor(gathered.view(world * K, frames, 7), outs)

    total_ms, clocks = _timed(step, K, args.warmup, world, dist, dev, local, after=final_gather)
    ms_per_step = total_ms / K
    value = world * frames * K / (total_ms / 1e3)
    if args.dump_outputs and rank == 0:
        # the later measurements below reuse `outs`: the last timed step's logits are written now
        dump_outputs(args.dump_outputs, {"logits": outs[K - 1].view(WINDOWS, LENGTH, 7)})

    # ---- the gathered logits are what the other rank computed: rank 0 recomputes rank 1's last step
    gather_verified = None
    if world > 1 and rank == 0:
        i_last = K - 1
        other = {k: v.to(dev) for k, v in host_batch(batch_seed(i_last % ROT, 1)).items()}
        mine = model(other).view(frames, 7)
        gather_verified = bool(torch.equal(mine, gathered[1, i_last % K])) and bool(torch.equal(outs, gathered[0]))
        del other

    # ---- the same loop for >= 2 s of device time: the power-capped steady state
    n_long = max(K, int(math.ceil(args.min_seconds * 1e3 / max(ms_per_step, 1e-3))))
    long_ms, long_clocks = _timed(step, n_long, 0, world, dist, dev, local, after=final_gather)
    long_run = {"steps": n_long, "seconds": long_ms / 1e3, "ms_per_step": long_ms / n_long,
                "value": world * frames * n_long / (long_ms / 1e3), "clocks": long_clocks}

    # ---- IR-50 alone (device events), for the tensor-pipe fraction of the whole backbone
    vid = devb[0]["video"].view(frames, 3, 40, 40)
    vb = model.spatial["visual"]
    ir50_ms = _events_ms(lambda i: vb(devb[i % ROT]["video"].view(frames, 3, 40, 40)), 10, warm=1)

    # ---- end to end through the public API: pinned host -> device, forward, logits -> host
    pinned = [{k: v.pin_memory() for k, v in h.items()} for h in host]
    out_host = torch.empty(WINDOWS, LENGTH, 7).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in pinned[0].values())
    d2h = out_host.numel() * out_host.element_size()
    # the H2D copy of step i+1 runs on a side stream while step i computes (pipeline.HostPrefetcher);
    # every step's copies and its D2H read are inside the timed region
    from feature_vs_text_compound_emotion_b200.pipeline import HostPrefetcher
    pf = HostPrefetcher(dev)
    cnt = [0]

    def e2e_run(n):
        def fn(b):
            out = step(cnt[0], b)
            cnt[0] += 1
            return out
        pf.run((pinned[i % ROT] for i in range(n)), fn, lambda i, out: out_host.copy_(out, non_blocking=True))
        final_gather()

    n_e2e = max(K, n_long // 2)
    e2e_run(2)
    e2e_ms, _ = _timed(lambda i: e2e_run(n_e2e) if i == 0 else None, 1, 0, world, dist, dev, local)
    e2e_value = world * frames * n_e2e / (e2e_ms / 1e3)

    # ---- compact records of the other BASELINE configs (every rank takes part: train all-reduces at N > 1)
    sub = {}
    if not args.no_sub_records:
        torch.cuda.empty_cache()
        tr = measure_train(dev, world, rank, local, dist, 16, 5, 3, with_e2e=False)
        sub["train"] = {"workload": "configs[3]: fusion-head training step, 16 windows x 300 frames per GPU, AdamW, "
                                    + ("one NCCL all-reduce of the 20 MB gradient bucket per step" if world > 1 else "single GPU"),
                        "frames_per_s": tr["value"], "ms_per_step": tr["ms_per_step"], "steps": 5, "precision": tr["precision"],
                        "loss_first_last": tr["loss_first_last"]}
        torch.cuda.empty_cache()
        vm = build_model(dev, ["video", "logmel", "bert"])
        fv = measure_videos(dev, world, rank, local, dist, 8 * world, 2, 1, with_e2e=False, model=vm)
        sub["full"] = {"workload": f"configs[2]: {8 * world} whole videos (T_v~U[150,3000]) from stored uint8 crops + log-mel + BERT "
                                   "-> eval transform -> IR-50 / VGGish -> TCN -> fusion -> stitch -> vote",
                       "unique_frames_per_s": fv["value"], "ms_per_pass": fv["ms_per_step"], "unique_frames": fv["frames_total"],
                       "windows": fv["windows"], "example_vote": fv.get("example_vote")}
        sv = measure_videos(dev, world, rank, local, dist, 128, 1, 1, with_e2e=False, model=vm)
        del vm
        sub["sweep"] = {"workload": "configs[4] (reduced): 128 whole videos sharded over the ranks, longest first (STRONG scaling: the "
                                    "total is fixed; bench.py --workload sweep runs the 1000-video version)",
                        "unique_frames_per_s": sv["value"], "ms_per_pass": sv["ms_per_step"], "unique_frames": sv["frames_total"],
                        "windows": sv["windows"]}
        torch.cuda.empty_cache()

    if rank != 0:
        return

    burst, sustained, hbm, src = _peaks()
    fpp = modules.Backbone.frames_per_pass
    dom_frames = min(fpp, frames)
    dom_ms, dom_flops, dom_variant = time_dominant_conv(dev, dom_frames)
    achieved = dom_flops / (dom_ms * 1e-3) / 1e12
    eng = vb.backbone.engine()
    # the plan's own choice for that layer class (unit 10 conv1 = 256->256 @10x10): must be the variant timed above
    plan_variant = eng.op_variant(2 * 10, frames)
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "dominant_conv_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if str(tj.get("kernel", "")).startswith(dom_variant):  # only a capture of the SAME variant may be quoted
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), f"profiles/dominant_conv_traffic.json ({tj.get('capture', 'ncu --set full')})"
    tcn_engines, _ = model._head_engines()
    launches = (eng.launches(frames) + sum(t.launches for t in tcn_engines.values()) + 1) * K
    eng.forward(vid)
    layers = ir50_layer_table(eng, frames)
    line = {
        "metric": "frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": K,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"LFAN inference (IR-50+TCN+fusion), {WINDOWS} windows x {LENGTH} frames of 40x40 crops per GPU",
                   "frames_per_step_per_gpu": frames, "frames_per_pass": fpp, "backbone_dtype": "bf16 in, fp32 accumulate",
                   "head_dtype": "tf32 (tcgen05 kind::tf32 TCN), fp32 fusion head",
                   "l2": f"inputs rotate over {ROT} buffers (219 MB > L2); each step streams >1 GB of activations",
                   "collective": "ONE all_gather of the per-frame logits of all K steps, after the last step, inside the timed region"
                                 if world > 1 else "none"},
        "clocks": clocks,
        "long_run": long_run,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": n_e2e},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": f"{dom_variant} 256->256 3x3 @10x10 (PReLU epilogue), timed alone",
                     "plan_variant_for_this_layer": plan_variant,
                     "frames_per_launch": dom_frames, "ms_per_launch": dom_ms, "peak_source": f"{src} burst"},
        "ir50": {"ms": ir50_ms, "tflops": IR50_GFLOP_PER_FRAME * frames / ir50_ms,
                 "frac_of_burst_peak": IR50_GFLOP_PER_FRAME * frames / ir50_ms / burst,
                 "frac_of_sustained_peak": IR50_GFLOP_PER_FRAME * frames / ir50_ms / sustained,
                 "share_of_step": ir50_ms / ms_per_step},
        "ir50_layers": layers,
        "roofline_hbm": hbm_rooflines(dev, model, devb, frames),
    }
    if gather_verified is not None:
        line["gather_verified"] = gather_verified
    if not args.no_sub_records:
        # rank 0 alone gets here: nothing below may touch the process group
        for name, fn in (("head_only", measure_head_only), ("alt_heads", measure_alt_heads)):
            try:
                sub[name] = fn(dev)
            except Exception as e:                                  # a side record must not cost the headline line
                sub[name] = {"error": f"{type(e).__name__}: {e}"}
        line.update(sub)
    if world == 1 and not args.no_library_bar:
        line["library_bar"] = library_bar(dev, frames)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_record(20.0, os.cpu_count() or 1)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="infer", choices=["infer", "full", "sweep", "train"],
                    help="infer: BASELINE configs[1] shape through the whole path (default, the headline line); "
                         "full: configs[2] -- 56 variable-length videos from stored uint8 crops + log-mel + BERT; "
                         "sweep: configs[4] -- 1000 videos sharded over the ranks (strong scaling); "
                         "train: configs[3] -- fusion-head training step, B=16 windows per rank, NCCL grad all-reduce")
    ap.add_argument("--videos", type=int, default=0, help="override the number of videos of full/sweep")
    ap.add_argument("--train-batch", type=int, default=16)
    ap.add_argument("--frames-per-pass", type=int, default=int(os.environ.get("CER_FRAMES_PER_PASS", "0")))
    ap.add_argument("--min-seconds", type=float, default=2.0, help="length of the long_run measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--no-sub-records", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the per-frame logits of the last timed step (rank 0, "
                         f"{WINDOWS} x {LENGTH} x 7) as DIR/logits.npy (float32); --workload infer only")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "infer"):
        ap.error("--dump-outputs is implemented for --impl b200 --workload infer")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import datetime
        import torch.distributed as dist
        # no phase of this script keeps a rank away from a collective for more than a minute: a 5-minute watchdog turns
        # a mismatch into a prompt error instead of NCCL's default 10-minute hang
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    torch.set_grad_enabled(False)

    from feature_vs_text_compound_emotion_b200 import modules
    if args.frames_per_pass > 0:
        modules.Backbone.frames_per_pass = args.frames_per_pass
    try:
        if args.workload in ("full", "sweep"):
            run_videos(args, dev, world, rank, local, dist)
        elif args.workload == "train":
            run_train(args, dev, world, rank, local, dist)
        else:
            run_infer(args, dev, world, rank, local, dist)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
