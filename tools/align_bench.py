"""Throughput of five-point face alignment on the device (faces.align on csrc/align.cu) against cv2.warpAffine on all
host cores, with the card's name and power limit read in the same run.

    python tools/align_bench.py --out profiles/r09_align.json

Workloads: 720p and 1080p frames with 1 and 4 faces per frame, 256 x 256 crops, 256 faces per call, faces placed as
in the GPU tests (oracle/gen_align_golden.workload_faces).  Per workload:
  * ``align_ms``: faces.align per call (fit + index upload + warp), CUDA events over ``--reps`` calls;
  * ``warp_ms``: cer_face_warp alone on the same matrices;
  * ``gbps``: algorithmic bytes over warp_ms: the crops written (N * 256 * 256 * 3) plus the source bytes under each
    crop's footprint (256^2 * |det(inverse)| pixels * 3, not clipped at the frame's edge), computed from shapes;
  * ``cv2_faces_per_s``: cv2.warpAffine of the same faces on a thread pool of os.cpu_count() threads (cv2 releases the
    GIL; its own threading off), matrices fitted beforehand; "not measured" when cv2 is not installed.
Frames are seeded uint8 noise.  Every call reads the same faces: their source footprints (37 - 84 MB) fit the 126 MB
L2, so after the first call much of the source is read from L2, not HBM; the 50 MB of crops are written each call.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from feature_vs_text_compound_emotion_b200 import _capi, faces  # noqa: E402
from oracle import face_align_oracle as O  # noqa: E402
from oracle import gen_align_golden as G  # noqa: E402

S = 256
N_FACES = 256
WORKLOADS = [("720p_1face", 720, 1280, 1), ("720p_4faces", 720, 1280, 4),
             ("1080p_1face", 1080, 1920, 1), ("1080p_4faces", 1080, 1920, 4)]


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


def cv2_rate(host_frames, idx, fwd, n_threads):
    try:
        import cv2
    except ImportError:
        return "not measured (cv2 not installed)"
    cv2.setNumThreads(1)
    work = [(host_frames[f], M) for f, M in zip(idx, fwd)]
    with ThreadPoolExecutor(n_threads) as pool:
        list(pool.map(lambda a: cv2.warpAffine(a[0], a[1], (S, S)), work[:n_threads]))
        t = time.perf_counter()
        list(pool.map(lambda a: cv2.warpAffine(a[0], a[1], (S, S)), work))
        dt = time.perf_counter() - t
    return len(work) / dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default="profiles/r09_align.json")
    args = ap.parse_args()
    _capi.require_gpu()
    dev = torch.device("cuda:0")
    rec = {"card": card(), "crop": S, "faces_per_call": N_FACES, "host_threads": os.cpu_count(), "workloads": {}}
    for name, h, w, k in WORKLOADS:
        n_frames = N_FACES // k
        g = torch.Generator(device=dev).manual_seed(1)
        frames = torch.randint(0, 256, (n_frames, h, w, 3), generator=g, dtype=torch.uint8, device=dev)
        lm, idx = G.workload_faces([k] * n_frames, h, w, seed=2)
        lm_dev = torch.from_numpy(lm).to(dev)
        ref = faces.reference_points(S)
        fwd_dev, inv_dev = faces._fit(lm_dev, ref)
        idx_dev = torch.from_numpy(idx).to(dev)
        out = torch.empty(N_FACES, S, S, 3, dtype=torch.uint8, device=dev)
        lib, st = _capi.lib(), _capi.current_stream_ptr(dev)

        def warp():
            _capi.check(lib.cer_face_warp(frames.data_ptr(), n_frames, h, w, idx_dev.data_ptr(), inv_dev.data_ptr(),
                                          N_FACES, S, out.data_ptr(), st), "cer_face_warp")

        align_ms = timed_ms(lambda: faces.align(frames, lm_dev, idx), args.reps, args.warmup)
        warp_ms = timed_ms(warp, args.reps, args.warmup)
        inv = inv_dev.cpu().numpy()
        src_px = float(sum(S * S * abs(A[0, 0] * A[1, 1] - A[0, 1] * A[1, 0]) for A in inv))
        nbytes = N_FACES * S * S * 3 + src_px * 3
        fwd = fwd_dev.cpu().numpy()
        host = frames.cpu().numpy()
        rate = cv2_rate(host, idx, fwd, os.cpu_count())
        rec["workloads"][name] = {"frame": [h, w], "faces_per_frame": k, "align_ms": align_ms, "warp_ms": warp_ms,
                                  "align_faces_per_s": N_FACES / align_ms * 1e3, "warp_faces_per_s": N_FACES / warp_ms * 1e3,
                                  "algorithmic_bytes": nbytes, "gbps": nbytes / warp_ms / 1e6, "cv2_faces_per_s": rate}
        print(name, json.dumps(rec["workloads"][name]), flush=True)
        # the device crops are cv2's crops for the device matrices (spot check of 4 faces with the oracle)
        got = out.cpu().numpy()
        for i in range(0, N_FACES, N_FACES // 4):
            assert np.array_equal(got[i], O.warp(host[idx[i]], fwd[i], S)), (name, i)
        del frames, host
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(rec, open(args.out, "w"), indent=1)
    print(json.dumps(rec["card"]))


if __name__ == "__main__":
    main()
