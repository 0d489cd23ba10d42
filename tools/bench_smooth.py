"""Cost of smoothing tracked joints: hpd_track against hpd_track_smooth per call, and frame-stream inference with
tracking against tracking plus smoothing.

  python tools/bench_smooth.py [--frames N] [--reps R] [--out profiles/r10_smooth.json]

hpd_track vs hpd_track_smooth (CUDA events, median of --reps calls each, after a warm-up; the two trackers'
calls alternate so that both see the same machine): calls of 8 and 64 frames of 30-person records (K = 17, E = 2,
every slot filled, bench_track.walking_records), max_age 1 and 8.  Each tracker's state carries over from call to call
as in a video.

model.stream frames/s (host clock over the whole iteration, after a warm-up pass of both): synthetic 640x480 uint8
frames, input size 512, HigherHRNet-W32 with PyTorch's default init (hpdecode.synth_net), flip test on, batch 8,
depth 4; track=True and track=True with smooth=OneEuro(30) alternated, each --stream-reps times.  The network
dominates these numbers.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "pytorch-human-pose_b200"))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_stream import frames_of, gpu_info  # noqa: E402
from bench_track import walking_records  # noqa: E402


def time_pair(frames_per_call, max_age, reps):
    from hpdecode import OneEuro, PoseTracker
    recs = walking_records(frames_per_call * (reps + 10))
    chunks = [recs[i * frames_per_call:(i + 1) * frames_per_call] for i in range(reps + 10)]
    trackers = {"hpd_track": PoseTracker(17, 30, 2, "cuda:0", max_age=max_age),
                "hpd_track_smooth": PoseTracker(17, 30, 2, "cuda:0", max_age=max_age, smoothing=OneEuro(30.0))}
    calls = {"hpd_track": lambda tr, c: tr.update(c), "hpd_track_smooth": lambda tr, c: tr.update_smoothed(c)}
    times = {k: [] for k in trackers}
    for i, c in enumerate(chunks):
        for name, tr in trackers.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            calls[name](tr, c)
            e1.record()
            e1.synchronize()
            if i >= 10:
                times[name].append(e0.elapsed_time(e1))
    row = {"frames_per_call": frames_per_call, "max_age": max_age}
    for name, t in times.items():
        med = float(np.median(t))
        row[name] = {"median_ms_per_call": med, "us_per_frame": med * 1e3 / frames_per_call,
                     "p90_ms": float(np.percentile(t, 90))}
    row["smooth_over_track"] = row["hpd_track_smooth"]["median_ms_per_call"] / row["hpd_track"]["median_ms_per_call"]
    return row


def stream_rates(n_frames, reps):
    from hpdecode import InferenceKeypointsModel, OneEuro, synth_net
    torch.manual_seed(0)
    model = InferenceKeypointsModel(synth_net.HigherHRNet(17, 32), use_flip=True, input_size=512, device="cuda:0")
    frames = frames_of(n_frames)
    modes = {"track": None, "track_smooth": OneEuro(30.0)}
    rows = {k: [] for k in modes}
    for sm in modes.values():                # warm-up of both paths
        assert sum(1 for _ in model.stream(frames, 8, 4, track=True, smooth=sm)) == n_frames
    for _ in range(reps):
        for name, sm in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = sum(1 for r in model.stream(frames, 8, 4, track=True, smooth=sm)
                    if (r.smoothed_coords is not None) == (sm is not None))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert n == n_frames
            rows[name].append(n_frames / dt)
            print(json.dumps({"mode": name, "frames_per_s": rows[name][-1]}), flush=True)
    return {"frames": n_frames, "batch_size": 8, "depth": 4, "frames_per_s_track": rows["track"],
            "frames_per_s_track_smooth": rows["track_smooth"],
            "median_smooth_over_track": float(np.median(rows["track_smooth"]) / np.median(rows["track"]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--stream-reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_smooth.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_smooth needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    result = {"gpu": gpu_info(), "track_calls": []}
    print(result["gpu"], flush=True)
    for max_age in (1, 8):
        for n in (8, 64):
            result["track_calls"].append(time_pair(n, max_age, args.reps))
            print(json.dumps(result["track_calls"][-1]), flush=True)
    result["stream"] = stream_rates(args.frames, args.stream_reps)
    result["stream"]["workload"] = "640x480 uint8 frames, input 512, HigherHRNet-W32 default init, flip test"
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
