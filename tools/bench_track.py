"""Cost of person tracking: hpd_track per call, and frame-stream inference with tracking off and on.

  python tools/bench_track.py [--frames N] [--reps R] [--out profiles/r9_track.json]

hpd_track (CUDA events, median of --reps calls, after a warm-up): calls of 8 and 64 frames of 30-person records
(K = 17, E = 2, every slot filled), max_age 1 and 8.  The records are a seeded scene of 30 people walking, so most
persons match a track; the state carries over from call to call as in a video.

model.stream frames/s (host clock over the whole iteration, after a warm-up pass): synthetic 640x480 uint8 frames,
input size 512, HigherHRNet-W32 with PyTorch's default init (hpdecode.synth_net), flip test on, batch 8, depth 4;
tracking off and on alternated, each --stream-reps times.  The network dominates these numbers.
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


def walking_records(n, K=17, M=30, E=2, seed=0):
    from oracle import track_oracle as T
    rng = np.random.default_rng(seed)
    shape = np.stack([(rng.random((M, K)) - 0.5) * 80, (rng.random((M, K)) - 0.5) * 160], -1)
    pos, vel = rng.uniform(0, 1500, (M, 2)), rng.normal(0, 3, (M, 2))
    frames = []
    for _ in range(n):
        pos = pos + vel
        frames.append([(pos[i] + shape[i] + rng.normal(0, 1, (K, 2)), np.ones(K, bool), float(rng.random()))
                       for i in range(M)])
    return torch.from_numpy(T.make_records(frames, K, M, E)).cuda()


def time_track(frames_per_call, max_age, reps):
    from hpdecode import PoseTracker
    recs = walking_records(frames_per_call * (reps + 10))
    tr = PoseTracker(17, 30, 2, "cuda:0", max_age=max_age)
    chunks = [recs[i * frames_per_call:(i + 1) * frames_per_call] for i in range(reps + 10)]
    for c in chunks[:10]:
        tr.update(c)
    times, ids = [], None
    for c in chunks[10:]:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ids = tr.update(c)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    med = float(np.median(times))
    return {"frames_per_call": frames_per_call, "max_age": max_age, "median_ms_per_call": med,
            "us_per_frame": med * 1e3 / frames_per_call, "p90_ms": float(np.percentile(times, 90)),
            "matched_share_last_call": float((ids >= 0).float().mean())}


def stream_rates(n_frames, reps):
    from hpdecode import InferenceKeypointsModel, synth_net
    torch.manual_seed(0)
    model = InferenceKeypointsModel(synth_net.HigherHRNet(17, 32), use_flip=True, input_size=512, device="cuda:0")
    frames = frames_of(n_frames)
    rows = {False: [], True: []}
    for track in (False, True):                # warm-up of both paths
        assert sum(1 for _ in model.stream(frames, 8, 4, track=track)) == n_frames
    for _ in range(reps):
        for track in (False, True):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = sum(1 for r in model.stream(frames, 8, 4, track=track) if (r.track_ids is not None) == track)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert n == n_frames
            rows[track].append(n_frames / dt)
            print(json.dumps({"track": track, "frames_per_s": rows[track][-1]}), flush=True)
    return {"frames": n_frames, "batch_size": 8, "depth": 4, "frames_per_s_off": rows[False],
            "frames_per_s_on": rows[True], "median_on_over_off": float(np.median(rows[True]) / np.median(rows[False]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--stream-reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_track.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_track needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    result = {"gpu": gpu_info(), "hpd_track": []}
    print(result["gpu"], flush=True)
    for max_age in (1, 8):
        for n in (8, 64):
            result["hpd_track"].append(time_track(n, max_age, args.reps))
            print(json.dumps(result["hpd_track"][-1]), flush=True)
    result["stream"] = stream_rates(args.frames, args.stream_reps)
    result["stream"]["workload"] = "640x480 uint8 frames, input 512, HigherHRNet-W32 default init, flip test"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
