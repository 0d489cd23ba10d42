"""Cost of drawing poses onto frames: hpd_render_poses against a plain device-to-device copy of the same frames, and
frame-stream inference with and without render.

  python tools/bench_render.py [--reps R] [--stream-frames N] [--stream-reps S] [--out profiles/r11_render.json]

Kernel time per frame (CUDA events around --reps launches, after a warm-up): 30 persons of 17 joints (COCO skeleton,
default PoseStyle: 3 px limbs, 4 px joints, tracked colours) spread over 640x480, 1920x1080 and 3840x2160 frames,
8 frames per launch, each frame in its own buffer; the copy is ``out.copy_(in)`` of the same 8 frames, timed the same
way and alternated with the kernel, so both see the same machine.  Frames and outputs of one size are 8 x 25 MB at
4K: the 4K working set is larger than the 126 MB L2, the smaller ones are not (both the copy and the kernel then
read from L2 after the first pass).

model.stream frames/s (host clock over the whole iteration, after a warm-up pass of both): 1920x1080 host uint8
frames, input size 512, HigherHRNet-W32 with PyTorch's default init (hpdecode.synth_net), flip test, batch 8, depth 4,
track=True; render off and on alternated.  With render on, every drawn frame is also copied back to the host
(6.2 MB per 1080p frame).  The card's name and power limit are read in the same run.
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

from bench_stream import gpu_info  # noqa: E402
from oracle import track_oracle as T  # noqa: E402

SIZES = ((480, 640), (1080, 1920), (2160, 3840))


def crowd_records(h, w, n, seed=0):
    """n frames of 30 standing persons (about h/4 tall) at random places, every joint visible."""
    rng = np.random.default_rng(seed)
    # a standing COCO pose in units of the person's height: nose, eyes, ears, shoulders, elbows, wrists, hips,
    # knees, ankles
    pose = np.array([[0, .05], [-.02, .03], [.02, .03], [-.05, .05], [.05, .05], [-.12, .18], [.12, .18], [-.16, .33],
                     [.16, .33], [-.17, .47], [.17, .47], [-.08, .52], [.08, .52], [-.09, .74], [.09, .74], [-.09, .96],
                     [.09, .96]])
    frames = []
    for _ in range(n):
        persons = []
        for _ in range(30):
            s = h / 4 * rng.uniform(0.7, 1.3)
            c = rng.uniform((0, 0), (w, h - s))
            persons.append((c + pose * s + rng.normal(0, 0.01 * s, pose.shape), np.ones(17, bool), 0.9))
        frames.append(persons)
    return torch.from_numpy(T.make_records(frames, 17, 30, 2)).cuda()


def time_kernel(h, w, reps, batch=8):
    from hpdecode import PoseRenderer, PoseStyle, ops
    r = PoseRenderer(17, 30, 2, PoseStyle())
    recs = crowd_records(h, w, batch)
    ids = torch.arange(batch * 30, dtype=torch.int32, device="cuda").reshape(batch, 30)
    ins = [torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(batch)]
    outs = [torch.empty_like(f) for f in ins]
    fns = {"render": lambda: ops.run_render(r.params, ins, outs, recs, ids),
           "copy": lambda: [o.copy_(f) for o, f in zip(outs, ins)]}
    for fn in fns.values():
        for _ in range(5):
            fn()
    times = {k: [] for k in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / batch)
    row = {"h": h, "w": w, "persons": 30, "frames_per_launch": batch, "frame_bytes": h * w * 3}
    for name, t in times.items():
        row[name] = {"median_us_per_frame": float(np.median(t)), "p10_us": float(np.percentile(t, 10)),
                     "p90_us": float(np.percentile(t, 90))}
    row["render_over_copy"] = row["render"]["median_us_per_frame"] / row["copy"]["median_us_per_frame"]
    row["render_GBps"] = 2 * h * w * 3 / row["render"]["median_us_per_frame"] / 1e3
    row["copy_GBps"] = 2 * h * w * 3 / row["copy"]["median_us_per_frame"] / 1e3
    return row


def stream_rates(n_frames, reps):
    from hpdecode import InferenceKeypointsModel, PoseStyle, synth_net
    torch.manual_seed(0)
    model = InferenceKeypointsModel(synth_net.HigherHRNet(17, 32), use_flip=True, input_size=512, device="cuda:0")
    rng = np.random.default_rng(0)
    frames = [rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8) for _ in range(n_frames)]
    modes = {"render_off": None, "render_on": PoseStyle()}
    rows = {k: [] for k in modes}
    for st in modes.values():                # warm-up of both paths
        assert sum(1 for _ in model.stream(frames, 8, 4, track=True, render=st)) == n_frames
    for _ in range(reps):
        for name, st in modes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = sum(1 for r in model.stream(frames, 8, 4, track=True, render=st)
                    if (r.rendered is not None) == (st is not None))
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            assert n == n_frames
            rows[name].append(n_frames / dt)
            print(json.dumps({"mode": name, "frames_per_s": rows[name][-1]}), flush=True)
    return {"frames": n_frames, "batch_size": 8, "depth": 4, "track": True,
            "frames_per_s_render_off": rows["render_off"], "frames_per_s_render_on": rows["render_on"],
            "median_on_over_off": float(np.median(rows["render_on"]) / np.median(rows["render_off"])),
            "note": "render on includes one device-to-host copy of every drawn frame (6.2 MB at 1080p)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--stream-frames", type=int, default=128)
    ap.add_argument("--stream-reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_render.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_render needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    result = {"gpu": gpu_info(), "kernel": []}
    print(result["gpu"], flush=True)
    for h, w in SIZES:
        result["kernel"].append(time_kernel(h, w, args.reps))
        print(json.dumps(result["kernel"][-1]), flush=True)
    result["stream"] = stream_rates(args.stream_frames, args.stream_reps)
    result["stream"]["workload"] = "1920x1080 host uint8 frames, input 512, HigherHRNet-W32 default init, flip test"
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
