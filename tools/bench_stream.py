"""Frames/s of frame-stream inference from host uint8 frames, and the input side alone.

  python tools/bench_stream.py [--frames N] [--bf16] [--out profiles/stream.json]

Workload: synthetic 640x480 uint8 frames (seeded), input size 512, HigherHRNet-W32 with PyTorch's default init
(hpdecode.synth_net), flip test on.  Rows:
  * per_frame: the reference's loop, ``model(frame)`` once per frame (batch 1, maps copied back, one sync per frame);
  * stream: ``model.stream(frames, batch_size, depth)`` for batch_size in {1, 8, 32} and depth in {1, 4};
  * with --bf16, the same rows with autocast_dtype=torch.bfloat16.
Each row is timed with a host clock over the whole iteration (the stream's results wait for every batch), after a
warm-up pass over the same frames.  The network dominates these numbers; they are end-to-end rates, not kernel times.

Input side (CUDA events, median of --reps): the inputs of test scales 0.5 / 1.0 / 1.5 at input size 640 (config 3's
scales) plus the flip-test copies for a batch of 640x480 images already on the device:
  * ``hpd_prepare_inputs``: one launch per 32 (scale, image) pairs;
  * ``hpd_prepare_input`` once per scale + ``torch.flip(x, [3])`` per scale (what predict_batch runs).
Both outputs are checked for equality before timing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "pytorch-human-pose_b200"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name()


def frames_of(n, seed=0):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for _ in range(n)]


def time_rate(fn, frames):
    fn(frames)                        # warm-up: every shape of the timed pass, allocator, cuDNN plans
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = fn(frames)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert n == len(frames)
    return {"frames": len(frames), "seconds": dt, "frames_per_s": len(frames) / dt}


def end_to_end(args, dtype):
    from hpdecode import InferenceKeypointsModel, synth_net
    torch.manual_seed(0)
    model = InferenceKeypointsModel(synth_net.HigherHRNet(17, 32), use_flip=True, input_size=512, device="cuda:0",
                                    autocast_dtype=dtype)
    frames = frames_of(args.frames)
    rows = [dict(mode="per_frame", batch_size=1, depth=1,
                 **time_rate(lambda fs: sum(1 for f in fs if model(f) is not None), frames[: args.per_frame]))]
    print(json.dumps({"dtype": str(dtype), **rows[-1]}), flush=True)
    for bs in (1, 8, 32):
        for depth in (1, 4):
            r = time_rate(lambda fs: sum(1 for _ in model.stream(fs, bs, depth)), frames)
            rows.append(dict(mode="stream", batch_size=bs, depth=depth, **r))
            print(json.dumps({"dtype": str(dtype), **rows[-1]}), flush=True)
    base = rows[0]["frames_per_s"]
    for r in rows:
        r["vs_per_frame"] = r["frames_per_s"] / base
    return rows


def input_side(args):
    from hpdecode import geometry
    scales, B = (0.5, 1.0, 1.5), args.input_batch
    imgs = [torch.from_numpy(f).cuda() for f in frames_of(B, seed=1)]
    sizes_hw, fwd, _ = geometry.multi_scale_geometry([im.shape[:2] for im in imgs], 640, scales)
    fwd_t = torch.from_numpy(fwd)
    mean, std = list(geometry.MEAN), list(geometry.STD)

    def fused():
        return torch.ops.hpd.prepare_inputs(imgs, fwd_t, sizes_hw, True, mean, std)

    def separate():
        xs = [torch.ops.hpd.prepare_input(imgs, fwd_t[t], sizes_hw[2 * t], sizes_hw[2 * t + 1], mean, std)
              for t in range(len(scales))]
        return xs, [torch.flip(x, [3]) for x in xs]

    a, b = fused(), separate()
    for x, y in zip(a[0] + a[1], b[0] + b[1]):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    out_bytes = sum(2 * x.numel() * 4 for x in a[0])
    res = {}
    for name, fn in (("prepare_inputs", fused), ("prepare_input_x3_plus_flip", separate)) * 2:   # alternated
        for _ in range(5):
            fn()
        times = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        res.setdefault(name, []).append(float(np.median(times)))
    out = {k: {"median_ms_per_pass": v, "output_GB_per_s": [out_bytes / (t * 1e-3) / 1e9 for t in v]} for k, v in res.items()}
    out["images"], out["scales"], out["input_size"], out["flip"] = B, list(scales), 640, True
    out["output_bytes"] = out_bytes
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=128)
    ap.add_argument("--per-frame", type=int, default=32, help="frames of the per-frame baseline")
    ap.add_argument("--bf16", action="store_true")
    ap.add_argument("--input-batch", type=int, default=8)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "stream.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stream needs a CUDA device")
    torch.backends.cudnn.benchmark = True
    result = {"gpu": gpu_info(), "workload": "640x480 uint8 frames, input 512, HigherHRNet-W32 default init, flip test"}
    result["input_side"] = input_side(args)
    print(json.dumps(result["input_side"]), flush=True)
    if not args.skip_e2e:
        result["fp32"] = end_to_end(args, None)
        if args.bf16:
            result["bf16"] = end_to_end(args, torch.bfloat16)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
