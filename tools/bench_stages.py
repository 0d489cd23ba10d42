"""Single-stage heads (HRNet with the associative-embedding head): agg_nms_x4_kernel against the generic kernel on the
same inputs, and the pipelined decode rate of 1-stage against 2-stage heads.

Workload: synthetic W32 network (hpdecode.synth_net, num_deconvs=0 and 1) at 512 x 512, flip test, B = 64.  The
network outputs of one batch (142 MB per run, 285 MB with the flipped run) are larger than the B200's 126 MB L2, so
the kernels read them from HBM.  The two aggregation kernels alternate launch by launch, timed with CUDA events.
The peak the bandwidth is compared with is measured in the same run: a device-to-device copy of 4 GB.

    python tools/bench_stages.py --out profiles/r8_stages.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "pytorch-human-pose_b200"), ROOT]

import torch  # noqa: E402

from hpdecode import BottomUpDecoder, DecodePipeline, ops, synth_net  # noqa: E402


def _gpu():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def _copy_peak(nbytes=4 << 30, reps=10):
    a = torch.empty(nbytes // 4, device="cuda:0")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) / 1e3)


def _agg_bytes(B, K, H, W, flip):
    q = (H // 4) * (W // 4)
    reads = B * K * q * 4 * ((2 if flip else 1) + 1)            # heatmap (+ flipped run) and the first tag component
    wpr, HB = (W + 31) // 32, (H + 3) // 4
    writes = B * K * (H * W + 3 * H * wpr + 2 * HB * wpr) * 4    # agg_hm, mask / wmax / hmax, tag bounds
    return reads + writes


def _time_agg(scales, B, K, H, W, E, launches):
    params = {f: ops.make_params(B, K, H, W, E, 30, 0.05, 0.5) for f in (0, 1)}
    params[1].force_generic = 1
    bufs = ops.DecodeBuffers(B, K, H, W, E, 30, "cuda:0", tags=False)
    ms = {0: [], 1: []}
    for f in (0, 1, 0, 1):                                      # warm-up: module load, shared-memory opt-in
        ops.run_stage("aggregate_nms", bufs, params[f], scales=scales)
    for _ in range(launches):
        for f in (0, 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.run_stage("aggregate_nms", bufs, params[f], scales=scales)
            e1.record()
            e1.synchronize()
            ms[f].append(e0.elapsed_time(e1))
    return ms


def _pipeline_rate(scales, H, W, batches, depth=3):
    dec = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0")
    pipe = DecodePipeline(dec, depth=depth)
    B = ops.stage_scale(scales[0])["hm"][0].shape[0]
    for _ in range(depth):
        pipe.submit(scales, (H, W))
    pipe.drain()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(batches):
        pipe.submit(scales, (H, W))
    pipe.drain()
    e1.record()
    torch.cuda.synchronize()
    return batches * B / (e0.elapsed_time(e1) / 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--batches", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stages needs a GPU")
    B, S, K = args.batch, args.size, 17
    res = {"gpu": _gpu(), "workload": f"W32 {S}x{S}, flip, B={B}, K={K}, synthetic network outputs"}
    one = synth_net.network_outputs(B, S, flip=True, seed=0, num_deconvs=0)
    two = synth_net.network_outputs(B, S, flip=True, seed=0, num_deconvs=1)
    torch.cuda.synchronize()
    peak = _copy_peak()
    ms = _time_agg([one], B, K, S, S, 2, args.launches)
    nbytes = _agg_bytes(B, K, S, S, True)
    med = {f: sorted(v)[len(v) // 2] for f, v in ms.items()}
    res["aggregation"] = {
        "launches_each": args.launches,
        "x4_ms": ms[0], "generic_ms": ms[1],
        "x4_median_ms": med[0], "generic_median_ms": med[1], "speedup_median": med[1] / med[0],
        "bytes_moved_x4": nbytes,
        "x4_tb_per_s": nbytes / (med[0] / 1e3) / 1e12,
        "measured_copy_peak_tb_per_s": peak / 1e12,
        "x4_share_of_measured_peak": nbytes / (med[0] / 1e3) / peak,
        "x4_share_of_datasheet_7p7_tb_per_s": nbytes / (med[0] / 1e3) / 7.7e12,
    }
    res["pipelined_images_per_s"] = {"one_stage": _pipeline_rate([one], S, S, args.batches),
                                     "two_stage": _pipeline_rate([two], S, S, args.batches),
                                     "depth": 3, "batches": args.batches}
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
