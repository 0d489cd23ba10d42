"""Time the decode on float32, float16 and bfloat16 network outputs of the same seeded HigherHRNet run.

Workloads (bench.py's inputs: synth_net, weights from seed 1, images from seed 2):
  cfg2  HigherHRNet-W32 512x512, flip, batch 64 (agg_nms_x2_kernel)
  cfg3  HigherHRNet-W48 640x640, test scales 0.5/1.0/1.5, flip, batch 32 (agg_nms_ms_kernel); fp16 is also timed
        through the generic kernel (force_generic bit 0), the only kernel that took 16-bit multi-scale inputs before.
Both workloads also time "bfloat16_via_float32": the bf16 outputs converted with .float() inside the timed region,
then the float32 decode -- what a bf16 caller had to do before the decode read bf16.
The 16-bit inputs are the float32 outputs rounded once (hm_lo / tag stay channel slices of one tensor).  Before any
timing, each 16-bit decode is checked against the float32 decode of its up-cast inputs (every stage output, bit for
bit).  Two regions are timed with CUDA events: the aggregation kernel alone (hpd_aggregate_nms) and the whole
sequential decode step (hpd_decode on one stream).  The variants alternate within each repeat; the medians and the
spread (min, max) over the repeats are reported.  Inputs exceed the 126 MB L2 (cfg2 float32: 856 MB).

    python tools/bench_16bit.py --out profiles/r5_16bit.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-human-pose_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    "cfg2": dict(arch=32, size=512, batch=64, scales=(1.0,), tag_scale=0),
    "cfg3": dict(arch=48, size=640, batch=32, scales=(0.5, 1.0, 1.5), tag_scale=1),
}


def to16(s, dtype):
    out = {}
    for suf in ("", "_f"):
        K = s["hm_lo" + suf].shape[1]
        both = torch.cat((s["hm_lo" + suf], s["tag" + suf]), 1).to(dtype)
        out["hm_lo" + suf], out["tag" + suf] = both[:, :K], both[:, K:]
        out["hm_hi" + suf] = s["hm_hi" + suf].to(dtype)
    return out


def input_bytes(scales):
    return sum(t.numel() * t.element_size() for s in scales for t in s.values())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg2,cfg3")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=15)
    ap.add_argument("--iters", type=int, default=5, help="launches per timed sample")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_16bit needs a CUDA device")
    from hpdecode import ops, synth_net

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rec = {"what": "decode of float32 / float16 / bfloat16 network outputs: aggregation kernel and whole sequential "
                   "decode step, CUDA events, variants alternating", "gpu": smi[0] if smi else "unknown",
           "device": torch.cuda.get_device_name(0), "torch": torch.__version__, "warmup": a.warmup,
           "repeats": a.repeats, "iters_per_sample": a.iters, "workloads": {}}
    for name in a.workloads.split(","):
        wl = WORKLOADS[name]
        B, S = wl["batch"], wl["size"]
        f32 = [synth_net.network_outputs(B, int(round(S * s / 64.0)) * 64, flip=True, seed=1, C=wl["arch"],
                                         device="cuda:0", chunk=8 if S <= 512 else 4) for s in wl["scales"]]
        ins = {"float32": f32, "float16": [to16(s, torch.float16) for s in f32],
               "bfloat16": [to16(s, torch.bfloat16) for s in f32]}
        variants = [("float32", "float32", 0), ("float16", "float16", 0), ("bfloat16", "bfloat16", 0),
                    ("bfloat16_via_float32", "bfloat16", 0)]
        if len(wl["scales"]) > 1:
            variants.insert(2, ("float16_generic", "float16", 1))
        p = ops.make_params(B, 17, S, S, 2, 30, 0.05, 0.5, num_scales=len(wl["scales"]), tag_scale=wl["tag_scale"])
        bufs = {v: ops.DecodeBuffers(B, 17, S, S, 2, 30, "cuda:0", tags=False) for v, _, _ in variants}

        def run(v, src, force, whole):
            p.force_generic = force
            scales = ins[src]
            if v.endswith("_via_float32"):
                scales = [{k: t.float() for k, t in s.items()} for s in scales]
            if whole:
                ops.run_decode(scales, bufs[v], p)
            else:
                ops.run_stage("aggregate_nms", bufs[v], p, scales=scales)

        # correctness before timing: each 16-bit decode equals the float32 decode of its up-cast inputs
        checks = {}
        for v, src, force in variants:
            if src == "float32" or v.endswith("_via_float32"):
                continue
            ref = ops.DecodeBuffers(B, 17, S, S, 2, 30, "cuda:0", tags=False)
            p.force_generic = force
            ops.run_decode([{k: t.float() for k, t in s.items()} for s in ins[src]], ref, p)
            run(v, src, force, True)
            torch.cuda.synchronize()
            same = all(torch.equal(getattr(ref, f).view(torch.int32) if getattr(ref, f).is_floating_point() else getattr(ref, f),
                                   getattr(bufs[v], f).view(torch.int32) if getattr(bufs[v], f).is_floating_point() else getattr(bufs[v], f))
                       for f in ("agg_hm", "nms_mask", "hm_wmax", "tag_bmin", "tag_bmax", "scores_k", "idx_k", "tags_k",
                                 "poses", "person_scores", "n_person", "flags"))
            checks[v] = bool(same)
            del ref
            if not same:
                raise SystemExit(f"{name} {v}: the 16-bit decode differs from the float32 decode of the up-cast inputs")
        times = {(v, w): [] for v, _, _ in variants for w in (False, True)}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for rep in range(a.warmup + a.repeats):
            for whole in (False, True):
                for v, src, force in variants:
                    ev0.record()
                    for _ in range(a.iters):
                        run(v, src, force, whole)
                    ev1.record()
                    ev1.synchronize()
                    if rep >= a.warmup:
                        times[(v, whole)].append(ev0.elapsed_time(ev1) / a.iters)
        out = {"config": f"HigherHRNet-W{wl['arch']} {S}x{S}, scales {list(wl['scales'])}, flip, batch {B}",
               "checked_bit_exact_vs_upcast_float32": checks, "variants": {}}
        for v, src, force in variants:
            agg, dec = np.array(times[(v, False)]), np.array(times[(v, True)])
            out["variants"][v] = {
                "input_dtype": src, "force_generic": force, "input_bytes": input_bytes(ins[src]),
                "aggregate_ms_median": float(np.median(agg)), "aggregate_ms_min": float(agg.min()),
                "aggregate_ms_max": float(agg.max()), "decode_ms_median": float(np.median(dec)),
                "decode_ms_min": float(dec.min()), "decode_ms_max": float(dec.max()),
                "aggregate_input_GBps": input_bytes(ins[src]) / (np.median(agg) * 1e-3) / 1e9,
            }
        rec["workloads"][name] = out
        print(json.dumps({name: out}), flush=True)
        del ins, bufs, f32
        torch.cuda.empty_cache()
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
