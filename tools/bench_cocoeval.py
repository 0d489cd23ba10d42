"""Time the device COCO keypoint evaluation against the NumPy oracle on a seeded val2017-sized set.

5000 images, 0-15 ground-truth persons and 30 detections each (synth.coco_eval_set).  The device evaluation
(hpd_coco_eval through KeypointEvaluator.evaluate_results' packed rows, inputs resident, summary included) is timed
with CUDA events: warm-up, then ``--repeats`` runs.  The oracle runs once on the host.  Both must agree exactly on
precision / recall / scores / stats.  Writes a JSON record with the card name and power limit read in the same run.

    python tools/bench_cocoeval.py --out profiles/r4_cocoeval.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "pytorch-human-pose_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--dets", type=int, default=30)
    ap.add_argument("--max-gts", type=int, default=15)
    ap.add_argument("--seed", type=int, default=2017)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cocoeval needs a CUDA device")
    from hpdecode import KeypointEvaluator, KeypointGroundTruth, ops, synth
    from hpdecode.cocoeval import CocoEvalResult
    from oracle import coco_eval_oracle as O

    dataset, results = synth.coco_eval_set(a.images, seed=a.seed, max_gts=a.max_gts, dets_per_image=a.dets)
    E = KeypointEvaluator(KeypointGroundTruth.from_coco(dataset, "cuda:0"))
    view = E.results_view(results)            # resident packed detection rows
    p = E.params()
    T, R, A = p.num_iou_thrs, p.num_rec_thrs, p.num_areas
    f64 = dict(device="cuda:0", dtype=torch.float64)
    outs = [torch.empty((T, R, A), **f64), torch.empty((T, A), **f64), torch.empty((T, R, A), **f64), None, None, None]

    def run():
        ops.run_coco_eval(p, *view, E.gt_tensors(), outs)

    for _ in range(a.warmup):
        run()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(a.repeats):
        ev0.record()
        run()
        ev1.record()
        ev1.synchronize()
        times.append(ev0.elapsed_time(ev1))
    t0 = time.perf_counter()
    end_to_end = E.evaluate_results(results)   # packing the dicts + evaluation + host summary
    e2e_ms = (time.perf_counter() - t0) * 1e3
    dev = CocoEvalResult(E.max_dets, outs[:3] + [None] * 3, False)

    t0 = time.perf_counter()
    ev = O.COCOevalKeypoints(dataset, results).run()
    oracle_s = time.perf_counter() - t0
    agree = all(np.array_equal(x, y) for x, y in ((dev.precision, ev.eval['precision']), (dev.recall, ev.eval['recall']),
                                                   (dev.scores, ev.eval['scores']), (dev.stats, ev.stats),
                                                   (end_to_end.stats, ev.stats)))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rec = {
        "what": "COCO keypoint evaluation (evaluate + accumulate) of a seeded val2017-shaped set",
        "images": a.images, "dets_per_image": a.dets, "max_gts": a.max_gts, "gts": len(dataset["annotations"]),
        "detections": len(results), "seed": a.seed,
        "device_ms_median": float(np.median(times)), "device_ms_min": float(np.min(times)),
        "device_ms_max": float(np.max(times)), "repeats": a.repeats, "warmup": a.warmup,
        "evaluate_results_ms_incl_packing_and_summary": e2e_ms,
        "oracle_numpy_s": oracle_s, "exact_agreement": bool(agree), "oks_margin": ev.oks_margin(),
        "stats": [float(x) for x in ev.stats], "gpu": smi[0] if smi else "unknown",
        "torch": torch.__version__, "numpy": np.__version__,
    }
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not agree:
        raise SystemExit("device and oracle disagree")


if __name__ == "__main__":
    main()
