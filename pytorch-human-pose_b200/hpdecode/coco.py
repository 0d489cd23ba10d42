"""COCO keypoint results from decoded batches (SURVEY.md 8(f)-2): the feed of
/root/reference/src/keypoints/bin/eval.py:18-49.

The record of a person -- ``[x, y, 1] * K`` in raw-image coordinates plus the person score -- is laid out by the
decode's last kernel (HpdRecordLayout.coco, csrc/refine.cu); this module only walks the host copy of a batch's
records and attaches image ids.  ``evaluate_dataset_batched`` is ``evaluate_dataset`` with the dataset loop
feeding the batched decoder B images at a time instead of one.
"""
from pathlib import Path
from typing import List, Optional, Sequence

from .decoder import Records


def batch_to_coco(image_ids: Sequence[int], records: Records) -> List[dict]:
    """records: host records of one decoded batch (DecodeResult.host()); one dict per person, image order kept."""
    out: List[dict] = []
    for b, image_id in enumerate(image_ids):
        out.extend(records.coco_records(b, image_id))
    return out


def result_to_coco(image_id: int, result) -> List[dict]:
    """eval.py:31-47 for one InferenceKeypointsResult (the reference's per-image path)."""
    recs = []
    for kpts, score in zip(result.kpts_coords, result.obj_scores):
        flat = [0.0] * (3 * len(kpts))
        flat[0::3] = [float(v) for v in kpts[:, 0]]
        flat[1::3] = [float(v) for v in kpts[:, 1]]
        flat[2::3] = [1.0] * len(kpts)
        recs.append({"image_id": int(image_id), "category_id": 1, "keypoints": flat, "score": float(score)})
    return recs


def image_id_of(filepath: str) -> int:
    """eval.py:23: COCO file name -> image id."""
    return int(Path(filepath).stem.lstrip("0"))


def evaluate_dataset_batched(model, dataset, batch_size: int = 32, limit: Optional[int] = None) -> List[dict]:
    """bin/eval.py:18-49 with a batched loop.  ``dataset`` needs what the reference's loop uses:
    ``images_filepaths`` and ``load_image(idx)`` (datasets/coco.py).  Images are loaded ``batch_size`` at a time,
    grouped by resized size inside ``model.predict_batch``-like steps, decoded on the device, and the COCO dicts
    are read from the records' COCO section -- no per-person host arithmetic."""
    from . import geometry
    n = len(dataset) if limit is None else min(limit, len(dataset))
    results: List[dict] = []
    min_scale = min(model.test_scales)
    for i0 in range(0, n, batch_size):
        idxs = list(range(i0, min(i0 + batch_size, n)))
        images = [dataset.load_image(i) for i in idxs]
        ids = [image_id_of(dataset.images_filepaths[i]) for i in idxs]
        per_image: List[List[dict]] = [[] for _ in idxs]
        groups = geometry.group_by_resized_size([im.shape[:2] for im in images], model.input_size, 1.0, min_scale)
        for size, members in groups.items():
            imgs = [images[j] for j in members]
            x, _, _, minv = geometry.prepare_input(imgs, model.input_size, model.device, 1.0, min_scale, return_inverse=True)
            extra = [geometry.prepare_input(imgs, model.input_size, model.device, s, min_scale)[0]
                     for s in model.test_scales if s != 1.0]
            rec = model.forward_decode(x, inv_affine=minv, extra_scales=extra).host()
            for b, j in enumerate(members):
                per_image[j] = rec.coco_records(b, ids[j])
        for recs in per_image:          # dataset order, like the reference's loop
            results.extend(recs)
    return results


def eval_coco(gt, results, device="cuda:0", verbose: bool = True):
    """bin/eval.py:52-65 on the device: COCO(gt).loadRes(results) and COCOeval(..., "keypoints") evaluate /
    accumulate / summarize.  gt: a COCO keypoint annotation dict or the path of its JSON file; results: a list of
    result dicts or the path of their JSON file.  Prints the summary like pycocotools and returns the
    CocoEvalResult (``stats`` holds the ten numbers)."""
    import json
    from .cocoeval import KeypointEvaluator, KeypointGroundTruth
    if not isinstance(gt, dict):
        with open(gt) as f:
            gt = json.load(f)
    if not isinstance(results, (list, tuple)):
        with open(results) as f:
            results = json.load(f)
    res = KeypointEvaluator(KeypointGroundTruth.from_coco(gt, device)).evaluate_results(results)
    if verbose:
        print("\n".join(res.summary()))
    return res
