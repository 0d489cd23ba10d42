"""COCO keypoint evaluation on the device: the AP / AR that bin/eval.py:52-65 gets from pycocotools'
``COCOeval(gt, dt, "keypoints")`` with ``evaluate()``, ``accumulate()`` and ``summarize()``.

``hpd_coco_eval`` (csrc/cocoeval.cu) computes the OKS of every (detection, gt) pair, the greedy matching of every area
range and OKS threshold, the global score order and accumulate's precision / recall / score arrays.  Detections are read
where they are: in the decode's result records (``evaluate_records``), or packed from COCO result dicts
(``evaluate_results``, the ``loadRes`` path).  The ten summary numbers are a mean over those arrays, computed here with
pycocotools' own ``_summarize`` code.

One category (person, id 1) and one maxDets entry, as in pycocotools' keypoint parameters (``setKpParams``).
"""
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops

COCO_KPT_OKS_SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89,
                                .89]) / 10.0
# Params.setKpParams
IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
AREA_RNG = [[0 ** 2, 1e5 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
AREA_RNG_LBL = ['all', 'medium', 'large']


class KeypointGroundTruth:
    """The ground truth of the evaluated images on the device, padded to G annotations per image (category 1, each
    image's annotations in dataset order, images in ascending id order like COCOeval's ``p.imgIds``)."""

    def __init__(self, image_ids: Sequence[int], dataset_image_ids, kpts: np.ndarray, area: np.ndarray,
                 bbox: np.ndarray, iscrowd: np.ndarray, ignore: np.ndarray, n_gt: np.ndarray, device):
        self.image_ids = [int(i) for i in image_ids]
        self.index = {i: n for n, i in enumerate(self.image_ids)}
        self.dataset_image_ids = set(int(i) for i in dataset_image_ids)
        self.num_kpts = kpts.shape[2]
        dev = torch.device(device)
        self.kpts = torch.from_numpy(kpts).to(dev)
        self.area = torch.from_numpy(area).to(dev)
        self.bbox = torch.from_numpy(bbox).to(dev)
        self.iscrowd = torch.from_numpy(iscrowd).to(dev)
        self.ignore = torch.from_numpy(ignore).to(dev)
        self.n_gt = torch.from_numpy(n_gt).to(dev)

    @property
    def device(self):
        return self.kpts.device

    @classmethod
    def from_coco(cls, dataset: dict, device, image_ids: Optional[Sequence[int]] = None) -> "KeypointGroundTruth":
        """dataset: a COCO keypoint annotation dict (``images``, ``annotations``).  image_ids: the evaluated images
        (COCOeval's ``p.imgIds``; default: every image of the dataset).  ``ignore`` is COCOeval._prepare's:
        iscrowd, or no labelled keypoint."""
        all_ids = [int(img['id']) for img in dataset['images']]
        ids = [int(i) for i in np.unique(all_ids if image_ids is None else list(image_ids))]
        index = {i: n for n, i in enumerate(ids)}
        per: List[List[dict]] = [[] for _ in ids]
        for ann in dataset['annotations']:
            n = index.get(int(ann['image_id']))
            if n is not None and ann['category_id'] == 1:
                per[n].append(ann)
        anns = [a for p in per for a in p]
        K = len(anns[0]['keypoints']) // 3 if anns else 17
        I, G = len(ids), max([1] + [len(p) for p in per])
        if not ids:
            raise _lib.HpdError("coco_eval: no images to evaluate")
        if G > _lib.HPD_COCO_MAX_PER_IMAGE:
            raise _lib.HpdError(f"coco_eval: at most {_lib.HPD_COCO_MAX_PER_IMAGE} annotations per image (got {G})")
        kpts = np.zeros((I, G, K, 3))
        area, bbox = np.zeros((I, G)), np.zeros((I, G, 4))
        iscrowd, ignore = np.zeros((I, G), np.uint8), np.zeros((I, G), np.uint8)
        n_gt = np.array([len(p) for p in per], np.int32)
        for i, p in enumerate(per):
            for g, ann in enumerate(p):
                if len(ann['keypoints']) != 3 * K:
                    raise _lib.HpdError(f"coco_eval: annotation {ann.get('id')} has {len(ann['keypoints'])} keypoint "
                                        f"values, expected {3 * K}")
                kpts[i, g] = np.asarray(ann['keypoints'], np.float64).reshape(K, 3)
                area[i, g] = ann['area']
                bbox[i, g] = ann['bbox']
                crowd = 'iscrowd' in ann and ann['iscrowd']
                iscrowd[i, g] = int(ann.get('iscrowd', 0))
                ignore[i, g] = bool((ann['num_keypoints'] == 0) or crowd)
        return cls(ids, all_ids, kpts, area, bbox, iscrowd, ignore, n_gt, device)


class CocoEvalResult:
    """accumulate's arrays in pycocotools' shapes (host, float64): ``precision`` / ``scores`` [T,R,1,A,1],
    ``recall`` [T,1,A,1]; ``stats`` (summarize's ten numbers) and ``summary()`` (its printed lines).
    With ``debug``: the device tensors ``oks`` [I,max_dets,G], ``codes`` [A,T,I,max_dets] and ``npig`` [A]."""

    def __init__(self, max_dets: int, outs: List[torch.Tensor], debug: bool):
        T, R, A = outs[0].shape
        self.max_dets = max_dets
        self.precision = outs[0].cpu().numpy().reshape(T, R, 1, A, 1)
        self.recall = outs[1].cpu().numpy().reshape(T, 1, A, 1)
        self.scores = outs[2].cpu().numpy().reshape(T, R, 1, A, 1)
        self.oks, self.codes, self.npig = (outs[3], outs[4], outs[5]) if debug else (None, None, None)
        self.stats, self._lines = summarize_kps(IOU_THRS, AREA_RNG_LBL, [max_dets], self.precision, self.recall)

    def summary(self) -> List[str]:
        return list(self._lines)


def summarize_kps(iou_thrs, area_lbl, max_dets, precision, recall) -> Tuple[np.ndarray, List[str]]:
    """COCOeval.summarize's _summarize / _summarizeKps on accumulate's arrays (pycocotools cocoeval.py), with
    maxDets[-1] where pycocotools writes 20 (the same at the default)."""
    lines = []

    def _summarize(ap=1, iouThr=None, areaRng='all', maxDets=100):
        iStr = ' {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}'
        titleStr = 'Average Precision' if ap == 1 else 'Average Recall'
        typeStr = '(AP)' if ap == 1 else '(AR)'
        iouStr = '{:0.2f}:{:0.2f}'.format(iou_thrs[0], iou_thrs[-1]) \
            if iouThr is None else '{:0.2f}'.format(iouThr)
        aind = [i for i, aRng in enumerate(area_lbl) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(max_dets) if mDet == maxDets]
        if ap == 1:
            s = precision
            if iouThr is not None:
                t = np.where(iouThr == iou_thrs)[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            s = recall
            if iouThr is not None:
                t = np.where(iouThr == iou_thrs)[0]
                s = s[t]
            s = s[:, :, aind, mind]
        if len(s[s > -1]) == 0:
            mean_s = -1
        else:
            mean_s = np.mean(s[s > -1])
        lines.append(iStr.format(titleStr, typeStr, iouStr, areaRng, maxDets, mean_s))
        return mean_s

    md = max_dets[-1]
    stats = np.zeros((10,))
    stats[0] = _summarize(1, maxDets=md)
    stats[1] = _summarize(1, maxDets=md, iouThr=.5)
    stats[2] = _summarize(1, maxDets=md, iouThr=.75)
    stats[3] = _summarize(1, maxDets=md, areaRng='medium')
    stats[4] = _summarize(1, maxDets=md, areaRng='large')
    stats[5] = _summarize(0, maxDets=md)
    stats[6] = _summarize(0, maxDets=md, iouThr=.5)
    stats[7] = _summarize(0, maxDets=md, iouThr=.75)
    stats[8] = _summarize(0, maxDets=md, areaRng='medium')
    stats[9] = _summarize(0, maxDets=md, areaRng='large')
    return stats, lines


class KeypointEvaluator:
    """COCOeval(gt, dt, "keypoints") on the device, for the images of ``gt``."""

    def __init__(self, gt: KeypointGroundTruth, sigmas=COCO_KPT_OKS_SIGMAS, max_dets: int = 20):
        sigmas = np.asarray(sigmas, np.float64)
        if sigmas.shape != (gt.num_kpts,):
            raise _lib.HpdError(f"coco_eval: need one sigma per joint ({gt.num_kpts}), got shape {sigmas.shape}")
        self.gt, self.max_dets = gt, int(max_dets)
        self.kpt_vars = (sigmas * 2) ** 2        # computeOks: vars = (sigmas * 2)**2

    def _image_index(self, image_id: int, seen: Dict[int, int]) -> int:
        i = self.gt.index.get(int(image_id))
        if i is None:
            raise _lib.HpdError(f"coco_eval: image {image_id} is not among the ground truth's images")
        if i in seen:
            raise _lib.HpdError(f"coco_eval: image {image_id} has detections in two places")
        seen[i] = 1
        return i

    def params(self):
        """HpdCocoEvalParams of this evaluation."""
        g = self.gt
        return ops.coco_eval_params(len(g.image_ids), g.num_kpts, self.max_dets, g.kpts.shape[1], IOU_THRS.tolist(),
                                    REC_THRS.tolist(), [float(v) for r in AREA_RNG for v in r], self.kpt_vars.tolist())

    def gt_tensors(self):
        g = self.gt
        return g.kpts, g.area, g.bbox, g.iscrowd, g.ignore, g.n_gt

    def _run(self, view, debug) -> CocoEvalResult:
        records, rows, off_coco, off_count, person_stride, max_per_row = view
        area = [float(v) for r in AREA_RNG for v in r]
        outs = torch.ops.hpd.coco_eval(records, torch.from_numpy(rows), off_coco, off_count, person_stride, max_per_row,
                                       *self.gt_tensors(), IOU_THRS.tolist(), REC_THRS.tolist(), area,
                                       self.kpt_vars.tolist(), self.max_dets, debug)
        return CocoEvalResult(self.max_dets, outs, debug)

    def records_view(self, batches: Sequence[Tuple[torch.Tensor, Sequence[int]]], M: int, K: int, E: int):
        """(records, row_of_image, off_coco, off_count, person_stride, max_per_row) for ops.run_coco_eval."""
        if K != self.gt.num_kpts:
            raise _lib.HpdError(f"coco_eval: records hold {K} joints, the ground truth {self.gt.num_kpts}")
        L = ops.record_layout(K, M, E)
        rows = np.full(len(self.gt.image_ids), -1, np.int64)
        seen: Dict[int, int] = {}
        tensors, start = [], 0
        for rec, ids in batches:
            if rec.dim() != 2 or rec.shape[1] < L.row_bytes or len(ids) > rec.shape[0]:
                raise _lib.HpdError(f"coco_eval: records must be [B, {L.row_bytes}] with one image id per row")
            for b, image_id in enumerate(ids):
                rows[self._image_index(image_id, seen)] = start + b
            tensors.append(rec)
            start += rec.shape[0]
        return tensors, rows, L.off_coco, L.off_n_person, L.coco_stride, M

    def results_view(self, results: Sequence[dict]):
        """COCO.loadRes's input packed into detection rows on the device: the same view as records_view."""
        K = self.gt.num_kpts
        C = 3 * K + 1
        per: Dict[int, List[dict]] = {}
        for r in results:
            image_id = int(r['image_id'])
            if image_id not in self.gt.dataset_image_ids:
                raise _lib.HpdError(f"coco_eval: result for image {image_id}, which is not in the ground truth")
            if r['category_id'] != 1 or image_id not in self.gt.index:
                continue
            if len(r['keypoints']) != 3 * K:
                raise _lib.HpdError(f"coco_eval: a result has {len(r['keypoints'])} keypoint values, expected {3 * K}")
            per.setdefault(image_id, []).append(r)
        D = max([1] + [len(v) for v in per.values()])
        if D > _lib.HPD_COCO_MAX_PER_IMAGE:
            raise _lib.HpdError(f"coco_eval: at most {_lib.HPD_COCO_MAX_PER_IMAGE} detections per image (got {D})")
        packed = np.zeros((max(len(per), 1), D * C + 1), np.float64)     # rows: [D][3K+1] persons, then the count
        rows = np.full(len(self.gt.image_ids), -1, np.int64)
        for n, (image_id, dets) in enumerate(per.items()):
            rows[self.gt.index[image_id]] = n
            for j, r in enumerate(dets):
                packed[n, j * C:j * C + 3 * K] = r['keypoints']
                packed[n, j * C + 3 * K] = r['score']
            packed[n, D * C:].view(np.int32)[0] = len(dets)
        rec = torch.from_numpy(packed.view(np.uint8)).to(self.gt.device)
        return [rec], rows, 0, 8 * D * C, C, D

    def evaluate_records(self, batches: Sequence[Tuple[torch.Tensor, Sequence[int]]], M: int, K: int, E: int,
                         debug: bool = False) -> CocoEvalResult:
        """batches: (records [B,row_bytes] uint8 on the device, image ids of its B rows) per decoded batch, as
        DecodeResult.packed() gives them; read in place.  An image may appear once; images of the ground truth
        without a row have no detections."""
        return self._run(self.records_view(batches, M, K, E), debug)

    def evaluate_results(self, results: Sequence[dict], debug: bool = False) -> CocoEvalResult:
        """COCO result dicts (``image_id``, ``category_id``, ``keypoints``, ``score``): COCO.loadRes, then the
        evaluation.  Each image keeps its detections in the order of the list (score ties are broken by it)."""
        return self._run(self.results_view(results), debug)
