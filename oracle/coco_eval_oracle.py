"""NumPy restatement of pycocotools 2.0.x ``cocoeval.py`` for ``iouType="keypoints"`` (and the keypoint branch of
``coco.py: COCO.loadRes``): the CPU oracle of ``hpd_coco_eval``.

pycocotools is not installable offline, so its published source is restated here function by function, keeping its
own expressions and their order so the two can be diffed line by line.  Only what the keypoint evaluation of one
category (person, id 1) reads is kept.  Inputs are plain COCO dicts: the ground-truth dataset (``images``,
``annotations``) and the result list (``image_id``, ``category_id``, ``keypoints``, ``score``).

Exactness: every step after ``computeOks`` is comparisons, integer counts and the same IEEE operations in the same
order, so the device reproduces it exactly.  ``computeOks`` itself ends in ``np.exp``, whose last bit depends on the
host's NumPy build; ``oks_margin`` reports how far the OKS values of a scene are from every decision they feed.
"""
import copy
from collections import defaultdict

import numpy as np

KPT_OKS_SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0

# dtIgnore / dtMatches of one (area, threshold, image, rank) slot folded into one code, as the device writes it
ABSENT, TP, FP, IGNORED = 0, 1, 2, 3


class Params:
    """cocoeval.py: Params.setKpParams (+ the imgIds / catIds defaults of Params.__init__)."""

    def __init__(self, img_ids, sigmas=None, max_dets=20):
        self.imgIds = list(img_ids)
        self.catIds = [1]
        self.iouThrs = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
        self.recThrs = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
        self.maxDets = [max_dets]
        self.areaRng = [[0 ** 2, 1e5 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
        self.areaRngLbl = ['all', 'medium', 'large']
        self.useCats = 1
        self.kpt_oks_sigmas = KPT_OKS_SIGMAS if sigmas is None else np.asarray(sigmas, np.float64)


def load_res(gt_image_ids, results):
    """coco.py: COCO.loadRes, keypoint branch: each result gets area / bbox from the min and max of its x and y and
    id = index + 1.  The dicts are copied (loadRes annotates the caller's)."""
    anns = copy.deepcopy(list(results))
    ann_img_ids = [ann['image_id'] for ann in anns]
    assert set(ann_img_ids) == (set(ann_img_ids) & set(gt_image_ids)), \
        'Results do not correspond to current coco set'
    for id, ann in enumerate(anns):
        s = ann['keypoints']
        x = s[0::3]
        y = s[1::3]
        x0, x1, y0, y1 = np.min(x), np.max(x), np.min(y), np.max(y)
        ann['area'] = (x1 - x0) * (y1 - y0)
        ann['id'] = id + 1
        ann['bbox'] = [x0, y0, x1 - x0, y1 - y0]
    return anns


class COCOevalKeypoints:
    """cocoeval.py: COCOeval(cocoGt, cocoDt, iouType='keypoints') restricted to category 1."""

    def __init__(self, gt_dataset, results, sigmas=None, max_dets=20, img_ids=None):
        self.gt_dataset = gt_dataset
        all_ids = sorted(img['id'] for img in gt_dataset['images'])       # Params: imgIds = sorted(cocoGt.getImgIds())
        self.params = Params(all_ids if img_ids is None else img_ids, sigmas, max_dets)
        self.dts_all = load_res(all_ids, results)
        self.eval = {}
        self.stats = None
        self.summary_lines = []

    def _prepare(self):
        """cocoeval.py: COCOeval._prepare (useCats): anns of the evaluated images and categories, in dataset order;
        ignore = iscrowd, then (num_keypoints == 0) or ignore."""
        p = self.params
        img_set, cat_set = set(p.imgIds), set(p.catIds)
        gts = [copy.copy(a) for a in self.gt_dataset['annotations']
               if a['image_id'] in img_set and a['category_id'] in cat_set]
        dts = [d for d in self.dts_all if d['image_id'] in img_set and d['category_id'] in cat_set]
        for gt in gts:
            gt['ignore'] = gt['ignore'] if 'ignore' in gt else 0
            gt['ignore'] = 'iscrowd' in gt and gt['iscrowd']
            gt['ignore'] = (gt['num_keypoints'] == 0) or gt['ignore']
        self._gts = defaultdict(list)
        self._dts = defaultdict(list)
        for gt in gts:
            self._gts[gt['image_id'], gt['category_id']].append(gt)
        for dt in dts:
            self._dts[dt['image_id'], dt['category_id']].append(dt)

    def evaluate(self):
        """cocoeval.py: COCOeval.evaluate."""
        p = self.params
        p.imgIds = list(np.unique(p.imgIds))
        p.catIds = list(np.unique(p.catIds))
        p.maxDets = sorted(p.maxDets)
        self._prepare()
        catIds = p.catIds
        self.ious = {(imgId, catId): self.computeOks(imgId, catId) for imgId in p.imgIds for catId in catIds}
        maxDet = p.maxDets[-1]
        self.evalImgs = [self.evaluateImg(imgId, catId, areaRng, maxDet)
                         for catId in catIds for areaRng in p.areaRng for imgId in p.imgIds]
        self._paramsEval = copy.deepcopy(self.params)

    def computeOks(self, imgId, catId):
        """cocoeval.py: COCOeval.computeOks."""
        p = self.params
        gts = self._gts[imgId, catId]
        dts = self._dts[imgId, catId]
        inds = np.argsort([-d['score'] for d in dts], kind='mergesort')
        dts = [dts[i] for i in inds]
        if len(dts) > p.maxDets[-1]:
            dts = dts[0:p.maxDets[-1]]
        if len(gts) == 0 or len(dts) == 0:
            return []
        ious = np.zeros((len(dts), len(gts)))
        sigmas = p.kpt_oks_sigmas
        vars = (sigmas * 2) ** 2
        k = len(sigmas)
        for j, gt in enumerate(gts):
            g = np.array(gt['keypoints'])
            xg = g[0::3]; yg = g[1::3]; vg = g[2::3]
            k1 = np.count_nonzero(vg > 0)
            bb = gt['bbox']
            x0 = bb[0] - bb[2]; x1 = bb[0] + bb[2] * 2
            y0 = bb[1] - bb[3]; y1 = bb[1] + bb[3] * 2
            for i, dt in enumerate(dts):
                d = np.array(dt['keypoints'])
                xd = d[0::3]; yd = d[1::3]
                if k1 > 0:
                    dx = xd - xg
                    dy = yd - yg
                else:
                    z = np.zeros((k))
                    dx = np.max((z, x0 - xd), axis=0) + np.max((z, xd - x1), axis=0)
                    dy = np.max((z, y0 - yd), axis=0) + np.max((z, yd - y1), axis=0)
                e = (dx ** 2 + dy ** 2) / vars / (gt['area'] + np.spacing(1)) / 2
                if k1 > 0:
                    e = e[vg > 0]
                ious[i, j] = np.sum(np.exp(-e)) / e.shape[0]
        return ious

    def evaluateImg(self, imgId, catId, aRng, maxDet):
        """cocoeval.py: COCOeval.evaluateImg."""
        p = self.params
        gt = self._gts[imgId, catId]
        dt = self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return None
        for g in gt:
            if g['ignore'] or (g['area'] < aRng[0] or g['area'] > aRng[1]):
                g['_ignore'] = 1
            else:
                g['_ignore'] = 0
        # sort dt highest score first, sort gt ignore last
        gtind = np.argsort([g['_ignore'] for g in gt], kind='mergesort')
        gt = [gt[i] for i in gtind]
        dtind = np.argsort([-d['score'] for d in dt], kind='mergesort')
        dt = [dt[i] for i in dtind[0:maxDet]]
        iscrowd = [int(o['iscrowd']) for o in gt]
        # load computed ious
        ious = self.ious[imgId, catId][:, gtind] if len(self.ious[imgId, catId]) > 0 else self.ious[imgId, catId]
        T = len(p.iouThrs)
        G = len(gt)
        D = len(dt)
        gtm = np.zeros((T, G))
        dtm = np.zeros((T, D))
        gtIg = np.array([g['_ignore'] for g in gt])
        dtIg = np.zeros((T, D))
        if not len(ious) == 0:
            for tind, t in enumerate(p.iouThrs):
                for dind, d in enumerate(dt):
                    # information about best match so far (m=-1 -> unmatched)
                    iou = min([t, 1 - 1e-10])
                    m = -1
                    for gind, g in enumerate(gt):
                        # if this gt already matched, and not a crowd, continue
                        if gtm[tind, gind] > 0 and not iscrowd[gind]:
                            continue
                        # if dt matched to reg gt, and on ignore gt, stop
                        if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                            break
                        # continue to next gt unless better match made
                        if ious[dind, gind] < iou:
                            continue
                        # if match successful and best so far, store appropriately
                        iou = ious[dind, gind]
                        m = gind
                    # if match made store id of match for both dt and gt
                    if m == -1:
                        continue
                    dtIg[tind, dind] = gtIg[m]
                    dtm[tind, dind] = gt[m]['id']
                    gtm[tind, m] = d['id']
        # set unmatched detections outside of area range to ignore
        a = np.array([d['area'] < aRng[0] or d['area'] > aRng[1] for d in dt]).reshape((1, len(dt)))
        dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
        return {
            'image_id': imgId, 'category_id': catId, 'aRng': aRng, 'maxDet': maxDet,
            'dtIds': [d['id'] for d in dt], 'gtIds': [g['id'] for g in gt],
            'dtMatches': dtm, 'gtMatches': gtm, 'dtScores': [d['score'] for d in dt],
            'gtIgnore': gtIg, 'dtIgnore': dtIg,
        }

    def accumulate(self):
        """cocoeval.py: COCOeval.accumulate."""
        p = self.params
        T = len(p.iouThrs)
        R = len(p.recThrs)
        K = len(p.catIds)
        A = len(p.areaRng)
        M = len(p.maxDets)
        precision = -np.ones((T, R, K, A, M))  # -1 for the precision of absent categories
        recall = -np.ones((T, K, A, M))
        scores = -np.ones((T, R, K, A, M))
        _pe = self._paramsEval
        setK = set(_pe.catIds)
        setA = set(map(tuple, _pe.areaRng))
        setM = set(_pe.maxDets)
        setI = set(_pe.imgIds)
        k_list = [n for n, k in enumerate(p.catIds) if k in setK]
        m_list = [m for n, m in enumerate(p.maxDets) if m in setM]
        a_list = [n for n, a in enumerate(map(lambda x: tuple(x), p.areaRng)) if a in setA]
        i_list = [n for n, i in enumerate(p.imgIds) if i in setI]
        I0 = len(_pe.imgIds)
        A0 = len(_pe.areaRng)
        for k, k0 in enumerate(k_list):
            Nk = k0 * A0 * I0
            for a, a0 in enumerate(a_list):
                Na = a0 * I0
                for m, maxDet in enumerate(m_list):
                    E = [self.evalImgs[Nk + Na + i] for i in i_list]
                    E = [e for e in E if e is not None]
                    if len(E) == 0:
                        continue
                    dtScores = np.concatenate([e['dtScores'][0:maxDet] for e in E])
                    inds = np.argsort(-dtScores, kind='mergesort')
                    dtScoresSorted = dtScores[inds]
                    dtm = np.concatenate([e['dtMatches'][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    dtIg = np.concatenate([e['dtIgnore'][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    gtIg = np.concatenate([e['gtIgnore'] for e in E])
                    npig = np.count_nonzero(gtIg == 0)
                    if npig == 0:
                        continue
                    tps = np.logical_and(dtm, np.logical_not(dtIg))
                    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                    tp_sum = np.cumsum(tps, axis=1).astype(dtype=np.float64)
                    fp_sum = np.cumsum(fps, axis=1).astype(dtype=np.float64)
                    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                        tp = np.array(tp)
                        fp = np.array(fp)
                        nd = len(tp)
                        rc = tp / npig
                        pr = tp / (fp + tp + np.spacing(1))
                        q = np.zeros((R,))
                        ss = np.zeros((R,))
                        if nd:
                            recall[t, k, a, m] = rc[-1]
                        else:
                            recall[t, k, a, m] = 0
                        pr = pr.tolist()
                        q = q.tolist()
                        for i in range(nd - 1, 0, -1):
                            if pr[i] > pr[i - 1]:
                                pr[i - 1] = pr[i]
                        inds = np.searchsorted(rc, p.recThrs, side='left')
                        try:
                            for ri, pi in enumerate(inds):
                                q[ri] = pr[pi]
                                ss[ri] = dtScoresSorted[pi]
                        except IndexError:
                            pass
                        precision[t, :, k, a, m] = np.array(q)
                        scores[t, :, k, a, m] = np.array(ss)
        self.eval = {'params': p, 'counts': [T, R, K, A, M], 'precision': precision, 'recall': recall, 'scores': scores}

    def summarize(self):
        """cocoeval.py: COCOeval.summarize -> _summarizeKps.  pycocotools hard-codes maxDets=20 there; this uses
        maxDets[-1], which is the same number at the default."""
        self.stats, self.summary_lines = summarize_kps(self.params, self.eval['precision'], self.eval['recall'])
        return self.stats

    def run(self):
        self.evaluate()
        self.accumulate()
        self.summarize()
        return self

    # ---- what the device writes besides the accumulate arrays (test hooks) --------------------------------
    def oks_matrix(self, img_id):
        """computeOks of one image: [min(D, maxDet), G] in score order x dataset gt order (empty: [])."""
        return self.ious[img_id, 1]

    def codes(self):
        """u8 [A][T][I][maxDet]: ABSENT / TP / FP / IGNORED per (area, threshold, image, score rank)."""
        p = self.params
        T, A, I, md = len(p.iouThrs), len(p.areaRng), len(p.imgIds), p.maxDets[-1]
        out = np.zeros((A, T, I, md), np.uint8)
        for a in range(A):
            for i in range(I):
                e = self.evalImgs[a * I + i]
                if e is None:
                    continue
                for r in range(len(e['dtIds'])):
                    for t in range(T):
                        matched = e['dtMatches'][t, r] != 0
                        out[a, t, i, r] = IGNORED if e['dtIgnore'][t, r] else (TP if matched else FP)
        return out

    def npig(self):
        """Number of non-ignored gts per area range (accumulate's npig)."""
        p = self.params
        I = len(p.imgIds)
        return np.array([sum(int(np.count_nonzero(e['gtIgnore'] == 0))
                             for e in self.evalImgs[a * I:(a + 1) * I] if e is not None)
                         for a in range(len(p.areaRng))], np.int64)

    def oks_margin(self):
        """The smallest distance of an OKS value to a decision it feeds: to every min(t, 1-1e-10), and between two
        distinct values of one detection's row that could both hold a match (>= the lowest threshold).  Beyond a
        few ulp the device takes every decision the same way (its exp differs from NumPy's in the last bits)."""
        bars = np.minimum(self.params.iouThrs, 1 - 1e-10)
        margin = np.inf
        for m in self.ious.values():
            if len(m) == 0:
                continue
            m = np.asarray(m)
            margin = min(margin, float(np.min(np.abs(m[..., None] - bars))))
            for row in m:
                v = np.unique(row[row >= bars[0] - 1e-6])
                if len(v) > 1:
                    margin = min(margin, float(np.min(np.diff(v))))
        return margin


def summarize_kps(p, precision, recall):
    """cocoeval.py: COCOeval.summarize._summarize / _summarizeKps on accumulate's arrays -> (stats [10], printed
    lines).  The host half of the device path runs this same function."""
    lines = []

    def _summarize(ap=1, iouThr=None, areaRng='all', maxDets=100):
        iStr = ' {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}'
        titleStr = 'Average Precision' if ap == 1 else 'Average Recall'
        typeStr = '(AP)' if ap == 1 else '(AR)'
        iouStr = '{:0.2f}:{:0.2f}'.format(p.iouThrs[0], p.iouThrs[-1]) \
            if iouThr is None else '{:0.2f}'.format(iouThr)
        aind = [i for i, aRng in enumerate(p.areaRngLbl) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(p.maxDets) if mDet == maxDets]
        if ap == 1:
            # dimension of precision: [TxRxKxAxM]
            s = precision
            # IoU
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            # dimension of recall: [TxKxAxM]
            s = recall
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, aind, mind]
        if len(s[s > -1]) == 0:
            mean_s = -1
        else:
            mean_s = np.mean(s[s > -1])
        lines.append(iStr.format(titleStr, typeStr, iouStr, areaRng, maxDets, mean_s))
        return mean_s

    md = p.maxDets[-1]
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
