"""TEST / BASELINE INFRASTRUCTURE ONLY -- Python port of the reference decode (torch CPU + NumPy).

The reference is pure Python and cannot travel to the GPU box, so this module is what
``bench.py --impl reference`` and the ``cpu_baseline`` leg time: the same library calls the
reference makes (F.interpolate, max_pool2d, topk, gather on the CPU; NumPy means / norms / full-map
passes; the pure-Python Hungarian solver of oracle/refshim/munkres.py), so its cost structure is
the reference's.  The bookkeeping is restated with flat arrays instead of the reference's dicts.
Pinned bit-exactly against the unmodified reference (tests/test_oracle_reference.py, build
container only) and against the C++ oracle (tests/test_oracle.py).

Reference lines followed (relative to /root/reference): model.py:85-96, results.py:46-67,225-234,
grouping.py:55-59,80-283.  Never imported by the product package.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
if os.path.join(_HERE, "refshim") not in sys.path:
    sys.path.insert(0, os.path.join(_HERE, "refshim"))
from munkres import Munkres  # noqa: E402  (restated stand-in, see its header)

COCO_FLIP_INDEX = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15]
JOINTS_ORDER = [0, 1, 2, 3, 4, 5, 6, 11, 12, 7, 8, 9, 10, 13, 14, 15, 16]


def _up(x, h, w):
    return F.interpolate(x, size=[h, w], mode="bilinear", align_corners=False)


def aggregate(scales, out_hw, tag_scale=0):
    """One image: list of per-scale dicts of [K,h,w] arrays -> (hm [K,H,W], tags [K,H,W,E]) tensors."""
    H, W = out_hw
    fulls, tag_maps = [], None
    for si, s in enumerate(scales):
        t = {k: torch.from_numpy(np.ascontiguousarray(v))[None] for k, v in s.items() if v is not None}
        lo, hi, tags = t["hm_lo"], t["hm_hi"], [t["tag"]]
        if "hm_lo_f" in t:
            lo = (lo + torch.flip(t["hm_lo_f"], [3])[:, COCO_FLIP_INDEX]) / 2
            hi = (hi + torch.flip(t["hm_hi_f"], [3])[:, COCO_FLIP_INDEX]) / 2
            tags.append(torch.flip(t["tag_f"], [3])[:, COCO_FLIP_INDEX])
        stage_mean = torch.stack([_up(lo, hi.shape[2], hi.shape[3]), hi]).mean(dim=0)
        fulls.append(_up(stage_mean, H, W))
        if si == tag_scale:
            tag_maps = tags
    hm = fulls[0] if len(fulls) == 1 else torch.stack(fulls).mean(dim=0)
    tg = torch.stack([_up(x, H, W) for x in tag_maps], dim=4)
    return hm[0], tg[0]


def nms(hm):
    pooled = F.max_pool2d(hm, 5, 1, 2)
    return hm * torch.eq(pooled, hm).float()


def top_k(hm, tags, M):
    K, H, W = hm.shape
    flat = nms(hm[None])[0].view(K, -1)
    scores, idx = flat.topk(M, dim=1)
    tflat = tags.view(K, H * W, -1)
    tags_k = torch.stack([torch.gather(tflat[..., e], 1, idx) for e in range(tflat.size(2))], dim=2)
    coords = torch.stack((idx % W, (idx / W).long()), dim=2)
    return tags_k.numpy(), coords.numpy().astype(np.int32), scores.numpy(), idx.numpy().astype(np.int32)


def match_by_tag(tags_k, coords_k, scores_k, M, det_thr, tag_thr, joints_order=None, trace=None):
    """``joints_order`` replaces grouping.py:63-65's order; ``trace`` (a list) receives one dict per joint step with
    detections: the selection mask, the person keys and tag lists before the step, the distances and the solver's
    pairs (tests count the branches their scenes reach from it)."""
    K, _, E = tags_k.shape
    keys = []          # float32 key per person, insertion order
    rows = []          # [K, 3+E] float64 per person
    tag_lists = []     # list of float32 tag vectors per person

    def seed(k, joint, tag):
        for p, key in enumerate(keys):
            if key == tag[0]:
                rows[p][k] = joint
                tag_lists[p] = [tag]
                return
        keys.append(tag[0])
        r = np.zeros((K, 3 + E))
        r[k] = joint
        rows.append(r)
        tag_lists.append([tag])

    for it in range(K):
        k = joints_order[it] if joints_order is not None else (JOINTS_ORDER[it] if K == 17 else it)
        tags = tags_k[k]
        joints = np.concatenate((coords_k[k], scores_k[k, :, None], tags), 1)
        sel = joints[:, 2] > det_thr
        tags, joints = tags[sel], joints[sel]
        if joints.shape[0] == 0:
            continue
        step = None if trace is None else dict(k=k, sel=sel, tags=tags, keys=list(keys),
                                               tag_lists=[list(t) for t in tag_lists[:M]], dist=None, pairs=[])
        if step is not None:
            trace.append(step)
        if it == 0 or not keys:
            for tag, joint in zip(tags, joints):
                seed(k, joint, tag)
            continue
        G = min(len(keys), M)
        means = np.array([np.mean(tag_lists[p], axis=0) for p in range(G)])
        dist = np.linalg.norm(joints[:, None, 3:] - means[None, :, :], ord=2, axis=2)
        saved = np.copy(dist)
        cost = np.round(dist) * 100 - joints[:, 2:3]
        n_new = joints.shape[0]
        if n_new > G:
            cost = np.concatenate((cost, np.zeros((n_new, n_new - G)) + 1e10), axis=1)
        pairs = Munkres().compute(cost)
        if step is not None:
            step.update(dist=saved, pairs=pairs)
        for r, c in pairs:
            if r < n_new and c < G and saved[r][c] < tag_thr:
                rows[c][k] = joints[r]
                tag_lists[c].append(tags[r])
            else:
                seed(k, joints[r], tags[r])
    if not rows:
        return np.zeros((0,), np.float32)
    return np.array(rows).astype(np.float32)[:M]


def _quarter(hm_k, x, y, fx, fy):
    H, W = hm_k.shape
    fx += 0.25 if hm_k[y, min(x + 1, W - 1)] > hm_k[y, max(x - 1, 0)] else -0.25
    fy += 0.25 if hm_k[min(y + 1, H - 1), x] > hm_k[max(y - 1, 0), x] else -0.25
    return fx, fy


def adjust(grouped, hm):
    for p in range(grouped.shape[0]):
        for k in range(grouped.shape[1]):
            if grouped[p, k, 2] == 0:
                continue
            fx, fy = grouped[p, k, 0], grouped[p, k, 1]
            fx, fy = _quarter(hm[k], int(fx), int(fy), fx, fy)
            grouped[p, k, :2] = (fx + 0.5, fy + 0.5)
    return grouped


def refine(hm, tags, person):
    K, H, W = hm.shape
    have = [tags[k, int(person[k, 1]), int(person[k, 0])] for k in range(K) if person[k, 2] > 0]
    mean_tag = np.mean(have, axis=0)[None, None, :]
    cand = []
    for k in range(K):
        d = ((tags[k] - mean_tag) ** 2).sum(axis=2) ** 0.5
        y, x = np.unravel_index(np.argmax(hm[k] - np.round(d)), (H, W))
        val = hm[k, y, x]
        fx, fy = _quarter(hm[k], x, y, x + 0.5, y + 0.5)
        cand.append((fx, fy, val))
    cand = np.array(cand)
    repl = np.bitwise_and(cand[:, 2] > 0, person[:, 2] == 0)
    person[repl, :3] = cand[repl]
    return person


def parse(hm, tags, M=30, det_thr=0.05, tag_thr=0.5, do_adjust=True, do_refine=True):
    """hm [K,H,W], tags [K,H,W,E] torch CPU tensors -> (grouped_joints, person_scores)."""
    tags_k, coords_k, scores_k, _ = top_k(hm, tags, M)
    grouped = match_by_tag(tags_k, coords_k, scores_k, M, det_thr, tag_thr)
    if len(grouped) == 0:
        g = np.concatenate([coords_k[:, 0], scores_k[:, 0, None], tags_k[:, 0]], axis=-1)[None]
        grouped = np.nan_to_num(g, nan=0)
        grouped[..., 2] = 0.01
    hm_np, tags_np = hm.numpy(), tags.numpy()
    if do_adjust:
        grouped = adjust(grouped, hm_np)
    scores = grouped[..., 2].mean(1)
    if do_refine:
        for p in range(len(grouped)):
            grouped[p] = refine(hm_np, tags_np, grouped[p])
    return grouped, scores


def decode_image(scales, out_hw, M=30, det_thr=0.05, tag_thr=0.5, tag_scale=0):
    """Whole path for one image (what bench.py --impl reference times)."""
    hm, tags = aggregate(scales, out_hw, tag_scale)
    return parse(hm, tags, M, det_thr, tag_thr)
