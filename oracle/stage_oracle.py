"""TEST INFRASTRUCTURE ONLY -- the aggregation of heads with 1 to 4 heatmap stages, restated twice.

``aggregate`` composes the C++ oracle's primitives (oracle/libhpd_oracle.so: torch-CPU bilinear resize, the tag map)
with float32 NumPy element-wise arithmetic; ``aggregate_torch`` replays the reference's torch calls (model.py:85-96,
results.py:46-54,225-230), whose stage handling is written for a list of stages:

  1. flip average per stage:  P_i = (hm_i + flipW(hm_f_i)[:, FLIP]) / 2            (model.py:85-96)
  2. resize to the last stage: U_i = interp(P_i, size of P_{n-1}), U_{n-1} = P_{n-1} (match_heatmaps_size)
  3. stage mean:               A = ((U_0 + U_1) + ...) / n, float32, true division   (torch.stack(...).mean(0))
  4. interp(A, (H, W)), then the mean over test scales; tags from scales[tag_scale].

For two stages both equal oracle.cpu_oracle.aggregate / oracle.py_port.aggregate / oracle.ref_runner.aggregate_torch
bit for bit (tests/test_stages_cpu.py).  A scale is {"hm": [stages], "tag"[, "hm_f": [stages], "tag_f"]} or the
two-stage {"hm_lo", "hm_hi", "tag"[, "hm_lo_f", "hm_hi_f", "tag_f"]}, each map a [K,h,w] float32 array of one image.
The product package (hpdecode) never imports this module.
"""
import ctypes

import numpy as np
import torch
import torch.nn.functional as F

from . import cpu_oracle

COCO_FLIP_INDEX = cpu_oracle.COCO_FLIP_INDEX


def stages(s):
    """(heatmap stages, flipped-run stages or None) of one scale dict in either format."""
    if "hm" in s:
        return list(s["hm"]), (list(s["hm_f"]) if s.get("hm_f") else None)
    return [s["hm_lo"], s["hm_hi"]], ([s["hm_lo_f"], s["hm_hi_f"]] if s.get("hm_lo_f") is not None else None)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def aggregate(scales, out_hw, tag_scale: int = 0, flip_index=None):
    """Network outputs of one image -> (agg_hm [K,H,W], tags [K,H,W,E]), float32 arrays."""
    H, W = out_hw
    per_scale = []
    for s in scales:
        hms, hms_f = stages(s)
        hms = [_f32(m) for m in hms]
        K, n = hms[0].shape[0], len(hms)
        fi = list(flip_index) if flip_index is not None else [COCO_FLIP_INDEX[k] if k < 17 else k for k in range(K)]
        if hms_f is not None:     # (a + flipW(b)[FLIP]) * 0.5, each operation rounded to float32
            hms = [(h + _f32(f)[fi][..., ::-1]) * np.float32(0.5) for h, f in zip(hms, hms_f)]
        hh, hw = hms[-1].shape[1:]
        if n == 1:
            mean = hms[0]
        else:
            acc = cpu_oracle.resize_bilinear(hms[0], hh, hw)
            for m in hms[1:-1]:
                acc = acc + cpu_oracle.resize_bilinear(m, hh, hw)
            mean = (acc + hms[-1]) / np.float32(n)
        per_scale.append(cpu_oracle.resize_bilinear(mean, H, W))
    agg = per_scale[0]
    if len(per_scale) > 1:        # torch.stack(per_scale).mean(0): sequential sum, true division
        for m in per_scale[1:]:
            agg = agg + m
        agg = agg / np.float32(len(per_scale))
    ts = scales[tag_scale]
    tag = _f32(ts["tag"])
    tagf = _f32(ts["tag_f"]) if ts.get("tag_f") is not None else None
    E = 2 if tagf is not None else 1
    tags = np.empty((tag.shape[0], H, W, E), np.float32)
    fi_c = None if flip_index is None else np.ascontiguousarray(flip_index, np.int32)
    cpu_oracle.lib().hpo_aggregate_tags(cpu_oracle._p(tag), cpu_oracle._p(tagf), cpu_oracle._p(fi_c, ctypes.c_int),
                                        tag.shape[0], tag.shape[1], tag.shape[2], H, W, cpu_oracle._p(tags))
    return _f32(agg), tags


def _interp(x, h, w):
    return F.interpolate(x, size=[h, w], mode="bilinear", align_corners=False)


def aggregate_torch(scales, out_hw, tag_scale=0):
    """The same with the reference's torch CPU calls; returns torch tensors (hm [K,H,W], tags [K,H,W,E])."""
    H, W = out_hw
    per_scale, tags_list = [], None
    T = lambda v: torch.from_numpy(np.ascontiguousarray(v))[None]
    for si, s in enumerate(scales):
        hm_list, fl_list = stages(s)
        hms = [T(v) for v in hm_list]
        tags = [T(s["tag"])]
        if fl_list is not None:
            hms = [(h + torch.flip(T(f), [3])[:, COCO_FLIP_INDEX]) / 2 for h, f in zip(hms, fl_list)]
            tags.append(torch.flip(T(s["tag_f"]), [3])[:, COCO_FLIP_INDEX])
        h, w = hms[-1].shape[-2:]
        hms = [_interp(x, h, w) for x in hms[:-1]] + [hms[-1]]     # match_heatmaps_size
        per_scale.append(_interp(torch.stack(hms).mean(dim=0), H, W))
        if si == tag_scale:
            tags_list = tags
    hm = per_scale[0] if len(per_scale) == 1 else torch.stack(per_scale).mean(dim=0)
    tg = torch.stack([_interp(t, H, W) for t in tags_list], dim=4)
    return hm[0], tg[0]
