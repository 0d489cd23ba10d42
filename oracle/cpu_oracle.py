"""TEST INFRASTRUCTURE ONLY -- ctypes front-end of oracle/libhpd_oracle.so.

Allowed importers: tests/, __graft_entry__.smoke(), bench.py (cpu_baseline and
--impl reference legs).  The product package (hpdecode) must never import this.

Every function takes/returns contiguous numpy arrays; see hpd_oracle.cpp for the
reference file:line each one follows.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libhpd_oracle.so")
_lib = None

COCO_FLIP_INDEX = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15]  # transforms.py:11
JOINTS_ORDER = [0, 1, 2, 3, 4, 5, 6, 11, 12, 7, 8, 9, 10, 13, 14, 15, 16]      # grouping.py:63-65


def build(force: bool = False) -> str:
    """Compile the oracle with oracle/Makefile (g++).  Building the checker is not using it."""
    src = os.path.join(_HERE, "hpd_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libhpd_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.hpo_abi_version.restype = ctypes.c_int
    return _lib


def _p(a, ct=ctypes.c_float):
    if a is None:
        return None
    return a.ctypes.data_as(ctypes.POINTER(ct))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def resize_bilinear(x: np.ndarray, oh: int, ow: int) -> np.ndarray:
    """F.interpolate(x, size=[oh, ow], mode='bilinear', align_corners=False) on [..., h, w]."""
    x = _f32(x)
    ih, iw = x.shape[-2:]
    planes = int(np.prod(x.shape[:-2], dtype=np.int64))
    out = np.empty(x.shape[:-2] + (oh, ow), np.float32)
    lib().hpo_resize_bilinear(_p(x), planes, ih, iw, _p(out), oh, ow)
    return out


def aggregate(scales, out_hw, tag_scale: int = 0, flip_index=None):
    """Network outputs of one image -> (agg_hm [K,H,W], tags [K,H,W,E]).

    scales: list of dicts with keys hm_lo, hm_hi, tag and (flip test) hm_lo_f, hm_hi_f, tag_f,
            each a [K,h,w] float32 array (raw outputs of the un-flipped / flipped forward).
    Restates model.py:85-96 + results.py:225-230; for len(scales) > 1 the per-scale full-res
    heatmaps are averaged (torch.stack(...).mean(0)) and tags come from scales[tag_scale].
    """
    H, W = out_hw
    L = lib()
    fi = None if flip_index is None else np.ascontiguousarray(flip_index, np.int32)
    per_scale = []
    for s in scales:
        lo, hi = _f32(s["hm_lo"]), _f32(s["hm_hi"])
        K = lo.shape[0]
        lof = _f32(s["hm_lo_f"]) if s.get("hm_lo_f") is not None else None
        hif = _f32(s["hm_hi_f"]) if s.get("hm_hi_f") is not None else None
        out = np.empty((K, H, W), np.float32)
        L.hpo_aggregate_heatmaps_scale(_p(lo), _p(hi), _p(lof), _p(hif), _p(fi, ctypes.c_int), K,
                                       lo.shape[1], lo.shape[2], hi.shape[1], hi.shape[2], H, W, _p(out))
        per_scale.append(out)
    if len(per_scale) == 1:
        agg = per_scale[0]
    else:
        agg = np.empty_like(per_scale[0])
        arr = (ctypes.POINTER(ctypes.c_float) * len(per_scale))(*[_p(m) for m in per_scale])
        L.hpo_scale_mean(arr, len(per_scale), ctypes.c_size_t(agg.size), _p(agg))
    ts = scales[tag_scale]
    tag = _f32(ts["tag"])
    tagf = _f32(ts["tag_f"]) if ts.get("tag_f") is not None else None
    E = 2 if tagf is not None else 1
    tags = np.empty((tag.shape[0], H, W, E), np.float32)
    L.hpo_aggregate_tags(_p(tag), _p(tagf), _p(fi, ctypes.c_int), tag.shape[0], tag.shape[1], tag.shape[2],
                         H, W, _p(tags))
    return agg, tags


def nms(hm: np.ndarray):
    """grouping.py:80-83 on [..., H, W]; returns (nms'd map, keep mask uint8)."""
    hm = _f32(hm)
    H, W = hm.shape[-2:]
    planes = int(np.prod(hm.shape[:-2], dtype=np.int64))
    out = np.empty_like(hm)
    keep = np.empty(hm.shape, np.uint8)
    lib().hpo_nms(_p(hm), planes, H, W, _p(out), _p(keep, ctypes.c_uint8))
    return out, keep


def top_k(nms_hm: np.ndarray, tags: np.ndarray, M: int):
    """grouping.py:150-170 given the NMS'd map [K,H,W] and tags [K,H,W,E]."""
    nms_hm, tags = _f32(nms_hm), _f32(tags)
    K, H, W = nms_hm.shape
    E = tags.shape[3]
    tags_k = np.empty((K, M, E), np.float32)
    coords_k = np.empty((K, M, 2), np.int32)
    scores_k = np.empty((K, M), np.float32)
    idx_k = np.empty((K, M), np.int32)
    rc = lib().hpo_topk(_p(nms_hm), _p(tags), K, H, W, E, M, _p(tags_k), _p(coords_k, ctypes.c_int32),
                        _p(scores_k), _p(idx_k, ctypes.c_int32))
    if rc:
        raise ValueError("oracle top_k needs H*W >= 64*M (torch partial_sort regime)")
    return tags_k, coords_k, scores_k, idx_k


def munkres(cost: np.ndarray) -> np.ndarray:
    cost = np.ascontiguousarray(cost, np.float64)
    r, c = cost.shape
    out = np.empty(r, np.int32)
    rc = lib().hpo_munkres(_p(cost, ctypes.c_double), r, c, _p(out, ctypes.c_int32))
    if rc:
        raise ValueError("oracle munkres needs rows <= cols <= 32")
    return out


def match_by_tag(tags_k, coords_k, scores_k, det_thr: float, tag_thr: float, M: int = None):
    tags_k, scores_k = _f32(tags_k), _f32(scores_k)
    coords_k = np.ascontiguousarray(coords_k, np.int32)
    K, Mk, E = tags_k.shape
    M = Mk if M is None else M
    assert M == Mk
    poses = np.empty((M, K, 3 + E), np.float32)
    n = ctypes.c_int32(0)
    nt = ctypes.c_int32(0)
    rc = lib().hpo_match_by_tag(_p(tags_k), _p(coords_k, ctypes.c_int32), _p(scores_k), K, M, E,
                                ctypes.c_double(det_thr), ctypes.c_double(tag_thr), None, _p(poses),
                                ctypes.byref(n), ctypes.byref(nt), None)
    if rc:
        raise ValueError("oracle match_by_tag limits exceeded")
    return poses[: n.value].copy(), nt.value


def parse(hm: np.ndarray, tags: np.ndarray, M: int = 30, det_thr: float = 0.1, tag_thr: float = 1.0,
          adjust: bool = True, refine: bool = True):
    """grouping.py:252-283 on one image's aggregated maps.  Returns a dict."""
    hm, tags = _f32(hm), _f32(tags)
    K, H, W = hm.shape
    if tags.ndim == 3:
        tags = tags[..., None]
    E = tags.shape[3]
    poses = np.zeros((M, K, 3 + E), np.float32)
    scores = np.zeros((M,), np.float32)
    n = ctypes.c_int32(0)
    fb = ctypes.c_int32(0)
    tags_k = np.empty((K, M, E), np.float32)
    coords_k = np.empty((K, M, 2), np.int32)
    scores_k = np.empty((K, M), np.float32)
    idx_k = np.empty((K, M), np.int32)
    rc = lib().hpo_parse(_p(hm), _p(tags), K, H, W, E, M, ctypes.c_double(det_thr), ctypes.c_double(tag_thr),
                         int(adjust), int(refine), _p(poses), _p(scores), ctypes.byref(n), ctypes.byref(fb),
                         _p(tags_k), _p(coords_k, ctypes.c_int32), _p(scores_k), _p(idx_k, ctypes.c_int32))
    if rc:
        raise ValueError("oracle parse: unsupported shape (need H*W >= 64*M, K,M <= 32, E <= 2)")
    P = n.value
    return dict(grouped_joints=poses[:P].copy(), person_scores=scores[:P].copy(), fallback=bool(fb.value),
                tags_k=tags_k, coords_k=coords_k, scores_k=scores_k, idx_k=idx_k)
