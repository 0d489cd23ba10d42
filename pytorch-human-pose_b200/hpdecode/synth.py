"""Seeded synthetic network outputs for tests, smoke() and bench.py.

There is no dataset and no checkpoint offline, so workloads are synthetic.  Everything here
is built from a counter-based integer hash and IEEE float32 element-wise adds/multiplies only
(no transcendental library calls on arrays), so a given seed produces bit-identical tensors in
the build container and on the GPU box -- goldens recorded from the reference on these tensors
(tests/golden/) stay valid everywhere.

Two families, both at NETWORK-OUTPUT resolution so the whole decode path runs
(SURVEY.md 8(d)):
  * ``netlike``  -- smooth random fields with the value ranges seen from a default-init
    HigherHRNet (hm_lo ~ [-0.45, 0.62], hm_hi ~ [-0.25, 0.23], tags ~ [-0.45, 0.51]), some
    channels entirely negative (exercises the +-0 tail of top-k).
  * ``crowd``    -- planted persons x 17 joints: Gaussian-like peaks with distinct amplitudes,
    a constant tag per person inside a disc, small additive noise (the grouping-bound case,
    BASELINE config 4); ``quantised=True`` rounds amplitudes/tags to provoke exact ties.
Each generator returns a list (one entry per test scale) of dicts
``{hm_lo, hm_hi, tag[, hm_lo_f, hm_hi_f, tag_f]}`` of float32 arrays shaped [B, K, h, w]; the
``*_f`` entries are what the network would output for the horizontally flipped image.
"""
import math

import numpy as np

COCO_FLIP_INDEX = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15]


def hash_u32(n: int, seed: int) -> np.ndarray:
    """lowbias32-style integer hash of the counters 0..n-1 (exact on every platform)."""
    x = np.arange(n, dtype=np.uint64) + np.uint64((seed * 0x9E3779B1) & 0xFFFFFFFF)
    x &= np.uint64(0xFFFFFFFF)
    for mul, sh in ((0x7FEB352D, 15), (0x846CA68B, 16)):
        x ^= x >> np.uint64(sh)
        x = (x * np.uint64(mul)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    return x.astype(np.uint32)


def uniform(shape, seed: int) -> np.ndarray:
    """U[0,1) float32 with 24 random bits per element."""
    n = int(np.prod(shape))
    return ((hash_u32(n, seed) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)).reshape(shape)


def noise(shape, seed: int) -> np.ndarray:
    """Zero-mean, unit-variance-ish (Irwin-Hall of 4 uniforms) float32 noise."""
    u = uniform((4,) + tuple(shape), seed)
    s = (u[0] + u[1]) + (u[2] + u[3])
    return (s - np.float32(2.0)) * np.float32(math.sqrt(3.0))


def _box3(a: np.ndarray) -> np.ndarray:
    """3x3 box sum with edge replication on the last two axes (plain float32 adds)."""
    p = np.concatenate([a[..., :1, :], a, a[..., -1:, :]], axis=-2)
    r = (p[..., :-2, :] + p[..., 1:-1, :]) + p[..., 2:, :]
    p = np.concatenate([r[..., :, :1], r, r[..., :, -1:]], axis=-1)
    return (p[..., :, :-2] + p[..., :, 1:-1]) + p[..., :, 2:]


def _flip_view(a: np.ndarray) -> np.ndarray:
    """What the flipped forward would output if the net were exactly flip-equivariant."""
    return np.ascontiguousarray(a[:, COCO_FLIP_INDEX][..., ::-1])


def netlike(batch: int, size: int = 512, flip: bool = True, seed: int = 0, num_kpts: int = 17,
            scales=(1.0,), negative_channels=(0, 2, 4, 10, 11)):
    out = []
    for si, sc in enumerate(scales):
        s_in = int(round(size * sc / 64.0)) * 64 if sc != 1.0 else size
        q, h = s_in // 4, s_in // 2
        d = {}
        for name, res, amp, off, sd in (("hm_lo", q, 0.075, 0.05, 1), ("hm_hi", h, 0.035, -0.01, 2), ("tag", q, 0.07, 0.02, 3)):
            base_seed = seed * 1000 + si * 100 + sd * 10
            f = _box3(noise((batch, num_kpts, res, res), base_seed)) * np.float32(amp) + np.float32(off)
            if name != "tag":
                for c in negative_channels:
                    if c < num_kpts:
                        f[:, c] = f[:, c] * np.float32(0.3) - np.float32(0.3 if name == "hm_lo" else 0.12)
            d[name] = np.ascontiguousarray(f, np.float32)
            if flip:
                g = _flip_view(f) + noise((batch, num_kpts, res, res), base_seed + 5) * np.float32(amp * 0.2)
                d[name + "_f"] = np.ascontiguousarray(g, np.float32)
        out.append(d)
    return out


def _gauss_table(sigma: float, radius: int) -> np.ndarray:
    t = np.zeros((2 * radius + 1, 2 * radius + 1), np.float32)
    for dy in range(-radius, radius + 1):
        for dx in range(-radius, radius + 1):
            t[dy + radius, dx + radius] = round(math.exp(-(dx * dx + dy * dy) / (2.0 * sigma * sigma)), 6)
    return t


def crowd(batch: int, size: int = 512, persons: int = 30, flip: bool = True, seed: int = 0, num_kpts: int = 17,
          quantised: bool = False, tag_spread: float = 2.0, missing_frac: float = 0.15, noise_amp: float = 0.02):
    """Planted persons (BASELINE config 4).  Deterministic placement from the integer hash."""
    q, h = size // 4, size // 2
    gq, gh = _gauss_table(1.0, 3), _gauss_table(2.0, 6)
    hm_lo = noise((batch, num_kpts, q, q), seed * 1000 + 1) * np.float32(noise_amp)
    hm_hi = noise((batch, num_kpts, h, h), seed * 1000 + 2) * np.float32(noise_amp)
    tag = noise((batch, num_kpts, q, q), seed * 1000 + 3) * np.float32(0.01)
    n = batch * persons * num_kpts
    ux = uniform((n,), seed * 1000 + 4).reshape(batch, persons, num_kpts)
    uy = uniform((n,), seed * 1000 + 5).reshape(batch, persons, num_kpts)
    ua = uniform((n,), seed * 1000 + 6).reshape(batch, persons, num_kpts)
    um = uniform((n,), seed * 1000 + 7).reshape(batch, persons, num_kpts)
    ut = noise((n,), seed * 1000 + 8).reshape(batch, persons, num_kpts)
    for b in range(batch):
        for p in range(persons):
            base_tag = np.float32(tag_spread * (p - persons // 2))
            if quantised:
                base_tag = np.float32(base_tag * 0.15)
            for k in range(num_kpts):
                if um[b, p, k] < missing_frac:
                    continue
                cx = 4 + int(ux[b, p, k] * (q - 8))
                cy = 4 + int(uy[b, p, k] * (q - 8))
                amp = np.float32(0.5) + np.float32(0.5) * ua[b, p, k]
                if quantised:
                    amp = np.float32(round(float(amp) * 20.0) / 20.0)
                t = base_tag + (np.float32(0.0) if quantised else np.float32(0.05) * ut[b, p, k])
                hm_lo[b, k, cy - 3:cy + 4, cx - 3:cx + 4] = np.maximum(hm_lo[b, k, cy - 3:cy + 4, cx - 3:cx + 4], gq * amp)
                y2, x2 = 2 * cy, 2 * cx
                ys, xs = max(y2 - 6, 0), max(x2 - 6, 0)
                ye, xe = min(y2 + 7, h), min(x2 + 7, h)
                sub = gh[ys - (y2 - 6):ye - (y2 - 6), xs - (x2 - 6):xe - (x2 - 6)] * amp
                hm_hi[b, k, ys:ye, xs:xe] = np.maximum(hm_hi[b, k, ys:ye, xs:xe], sub)
                tag[b, k, cy - 2:cy + 3, cx - 2:cx + 3] = t
    d = {"hm_lo": hm_lo, "hm_hi": hm_hi, "tag": tag}
    if flip:
        d["hm_lo_f"] = _flip_view(hm_lo) + noise(hm_lo.shape, seed * 1000 + 11) * np.float32(noise_amp * 0.5)
        d["hm_hi_f"] = _flip_view(hm_hi) + noise(hm_hi.shape, seed * 1000 + 12) * np.float32(noise_amp * 0.5)
        d["tag_f"] = _flip_view(tag) + noise(tag.shape, seed * 1000 + 13) * np.float32(0.005)
    return [{k: np.ascontiguousarray(v, np.float32) for k, v in d.items()}]


def image_slice(scales, b: int):
    """Per-image view ([K,h,w] arrays) of a generator's output."""
    return [{k: v[b] for k, v in s.items()} for s in scales]


class _Draws:
    """Consumes U[0,1) float64 values of one seeded hash stream (float32 resolution), block by block."""

    def __init__(self, seed: int, block: int = 1 << 16):
        self.seed, self.block, self.n = seed, block, 0
        self.buf, self.pos = np.zeros(0), 0

    def take(self, n: int) -> np.ndarray:
        if self.pos + n > len(self.buf):
            self.buf = np.concatenate([self.buf[self.pos:], uniform((max(self.block, n),), self.seed * 7919 + self.n)
                                       .astype(np.float64)])
            self.pos, self.n = 0, self.n + 1
        out = self.buf[self.pos:self.pos + n]
        self.pos += n
        return out

    def one(self) -> float:
        return float(self.take(1)[0])


def coco_eval_set(num_images: int, seed: int = 0, num_kpts: int = 17, max_gts: int = 15, dets_per_image: int = 30,
                  sigmas=None, spread: float = 1.0, crowd_frac: float = 0.05, no_kpt_frac: float = 0.05,
                  no_gt_frac: float = 0.1, no_det_frac: float = 0.05, score_levels: int = 0):
    """A seeded COCO keypoint evaluation set: (annotation dict, result list), shaped like val2017 person keypoints.

    Each image has 0..max_gts ground-truth persons (none with probability ``no_gt_frac``) spread over the three area
    bands (small < 32², medium, large > 96²), some crowd (``crowd_frac``) and some without a labelled joint
    (``no_kpt_frac``, num_keypoints == 0).  It has ``dets_per_image`` detections (none with probability
    ``no_det_frac``): most ground-truth persons get one whose joints are the ground truth's moved by up to
    ``spread`` x 3 OKS standard deviations (so OKS values cover the whole range), some a second, lower-scored one,
    and the rest are false positives.  ``score_levels`` > 0 rounds scores to that many levels: ties inside and
    across images.  The result list holds the images in a shuffled order, each image's detections together."""
    K = num_kpts
    if sigmas is not None:
        sig = np.asarray(sigmas, np.float64)
    elif K == 17:
        sig = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0
    else:
        sig = np.full(K, 0.05)
    rnd = _Draws(seed)
    images, anns, per_image = [], [], []
    image_id = 0
    for i in range(num_images):
        image_id += 1 + int(rnd.one() * 3)
        images.append({"id": image_id, "width": 640, "height": 480})
        ng = 0 if rnd.one() < no_gt_frac else int(rnd.one() * (max_gts + 1))
        gts = []
        for _ in range(ng):
            band = rnd.one()
            s = (20.0 if band < 0.3 else 60.0 if band < 0.65 else 160.0) * (0.7 + 0.6 * rnd.one())
            cx, cy = 40.0 + 560.0 * rnd.one(), 40.0 + 400.0 * rnd.one()
            u = rnd.take(3 * K)
            x = cx + (u[:K] - 0.5) * s
            y = cy + (u[K:2 * K] - 0.5) * s
            v = np.where(u[2 * K:] > 0.2, 2.0, np.where(u[2 * K:] > 0.1, 1.0, 0.0))
            if rnd.one() < no_kpt_frac:
                v[:] = 0.0
            x, y = np.where(v > 0, x, 0.0), np.where(v > 0, y, 0.0)
            bbox = [cx - 0.6 * s, cy - 0.6 * s, 1.2 * s, 1.2 * s]
            area = s * s * (0.5 + 0.4 * rnd.one())
            kp = np.stack([x, y, v], 1).ravel()
            ann = {"id": len(anns) + 1, "image_id": image_id, "category_id": 1, "keypoints": kp.tolist(),
                   "num_keypoints": int(np.count_nonzero(v > 0)), "area": area, "bbox": bbox,
                   "iscrowd": int(rnd.one() < crowd_frac)}
            anns.append(ann)
            gts.append((cx, cy, s, x, y, v, area))
        dets = []
        if rnd.one() >= no_det_frac:
            for cx, cy, s, x, y, v, area in gts:
                for copy in range(2):
                    if rnd.one() > (0.85 if copy == 0 else 0.2) or len(dets) >= dets_per_image:
                        continue
                    level = 3.0 * spread * rnd.one()
                    u = rnd.take(2 * K)
                    sd = sig * 2 * np.sqrt(area) * level
                    xd = np.where(v > 0, x, cx) + (u[:K] - 0.5) * 2 * sd
                    yd = np.where(v > 0, y, cy) + (u[K:] - 0.5) * 2 * sd
                    dets.append((xd, yd, rnd.one() * (0.5 if copy else 1.0)))
            while len(dets) < dets_per_image:
                s = 10.0 + 150.0 * rnd.one()
                cx, cy = 640.0 * rnd.one(), 480.0 * rnd.one()
                u = rnd.take(2 * K)
                dets.append((cx + (u[:K] - 0.5) * s, cy + (u[K:] - 0.5) * s, 0.6 * rnd.one()))
        order = np.argsort(rnd.take(len(dets)), kind="mergesort")
        recs = []
        for j in order:
            xd, yd, score = dets[j]
            if score_levels:
                score = round(score * score_levels) / score_levels
            kp = np.stack([xd, yd, np.ones(K)], 1).ravel()
            recs.append({"image_id": image_id, "category_id": 1, "keypoints": kp.tolist(), "score": float(score)})
        per_image.append(recs)
    results = [r for i in np.argsort(rnd.take(num_images), kind="mergesort") for r in per_image[i]]
    dataset = {"images": images, "annotations": anns, "categories": [{"id": 1, "name": "person"}]}
    return dataset, results
