"""NumPy statement of the pose renderer (hpd_render_poses, include/hpdecode.h): every drawn person's limbs and joints
painted into a copy of the frame.

Test infrastructure only; the product never imports it.  Every step is one float64 NumPy operation (correctly
rounded, no FMA) in the kernel's order, so the kernel's pixels are compared byte for byte.  Each primitive is
evaluated over its bounding box, widened by one pixel and clamped to the frame; pixels outside it are not covered.

- Persons drawn: none when the record's flags bit 0 (the empty-scene fallback) is set, else p < clamp(n_person, 0, M)
  in ascending p.
- Joint k of person p is at coords[p][k] when coords are given, else at the COCO-section (x, y); it is visible when
  float(poses[p][k][2]) > kpt_thr and both coordinates are finite with |x|, |y| <= 2^20.
- Pixel (c, r) is the point X = c, Y = r.  Disc of radius R at (jx, jy): (X-jx)*(X-jx) + (Y-jy)*(Y-jy) <= R*R.
  Limb (a, b) with h = thickness / 2: ex = bx-ax, ey = by-ay, L2 = ex*ex + ey*ey, px = X-ax, py = Y-ay,
  t = px*ex + py*ey; t <= 0: px*px + py*py <= h*h; t >= L2: (X-bx)*(X-bx) + (Y-by)*(Y-by) <= h*h; else
  cr = px*ey - py*ex and cr*cr <= (h*h)*L2.
- Per person: limbs in list order (both joints visible, thickness > 0), then joints 0..K-1 (visible, radius > 0).
  A later primitive paints over an earlier one.  Limb colour: limb_colors[l] without ids; with ids,
  track_colors[id % len(track_colors)] for id >= 0 and untracked_color for id < 0.  Joints: joint_color.

``style`` is any object with the attributes of hpdecode.PoseStyle: limbs, limb_colors, joint_color, track_colors,
untracked_color, thickness, joint_radius, kpt_thr.
"""
import math

import numpy as np

from oracle.track_oracle import record_layout

MAX_COORD = 2.0 ** 20


def persons(record, K, M, E):
    """(n drawn, COCO-section xy float64 [M,K,2], joint scores float32 [M,K]) of one record."""
    row, oc, op, osc, on, of = record_layout(K, M, E)
    raw = np.ascontiguousarray(record, np.uint8)[:row]
    n = min(max(int(raw[on:on + 4].view(np.int32)[0]), 0), M)
    if int(raw[of:of + 4].view(np.int32)[0]) & 1:
        n = 0
    coco = raw[oc:op].view(np.float64).reshape(M, 3 * K + 1)[:, :3 * K].reshape(M, K, 3)
    poses = raw[op:osc].view(np.float32).reshape(M, K, 3 + E)
    return n, coco[..., :2], poses[..., 2]


def visible(x, y, score, kpt_thr):
    return float(score) > kpt_thr and abs(x) <= MAX_COORD and abs(y) <= MAX_COORD     # False for NaN and inf


def _box(lo_x, hi_x, lo_y, hi_y, margin, h, w):
    """Pixel ranges (ys, xs) of [lo - margin, hi + margin] clamped to the frame, or None when empty."""
    x0, x1 = max(math.floor(lo_x - margin), 0), min(math.ceil(hi_x + margin), w - 1)
    y0, y1 = max(math.floor(lo_y - margin), 0), min(math.ceil(hi_y + margin), h - 1)
    if x0 > x1 or y0 > y1:
        return None
    return (slice(y0, y1 + 1), slice(x0, x1 + 1),
            np.arange(y0, y1 + 1, dtype=np.float64)[:, None], np.arange(x0, x1 + 1, dtype=np.float64)[None, :])


def disc_mask(X, Y, jx, jy, R):
    return (X - jx) * (X - jx) + (Y - jy) * (Y - jy) <= R * R


def limb_mask(X, Y, ax, ay, bx, by, h):
    hh = h * h
    ex, ey = bx - ax, by - ay
    L2 = ex * ex + ey * ey
    px, py = X - ax, Y - ay
    t = px * ex + py * ey
    cr = px * ey - py * ex
    return np.where(t <= 0, px * px + py * py <= hh,
                    np.where(t >= L2, (X - bx) * (X - bx) + (Y - by) * (Y - by) <= hh, cr * cr <= hh * L2))


def render(frame, record, K, M, E, style, ids=None, coords=None):
    """frame uint8 [h,w,3] (left unchanged), one record (uint8 [row_bytes]), optional ids int32 [M] and coords
    float64 [M,K,2] -> a new uint8 [h,w,3]."""
    out = np.array(frame, np.uint8, copy=True)
    h, w = out.shape[:2]
    n, xy, score = persons(record, K, M, E)
    if coords is not None:
        xy = np.asarray(coords, np.float64)
    half, R = float(style.thickness) / 2, float(style.joint_radius)
    tc = style.track_colors
    for p in range(n):
        pts = [(float(xy[p, k, 0]), float(xy[p, k, 1])) for k in range(K)]
        vis = [visible(x, y, score[p, k], float(style.kpt_thr)) for k, (x, y) in enumerate(pts)]
        if ids is not None:
            col = tc[int(ids[p]) % len(tc)] if int(ids[p]) >= 0 else style.untracked_color
        if half > 0:
            for l, (a, b) in enumerate(style.limbs):
                if not (vis[a] and vis[b]):
                    continue
                (ax, ay), (bx, by) = pts[a], pts[b]
                box = _box(min(ax, bx), max(ax, bx), min(ay, by), max(ay, by), half + 1, h, w)
                if box is not None:
                    ys, xs, Y, X = box
                    out[ys, xs][limb_mask(X, Y, ax, ay, bx, by, half)] = col if ids is not None else style.limb_colors[l]
        if R > 0:
            for k, (x, y) in enumerate(pts):
                if vis[k]:
                    box = _box(x, x, y, y, R + 1, h, w)
                    if box is not None:
                        ys, xs, Y, X = box
                        out[ys, xs][disc_mask(X, Y, x, y, R)] = style.joint_color
    return out
