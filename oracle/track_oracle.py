"""NumPy statement of the person tracker (hpd_track, include/hpdecode.h): greedy OKS matching of each frame's persons
to the tracks of earlier frames, modelled on mmpose's video-demo tracker (_track_by_oks, tracking_thr, min_keypoints).

Test infrastructure only; the product never imports it.  Everything is float64 in the kernel's operation order; the
OKS sum is np.sum (NumPy's pairwise order), its terms np.exp (within 1 ulp of CUDA's exp, so ids are compared exactly
only where no decision is closer than a margin to the threshold or to its runner-up: see ``Tracker.margins``).

- Persons of a frame: p < n_person; none when flags bit 0 (the empty-scene fallback) is set.  Joint k is at
  coco[p][3k], coco[p][3k+1] and visible when poses[p][k][2] > 0; the score is person_scores[p] (float32).
- Area: (max x - min x) * (max y - min y) over the visible joints, 0 with fewer than two.
- OKS(d, t) over J = joints visible in both (0 if none): s = (area_d + area_t) / 2,
  e = (dx**2 + dy**2) / vars / (s + np.spacing(1)) / 2, OKS = np.sum(np.exp(-e)) / |J|.
- Persons in descending score (ties: lower index) take the live, unclaimed track of highest OKS (ties: smaller id) if
  OKS > oks_thr; else a new id if >= min_keypoints joints are visible, else -1.  Tracks started in this frame are not
  candidates in it.  Unclaimed tracks age by one after the frame and are dropped at age max_age.
"""
import numpy as np

COCO_SIGMAS = np.array([.26, .25, .25, .35, .35, .79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89]) / 10.0


def record_layout(K, M, E):
    """HpdRecordLayout (common.cuh: record_layout) -> (row_bytes, off_coco, off_poses, off_person_scores, off_n_person,
    off_flags)."""
    off_coco = 0
    off_poses = off_coco + 8 * M * (3 * K + 1)
    off_scores = off_poses + 4 * M * K * (3 + E)
    off_n = off_scores + 4 * M
    off_flags = off_n + 4
    return (off_flags + 4 + 7) // 8 * 8, off_coco, off_poses, off_scores, off_n, off_flags


def frame_persons(raw, K, M, E):
    """One record (uint8 [row_bytes]) -> (xy float64 [n,K,2], vis bool [n,K], scores float32 [n])."""
    row, oc, op, osc, on, of = record_layout(K, M, E)
    raw = np.ascontiguousarray(raw, np.uint8)[:row]
    n = min(max(int(raw[on:on + 4].view(np.int32)[0]), 0), M)
    if int(raw[of:of + 4].view(np.int32)[0]) & 1:
        n = 0
    coco = raw[oc:op].view(np.float64).reshape(M, 3 * K + 1)[:n, :3 * K].reshape(n, K, 3)
    poses = raw[op:osc].view(np.float32).reshape(M, K, 3 + E)[:n]
    scores = raw[osc:on].view(np.float32)[:n]
    return coco[..., :2].copy(), poses[..., 2] > 0, scores.copy()


def area_of(xy, vis):
    if vis.sum() < 2:
        return 0.0
    x, y = xy[vis, 0], xy[vis, 1]
    return float((x.max() - x.min()) * (y.max() - y.min()))


def oks(xy_d, vis_d, area_d, xy_t, vis_t, area_t, kpt_vars):
    J = vis_d & vis_t
    if not J.any():
        return 0.0
    dx = xy_d[J, 0] - xy_t[J, 0]
    dy = xy_d[J, 1] - xy_t[J, 1]
    s = (area_d + area_t) / 2
    e = (dx ** 2 + dy ** 2) / kpt_vars[J] / (s + np.spacing(1)) / 2
    return float(np.sum(np.exp(-e)) / e.shape[0])


class Tracker:
    def __init__(self, K=17, M=30, E=2, oks_thr=0.3, max_age=1, min_keypoints=3, kpt_vars=None):
        self.K, self.M, self.E = K, M, E
        self.oks_thr, self.max_age, self.min_keypoints = float(oks_thr), int(max_age), int(min_keypoints)
        self.kpt_vars = (COCO_SIGMAS * 2) ** 2 if kpt_vars is None else np.asarray(kpt_vars, np.float64)
        self.tracks = []      # dicts: id, xy, vis, area, age -- in id order
        self.next_id = 0
        self.margins = []     # per decision: |best - oks_thr| and, for a match, best - the best other OKS

    def reset(self):
        self.tracks = []

    def frame(self, xy, vis, scores):
        """One frame's persons -> ids int32 [M]."""
        n = len(scores)
        ids = np.full(self.M, -1, np.int32)
        areas = [area_of(xy[p], vis[p]) for p in range(n)]
        order = sorted(range(n), key=lambda p: (-float(scores[p]), p))
        live = self.tracks
        table = [[oks(xy[p], vis[p], areas[p], t["xy"], t["vis"], t["area"], self.kpt_vars) for t in live]
                 for p in range(n)]
        claimed, new = set(), []
        for p in order:
            cands = [(table[p][j], j) for j in range(len(live)) if j not in claimed]
            best_j = None
            if cands:
                best_v = max(v for v, _ in cands)
                best_j = min(j for v, j in cands if v == best_v)      # equal OKS: the smaller id (ids ascend with j)
                others = [v for v, _ in cands if v != best_v]
                self.margins.append(abs(best_v - self.oks_thr))
                if others and best_v > self.oks_thr:      # the runner-up matters only when the best one is taken
                    self.margins.append(best_v - max(others))
            if best_j is not None and best_v > self.oks_thr:
                claimed.add(best_j)
                t = live[best_j]
                t.update(xy=xy[p].copy(), vis=vis[p].copy(), area=areas[p], age=0)
                ids[p] = t["id"]
            elif vis[p].sum() >= self.min_keypoints:
                ids[p] = self.next_id
                new.append(dict(id=self.next_id, xy=xy[p].copy(), vis=vis[p].copy(), area=areas[p], age=0))
                self.next_id += 1
        for j, t in enumerate(live):
            if j not in claimed:
                t["age"] += 1
        self.tracks = [t for t in live if t["age"] < self.max_age] + new
        return ids

    def update(self, records):
        """uint8 [n, row_bytes] records in time order -> ids int32 [n, M]."""
        return np.stack([self.frame(*frame_persons(r, self.K, self.M, self.E)) for r in np.asarray(records)])


def make_records(frames, K, M, E, fallback=()):
    """Result records of synthetic frames: frames[f] is a list of persons (xy float64 [K,2], vis bool [K], score);
    frames whose index is in ``fallback`` carry the empty-scene fallback flag and one pseudo-person instead.
    -> uint8 [n, row_bytes]."""
    row, oc, op, osc, on, of = record_layout(K, M, E)
    out = np.zeros((len(frames), row), np.uint8)
    for f, persons in enumerate(frames):
        r = out[f]
        coco = r[oc:op].view(np.float64).reshape(M, 3 * K + 1)
        poses = r[op:osc].view(np.float32).reshape(M, K, 3 + E)
        scores = r[osc:on].view(np.float32)
        if f in fallback:
            persons = [(np.full((K, 2), 7.0), np.ones(K, bool), 0.01)]
        assert len(persons) <= M
        for p, (xy, vis, score) in enumerate(persons):
            coco[p, 0:3 * K:3], coco[p, 1:3 * K:3], coco[p, 2:3 * K:3] = xy[:, 0], xy[:, 1], 1.0
            coco[p, 3 * K] = score
            poses[p, :, :2] = xy
            poses[p, :, 2] = np.where(vis, 0.5, 0.0)
            scores[p] = score
        r[on:on + 4].view(np.int32)[0] = len(persons)
        r[of:of + 4].view(np.int32)[0] = 1 if f in fallback else 0
    return out
