"""TEST INFRASTRUCTURE ONLY -- grouping scenes: top-k tensors built by hand, not decoded.

Each builder returns a ``Scene``: the inputs of MPPEHeatmapParser.match_by_tag (grouping.py:85-145) for one image,
``tags_k [K,M,E]`` float32, ``coords_k [K,M,2]`` int32, ``scores_k [K,M]`` float32, the two thresholds and an
optional joint order.  The scenes are built to reach the branches of the grouping that decoded maps rarely reach:
Hungarian ties and long solves, dict-key clashes (the one-by-one placement), thresholds hit exactly, unsorted
scores, the float32 mean order, a custom joint order, the empty-scene fallback and non-finite values.  Everything
is seeded.  Only tests import this module; the product package never does.
"""
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

F32 = np.float32


@dataclass
class Scene:
    name: str
    tags_k: np.ndarray
    coords_k: np.ndarray
    scores_k: np.ndarray
    det_thr: float
    tag_thr: float
    joints_order: Optional[List[int]] = None
    finite: bool = True       # False: the reference's munkres would not return (run through the library's guard only)

    @property
    def shape(self):
        K, M, E = self.tags_k.shape
        return K, M, E


def _coords(rng, K, M, lo=0, hi=512):
    return rng.integers(lo, hi, (K, M, 2)).astype(np.int32)


def _grid_crowd(name, seed, K, M, E, persons, first_present, present, offsets, pitch=1.0, score_grid=0.25,
                det_thr=0.1, tag_thr=3.0, junk=0.0):
    """Persons with tags on a grid of ``pitch`` (E = 2: second component on the same grid, permuted); each joint
    shows a random subset of them (the first joint ``first_present`` persons, later ones ``present`` of them) with
    tags at the person's tag plus an offset drawn from ``offsets`` and scores on a ``score_grid`` grid above
    det_thr, sorted by score like top-k.  Ranks below the detections get the score ``junk`` (<= det_thr)."""
    rng = np.random.default_rng(seed)
    base = np.zeros((persons, E), np.float64)
    base[:, 0] = rng.permutation(persons) * pitch
    if E == 2:
        base[:, 1] = rng.permutation(persons) * pitch
    tags = np.zeros((K, M, E), F32)
    scores = np.full((K, M), junk, F32)
    for k in range(K):
        cnt = min(first_present if k == 0 else present, persons, M)
        who = rng.choice(persons, cnt, replace=False)
        sc = (rng.integers(1, 1 + int(round(1 / score_grid)), cnt) * score_grid).astype(F32)
        sc = np.maximum(sc, F32(det_thr + score_grid)) if det_thr >= 0 else sc
        order = np.argsort(-sc, kind="stable")
        for r, i in enumerate(order):
            tags[k, r] = (base[who[i]] + rng.choice(offsets, E)).astype(F32)
            scores[k, r] = sc[i]
        tags[k, cnt:] = rng.integers(-50, 50, (M - cnt, E)).astype(F32)
    return Scene(name, tags, _coords(rng, K, M), scores, det_thr, tag_thr)


HALF = [-2.5, -1.5, -0.5, 0.5, 1.5, 2.5]


def hungarian_ties() -> List[Scene]:
    """E = 1 persons on an integer grid, detections at half-integer offsets (np.round's half-to-even ties on the
    distance), scores on a 1/4 grid (equal costs); nr < G, nr == G, nr > G; M = 32 with n = 32."""
    out = []
    for i, (M, persons, first, present) in enumerate([(30, 20, 20, 12), (30, 16, 16, 16), (30, 24, 8, 24),
                                                      (32, 32, 32, 32), (32, 32, 32, 32), (32, 40, 32, 32)]):
        for j, offs in enumerate((HALF, HALF + [0.0, 1.0, -1.0])):
            out.append(_grid_crowd(f"ties{i}{j}_m{M}_p{persons}", 100 + 10 * i + j, 17, M, 1, persons, first,
                                   present, offs, tag_thr=2.6))
    # dense grids: persons one tag unit apart, detections up to 3.5 away -> long solves
    for j in range(4):
        out.append(_grid_crowd(f"ties_dense{j}", 150 + j, 17, 32, 1, 32, 32, 32, [-3.5, -2.5, 0.5, 1.5, 2.5, 3.5],
                               pitch=1.0, score_grid=0.25, tag_thr=4.0))
    for j in range(2):
        out.append(_grid_crowd(f"ties_e2_{j}", 160 + j, 17, 32, 2, 32, 32, 28, HALF, tag_thr=3.0))
    return out


def dict_keys() -> List[Scene]:
    """E = 2 detections whose float32 tag[0] equals an existing person's key or another new detection's key while
    tag[1] keeps them unmatched (the one-by-one placement); +0 / -0 keys; persons beyond M; M in {1, 2, 5}."""
    out = []
    for M in (1, 2, 5, 8, 30):
        for j in range(3):
            rng = np.random.default_rng(200 + 7 * M + j)
            K = 17
            levels = [0.0, -0.0, 0.5, 1.0, 1.5, 2.0, 3.0] if j != 2 else [0.0, -0.0, 1.0]
            tags = np.zeros((K, M, 2), F32)
            tags[..., 0] = rng.choice(levels, (K, M))
            tags[..., 1] = rng.integers(0, 4, (K, M)) * F32(4.0)      # 4 apart: tag_thr 1.5 rarely matches
            scores = np.sort(rng.integers(1, 8, (K, M)).astype(F32) / 8, axis=1)[:, ::-1].copy()
            scores[rng.random((K, M)) < 0.15] = 0.0
            scores = -np.sort(-scores, axis=1)
            out.append(Scene(f"keys_m{M}_{j}", tags, _coords(rng, K, M), scores, 0.1, 1.5))
    return out


def thresholds() -> List[Scene]:
    """Scores equal to float32(det_thr) (det_thr given as float(np.float32(x)) and as x, compared in float64);
    distances exactly tag_thr and one ulp below; a negative det_thr with -0 and negative scores."""
    out = []
    K, M = 17, 8
    rng = np.random.default_rng(300)
    for x in (0.1, 0.3):
        for thr in (float(F32(x)), x):
            tags = (np.arange(M, dtype=F32)[None, :, None] * F32(10) + np.zeros((K, 1, 1), F32))
            scores = np.full((K, M), F32(x), F32)
            scores[:, ::3] = F32(0.75)
            scores = -np.sort(-scores, axis=1)
            out.append(Scene(f"det_eq_{x}_{'f32' if thr != x else 'f64'}", tags, _coords(rng, K, M), scores, thr, 1.0))
    # persons at 2, 12, 22, ...; every later detection sits exactly 0.5 (E = 1) / 0.625 (E = 2: 0.375, 0.5) away
    for E, d in ((1, 0.5), (2, 0.625)):
        for below in (False, True):
            tags = np.zeros((K, M, E), F32)
            tags[..., 0] = np.arange(M, dtype=F32) * 10 + 2
            if E == 2:
                tags[..., 1] = np.arange(M, dtype=F32) * 10
            sign = np.where(np.arange(K) % 2 == 0, 1, -1).astype(F32)[:, None]
            tags[1:, :, 0] += sign[1:] * F32(0.5 if E == 1 else 0.375)
            if E == 2:
                tags[1:, :, 1] += F32(0.5)
            thr = float(np.nextafter(d, 1.0)) if below else d
            scores = np.full((K, M), F32(0.5), F32)
            # the second joint in order meets tag lists of length 1, i.e. means exactly at the first joint's tags
            out.append(Scene(f"tag_eq_e{E}_{'below' if below else 'equal'}", tags, _coords(rng, K, M), scores,
                             0.1, thr))
    for j in range(2):
        rng2 = np.random.default_rng(310 + j)
        tags = (rng2.integers(0, 6, (K, M, 1)) * F32(1.0)).astype(F32)
        scores = -np.sort(-rng2.choice(np.array([0.25, 0.0, -0.0, -0.25, -0.5, -0.75], F32), (K, M)), axis=1)
        out.append(Scene(f"neg_det_thr{j}", tags, _coords(rng2, K, M), scores, -0.5, 1.0))
    return out


def foreign() -> List[Scene]:
    """Data no top-k produces: unsorted scores with holes below det_thr (the kernel's compaction), scores above
    100 (negative costs), negative coordinates and coordinates >= 2^24."""
    out = []
    for j, (M, E) in enumerate([(30, 1), (30, 2), (32, 2), (7, 1)]):
        s = _grid_crowd(f"unsorted{j}", 400 + j, 17, M, E, min(M, 20), min(M, 20), 14, HALF + [0.0], tag_thr=2.6)
        rng = np.random.default_rng(410 + j)
        for k in range(17):
            p = rng.permutation(M)
            s.scores_k[k] = s.scores_k[k, p]
            s.tags_k[k] = s.tags_k[k, p]
        out.append(s)
    for j in range(2):
        s = _grid_crowd(f"big_scores{j}", 420 + j, 17, 30, 2 - j, 20, 20, 15, HALF, tag_thr=2.6)
        s.scores_k *= F32(400.0)                        # up to 400: cost = rint(d) * 100 - score < 0
        s.det_thr = 60.0
        out.append(s)
    for j in range(2):
        s = _grid_crowd(f"far_coords{j}", 430 + j, 17, 30, 1 + j, 20, 20, 15, HALF, tag_thr=2.6)
        rng = np.random.default_rng(440 + j)
        s.coords_k = rng.integers(-(1 << 30), 1 << 30, s.coords_k.shape).astype(np.int32)
        s.coords_k[:, ::2, 0] = (1 << 24) + rng.integers(1, 1000, s.coords_k[:, ::2, 0].shape)   # odd: rounds
        s.coords_k[:, 1::3, 1] = -rng.integers(1, 1 << 26, s.coords_k[:, 1::3, 1].shape)
        out.append(s)
    return out


def _pairwise_mean(vals):
    """NumPy's float32 mean over a [n, 1] tag list (pairwise-8 summation)."""
    return np.mean(np.array(vals, F32).reshape(-1, 1), axis=0)[0]


def _sequential_mean(vals):
    s = F32(0)
    for v in vals:
        s = F32(s + F32(v))
    return F32(s / F32(len(vals)))


def mean_order() -> List[Scene]:
    """E = 1, K = 32: two persons whose tag lists grow to L in 9..31 entries; at step L a detection sits between
    the tag_thr decisions of NumPy's pairwise-8 float32 mean and a sequential one (asserted: the sequential mean
    would flip the match)."""
    out = []
    K, M = 32, 2
    for L in (9, 12, 16, 17, 24, 31):
        rng = np.random.default_rng(500 + L)
        for _ in range(1000):
            vals = (F32(1000.0) + rng.integers(-1000, 1000, L).astype(F32) * F32(2.0 ** -12)).astype(F32)
            mp, ms = _pairwise_mean(vals), _sequential_mean(vals)
            if mp != ms:
                break
        assert mp != ms, "no discriminating tag list found"
        x = F32(mp + F32(0.75))
        dp, ds = abs(float(x) - float(mp)), abs(float(x) - float(ms))
        tag_thr = (dp + ds) / 2          # dp < tag_thr <= ds or the reverse
        assert (dp < tag_thr) != (ds < tag_thr)
        tags = np.zeros((K, M, 1), F32)
        tags[:, 1, 0] = F32(-1000.0)      # the second person, far away, always matches
        tags[:L, 0, 0] = vals
        tags[L:, 0, 0] = x
        scores = np.full((K, M), F32(0.5), F32)
        out.append(Scene(f"mean_order_L{L}", tags, _coords(rng, K, M), scores, 0.1, tag_thr))
    return out


def joints_order() -> List[Scene]:
    """K = 23 with a random joint order (HpdParams.joints_order / hpo_match_by_tag's joints_order)."""
    out = []
    for j, E in enumerate((1, 2, 2)):
        s = _grid_crowd(f"order_k23_{j}", 600 + j, 23, 30, E, 18, 18, 12, HALF + [0.0], tag_thr=2.6)
        s.joints_order = [int(v) for v in np.random.default_rng(610 + j).permutation(23)]
        out.append(s)
    return out


def fallback() -> List[Scene]:
    """No score above det_thr and NaN among the rank-0 tags: the empty-scene fallback (flags bit 0), whose
    pseudo-person maps NaN tags to 0.  No solver runs."""
    out = []
    for E in (1, 2):
        rng = np.random.default_rng(700 + E)
        K, M = 17, 30
        tags = rng.standard_normal((K, M, E)).astype(F32)
        tags[::3, 0, 0] = np.nan
        tags[1::4, 0, E - 1] = np.nan
        scores = -np.sort(-rng.random((K, M)).astype(F32) * F32(0.1), axis=1)
        out.append(Scene(f"fallback_e{E}", tags, _coords(rng, K, M), scores, 0.1, 1.0, finite=False))
    return out


def non_finite() -> List[Scene]:
    """NaN and +-inf tags, inf scores, tags of about 1e18: costs the reference's munkres never returns on."""
    out = []
    bad = [("nan_tag", "tag", np.nan), ("inf_tag", "tag", np.inf), ("ninf_tag", "tag", -np.inf),
           ("inf_score", "score", np.inf), ("huge_tag", "tag", 1e18), ("nhuge_tag", "tag", -3e18)]
    for i, (what, field, v) in enumerate(bad):
        for E in (1, 2):
            s = _grid_crowd(f"{what}_e{E}", 800 + 2 * i + E, 17, 30, E, 20, 20, 15, HALF, tag_thr=2.6)
            s.name, s.finite = f"{what}_e{E}", False
            rng = np.random.default_rng(900 + 2 * i + E)
            ks = rng.choice(np.arange(1, 17), 4, replace=False)
            for k in ks:
                r = int(rng.integers(0, 10))
                if field == "tag":
                    s.tags_k[k, r, int(rng.integers(0, E))] = v
                else:
                    s.scores_k[k, r] = v
                    s.scores_k[k] = -np.sort(-s.scores_k[k])
            out.append(s)
    # the issue's two-person case: a NaN tag on a detection of the second joint
    tags = np.array([[[0.0], [5.0]], [[np.nan], [5.0]]], F32)
    out.append(Scene("nan_two_persons", tags, np.zeros((2, 2, 2), np.int32), np.full((2, 2), 0.9, F32), 0.1, 1.0,
                     finite=False))
    return out


FAMILIES = dict(hungarian_ties=hungarian_ties, dict_keys=dict_keys, thresholds=thresholds, foreign=foreign,
                mean_order=mean_order, joints_order=joints_order, fallback=fallback, non_finite=non_finite)


def all_scenes() -> List[Scene]:
    return [s for f in FAMILIES.values() for s in f()]
