"""-m gpu: the sparse refine (csrc/refine.cu) and its prefilter against the CPU oracle, on scenes built to reach the
edges of the search: value ties across words, rows, 4-row bands and the two sweeps, winners among and outside the
top-k seeds, half-way tag distances, words on the sweep boundary, word bounds equal to the running best, bests with
hm <= 0, a pairwise-8 mean tag, winners on the image border and in the last partial word of a row.

The scenes are network outputs (hm_lo = 0, hm_hi = 2 X, so the aggregated heatmap is the x2 upsampling of X), so the
real aggregation kernels run and derive the tag bounds refine prunes with.  Heatmap and tag values are small dyadic
numbers, and tags are constant over the quarter-res taps of the pixels that matter, so the bilinear taps reproduce
them exactly and the builder can place exact tag distances.  Every scene checks, from the oracle's own maps, that the
edges it was built for really occur.

Besides the decode's outputs, the refine workspace is read back after every decode: for each listed (person, joint)
pair its final key must be the oracle's argmax (value and first index), which also pins pairs whose best is not
replaced."""
import numpy as np
import pytest
import torch

from oracle import cpu_oracle

pytestmark = pytest.mark.gpu

COCO_FLIP = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15]
DET_V = 4.0            # X value of a detected joint: its unique full-res maximum is 0.765625 * 4 = 3.0625
DET_THR, TAG_THR = 3.0, 1.0
BG_TAG = 200.0         # tag of everything that is not part of a spot: far from every person


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------------------------
# scene builder
# ------------------------------------------------------------------------------------------------------------------
class Scene:
    """Network outputs of one image, built spot by spot.  Cell (ci, cj) covers quarter-res rows 4ci..4ci+3 and columns
    4cj..4cj+3 (full-res 16 x 16 pixels); a spot's tag block covers quarter-res rows / columns 4c..4c+2, which are all
    the taps of full-res pixels 16c+2 .. 16c+9."""

    def __init__(self, H, W, K, E, seed):
        self.H, self.W, self.K, self.E = H, W, K, E
        self.X = np.zeros((K, H // 2, W // 2), np.float32)           # stage mean (half res)
        self.lo = np.zeros((K, H // 4, W // 4), np.float32)          # hm_lo (only -0 regions)
        self.t0 = np.full((K, H // 4, W // 4), BG_TAG, np.float32)
        self.t1 = np.zeros((K, H // 4, W // 4), np.float32)
        self.nci, self.ncj = H // 16, W // 16
        self.rng = np.random.default_rng(seed)
        self.free = {}

    def cells(self, k):
        if k not in self.free:
            # the border cells hold the edge spots, unless the image ends in a strip no cell covers
            ri = range(1, self.nci - (1 if self.H % 64 == 0 else 0))
            rj = range(1, self.ncj - (1 if self.W % 64 == 0 else 0))
            c = [(i, j) for i in ri for j in rj]
            self.free[k] = [c[i] for i in self.rng.permutation(len(c))]
        return self.free[k]

    def take(self, k, cell=None):
        f = self.cells(k)
        if cell is None:
            return f.pop()
        f.remove(cell)
        return cell

    def tag_block(self, k, r0, r1, c0, c1, t):
        self.t0[k, r0:r1, c0:c1] = t[0]
        self.t1[k, r0:r1, c0:c1] = t[1] if len(t) > 1 else 0.0

    def detected(self, k, cell, T):
        """A detected joint: unique full-res maximum 0.765625 * DET_V at (16ci+5, 16cj+5), tag T."""
        ci, cj = cell
        r, c = 8 * ci + 2, 8 * cj + 2
        self.X[k, r:r + 2, c:c + 2] = DET_V * np.array([[1, .5], [.5, .25]], np.float32)
        self.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj, 4 * cj + 3, T)

    def spot(self, k, cell, v, t):
        """A 2 x 2 full-res plateau of value v at rows 16ci+5..6, columns 16cj+5..6 (ringed by 0.75 v), tag t."""
        ci, cj = cell
        self.X[k, 8 * ci + 2:8 * ci + 4, 8 * cj + 2:8 * cj + 4] = v
        self.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj, 4 * cj + 3, t)

    def zero_spot(self, k, cell, t, negative):
        """hm = -0 (negative) or +0 over the cell, tag t over the spot block: every value there is 0."""
        ci, cj = cell
        if negative:   # -0 in hm_lo and hm_hi one cell around the spot (zeros only: neighbouring spots stay)
            for a, r in ((self.lo, 4), (self.X, 8)):
                blk = a[k, max(r * ci - r, 0):r * ci + 2 * r, max(r * cj - r, 0):r * cj + 2 * r]
                blk[blk == 0] = -0.0
        self.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj, 4 * cj + 3, t)

    def grad_row(self, k, cell, T):
        """Tag T+2 on quarter rows 4ci, 4ci+1 and T below: the winner (16ci+7, hm 1.75, tag T+1.25) reads quarter row
        4ci+2 -- the third row of its band's bound -- and ties with (16ci+9, hm 0.75, tag T+0.25) in the next band."""
        ci, cj = cell
        self.X[k, 8 * ci + 3, 8 * cj + 2:8 * cj + 4] = 2.0
        self.X[k, 8 * ci + 4, 8 * cj + 2:8 * cj + 4] = 1.0
        self.tag_block(k, 4 * ci, 4 * ci + 2, 4 * cj, 4 * cj + 3, (T[0] + 2,) + T[1:])
        self.tag_block(k, 4 * ci + 2, 4 * ci + 4, 4 * cj, 4 * cj + 3, T)

    def grad_col(self, k, cell, T):
        """The same along x: the winner (x = 16cj+7, tag T+1.25) interpolates two different quarter-res columns."""
        ci, cj = cell
        self.X[k, 8 * ci + 2:8 * ci + 4, 8 * cj + 3] = 2.0
        self.X[k, 8 * ci + 2:8 * ci + 4, 8 * cj + 4] = 1.0
        self.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj, 4 * cj + 2, (T[0] + 2,) + T[1:])
        self.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj + 2, 4 * cj + 4, T)

    def edge(self, k, side, cell, v, t):
        """A unique maximum v on the image border: x = 0 ('l'), x = W-1 ('r') or y = H-1 ('b')."""
        ci, cj = cell
        hh, hw, th, tw = self.H // 2, self.W // 2, self.H // 4, self.W // 4
        prof = np.array([1.0, 0.5], np.float32) * v
        if side == "l":
            self.X[k, 8 * ci + 2:8 * ci + 4, 0:2] = prof
            self.tag_block(k, 4 * ci, 4 * ci + 3, 0, 2, t)
        elif side == "r":
            self.X[k, 8 * ci + 2:8 * ci + 4, hw - 2:hw] = prof[::-1]
            self.tag_block(k, 4 * ci, 4 * ci + 3, tw - 2, tw, t)
        else:
            self.X[k, hh - 2:hh, 8 * cj + 2:8 * cj + 4] = prof[::-1, None]
            self.tag_block(k, th - 2, th, 4 * cj, 4 * cj + 3, t)

    def outputs(self, flip_index, hm_scale=1.0):
        """{hm_lo, hm_hi, tag[, *_f]} [1,K,h,w]: the flipped run holds the mirrored, joint-permuted maps, so the flip
        average reproduces hm_hi = 2 X and the second tag component is t1."""
        s = {"hm_lo": self.lo * np.float32(hm_scale), "hm_hi": self.X * np.float32(2 * hm_scale), "tag": self.t0}
        if self.E == 2:
            fl = list(flip_index)
            s.update(hm_lo_f=s["hm_lo"][fl][..., ::-1], hm_hi_f=s["hm_hi"][fl][..., ::-1], tag_f=self.t1[fl][..., ::-1])
        return {n: np.ascontiguousarray(a[None], np.float32) for n, a in s.items()}


# pair recipes: (kind, [(value, tag offset (d0, d1), placement)]) -- the first spot has the lower index unless noted
def _plant(sc, k, T, kind):
    def off(d):
        return (T[0] + d[0],) + ((T[1] + d[1],) if sc.E == 2 else ())

    def two():
        a, b = sc.take(k), sc.take(k)
        return (a, b) if a < b else (b, a)

    if kind == "tie_bands":            # 0.75 at d 0 (lower index) against 1.75 at d 1
        a, b = two()
        sc.spot(k, a, 0.75, off((0, 0))); sc.spot(k, b, 1.75, off((1, 0)))
    elif kind == "tie_rev":            # 1.75 at d 1 (lower index) against 0.75 at d 0
        a, b = two()
        sc.spot(k, a, 1.75, off((1, 0))); sc.spot(k, b, 0.75, off((0, 0)))
    elif kind == "seed_hi":            # a top-k seed (2.75 at d 2) ties with a lower-index non-seed (0.75 at d 0)
        a, b = two()
        sc.spot(k, a, 0.75, off((0, 0))); sc.spot(k, b, 2.75, off((2, 0)))
    elif kind == "seed_lo":            # the lower-index one is the seed
        a, b = two()
        sc.spot(k, a, 2.75, off((-2, 0))); sc.spot(k, b, 0.75, off((0, 0)))
    elif kind == "half05":             # d = 0.5 rounds to 0: 1.0 beats 0.875 (round-half-up would pick the latter)
        a, b = two()
        sc.spot(k, a, 0.875, off((0, 0))); sc.spot(k, b, 1.0, off((0.5, 0)))
    elif kind == "half25":             # d = 2.5 (E = 2: from (1.5, 2)) rounds to 2: 2.5 - 2 beats 0.375
        a, b = two()
        sc.spot(k, a, 0.375, off((0, 0)))
        sc.spot(k, b, 2.5, off((1.5, 2.0) if sc.E == 2 else (2.5, 0)))
    elif kind == "half15":             # d = 1.5 rounds to 2 (half-even and half-up agree): 2.5 - 2 ties with 0.5 at d 0
        a, b = two()                   # at the lower index; rounding half down would make the 2.5 win with 1.5
        sc.spot(k, a, 0.5, off((0, 0))); sc.spot(k, b, 2.5, off((-1.5, 0)))
    elif kind == "slack":              # tag T + 2^-6: inside the slack refine_scan_kernel widens the block's bounds by
        a, b = two()                   # (>= 1e-4 * (1 + |T| + 200) with the background tag in the block)
        sc.spot(k, a, 1.0, off((0, 0))); sc.spot(k, b, 1.25, off((2.0 ** -6, 0)))
    elif kind == "split":              # one 2.5 spot at d 0; in a crowded plane its words sit on the sweep boundary
        sc.spot(k, sc.take(k), 2.5, off((0, 0)))
    elif kind == "grad_row":
        sc.grad_row(k, sc.take(k), off((0, 0)))
    elif kind == "grad_col":
        sc.grad_col(k, sc.take(k), off((0, 0)))
    elif kind in ("neg0", "pos0"):     # the best is 0 at hm -0 / +0: nothing is replaced
        sc.zero_spot(k, sc.take(k), off((0, 0)), kind == "neg0")
        sc.spot(k, sc.take(k), 0.5, off((1, 0)))
    elif kind in ("edge_l", "edge_r", "edge_b"):
        side = kind[-1]
        pick = [c for c in sc.cells(k) if (side != "b" or c[1] < sc.ncj - 1)]
        cell = sc.take(k, pick[0])
        sc.edge(k, side, cell, 1.25, off((0, 0)))
        sc.spot(k, sc.take(k), 1.0, off((0, 0)))
    else:
        raise ValueError(kind)


KINDS = ["tie_bands", "tie_rev", "seed_hi", "seed_lo", "half05", "half25", "half15", "split", "grad_row", "grad_col",
         "neg0", "pos0", "slack"]


def _build(name):
    """-> dict(scene, scales (numpy, one image), H, W, K, M, E, flip_index, persons, missing)."""
    if name == "crowd32":
        # M = 32 persons, all missing joint 16 (a full warp of pairs), persons 0..14 also joint p+1 (single pairs)
        H = W = 256; K, M, E = 17, 32, 2
        sc = Scene(H, W, K, E, seed=1)
        P = 32
        tags = [((p - 16) * 8.0, 0.0) for p in range(P)]
        missing = {p: {16} | ({p + 1} if p < 15 else set()) for p in range(P)}
        kinds = KINDS + ["edge_l", "edge_r", "edge_b"]
    elif name == "e1_pairwise":
        # E = 1, no flip; person 0 has 16 detected joints whose tags need more bits than float32 keeps, so the
        # pairwise-8 mean differs from a sequential one; its missing joint is decided by that difference
        H = W = 256; K, M, E = 17, 20, 1
        sc = Scene(H, W, K, E, seed=2)
        P = 12
        tags = [((p - 6) * 8.0,) for p in range(P)]
        missing = {p: {(p * 5 + 3) % 16 + 1, (p * 7 + 1) % 16 + 1} for p in range(1, P)}
        missing[0] = {16}
        kinds = KINDS
    elif name == "generic248":
        # W % 32 != 0 (generic kernel, +-inf bounds): winners at x = 0, x = W-1, y = H-1 and in the last partial word
        H, W = 184, 248; K, M, E = 17, 16, 2
        sc = Scene(H, W, K, E, seed=3)
        P = 8
        tags = [((p - 4) * 8.0, 0.0) for p in range(P)]
        missing = {p: {16, (p % 8) * 2 + 1} for p in range(P)}
        kinds = ["edge_l", "edge_r", "edge_b", "lastword"] + KINDS
    else:
        raise ValueError(name)
    flip_index = COCO_FLIP
    person_cells = [sc.cells(0)[i] for i in range(P)]
    for k in range(K):
        for c in person_cells:
            sc.take(k, c)
    i = 0
    for p in range(P):
        for k in range(K):
            if k in missing[p]:
                kind = kinds[i % len(kinds)]
                i += 1
                if kind == "lastword":
                    cell = sc.take(k, [c for c in sc.cells(k) if c[1] == W // 32 * 2][0])   # x = 16cj+5 >= W // 32 * 32
                    sc.spot(k, cell, 1.25, tags[p]); sc.spot(k, sc.take(k), 1.0, tags[p])
                else:
                    _plant(sc, k, tags[p], kind)
            else:
                sc.detected(k, person_cells[p], tags[p])
    if name == "e1_pairwise":
        # person 0: tags 1000 + odd multiples of 2^-12 on its detected joints
        ks = [k for k in range(K) if k not in missing[0]]
        while True:
            vals = (1000 + (2 * sc.rng.integers(0, 2048, len(ks)) + 1) / 4096).astype(np.float32)
            if np.mean(vals) != _seq_mean(vals):
                break
        ci, cj = person_cells[0]
        for k, v in zip(ks, vals):
            sc.tag_block(k, 4 * ci, 4 * ci + 3, 4 * cj, 4 * cj + 3, (v,))
    return dict(scene=sc, H=H, W=W, K=K, M=M, E=E, flip_index=flip_index, P=P, missing=missing,
                person_cells=person_cells, name=name)


def _seq_mean(vals):
    t = np.float32(0)
    for v in vals:
        t = np.float32(t + v)
    return np.float32(t / np.float32(len(vals)))


def _finish_e1_pairwise(case):
    """Place person 0's deciding spots once its mean tag is known: A (hm 1.0) at distance exactly 0.5 from the
    pairwise-8 mean, on the side where a sequential mean puts it past 0.5; B (hm 0.5) at distance 0."""
    sc = case["scene"]
    hm, tg = cpu_oracle.aggregate([{k: v[0] for k, v in sc.outputs(case["flip_index"]).items()}], (case["H"], case["W"]),
                                  flip_index=case["flip_index"])
    ref = cpu_oracle.parse(hm, tg, case["M"], DET_THR, TAG_THR, refine=False)
    gj = ref["grouped_joints"]
    p0 = [p for p in range(gj.shape[0]) if gj[p, 0, 3] > 900][0]
    have = np.array([tg[k, int(gj[p0, k, 1]), int(gj[p0, k, 0]), 0] for k in range(case["K"]) if gj[p0, k, 2] > 0],
                    np.float32)
    t_pair, t_seq = np.float32(np.mean(have)), _seq_mean(have)
    assert t_pair != t_seq, "person 0's tags do not tell the pairwise-8 mean from a sequential one"
    a = np.float32(t_pair - np.float32(0.5)) if t_seq > t_pair else np.float32(t_pair + np.float32(0.5))
    k = 16
    ca, cb = sc.take(k), sc.take(k)
    ca, cb = (ca, cb) if ca > cb else (cb, ca)       # A at the higher index: it wins on value alone
    sc.spot(k, ca, 1.0, (a,))
    sc.spot(k, cb, 0.5, (t_pair,))
    case["t_pair"], case["t_seq"] = t_pair, t_seq


_CACHE = {}


def _case(name):
    """Scene + oracle results, computed once per session."""
    if name in _CACHE:
        return _CACHE[name]
    case = _build(name)
    if name == "e1_pairwise":
        _finish_e1_pairwise(case)
    sc = case["scene"]
    case["scales"] = [sc.outputs(case["flip_index"])]
    _oracle(case, case["scales"])
    _CACHE[name] = case
    return case


def _oracle(case, scales, into=None):
    """Oracle maps, parse with and without refine, and the argmax of every listed (person, missing joint) pair."""
    out = case if into is None else into
    H, W, K, M = case["H"], case["W"], case["K"], case["M"]
    img = [{k: v[0] for k, v in s.items()} for s in scales]
    hm, tg = cpu_oracle.aggregate(img, (H, W), flip_index=case["flip_index"], tag_scale=case.get("tag_scale", 0))
    out["hm"], out["tg"] = hm, tg
    out["ref"] = cpu_oracle.parse(hm, tg, M, DET_THR, TAG_THR)
    out["noref"] = cpu_oracle.parse(hm, tg, M, DET_THR, TAG_THR, refine=False)
    out["pairs"] = _pairs(hm, tg, out["noref"]["grouped_joints"])
    return out


def _value_map(hm, tg, T, E, rnd=np.round):
    a = (tg[..., 0] - T[0]).astype(np.float32)
    s = (a * a).astype(np.float32)
    if E > 1:
        b = (tg[..., 1] - T[1]).astype(np.float32)
        s = (s + (b * b).astype(np.float32)).astype(np.float32)
    d = np.sqrt(s).astype(np.float32)
    return (hm - rnd(d).astype(np.float32)).astype(np.float32) + np.float32(0.0), d


def _pairs(hm, tg, noref):
    """{(p, k): dict(T, idx, val)} -- grouping.py:193-250 restated per pair (first index of the maximum)."""
    K, H, W = hm.shape
    E = tg.shape[3]
    out = {}
    for p in range(noref.shape[0]):
        person = noref[p]
        have = [tg[k, int(person[k, 1]), int(person[k, 0])] for k in range(K) if person[k, 2] > 0]
        T = np.mean(np.array(have, np.float32), axis=0).astype(np.float32) if have else np.full(E, np.nan, np.float32)
        for k in range(K):
            if person[k, 2] != 0:
                continue
            v, d = _value_map(hm[k], tg[k], T, E)
            idx = int(np.argmax(v))
            out[(p, k)] = dict(T=T, idx=idx, val=v.reshape(-1)[idx], v=v.reshape(-1), d=d.reshape(-1))
    return out


def _x2_bounds(t0q, H, W):
    """tag_bmin / tag_bmax as agg_nms_x2_kernel derives them from the quarter-res first tag component: block (band g,
    word w) covers quarter-res rows g-1..g+1 and columns 8w-1..8w+8, clamped to the map."""
    K, th, tw = t0q.shape
    HB, wpr = (H + 3) // 4, (W + 31) // 32
    lo, hi = np.empty((K, HB, wpr), np.float32), np.empty((K, HB, wpr), np.float32)
    for g in range(HB):
        rows = np.clip(np.arange(g - 1, g + 2), 0, th - 1)
        for w in range(wpr):
            blk = t0q[:, rows][:, :, np.clip(np.arange(8 * w - 1, 8 * w + 9), 0, tw - 1)]
            lo[:, g, w], hi[:, g, w] = blk.min(axis=(1, 2)), blk.max(axis=(1, 2))
    return lo, hi


def _reach(hmx, lo, hi, T):
    """refine_scan_kernel's upper bound of a word's value for mean tag T (float32, the kernel's operation order);
    also whether the block's tag range ends within the slack of T."""
    f = np.float32
    with np.errstate(invalid="ignore", over="ignore"):
        slack = f(f(1e-4) * f(f(f(1) + f(abs(T))) + f(max(abs(lo), abs(hi)))))
        gap = max(f(lo - T), f(T - hi), f(0))
        dmin = max(f(gap - slack), f(0))
    return f(f(hmx - np.round(dmin)) + f(0)), bool(f(0) < gap <= slack)


def _coverage(case):
    """Counts of the edges the scene was built to hit, measured on the oracle's maps."""
    hm, ref, pairs = case["hm"], case["ref"], case["pairs"]
    K, H, W = hm.shape
    wpr = (W + 31) // 32
    if W % 32 == 0:     # the x2 kernel's bounds; the generic kernel's are -inf / +inf
        blo, bhi = _x2_bounds(case["scene"].t0, H, W)
    else:
        blo, bhi = np.full((K, (H + 3) // 4, wpr), -np.inf, np.float32), np.full((K, (H + 3) // 4, wpr), np.inf, np.float32)
    flat = hm.reshape(K, -1)
    idx_k, scores_k = ref["idx_k"], ref["scores_k"]
    words = np.full((K, H, wpr * 32), -np.inf, np.float32)
    words[:, :, :W] = hm
    wmax = words.reshape(K, H, wpr, 32).max(axis=3).reshape(K, -1)
    word_of = lambda i: (i // W) * wpr + (i % W) // 32
    c = dict(pairs=len(pairs), tied=0, tied_rows=0, tied_bands=0, tied_sweeps=0, later_sweep_lower=0, seed_winner_tied=0,
             seed_tie_above=0, sweep1=0, on_split=0, on_split_not_seed=0, half_rounding=0, nonpos=0, neg0=0,
             half_down=0, bound_eq=0, slack=0, edge_x0=0, edge_xw=0, edge_yh=0, last_word=0)
    per_plane = {}
    for (p, k), r in pairs.items():
        per_plane[k] = per_plane.get(k, 0) + 1
        v, idx, val = r["v"], r["idx"], r["val"]
        split = scores_k[k, -1]
        sweep = lambda i: 0 if wmax[k, word_of(i)] >= split else 1
        ties = np.flatnonzero(v == val)
        tw = {word_of(i) for i in ties}
        seeds = set(int(i) for i in idx_k[k])
        if len(tw) > 1:
            c["tied"] += 1
            c["tied_rows"] += len({i // W for i in ties}) > 1
            c["tied_bands"] += len({i // W // 4 for i in ties}) > 1
            sw = {sweep(i) for i in ties}
            c["tied_sweeps"] += len(sw) > 1
            c["later_sweep_lower"] += sweep(idx) == 1 and 0 in sw
            c["seed_winner_tied"] += idx in seeds
            c["seed_tie_above"] += idx not in seeds and any(int(i) in seeds for i in ties)
        c["sweep1"] += sweep(idx) == 1
        on = wmax[k, word_of(idx)] == split
        c["on_split"] += bool(on)
        c["on_split_not_seed"] += bool(on) and idx not in seeds
        v_up, _ = _value_map(hm[k], case["tg"][k], r["T"], case["tg"].shape[3], rnd=lambda d: np.floor(d + np.float32(0.5)))
        c["half_rounding"] += int(np.argmax(v_up)) != idx
        v_dn, _ = _value_map(hm[k], case["tg"][k], r["T"], case["tg"].shape[3], rnd=lambda d: np.ceil(d - np.float32(0.5)))
        c["half_down"] += int(np.argmax(v_dn)) != idx
        c["nonpos"] += not (flat[k, idx] > 0)
        c["neg0"] += bool(flat[k, idx] == 0 and np.signbit(flat[k, idx]))
        y, x = divmod(idx, W)
        c["edge_x0"] += x == 0
        c["edge_xw"] += x == W - 1
        c["edge_yh"] += y == H - 1
        c["last_word"] += W % 32 != 0 and x >= (W // 32) * 32
        # the winner is no seed, a tie at a higher index is one (so the running best holds the winning value before
        # the scan starts), and the bound of the winner's word equals that value exactly: only ">=" expands the word
        reach, in_slack = _reach(wmax[k, word_of(idx)], blo[k, y // 4, x // 32], bhi[k, y // 4, x // 32], r["T"][0])
        c["bound_eq"] += (idx not in seeds and any(int(i) in seeds and i > idx for i in ties)
                          and reach == val + np.float32(0))
        # the winner's block ends within the slack of T (the bound prunes nothing there, as the pixel's distance is
        # the small non-zero gap)
        c["slack"] += in_slack
    c["pairs_per_plane_max"] = max(per_plane.values()) if per_plane else 0
    c["single_pair_planes"] = sum(1 for n in per_plane.values() if n == 1)
    gj, gn = ref["grouped_joints"], case["noref"]["grouped_joints"]
    c["refined_differ"] = int((_bits(gj) != _bits(gn)).any(axis=2).sum())
    return c


# measured on the scenes as built (the builder is deterministic): a later edit that loses any of these fails
EXPECT = {
    "crowd32": dict(pairs=47, pairs_per_plane_max=32, single_pair_planes=15, tied=45, tied_rows=45, tied_bands=23,
                    tied_sweeps=14, later_sweep_lower=8, seed_winner_tied=8, seed_tie_above=13, sweep1=28, on_split=13,
                    on_split_not_seed=8, half_rounding=6, half_down=3, nonpos=6, neg0=2, bound_eq=9, slack=3,
                    edge_x0=3, edge_xw=3, edge_yh=2, refined_differ=41),
    "e1_pairwise": dict(pairs=21, tied=21, tied_bands=11, tied_sweeps=1, seed_tie_above=5, sweep1=1, on_split_not_seed=6,
                        half_rounding=5, half_down=2, nonpos=2, neg0=1, bound_eq=5, slack=1, refined_differ=19),
    "generic248": dict(pairs=16, single_pair_planes=8, tied=15, tied_bands=6, tied_sweeps=2, seed_tie_above=1, sweep1=3,
                       on_split_not_seed=2, half_rounding=2, half_down=1, nonpos=2, neg0=1, edge_x0=1, edge_xw=1,
                       edge_yh=1, last_word=4, refined_differ=14),
}

SCENES = list(EXPECT)


@pytest.mark.parametrize("name", SCENES)
def test_scene_reaches_its_edges(name):
    """The builder still produces what the scene is for (counts measured on the oracle's maps)."""
    case = _case(name)
    cov = _coverage(case)
    print(name, cov)
    for key, n in EXPECT[name].items():
        assert cov[key] >= n, f"{name}: {key} = {cov[key]} < {n} ({cov})"
    if name == "e1_pairwise":
        p0 = [p for p in range(case["noref"]["grouped_joints"].shape[0])
              if case["noref"]["grouped_joints"][p, 0, 3] > 900][0]
        r = case["pairs"][(p0, 16)]
        v_seq, _ = _value_map(case["hm"][16], case["tg"][16], np.array([case["t_seq"]], np.float32), 1)
        assert int(np.argmax(v_seq)) != r["idx"], "the pairwise-8 mean does not decide person 0's missing joint"


# ------------------------------------------------------------------------------------------------------------------
# decode paths
# ------------------------------------------------------------------------------------------------------------------
def _poison(bufs, params):
    for name in ("agg_hm", "tag_map", "poses", "person_scores", "scores_k", "tags_k", "hm_wmax", "nms_wmax",
                 "tag_bmin", "tag_bmax"):
        t = getattr(bufs, name)
        if t is not None and t.numel():
            t.fill_(float("nan"))
    for name in ("idx_k", "coords_k", "n_person", "flags", "nms_mask"):
        getattr(bufs, name).fill_(-1)
    bufs.records.fill_(0xFF)
    bufs.ensure_workspace(params).fill_(0xFF)


def _ordered(v):
    u = np.float32(v).view(np.uint32).astype(np.uint64)
    return int(~u & 0xFFFFFFFF) if u & 0x80000000 else int(u | 0x80000000)


def _check(bufs, want, what, M, K, E):
    """Records, idx_k, and the refine workspace's final key of every listed pair against the oracle."""
    from hpdecode.decoder import Records
    torch.cuda.synchronize()
    ref, pairs = want["ref"], want["pairs"]
    assert np.array_equal(bufs.idx_k[0].cpu().numpy(), ref["idx_k"]), f"{what}: idx_k"
    assert np.array_equal(_bits(bufs.scores_k[0].cpu().numpy()), _bits(ref["scores_k"])), f"{what}: scores_k"
    rec = Records(bufs.records.cpu().numpy(), M, K, E)
    gj, ps = rec.image(0)
    assert not ref["fallback"]
    assert gj.shape == ref["grouped_joints"].shape, f"{what}: person count {gj.shape[0]} != {ref['grouped_joints'].shape[0]}"
    bad = np.argwhere((_bits(gj) != _bits(ref["grouped_joints"])).any(axis=2))
    assert bad.size == 0, f"{what}: grouped joints differ at (person, joint) {bad[:8].tolist()}"
    assert np.array_equal(_bits(ps), _bits(ref["person_scores"])), f"{what}: person scores"
    assert np.array_equal(_bits(bufs.poses[0, :gj.shape[0]].cpu().numpy()), _bits(gj)), f"{what}: poses buffer"
    # refine workspace (csrc/refine.cu RefineWs, one image): keys [K][M] u64, T [M][2], miss_cnt [K], miss_pid [K][M]
    ws = bufs.workspace.cpu().numpy()
    al = lambda n: (n + 255) // 256 * 256
    keys = ws[:K * M * 8].view(np.uint64).reshape(K, M)
    o = al(K * M * 8)
    T = ws[o:o + M * 8].view(np.float32).reshape(M, 2)
    o += al(M * 8)
    cnt = ws[o:o + K * 4].view(np.int32)
    o += al(K * 4)
    pid = ws[o:o + K * M * 4].view(np.int32).reshape(K, M)
    listed = {(int(pid[k, s]), k): int(keys[k, s]) for k in range(K) for s in range(cnt[k])}
    assert set(listed) == set(pairs), f"{what}: listed pairs {sorted(set(listed) ^ set(pairs))[:8]} differ"
    wrong = []
    for (p, k), key in listed.items():
        r = pairs[(p, k)]
        assert np.array_equal(_bits(T[p, :E]), _bits(r["T"])), f"{what}: mean tag of person {p}"
        exp = (_ordered(r["val"]) << 32) | (~r["idx"] & 0xFFFFFFFF)
        if key != exp:
            wrong.append((p, k, r["idx"], int(~key & 0xFFFFFFFF)))
    assert not wrong, f"{what}: refine argmax (person, joint, want idx, got idx) {wrong[:8]}"


def _dev(scales, half=False):
    return [{k: torch.from_numpy(v).cuda().to(torch.float16 if half else torch.float32) for k, v in s.items()}
            for s in scales]


def _params(case, **kw):
    from hpdecode import ops
    return ops.make_params(1, case["K"], case["H"], case["W"], case["E"], case["M"], DET_THR, TAG_THR,
                           flip_index=case["flip_index"], **kw)


def _run(case, scales_dev, tags, want, what, force_generic=0, num_scales=1):
    from hpdecode import ops
    K, H, W, E, M = case["K"], case["H"], case["W"], case["E"], case["M"]
    p = _params(case, num_scales=num_scales)
    p.force_generic = force_generic
    bufs = ops.DecodeBuffers(1, K, H, W, E, M, "cuda:0", tags=tags)
    _poison(bufs, p)
    ops.run_decode(scales_dev, bufs, p)
    _check(bufs, want, what, M, K, E)
    return bufs


@pytest.mark.parametrize("name", SCENES)
def test_decoder_default_and_tag_map(name):
    """BottomUpDecoder's default (tag-less: interpolated tags, word_tags shuffles) and keep_tag_map=True."""
    from hpdecode import BottomUpDecoder
    case = _case(name)
    K, H, W, E, M = case["K"], case["H"], case["W"], case["E"], case["M"]
    for keep in (False, True):
        dec = BottomUpDecoder(K, M, DET_THR, TAG_THR, "cuda:0", keep_tag_map=keep)
        bufs = dec.buffers(1, H, W, E)
        _poison(bufs, _params(case))
        res = dec.decode(_dev(case["scales"]), (H, W))
        assert (res.bufs.tag_map is None) == (not keep)
        _check(res.bufs, case, f"{name} keep_tag_map={keep}", M, K, E)
        if W % 32 == 0:   # the x2 kernel derived real bounds
            assert bool(torch.isfinite(res.bufs.tag_bmin).any())


@pytest.mark.parametrize("name", SCENES)
def test_generic_kernel_and_heap_topk(name):
    """force_generic = 1: the generic aggregation kernel (+-inf tag bounds) and the literal-heap top-k."""
    case = _case(name)
    for tags in (False, True):
        bufs = _run(case, _dev(case["scales"]), tags, case, f"{name} generic tags={tags}", force_generic=1)
        assert bool((bufs.tag_bmin == -np.inf).all()) and bool((bufs.tag_bmax == np.inf).all())


@pytest.mark.parametrize("name", SCENES)
def test_half_inputs(name):
    """fp16 network outputs: against the oracle on the up-cast values."""
    case = _case(name)
    half = [{k: v.astype(np.float16).astype(np.float32) for k, v in s.items()} for s in case["scales"]]
    want = _oracle(case, half, into={})
    for tags in (False, True):
        _run(case, _dev(case["scales"], half=True), tags, want, f"{name} half tags={tags}")


@pytest.mark.parametrize("name", ["crowd32", "e1_pairwise"])
def test_two_scales_multiscale_kernel(name):
    """Two test scales (agg_nms_ms_kernel, real bounds): the scene at 2x its values next to an all-zero second
    scale (0.75 x the output), so the scale mean is the scene again."""
    case = _case(name)
    H, W = case["H"], case["W"]
    s0 = case["scene"].outputs(case["flip_index"], hm_scale=2.0)
    z = {k: np.zeros((1, case["K"], 3 * H // 8 if "lo" in k else 3 * H // 4, 3 * W // 8 if "lo" in k else 3 * W // 4),
                     np.float32) for k in s0 if "tag" not in k}
    scales = [s0, z]
    want = _oracle(case, scales, into={})
    for r in ("ref", "noref"):
        assert np.array_equal(_bits(want[r]["grouped_joints"]), _bits(case[r]["grouped_joints"]))
    for tags in (False, True):
        bufs = _run(case, _dev(scales), tags, want, f"{name} two scales tags={tags}", num_scales=2)
        assert bool(torch.isfinite(bufs.tag_bmin).float().mean() > 0.5)


@pytest.mark.parametrize("name", SCENES)
def test_aggregated_map_entry(name):
    """hpd_decode with scales == NULL (MPPEHeatmapParser.parse): the bounds are hpd_nms's +-inf."""
    from hpdecode import MPPEHeatmapParser, ops
    case = _case(name)
    K, H, W, E, M = case["K"], case["H"], case["W"], case["E"], case["M"]
    hm, tg = torch.from_numpy(case["hm"])[None].cuda(), torch.from_numpy(case["tg"])[None].cuda()
    bufs = ops.DecodeBuffers(1, K, H, W, E, M, "cuda:0", hm.clone(), tg.clone())
    p = _params(case)
    _poison(bufs, p)
    bufs.agg_hm.copy_(hm)
    bufs.tag_map.copy_(tg)
    ops.run_decode(None, bufs, p)
    _check(bufs, case, f"{name} aggregated maps", M, K, E)
    assert bool((bufs.tag_bmin == -np.inf).all()) and bool((bufs.tag_bmax == np.inf).all())
    gj, ps = MPPEHeatmapParser(K, M, DET_THR, TAG_THR).parse(torch.from_numpy(case["hm"]), torch.from_numpy(case["tg"]))
    assert np.array_equal(_bits(gj), _bits(case["ref"]["grouped_joints"]))
    assert np.array_equal(_bits(ps), _bits(case["ref"]["person_scores"]))


def test_pipeline_with_cuda_graphs():
    """DecodePipeline (tag-less lanes, CUDA graphs) on the crowd scene: every submit's lane is poisoned before it and
    checked after it, so each graph replay must have written its own results."""
    from hpdecode import BottomUpDecoder
    from hpdecode.decoder import DecodePipeline
    case = _case("crowd32")
    K, H, W, E, M = case["K"], case["H"], case["W"], case["E"], case["M"]
    dec = BottomUpDecoder(K, M, DET_THR, TAG_THR, "cuda:0")
    pipe = DecodePipeline(dec, depth=2, use_graphs=True)
    scales = _dev(case["scales"])
    for i in range(4):
        _poison(dec.buffers(1, H, W, E, slot=i % 2), _params(case))
        res = pipe.submit(scales, (H, W))
        pipe.drain()
        _check(res.bufs, case, f"pipeline submit {i}", M, K, E)
    assert pipe.graph_replays == 4


def test_python_port_refine_on_small_scene():
    """The reference's own NumPy refine (oracle/py_port) on the generic scene's maps, against the decode."""
    from hpdecode import BottomUpDecoder
    from oracle import py_port
    case = _case("generic248")
    K, H, W, E, M = case["K"], case["H"], case["W"], case["E"], case["M"]
    gj, ps = py_port.parse(torch.from_numpy(case["hm"]), torch.from_numpy(case["tg"]), M, DET_THR, TAG_THR)
    assert np.array_equal(_bits(gj), _bits(case["ref"]["grouped_joints"]))
    got, gps = BottomUpDecoder(K, M, DET_THR, TAG_THR, "cuda:0").decode(_dev(case["scales"]), (H, W)).to_numpy()[0]
    assert np.array_equal(_bits(got), _bits(gj)) and np.array_equal(_bits(gps), _bits(ps))


# ------------------------------------------------------------------------------------------------------------------
# prefilter invariants
# ------------------------------------------------------------------------------------------------------------------
def _bound_violations(bmin, bmax, t0):
    """Pixels whose first tag component lies outside their 4-row x 32-pixel block's [tag_bmin, tag_bmax], widened by
    the slack refine_scan_kernel applies (the same float32 formula, with the pixel's own tag as T)."""
    K, H, W = t0.shape
    wpr = (W + 31) // 32
    yb, xb = np.arange(H)[:, None] // 4, np.arange(W)[None, :] // 32
    lo, hi = bmin[:, yb, xb], bmax[:, yb, xb]
    with np.errstate(invalid="ignore", over="ignore"):
        slack = (np.float32(1e-4) * ((np.float32(1) + np.abs(t0)).astype(np.float32) +
                                     np.maximum(np.abs(lo), np.abs(hi)))).astype(np.float32)
        out = ((lo - t0).astype(np.float32) > slack) | ((t0 - hi).astype(np.float32) > slack) | np.isnan(lo) | np.isnan(hi)
    assert wpr == bmin.shape[-1]
    return int(out.sum())


def _word_max(a, wpr):
    K, H, W = a.shape
    w = np.full((K, H, wpr * 32), -np.inf, np.float32)
    w[:, :, :W] = a
    return w.reshape(K, H, wpr, 32).max(axis=3)


def _aggregate(scales_np, H, W, E, half, tags, force_generic=0, tag_scale=0):
    from hpdecode import ops
    K = scales_np[0]["hm_lo"].shape[1]
    p = ops.make_params(1, K, H, W, E, 30, 0.05, 0.5, num_scales=len(scales_np), tag_scale=tag_scale)
    p.force_generic = force_generic
    bufs = ops.DecodeBuffers(1, K, H, W, E, 30, "cuda:0", tags=tags)
    _poison(bufs, p)
    ops.run_stage("aggregate_nms", bufs, p, scales=_dev(scales_np, half=half))
    torch.cuda.synchronize()
    return bufs


def _check_prefilter(bufs, scales_np, H, W, half, what, tag_scale=0):
    img = [{k: (v.astype(np.float16) if half else v).astype(np.float32)[0] for k, v in s.items()} for s in scales_np]
    K = img[0]["hm_lo"].shape[0]
    hm, tg = cpu_oracle.aggregate(img, (H, W), tag_scale=tag_scale, flip_index=COCO_FLIP if K == 17 else list(range(K)))
    wpr = (W + 31) // 32
    bmin, bmax = bufs.tag_bmin[0].cpu().numpy(), bufs.tag_bmax[0].cpu().numpy()
    assert bool(np.isfinite(bmin).all() and np.isfinite(bmax).all()), f"{what}: a bound is not finite"
    assert _bound_violations(bmin, bmax, tg[..., 0]) == 0, f"{what}: a tag lies outside its block's bounds"
    assert np.array_equal(bufs.hm_wmax[0].cpu().numpy(), _word_max(hm, wpr)), f"{what}: hm_wmax"
    nm, _ = cpu_oracle.nms(hm)
    assert np.array_equal(bufs.nms_wmax[0].cpu().numpy(), _word_max(nm, wpr)), f"{what}: nms_wmax"
    return hm, tg


def _rand_outputs(lh, lw, E, seed, K=5):
    rng = np.random.default_rng(seed)
    s = {"hm_lo": rng.standard_normal((1, K, lh, lw)), "hm_hi": rng.standard_normal((1, K, 2 * lh, 2 * lw)),
         # tags: smooth ramps plus noise, so that blocks differ and the border rows / columns carry the extremes
         "tag": (rng.standard_normal((1, K, lh, lw)) + np.linspace(-3, 3, lw)[None, None, None, :]
                 + np.linspace(2, -2, lh)[None, None, :, None])}
    if E == 2:
        s.update(hm_lo_f=rng.standard_normal((1, K, lh, lw)), hm_hi_f=rng.standard_normal((1, K, 2 * lh, 2 * lw)),
                 tag_f=rng.standard_normal((1, K, lh, lw)))
    return {k: v.astype(np.float32) for k, v in s.items()}


@pytest.mark.parametrize("lh,lw", [(40, 40), (40, 64), (48, 128)])      # W = 160 / 256 / 512: NW = 1 / 2 / 4
@pytest.mark.parametrize("E", [1, 2])
@pytest.mark.parametrize("half", [False, True])
def test_x2_kernel_bounds_and_word_maxima(lh, lw, E, half):
    """agg_nms_x2_kernel into buffer sets with and without a tag map: every tag inside its block's bounds (borders
    included), word maxima equal to the oracle's, and the generic kernel's bounds exactly -inf / +inf."""
    s = _rand_outputs(lh, lw, E, seed=lh * 7 + lw + E + 100 * half)
    H, W = 4 * lh, 4 * lw
    for tags in (False, True):
        bufs = _aggregate([s], H, W, E, half, tags)
        _check_prefilter(bufs, [s], H, W, half, f"x2 {H}x{W} E={E} half={half} tags={tags}")
    g = _aggregate([s], H, W, E, half, False, force_generic=1)
    assert bool((g.tag_bmin == -np.inf).all()) and bool((g.tag_bmax == np.inf).all())


@pytest.mark.parametrize("H,W,ratios,tag_scale,E", [(256, 384, (0.5, 0.75), 0, 1), (320, 512, (0.25, 0.5), 1, 2)])
def test_multiscale_kernel_bounds_and_word_maxima(H, W, ratios, tag_scale, E):
    rng = np.random.default_rng(H + W)
    scales = []
    for r in ratios:
        hh, hw = int(round(H * r)), int(round(W * r))
        s = _rand_outputs(hh // 2, hw // 2, E, seed=int(rng.integers(1 << 30)))
        scales.append(s)
    for tags in (False, True):
        bufs = _aggregate(scales, H, W, E, False, tags, tag_scale=tag_scale)
        _check_prefilter(bufs, scales, H, W, False, f"ms {H}x{W} tags={tags}", tag_scale=tag_scale)


def test_nms_entry_writes_infinite_bounds():
    from hpdecode import ops
    hm = torch.randn(1, 5, 160, 200, device="cuda:0")
    bufs = ops.DecodeBuffers(1, 5, 160, 200, 1, 30, "cuda:0", hm, torch.empty((0,), device="cuda:0"))
    p = ops.make_params(1, 5, 160, 200, 1, 30, 0.05, 0.5)
    for t in (bufs.tag_bmin, bufs.tag_bmax, bufs.hm_wmax):
        t.fill_(float("nan"))
    ops.run_stage("nms", bufs, p)
    torch.cuda.synchronize()
    assert bool((bufs.tag_bmin == -np.inf).all()) and bool((bufs.tag_bmax == np.inf).all())
    assert np.array_equal(bufs.hm_wmax[0].cpu().numpy(), _word_max(hm[0].cpu().numpy(), 7))


def test_crowd_scene_bounds_are_mostly_finite():
    """On the crowd scene the x2 kernel bounds most blocks: a regression to "no bound" fails here."""
    case = _case("crowd32")
    for tags in (False, True):
        bufs = _aggregate(case["scales"], case["H"], case["W"], case["E"], False, tags)
        _check_prefilter(bufs, case["scales"], case["H"], case["W"], False, f"crowd32 tags={tags}")
        assert np.isfinite(bufs.tag_bmin[0].cpu().numpy()).mean() > 0.9


# ------------------------------------------------------------------------------------------------------------------
# a tag map finer than the output (word_tags' span > 32 branch)
# ------------------------------------------------------------------------------------------------------------------
def test_tag_map_finer_than_output():
    """128 x 128 output from 160-wide hm_hi / tag maps (hm_lo 80): every tag read in refine takes tag_at, since a
    word's 32 pixels span 40 tag columns."""
    from hpdecode import ops
    rng = np.random.default_rng(77)
    K, M, E = 17, 20, 2
    s = {"hm_lo": rng.standard_normal((1, K, 80, 80)) * 0.04, "hm_hi": rng.standard_normal((1, K, 160, 160)) * 0.04,
         "tag": rng.standard_normal((1, K, 160, 160)) * 0.5}
    for k in range(K):
        ys, xs = rng.integers(2, 78, 12), rng.integers(2, 78, 12)
        s["hm_lo"][0, k, ys, xs] = rng.random(12) * 0.6 + 0.3
    s.update(hm_lo_f=s["hm_lo"][:, COCO_FLIP, :, ::-1], hm_hi_f=s["hm_hi"][:, COCO_FLIP, :, ::-1],
             tag_f=rng.standard_normal((1, K, 160, 160)) * 0.5)
    s = {k: np.ascontiguousarray(v, np.float32) for k, v in s.items()}
    hm, tg = cpu_oracle.aggregate([{k: v[0] for k, v in s.items()}], (128, 128), flip_index=COCO_FLIP)
    ref = cpu_oracle.parse(hm, tg, M, 0.1, 0.5)
    noref = cpu_oracle.parse(hm, tg, M, 0.1, 0.5, refine=False)
    assert (_bits(ref["grouped_joints"]) != _bits(noref["grouped_joints"])).any(), "refine changes nothing here"
    want = dict(ref=ref, pairs=_pairs(hm, tg, noref["grouped_joints"]))
    assert len(want["pairs"]) > 0
    for tags in (False, True):
        p = ops.make_params(1, K, 128, 128, E, M, 0.1, 0.5)
        bufs = ops.DecodeBuffers(1, K, 128, 128, E, M, "cuda:0", tags=tags)
        _poison(bufs, p)
        ops.run_decode(_dev([s]), bufs, p)
        _check(bufs, want, f"tag map 160 -> 128 tags={tags}", M, K, E)
        assert np.array_equal(_bits(bufs.agg_hm[0].cpu().numpy()), _bits(hm))
        assert np.array_equal(_bits(bufs.agg_tags[0].cpu().numpy()), _bits(tg))
