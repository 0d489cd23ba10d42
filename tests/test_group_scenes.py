"""CPU suite for the grouping scenes of oracle/group_scenes.py: the C++ oracle's match_by_tag equals the Python
port's bit for bit on every finite scene; the scenes reach the branches they are built for (floors on each count,
so a later edit to a builder cannot quietly stop reaching one); the solver never needs more than n step-6 calls
between two augmentations, on the scenes and on the goldens' top-k inputs (the bound group.cu's step-6 cap relies
on); and on non-finite scenes the oracle applies the library's cost guard: it returns, sets flags bit 1, and equals
the Python port whose solver sees the guarded matrix."""
import ctypes
import os

import numpy as np
import pytest

from oracle import golden_cases, group_scenes, py_port

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SCENES = group_scenes.all_scenes()
FINITE = [s for s in SCENES if s.finite]
NON_FINITE = [s for s in SCENES if not s.finite]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def oracle_match(oracle, s):
    """hpo_match_by_tag called directly, with the scene's joint order and the flags output:
    (poses [M,K,3+E] with zero rows from n_person on, n_person, flags)."""
    L = oracle.lib()
    K, M, E = s.shape
    poses = np.full((M, K, 3 + E), np.nan, np.float32)
    n, nt, fl = ctypes.c_int32(-1), ctypes.c_int32(-1), ctypes.c_int32(-1)
    jo = None if s.joints_order is None else np.ascontiguousarray(s.joints_order, np.int32)
    rc = L.hpo_match_by_tag(oracle._p(np.ascontiguousarray(s.tags_k)), oracle._p(np.ascontiguousarray(s.coords_k), ctypes.c_int32),
                            oracle._p(np.ascontiguousarray(s.scores_k)), K, M, E, ctypes.c_double(s.det_thr),
                            ctypes.c_double(s.tag_thr), oracle._p(jo, ctypes.c_int), oracle._p(poses),
                            ctypes.byref(n), ctypes.byref(nt), ctypes.byref(fl))
    assert rc == 0
    return poses, n.value, fl.value


class SolverLog:
    """Wraps the munkres stand-in (the module py_port imports as ``munkres``): per solve, n, the step-6 calls and
    the most step-6 calls between two augmentations (step 5) or before the first."""

    def __init__(self, monkeypatch):
        from munkres import Munkres
        self.solves = []
        compute, step5, step6 = Munkres.compute, Munkres._step5, Munkres._step6
        log = self

        def _compute(self, m):
            log.solves.append(dict(n=max(len(m), len(m[0])), s6=0, run=0, maxrun=0))
            return compute(self, m)

        def _step5(self):
            log.solves[-1]["run"] = 0
            return step5(self)

        def _step6(self):
            d = log.solves[-1]
            d["s6"] += 1
            d["run"] += 1
            d["maxrun"] = max(d["maxrun"], d["run"])
            return step6(self)

        monkeypatch.setattr(Munkres, "compute", _compute)
        monkeypatch.setattr(Munkres, "_step5", _step5)
        monkeypatch.setattr(Munkres, "_step6", _step6)


def _sequential_mean(tl):
    s = np.float32(0)
    for t in tl:
        s = np.float32(s + np.float32(t[0]))
    return np.float32(s / np.float32(len(tl)))


def count_branches(s, trace, solves):
    """What one replayed scene reached, counted the way group.cu branches."""
    K, M, E = s.shape
    c = dict(ordered=0, compaction=0, n32=0, nr_gt_g=0, nr_lt_g=0, half_ties=0, dist_eq_thr=0, beyond_m=0,
             long_solves=0, discriminating_means=0)
    for st in trace:
        sel, tags, keys = st["sel"], st["tags"], st["keys"]
        nr = int(sel.sum())
        c["compaction"] += int(not sel[:nr].all())
        c["beyond_m"] += int(len(keys) > M)
        ok = [False] * nr
        if st["dist"] is not None:
            G = min(len(keys), M)
            n = max(G, nr)
            c["n32"] += int(n == 32)
            c["nr_gt_g"] += int(nr > G)
            c["nr_lt_g"] += int(nr < G)
            d = st["dist"]
            c["half_ties"] += int((d - np.floor(d) == 0.5).sum())
            c["dist_eq_thr"] += int((d == s.tag_thr).sum())
            for r, col in st["pairs"]:
                if r < nr and col < G:
                    ok[r] = bool(d[r][col] < s.tag_thr)
                    if E == 1 and len(st["tag_lists"][col]) >= 8:
                        ds = abs(float(tags[r][0]) - float(_sequential_mean(st["tag_lists"][col])))
                        c["discriminating_means"] += int(ok[r] != (ds < s.tag_thr))
        # group.cu places the step one by one when an unmatched detection's key equals a stored person's key or
        # another unmatched detection's key (+0 == -0)
        new = [np.float32(tags[a][0]) for a in range(nr) if not ok[a]]
        stored = [np.float32(k) for k in keys[:M]]
        c["ordered"] += int(any(t in stored for t in new) or len({float(t) + 0.0 for t in new}) != len(new))
    c["long_solves"] = sum(d["s6"] >= 10 for d in solves)
    return c


@pytest.mark.parametrize("scene", FINITE, ids=[s.name for s in FINITE])
def test_cpp_oracle_equals_python_port(scene, oracle):
    K, M, E = scene.shape
    poses, n, fl = oracle_match(oracle, scene)
    want = py_port.match_by_tag(scene.tags_k, scene.coords_k, scene.scores_k, M, scene.det_thr, scene.tag_thr,
                                joints_order=scene.joints_order)
    assert n == want.shape[0] if want.size else n == 0
    assert np.array_equal(_bits(poses[:n]), _bits(want.reshape(n, K, 3 + E)))
    assert not poses[n:].any()
    assert fl == 0


def test_scenes_reach_their_branches(monkeypatch):
    log = SolverLog(monkeypatch)
    total, most_step6 = {}, 0
    for s in FINITE:
        trace, first = [], len(log.solves)
        K, M, E = s.shape
        py_port.match_by_tag(s.tags_k, s.coords_k, s.scores_k, M, s.det_thr, s.tag_thr, s.joints_order, trace)
        for key, v in count_branches(s, trace, log.solves[first:]).items():
            total[key] = total.get(key, 0) + v
        most_step6 = max(most_step6, sum(d["s6"] for d in log.solves[first:]))
    print(total, "most step-6 calls in one scene:", most_step6)
    # the committed goldens reach: one n = 32 case, at most 124 step-6 calls per case, no compaction
    # the floors sit below what the scenes reach today (570, 51, 187, 178 / 316, 22633, 1923, 318, 105, 54, 235)
    assert total["ordered"] >= 300
    assert total["compaction"] >= 40
    assert total["n32"] >= 150
    assert total["nr_gt_g"] >= 100 and total["nr_lt_g"] >= 200
    assert total["half_ties"] >= 15000
    assert total["dist_eq_thr"] >= 1000
    assert total["beyond_m"] >= 200
    assert total["long_solves"] >= 80
    assert total["discriminating_means"] >= 30
    assert most_step6 > 124


def test_step6_calls_between_augmentations_at_most_n(monkeypatch):
    """With finite costs below 2^63 every step 6 makes a new zero, and each one covers a row or ends in an
    augmentation: so at most n step-6 calls separate two augmentations.  group.cu's cap (n (n + 1) per solve) is
    therefore never reached on such inputs."""
    log = SolverLog(monkeypatch)
    for s in FINITE:
        K, M, E = s.shape
        py_port.match_by_tag(s.tags_k, s.coords_k, s.scores_k, M, s.det_thr, s.tag_thr, s.joints_order)
    for name in golden_cases.CASES:
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        M, det, tthr = golden_cases.CASES[name][3:]
        py_port.match_by_tag(g["tags_k"], g["coords_k"], g["scores_k"], M, det, tthr)
    assert len(log.solves) > 1000
    worst = max(d["maxrun"] / d["n"] for d in log.solves)
    assert worst <= 1.0, worst


def _guarded_munkres():
    from munkres import Munkres

    class Guarded(Munkres):
        """The library's rule: a cost that is not finite or whose magnitude is >= 2^63 becomes 1e10."""

        def compute(self, cost):
            cost = np.asarray(cost, np.float64)
            with np.errstate(invalid="ignore"):
                bad = ~(np.abs(cost) < 2.0 ** 63)
            return super().compute(np.where(bad, 1e10, cost))
    return Guarded


@pytest.mark.parametrize("scene", NON_FINITE, ids=[s.name for s in NON_FINITE])
def test_oracle_guards_non_finite_costs(scene, oracle, monkeypatch):
    """The reference's munkres never returns on these scenes (NaN rows, inf - inf, costs >= 2^63).  The oracle
    returns, flags the image, and equals the Python port whose solver sees the guarded cost matrix."""
    K, M, E = scene.shape
    poses, n, fl = oracle_match(oracle, scene)
    monkeypatch.setattr(py_port, "Munkres", _guarded_munkres())
    with np.errstate(invalid="ignore", over="ignore"):
        want = py_port.match_by_tag(scene.tags_k, scene.coords_k, scene.scores_k, M, scene.det_thr, scene.tag_thr,
                                    joints_order=scene.joints_order)
    assert n == (want.shape[0] if want.size else 0)
    assert np.array_equal(_bits(poses[:n]), _bits(want.reshape(n, K, 3 + E)))
    assert not poses[n:].any()
    if scene.name.startswith("fallback"):
        assert n == 0 and fl == 0          # no detection, no solver: the fallback is the caller's (bit 0)
    else:
        assert fl == 2


def test_guard_leaves_finite_costs_alone(oracle):
    """Costs just below 2^63 in magnitude stay; at 2^63 they are guarded (the sentinel of step 6)."""
    K, M, E = 2, 2, 1
    tags = np.array([[[0.0], [1e3]], [[0.0], [1e3]]], np.float32)
    scores = np.full((K, M), 0.5, np.float32)
    base = group_scenes.Scene("probe", tags, np.zeros((K, M, 2), np.int32), scores, 0.1, 1.0)
    _, n, fl = oracle_match(oracle, base)
    assert (n, fl) == (2, 0)
    # a tag 9.2e16 from a person: rint(d) * 100 = 9.2e18 < 2^63; 9.3e16 -> 9.3e18 >= 2^63
    for t, want in ((9.2e16, 0), (9.3e16, 2)):
        tg = tags.copy()
        tg[1, 1, 0] = np.float32(t)
        _, _, fl = oracle_match(oracle, group_scenes.Scene("probe", tg, base.coords_k, scores, 0.1, 1.0))
        assert fl == want, t
