"""CPU suite for person tracking: known-answer sequences for the NumPy tracker (oracle/track_oracle.py) that the kernel
is tested against, argument validation of hpd_track_state_bytes / hpd_track_reset / hpd_track (every rejection
happens before a launch), and the C layout of HpdTrackParams."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import track_oracle as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, M, E = 17, 30, 2


def _pose(cx, cy, w=80.0, h=160.0, vis=None, seed=0):
    """A person: K joints spread over a w x h box centred at (cx, cy) (the same shape for a given seed)."""
    rng = np.random.default_rng(seed)
    xy = np.stack([cx + (rng.random(K) - 0.5) * w, cy + (rng.random(K) - 0.5) * h], 1)
    v = np.ones(K, bool) if vis is None else np.asarray(vis, bool)
    return xy, v


def _p(cx, cy, score=0.9, **kw):
    xy, v = _pose(cx, cy, **kw)
    return (xy, v, score)


def _run(frames, fallback=(), **kw):
    tr = T.Tracker(K, M, E, **kw)
    return tr, tr.update(T.make_records(frames, K, M, E, fallback))


def test_walker_keeps_its_id():
    _, ids = _run([[_p(100 + 4 * f, 200)] for f in range(12)])
    assert (ids[:, 0] == 0).all() and (ids[:, 1:] == -1).all()


def test_crossing_people_keep_their_ids():
    frames = [[_p(100 + 10 * f, 200, 0.9, seed=1), _p(300 - 10 * f, 260, 0.8, seed=2)] for f in range(21)]
    _, ids = _run(frames)
    assert (ids[:, 0] == 0).all() and (ids[:, 1] == 1).all()


@pytest.mark.parametrize("max_age,want", [(1, 1), (2, 0), (3, 0)])
def test_one_frame_gap(max_age, want):
    frames = [[_p(100, 200)], [_p(102, 200)], [], [_p(104, 200)]]
    _, ids = _run(frames, max_age=max_age)
    assert list(ids[:, 0]) == [0, 0, -1, want]


def test_two_frame_gap_needs_max_age_3():
    frames = [[_p(100, 200)], [], [], [_p(102, 200)]]
    assert _run(frames, max_age=2)[1][3, 0] == 1
    assert _run(frames, max_age=3)[1][3, 0] == 0


def test_min_keypoints_gives_minus_one_and_no_track():
    few = np.zeros(K, bool)
    few[:2] = True
    three = few.copy()
    three[2] = True
    frames = [[_p(100, 200, vis=few)], [_p(100, 200, vis=three)], [_p(101, 200, vis=three)]]
    tr, ids = _run(frames, min_keypoints=3)
    assert list(ids[:, 0]) == [-1, 0, 0] and tr.next_id == 1
    assert list(_run(frames, min_keypoints=2)[1][:, 0]) == [0, 0, 0]
    assert list(_run(frames, min_keypoints=0)[1][:, 0]) == [0, 0, 0]


@pytest.mark.parametrize("max_age,want", [(1, 1), (2, 0)])
def test_fallback_frame_ages_the_tracks(max_age, want):
    frames = [[_p(100, 200)], [_p(100, 200)], [_p(102, 200)]]
    _, ids = _run(frames, fallback=(1,), max_age=max_age)
    assert (ids[1] == -1).all()
    assert list(ids[[0, 2], 0]) == [0, want]


def test_exact_oks_tie_goes_to_the_lower_id():
    """Two identical poses become tracks 0 and 1; a person next to both matches them with the same OKS, bit for bit,
    and takes id 0; a second such person then takes 1."""
    twin = _pose(100, 200)
    frames = [[(twin[0], twin[1], 0.8), (twin[0].copy(), twin[1], 0.9)],
              [_p(101, 200, 0.7)],
              [_p(101, 200, 0.7), _p(101, 200, 0.6)]]
    tr, ids = _run(frames, max_age=2)
    assert list(ids[0, :2]) == [1, 0]                   # the higher score is visited first and gets id 0
    assert ids[1, 0] == 0
    assert list(ids[2, :2]) == [0, 1]


@pytest.mark.parametrize("first", [0, 1])
def test_exact_score_tie_goes_to_the_lower_index(first):
    same = _pose(100, 200)
    scores = [0.5, 0.5] if first == 0 else [0.4, 0.5]
    frames = [[_p(100, 200, 0.9)], [(same[0], same[1], scores[0]), (same[0].copy(), same[1], scores[1])]]
    _, ids = _run(frames)
    assert ids[1, first] == 0 and ids[1, 1 - first] == 1


def test_ids_are_never_reused_after_reset():
    tr = T.Tracker(K, M, E)
    a = tr.update(T.make_records([[_p(100, 200), _p(400, 200, 0.5, seed=3)]], K, M, E))
    tr.reset()
    b = tr.update(T.make_records([[_p(100, 200)]], K, M, E))
    assert list(a[0, :2]) == [0, 1] and b[0, 0] == 2


def test_oks_matches_the_definition():
    """OKS against its formula (pycocotools' computeOks with the two poses' mean area) on a hand-sized case."""
    xy_d, vis = _pose(100, 200)
    xy_t = xy_d + 3.0
    vis_t = vis.copy()
    vis_t[5:] = False
    var = (T.COCO_SIGMAS * 2) ** 2
    a_d, a_t = T.area_of(xy_d, vis), T.area_of(xy_t, vis_t)
    got = T.oks(xy_d, vis, a_d, xy_t, vis_t, a_t, var)
    s = (a_d + a_t) / 2
    want = np.mean([math.exp(-18.0 / var[k] / (s + 2.0 ** -52) / 2) for k in range(5)])
    assert got == pytest.approx(want, rel=1e-15)
    assert T.oks(xy_d, vis, a_d, xy_t, ~vis, a_t, var) == 0.0
    assert T.area_of(xy_d, np.eye(K, dtype=bool)[0]) == 0.0


def test_oracle_layout_matches_the_library():
    from hpdecode import ops
    for k, m, e in ((17, 30, 2), (14, 1, 1), (32, 32, 2)):
        L = ops.record_layout(k, m, e)
        assert T.record_layout(k, m, e) == (L.row_bytes, L.off_coco, L.off_poses, L.off_person_scores, L.off_n_person,
                                            L.off_flags)


def test_default_sigmas_are_cocoeval_s():
    from hpdecode.cocoeval import COCO_KPT_OKS_SIGMAS
    assert np.array_equal(T.COCO_SIGMAS, COCO_KPT_OKS_SIGMAS)


# ---- C ABI ------------------------------------------------------------------------------------------------------
def _params(**kw):
    from hpdecode import ops
    p = ops.track_params(K, M, E, 1, 3, 0.3, ((T.COCO_SIGMAS * 2) ** 2).tolist())
    for name, v in kw.items():
        if name == "kpt_vars":
            p.kpt_vars[v[0]] = v[1]
        else:
            setattr(p, name, v)
    return p


BAD = [
    (dict(max_age=0), b"max_age"), (dict(max_age=9), b"max_age"), (dict(num_kpts=0), b"num_kpts"),
    (dict(num_kpts=33), b"num_kpts"), (dict(max_people=0), b"max_people"), (dict(max_people=33), b"max_people"),
    (dict(emb=3), b"emb"), (dict(emb=0), b"emb"), (dict(min_keypoints=-1), b"min_keypoints"),
    (dict(min_keypoints=K + 1), b"min_keypoints"), (dict(oks_thr=float("nan")), b"oks_thr"),
    (dict(oks_thr=float("inf")), b"oks_thr"), (dict(kpt_vars=(3, 0.0)), b"kpt_vars[3]"),
    (dict(kpt_vars=(16, -1.0)), b"kpt_vars[16]"), (dict(kpt_vars=(0, float("nan"))), b"kpt_vars[0]"),
    (dict(kpt_vars=(5, float("inf"))), b"kpt_vars[5]"),
]


def _state_bytes(L, p):
    n = ctypes.c_size_t(0)
    assert L.hpd_track_state_bytes(ctypes.byref(p), ctypes.byref(n)) == 0
    return n.value


def _rejects(L, fn, args, who, what):
    rc = getattr(L, fn)(*args)
    msg = L.hpd_last_error_string()
    assert rc == 1, what
    assert msg.startswith(who.encode()), (what, msg)
    assert L.hpd_last_launch_count() == 0, what
    return msg


@pytest.mark.parametrize("bad,word", BAD)
def test_every_entry_point_rejects_bad_params(bad, word):
    from hpdecode import _lib
    L = _lib.lib()
    good = _state_bytes(L, _params())
    p = _params(**bad)
    n = ctypes.c_size_t(0)
    for fn, args in (("hpd_track_state_bytes", (ctypes.byref(p), ctypes.byref(n))),
                     ("hpd_track_reset", (ctypes.byref(p), 4096, 1 << 20, 1, None)),
                     ("hpd_track", (ctypes.byref(p), 4096, 4, 1 << 16, 1 << 20, 1 << 24, None))):
        assert word in _rejects(L, fn, args, fn, bad), (fn, bad)
    assert good > 0


def test_entry_points_reject_bad_pointers_and_sizes():
    from hpdecode import _lib
    L = _lib.lib()
    p = _params()
    need = _state_bytes(L, p)
    n = ctypes.c_size_t(0)
    _rejects(L, "hpd_track_state_bytes", (None, ctypes.byref(n)), "hpd_track_state_bytes", "NULL params")
    _rejects(L, "hpd_track_state_bytes", (ctypes.byref(p), None), "hpd_track_state_bytes", "NULL out")
    bp = ctypes.byref(p)
    for args, word in (((bp, None, need, 1, None), b"NULL"), ((bp, 4096, need - 1, 1, None), b"too small"),
                       ((bp, 4100, need, 0, None), b"aligned")):
        assert word in _rejects(L, "hpd_track_reset", args, "hpd_track_reset", word)
    rec, st, ids = 4096, 1 << 16, 1 << 24
    for args, word in (((None, rec, 4, st, need, ids, None), b"params"), ((bp, None, 4, st, need, ids, None), b"records"),
                       ((bp, rec + 4, 4, st, need, ids, None), b"aligned"), ((bp, rec, 0, st, need, ids, None), b"n_frames"),
                       ((bp, rec, -1, st, need, ids, None), b"n_frames"), ((bp, rec, 4, None, need, ids, None), b"state"),
                       ((bp, rec, 4, st, need - 1, ids, None), b"too small"), ((bp, rec, 4, st, 0, ids, None), b"too small"),
                       ((bp, rec, 4, st + 4, need, ids, None), b"aligned"), ((bp, rec, 4, st, need, None, None), b"track_ids"),
                       ((bp, rec, 4, st, need, ids + 2, None), b"aligned")):
        assert word in _rejects(L, "hpd_track", args, "hpd_track", word), word


def test_state_holds_max_people_times_max_age_tracks():
    from hpdecode import _lib
    L = _lib.lib()
    one = _state_bytes(L, _params(max_age=1))
    eight = _state_bytes(L, _params(max_age=8))
    assert eight - 16 == 8 * (one - 16) and (one - 16) % M == 0


def test_track_params_struct_matches_c_layout(tmp_path):
    from hpdecode import _lib
    probe = tmp_path / "probe.c"
    fields = ("num_kpts", "max_people", "emb", "max_age", "min_keypoints", "reserved_", "oks_thr", "kpt_vars")
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){printf("%zu %d %d'
                     + " %zu" * len(fields) + '\\n",sizeof(HpdTrackParams),HPD_TRACK_MAX_AGE,HPD_ABI_VERSION,'
                     + ",".join(f"offsetof(HpdTrackParams,{f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    S = _lib.HpdTrackParams
    assert got == [ctypes.sizeof(S), _lib.HPD_TRACK_MAX_AGE, _lib.HPD_ABI_VERSION] + [getattr(S, f).offset for f in fields]
    assert ctypes.sizeof(S) == 288


def test_pose_tracker_fails_loudly_without_cuda():
    import torch
    from hpdecode import PoseTracker, _lib
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.HpdError):
        PoseTracker()


def test_track_op_fake_shapes():
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    import hpdecode  # noqa: F401
    with FakeTensorMode():
        out = torch.ops.hpd.track(torch.empty(5, 100, dtype=torch.uint8), torch.empty(64, dtype=torch.uint8), 17, 30, 2,
                                  1, 3, 0.3, [0.1] * 17)
        assert tuple(out.shape) == (5, 30) and out.dtype == torch.int32
