"""CPU suite for drawing poses onto frames: closed forms of the NumPy rule (oracle/render_oracle.py) that the kernel is
tested against, the oracle against a per-pixel brute force, argument validation of hpd_render_poses (every rejection
happens before a launch), the C layouts of HpdRenderParams / HpdRenderFrame, and the Python front end (PoseStyle,
PoseRenderer, the op's fake, FrameStream's render argument)."""
import ctypes
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import render_oracle as R
from oracle import track_oracle as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, M, E = 17, 30, 2
RED, GREEN, BLUE, WHITE = (255, 0, 0), (0, 255, 0), (0, 0, 255), (255, 255, 255)


def _style(**kw):
    base = dict(limbs=(), limb_colors=(), joint_color=WHITE, track_colors=(RED, GREEN, BLUE), untracked_color=(9, 9, 9),
                thickness=0.0, joint_radius=0.0, kpt_thr=0.0)
    base.update(kw)
    return SimpleNamespace(**base)


def _person(points, score=0.9):
    """A person with the given joints visible at (x, y) (dict k -> (x, y)); every other joint hidden at 0."""
    xy = np.zeros((K, 2))
    vis = np.zeros(K, bool)
    for k, p in points.items():
        xy[k], vis[k] = p, True
    return xy, vis, score


def _covered(out, color):
    return {(int(x), int(y)) for y, x in zip(*np.nonzero((out == np.array(color, np.uint8)).all(-1)))}


def test_disc_with_an_integer_centre_covers_the_29_lattice_points():
    rec = T.make_records([[_person({0: (10.0, 12.0)})]], K, M, E)[0]
    out = R.render(np.zeros((25, 21, 3), np.uint8), rec, K, M, E, _style(joint_radius=3.0))
    got = _covered(out, WHITE)
    want = {(10 + dx, 12 + dy) for dx in range(-3, 4) for dy in range(-3, 4) if dx * dx + dy * dy <= 9}
    assert len(want) == 29 and got == want


def test_horizontal_limb_covers_its_band_and_round_caps():
    rec = T.make_records([[_person({0: (5.0, 10.0), 1: (25.0, 10.0)})]], K, M, E)[0]
    out = R.render(np.zeros((21, 32, 3), np.uint8), rec, K, M, E,
                   _style(limbs=((0, 1),), limb_colors=(RED,), thickness=4.0))
    want = {(x, y) for x in range(32) for y in range(21)
            if (5 <= x <= 25 and abs(y - 10) <= 2) or (x - 5) ** 2 + (y - 10) ** 2 <= 4 or (x - 25) ** 2 + (y - 10) ** 2 <= 4}
    assert _covered(out, RED) == want
    assert {y for _, y in want} == set(range(8, 13)) and (3, 10) in want and (2, 10) not in want


def test_zero_length_limb_equals_a_disc_of_radius_h():
    pt = (7.3, 8.6)
    rec = T.make_records([[_person({2: pt, 5: pt})]], K, M, E)[0]
    frame = np.zeros((20, 20, 3), np.uint8)
    limb = R.render(frame, rec, K, M, E, _style(limbs=((2, 5),), limb_colors=(RED,), thickness=6.0))
    disc = R.render(frame, T.make_records([[_person({2: pt})]], K, M, E)[0], K, M, E,
                    _style(joint_color=RED, joint_radius=3.0))
    assert np.array_equal(limb, disc) and len(_covered(limb, RED)) > 20


def test_later_persons_and_joints_paint_over_earlier_primitives():
    a = _person({0: (5.0, 5.0), 1: (15.0, 5.0)})
    b = _person({0: (10.0, 0.0), 1: (10.0, 10.0)})
    rec = T.make_records([[a, b]], K, M, E)[0]
    st = _style(limbs=((0, 1),), limb_colors=(RED,), thickness=3.0, joint_radius=1.0)
    ids = np.full(M, -1, np.int32)
    ids[:2] = [0, 1]
    out = R.render(np.zeros((16, 20, 3), np.uint8), rec, K, M, E, st, ids=ids)
    assert tuple(out[5, 10]) == GREEN          # person 1 (id 1) crosses person 0 (id 0) and wins
    assert tuple(out[5, 7]) == RED             # person 0 alone
    assert tuple(out[5, 5]) == WHITE and tuple(out[0, 10]) == WHITE and tuple(out[5, 15]) == WHITE   # joints on top
    ids[1] = -1
    out = R.render(np.zeros((16, 20, 3), np.uint8), rec, K, M, E, st, ids=ids)
    assert tuple(out[5, 10]) == (9, 9, 9)      # untracked
    ids[:2] = [5, 4]                           # 5 % 3 = 2, 4 % 3 = 1
    out = R.render(np.zeros((16, 20, 3), np.uint8), rec, K, M, E, st, ids=ids)
    assert tuple(out[5, 7]) == BLUE and tuple(out[5, 10]) == GREEN


def _garbage_record(n_person=1, flags=0):
    """One visible person, then rows past n_person full of visible-looking garbage."""
    rng = np.random.default_rng(0)
    persons = [_person({0: (4.0, 4.0), 1: (9.0, 4.0)})] + [
        (rng.uniform(0, 12, (K, 2)), np.ones(K, bool), 0.5) for _ in range(M - 1)]
    rec = T.make_records([persons], K, M, E)[0]
    row, oc, op, osc, on, of = T.record_layout(K, M, E)
    rec[on:on + 4].view(np.int32)[0] = n_person
    rec[of:of + 4].view(np.int32)[0] = flags
    return rec


@pytest.mark.parametrize("n_person,flags,drawn", [(1, 0, True), (0, 0, False), (-3, 0, False), (1, 1, False),
                                                  (M, 1, False), (5, 3, False)])
def test_rows_past_n_person_and_fallback_frames_are_not_drawn(n_person, flags, drawn):
    frame = np.random.default_rng(1).integers(0, 256, (14, 14, 3), dtype=np.uint8)
    rec = _garbage_record(1 if n_person == 1 else n_person, flags)
    st = _style(limbs=((0, 1), (2, 3)), limb_colors=(RED, RED), thickness=2.0, joint_radius=1.5)
    out = R.render(frame, rec, K, M, E, st)
    if drawn:
        assert not np.array_equal(out, frame) and tuple(out[4, 6]) == RED
        only = R.render(frame, T.make_records([[_person({0: (4.0, 4.0), 1: (9.0, 4.0)})]], K, M, E)[0], K, M, E, st)
        assert np.array_equal(out, only)      # the garbage rows past n_person changed nothing
    else:
        assert np.array_equal(out, frame)


@pytest.mark.parametrize("bad", ["score", "nan", "inf", "far", "far_neg"])
def test_invisible_joints_draw_nothing(bad):
    frame = np.random.default_rng(2).integers(0, 256, (16, 16, 3), dtype=np.uint8)
    xy = np.full((K, 2), 8.0)
    xy[1] = (12.0, 8.0)
    vis = np.ones(K, bool)
    if bad == "score":
        vis[:] = False                          # poses score 0, at kpt_thr 0
    else:
        v = {"nan": np.nan, "inf": np.inf, "far": 2.0 ** 20 + 2 ** -32, "far_neg": -2.0 ** 21}[bad]
        xy[:, 1 if bad != "far_neg" else 0] = v
    rec = T.make_records([[(xy, vis, 0.9)]], K, M, E)[0]
    st = _style(limbs=((0, 1),), limb_colors=(RED,), thickness=3.0, joint_radius=2.0)
    assert np.array_equal(R.render(frame, rec, K, M, E, st), frame)


def test_kpt_thr_is_strict_and_compared_in_float64():
    xy = np.full((K, 2), 5.0)
    rec = T.make_records([[(xy, np.ones(K, bool), 0.9)]], K, M, E)[0]   # scores 0.5 (float32, exact)
    frame = np.zeros((11, 11, 3), np.uint8)
    assert np.array_equal(R.render(frame, rec, K, M, E, _style(joint_radius=1.0, kpt_thr=0.5)), frame)
    assert tuple(R.render(frame, rec, K, M, E, _style(joint_radius=1.0, kpt_thr=np.nextafter(0.5, 0)))[5, 5]) == WHITE


def test_coords_replace_the_records_coordinates():
    rec = T.make_records([[_person({0: (2.0, 2.0)})]], K, M, E)[0]
    coords = np.zeros((M, K, 2))
    coords[0, 0] = (8.0, 6.0)
    out = R.render(np.zeros((10, 10, 3), np.uint8), rec, K, M, E, _style(joint_radius=0.5), coords=coords)
    assert _covered(out, WHITE) == {(8, 6)}


def _brute(frame, rec, style, ids=None, coords=None):
    """Per pixel, every primitive in paint order with Python floats: the last one that covers it wins."""
    n, xy, score = R.persons(rec, K, M, E)
    if coords is not None:
        xy = coords
    out = frame.copy()
    h, w = frame.shape[:2]
    half, rad = style.thickness / 2, style.joint_radius
    prims = []
    for p in range(n):
        pts = [(float(xy[p, k, 0]), float(xy[p, k, 1])) for k in range(K)]
        vis = [R.visible(x, y, score[p, k], style.kpt_thr) for k, (x, y) in enumerate(pts)]
        col = None if ids is None else (style.track_colors[ids[p] % len(style.track_colors)] if ids[p] >= 0
                                        else style.untracked_color)
        for l, (a, b) in enumerate(style.limbs):
            if half > 0 and vis[a] and vis[b]:
                prims.append(("limb", pts[a], pts[b], col or style.limb_colors[l]))
        for k in range(K):
            if rad > 0 and vis[k]:
                prims.append(("disc", pts[k], None, style.joint_color))
    for r in range(h):
        for c in range(w):
            X, Y = float(c), float(r)
            for kind, (ax, ay), b, col in prims:
                if kind == "disc":
                    cov = (X - ax) * (X - ax) + (Y - ay) * (Y - ay) <= rad * rad
                else:
                    bx, by = b
                    ex, ey = bx - ax, by - ay
                    L2 = ex * ex + ey * ey
                    px, py = X - ax, Y - ay
                    t = px * ex + py * ey
                    if t <= 0:
                        cov = px * px + py * py <= half * half
                    elif t >= L2:
                        cov = (X - bx) * (X - bx) + (Y - by) * (Y - by) <= half * half
                    else:
                        cr = px * ey - py * ex
                        cov = cr * cr <= (half * half) * L2
                if cov:
                    out[r, c] = col
    return out


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_a_per_pixel_brute_force(seed):
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(5, 40)), int(rng.integers(5, 40))
    persons = []
    for _ in range(int(rng.integers(1, 5))):
        xy = rng.uniform(-8, max(h, w) + 8, (K, 2))
        if seed % 2:
            xy = np.round(xy * 2) / 2                     # half-integer coordinates: exact boundary cases
        persons.append((xy, rng.random(K) < 0.8, 0.5))
    rec = T.make_records([persons], K, M, E)[0]
    limbs = tuple(tuple(int(j) for j in rng.choice(K, 2, replace=False)) for _ in range(int(rng.integers(0, 12))))
    palette = [tuple(int(c) for c in rng.integers(0, 256, 3)) for _ in range(40)]
    st = _style(limbs=limbs, limb_colors=palette[:len(limbs)], joint_color=palette[30], track_colors=palette[31:36],
                untracked_color=palette[36], thickness=float(rng.choice([0, 1, 2.5, 4, 7])),
                joint_radius=float(rng.choice([0, 1, 1.5, 3])))
    frame = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    ids = rng.integers(-1, 9, M).astype(np.int32) if seed % 3 else None
    coords = rng.uniform(-4, 40, (M, K, 2)) if seed == 4 else None
    assert np.array_equal(R.render(frame, rec, K, M, E, st, ids, coords), _brute(frame, rec, st, ids, coords))


# ---- C ABI ------------------------------------------------------------------------------------------------------
def _params(**kw):
    from hpdecode import ops
    limbs = [0, 1, 1, 2, 2, 3]
    p = ops.render_params(K, M, E, limbs, [1, 2, 3] * 3, [4, 5, 6], [7, 8, 9] * 4, [0, 0, 0], 3.0, 4.0, 0.0)
    for name, v in kw.items():
        if name == "limb":
            p.limbs[v[0]][0], p.limbs[v[0]][1] = v[1], v[2]
        else:
            setattr(p, name, v)
    return p


def _frames(*specs):
    """HpdRenderFrame array from (in, out, in_stride, out_stride, h, w) tuples (fake device addresses)."""
    from hpdecode import _lib
    arr = (_lib.HpdRenderFrame * len(specs))()
    for a, (i, o, si, so, h, w) in zip(arr, specs):
        setattr(a, "in", i)
        a.out, a.in_stride_row, a.out_stride_row, a.h, a.w = o, si, so, h, w
    return arr


def _rejects(args, what):
    from hpdecode import _lib
    L = _lib.lib()
    rc = L.hpd_render_poses(*args)
    msg = L.hpd_last_error_string()
    assert rc == 1, what
    assert msg.startswith(b"hpd_render_poses"), (what, msg)
    assert L.hpd_last_launch_count() == 0, what
    return msg


IN, OUT, REC = 1 << 30, 1 << 34, 1 << 20
GOOD = (IN, OUT, 300, 300, 50, 100)

BAD_PARAMS = [
    (dict(num_kpts=0), b"num_kpts"), (dict(num_kpts=33), b"num_kpts"), (dict(max_people=0), b"max_people"),
    (dict(max_people=33), b"max_people"), (dict(emb=0), b"emb"), (dict(emb=3), b"emb"),
    (dict(num_limbs=-1), b"num_limbs"), (dict(num_limbs=65), b"num_limbs"), (dict(limb=(1, 0, K)), b"limbs[1]"),
    (dict(limb=(2, -1, 3)), b"limbs[2]"), (dict(limb=(0, 4, 4)), b"limbs[0] joins joint 4 to itself"),
    (dict(thickness=-1.0), b"thickness"), (dict(thickness=1024.5), b"thickness"),
    (dict(thickness=float("nan")), b"thickness"), (dict(thickness=float("inf")), b"thickness"),
    (dict(joint_radius=-0.5), b"joint_radius"), (dict(joint_radius=2e3), b"joint_radius"),
    (dict(joint_radius=float("nan")), b"joint_radius"), (dict(kpt_thr=float("nan")), b"kpt_thr"),
    (dict(kpt_thr=float("-inf")), b"kpt_thr"), (dict(num_track_colors=0), b"num_track_colors"),
    (dict(num_track_colors=33), b"num_track_colors"),
]


@pytest.mark.parametrize("bad,word", BAD_PARAMS)
def test_render_rejects_bad_params(bad, word):
    p = _params(**bad)
    assert word in _rejects((ctypes.byref(p), _frames(GOOD), 1, REC, None, None, None), bad)


def test_limbs_past_num_limbs_are_not_checked_and_bounds_pass():
    """Entries past num_limbs are ignored; 0 and 1024 are valid sizes: the call gets as far as the records check."""
    for kw in (dict(limb=(5, 40, 40)), dict(thickness=0.0, joint_radius=1024.0), dict(thickness=1024.0, joint_radius=0.0),
               dict(num_limbs=0, limb=(0, 0, 0)), dict(num_track_colors=32), dict(kpt_thr=-1e300)):
        p = _params(**kw)
        msg = _rejects((ctypes.byref(p), _frames(GOOD), 1, None, None, None, None), kw)
        assert b"records is NULL" in msg, (kw, msg)


def test_render_rejects_bad_pointers_and_frames():
    p = ctypes.byref(_params())
    g = _frames(GOOD)
    for args, word in (((None, g, 1, REC, None, None, None), b"params"),
                       ((p, g, 0, REC, None, None, None), b"n_frames"),
                       ((p, g, -1, REC, None, None, None), b"n_frames"),
                       ((p, None, 1, REC, None, None, None), b"frames_host"),
                       ((p, g, 1, None, None, None, None), b"records is NULL"),
                       ((p, g, 1, REC + 4, None, None, None), b"records must be 8-byte aligned"),
                       ((p, g, 1, REC, 4098, None, None), b"track_ids must be 4-byte aligned"),
                       ((p, g, 1, REC, 4096, 4100, None), b"coords must be 8-byte aligned")):
        assert word in _rejects(args, word), word
    bad_frames = [((0, OUT, 300, 300, 50, 100), b"frame 0: in / out"), ((IN, 0, 300, 300, 50, 100), b"frame 0: in / out"),
                  ((IN, OUT, 300, 300, 0, 100), b"size"), ((IN, OUT, 300, 300, 50, 0), b"size"),
                  ((IN, OUT, 300, 300, 32768, 100), b"size"), ((IN, OUT, 3 * 32768, 3 * 32768, 5, 32768), b"size"),
                  ((IN, OUT, 299, 300, 50, 100), b"strides"), ((IN, OUT, 300, 299, 50, 100), b"strides"),
                  ((IN, OUT, -300, 300, 50, 100), b"strides"), ((IN, OUT, 300, (1 << 47) + 1, 50, 100), b"strides")]
    for spec, word in bad_frames:
        assert word in _rejects((p, _frames(spec), 1, REC, None, None, None), spec), spec
        msg = _rejects((p, _frames(GOOD, spec), 2, REC, None, None, None), spec)
        assert word.replace(b"frame 0", b"frame 1") in msg and b"frame 1" in msg, (spec, msg)


def test_render_rejects_overlapping_outputs():
    p = ctypes.byref(_params())
    span = 49 * 300 + 300                       # bytes a 50x100 frame with 300-byte rows spans
    cases = [
        ((IN, IN, 300, 300, 50, 100),), ((IN, IN + span - 1, 300, 300, 50, 100),),
        ((IN + span - 1, IN, 300, 300, 50, 100),),
        (GOOD, (IN + (1 << 24), OUT + span - 1, 300, 300, 50, 100)),            # outputs overlap
        (GOOD, (IN + (1 << 24), IN + 5, 300, 300, 50, 100)),                    # frame 1 writes into frame 0's input
        (GOOD, (OUT - span + 1, IN + (1 << 24), 300, 300, 50, 100)),            # frame 0 writes into frame 1's input
    ]
    for specs in cases:
        assert b"overlaps" in _rejects((p, _frames(*specs), len(specs), REC, None, None, None), specs), specs
    # (touching ranges and a shared input are accepted: tests/test_gpu_render.py draws such a call on real buffers)


def test_render_structs_match_c_layout(tmp_path):
    from hpdecode import _lib
    specs = {"HpdRenderParams": ("num_kpts", "max_people", "emb", "num_limbs", "limbs", "limb_rgb", "joint_rgb",
                                 "untracked_rgb", "num_track_colors", "track_rgb", "thickness", "joint_radius",
                                 "kpt_thr"),
             "HpdRenderFrame": ("in", "out", "in_stride_row", "out_stride_row", "h", "w")}
    probe = tmp_path / "probe.c"
    body = []
    for name, fields in specs.items():
        body.append(f'printf("%zu' + " %zu" * len(fields) + f'\\n",sizeof({name}),'
                    + ",".join(f"offsetof({name},{f})" for f in fields) + ");")
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){' + "".join(body)
                     + "return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    lines = subprocess.check_output([str(exe)]).decode().splitlines()
    for line, (name, fields) in zip(lines, specs.items()):
        S = getattr(_lib, name)
        assert [int(x) for x in line.split()] == [ctypes.sizeof(S)] + [getattr(S, f).offset for f in fields], name


# ---- Python -----------------------------------------------------------------------------------------------------
def test_pose_style_defaults_and_validation():
    from hpdecode import PoseStyle
    s = PoseStyle()
    assert (s.thickness, s.joint_radius, s.kpt_thr) == (3.0, 4.0, 0.0) and s.limbs is None
    assert 18 <= len(s.track_colors) <= 32 and len(set(s.track_colors)) == len(s.track_colors)
    with pytest.raises(Exception):
        s.thickness = 1.0                                       # frozen
    from hpdecode.model import COCO_LIMBS
    assert s.resolved_limbs(17) == tuple(COCO_LIMBS) and len(s.resolved_limb_colors(19)) == 19
    with pytest.raises(ValueError, match="limbs are required"):
        s.resolved_limbs(14)
    t = PoseStyle(limbs=[[0, 1], (1, 2)], limb_colors=[[1, 2, 3], (4, 5, 6)], thickness=0, joint_radius=1024)
    assert t.limbs == ((0, 1), (1, 2)) and t.limb_colors == ((1, 2, 3), (4, 5, 6)) and t.thickness == 0.0
    assert t.resolved_limbs(3) == t.limbs
    with pytest.raises(ValueError, match="num_kpts"):
        t.resolved_limbs(2)
    n = PoseStyle(limbs=np.array([[0, 1], [1, 2]]), limb_colors=np.array([[1, 2, 3], [4, 5, 6]], np.uint8),
                  track_colors=np.arange(6, dtype=np.int64).reshape(2, 3), joint_color=np.array([7, 8, 9]))
    assert n.limbs == ((0, 1), (1, 2)) and n.limb_colors == ((1, 2, 3), (4, 5, 6)) and n.joint_color == (7, 8, 9)
    assert n.track_colors == ((0, 1, 2), (3, 4, 5)) and all(type(v) is int for c in n.track_colors for v in c)
    for kw, word in ((dict(limbs=[(0, 0)]), "distinct"), (dict(limbs=[(-1, 2)]), "distinct"),
                     (dict(limbs=[(0, 1)] * 65), "64"), (dict(limb_colors=[(0, 0, 0)]), "one limb colour"),
                     (dict(track_colors=()), "track colours"), (dict(track_colors=[(1, 1, 1)] * 33), "track colours"),
                     (dict(joint_color=(0, 0, 256)), "joint_color"), (dict(untracked_color=(-1, 0, 0)), "untracked"),
                     (dict(thickness=-1), "thickness"), (dict(thickness=1025), "thickness"),
                     (dict(thickness=float("nan")), "thickness"), (dict(joint_radius=float("inf")), "joint_radius"),
                     (dict(kpt_thr=float("nan")), "kpt_thr")):
        with pytest.raises(ValueError, match=word):
            PoseStyle(**kw)
    for kw in (dict(limbs=[(0, 1, 2)]), dict(limbs=[(0.0, 1)]), dict(joint_color=(1, 2)), dict(joint_color=(1.0, 2, 3)), dict(joint_color=(True, 2, 3)),
               dict(thickness="3"), dict(joint_radius=True), dict(kpt_thr=None), dict(track_colors=[5])):
        with pytest.raises(TypeError):
            PoseStyle(**kw)


def test_render_params_from_a_style_pass_the_library_checks():
    from hpdecode import PoseStyle, _lib, ops
    s = PoseStyle()
    limbs = s.resolved_limbs(17)
    p = ops.render_params(17, 30, 2, [j for l in limbs for j in l], [c for col in s.resolved_limb_colors(19) for c in col],
                          list(s.joint_color), [c for col in s.track_colors for c in col], list(s.untracked_color),
                          s.thickness, s.joint_radius, s.kpt_thr)
    assert p.num_limbs == 19 and p.num_track_colors == len(s.track_colors) and tuple(p.limbs[3]) == limbs[3]
    assert b"records is NULL" in _rejects((ctypes.byref(p), _frames(GOOD), 1, None, None, None, None), "style")
    with pytest.raises(_lib.HpdError):
        ops.render_params(17, 30, 2, [0, 1, 2], [0] * 3, [0] * 3, [0] * 3, [0] * 3, 1.0, 1.0, 0.0)


def test_render_op_fake_shapes():
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    import hpdecode  # noqa: F401
    with FakeTensorMode():
        frames = [torch.empty(48, 64, 3, dtype=torch.uint8), torch.empty(7, 5, 3, dtype=torch.uint8)]
        out = torch.ops.hpd.render_poses(frames, torch.empty(2, 100, dtype=torch.uint8), None, None, 17, 30, 2, [0, 1],
                                         [1, 2, 3], [0, 0, 0], [9, 9, 9], [1, 1, 1], 3.0, 4.0, 0.0)
        assert [tuple(o.shape) for o in out] == [(48, 64, 3), (7, 5, 3)] and all(o.dtype == torch.uint8 for o in out)


def test_pose_renderer_fails_loudly_without_cuda():
    import torch
    from hpdecode import PoseRenderer, PoseStyle, _lib
    with pytest.raises(TypeError):
        PoseRenderer(style=3.0)
    with pytest.raises(ValueError, match="limbs are required"):
        PoseRenderer(num_kpts=14)
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.HpdError):
        PoseRenderer(style=PoseStyle())


def test_frame_stream_render_must_be_a_pose_style():
    from hpdecode import FrameStream
    with pytest.raises(TypeError, match="PoseStyle"):
        FrameStream(None, render=True)
    with pytest.raises(TypeError, match="PoseStyle"):
        FrameStream(None, track=True, render={"thickness": 3})
