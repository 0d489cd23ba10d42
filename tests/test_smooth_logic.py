"""CPU suite for the smoothing of tracked joints: known answers of the Python filter (oracle/smooth_oracle.py) that the
kernel is tested against, argument validation of hpd_track_smooth_state_bytes / hpd_track_smooth (every rejection
happens before a launch), the C layout of HpdSmoothParams, and the Python front end (OneEuro, the op's fake)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import smooth_oracle as S
from oracle import track_oracle as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K, M, E = 17, 30, 2


def _person(x, y, vis=None, score=0.9):
    """A person whose every joint sits at (x, y) (numbers that make the closed forms easy to state)."""
    xy = np.tile(np.array([[x, y]], np.float64), (K, 1))
    return xy, np.ones(K, bool) if vis is None else np.asarray(vis, bool), score


def _run(frames, ids, fallback=(), **kw):
    """The filter over synthetic frames with the given ids per frame (a list per frame, one id per person)."""
    recs = T.make_records(frames, K, M, E, fallback)
    full = np.full((len(frames), M), -1, np.int32)
    for f, i in enumerate(ids):
        full[f, :len(i)] = i
    orc = S.OneEuroOracle(K, M, E, **kw)
    return orc, orc.update(recs, full)


def _alpha(cutoff, te):
    r = 2 * math.pi * cutoff * te
    return r / (r + 1)


def test_constant_input_stays_constant():
    _, out = _run([[_person(123.25, 456.5)]] * 20, [[4]] * 20, fps=30.0, min_cutoff=0.7, beta=0.3)
    assert np.allclose(out[:, 0, :, 0], 123.25, rtol=1e-15, atol=0)
    assert np.allclose(out[:, 0, :, 1], 456.5, rtol=1e-15, atol=0)


@pytest.mark.parametrize("fps,fc", [(30.0, 1.0), (60.0, 0.2), (7.5, 3.0)])
def test_step_follows_a_first_order_low_pass(fps, fc):
    """beta = 0: a constant cutoff, so x^_n = 1 - (1 - a)^n for a unit step after the seed."""
    n = 40
    frames = [[_person(0.0, 10.0)]] + [[_person(1.0, 10.0)]] * (n - 1)
    _, out = _run(frames, [[0]] * n, fps=fps, min_cutoff=fc, beta=0.0)
    a = _alpha(fc, 1 / fps)
    want = 1 - (1 - a) ** np.arange(n)
    assert np.allclose(out[:, 0, 3, 0], want, rtol=1e-12, atol=1e-15)
    assert np.allclose(out[:, 0, :, 1], 10.0, rtol=1e-15, atol=0)


@pytest.mark.parametrize("fps,fc", [(30.0, 1.0), (25.0, 2.5)])
def test_ramp_follows_a_first_order_low_pass(fps, fc):
    """beta = 0, x_n = v n: the lag e_n = x_n - x^_n obeys e_n = (1 - a)(e_{n-1} + v), so e_n = v (1-a)(1-(1-a)^n) / a."""
    n, v = 50, 3.0
    _, out = _run([[_person(v * f, 0.0)] for f in range(n)], [[7]] * n, fps=fps, min_cutoff=fc)
    a = _alpha(fc, 1 / fps)
    f = np.arange(n)
    want = v * f - v * (1 - a) * (1 - (1 - a) ** f) / a
    assert np.allclose(out[:, 0, 0, 0], want, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("g", [1, 2, 5])
def test_a_hidden_joint_returns_with_the_gap_in_te(g):
    """Joint 2 is hidden for g frames while the track goes on: on its return te = (g + 1) / fps."""
    hid = np.ones(K, bool)
    hid[2] = False
    frames = [[_person(0.0, 0.0)]] + [[_person(0.0, 0.0, vis=hid)]] * g + [[_person(1.0, 0.0)]]
    _, out = _run(frames, [[0]] * (g + 2), fps=30.0, min_cutoff=1.5)
    assert out[-1, 0, 2, 0] == pytest.approx(_alpha(1.5, (g + 1) / 30.0), rel=1e-14)
    assert out[-1, 0, 3, 0] == pytest.approx(_alpha(1.5, 1 / 30.0), rel=1e-14)
    assert (out[1:-1, 0, 2, 0] == 0.0).all()          # hidden: the raw coordinate


@pytest.mark.parametrize("g", [1, 3])
def test_a_track_refound_after_a_gap_has_the_gap_in_te(g):
    frames = [[_person(0.0, 0.0)]] + [[]] * g + [[_person(1.0, 0.0)]]
    _, out = _run(frames, [[5]] + [[]] * g + [[5]], fps=24.0, min_cutoff=1.0)
    assert out[-1, 0, 0, 0] == pytest.approx(_alpha(1.0, (g + 1) / 24.0), rel=1e-14)


def test_speed_term_raises_the_cutoff():
    """beta > 0 follows a moving joint more closely than beta = 0."""
    frames = [[_person(20.0 * f, 0.0)] for f in range(15)]
    _, slow = _run(frames, [[0]] * 15, fps=30.0, beta=0.0)
    _, fast = _run(frames, [[0]] * 15, fps=30.0, beta=0.05)
    lag = lambda out: 20.0 * 14 - out[-1, 0, 0, 0]       # noqa: E731
    assert 0 < lag(fast) < lag(slow)


def test_untracked_invisible_and_fallback_are_raw_and_padding_is_zero():
    vis = np.ones(K, bool)
    vis[[1, 4]] = False
    frames = [[_person(0.0, 0.0), _person(50.0, 60.0)],
              [_person(10.0, 0.0, vis=vis), _person(70.0, 80.0)],
              [_person(3.0, 4.0)]]
    _, out = _run(frames, [[0, -1], [0, -1], [0]], fallback=(2,), fps=30.0)
    recs = T.make_records(frames, K, M, E, (2,))
    raw = recs[:, :8 * M * (3 * K + 1)].view(np.float64).reshape(3, M, 3 * K + 1)[:, :, :3 * K].reshape(3, M, K, 3)
    assert np.array_equal(out[1, 0, [1, 4]], raw[1, 0, [1, 4], :2])      # invisible joints
    assert not np.array_equal(out[1, 0, 0], raw[1, 0, 0, :2])           # a visible one is filtered
    assert np.array_equal(out[:2, 1], raw[:2, 1, :, :2])                 # id -1
    assert np.array_equal(out[2, 0], raw[2, 0, :, :2]) and (out[2, 0] == 7.0).all()   # the fallback pseudo-person
    assert (out[:2, 2:] == 0).all() and (out[2, 1:] == 0).all()          # rows past n_person


def test_reset_unseeds():
    frames = [[_person(0.0, 0.0)], [_person(1.0, 0.0)], [_person(2.0, 0.0)]]
    orc, _ = _run(frames[:2], [[0], [0]], fps=30.0)
    orc.reset()
    recs = T.make_records(frames[2:], K, M, E)
    out = orc.update(recs, np.array([[0] + [-1] * (M - 1)], np.int32))
    assert (out[0, 0, :, 0] == 2.0).all()


# ---- C ABI ------------------------------------------------------------------------------------------------------
def _tparams(**kw):
    from hpdecode import ops
    p = ops.track_params(K, M, E, 1, 3, 0.3, ((T.COCO_SIGMAS * 2) ** 2).tolist())
    for name, v in kw.items():
        if name == "kpt_vars":
            p.kpt_vars[v[0]] = v[1]
        else:
            setattr(p, name, v)
    return p


def _sparams(**kw):
    from hpdecode import ops
    sp = ops.smooth_params(30.0, 1.0, 0.0, 1.0)
    for name, v in kw.items():
        setattr(sp, name, v)
    return sp


def _rejects(L, fn, args, what):
    rc = getattr(L, fn)(*args)
    msg = L.hpd_last_error_string()
    assert rc == 1, what
    assert msg.startswith(fn.encode()), (what, msg)
    assert L.hpd_last_launch_count() == 0, what
    return msg


def _smooth_bytes(L, p):
    n = ctypes.c_size_t(0)
    assert L.hpd_track_smooth_state_bytes(ctypes.byref(p), ctypes.byref(n)) == 0
    return n.value


BAD_TRACK = [
    (dict(max_age=0), b"max_age"), (dict(max_age=9), b"max_age"), (dict(num_kpts=0), b"num_kpts"),
    (dict(num_kpts=33), b"num_kpts"), (dict(max_people=0), b"max_people"), (dict(max_people=33), b"max_people"),
    (dict(emb=3), b"emb"), (dict(min_keypoints=-1), b"min_keypoints"), (dict(min_keypoints=K + 1), b"min_keypoints"),
    (dict(oks_thr=float("nan")), b"oks_thr"), (dict(kpt_vars=(3, 0.0)), b"kpt_vars[3]"),
    (dict(kpt_vars=(5, float("inf"))), b"kpt_vars[5]"),
]

BAD_SMOOTH = [
    (dict(min_cutoff=0.0), b"min_cutoff"), (dict(min_cutoff=-1.0), b"min_cutoff"), (dict(min_cutoff=2e6), b"min_cutoff"),
    (dict(min_cutoff=float("nan")), b"min_cutoff"), (dict(min_cutoff=float("inf")), b"min_cutoff"),
    (dict(beta=-1e-9), b"beta"), (dict(beta=1.5e6), b"beta"), (dict(beta=float("nan")), b"beta"),
    (dict(beta=float("inf")), b"beta"), (dict(d_cutoff=0.0), b"d_cutoff"), (dict(d_cutoff=-2.0), b"d_cutoff"),
    (dict(d_cutoff=1e7), b"d_cutoff"), (dict(d_cutoff=float("nan")), b"d_cutoff"), (dict(fps=0.0), b"fps"),
    (dict(fps=-30.0), b"fps"), (dict(fps=1e-310), b"fps"), (dict(fps=9.99e-4), b"fps"), (dict(fps=1.1e6), b"fps"),
    (dict(fps=float("nan")), b"fps"), (dict(fps=float("inf")), b"fps"),
]


@pytest.mark.parametrize("bad,word", BAD_TRACK)
def test_smooth_entry_points_reject_bad_track_params(bad, word):
    from hpdecode import _lib
    L = _lib.lib()
    p, sp, n = _tparams(**bad), _sparams(), ctypes.c_size_t(0)
    for fn, args in (("hpd_track_smooth_state_bytes", (ctypes.byref(p), ctypes.byref(n))),
                     ("hpd_track_smooth", (ctypes.byref(p), ctypes.byref(sp), 4096, 4, 1 << 16, 1 << 24, 1 << 20,
                                           1 << 22, None))):
        assert word in _rejects(L, fn, args, bad), (fn, bad)


@pytest.mark.parametrize("bad,word", BAD_SMOOTH)
def test_track_smooth_rejects_bad_smooth_params(bad, word):
    from hpdecode import _lib
    L = _lib.lib()
    p = _tparams()
    need = _smooth_bytes(L, p)
    sp = _sparams(**bad)
    assert word in _rejects(L, "hpd_track_smooth", (ctypes.byref(p), ctypes.byref(sp), 4096, 4, 1 << 16, need, 1 << 20,
                                                    1 << 22, None), bad)


def test_smooth_params_at_their_bounds_pass_validation():
    """The bounds themselves are accepted: the call gets as far as the launch checks (records NULL here)."""
    from hpdecode import _lib
    L = _lib.lib()
    p = _tparams()
    need = _smooth_bytes(L, p)
    for kw in (dict(min_cutoff=1e6, beta=1e6, d_cutoff=1e6, fps=1e6), dict(min_cutoff=5e-324, beta=0.0,
                                                                           d_cutoff=5e-324, fps=1e-3)):
        sp = _sparams(**kw)
        msg = _rejects(L, "hpd_track_smooth", (ctypes.byref(p), ctypes.byref(sp), None, 4, 1 << 16, need, 1 << 20,
                                               1 << 22, None), kw)
        assert b"records is NULL" in msg, (kw, msg)


def test_smooth_entry_points_reject_bad_pointers_and_sizes():
    from hpdecode import _lib
    L = _lib.lib()
    p, sp = _tparams(), _sparams()
    need = _smooth_bytes(L, p)
    plain = ctypes.c_size_t(0)
    assert L.hpd_track_state_bytes(ctypes.byref(p), ctypes.byref(plain)) == 0
    assert need > plain.value
    n = ctypes.c_size_t(0)
    _rejects(L, "hpd_track_smooth_state_bytes", (None, ctypes.byref(n)), "NULL params")
    assert b"out_bytes" in _rejects(L, "hpd_track_smooth_state_bytes", (ctypes.byref(p), None), "NULL out")
    bp, bs = ctypes.byref(p), ctypes.byref(sp)
    rec, st, ids, xy = 4096, 1 << 16, 1 << 24, 1 << 22
    for args, word in (((None, bs, rec, 4, st, need, ids, xy, None), b"params"),
                       ((bp, None, rec, 4, st, need, ids, xy, None), b"smooth params"),
                       ((bp, bs, None, 4, st, need, ids, xy, None), b"records"),
                       ((bp, bs, rec + 4, 4, st, need, ids, xy, None), b"records must be 8-byte aligned"),
                       ((bp, bs, rec, 0, st, need, ids, xy, None), b"n_frames"),
                       ((bp, bs, rec, -1, st, need, ids, xy, None), b"n_frames"),
                       ((bp, bs, rec, 4, st, need, None, xy, None), b"track_ids"),
                       ((bp, bs, rec, 4, st, need, ids + 2, xy, None), b"track_ids must be 4-byte aligned"),
                       ((bp, bs, rec, 4, st, need, ids, None, None), b"coords"),
                       ((bp, bs, rec, 4, st, need, ids, xy + 4, None), b"coords must be 8-byte aligned"),
                       ((bp, bs, rec, 4, None, need, ids, xy, None), b"state"),
                       ((bp, bs, rec, 4, st + 4, need, ids, xy, None), b"state must be 8-byte aligned"),
                       ((bp, bs, rec, 4, st, need - 1, ids, xy, None), b"too small"),
                       ((bp, bs, rec, 4, st, plain.value, ids, xy, None), b"too small")):
        assert word in _rejects(L, "hpd_track_smooth", args, word), word


def test_smooth_state_grows_with_max_age():
    from hpdecode import _lib
    L = _lib.lib()
    def extra(max_age):       # the filters' share of the state
        p = _tparams(max_age=max_age)
        n = ctypes.c_size_t(0)
        assert L.hpd_track_state_bytes(ctypes.byref(p), ctypes.byref(n)) == 0
        return _smooth_bytes(L, p) - n.value

    assert extra(8) == 8 * extra(1) and extra(1) % M == 0 and extra(1) > 0


def test_smooth_params_struct_matches_c_layout(tmp_path):
    from hpdecode import _lib
    probe = tmp_path / "probe.c"
    fields = ("min_cutoff", "beta", "d_cutoff", "fps")
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){printf("%zu'
                     + " %zu" * len(fields) + '\\n",sizeof(HpdSmoothParams),'
                     + ",".join(f"offsetof(HpdSmoothParams,{f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    S_ = _lib.HpdSmoothParams
    assert got == [ctypes.sizeof(S_)] + [getattr(S_, f).offset for f in fields]
    assert ctypes.sizeof(S_) == 32


# ---- Python -----------------------------------------------------------------------------------------------------
def test_one_euro_defaults_and_validation():
    from hpdecode import OneEuro
    oe = OneEuro(30)
    assert (oe.fps, oe.min_cutoff, oe.beta, oe.d_cutoff) == (30.0, 1.0, 0.0, 1.0) and isinstance(oe.fps, float)
    with pytest.raises(Exception):
        oe.fps = 60.0                                    # frozen
    assert OneEuro(1e-3, 1e6, 1e6, 1e6).beta == 1e6
    for kw, word in ((dict(fps=0), "fps"), (dict(fps=-1), "fps"), (dict(fps=1e-4), "fps"), (dict(fps=2e6), "fps"),
                     (dict(fps=float("nan")), "fps"), (dict(fps=30, beta=-1), "beta"),
                     (dict(fps=30, beta=float("inf")), "beta"), (dict(fps=30, min_cutoff=0), "min_cutoff"),
                     (dict(fps=30, d_cutoff=0), "d_cutoff"), (dict(fps=30, d_cutoff=1e7), "d_cutoff"),
                     (dict(fps=30, min_cutoff=float("nan")), "min_cutoff")):
        with pytest.raises(ValueError, match=word):
            OneEuro(**kw)
    for kw in (dict(fps="30"), dict(fps=True), dict(fps=30, beta=None)):
        with pytest.raises(TypeError):
            OneEuro(**kw)


def test_frame_stream_smooth_needs_track():
    from hpdecode import FrameStream, OneEuro
    with pytest.raises(ValueError, match="track"):
        FrameStream(None, smooth=OneEuro(30))
    with pytest.raises(TypeError):
        FrameStream(None, track=True, smooth=30.0)


def test_track_smooth_op_fake_shapes():
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    import hpdecode  # noqa: F401
    with FakeTensorMode():
        ids, xy = torch.ops.hpd.track_smooth(torch.empty(5, 100, dtype=torch.uint8), torch.empty(64, dtype=torch.uint8),
                                             17, 30, 2, 1, 3, 0.3, [0.1] * 17, 30.0, 1.0, 0.0, 1.0)
        assert tuple(ids.shape) == (5, 30) and ids.dtype == torch.int32
        assert tuple(xy.shape) == (5, 30, 17, 2) and xy.dtype == torch.float64


def test_pose_tracker_with_smoothing_fails_loudly_without_cuda():
    import torch
    from hpdecode import OneEuro, PoseTracker, _lib
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.HpdError):
        PoseTracker(smoothing=OneEuro(30))
