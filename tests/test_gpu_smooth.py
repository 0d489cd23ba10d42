"""-m gpu: smoothing of tracked joints on the device (hpd_track_smooth, PoseTracker(smoothing=...),
model.stream(track=True, smooth=...)) against the Python filter (oracle/smooth_oracle.py).

The filter has no exp: every step is a correctly rounded float64 operation, so the coordinates are compared bit for
bit.  The oracle is fed the kernel's own ids, so the comparison does not depend on the OKS decisions; the ids
themselves must equal hpd_track's on the same records."""
import numpy as np
import pytest
import torch

from oracle import smooth_oracle as S
from oracle import track_oracle as T
from oracle.gen_golden_input import image_of

pytestmark = pytest.mark.gpu

POISON = 0x5A5A5A5A
SIGMAS_14 = np.array([.79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89, .5, .6]) / 10.0


def _sigmas(K):
    if K == 17:
        return T.COCO_SIGMAS
    if K == 14:
        return SIGMAS_14
    return np.linspace(0.025, 0.107, K)


def _scene(seed, n_frames, M, K, max_age, churn=False):
    """Seeded frames: people move along smooth curved paths with per-frame jitter, appear and disappear, vanish for 1
    to max_age + 1 frames; each joint's visibility flickers; some persons have few visible joints; fallback frames.
    churn: every person jumps every frame, so each frame starts new tracks and the table fills to M * max_age."""
    rng = np.random.default_rng(seed)
    P = M + 8
    shape = np.stack([(rng.random((P, K)) - 0.5) * rng.uniform(40, 200, (P, 1)),
                      (rng.random((P, K)) - 0.5) * rng.uniform(80, 300, (P, 1))], -1)
    c0 = rng.uniform(200, 1000, (P, 2))
    amp, w, ph = rng.uniform(20, 200, (P, 2)), rng.uniform(0.02, 0.15, (P, 2)), rng.uniform(0, 6.3, (P, 2))
    on = rng.random(P) < 0.8
    left = rng.integers(1, 12, P)
    flicker = rng.uniform(0.0, 0.3, (P, K))          # per joint: the chance to be hidden in a frame
    frames, fallback = [], set()
    for f in range(n_frames):
        left -= 1
        for i in np.nonzero(left <= 0)[0]:
            on[i] = not on[i]
            left[i] = rng.integers(3, 14) if on[i] else rng.integers(1, max_age + 2)
        pos = c0 + amp * np.sin(w * f + ph)
        if churn:
            pos = rng.uniform(0, 5000, (P, 2))
        if rng.random() < 0.06:
            fallback.add(f)
        persons = []
        for i in rng.permutation(np.nonzero(on)[0]):
            xy = pos[i] + shape[i] + rng.normal(0, 1.5, (K, 2))
            vis = rng.random(K) >= (flicker[i] if rng.random() > 0.1 else 0.9)
            persons.append((xy, vis, float(np.float32(rng.random()))))
        frames.append(persons[:M])
    return frames, fallback


def _setup(K, M, E, max_age, min_kp, thr, sm):
    from hpdecode import ops
    kv = (_sigmas(K) * 2) ** 2
    p = ops.track_params(K, M, E, max_age, min_kp, thr, kv.tolist())
    sp = ops.smooth_params(*sm)
    state = torch.empty((ops.track_smooth_state_bytes(p),), dtype=torch.uint8, device="cuda")
    ops.run_track_reset(p, state, clear_ids=True)
    plain = torch.empty((ops.track_state_bytes(p),), dtype=torch.uint8, device="cuda")
    ops.run_track_reset(p, plain, clear_ids=True)
    return p, sp, state, plain


def _smooth(recs, p, sp, state, calls):
    """hpd_track_smooth over the records in calls of `calls` frames, into poisoned outputs; one launch per call."""
    from hpdecode import _lib, ops
    L = _lib.lib()
    ids, xy = [], []
    for f0 in range(0, recs.shape[0], calls):
        chunk = recs[f0:f0 + calls]
        n = chunk.shape[0]
        out = torch.full((n, p.max_people), POISON, dtype=torch.int32, device="cuda")
        co = torch.full((n, p.max_people, p.num_kpts, 2), float("nan"), dtype=torch.float64, device="cuda")
        ops.run_track_smooth(p, sp, chunk, state, out, co)
        assert L.hpd_last_launch_count() == 1
        ids.append(out)
        xy.append(co)
    return torch.cat(ids).cpu().numpy(), torch.cat(xy).cpu().numpy()


def _plain(recs, p, state):
    from hpdecode import ops
    out = torch.full((recs.shape[0], p.max_people), POISON, dtype=torch.int32, device="cuda")
    return ops.run_track(p, recs, state, out).cpu().numpy()


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


CASES = [  # M, K, E, max_age, min_keypoints, oks_thr, churn, (fps, min_cutoff, beta, d_cutoff)
    (1, 17, 2, 1, 3, 0.3, False, (30.0, 1.0, 0.0, 1.0)),
    (1, 14, 1, 3, 3, 0.3, False, (25.0, 0.5, 0.01, 1.0)),
    (30, 17, 2, 1, 3, 0.3, False, (30.0, 1.0, 0.0, 1.0)),
    (30, 17, 1, 8, 0, 0.3, False, (60.0, 0.3, 0.05, 2.0)),
    (30, 14, 2, 4, 3, 0.5, False, (24.0, 1.7, 0.7, 0.5)),
    (32, 17, 2, 8, 3, 0.3, False, (29.97, 1.0, 0.007, 1.0)),
    (32, 14, 1, 5, 14, 0.2, False, (120.0, 2.0, 0.0, 3.0)),
    (30, 17, 2, 8, 3, 0.3, True, (30.0, 1.0, 0.1, 1.0)),
    (32, 14, 1, 8, 0, 0.3, True, (15.0, 0.8, 0.0, 1.0)),
    (32, 32, 2, 8, 3, 0.3, False, (30.0, 1.0, 0.02, 1.0)),
    (32, 32, 1, 8, 0, 0.3, True, (50.0, 1.0, 0.5, 1.0)),
]


def _id(c):
    return "M%d-K%d-E%d-age%d-min%d-thr%g%s-fps%g-beta%g" % (c[:6] + ("-churn" if c[6] else "", c[7][0], c[7][2]))


@pytest.mark.parametrize("case", CASES, ids=_id)
def test_coords_equal_the_oracle_bit_for_bit(case):
    M, K, E, max_age, min_kp, thr, churn, sm = case
    frames, fb = _scene(CASES.index(case), 96, M, K, max_age, churn)
    recs = torch.from_numpy(T.make_records(frames, K, M, E, fb)).cuda()
    p, sp, state, plain = _setup(K, M, E, max_age, min_kp, thr, sm)
    ids, xy = _smooth(recs, p, sp, state, recs.shape[0])
    assert np.array_equal(ids, _plain(recs, p, plain))                # smoothing changes no id
    orc = S.OneEuroOracle(K, M, E, *sm)
    host = recs.cpu().numpy()
    assert _same_bits(xy, orc.update(host, ids))
    assert (ids >= 0).sum() > len(frames) // 2                          # the scene does exercise the tracker
    raw = host[:, :8 * M * (3 * K + 1)].view(np.float64).reshape(-1, M, 3 * K + 1)[:, :, :3 * K]
    raw = raw.reshape(-1, M, K, 3)[..., :2]
    assert (xy != raw).any()                                            # ... and the filter
    # the same frames again continue the tracks and the filters (the state carried them)
    ids2, xy2 = _smooth(recs, p, sp, state, 64)
    assert np.array_equal(ids2, _plain(recs, p, plain))
    assert _same_bits(xy2, orc.update(host, ids2))


@pytest.mark.parametrize("case", [CASES[2], CASES[5], CASES[7], CASES[9]], ids=["age1", "age8", "churn", "K32"])
def test_call_size_does_not_change_ids_or_coords(case):
    M, K, E, max_age, min_kp, thr, churn, sm = case
    frames, fb = _scene(11, 130, M, K, max_age, churn)
    recs = torch.from_numpy(T.make_records(frames, K, M, E, fb)).cuda()
    runs = []
    for calls in (1, 3, 8, 64):
        p, sp, state, _ = _setup(K, M, E, max_age, min_kp, thr, sm)
        runs.append(_smooth(recs, p, sp, state, calls))
    orc = S.OneEuroOracle(K, M, E, *sm)
    assert _same_bits(runs[0][1], orc.update(recs.cpu().numpy(), runs[0][0]))
    for ids, xy in runs[1:]:
        assert np.array_equal(ids, runs[0][0]) and _same_bits(xy, runs[0][1])


def test_reset_makes_the_next_frame_raw():
    from hpdecode import ops
    M, K, E, max_age, min_kp, thr, _, sm = CASES[5]
    frames, _ = _scene(3, 40, M, K, max_age)
    recs = torch.from_numpy(T.make_records(frames, K, M, E)).cuda()
    p, sp, state, _ = _setup(K, M, E, max_age, min_kp, thr, sm)
    ids, xy = _smooth(recs[:30], p, sp, state, 30)
    ops.run_track_reset(p, state, clear_ids=False)
    ids2, xy2 = _smooth(recs[30:], p, sp, state, 10)
    host = recs.cpu().numpy()
    raw = host[30, :8 * M * (3 * K + 1)].view(np.float64).reshape(M, 3 * K + 1)[:, :3 * K].reshape(M, K, 3)[..., :2]
    n = int(host[30, T.record_layout(K, M, E)[4]:][:4].view(np.int32)[0])
    assert n > 0 and (ids2[0, :n] >= 0).any() and ids2[0][ids2[0] >= 0].min() > ids.max()
    assert _same_bits(xy2[0, :n], raw[:n]) and (xy2[0, n:] == 0).all()
    orc = S.OneEuroOracle(K, M, E, *sm)
    orc.update(host[:30], ids)
    orc.reset()
    assert _same_bits(xy2, orc.update(host[30:], ids2))


def test_pose_tracker_smoothing():
    from hpdecode import OneEuro, PoseTracker, _lib
    M, K, E = 30, 17, 2
    frames, fb = _scene(5, 24, M, K, 2)
    recs = torch.from_numpy(T.make_records(frames, K, M, E, fb)).cuda()
    sm = OneEuro(30.0, min_cutoff=0.8, beta=0.02)
    tr = PoseTracker(K, M, E, "cuda:0", max_age=2, smoothing=sm)
    ref = PoseTracker(K, M, E, "cuda:0", max_age=2)
    a = tr.update(recs[:8])                               # update() advances the filter too
    b, xy = tr.update_smoothed(recs[8:])
    assert a.dtype == torch.int32 and a.is_cuda and tuple(a.shape) == (8, M)
    assert xy.dtype == torch.float64 and xy.is_cuda and tuple(xy.shape) == (16, M, K, 2)
    assert torch.equal(torch.cat([a, b]), ref.update(recs))
    orc = S.OneEuroOracle(K, M, E, sm.fps, sm.min_cutoff, sm.beta, sm.d_cutoff)
    want = orc.update(recs.cpu().numpy(), torch.cat([a, b]).cpu().numpy())
    assert _same_bits(xy.cpu().numpy(), want[8:])
    tr.reset()
    ids, xy = tr.update_smoothed(recs[:0])
    assert tuple(ids.shape) == (0, M) and tuple(xy.shape) == (0, M, K, 2)
    with pytest.raises(_lib.HpdError, match="without smoothing"):
        ref.update_smoothed(recs[:1])


# ---- model.stream(track=True, smooth=...) -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def _deterministic():
    saved = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = saved


def _model():
    from hpdecode import InferenceKeypointsModel, synth_net
    torch.manual_seed(0)
    return InferenceKeypointsModel(synth_net.HigherHRNet(17, 16), use_flip=True, input_size=128, device="cuda:0")


def _video(n, sizes=((90, 120),), run=None):
    """A panning camera: each frame is the previous one shifted by 3 px; the size changes every ``run`` frames."""
    out, base = [], image_of(200, 260, 3)
    for i in range(n):
        h, w = sizes[(i // run) % len(sizes)] if run else sizes[0]
        out.append(np.ascontiguousarray(np.roll(base, 3 * i, axis=1)[:h, :w]))
    return out


def _oracle_coords(recs, sizes, sm):
    """The filter over the stream's own records and ids in submission order, reset where the frame size changes."""
    orc = S.OneEuroOracle(17, 30, 2, sm.fps, sm.min_cutoff, sm.beta, sm.d_cutoff)
    out, prev = [], None
    for r, hw in zip(recs, sizes):
        if prev is not None and hw != prev:
            orc.reset()
        prev = hw
        out.append(orc.update(r.raw, r.track_ids)[0])
    return np.stack(out)


@pytest.mark.parametrize("batch_size,depth", [(1, 1), (4, 4), (3, 2)])
@pytest.mark.parametrize("sizes,run", [(((90, 120),), None), (((90, 120), (120, 90)), 6)], ids=["one-size", "resize"])
def test_stream_smoothed_coords_equal_the_oracle(_deterministic, batch_size, depth, sizes, run):
    from hpdecode import OneEuro
    model = _model()
    frames = _video(18, sizes, run)
    sm = OneEuro(25.0, min_cutoff=0.5, beta=0.01)
    recs = list(model.stream(frames, batch_size=batch_size, depth=depth, records=True, track=True, smooth=sm))
    got = np.concatenate([r.smoothed_coords for r in recs])
    assert got.dtype == np.float64 and got.shape == (18, 30, 17, 2)
    want = _oracle_coords(recs, [f.shape for f in frames], sm)
    assert _same_bits(got, want)
    tracked = np.concatenate([r.track_ids for r in recs])
    plain = list(model.stream(frames, batch_size=batch_size, depth=depth, records=True, track=True))
    assert np.array_equal(tracked, np.concatenate([r.track_ids for r in plain]))     # the same ids as without smooth
    assert all(r.smoothed_coords is None for r in plain)
    res = list(model.stream(frames, batch_size=batch_size, depth=depth, track=True, smooth=sm))
    for r, rec, xy in zip(res, recs, want):
        P = len(r.obj_scores)
        assert r.smoothed_coords.dtype == r.kpts_coords.dtype and r.smoothed_coords.shape == r.kpts_coords.shape
        assert np.array_equal(r.smoothed_coords, xy[:int(rec.n_person[0])].astype(r.kpts_coords.dtype))
        assert np.array_equal(r.track_ids, rec.track_ids[0, :P])
        assert np.array_equal(r.kpts_coords, rec.final_coords(0))


def test_stream_without_smoothing_has_no_smoothed_coords(_deterministic):
    from hpdecode import OneEuro
    model = _model()
    frames = _video(5)
    assert all(r.smoothed_coords is None for r in model.stream(frames, batch_size=2, depth=2))
    assert all(r.smoothed_coords is None for r in model.stream(frames, batch_size=2, depth=2, records=True))
    assert all(r.smoothed_coords is None for r in model.stream(frames, batch_size=2, depth=2, track=True))
    with pytest.raises(ValueError, match="track"):
        list(model.stream(frames, smooth=OneEuro(30)))
