"""-m gpu: person tracking on the device (hpd_track, PoseTracker, model.stream(track=True)) against the NumPy tracker
(oracle/track_oracle.py).

CUDA's exp and NumPy's differ by up to 1 ulp, so ids are compared exactly on scenes where the oracle's margins -- every
best OKS against the threshold and, for a match, against the best other OKS -- are larger than that can move them.
Exact ties come from identical poses and are bit-identical on both sides; they are not margins."""
import numpy as np
import pytest
import torch

from oracle import track_oracle as T
from oracle.gen_golden_input import image_of

pytestmark = pytest.mark.gpu

MARGIN = 1e-12
POISON = 0x5A5A5A5A
SIGMAS_14 = np.array([.79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89, .5, .6]) / 10.0


def _scene(seed, n_frames, M, K, max_age, churn=False):
    """Seeded frames: people walk (and cross), appear and disappear, vanish for 1 to max_age + 1 frames, some with few
    visible joints; fallback frames; duplicated persons (exact OKS ties next frame) and duplicated scores.  churn: every
    person jumps every frame, so each frame starts new tracks and the table fills to M * max_age."""
    rng = np.random.default_rng(seed)
    P = M + 8
    shape = np.stack([(rng.random((P, K)) - 0.5) * rng.uniform(40, 200, (P, 1)),
                      (rng.random((P, K)) - 0.5) * rng.uniform(80, 300, (P, 1))], -1)
    pos = rng.uniform(0, 1200, (P, 2))
    vel = rng.normal(0, 8, (P, 2))
    on = rng.random(P) < 0.8
    left = rng.integers(1, 12, P)
    frames, fallback = [], set()
    for f in range(n_frames):
        left -= 1
        for i in np.nonzero(left <= 0)[0]:
            on[i] = not on[i]
            left[i] = rng.integers(3, 14) if on[i] else rng.integers(1, max_age + 2)
        pos += vel
        if churn:
            pos = rng.uniform(0, 5000, (P, 2))
        if rng.random() < 0.06:
            fallback.add(f)
        persons = []
        for i in rng.permutation(np.nonzero(on)[0]):
            xy = pos[i] + shape[i] + rng.normal(0, 1.5, (K, 2))
            vis = rng.random(K) < (0.9 if rng.random() > 0.1 else 0.1)
            score = float(np.float32(rng.choice([rng.random(), 0.5])))     # 0.5: frequent exact score ties
            persons.append((xy, vis, score))
        if persons and rng.random() < 0.15:                                 # an exact duplicate
            xy, vis, score = persons[0]
            persons.append((xy.copy(), vis.copy(), score if rng.random() < 0.5 else score * 0.5))
        frames.append(persons[:M])
    return frames, fallback


def _near_ties(K, M, max_age, oks_thr, kpt_vars):
    """Decisions a hair apart: a person between two tracks 5 px and 5 + 1e-6 px away, and persons whose OKS is 1e-7
    above or below the threshold (found by bisection on the oracle's OKS).  Empty frames drop the tracks between
    groups."""
    rng = np.random.default_rng(7)
    base = np.stack([(rng.random(K) - 0.5) * 80, (rng.random(K) - 0.5) * 160], -1) + 9000
    vis = np.ones(K, bool)
    a = T.area_of(base, vis)
    gap = [[] for _ in range(max_age)]
    frames = list(gap)
    if M >= 2:
        frames += [[(base - [5, 0], vis, 0.9), (base + [5 + 1e-6, 0], vis, 0.8)], [(base, vis, 0.7)]] + gap
        frames += [[(base - [5 + 1e-6, 0], vis, 0.9), (base + [5, 0], vis, 0.8)], [(base, vis, 0.7)]] + gap
    for sign in (1, -1):
        lo, hi = 0.0, 400.0       # OKS falls with the shift
        for _ in range(200):
            mid = (lo + hi) / 2
            if T.oks(base + [mid, 0], vis, a, base, vis, a, kpt_vars) > oks_thr + sign * 1e-7:
                lo = mid
            else:
                hi = mid
        frames += [[(base, vis, 0.9)], [(base + [lo, 0], vis, 0.9)]] + gap
    return frames


def _records(frames, fallback, K, M, E):
    return torch.from_numpy(T.make_records(frames, K, M, E, fallback)).cuda()


def _kernel(recs, p, state, calls):
    """hpd_track over the records in calls of `calls` frames, into poisoned outputs; one launch per call."""
    from hpdecode import _lib, ops
    L = _lib.lib()
    outs = []
    for f0 in range(0, recs.shape[0], calls):
        chunk = recs[f0:f0 + calls]
        out = torch.full((chunk.shape[0], p.max_people), POISON, dtype=torch.int32, device="cuda")
        ops.run_track(p, chunk, state, out)
        assert L.hpd_last_launch_count() == 1
        outs.append(out)
    return torch.cat(outs).cpu().numpy()


def _setup(K, M, E, max_age, min_kp, oks_thr):
    from hpdecode import ops
    sig = T.COCO_SIGMAS if K == 17 else SIGMAS_14
    kv = (sig * 2) ** 2
    p = ops.track_params(K, M, E, max_age, min_kp, oks_thr, kv.tolist())
    state = torch.empty((ops.track_state_bytes(p),), dtype=torch.uint8, device="cuda")
    ops.run_track_reset(p, state, clear_ids=True)
    return p, state, T.Tracker(K, M, E, oks_thr, max_age, min_kp, kv)


CASES = [  # M, K, E, max_age, min_keypoints, oks_thr, churn
    (1, 17, 2, 1, 3, 0.3, False), (1, 14, 1, 3, 3, 0.3, False), (30, 17, 2, 1, 3, 0.3, False),
    (30, 17, 1, 2, 0, 0.3, False), (30, 14, 2, 4, 3, 0.5, False), (32, 17, 2, 8, 3, 0.3, False),
    (32, 14, 1, 5, 14, 0.2, False), (30, 17, 2, 6, 3, 0.3, False), (32, 17, 1, 7, 3, 0.7, False),
    (30, 17, 2, 3, 3, 0.3, False), (30, 17, 2, 8, 3, 0.3, True), (32, 14, 1, 8, 0, 0.3, True), (1, 17, 1, 8, 3, 0.3, True),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "M%d-K%d-E%d-age%d-min%d-thr%g%s" % (c[:6] + ("-churn" if c[6] else "",)))
def test_ids_equal_the_oracle(case):
    M, K, E, max_age, min_kp, thr, churn = case
    frames, fb = _scene(CASES.index(case), 96, M, K, max_age, churn)
    frames += _near_ties(K, M, max_age, thr, ((T.COCO_SIGMAS if K == 17 else SIGMAS_14) * 2) ** 2)
    recs = _records(frames, fb, K, M, E)
    p, state, oracle = _setup(K, M, E, max_age, min_kp, thr)
    want = oracle.update(recs.cpu().numpy())
    assert min(oracle.margins) > MARGIN
    got = _kernel(recs, p, state, recs.shape[0])
    assert np.array_equal(got, want)
    assert (want >= 0).sum() > len(frames) // 2 and want.max() > 0        # the scene does exercise the tracker
    # the same frames again continue the ids (the state carried them)
    more = _kernel(recs, p, state, 64)
    assert np.array_equal(more, oracle.update(recs.cpu().numpy()))
    assert min(oracle.margins) > MARGIN


@pytest.mark.parametrize("case", [CASES[2], CASES[5], CASES[10]], ids=["age1", "age8", "churn"])
def test_call_size_does_not_change_the_ids(case):
    M, K, E, max_age, min_kp, thr, churn = case
    frames, fb = _scene(11, 130, M, K, max_age, churn)
    recs = _records(frames, fb, K, M, E)
    runs = []
    for calls in (1, 3, 8, 64):
        p, state, _ = _setup(K, M, E, max_age, min_kp, thr)
        runs.append(_kernel(recs, p, state, calls))
    for r in runs[1:]:
        assert np.array_equal(r, runs[0])


def test_pose_tracker_reset_keeps_counting():
    from hpdecode import PoseTracker
    frames, fb = _scene(5, 20, 30, 17, 2)
    recs = _records(frames, fb, 17, 30, 2)
    tr = PoseTracker(17, 30, 2, "cuda:0", max_age=2)
    oracle = T.Tracker(17, 30, 2, max_age=2)
    a = tr.update(recs[:10])
    tr.reset()
    b = tr.update(recs[10:])
    want_a = oracle.update(recs[:10].cpu().numpy())
    oracle.reset()
    want_b = oracle.update(recs[10:].cpu().numpy())
    assert a.dtype == torch.int32 and a.is_cuda and tuple(a.shape) == (10, 30)
    assert np.array_equal(a.cpu().numpy(), want_a) and np.array_equal(b.cpu().numpy(), want_b)
    a, b = a.cpu().numpy(), b.cpu().numpy()
    assert b[b >= 0].min() > a.max()
    assert tuple(tr.update(recs[:0]).shape) == (0, 30)


def test_track_op_rejects_foreign_records():
    from hpdecode import PoseTracker, _lib
    tr = PoseTracker(17, 30, 2, "cuda:0")
    row = T.record_layout(17, 30, 2)[0]
    for bad in (torch.zeros((2, row), dtype=torch.uint8), torch.zeros((2, row + 8), dtype=torch.uint8, device="cuda"),
                torch.zeros((2, row), dtype=torch.int32, device="cuda"),
                torch.zeros((2, 2 * row), dtype=torch.uint8, device="cuda")[:, :row]):
        with pytest.raises(_lib.HpdError):
            tr.update(bad)


# ---- model.stream(track=True) -------------------------------------------------------------------------------------
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


def _oracle_ids(raws, sizes):
    """The oracle over the stream's own records in submission order, reset where the frame size changes."""
    tr = T.Tracker(17, 30, 2)
    ids, prev = [], None
    for raw, hw in zip(raws, sizes):
        if prev is not None and hw != prev:
            tr.reset()
        prev = hw
        ids.append(tr.update(raw[None])[0])
    return np.stack(ids), tr


@pytest.mark.parametrize("batch_size", [1, 4])
@pytest.mark.parametrize("depth", [1, 4])
def test_stream_track_ids_equal_the_oracle(_deterministic, batch_size, depth):
    model = _model()
    frames = _video(21)
    recs = list(model.stream(frames, batch_size=batch_size, depth=depth, records=True, track=True))
    raws = [r.raw[0] for r in recs]
    got = np.concatenate([r.track_ids for r in recs])
    want, tr = _oracle_ids(raws, [f.shape for f in frames])
    assert min(tr.margins) > MARGIN
    assert np.array_equal(got, want) and got.dtype == np.int32
    assert (got >= 0).any()
    res = list(model.stream(frames, batch_size=batch_size, depth=depth, track=True))
    for r, rec, ids in zip(res, recs, want):
        P = len(r.obj_scores)
        assert r.track_ids.dtype == np.int32 and np.array_equal(r.track_ids, ids[:P])
        assert np.array_equal(r.kpts_coords, rec.final_coords(0))


def test_stream_size_change_resets_the_tracks(_deterministic):
    model = _model()
    frames = _video(18, sizes=((90, 120), (120, 90)), run=6)
    recs = list(model.stream(frames, batch_size=4, depth=4, records=True, track=True))
    got = np.stack([r.track_ids[0] for r in recs])
    want, tr = _oracle_ids([r.raw[0] for r in recs], [f.shape for f in frames])
    assert min(tr.margins) > MARGIN and np.array_equal(got, want)
    for seg in (6, 12):      # ids after a size change are all new
        before, after = got[:seg], got[seg:seg + 6]
        if (after >= 0).any() and (before >= 0).any():
            assert after[after >= 0].min() > before.max()


def test_stream_without_tracking_has_no_ids(_deterministic):
    model = _model()
    frames = _video(5)
    assert all(r.track_ids is None for r in model.stream(frames, batch_size=2, depth=2))
    assert all(r.track_ids is None for r in model.stream(frames, batch_size=2, depth=2, records=True))
