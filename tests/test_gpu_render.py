"""-m gpu: drawing poses onto frames on the device (hpd_render_poses, PoseRenderer, model.stream(render=...)) against
the NumPy rule (oracle/render_oracle.py), byte for byte.

Every output is poisoned before the call (its row padding included, which must stay poisoned) and every input must be
unchanged after it.  Scenes put persons partly and wholly off the frame and, with integer coordinates and sizes, pixels
exactly on a disc's or a limb's boundary (d^2 = r^2)."""
import math

import numpy as np
import pytest
import torch

from oracle import render_oracle as R
from oracle import track_oracle as T
from oracle.gen_golden_input import image_of

pytestmark = pytest.mark.gpu

POISON = 0xA5


def _style(rng, K, L, thickness, radius, kpt_thr=0.0):
    from hpdecode import PoseStyle
    limbs = [tuple(int(j) for j in rng.choice(K, 2, replace=False)) for _ in range(L)]
    col = lambda: tuple(int(c) for c in rng.integers(0, 256, 3))   # noqa: E731
    return PoseStyle(limbs=limbs, limb_colors=[col() for _ in range(L)], joint_color=col(),
                     track_colors=[col() for _ in range(int(rng.integers(1, 33)))], untracked_color=col(),
                     thickness=thickness, joint_radius=radius, kpt_thr=kpt_thr)


def _scene(rng, h, w, M, K, n_frames, snap):
    """Per frame up to M persons of K joints around the frame (some partly or wholly off it); snap: integer or
    half-integer coordinates (exact boundaries with integer sizes).  Fallback frames and scores below the threshold."""
    frames, fallback = [], set()
    for f in range(n_frames):
        persons = []
        for _ in range(int(rng.integers(0, M + 1))):
            c = rng.uniform(-0.3, 1.3, 2) * (w, h)
            spread = rng.uniform(2, max(4, min(h, w) / 3))
            xy = c + rng.normal(0, spread, (K, 2))
            if rng.random() < 0.05:
                xy += (w + 200, 0)                            # wholly off the frame
            if snap:
                xy = np.round(xy * 2) / 2
            persons.append((xy, rng.random(K) < 0.85, float(np.float32(rng.random()))))
        if rng.random() < 0.08:
            fallback.add(f)
        frames.append(persons)
    return T.make_records(frames, K, M, 2, fallback)


def _frames(rng, shapes, pad_in, pad_out, offset):
    """Inputs (random pixels) and poisoned outputs as strided views: rows pad_* bytes longer than 3w, the base
    ``offset`` bytes into its buffer (odd values give unaligned rows)."""
    ins, outs, keep = [], [], []
    for h, w in shapes:
        views = []
        for pad, poison in ((pad_in, False), (pad_out, True)):
            stride = 3 * w + pad
            buf = torch.empty(offset + h * stride + 16, dtype=torch.uint8, device="cuda")
            if poison:
                buf.fill_(POISON)
            else:
                buf.copy_(torch.from_numpy(rng.integers(0, 256, buf.numel(), dtype=np.uint8)))
            views.append((buf, buf.as_strided((h, w, 3), (stride, 3, 1), offset)))
        (bi, vi), (bo, vo) = views
        ins.append(vi)
        outs.append(vo)
        keep.append((bi, bi.clone(), bo, vo))
    return ins, outs, keep


def _check(style, K, M, recs, ids, coords, ins, outs, keep):
    host_ids = None if ids is None else ids.cpu().numpy()
    host_xy = None if coords is None else coords.cpu().numpy()
    host_recs = recs.cpu().numpy()
    for f, (bi, bi0, bo, vo) in enumerate(keep):
        assert torch.equal(bi, bi0), "input %d changed" % f
        want = R.render(ins[f].cpu().numpy(), host_recs[f], K, M, 2, _Resolved(style, K),
                        None if host_ids is None else host_ids[f], None if host_xy is None else host_xy[f])
        got = vo.cpu().numpy()
        assert np.array_equal(got, want), "frame %d: %d pixels differ" % (f, int((got != want).any(-1).sum()))
        # everything of the output buffer outside the frame's 3w bytes per row is still poisoned
        mask = torch.ones_like(bo, dtype=torch.bool)
        mask.as_strided(vo.shape, vo.stride(), vo.storage_offset()).fill_(False)
        assert bool((bo[mask] == POISON).all()), "frame %d: bytes outside the frame were written" % f


class _Resolved:
    """A PoseStyle with its defaults resolved for K joints, as the renderer resolves them."""

    def __init__(self, style, K):
        self.limbs = style.resolved_limbs(K)
        self.limb_colors = style.resolved_limb_colors(len(self.limbs))
        for n in ("joint_color", "track_colors", "untracked_color", "thickness", "joint_radius", "kpt_thr"):
            setattr(self, n, getattr(style, n))


def _run(style, K, M, recs, ins, outs, ids=None, coords=None):
    from hpdecode import PoseRenderer, _lib, ops
    r = PoseRenderer(K, M, 2, style)
    ops.run_render(r.params, ins, outs, recs, ids, coords)
    assert _lib.lib().hpd_last_launch_count() == math.ceil(len(ins) / 32)
    torch.cuda.synchronize()


CASES = [  # (h, w), n_frames, M, K, L, thickness, radius, ids, coords, pads (in, out, offset), snap
    ((1, 1), 1, 1, 17, 19, 3.0, 4.0, None, False, (0, 0, 0), True),
    ((7, 5), 3, 3, 14, 13, 2.0, 1.0, "ids", False, (1, 3, 1), True),
    ((33, 65), 5, 30, 17, 19, 4.0, 3.0, "ids", True, (0, 5, 3), True),
    ((33, 65), 4, 32, 32, 64, 1.0, 1.5, None, False, (8, 8, 0), False),
    ((480, 640), 2, 30, 17, 19, 3.0, 4.0, None, False, (0, 0, 0), False),
    ((480, 640), 2, 32, 32, 0, 0.0, 30.0, None, False, (2, 7, 5), True),
    ((480, 640), 1, 1, 14, 13, 40.0, 0.0, "ids", True, (0, 0, 0), False),
    ((1080, 1920), 2, 30, 17, 19, 6.0, 8.0, "ids", False, (0, 0, 0), True),
    ((1080, 1920), 1, 32, 32, 64, 13.0, 2.0, "big_ids", False, (3, 0, 1), False),
    ((2160, 3840), 1, 30, 17, 19, 10.0, 12.0, "ids", True, (0, 0, 0), False),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%dx%d-n%d-M%d-K%d-L%d-t%g-r%g-%s%s-pad%s" % (
    c[0] + c[1:7] + (c[7] or "noids", "-coords" if c[8] else "", "_".join(map(str, c[9])))))
def test_render_equals_the_oracle_byte_for_byte(case):
    (h, w), n, M, K, L, th, rad, ids_kind, use_xy, (pad_in, pad_out, off), snap = case
    rng = np.random.default_rng(CASES.index(case))
    style = _style(rng, K, L, th, rad, kpt_thr=float(rng.choice([0.0, 0.2])))
    recs = torch.from_numpy(_scene(rng, h, w, M, K, n, snap)).cuda()
    ids = coords = None
    if ids_kind:
        hi = 1 << 30 if ids_kind == "big_ids" else 40
        ids = torch.from_numpy(rng.integers(-1, hi, (n, M)).astype(np.int32)).cuda()
    if use_xy:
        xy = rng.uniform(-0.2, 1.2, (n, M, K, 2)) * (w, h)
        xy[rng.random((n, M, K)) < 0.05] = np.nan
        coords = torch.from_numpy(np.round(xy) if snap else xy).cuda()
    ins, outs, keep = _frames(rng, [(h, w)] * n, pad_in, pad_out, off)
    _run(style, K, M, recs, ins, outs, ids, coords)
    _check(style, K, M, recs, ids, coords, ins, outs, keep)


def test_exact_boundaries():
    """Integer joints with integer radii and half-widths: pixels at d^2 = r^2 are covered, the next ones are not."""
    from hpdecode import PoseStyle
    K, M = 17, 4
    xy = np.full((K, 2), 40.0)
    xy[1] = (80.0, 40.0)
    xy[2] = (40.0, 70.0)
    xy[3] = (64.0, 72.0)          # joint 0 + 8 * (3, 4): a limb along a 3-4-5 direction
    recs = torch.from_numpy(T.make_records([[(xy, np.ones(K, bool), 0.9)]], K, M, 2)).cuda()
    style = PoseStyle(limbs=[(0, 1), (0, 3)], limb_colors=[(255, 0, 0), (0, 255, 0)], thickness=10.0, joint_radius=5.0)
    rng = np.random.default_rng(0)
    ins, outs, keep = _frames(rng, [(100, 100)], 0, 0, 0)
    _run(style, K, M, recs, ins, outs)
    _check(style, K, M, recs, None, None, ins, outs, keep)
    got = outs[0].cpu().numpy()
    assert tuple(got[45, 60]) == (255, 0, 0) and tuple(got[46, 60]) != (255, 0, 0)     # h = 5: y = 45 on the edge
    assert tuple(got[43, 44]) == style.joint_color and tuple(got[44, 44]) != style.joint_color   # 3-4-5 on the disc
    assert tuple(got[72, 64]) == style.joint_color


@pytest.mark.parametrize("n", [1, 31, 32, 33, 64])
def test_frame_counts_and_launches(n):
    rng = np.random.default_rng(100 + n)
    K, M = 17, 8
    shapes = [(int(rng.integers(1, 90)), int(rng.integers(1, 130))) for _ in range(n)]
    recs = np.concatenate([_scene(rng, h, w, M, K, 1, bool(i % 2)) for i, (h, w) in enumerate(shapes)])
    recs = torch.from_numpy(recs).cuda()
    style = _style(rng, K, 19, 3.0, 2.5)
    ids = torch.from_numpy(rng.integers(-1, 50, (n, M)).astype(np.int32)).cuda()
    ins, outs, keep = _frames(rng, shapes, 3, 1, 1)
    _run(style, K, M, recs, ins, outs, ids)
    _check(style, K, M, recs, ids, None, ins, outs, keep)


def test_touching_ranges_and_a_shared_input_are_accepted():
    """Three frames read one input; each output starts where the previous range ends (no byte in common)."""
    rng = np.random.default_rng(9)
    K, M, h, w = 17, 30, 50, 100
    span = (h - 1) * 3 * w + 3 * w
    buf = torch.full((4 * span,), POISON, dtype=torch.uint8, device="cuda")
    buf[:span].copy_(torch.from_numpy(rng.integers(0, 256, span, dtype=np.uint8)))
    view = lambda i: buf.as_strided((h, w, 3), (3 * w, 3, 1), i * span)   # noqa: E731
    recs = torch.from_numpy(_scene(rng, h, w, M, K, 3, True)).cuda()
    style = _style(rng, K, 19, 3.0, 2.0)
    src = buf[:span].clone()
    _run(style, K, M, recs, [view(0)] * 3, [view(1), view(2), view(3)])
    assert torch.equal(buf[:span], src)
    for f in range(3):
        want = R.render(view(0).cpu().numpy(), recs[f].cpu().numpy(), K, M, 2, _Resolved(style, K))
        assert np.array_equal(view(f + 1).cpu().numpy(), want)


def test_pose_renderer_returns_new_tensors_and_leaves_frames_alone():
    from hpdecode import PoseRenderer, PoseStyle, _lib
    rng = np.random.default_rng(7)
    K, M = 17, 30
    recs = torch.from_numpy(_scene(rng, 120, 160, M, K, 3, False)).cuda()
    frames = [torch.from_numpy(rng.integers(0, 256, (120, 160, 3), dtype=np.uint8)).cuda() for _ in range(3)]
    frames[1] = torch.from_numpy(rng.integers(0, 256, (120, 200, 3), dtype=np.uint8)).cuda()[:, :160]   # a strided view
    before = [f.clone() for f in frames]
    style = PoseStyle()
    out = PoseRenderer(K, M, 2, style, "cuda").render(frames, recs)
    with pytest.raises(_lib.HpdError, match="records on cpu"):
        PoseRenderer(K, M, 2, style).render(frames, recs.cpu())
    for f, b, o, r in zip(frames, before, out, recs.cpu().numpy()):
        assert torch.equal(f, b) and o.is_contiguous() and o.dtype == torch.uint8 and o.shape == f.shape
        assert np.array_equal(o.cpu().numpy(), R.render(f.cpu().numpy(), r, K, M, 2, _Resolved(style, K)))


# ---- model.stream(render=...) -------------------------------------------------------------------------------------
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
    out, base = [], image_of(200, 260, 3)
    for i in range(n):
        h, w = sizes[(i // run) % len(sizes)] if run else sizes[0]
        out.append(np.ascontiguousarray(np.roll(base, 3 * i, axis=1)[:h, :w]))
    return out


def _same(a, b):
    if a is None or b is None:
        return a is b
    if isinstance(a, np.ndarray):
        return (a.dtype == b.dtype and a.shape == b.shape
                and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)))
    return a == b


@pytest.mark.parametrize("cuda_frames", [False, True], ids=["host", "cuda"])
@pytest.mark.parametrize("track,smooth", [(False, False), (True, False), (True, True)], ids=["plain", "track", "smooth"])
@pytest.mark.parametrize("sizes,run", [(((90, 120),), None), (((90, 120), (120, 90)), 5)], ids=["one-size", "resize"])
def test_stream_rendered_equals_the_oracle(_deterministic, cuda_frames, track, smooth, sizes, run):
    from hpdecode import OneEuro, PoseStyle
    model = _model()
    frames = _video(13, sizes, run)
    if cuda_frames:
        frames = [torch.from_numpy(f).cuda() for f in frames]
        before = [f.clone() for f in frames]
    sm = OneEuro(25.0, min_cutoff=0.5) if smooth else None
    style = PoseStyle(thickness=2.0, joint_radius=2.5, track_colors=[(255, 0, 0), (0, 255, 0), (0, 0, 255)])
    kw = dict(batch_size=4, depth=2, track=track, smooth=sm)
    recs = list(model.stream(frames, records=True, render=style, **kw))
    plain = list(model.stream(frames, records=True, **kw))
    res = list(model.stream(frames, render=style, **kw))
    res0 = list(model.stream(frames, **kw))
    drew = 0
    for f, r, p, x, x0 in zip(frames, recs, plain, res, res0):
        host_f = f.cpu().numpy() if cuda_frames else f
        got = r.rendered.cpu().numpy() if cuda_frames else r.rendered
        assert r.rendered.shape == (1,) + host_f.shape and isinstance(r.rendered, torch.Tensor) == cuda_frames
        ids = None if r.track_ids is None else r.track_ids[0]
        xy = None if r.smoothed_coords is None else r.smoothed_coords[0]
        want = R.render(host_f, r.raw[0], 17, 30, 2, _Resolved(style, 17), ids, xy)
        assert np.array_equal(got[0], want)
        drew += int((want != host_f).any())
        # everything else equals the stream without render
        assert np.array_equal(r.raw, p.raw) and _same(r.track_ids, p.track_ids) and _same(r.smoothed_coords,
                                                                                         p.smoothed_coords)
        assert p.rendered is None and x0.rendered is None
        xr = x.rendered.cpu().numpy() if cuda_frames else x.rendered
        assert np.array_equal(xr, want)
        for name in ("kpts_coords", "kpts_scores", "kpts_tags", "obj_scores", "track_ids", "smoothed_coords"):
            assert _same(getattr(x, name), getattr(x0, name)), name
        assert x.raw_image is f and x.limbs == x0.limbs
    assert drew > 0
    if cuda_frames:
        assert all(torch.equal(f, b) for f, b in zip(frames, before))
    else:
        assert all(isinstance(x.rendered, np.ndarray) and x.rendered.flags.owndata for x in res)
