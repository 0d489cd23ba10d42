"""-m gpu: group_kernel on its own against the C++ oracle, on the hand-built scenes of oracle/group_scenes.py.

Every scene runs through hpd_group with its outputs poisoned first (poses NaN, n_person / flags -1); all M pose rows
must equal the oracle's bit for bit (rows from n_person on zero), and n_person and flags must match.  Batches of up
to 8 images mix scenes of different families in one launch (one CTA per image: indexing, no state shared between
images).  The non-finite scenes check the cost guard (flags bit 1) against the oracle's statement of it."""
import collections

import numpy as np
import pytest
import torch

from oracle import group_scenes
from test_group_scenes import oracle_match

pytestmark = pytest.mark.gpu

SCENES = group_scenes.all_scenes()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def expected(oracle, s):
    """The oracle's grouping plus hpd_group's empty-scene fallback (grouping.py:262-269): pseudo-person 0 from
    rank 0 of every joint, score 0.01, NaN tags as 0, flags bit 0."""
    K, M, E = s.shape
    poses, n, fl = oracle_match(oracle, s)
    poses[n:] = 0
    if n == 0:
        poses[0, :, 0:2] = s.coords_k[:, 0, :]
        poses[0, :, 2] = np.float32(0.01)
        poses[0, :, 3:] = np.nan_to_num(s.tags_k[:, 0, :], nan=0.0, posinf=np.inf, neginf=-np.inf)
        n, fl = 1, fl | 1
    return poses, n, fl


def run_group(scenes, det_thr, tag_thr, joints_order=None):
    from hpdecode import ops
    K, M, E = scenes[0].shape
    t = torch.from_numpy(np.stack([s.tags_k for s in scenes])).cuda()
    c = torch.from_numpy(np.stack([s.coords_k for s in scenes])).cuda()
    sc = torch.from_numpy(np.stack([s.scores_k for s in scenes])).cuda()
    bufs = ops.DecodeBuffers.for_grouping(sc, c, t)
    bufs.poses.fill_(float("nan"))
    bufs.n_person.fill_(-1)
    bufs.flags.fill_(-1)
    params = ops.make_params(len(scenes), K, 1 << 12, 1 << 12, E, M, det_thr, tag_thr, joints_order=joints_order)
    ops.run_stage("group", bufs, params)
    torch.cuda.synchronize()
    return bufs.poses.cpu().numpy(), bufs.n_person.cpu().numpy(), bufs.flags.cpu().numpy()


def _check(oracle, scenes, poses, n_person, flags, det_thr, tag_thr, joints_order):
    for b, s in enumerate(scenes):
        s = group_scenes.Scene(s.name, s.tags_k, s.coords_k, s.scores_k, det_thr, tag_thr, joints_order, s.finite)
        want, n, fl = expected(oracle, s)
        assert (int(n_person[b]), int(flags[b])) == (n, fl), (b, s.name)
        assert np.array_equal(_bits(poses[b]), _bits(want)), (b, s.name)


@pytest.mark.parametrize("scene", SCENES, ids=[s.name for s in SCENES])
def test_group_kernel_matches_oracle(scene, oracle):
    poses, n_person, flags = run_group([scene], scene.det_thr, scene.tag_thr, scene.joints_order)
    _check(oracle, [scene], poses, n_person, flags, scene.det_thr, scene.tag_thr, scene.joints_order)
    assert bool(flags[0] & 2) == (scene.finite is False and not scene.name.startswith("fallback"))


def _batches():
    """Scenes of one shape (K, M, E) from different families, shuffled, in launches of up to 8 images; the first
    scene's thresholds and joint order apply to the whole launch."""
    by_shape = collections.defaultdict(list)
    for s in SCENES:
        by_shape[s.shape].append(s)
    rng = np.random.default_rng(17)
    out = []
    for shape, ss in sorted(by_shape.items()):
        if len(ss) < 2:
            continue
        ss = [ss[i] for i in rng.permutation(len(ss))]
        for i in range(0, len(ss), 8):
            if len(ss[i:i + 8]) > 1:
                out.append(ss[i:i + 8])
    return out


BATCHES = _batches()


@pytest.mark.parametrize("batch", BATCHES, ids=["+".join(s.name for s in b) for b in BATCHES])
def test_group_kernel_batches_mix_families(batch, oracle):
    first = batch[0]
    poses, n_person, flags = run_group(batch, first.det_thr, first.tag_thr, first.joints_order)
    _check(oracle, batch, poses, n_person, flags, first.det_thr, first.tag_thr, first.joints_order)


def test_batches_cover_several_families():
    fams = {name: {s.name for s in f()} for name, f in group_scenes.FAMILIES.items()}
    mixed = [b for b in BATCHES if len({f for s in b for f, names in fams.items() if s.name in names}) >= 3]
    assert len(mixed) >= 4 and max(len(b) for b in BATCHES) == 8


PUBLIC = ["ties30_m32_p32", "keys_m5_1", "unsorted1", "fallback_e2", "nan_tag_e2", "det_eq_0.1_f64"]


@pytest.mark.parametrize("name", PUBLIC)
def test_public_entry_points(name, oracle):
    """torch.ops.hpd.group and MPPEHeatmapParser.match_by_tag on single scenes (K = 17: the parser's joint order)."""
    from hpdecode import MPPEHeatmapParser
    s = next(x for x in SCENES if x.name == name)
    K, M, E = s.shape
    want, n, fl = expected(oracle, s)
    poses, n_person, flags = torch.ops.hpd.group(torch.from_numpy(s.tags_k[None]).cuda(),
                                                 torch.from_numpy(s.coords_k[None]).cuda(),
                                                 torch.from_numpy(s.scores_k[None]).cuda(), s.det_thr, s.tag_thr,
                                                 1 << 12, 1 << 12)
    assert (int(n_person[0]), int(flags[0])) == (n, fl)
    assert np.array_equal(_bits(poses[0].cpu().numpy()), _bits(want))
    parser = MPPEHeatmapParser(K, M, s.det_thr, s.tag_thr)
    got = parser.match_by_tag(s.tags_k, s.coords_k, s.scores_k)
    if fl & 1:
        assert got.shape[0] == 0           # the reference returns an empty array; parse() builds the fallback
    else:
        assert np.array_equal(_bits(got), _bits(want[:n]))
