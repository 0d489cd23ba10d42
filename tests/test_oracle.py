"""CPU suite: the oracle against the committed golden vectors (recorded from the unmodified
reference, oracle/gen_golden.py), the Python port against the same, and the Hungarian restatements
against each other and against scipy's optimal cost."""
import os
import sys

import numpy as np
import pytest

from hpdecode import synth
from oracle import golden_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _load(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


@pytest.mark.parametrize("name", list(golden_cases.CASES))
def test_cpp_oracle_reproduces_reference_goldens(name, oracle):
    g = _load(name)
    scales, size, M, det, tthr = golden_cases.make_inputs(name)
    assert golden_cases.inputs_digest(scales) == str(g["inputs_digest"]), "synthetic generator not reproducible here"
    hm, tg = oracle.aggregate(synth.image_slice(scales, 0), (size, size))
    assert golden_cases.sha(hm) == str(g["agg_hm_sha"])
    assert golden_cases.sha(tg) == str(g["agg_tags_sha"])
    nm, _ = oracle.nms(hm)
    assert golden_cases.sha(nm) == str(g["nms_sha"])
    r = oracle.parse(hm, tg, M, det, tthr)
    assert np.array_equal(r["idx_k"], g["idx_k"])
    assert np.array_equal(_bits(r["scores_k"]), _bits(g["scores_k"]))
    assert np.array_equal(r["coords_k"], g["coords_k"])
    assert np.array_equal(_bits(r["tags_k"]), _bits(g["tags_k"]))
    matched, _ = oracle.match_by_tag(r["tags_k"], r["coords_k"], r["scores_k"], det, tthr)
    if g["matched"].size == 0:
        assert matched.shape[0] == 0 and r["fallback"]
    else:
        assert np.array_equal(_bits(matched), _bits(g["matched"]))
    gj, ps = g["grouped_joints"], g["person_scores"]
    if gj.dtype == np.float64:          # empty-scene fallback: the reference returns float64
        from hpdecode.decoder import _finish
        poses, scores = _finish(r["grouped_joints"], r["person_scores"], 1)
        assert poses.dtype == np.float64 and np.array_equal(poses, gj) and np.array_equal(scores, ps)
    else:
        assert np.array_equal(_bits(r["grouped_joints"]), _bits(gj))
        assert np.array_equal(_bits(r["person_scores"]), _bits(ps))


@pytest.mark.parametrize("name", [n for n in golden_cases.CASES if "512" not in n])
def test_python_port_reproduces_reference_goldens(name):
    from oracle import py_port
    g = _load(name)
    scales, size, M, det, tthr = golden_cases.make_inputs(name)
    hm, tg = py_port.aggregate(synth.image_slice(scales, 0), (size, size))
    assert golden_cases.sha(hm.numpy()) == str(g["agg_hm_sha"])
    assert golden_cases.sha(tg.numpy()) == str(g["agg_tags_sha"])
    gj, ps = py_port.parse(hm, tg, M, det, tthr)
    assert gj.dtype == g["grouped_joints"].dtype
    assert np.array_equal(gj, g["grouped_joints"]) and np.array_equal(ps, g["person_scores"])


def test_munkres_restatements_agree_and_are_optimal(oracle):
    from scipy.optimize import linear_sum_assignment
    sys.path.insert(0, os.path.join(os.path.dirname(GOLDEN), "..", "oracle", "refshim"))
    from oracle.refshim.munkres import Munkres
    rng = np.random.default_rng(5)
    for t in range(300):
        r = int(rng.integers(1, 31))
        c = int(rng.integers(r, 31))
        # the reference's cost structure: rint(dist)*100 - score (score constant along a row) -> heavy ties
        dist = np.round(rng.random((r, c)) * rng.choice([1.5, 3.0, 6.0]))
        M = dist * 100 - rng.random((r, 1))
        if t % 3 == 0 and c > 1:
            M[:, c // 2:] = 1e10
        py = Munkres().compute(M.copy())
        cc = oracle.munkres(M)
        assert [j for _, j in py] == list(cc), f"case {t}: python and C++ restatements disagree"
        ri, ci = linear_sum_assignment(M)
        assert abs(M[np.arange(r), cc].sum() - M[ri, ci].sum()) <= 1e-6 * max(1.0, abs(M[ri, ci].sum()))


def test_bilinear_matches_torch_cpu_on_this_host(oracle):
    """App. A.2: torch's CPU kernel uses this FMA nesting whenever an output side exceeds 64 px
    (smaller outputs take another internal path; no BASELINE config gets there)."""
    import torch
    rng = np.random.default_rng(1)
    for (ih, iw, oh, ow) in [(48, 48, 96, 96), (64, 64, 128, 128), (128, 128, 512, 512), (60, 60, 80, 80),
                             (40, 56, 160, 224), (80, 80, 80, 80), (120, 120, 160, 160),
                             # the resizes of tests/test_gpu_refine.py: the 256 x 256 scenes, the generic scene
                             # (184 x 248), the second scale of the two-scale scene, tag maps finer than the output
                             # (downsampling), the x2 prefilter shapes and the multi-scale prefilter shapes
                             (128, 128, 256, 256), (64, 64, 256, 256), (46, 62, 92, 124), (92, 124, 184, 248),
                             (46, 62, 184, 248), (96, 96, 192, 192), (192, 192, 256, 256), (80, 80, 160, 160),
                             (160, 160, 128, 128), (200, 200, 128, 128), (40, 40, 80, 80), (40, 40, 160, 160),
                             (40, 64, 80, 128), (80, 128, 160, 256), (40, 64, 160, 256), (48, 128, 96, 256),
                             (96, 256, 192, 512), (48, 128, 192, 512), (64, 96, 128, 192), (128, 192, 256, 384),
                             (64, 96, 256, 384), (96, 144, 192, 288), (192, 288, 256, 384), (80, 128, 320, 512),
                             (160, 256, 320, 512)]:
        x = rng.standard_normal((3, ih, iw)).astype(np.float32)
        t = torch.nn.functional.interpolate(torch.from_numpy(x)[None], size=[oh, ow], mode="bilinear",
                                            align_corners=False)[0].numpy()
        assert np.array_equal(_bits(oracle.resize_bilinear(x, oh, ow)), _bits(t)), (ih, iw, oh, ow)


def test_multiscale_aggregate_matches_python_port(oracle):
    from oracle import py_port
    scales = synth.netlike(1, 512, True, seed=31, scales=(0.5, 1.0, 1.5))  # 0.5 -> 64->128: above the 64-px torch quirk
    img = synth.image_slice(scales, 0)
    hm_o, tg_o = oracle.aggregate(img, (512, 512), tag_scale=1)
    hm_p, tg_p = py_port.aggregate(img, (512, 512), tag_scale=1)
    assert np.array_equal(_bits(hm_o), _bits(hm_p.numpy()))
    assert np.array_equal(_bits(tg_o), _bits(tg_p.numpy()))


def test_topk_tie_order_is_heap_history(oracle):
    """All-equal input: the order is libstdc++'s heap permutation, not index order (App. A.4)."""
    import torch
    K, H, W, M = 1, 64, 64, 30
    z = np.zeros((K, H, W), np.float32)
    tags = np.zeros((K, H, W, 1), np.float32)
    _, _, _, idx = oracle.top_k(z, tags, M)
    want = torch.zeros(H * W).topk(M).indices.numpy()
    assert np.array_equal(idx[0], want)
    assert list(idx[0][:6]) == [18, 22, 10, 16, 26, 8]
