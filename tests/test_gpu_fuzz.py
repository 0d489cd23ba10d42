"""-m gpu: seeded differential test -- the whole decode against the CPU oracle on shapes and parameters the named
workloads do not reach: non-square maps whose width is not a multiple of 128 (partial warps, word rows that are
not a multiple of 4 -> scalar word-maximum loads), K other than 17, every top-k launch variant (8 warps per row,
one warp per row with the second launch for tied rows, the throughput hint), value grids coarse enough to tie inside
and at the boundary of the top M, channels with fewer than M positive peaks, E = 1 and 2, M from 8 to 32."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _case(seed):
    rng = np.random.default_rng(1000 + seed)
    B = int(rng.integers(1, 4))
    K = int(rng.choice([5, 17, 23]))
    M = int(rng.choice([8, 20, 30, 32]))
    flip = bool(rng.integers(0, 2))
    H = int(rng.choice([128, 136, 192, 256, 320]))
    W = int(rng.choice([128, 160, 200, 256, 384]))
    levels = int(rng.choice([0, 8, 64, 1024]))          # 0: continuous values; else peaks on a grid -> ties
    q = (H // 4, W // 4)
    h = (H // 2, W // 2)
    names = ("hm_lo", "hm_hi", "tag") + (("hm_lo_f", "hm_hi_f", "tag_f") if flip else ())
    s = {}
    for n in names:
        shape = (B, K) + (h if "hi" in n else q)
        s[n] = (rng.standard_normal(shape) * (0.5 if "tag" in n else 0.04)).astype(np.float32)
    for b in range(B):
        for k in range(K):
            n_peaks = int(rng.choice([0, 3, 12, 40, 90]))     # 0 / 3 / 12: fewer than M positive peaks
            ys, xs = rng.integers(1, q[0] - 1, n_peaks), rng.integers(1, q[1] - 1, n_peaks)
            amp = rng.random(n_peaks).astype(np.float32) * 0.6 + 0.3
            if levels:
                amp = (np.ceil(amp * levels) / levels).astype(np.float32)
            for n in ("hm_lo",) + (("hm_lo_f",) if flip else ()):
                xx = xs if n == "hm_lo" else q[1] - 1 - xs
                kk = k
                s[n][b, kk, ys, xx] = amp
    if levels:                                                  # the rest on the grid too: plateaus after upsampling
        for n in names:
            if "tag" not in n:
                s[n] = (np.round(s[n] * levels) / levels).astype(np.float32)
    det = float(rng.choice([0.05, 0.1, 0.3]))
    tthr = float(rng.choice([0.2, 0.5, 1.0]))
    mode = int(rng.integers(0, 3))                              # 0: default, 1: one warp per row, 2: throughput hint
    return dict(B=B, K=K, M=M, E=2 if flip else 1, H=H, W=W, scale=s, det=det, tthr=tthr, mode=mode)


@pytest.mark.parametrize("seed", range(60))
def test_random_configuration_matches_oracle(seed, oracle):
    _run_seed(seed, oracle, tags=True)


@pytest.mark.parametrize("seed", range(60))
def test_random_configuration_tagless_matches_oracle(seed, oracle):
    """The same cases through buffer sets without a tag map (the decoder's default): top-k, adjust and refine
    interpolate their tags (tag_at, word_tags) under random K and random flip involutions."""
    _run_seed(seed, oracle, tags=False)


def _run_seed(seed, oracle, tags):
    from hpdecode import ops
    from hpdecode.decoder import Records
    c = _case(seed)
    B, K, M, E, H, W = c["B"], c["K"], c["M"], c["E"], c["H"], c["W"]
    if H * W < 64 * M:
        pytest.skip("below torch's partial_sort regime")
    dev = {k: torch.from_numpy(v).cuda() for k, v in c["scale"].items()}
    flip_index = list(range(K))
    rng = np.random.default_rng(seed)
    if K > 2:                                                   # a random involution as the flip permutation
        pairs = rng.permutation(K)[: 2 * (K // 2)].reshape(-1, 2)
        for a, b2 in pairs:
            flip_index[a], flip_index[b2] = int(b2), int(a)
    bufs = ops.DecodeBuffers(B, K, H, W, E, M, "cuda:0", tags=tags)
    for t in (bufs.agg_hm, bufs.tag_map, bufs.poses, bufs.person_scores):
        if t is not None:
            t.fill_(float("nan"))
    bufs.idx_k.fill_(-1)
    p = ops.make_params(B, K, H, W, E, M, c["det"], c["tthr"], flip_index=flip_index)
    if c["mode"] == 1:
        p.force_generic = 2
    elif c["mode"] == 2:
        p.batches_in_flight = 8
    ops.run_decode([dev], bufs, p)
    torch.cuda.synchronize()
    rec = Records(bufs.records.cpu().numpy(), M, K, E)
    for b in range(B):
        hm_o, tg_o = oracle.aggregate([{k: v[b] for k, v in c["scale"].items()}], (H, W), flip_index=flip_index)
        assert np.array_equal(_bits(bufs.agg_hm[b].cpu().numpy()), _bits(hm_o)), f"seed {seed} image {b}: heatmaps"
        if tags:      # a tag-less set computes agg_tags on demand; its decode read none of it
            assert np.array_equal(_bits(bufs.agg_tags[b].cpu().numpy()), _bits(tg_o)), f"seed {seed} image {b}: tags"
        ref = oracle.parse(hm_o, tg_o, M, c["det"], c["tthr"])
        assert np.array_equal(bufs.idx_k[b].cpu().numpy(), ref["idx_k"]), f"seed {seed} image {b}: top-k indices ({c['mode']})"
        assert np.array_equal(_bits(bufs.scores_k[b].cpu().numpy()), _bits(ref["scores_k"]))
        gj, ps = rec.image(b)
        if ref["fallback"]:
            from hpdecode.decoder import _finish
            wg, wp = _finish(ref["grouped_joints"], ref["person_scores"], 1)
            assert np.array_equal(gj, wg) and np.array_equal(ps, wp)
        else:
            assert gj.shape == ref["grouped_joints"].shape, f"seed {seed} image {b}: persons"
            assert np.array_equal(_bits(gj), _bits(ref["grouped_joints"])), f"seed {seed} image {b}: grouped joints"
            assert np.array_equal(_bits(ps), _bits(ref["person_scores"])), f"seed {seed} image {b}: person scores"
