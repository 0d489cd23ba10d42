"""-m gpu: stage-level checks -- specialised vs generic aggregation kernel, strided inputs,
multi-scale aggregation, and the reference's public methods one by one through the drop-in classes."""
import os

import numpy as np
import pytest
import torch

from hpdecode import synth

pytestmark = pytest.mark.gpu


def _dev(scales):
    return [{k: torch.from_numpy(v).cuda() for k, v in s.items()} for s in scales]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _run_aggregate(scales, H, W, E, force_generic, tags_preflipped=False, tag_scale=0):
    from hpdecode import ops
    B = scales[0]["hm_lo"].shape[0]
    bufs = ops.DecodeBuffers(B, 17, H, W, E, 30, "cuda:0")
    for t in (bufs.agg_hm, bufs.agg_tags, bufs.nms_wmax, bufs.hm_wmax):
        t.fill_(float("nan"))
    bufs.nms_mask.fill_(-1)
    p = ops.make_params(B, 17, H, W, E, 30, 0.05, 0.5, num_scales=len(scales), tag_scale=tag_scale,
                        tags_preflipped=tags_preflipped)
    p.force_generic = int(force_generic)
    ops.run_stage("aggregate_nms", bufs, p, scales=scales)
    torch.cuda.synchronize()
    return bufs


def _assert_tag_map_matches_oracle(bufs, scales, H, W, oracle, tag_scale=0):
    """Every image's tag map against the oracle's aggregation of the same inputs."""
    for b in range(bufs.agg_tags.shape[0]):
        _, tg_o = oracle.aggregate([{k: v[b].cpu().numpy() for k, v in s.items()} for s in scales], (H, W),
                                   tag_scale=tag_scale)
        assert np.array_equal(_bits(bufs.agg_tags[b].cpu().numpy()), _bits(tg_o)), f"image {b}: tag map"


def _rand_maps(B, lh, lw, flip, seed):
    g = torch.Generator().manual_seed(seed)
    d = {"hm_lo": torch.randn(B, 17, lh, lw, generator=g), "hm_hi": torch.randn(B, 17, 2 * lh, 2 * lw, generator=g),
         "tag": torch.randn(B, 17, lh, lw, generator=g)}
    if flip:
        d.update(hm_lo_f=torch.randn(B, 17, lh, lw, generator=g), hm_hi_f=torch.randn(B, 17, 2 * lh, 2 * lw, generator=g),
                 tag_f=torch.randn(B, 17, lh, lw, generator=g))
    return {k: v.cuda() for k, v in d.items()}


@pytest.mark.parametrize("lh,lw,flip,B", [(128, 128, True, 2), (128, 128, False, 1), (48, 48, True, 1), (40, 72, True, 1),
                                           (160, 160, True, 1), (64, 176, False, 2), (32, 256, True, 1), (12, 12, True, 1)])
def test_specialised_kernel_is_bit_identical_to_generic(lh, lw, flip, B, oracle):
    """aggregate_nms_x2 vs the generic kernel on every output, incl. borders, partial warps (W % 128 != 0),
    several CTAs per row (W > 512) and tiny maps; the tag map (written by neither: aggregate_tags_kernel) vs the
    oracle."""
    s = _rand_maps(B, lh, lw, flip, seed=lh * 1000 + lw)
    H, W, E = 4 * lh, 4 * lw, 2 if flip else 1
    fast = _run_aggregate([s], H, W, E, False)
    slow = _run_aggregate([s], H, W, E, True)
    _assert_tag_map_matches_oracle(fast, [s], H, W, oracle)
    for name in ("agg_hm", "nms_mask", "nms_wmax", "hm_wmax"):
        a, b = getattr(fast, name).cpu().numpy(), getattr(slow, name).cpu().numpy()
        if name == "nms_wmax":   # prefilter values: the sign of a zero is unspecified
            assert np.array_equal(a, b), f"{name} differs ({lh}x{lw}, flip={flip})"
        else:
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"{name} differs ({lh}x{lw}, flip={flip})"


def test_tags_preflipped_mode():
    """from_preds' calling convention: second tag map already un-flipped / permuted (model.py:91-94)."""
    s = _rand_maps(1, 64, 64, True, seed=9)
    pre = dict(s)
    pre["tag_f"] = torch.flip(s["tag_f"], [3])[:, synth.COCO_FLIP_INDEX].contiguous()
    a = _run_aggregate([s], 256, 256, 2, False)
    for force in (False, True):
        b = _run_aggregate([pre], 256, 256, 2, force, tags_preflipped=True)
        assert torch.equal(a.agg_tags, b.agg_tags)


def test_strided_channel_slice_inputs():
    """hm_lo / tag arrive as channel slices of one 34-channel tensor (higher_hrnet.py:78-79)."""
    g = torch.Generator().manual_seed(3)
    both = torch.randn(2, 34, 64, 64, generator=g).cuda()
    hi = torch.randn(2, 17, 128, 128, generator=g).cuda()
    s_view = {"hm_lo": both[:, :17], "tag": both[:, 17:], "hm_hi": hi}
    s_copy = {k: v.contiguous() for k, v in s_view.items()}
    a = _run_aggregate([s_view], 256, 256, 1, False)
    b = _run_aggregate([s_copy], 256, 256, 1, False)
    c = _run_aggregate([s_view], 256, 256, 1, True)
    for name in ("agg_hm", "agg_tags", "nms_mask"):
        assert torch.equal(getattr(a, name), getattr(b, name)) and torch.equal(getattr(a, name), getattr(c, name))


def test_multiscale_aggregate_matches_oracle(oracle):
    """BASELINE config 3 semantics (scales 0.5/1.0/1.5 + flip, tags from scale 1.0): generic kernel."""
    scales = synth.netlike(1, 512, True, seed=41, scales=(0.5, 1.0, 1.5))
    bufs = _run_aggregate(_dev(scales), 512, 512, 2, False, tag_scale=1)
    hm_o, tg_o = oracle.aggregate(synth.image_slice(scales, 0), (512, 512), tag_scale=1)
    assert np.array_equal(_bits(bufs.agg_hm[0].cpu().numpy()), _bits(hm_o))
    assert np.array_equal(_bits(bufs.agg_tags[0].cpu().numpy()), _bits(tg_o))
    nm, keep = oracle.nms(hm_o)
    mask = bufs.nms_mask[0].cpu().numpy().view(np.uint32)
    bits = ((mask[..., None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(17, 512, -1)
    assert np.array_equal(bits.astype(np.uint8), keep)


def test_resize_op_matches_oracle(oracle):
    g = torch.Generator().manual_seed(5)
    for (ih, iw, oh, ow) in [(64, 64, 128, 128), (128, 96, 512, 384), (120, 120, 160, 160), (80, 80, 80, 80)]:
        x = torch.randn(2, 5, ih, iw, generator=g)
        got = torch.ops.hpd.resize_bilinear(x.cuda(), oh, ow).cpu().numpy()
        assert np.array_equal(_bits(got), _bits(oracle.resize_bilinear(x.numpy(), oh, ow)))


def test_parser_api_matches_oracle(oracle):
    """The reference's public methods one by one: nms, top_k, match_by_tag, adjust, refine, parse."""
    from hpdecode import MPPEHeatmapParser
    scales = synth.crowd(1, 256, persons=14, flip=True, seed=51)
    hm, tg = oracle.aggregate(synth.image_slice(scales, 0), (256, 256))
    parser = MPPEHeatmapParser(17, 30, 0.05, 0.5)
    thm, ttg = torch.from_numpy(hm), torch.from_numpy(tg)      # CPU tensors are accepted like in the reference
    nm, _ = oracle.nms(hm)
    assert np.array_equal(_bits(parser.nms(thm[None])[0].cpu().numpy()), _bits(nm))
    tags_k, coords_k, scores_k = parser.top_k(thm, ttg)
    ref = oracle.parse(hm, tg, 30, 0.05, 0.5)
    assert np.array_equal(coords_k, ref["coords_k"]) and coords_k.dtype == np.int32
    assert np.array_equal(_bits(tags_k), _bits(ref["tags_k"])) and np.array_equal(_bits(scores_k), _bits(ref["scores_k"]))
    matched = parser.match_by_tag(tags_k, coords_k, scores_k)
    want, _ = oracle.match_by_tag(ref["tags_k"], ref["coords_k"], ref["scores_k"], 0.05, 0.5)
    assert np.array_equal(_bits(matched), _bits(want))
    gj, ps = parser.parse(thm, ttg)
    assert np.array_equal(_bits(gj), _bits(ref["grouped_joints"])) and np.array_equal(_bits(ps), _bits(ref["person_scores"]))
    no_refine = oracle.parse(hm, tg, 30, 0.05, 0.5, refine=False)["grouped_joints"]
    adj = parser.adjust(matched.copy(), hm)
    assert np.array_equal(_bits(adj), _bits(no_refine))
    person = adj[0].copy()
    assert np.array_equal(_bits(parser.refine(hm, tg, person)), _bits(ref["grouped_joints"][0]))


def test_from_preds_and_fallback_dtype(oracle):
    """from_preds receives flip-averaged heatmaps and [tag, unflipped flip tag] like the reference; an empty
    scene returns the float64 pseudo-person (grouping.py:262-269)."""
    from hpdecode import InferenceKeypointsResult
    from oracle import golden_cases
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "empty256_fallback.npz"))
    scales, size, M, det, tthr = golden_cases.make_inputs("empty256_fallback")
    s = {k: torch.from_numpy(v) for k, v in scales[0].items()}
    FL = synth.COCO_FLIP_INDEX
    hms = [(s["hm_lo"] + torch.flip(s["hm_lo_f"], [3])[:, FL]) / 2, (s["hm_hi"] + torch.flip(s["hm_hi_f"], [3])[:, FL]) / 2]
    tags = [s["tag"], torch.flip(s["tag_f"], [3])[:, FL].contiguous()]
    res = InferenceKeypointsResult.from_preds(None, None, torch.zeros(3, size, size), [h.cuda() for h in hms],
                                              [t.cuda() for t in tags], [], (size, size), (size // 2, size // 2), det, tthr, M)
    assert res.kpts_scores.dtype == np.float64 and res.obj_scores.dtype == np.float64
    assert np.array_equal(res.kpts_scores, g["grouped_joints"][..., 2])
    assert np.array_equal(res.kpts_tags, g["grouped_joints"][..., 3:])
    assert np.array_equal(res.obj_scores, g["person_scores"])
    assert golden_cases.sha(res.kpts_heatmaps) == str(g["agg_hm_sha"])


@pytest.mark.parametrize("name", ["netlike192_flip", "crowd256_q_flip", "crowd256_val_m20", "empty256_fallback",
                                  "crowd512_30_flip", "netlike512_flip", "crowd256_m5", "crowd256_m32",
                                  "crowd256_tight_thr", "netlike256_some_negative", "crowd192_q_dense"])
def test_decode_matches_committed_reference_goldens(name):
    """The CUDA path against tests/golden/*.npz -- outputs of the reference's own grouping.py (unmodified) with
    the restated munkres stand-in underneath it (oracle/refshim/munkres.py, PARITY UNPINNED for equal-cost
    tie-breaks), recorded by oracle/gen_golden.py; the C++ oracle is not involved."""
    from hpdecode import BottomUpDecoder
    from oracle import golden_cases
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    scales, size, M, det, tthr = golden_cases.make_inputs(name)
    assert golden_cases.inputs_digest(scales) == str(g["inputs_digest"])
    dec = BottomUpDecoder(17, M, det, tthr, "cuda:0")
    res = dec.decode(_dev(scales), (size, size))
    assert golden_cases.sha(res.agg_hm[0].cpu().numpy()) == str(g["agg_hm_sha"])
    assert golden_cases.sha(res.agg_tags[0].cpu().numpy()) == str(g["agg_tags_sha"])
    assert np.array_equal(res.bufs.idx_k[0].cpu().numpy(), g["idx_k"])
    gj, ps = res.to_numpy()[0]
    assert gj.dtype == g["grouped_joints"].dtype
    assert np.array_equal(gj, g["grouped_joints"]) and np.array_equal(ps, g["person_scores"])


@pytest.mark.parametrize("size,levels,peaks", [
    (256, 64, 400),      # plenty of positive peaks on a coarse value grid: ties inside the top 30 and at its boundary
    (256, 4096, 60),     # few ties: the floor-mode result stands for most joints
    (128, 16, 25),       # fewer than 30 positive peaks: +-0 tail, one warp per row (too small for the split kernel)
    (512, 32, 2000),     # 8 warps per row with heavy ties
])
def test_topk_tie_order_matches_oracle(size, levels, peaks, oracle):
    """Top-k on heatmaps built to tie: isolated peaks with values on a coarse grid over a negative background.
    Indices, values and tags must be the reference's (std::partial_sort history order among equal values)."""
    from hpdecode import MPPEHeatmapParser
    rng = np.random.default_rng(size + levels + peaks)
    K = 17
    hm = -rng.random((K, size, size), dtype=np.float32) - 0.5
    for k in range(K):
        n = peaks if k % 3 else max(peaks // 8, 3)                 # every third joint has few peaks
        ys = rng.integers(2, size - 2, n)
        xs = rng.integers(2, size - 2, n)
        hm[k, ys, xs] = (rng.integers(1, levels + 1, n) / np.float32(levels)).astype(np.float32)
    tg = rng.standard_normal((K, size, size, 2)).astype(np.float32)
    parser = MPPEHeatmapParser(K, 30, 0.05, 0.5)
    tags_k, coords_k, scores_k = parser.top_k(torch.from_numpy(hm), torch.from_numpy(tg))
    nm, _ = oracle.nms(hm)
    want = oracle.top_k(nm, tg, 30)
    w_tags, w_coords, w_scores = want[0], want[1], want[2]
    assert np.array_equal(coords_k, w_coords)
    assert np.array_equal(_bits(scores_k), _bits(w_scores)) and np.array_equal(_bits(tags_k), _bits(w_tags))
    # and the reference's own call (grouping.py:153): torch's CPU topk on the flattened NMS'd map
    tv, ti = torch.from_numpy(nm).reshape(K, -1).topk(30, dim=1)
    assert np.array_equal(coords_k[..., 1] * size + coords_k[..., 0], ti.numpy())
    assert np.array_equal(_bits(scores_k), _bits(tv.numpy()))
    # the large-batch path on the same maps: one warp per row with tied rows handed to the second launch
    # (force_generic 2), and with tied rows streamed inline (6)
    from hpdecode import ops
    for force in (2, 6):
        bufs = ops.DecodeBuffers(1, K, size, size, 2, 30, "cuda:0", torch.from_numpy(hm)[None].cuda(), torch.from_numpy(tg)[None].cuda())
        p = ops.make_params(1, K, size, size, 2, 30, 0.05, 0.5)
        ops.run_stage("nms", bufs, p)
        bufs.idx_k.fill_(-1)                      # stale markers must not confuse the second launch
        p.force_generic = force
        ops.run_stage("topk", bufs, p)
        assert np.array_equal(bufs.idx_k[0].cpu().numpy(), ti.numpy().astype(np.int32)), f"force_generic={force}"
        assert np.array_equal(_bits(bufs.scores_k[0].cpu().numpy()), _bits(w_scores))
        assert np.array_equal(_bits(bufs.tags_k[0].cpu().numpy()), _bits(w_tags))


@pytest.mark.parametrize("gen,kw,size", [
    ("netlike", dict(batch=2, size=256, flip=True, seed=61), 256),
    ("crowd", dict(batch=2, size=256, persons=25, flip=True, seed=62, quantised=True), 256),
    ("crowd", dict(batch=1, size=512, persons=30, flip=False, seed=63, quantised=True), 512),
    ("netlike", dict(batch=1, size=512, flip=True, seed=64, negative_channels=(0, 1, 2, 3)), 512),
])
def test_topk_fast_path_equals_exact_heap_replay(gen, kw, size):
    """The sorted-register fast path (with its ambiguity detector) against the forced libstdc++-heap path."""
    from hpdecode import ops
    scales = _dev(getattr(synth, gen)(**kw))
    B = kw["batch"]
    E = 2 if kw["flip"] else 1
    outs = []
    # force_generic bits: 1 = exact heap only, 2 = one-warp-per-row kernel instead of the split kernel that
    # small batches get.  0: split + fast, 1: split kernel's sequential exact scan, 2: one warp per row + fast
    # (tied rows go to the second, 8-warps-per-row launch), 6: one warp per row, tied rows streamed inline through
    # the warp-wide heap, 3: one warp per row, literal libstdc++ scan
    for force in (0, 1, 2, 6, 3):
        bufs = ops.DecodeBuffers(B, 17, size, size, E, 30, "cuda:0")
        p = ops.make_params(B, 17, size, size, E, 30, 0.05, 0.5)
        ops.run_stage("aggregate_nms", bufs, p, scales=scales)
        p.force_generic = force
        ops.run_stage("topk", bufs, p)
        torch.cuda.synchronize()
        outs.append((bufs.idx_k.cpu().numpy(), bufs.scores_k.cpu().numpy(), bufs.tags_k.cpu().numpy()))
    for o in outs[1:]:
        assert np.array_equal(outs[0][0], o[0])
        assert np.array_equal(_bits(outs[0][1]), _bits(o[1])) and np.array_equal(_bits(outs[0][2]), _bits(o[2]))


def _ms_scales(B, H, W, ratios, flip, seed):
    """Network outputs for several test scales: hi at ratio*(H, W), lo / tag at half of that."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for r in ratios:
        hh, hw = int(round(H * r)), int(round(W * r))
        d = {"hm_lo": torch.randn(B, 17, hh // 2, hw // 2, generator=g), "hm_hi": torch.randn(B, 17, hh, hw, generator=g),
             "tag": torch.randn(B, 17, hh // 2, hw // 2, generator=g)}
        if flip:
            d.update({k + "_f": torch.randn_like(v) for k, v in list(d.items())})
        out.append({k: v.cuda() for k, v in d.items()})
    return out


@pytest.mark.parametrize("H,W,ratios,tag_scale,flip,B", [
    (512, 512, (0.25, 0.5, 0.75), 1, True, 2),      # BASELINE config 3 ratios (scales 0.5 / 1.0 / 1.5)
    (640, 640, (0.25, 0.5, 0.75), 1, True, 1),
    (256, 384, (0.5, 0.75), 0, False, 1),           # two scales, non-square, E = 1, NW = 2
    (512, 768, (0.5, 1.0), 0, True, 1),             # hi == output size (copy taps), several CTAs per row
    (320, 512, (0.25, 0.5), 1, True, 1),            # H not a multiple of 64
    (128, 256, (0.25, 0.75), 1, True, 1),           # narrowest width the kernel takes (2 warps per CTA)
    (64, 1280, (0.5, 0.75), 0, True, 1),            # two 5-warp CTAs per row band
])
def test_multiscale_kernel_is_bit_identical_to_generic(H, W, ratios, tag_scale, flip, B, oracle):
    scales = _ms_scales(B, H, W, ratios, flip, seed=H + W)
    E = 2 if flip else 1
    fast = _run_aggregate(scales, H, W, E, False, tag_scale=tag_scale)
    slow = _run_aggregate(scales, H, W, E, True, tag_scale=tag_scale)
    _assert_tag_map_matches_oracle(fast, scales, H, W, oracle, tag_scale)
    for name in ("agg_hm", "nms_mask", "nms_wmax", "hm_wmax"):
        a, b = getattr(fast, name).cpu().numpy(), getattr(slow, name).cpu().numpy()
        if name == "nms_wmax":
            assert np.array_equal(a, b), f"{name} differs"
        else:
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"{name} differs"
    # the tag bounds really bound the first tag component of every 4-row x 32-pixel block
    t0 = fast.agg_tags[..., 0]
    blk = t0.reshape(B, 17, H // 4, 4, W // 32, 32)
    lo, hi = blk.amin(dim=(3, 5)), blk.amax(dim=(3, 5))
    slack = 1e-4 * (1 + lo.abs().max())
    assert bool((fast.tag_bmin <= lo + slack).all()) and bool((fast.tag_bmax >= hi - slack).all())


@pytest.mark.parametrize("lh,lw,flip,B", [(64, 64, False, 2), (128, 128, True, 1), (48, 80, True, 1), (30, 30, False, 1)])
def test_half_inputs_equal_float_path_on_upcast_tensors(lh, lw, flip, B, oracle):
    """SURVEY 8(f)-3: fp16 network outputs (autocast, module.py:78).  The halves are widened on load, so every
    output must equal -- bit for bit -- the float32 path run on the up-cast tensors; specialised and generic
    kernel, strided channel-slice views included."""
    s32 = _rand_maps(B, lh, lw, flip, seed=7 + lh)
    s16 = {k: v.half() for k, v in s32.items()}
    up = {k: v.float() for k, v in s16.items()}
    H, W, E = 4 * lh, 4 * lw, 2 if flip else 1
    want = _run_aggregate([up], H, W, E, False)
    for force in (False, True):
        got = _run_aggregate([s16], H, W, E, force)
        for name in ("agg_hm", "agg_tags", "nms_mask", "hm_wmax"):
            assert torch.equal(getattr(got, name), getattr(want, name)), f"{name} (generic={force})"
    both = torch.cat([s16["hm_lo"], s16["tag"]], 1)                       # one 34-channel half tensor, sliced
    view = dict(s16, hm_lo=both[:, :17], tag=both[:, 17:])
    got = _run_aggregate([view], H, W, E, False)
    assert torch.equal(got.agg_hm, want.agg_hm) and torch.equal(got.agg_tags, want.agg_tags)
    hm_o, tg_o = oracle.aggregate([{k: v[0].cpu().numpy() for k, v in up.items()}], (H, W))
    assert np.array_equal(_bits(want.agg_hm[0].cpu().numpy()), _bits(hm_o))
    assert np.array_equal(_bits(want.agg_tags[0].cpu().numpy()), _bits(tg_o))
    from hpdecode._lib import HpdError
    with pytest.raises(HpdError):                                          # mixed dtypes are refused
        _run_aggregate([dict(s16, hm_hi=up["hm_hi"])], H, W, E, False)
