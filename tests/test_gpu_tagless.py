"""-m gpu: buffer sets without a full-resolution tag map.  The aggregation then writes no agg_tags and the tag stages
(top-k, adjust, refine) interpolate the tags they read from the network outputs; every output must be bit-identical to
a decode into a buffer set that holds the map (where the tag stages read the map), the map must equal the oracle's,
and the map computed afterwards (the lazy DecodeResult.agg_tags) must equal the one the decode wrote."""
import numpy as np
import pytest
import torch

from hpdecode import synth

pytestmark = pytest.mark.gpu

OUTPUTS = ("records", "poses", "person_scores", "n_person", "flags", "scores_k", "idx_k", "coords_k", "tags_k", "agg_hm",
           "nms_mask", "hm_wmax", "tag_bmin", "tag_bmax")


def _bits(t):
    a = t.cpu().numpy()
    return a.view(np.uint8 if a.dtype == np.uint8 else np.uint32)


def _assert_same(got, want, what):
    for name in OUTPUTS:
        assert np.array_equal(_bits(getattr(got, name)), _bits(getattr(want, name))), f"{what}: {name} differs"
    # nms_wmax: the sign of a zero word maximum is unspecified (the existing stage tests compare values too)
    assert torch.equal(got.nms_wmax, want.nms_wmax), f"{what}: nms_wmax differs"


def _dev(scales, half=False):
    return [{k: torch.from_numpy(v).cuda().to(torch.float16 if half else torch.float32) for k, v in s.items()}
            for s in scales]


def _decode_both(scales, H, W, tag_scale=0, force_generic=0, tags_preflipped=False, K=17, M=30):
    """run_decode into a tag-less and into a map-holding buffer set; returns both and the params."""
    from hpdecode import ops
    B = scales[0]["hm_lo"].shape[0]
    E = 2 if scales[tag_scale].get("tag_f") is not None else 1
    p = ops.make_params(B, K, H, W, E, M, 0.05, 0.5, num_scales=len(scales), tag_scale=tag_scale,
                        tags_preflipped=tags_preflipped)
    p.force_generic = force_generic
    out = []
    for tags in (False, True):
        bufs = ops.DecodeBuffers(B, K, H, W, E, M, "cuda:0", tags=tags)
        bufs.records.zero_()
        ops.run_decode(scales, bufs, p)
        out.append(bufs)
    torch.cuda.synchronize()
    assert out[0].tag_map is None and out[1].tag_map is not None
    return out[0], out[1], p


def _check_case(scales, H, W, what, oracle, oracle_scales=None, **kw):
    """oracle_scales: the inputs as the oracle takes them (un-flipped tag_f), if ``scales`` differ from them."""
    tagless, full, p = _decode_both(scales, H, W, **kw)
    _assert_same(tagless, full, what)
    ref = oracle_scales if oracle_scales is not None else scales
    for b in range(p.batch):
        _, tg_o = oracle.aggregate([{k: v[b].float().cpu().numpy() for k, v in s.items()} for s in ref], (H, W),
                                   tag_scale=p.tag_scale)
        assert np.array_equal(_bits(full.agg_tags[b]), np.ascontiguousarray(tg_o, np.float32).view(np.uint32)), \
            f"{what}: image {b}: tag map vs oracle"
    assert torch.equal(tagless.agg_tags, full.agg_tags), f"{what}: lazy agg_tags of the tag-less set"
    return tagless, full


def test_bench_workload_cfg2(oracle):
    """The flagship batch: HigherHRNet-W32 outputs, 64 x 512^2 + flip (agg_nms_x2_kernel, one warp per top-k row)."""
    from hpdecode import synth_net
    scale = synth_net.network_outputs(64, 512, flip=True, seed=1, C=32, device="cuda:0")
    tagless, _ = _check_case([scale], 512, 512, "cfg2", oracle)
    assert int(tagless.n_person.sum()) > 0


def test_cfg3_three_scales_w48_640(oracle):
    """Multi-scale kernel (tags from scale 1.0 of 0.5 / 1.0 / 1.5), W48 640^2 + flip."""
    from hpdecode import synth_net
    S = 640
    ins = [synth_net.network_outputs(2, int(round(S * sc / 64.0)) * 64, flip=True, seed=5, C=48, device="cuda:0", chunk=2)
           for sc in (0.5, 1.0, 1.5)]
    _check_case(ins, S, S, "cfg3", oracle, tag_scale=1)


@pytest.mark.parametrize("size,flip", [(256, True), (192, False)])
def test_half_inputs(size, flip, oracle):
    scales = _dev(synth.crowd(2, size, persons=10, flip=flip, seed=21), half=True)
    _check_case(scales, size, size, f"half {size} flip={flip}", oracle)


def test_tags_preflipped(oracle):
    s = _dev(synth.crowd(2, 256, persons=12, flip=True, seed=23))[0]
    pre = dict(s)
    pre["tag_f"] = torch.flip(s["tag_f"], [3])[:, synth.COCO_FLIP_INDEX].contiguous()
    a, _ = _check_case([pre], 256, 256, "preflipped", oracle, oracle_scales=[s], tags_preflipped=True)
    b, _ = _check_case([s], 256, 256, "not preflipped", oracle)
    assert torch.equal(a.tags_k, b.tags_k) and torch.equal(a.records, b.records)


def test_single_embedding_without_flip(oracle):
    _check_case(_dev(synth.netlike(2, 256, flip=False, seed=25)), 256, 256, "E=1", oracle)


@pytest.mark.parametrize("force_generic", [0, 1, 2, 4])
def test_generic_kernel_and_topk_variants(force_generic, oracle):
    """A size no specialised kernel takes (250 x 250 output from 64 x 64 tag maps: not x4, W % 32 != 0), and the
    standard size under force_generic (bit 0: generic aggregation + literal heap top-k; bits 1 / 2: top-k launches)."""
    scales = _dev(synth.crowd(2, 256, persons=10, flip=True, seed=27))
    _check_case(scales, 250, 250, f"generic 250, force_generic={force_generic}", oracle, force_generic=force_generic)
    _check_case(scales, 256, 256, f"256, force_generic={force_generic}", oracle, force_generic=force_generic)


def test_single_stage_calls():
    """run_stage one stage at a time on a tag-less set: the tag stages take the tag inputs from ``scales``, and
    refuse to run without them."""
    from hpdecode import _lib, ops
    scales = _dev(synth.crowd(2, 256, persons=10, flip=True, seed=29))
    _, full, p = _decode_both(scales, 256, 256)
    bufs = ops.DecodeBuffers(2, 17, 256, 256, 2, 30, "cuda:0", tags=False)
    bufs.records.zero_()
    for st in ("aggregate_nms", "topk", "group", "adjust_refine"):
        ops.run_stage(st, bufs, p, scales=scales)
    torch.cuda.synchronize()
    _assert_same(bufs, full, "run_stage")
    for st in ("topk", "adjust_refine"):
        with pytest.raises(_lib.HpdError, match="tag"):
            ops.run_stage(st, bufs, p)


def test_decoder_results_and_lazy_tag_map():
    """BottomUpDecoder builds tag-less sets by default; DecodeResult.agg_tags computes the map once, on demand."""
    from hpdecode import BottomUpDecoder
    scales = _dev(synth.crowd(2, 256, persons=10, flip=True, seed=31))
    res = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0").decode(scales, (256, 256))
    want = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0", keep_tag_map=True).decode(scales, (256, 256))
    assert res.bufs.tag_map is None and want.bufs.tag_map is not None
    _assert_same(res.bufs, want.bufs, "decoder")
    assert torch.equal(res.agg_tags, want.agg_tags) and res.agg_tags is res.agg_tags


def test_pipeline_with_cuda_graphs():
    """DecodePipeline (CUDA graphs, records ring) on tag-less lanes against a map-holding decode; a result's lazy tag
    map is computed from its lane's inputs, and refused once the lane has been reused."""
    from hpdecode import BottomUpDecoder, _lib, ops
    from hpdecode.decoder import DecodePipeline
    scales = _dev(synth.crowd(4, 256, persons=10, flip=True, seed=33))
    want = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0", keep_tag_map=True).decode(scales, (256, 256))
    dec = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0")
    ring = torch.zeros((2, 4, ops.record_layout(17, 30, 2).row_bytes), device="cuda:0", dtype=torch.uint8)
    pipe = DecodePipeline(dec, depth=2, records_ring=ring, use_graphs=True)
    staging = [[{k: torch.empty_like(v) for k, v in s.items()} for s in scales] for _ in range(2)]

    def h2d(ln):
        st = staging[ln["slot"]]
        for d, s in zip(st, scales):
            for k in d:
                d[k].copy_(s[k], non_blocking=True)
        return st

    results = [pipe.submit(scales, (256, 256), before_agg=h2d) for _ in range(3)]
    assert pipe.graph_replays == 3
    pipe.drain()
    torch.cuda.synchronize()
    last = results[-1]
    assert last.bufs._tag_inputs[0] is staging[0]      # the inputs as before_agg staged them
    for name in ("records", "poses", "person_scores", "n_person", "flags", "tags_k", "idx_k"):
        assert torch.equal(getattr(last.bufs, name), getattr(want.bufs, name)), name
    assert torch.equal(ring[0], want.bufs.records) and torch.equal(ring[1], want.bufs.records)
    assert torch.equal(last.agg_tags, want.agg_tags)
    with pytest.raises(_lib.HpdError, match="overwritten"):
        results[0].agg_tags
