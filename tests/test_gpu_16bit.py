"""-m gpu: 16-bit network outputs decoded in place.  bfloat16 on every aggregation kernel and every tag read, float16
and bfloat16 on the multi-scale kernel, and the autocast forward of InferenceKeypointsModel.

Widening a float16 or bfloat16 to float32 is exact, so the oracle for 16-bit inputs is the float32 path on the up-cast
tensors: every output of every stage must equal it bit for bit.  Outputs are NaN-poisoned before each decode, and the
kernel that ran is read from the profiler's launch names, so a silent fall-back to another kernel cannot pass."""
import numpy as np
import pytest
import torch
from torch import nn

from hpdecode import ops, synth

pytestmark = pytest.mark.gpu

BF16, F16 = torch.bfloat16, torch.float16
TYPE_NAME = {BF16: "__nv_bfloat16", F16: "__half"}
OUTPUTS = ("agg_hm", "tag_map", "nms_mask", "hm_wmax", "tag_bmin", "tag_bmax", "scores_k", "idx_k", "coords_k",
           "tags_k", "poses", "person_scores", "n_person", "flags", "records")


def _bits(t):
    a = t.cpu().numpy()
    return a.view({1: np.uint8, 4: np.uint32}[a.dtype.itemsize])


def _decode(scales, H, W, tag_scale=0, force=0, tags=True, K=17, M=30):
    """run_decode into a NaN-poisoned buffer set; .kernels = the names of the kernels the decode launched."""
    from torch.profiler import ProfilerActivity, profile
    B = scales[0]["hm_lo"].shape[0]
    E = 2 if scales[tag_scale].get("tag_f") is not None else 1
    p = ops.make_params(B, K, H, W, E, M, 0.05, 0.5, num_scales=len(scales), tag_scale=tag_scale)
    p.force_generic = force
    bufs = ops.DecodeBuffers(B, K, H, W, E, M, "cuda:0", tags=tags)
    for name in OUTPUTS + ("nms_wmax",):
        t = getattr(bufs, name)
        if t is not None:
            t.fill_(float("nan") if t.is_floating_point() else (255 if t.dtype == torch.uint8 else -1))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.run_decode(scales, bufs, p)
        torch.cuda.synchronize()
    bufs.kernels = " ".join(e.key for e in prof.key_averages())
    assert not bool(torch.isnan(bufs.agg_hm).any()), "agg_hm not fully written"
    return bufs


def _assert_same(got, want, what, skip=()):
    for name in OUTPUTS:
        if name in skip:
            continue
        a, b = getattr(got, name), getattr(want, name)
        assert (a is None) == (b is None), f"{what}: {name}"
        if a is not None:
            assert np.array_equal(_bits(a), _bits(b)), f"{what}: {name} differs"
    # the sign of a zero word maximum is unspecified between kernels: compared by value, like the stage tests
    assert torch.equal(got.nms_wmax, want.nms_wmax), f"{what}: nms_wmax differs"


def _kernel(bufs, name, dtype=None):
    assert name in bufs.kernels, f"{name} did not run: {bufs.kernels}"
    if dtype is not None:
        assert any(name in k and TYPE_NAME[dtype] + "," in k or name in k and TYPE_NAME[dtype] + ">" in k
                   for k in bufs.kernels.split("void ")), f"{name} did not run on {dtype}: {bufs.kernels}"


def _to16(s, dtype, misalign=False):
    """The scale dict in `dtype`; hm_lo / tag as channel slices of one 2K-channel tensor when they share a shape
    (HigherHRNet's head, higher_hrnet.py:78-79).  misalign: every map starts one element past an 8-byte boundary."""
    out = {}
    for suf in ("", "_f"):
        if s.get("hm_lo" + suf) is None:
            continue
        lo, tag, hi = s["hm_lo" + suf], s.get("tag" + suf), s["hm_hi" + suf]
        if tag is not None and tag.shape == lo.shape:
            both = torch.cat((lo, tag), 1).to(dtype)
            out["hm_lo" + suf], out["tag" + suf] = both[:, :lo.shape[1]], both[:, lo.shape[1]:]
        else:
            out["hm_lo" + suf] = lo.to(dtype)
            if tag is not None:
                out["tag" + suf] = tag.to(dtype)
        out["hm_hi" + suf] = hi.to(dtype)
    return _misalign(out) if misalign else out


def _misalign(s):
    """Copies whose bases are one element past an aligned address (no 16-bit map is then 8-byte aligned, no float32
    one 16-byte aligned)."""
    out = {}
    for k, v in s.items():
        buf = torch.empty(v.numel() + 1, device=v.device, dtype=v.dtype)
        out[k] = buf[1:].view(v.shape).copy_(v)
    return out


def _up(s, misalign=False):
    up = {k: v.float() for k, v in s.items()}
    return _misalign(up) if misalign else up


# The generic kernel derives no tag bounds: it writes tag_bmin / tag_bmax = -inf / +inf ("anything", a valid refine
# prefilter), where the x2 and multi-scale kernels write the real bounds.  Against it those two arrays are not compared;
# every output of the decode is.
BOUNDS = ("tag_bmin", "tag_bmax")


def _rand(B, lh, lw, flip, seed, H=None, W=None, hi_ratio=2):
    g = torch.Generator().manual_seed(seed)
    d = {"hm_lo": torch.randn(B, 17, lh, lw, generator=g),
         "hm_hi": torch.randn(B, 17, hi_ratio * lh, hi_ratio * lw, generator=g),
         "tag": torch.randn(B, 17, H // 4 if H else lh, W // 4 if W else lw, generator=g)}
    if flip:
        d.update({k + "_f": torch.randn(v.shape, generator=g) for k, v in list(d.items())})
    return {k: v.cuda() for k, v in d.items()}


def _check(s32, H, W, dtype, kernel, tag_scale=0, force=0, tags=True, misalign=False, what=""):
    s16 = [_to16(s, dtype, misalign) for s in s32]
    want = _decode([_up(s, misalign) for s in s16], H, W, tag_scale, force, tags)
    got = _decode(s16, H, W, tag_scale, force, tags)
    _kernel(got, kernel, dtype if kernel != "agg_nms_generic_kernel" else None)
    _assert_same(got, want, what)
    return s16, got


# ---- x2 kernel -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lh,lw,flip,B,tags", [(128, 128, True, 2, True), (128, 128, False, 1, False),
                                               (64, 176, True, 2, False), (48, 80, False, 1, True),
                                               (32, 256, True, 1, True), (12, 16, True, 3, False)])
def test_bf16_x2_kernel(lh, lw, flip, B, tags):
    """E = 1 / 2, tag map kept and tag-less, one / two / four warps per CTA, partial strips, tiny maps."""
    _check([_rand(B, lh, lw, flip, seed=lh + lw)], 4 * lh, 4 * lw, BF16, "agg_nms_x2_kernel", tags=tags,
           what=f"x2 {lh}x{lw} flip={flip} tags={tags}")


def test_bf16_x2_kernel_misaligned_inputs():
    """Bases one element past an aligned address: the x2 kernel stages with scalar loads."""
    _check([_rand(2, 64, 64, True, seed=3)], 256, 256, BF16, "agg_nms_x2_kernel", misalign=True, what="misaligned x2")


def test_bf16_cfg2_batch():
    """The flagship shape: HigherHRNet-W32 outputs, 64 x 512^2 + flip, tag-less (the decoder's default)."""
    from hpdecode import synth_net
    s = synth_net.network_outputs(64, 512, flip=True, seed=1, C=32, device="cuda:0")
    _, got = _check([s], 512, 512, BF16, "agg_nms_x2_kernel", tags=False, what="cfg2")
    assert int(got.n_person.sum()) > 0


# ---- generic kernel ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["forced", "250", "odd", "misaligned_ms"])
def test_bf16_generic_kernel(case):
    """bf16 through the generic kernel: forced (force_generic bit 0), and chosen by shape -- outputs that are not x4
    of the tag maps, odd sizes with W % 32 != 0, and a multi-scale layout whose inputs are not 8-byte aligned."""
    if case == "forced":
        _check([_rand(2, 64, 64, True, seed=11)], 256, 256, BF16, "agg_nms_generic_kernel", force=1, what=case)
    elif case == "250":
        _check([_rand(2, 64, 64, True, seed=12)], 250, 250, BF16, "agg_nms_generic_kernel", what=case)
    elif case == "odd":
        _check([_rand(1, 33, 45, False, seed=13)], 132, 180, BF16, "agg_nms_generic_kernel", tags=False, what=case)
    else:
        s = [_rand(1, 32, 32, True, seed=14, H=256, W=256), _rand(1, 48, 48, True, seed=15, H=256, W=256)]
        _check(s, 256, 256, BF16, "agg_nms_generic_kernel", misalign=True, what=case)


# ---- multi-scale kernel --------------------------------------------------------------------------------------------
def _ms_case(case):
    """(scales, H, W, tag_scale): hi at ratio * output, lo at half of hi, tags x4 below the output."""
    if case == "1scale":          # hm_hi at the output size: not the x2 layout, one scale
        return [_rand(1, 128, 128, True, seed=21, H=256, W=256)], 256, 256, 0
    if case == "2scales":         # two scales, E = 1, non-square
        return [_rand(1, 64, 96, False, seed=22, H=256, W=384), _rand(1, 96, 144, False, seed=23, H=256, W=384)], 256, 384, 0
    if case == "3scales":         # BASELINE config 3 ratios (test scales 0.5 / 1.0 / 1.5), flip, two images
        return [_rand(2, 64 * r, 64 * r, True, seed=24 + r, H=512, W=512) for r in (1, 2, 3)], 512, 512, 1
    from hpdecode import synth_net   # cfg3: HigherHRNet-W48 outputs at 640^2, scales 0.5 / 1.0 / 1.5 + flip
    S = 640
    return [synth_net.network_outputs(2, int(round(S * sc / 64.0)) * 64, flip=True, seed=5, C=48, device="cuda:0",
                                      chunk=2) for sc in (0.5, 1.0, 1.5)], S, S, 1


@pytest.mark.parametrize("dtype", [F16, BF16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("case", ["1scale", "2scales", "3scales", "cfg3_w48_640"])
def test_16bit_multiscale_kernel(case, dtype):
    """fp16 and bf16 through agg_nms_ms_kernel: equal to the float32 path on the up-cast tensors, and to the generic
    kernel on the same 16-bit inputs."""
    s32, H, W, ts = _ms_case(case)
    s16, got = _check(s32, H, W, dtype, "agg_nms_ms_kernel", tag_scale=ts, tags=case != "cfg3_w48_640", what=case)
    slow = _decode(s16, H, W, ts, force=1, tags=case != "cfg3_w48_640")
    _kernel(slow, "agg_nms_generic_kernel")
    assert "agg_nms_ms_kernel" not in slow.kernels
    _assert_same(got, slow, f"{case}: ms vs generic", skip=BOUNDS)
    assert bool((slow.tag_bmin == -float("inf")).all()) and bool((got.tag_bmin > -float("inf")).all())


# ---- lazy tag map, pipeline, validation-time and model entry points -------------------------------------------------
def _written(records, K=17, M=30, E=2):
    """The bytes of each record row the decode writes (the row is padded to 8 bytes)."""
    return records[:, :ops.record_layout(K, M, E).off_flags + 4]


def test_bf16_lazy_agg_tags_of_a_tagless_decode():
    from hpdecode import BottomUpDecoder
    s = _to16({k: torch.from_numpy(v).cuda() for k, v in synth.crowd(2, 256, persons=12, flip=True, seed=31)[0].items()}, BF16)
    res = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0").decode([s], (256, 256))
    assert res.bufs.tag_map is None
    want = _decode([_up(s)], 256, 256)
    assert np.array_equal(_bits(res.agg_tags), _bits(want.tag_map))
    assert torch.equal(_written(res.records), _written(want.records))


def test_bf16_decode_pipeline_with_cuda_graphs():
    from hpdecode import BottomUpDecoder, DecodePipeline
    s = _to16({k: torch.from_numpy(v).cuda() for k, v in synth.crowd(4, 256, persons=10, flip=True, seed=33)[0].items()}, BF16)
    want = _decode([_up(s)], 256, 256)
    pipe = DecodePipeline(BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0"), depth=2, use_graphs=True)
    for _ in range(4):
        res = pipe.submit([s], (256, 256))
        pipe.drain()
        torch.cuda.synchronize()
        assert torch.equal(_written(res.records), _written(want.records)) and torch.equal(res.poses, want.poses)
    assert pipe.graph_replays == 4


def test_set_preds_bf16(oracle):
    """KeypointsResult.set_preds (results.py:94-124) on bf16 network outputs: the float32 path on the up-cast tensors."""
    from hpdecode import KeypointsResult
    s = _to16({k: torch.from_numpy(v).cuda() for k, v in synth.crowd(1, 256, persons=9, flip=False, seed=77)[0].items()}, BF16)
    up = {k: v.float().cpu().numpy() for k, v in s.items()}
    r = KeypointsResult(torch.zeros(3, 256, 256), [s["hm_lo"], s["hm_hi"]], s["tag"], [], max_num_people=20, det_thr=0.1,
                        tag_thr=1.0)
    r.set_preds()
    hm_o, tg_o = oracle.aggregate([{k: v[0] for k, v in up.items()}], (256, 256))
    ref = oracle.parse(hm_o, tg_o, 20, 0.1, 1.0)
    gj = ref["grouped_joints"]
    assert gj.shape[0] >= 5
    f32 = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
    assert np.array_equal(f32(r.kpts_coords), f32(gj[..., :2])) and np.array_equal(f32(r.kpts_scores), f32(gj[..., 2]))
    assert np.array_equal(f32(r.kpts_tags), f32(gj[..., 3:])) and np.array_equal(f32(r.obj_scores), f32(ref["person_scores"]))
    assert np.array_equal(f32(r.tags_heatmaps), f32(tg_o))


class _CaptureNet(nn.Module):
    """Keeps every call's outputs up-cast to float32 on the host, and their dtype."""

    def __init__(self, net):
        super().__init__()
        self.net, self.calls = net, []

    def forward(self, x):
        (lo, hi), tag = self.net(x)
        self.calls.append(({lo.dtype, hi.dtype, tag.dtype},
                           [t.detach().float().cpu().numpy() for t in (lo, hi, tag)]))
        return [lo, hi], tag


@pytest.mark.parametrize("dtype,flip,test_scales,size", [(BF16, True, (1.0,), 256), (BF16, True, (0.5, 1.0, 1.5), 512),
                                                         (F16, False, (1.0,), 256)])
def test_model_autocast(dtype, flip, test_scales, size, oracle):
    """InferenceKeypointsModel(autocast_dtype=...): the net runs under autocast, its 16-bit outputs go to the decoder
    as they are, and the results are the oracle's decode of those outputs up-cast to float32."""
    from hpdecode import InferenceKeypointsModel, synth_net
    from oracle import input_oracle
    from oracle.gen_golden_input import image_of
    torch.manual_seed(4)
    net = _CaptureNet(synth_net.HigherHRNet(17, 32))
    model = InferenceKeypointsModel(net, use_flip=flip, input_size=size, device="cuda:0", test_scales=test_scales,
                                    autocast_dtype=dtype)
    raw = image_of(300, 421, 11)
    result = model(raw, None)
    assert all(c[0] == {dtype} for c in net.calls) and len(net.calls) == len(test_scales) * (2 if flip else 1)
    min_scale = min(test_scales)
    per = 2 if flip else 1
    scales = []
    for i in range(len(test_scales)):
        lo, hi, tag = net.calls[i * per][1]
        d = {"hm_lo": lo[0], "hm_hi": hi[0], "tag": tag[0]}
        if flip:
            lo, hi, tag = net.calls[i * per + 1][1]
            d.update(hm_lo_f=lo[0], hm_hi_f=hi[0], tag_f=tag[0])
        scales.append(d)
    (W, H), center, scale = input_oracle.get_multi_scale_size(300, 421, size, 1.0, min_scale)
    hm_o, tg_o = oracle.aggregate(scales, (H, W), tag_scale=test_scales.index(1.0))
    ref = oracle.parse(hm_o, tg_o, 30, 0.05, 0.5)
    gj = ref["grouped_joints"]
    minv = input_oracle.get_affine_transform(center, scale, (W, H), inverse=True)
    coords = input_oracle.affine_points(gj[..., :2].reshape(-1, 2), minv).reshape(gj.shape[0], -1, 2).astype(np.float32)
    f32 = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
    assert np.array_equal(f32(result.kpts_heatmaps), f32(hm_o)) and np.array_equal(f32(result.tags_heatmaps), f32(tg_o[..., 0]))
    assert np.array_equal(f32(result.kpts_coords), f32(coords))
    assert np.array_equal(f32(result.kpts_scores), f32(gj[..., 2])) and np.array_equal(f32(result.kpts_tags), f32(gj[..., 3:]))
    assert np.array_equal(f32(result.obj_scores), f32(ref["person_scores"]))


def test_model_without_autocast_hands_float32_to_the_decoder():
    """autocast_dtype=None keeps the float32 forward: the outputs the decoder reads are float32 tensors."""
    from hpdecode import InferenceKeypointsModel, synth_net
    torch.manual_seed(4)
    net = _CaptureNet(synth_net.HigherHRNet(17, 32))
    model = InferenceKeypointsModel(net, use_flip=True, input_size=256, device="cuda:0")
    outs = model._net_outputs(torch.randn(1, 3, 256, 256, device="cuda:0"))
    assert net.calls[0][0] == {torch.float32} and all(v.dtype == torch.float32 for v in outs.values())
    with pytest.raises(ValueError):
        InferenceKeypointsModel(net, device="cuda:0", autocast_dtype=torch.float64)
