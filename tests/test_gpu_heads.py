"""-m gpu: heads with 1 to 4 heatmap stages.  The single-stage kernel (agg_nms_x4_kernel) against the generic kernel
and the oracle, three / four stages and multi-scale single-stage heads through the generic kernel, two stages through
hpd_decode_stages against hpd_decode, and InferenceKeypointsModel / from_preds / set_preds on 1- and 3-stage heads.
Outputs are NaN-poisoned before each decode, and the kernel that ran is read from the profiler's launch names."""
import ctypes

import numpy as np
import pytest
import torch
from torch import nn

from hpdecode import _lib, ops
from oracle import stage_oracle

pytestmark = pytest.mark.gpu

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
OUTPUTS = ("agg_hm", "tag_map", "nms_mask", "hm_wmax", "scores_k", "idx_k", "coords_k", "tags_k", "poses",
           "person_scores", "n_person", "flags", "records")
GENERIC, X4 = "agg_nms_generic_kernel", "agg_nms_x4_kernel"


def _bits(t):
    a = t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    return a.view({1: np.uint8, 4: np.uint32}[a.dtype.itemsize])


def _decode(scales, H, W, tag_scale=0, force=0, tags=True, K=17, M=30, call=None):
    """run_decode (or ``call(params, bufs)``) into a NaN-poisoned buffer set."""
    st = [ops.stage_scale(s) for s in scales]
    B = st[0]["hm"][0].shape[0]
    E = 2 if st[tag_scale].get("tag_f") is not None else 1
    p = ops.make_params(B, K, H, W, E, M, 0.05, 0.5, num_scales=len(scales), tag_scale=tag_scale)
    p.force_generic = force
    bufs = ops.DecodeBuffers(B, K, H, W, E, M, "cuda:0", tags=tags)
    for name in OUTPUTS + ("nms_wmax", "tag_bmin", "tag_bmax"):
        t = getattr(bufs, name)
        if t is not None:
            t.fill_(float("nan") if t.is_floating_point() else (255 if t.dtype == torch.uint8 else -1))
    if call is None:
        ops.run_decode(scales, bufs, p)
    else:
        call(p, bufs)
    torch.cuda.synchronize()
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
    assert torch.equal(got.nms_wmax, want.nms_wmax), f"{what}: nms_wmax differs"


def _host(s, b):
    """Image b of a device scale dict (any format) as float32 host arrays in the stage format."""
    s = ops.stage_scale(s)
    f = lambda t: None if t is None else t[b].float().cpu().numpy()
    return {"hm": [f(t) for t in s["hm"]], "hm_f": [f(t) for t in s.get("hm_f") or []], "tag": f(s["tag"]),
            "tag_f": f(s.get("tag_f"))}


def _word_max(a, wpr):
    K, H, W = a.shape
    w = np.full((K, H, wpr * 32), -np.inf, np.float32)
    w[:, :, :W] = a
    return w.reshape(K, H, wpr, 32).max(axis=3)


def _x4_bounds(tag0, H, W):
    """tag_bmin / tag_bmax of a single-stage x4 layout: per 4 output rows x 32 columns, the range of the quarter-res
    tags the block's pixels interpolate from (rows g-1..g+1, columns 8w-1..8w+8, clamped to the map)."""
    K, th, tw = tag0.shape
    HB, wpr = (H + 3) // 4, (W + 31) // 32
    mn = np.empty((K, HB, wpr), np.float32)
    mx = np.empty_like(mn)
    for g in range(HB):
        rows = np.clip(np.arange(g - 1, g + 2), 0, th - 1)
        for w in range(wpr):
            cols = np.clip(np.arange(8 * w - 1, 8 * w + 9), 0, tw - 1)
            blk = tag0[:, rows][:, :, cols]
            mn[:, g, w], mx[:, g, w] = blk.min(axis=(1, 2)), blk.max(axis=(1, 2))
    return mn, mx


def _check_oracle(bufs, scales, H, W, oracle, tag_scale=0, M=30):
    """agg_hm, the word maxima and every image's poses / scores against the oracle's decode of the float32 inputs."""
    B = bufs.agg_hm.shape[0]
    wpr = (W + 31) // 32
    from hpdecode.decoder import Records
    rec = Records(bufs.records.cpu().numpy(), M, bufs.agg_hm.shape[1], bufs.shape[4])
    for b in range(B):
        hm, tg = stage_oracle.aggregate([_host(s, b) for s in scales], (H, W), tag_scale=tag_scale)
        assert np.array_equal(_bits(bufs.agg_hm[b]), hm.view(np.uint32)), f"image {b}: agg_hm differs from the oracle"
        assert np.array_equal(bufs.hm_wmax[b].cpu().numpy(), _word_max(hm, wpr)), f"image {b}: hm_wmax"
        nm, _ = oracle.nms(hm)
        assert np.array_equal(bufs.nms_wmax[b].cpu().numpy(), _word_max(nm, wpr)), f"image {b}: nms_wmax"
        ref = oracle.parse(hm, tg, M, 0.05, 0.5)
        gj, ps = rec.image(b)
        assert np.array_equal(_bits(gj), _bits(ref["grouped_joints"])), f"image {b}: poses differ from the oracle"
        assert np.array_equal(_bits(ps), _bits(ref["person_scores"])), f"image {b}: person scores differ"
        assert np.array_equal(bufs.idx_k[b].cpu().numpy(), ref["idx_k"]), f"image {b}: top-k indices differ"
        assert np.array_equal(_bits(bufs.scores_k[b]), _bits(ref["scores_k"])), f"image {b}: top-k scores differ"
    return rec


def _single_stage(B, qh, qw, flip, dtype, seed, K=17):
    """One-stage outputs: hm and tag as channel slices of one 2K-channel tensor (batch stride 2K*qh*qw), like the
    HRNet-AE head."""
    g = torch.Generator().manual_seed(seed)
    s = {"hm_f": [], "tag_f": None}
    for r in ("", "_f") if flip else ("",):
        both = torch.randn(B, 2 * K, qh, qw, generator=g).to("cuda:0", dtype)
        s["hm" + r], s["tag" + r] = [both[:, :K]], both[:, K:]
    return s


def _up(s):
    f = lambda t: None if t is None else t.float()
    return {"hm": [t.float() for t in s["hm"]], "hm_f": [t.float() for t in s["hm_f"]], "tag": f(s["tag"]),
            "tag_f": f(s["tag_f"])}


# ---- single-stage kernel -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("qh,qw,B,flip,dtype", [
    (64, 64, 3, True, F32),      # W 256: two warps per CTA, odd B
    (32, 128, 1, False, F32),    # W 512: four warps
    (48, 40, 2, True, F32),      # W 160: one warp, partial strip
    (64, 64, 3, True, F16), (40, 80, 1, False, F16),
    (64, 64, 3, True, BF16), (33, 64, 2, False, BF16),   # H = 132: a partial last band
    (128, 128, 1, True, F32),
])
def test_single_stage_kernel(qh, qw, B, flip, dtype, oracle):
    H, W = 4 * qh, 4 * qw
    s = _single_stage(B, qh, qw, flip, dtype, seed=qh * 131 + qw + B)
    for tags in (False, True):
        got = _decode([s], H, W, tags=tags)
        want = _decode([s], H, W, tags=tags, force=1)
        _assert_same(got, want, f"x4 vs generic {qh}x{qw} B={B} flip={flip} {dtype} tags={tags}")
        assert bool((want.tag_bmin == -np.inf).all()) and bool((want.tag_bmax == np.inf).all())
        if dtype != F32:   # a 16-bit decode is the float32 decode of the up-cast outputs
            _assert_same(got, _decode([_up(s)], H, W, tags=tags), f"16-bit vs float32 {dtype}")
    _check_oracle(got, [s], H, W, oracle)
    for b in range(B):
        mn, mx = _x4_bounds(s["tag"][b].float().cpu().numpy(), H, W)
        assert np.array_equal(got.tag_bmin[b].cpu().numpy(), mn) and np.array_equal(got.tag_bmax[b].cpu().numpy(), mx)
        _, tg = stage_oracle.aggregate([_host(s, b)], (H, W))
        t0 = tg[..., 0]
        bmin = got.tag_bmin[b].cpu().numpy()[:, np.arange(H)[:, None] // 4, np.arange(W)[None, :] // 32]
        bmax = got.tag_bmax[b].cpu().numpy()[:, np.arange(H)[:, None] // 4, np.arange(W)[None, :] // 32]
        assert bool(((t0 >= bmin) & (t0 <= bmax)).all()), "a tag lies outside its block's bounds"


@pytest.mark.parametrize("qh,qw,flip", [(48, 44, True), (40, 60, False), (1, 64, True)])
def test_single_stage_layouts_outside_the_fast_path(qh, qw, flip, oracle):
    """W % 32 != 0 or a one-row map: the generic kernel, equal to the oracle."""
    H, W = 4 * qh, 4 * qw
    if H * W < 64 * 30:
        H = 64
    s = _single_stage(2, qh, qw, flip, F32, seed=qh + qw)
    got = _decode([s], H, W)
    _check_oracle(got, [s], H, W, oracle)


def test_single_stage_misaligned_inputs(oracle):
    """Bases one element past a 16-byte boundary: the kernel's scalar staging."""
    s = _single_stage(2, 64, 64, True, F32, seed=5)
    out = {"hm_f": [], "tag_f": None}
    for key in ("hm", "hm_f"):
        out[key] = []
        for t in s[key]:
            buf = torch.empty(t.numel() + 1, device=t.device)
            out[key].append(buf[1:].view(t.shape).copy_(t))
    for key in ("tag", "tag_f"):
        buf = torch.empty(s[key].numel() + 1, device="cuda:0")
        out[key] = buf[1:].view(s[key].shape).copy_(s[key])
    got = _decode([out], 256, 256)
    _assert_same(got, _decode([s], 256, 256), "misaligned vs aligned")


_KERNEL_PROBE = """
import json, sys, torch
sys.path[:0] = sys.argv[1:3]
from hpdecode import ops, synth
from hpdecode import _lib
import ctypes

def single(B, qh, qw, dtype, flip=True, K=17):
    s = {"hm_f": [], "tag_f": None}
    for r in ("", "_f") if flip else ("",):
        both = torch.randn(B, 2 * K, qh, qw, device="cuda:0").to(dtype)
        s["hm" + r], s["tag" + r] = [both[:, :K]], both[:, K:]
    return s

def stages(B, sizes, K=17):
    r = lambda h, w: torch.randn(B, K, h, w, device="cuda:0")
    return {"hm": [r(h, w) for h, w in sizes], "tag": r(*sizes[0]), "hm_f": [], "tag_f": None}

def run(scales, H, W, tag_scale=0, force=0, legacy=False):
    st = [ops.stage_scale(s) for s in scales]
    B = st[0]["hm"][0].shape[0]
    E = 2 if st[tag_scale].get("tag_f") is not None else 1
    p = ops.make_params(B, 17, H, W, E, 30, 0.05, 0.5, num_scales=len(scales), tag_scale=tag_scale)
    p.force_generic = force
    bufs = ops.DecodeBuffers(B, 17, H, W, E, 30, "cuda:0", tags=False)
    ws = bufs.ensure_workspace(p)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        if legacy:
            arr, keep = ops._scales_struct(scales)
            b = bufs.struct()
            rc = _lib.lib().hpd_decode(ctypes.byref(p), arr, ctypes.byref(b), ws.data_ptr(), ws.numel(),
                                       torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "hpd_decode")
        else:
            ops.run_decode(scales, bufs, p)
        torch.cuda.synchronize()
    return sorted(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)

crowd = [{k: torch.from_numpy(v).cuda() for k, v in s.items()} for s in synth.crowd(2, 256, persons=4, flip=True, seed=3)]
full = crowd[0]
half = {k: v[:, :, ::2, ::2].contiguous() for k, v in full.items()}
out = {
    "x4_f32_nw2": run([single(3, 64, 64, torch.float32)], 256, 256),
    "x4_f16_nw1": run([single(2, 40, 40, torch.float16, flip=False)], 160, 160),
    "x4_bf16_nw4": run([single(1, 32, 128, torch.bfloat16)], 128, 512),
    "x4_forced": run([single(1, 64, 64, torch.float32)], 256, 256, force=1),
    "x4_width": run([single(1, 48, 44, torch.float32)], 192, 176),
    "three_stages": run([stages(1, [(40, 48), (80, 96), (160, 192)])], 160, 192),
    "ms_single": run([stages(1, [(32, 24)]), stages(1, [(64, 48)]), stages(1, [(96, 72)])], 256, 192, tag_scale=1),
    "two_x2_legacy": run(crowd, 256, 256, legacy=True),
    "two_x2_stages": run([ops.stage_scale(s) for s in crowd], 256, 256),
    "two_ms_legacy": run([half, full], 256, 256, tag_scale=1, legacy=True),
    "two_ms_stages": run([ops.stage_scale(half), ops.stage_scale(full)], 256, 256, tag_scale=1),
}
print(json.dumps(out))
"""


def test_aggregation_kernel_selection():
    """Which aggregation kernel each layout runs, read from the launch names.  The profile is taken in a fresh process:
    in a long pytest process, earlier profiler sessions can leave CUPTI delivering the runtime calls but not the kernel
    records.  Two-stage inputs run the same kernels through hpd_decode_stages as through hpd_decode."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-s", "-c", _KERNEL_PROBE, root, os.path.join(root, "pytorch-human-pose_b200")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    got = json.loads(out.stdout.strip().splitlines()[-1])
    agg = {case: [k for k in names if "agg_nms" in k] for case, names in got.items()}
    want = {"x4_f32_nw2": "agg_nms_x4_kernel<2, float>", "x4_f16_nw1": "agg_nms_x4_kernel<1, __half>",
            "x4_bf16_nw4": "agg_nms_x4_kernel<4, __nv_bfloat16>", "x4_forced": GENERIC, "x4_width": GENERIC,
            "three_stages": GENERIC, "ms_single": GENERIC, "two_x2_stages": "agg_nms_x2_kernel<",
            "two_ms_stages": "agg_nms_ms_kernel<"}
    for case, name in want.items():
        assert len(agg[case]) == 1 and name in agg[case][0], (case, got[case])
    assert got["two_x2_stages"] == got["two_x2_legacy"] and got["two_ms_stages"] == got["two_ms_legacy"], got


# ---- three / four stages, multi-scale single stage: generic kernel ------------------------------------------------
def _stages(B, sizes, flip, seed, K=17):
    g = torch.Generator().manual_seed(seed)
    r = lambda h, w: torch.randn(B, K, h, w, generator=g).cuda()
    s = {"hm": [r(h, w) for h, w in sizes], "tag": r(*sizes[0]), "hm_f": [], "tag_f": None}
    if flip:
        s.update(hm_f=[r(h, w) for h, w in sizes], tag_f=r(*sizes[0]))
    return s


@pytest.mark.parametrize("sizes,out_hw,flip", [
    ([(40, 48), (80, 96), (160, 192)], (160, 192), True),      # S/4, S/2, S
    ([(40, 48), (80, 96), (160, 192)], (160, 192), False),
    ([(72, 88)] * 4, (144, 176), True),                         # four equal stages
    ([(30, 50), (60, 100), (90, 150), (90, 150)], (180, 300), False),
])
def test_three_and_four_stages(sizes, out_hw, flip, oracle):
    s = _stages(2, sizes, flip, seed=len(sizes) + flip)
    got = _decode([s], *out_hw)
    _check_oracle(got, [s], *out_hw, oracle)


@pytest.mark.parametrize("flip", [True, False])
def test_multi_scale_single_stage(flip, oracle):
    H, W = 256, 192
    scales = [_stages(2, [(int(H / 4 * r), int(W / 4 * r))], flip, seed=int(10 * r)) for r in (0.5, 1.0, 1.5)]
    got = _decode(scales, H, W, tag_scale=1)
    _check_oracle(got, scales, H, W, oracle, tag_scale=1)


# ---- two stages through hpd_decode_stages -------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["x2", "ms", "generic"])
def test_two_stages_decode_stages_equals_decode(layout):
    from hpdecode import synth
    if layout == "ms":       # a half-size scale next to the full one: the multi-scale kernel
        H = W = 256
        full = synth.crowd(2, H, persons=4, flip=True, seed=3)[0]
        host = [{k: np.ascontiguousarray(v[:, :, ::2, ::2]) for k, v in full.items()}, full]
        ts = 1
    else:
        H = W = 256 if layout == "x2" else 248
        host = synth.crowd(2, H, persons=4, flip=True, seed=3)
        ts = 0
    scales = [{k: torch.from_numpy(v).cuda() for k, v in s.items()} for s in host]

    def legacy(p, bufs):
        L = _lib.lib()
        arr, _keep = ops._scales_struct(scales)
        ws = bufs.ensure_workspace(p)
        rc = L.hpd_decode(ctypes.byref(p), arr, ctypes.byref(bufs.struct()), ws.data_ptr(), ws.numel(),
                          torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "hpd_decode")
    want = _decode(scales, H, W, tag_scale=ts, call=legacy)
    got = _decode([ops.stage_scale(s) for s in scales], H, W, tag_scale=ts)
    _assert_same(got, want, f"decode_stages vs decode ({layout})")
    assert np.array_equal(_bits(got.tag_bmin), _bits(want.tag_bmin)) and np.array_equal(_bits(got.tag_bmax), _bits(want.tag_bmax))


# ---- tag-less sets, pipelines and CUDA graphs on single-stage inputs -----------------------------------------------
def test_single_stage_pipeline_graphs_and_tagless_sets():
    from hpdecode import BottomUpDecoder, DecodePipeline
    s = _single_stage(4, 64, 64, True, F32, seed=21)
    dec = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0")
    want = dec.decode([s], (256, 256), slot=50).records.clone()
    kept = BottomUpDecoder(17, 30, 0.05, 0.5, "cuda:0", keep_tag_map=True).decode([s], (256, 256))
    assert torch.equal(kept.records, want)
    lazy = dec.decode([s], (256, 256), slot=51)
    assert torch.equal(lazy.agg_tags, kept.agg_tags)
    for graphs in (False, True):
        pipe = DecodePipeline(dec, depth=2, use_graphs=graphs)
        res = [pipe.submit([s], (256, 256)) for _ in range(3)]
        pipe.drain()
        torch.cuda.synchronize()
        assert torch.equal(res[-1].records, want)
        if graphs:
            assert pipe.graph_replays == 3


def test_decode_stages_op():
    s = _single_stage(2, 64, 64, True, F32, seed=8)
    outs = torch.ops.hpd.decode_stages(s["hm"], s["hm_f"], [s["tag"]], [s["tag_f"]], 1, 256, 256, 30, 0.05, 0.5,
                                       True, True, 0)
    want = _decode([s], 256, 256)
    assert torch.equal(outs[0], want.agg_hm) and torch.equal(outs[2], want.poses)
    with pytest.raises(_lib.HpdError):
        torch.ops.hpd.decode_stages(s["hm"] * 5, [], [s["tag"]], [], 5, 256, 256, 30, 0.05, 0.5, True, True, 0)


# ---- InferenceKeypointsModel with 1- and 3-stage heads ------------------------------------------------------------
class _CaptureNet(nn.Module):
    """Keeps every call's outputs up-cast to float32 on the host."""

    def __init__(self, net):
        super().__init__()
        self.net, self.calls = net, []

    def forward(self, x):
        hms, tag = self.net(x)
        self.calls.append(([h.detach().float().cpu().numpy() for h in hms], tag.detach().float().cpu().numpy(),
                           {t.dtype for t in list(hms) + [tag]}))
        return hms, tag


@pytest.mark.parametrize("num_deconvs", [0, 2])
@pytest.mark.parametrize("dtype", [None, BF16])
def test_model_with_other_heads(num_deconvs, dtype, oracle):
    from hpdecode import InferenceKeypointsModel, synth_net
    from oracle import input_oracle
    from oracle.gen_golden_input import image_of
    torch.manual_seed(4)
    net = _CaptureNet(synth_net.HigherHRNet(17, 32, num_deconvs))
    size = 256
    model = InferenceKeypointsModel(net, use_flip=True, input_size=size, device="cuda:0", autocast_dtype=dtype)
    raws = [image_of(300, 421, 11), image_of(300, 421, 12)]
    f32 = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)

    def oracle_of(calls, b):
        (hms, tag, dts), (hms_f, tag_f, _) = calls
        assert dts == ({dtype} if dtype is not None else {torch.float32})
        assert len(hms) == num_deconvs + 1
        s = {"hm": [h[b] for h in hms], "hm_f": [h[b] for h in hms_f], "tag": tag[b], "tag_f": tag_f[b]}
        (W, H), center, scale = input_oracle.get_multi_scale_size(300, 421, size, 1.0, 1.0)
        hm_o, tg_o = stage_oracle.aggregate([s], (H, W))
        ref = oracle.parse(hm_o, tg_o, 30, 0.05, 0.5)
        minv = input_oracle.get_affine_transform(center, scale, (W, H), inverse=True)
        gj = ref["grouped_joints"]
        coords = input_oracle.affine_points(gj[..., :2].reshape(-1, 2), minv).reshape(gj.shape[0], -1, 2)
        return hm_o, tg_o, gj, ref["person_scores"], coords.astype(np.float32)

    one = model(raws[0], None)
    hm_o, tg_o, gj, ps, coords = oracle_of(net.calls[-2:], 0)
    assert np.array_equal(f32(one.kpts_heatmaps), f32(hm_o)) and np.array_equal(f32(one.tags_heatmaps), f32(tg_o[..., 0]))
    assert np.array_equal(f32(one.kpts_coords), f32(coords)) and np.array_equal(f32(one.obj_scores), f32(ps))
    assert np.array_equal(f32(one.kpts_scores), f32(gj[..., 2])) and np.array_equal(f32(one.kpts_tags), f32(gj[..., 3:]))
    batch = model.predict_batch(raws)
    for b, r in enumerate(batch):
        _, _, gj, ps, coords = oracle_of(net.calls[-2:], b)
        assert np.array_equal(f32(r.kpts_coords), f32(coords)) and np.array_equal(f32(r.obj_scores), f32(ps))
    streamed = list(model.stream(raws, batch_size=2, depth=2))
    for r, w in zip(streamed, batch):
        assert np.array_equal(f32(r.kpts_coords), f32(w.kpts_coords)) and np.array_equal(f32(r.obj_scores), f32(w.obj_scores))


@pytest.mark.parametrize("n", [1, 3])
def test_from_preds_and_set_preds(n, oracle):
    from hpdecode import KeypointsResult, InferenceKeypointsResult, geometry
    from oracle import input_oracle
    K, H, W = 17, 256, 192
    g = torch.Generator().manual_seed(n)
    sizes = [(H // 4, W // 4), (H // 2, W // 2), (H, W)][:n] if n == 3 else [(H // 4, W // 4)]
    hms = [torch.randn(1, K, h, w, generator=g) * 0.3 for h, w in sizes]
    tag = torch.randn(1, K, H // 4, W // 4, generator=g)
    x = torch.zeros(3, H, W)
    center, scale = (150, 100), (300.0, 200.0)
    res = InferenceKeypointsResult.from_preds(np.zeros((200, 300, 3), np.uint8), None, x, [h.cuda() for h in hms],
                                              [tag.cuda()], None, scale, center)
    s = {"hm": [h[0].numpy() for h in hms], "tag": tag[0].numpy()}
    hm_o, tg_o = stage_oracle.aggregate([s], (H, W))
    ref = oracle.parse(hm_o, tg_o, 30, 0.05, 0.5)
    f32 = lambda a: np.ascontiguousarray(a, np.float32).view(np.uint32)
    assert np.array_equal(f32(res.kpts_heatmaps), f32(hm_o))
    assert np.array_equal(f32(res.kpts_scores), f32(ref["grouped_joints"][..., 2]))
    minv = geometry.get_affine_transform(center, scale, 0, (W, H), inverse=True)
    gj = ref["grouped_joints"]
    want = input_oracle.affine_points(gj[..., :2].reshape(-1, 2), minv).reshape(gj.shape[0], -1, 2).astype(np.float32)
    assert np.array_equal(f32(res.kpts_coords), f32(want))
    kr = KeypointsResult(x, [h.cuda() for h in hms], tag.cuda(), None)
    kr.set_preds()
    assert np.array_equal(f32(kr.kpts_coords), f32(gj[..., :2])) and np.array_equal(f32(kr.obj_scores), f32(ref["person_scores"]))
    assert kr.kpts_heatmaps.shape == (K, H, W, n)
