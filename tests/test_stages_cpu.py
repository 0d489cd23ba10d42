"""CPU suite for heads with 1 to 4 heatmap stages: the oracle's n-stage aggregation against torch's own calls, the
HpdStageInputs layout, and the argument checks of hpd_aggregate_nms_stages / hpd_decode_stages (made before any
launch, so they run without a GPU)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import cpu_oracle, py_port, ref_runner, stage_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PTR = 1 << 20

# (stage sizes, output size): every resize target is larger than 64 on a side
LAYOUTS = {
    "single_s4": ([(40, 34)], (160, 136)),
    "s4_s2_s": ([(40, 34), (80, 68), (160, 136)], (160, 136)),
    "four_equal": ([(72, 88)] * 4, (144, 176)),
    "nonsquare_3": ([(30, 50), (60, 100), (90, 150)], (180, 300)),
    "two_nonsquare": ([(34, 40), (68, 80)], (136, 160)),
}


def _scale(sizes, flip, seed, K=17):
    rng = np.random.default_rng(seed)
    f = lambda h, w: rng.standard_normal((K, h, w)).astype(np.float32)
    th, tw = sizes[0]
    s = {"hm": [f(h, w) for h, w in sizes], "tag": f(th, tw)}
    if flip:
        s.update(hm_f=[f(h, w) for h, w in sizes], tag_f=f(th, tw))
    return s


def _bits(t):
    a = t.numpy() if isinstance(t, torch.Tensor) else t
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("flip", [True, False])
def test_stage_oracle_equals_the_torch_replay(layout, flip):
    sizes, out_hw = LAYOUTS[layout]
    scales = [_scale(sizes, flip, seed=len(sizes) * 10 + flip)]
    hm_t, tg_t = stage_oracle.aggregate_torch(scales, out_hw)
    hm_o, tg_o = stage_oracle.aggregate(scales, out_hw)
    assert np.array_equal(_bits(hm_o), _bits(hm_t)) and np.array_equal(_bits(tg_o), _bits(tg_t))


@pytest.mark.parametrize("flip", [True, False])
def test_multi_scale_single_stage_equals_the_torch_replay(flip):
    out_hw = (192, 160)
    scales = [_scale([(int(48 * r), int(40 * r))], flip, seed=i) for i, r in enumerate((0.5, 1.0, 1.5))]
    hm_t, tg_t = stage_oracle.aggregate_torch(scales, out_hw, tag_scale=1)
    hm_o, tg_o = stage_oracle.aggregate(scales, out_hw, tag_scale=1)
    assert np.array_equal(_bits(hm_o), _bits(hm_t)) and np.array_equal(_bits(tg_o), _bits(tg_t))


@pytest.mark.parametrize("sizes,out_hw", [([(36, 44), (72, 88)], (144, 176)), ([(34, 40), (68, 80)], (136, 160))])
@pytest.mark.parametrize("flip", [True, False])
@pytest.mark.parametrize("n_scales", [1, 2])
def test_two_stages_equal_the_existing_oracles(sizes, out_hw, flip, n_scales):
    """For the two-stage head the stage oracle and its torch replay give what the C++ oracle, the Python port and the
    reference replay give, bit for bit, with stage lists and with hm_lo / hm_hi dicts alike."""
    stage = [_scale(sizes, flip, seed=3 + i) for i in range(n_scales)]
    legacy = []
    for s in stage:
        d = {"hm_lo": s["hm"][0], "hm_hi": s["hm"][1], "tag": s["tag"]}
        if flip:
            d.update(hm_lo_f=s["hm_f"][0], hm_hi_f=s["hm_f"][1], tag_f=s["tag_f"])
        legacy.append(d)
    ts = n_scales - 1
    want_hm, want_tg = cpu_oracle.aggregate(legacy, out_hw, tag_scale=ts)
    for hm, tg in (py_port.aggregate(legacy, out_hw, tag_scale=ts), ref_runner.aggregate_torch(legacy, out_hw, tag_scale=ts),
                   stage_oracle.aggregate(stage, out_hw, tag_scale=ts), stage_oracle.aggregate(legacy, out_hw, tag_scale=ts),
                   stage_oracle.aggregate_torch(stage, out_hw, tag_scale=ts)):
        assert np.array_equal(_bits(hm), _bits(want_hm)) and np.array_equal(_bits(tg), _bits(want_tg))


def test_stage_inputs_layout_matches_c(tmp_path):
    from hpdecode import _lib
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){printf("%zu %zu %zu %zu '
                     '%zu %d\\n",sizeof(HpdStageInputs),offsetof(HpdStageInputs,hm_f),offsetof(HpdStageInputs,tag),'
                     'offsetof(HpdStageInputs,tag_f),offsetof(HpdStageInputs,num_stages),HPD_MAX_STAGES);return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    S = _lib.HpdStageInputs
    assert got == [ctypes.sizeof(S), S.hm_f.offset, S.tag.offset, S.tag_f.offset, S.num_stages.offset,
                   _lib.HPD_MAX_STAGES]


def _map(h, w, dtype=0):
    from hpdecode import _lib
    m = _lib.HpdMap()
    m.ptr, m.h, m.w, m.dtype = PTR, h, w, dtype
    m.stride_c, m.stride_b = h * w, 17 * h * w
    return m


def _stages(n, flip=True, dtype=0, size=64):
    from hpdecode import _lib
    s = _lib.HpdStageInputs()
    s.num_stages = n
    for i in range(min(n, _lib.HPD_MAX_STAGES)):
        s.hm[i] = _map(size, size, dtype)
        if flip:
            s.hm_f[i] = _map(size, size, dtype)
    s.tag = _map(size, size, dtype)
    if flip:
        s.tag_f = _map(size, size, dtype)
    return s


def _call(stages, E=2, decode=False):
    from hpdecode import _lib, ops
    L = _lib.lib()
    p = ops.make_params(1, 17, 256, 256, E, 30, 0.05, 0.5, num_scales=len(stages))
    arr = (_lib.HpdStageInputs * len(stages))(*stages)
    b = _lib.HpdBuffers()
    for n in ("agg_hm", "nms_mask", "nms_wmax", "hm_wmax", "tag_bmin", "tag_bmax"):
        setattr(b, n, PTR)
    if decode:
        rc = L.hpd_decode_stages(ctypes.byref(p), arr, ctypes.byref(b), ctypes.c_void_p(PTR), 0, None)
    else:
        rc = L.hpd_aggregate_nms_stages(ctypes.byref(p), arr, ctypes.byref(b), None)
    return rc, L.hpd_last_error_string().decode()


@pytest.mark.parametrize("decode", [False, True])
@pytest.mark.parametrize("n", [0, 5, -1])
def test_num_stages_out_of_range(n, decode):
    rc, msg = _call([_stages(n)], decode=decode)
    assert rc == 1 and f"num_stages must be in [1,4] (got {n})" in msg, msg


@pytest.mark.parametrize("decode", [False, True])
def test_missing_stage(decode):
    s = _stages(3)
    s.hm[1] = type(s.hm[1])()
    rc, msg = _call([s], decode=decode)
    assert rc == 1 and "hm[1]: missing" in msg, msg


@pytest.mark.parametrize("decode", [False, True])
def test_flipped_stage_mismatch(decode):
    s = _stages(3)
    s.hm_f[2] = type(s.hm_f[2])()                       # one flipped stage missing
    rc, msg = _call([s], decode=decode)
    assert rc == 1 and "flip inputs must be given for all stages and scales or for none" in msg, msg
    s = _stages(3)
    s.hm_f[1] = _map(32, 64)                            # one flipped stage of another shape
    rc, msg = _call([s], decode=decode)
    assert rc == 1 and "flipped-run maps must have the shapes of the un-flipped run" in msg, msg
    rc, msg = _call([_stages(1, flip=False), _stages(1)], decode=decode)   # flip on one scale only
    assert rc == 1 and "flip inputs" in msg, msg


@pytest.mark.parametrize("decode", [False, True])
def test_mixed_dtypes(decode):
    s = _stages(4, dtype=2)
    s.hm_f[3] = _map(64, 64, 1)
    rc, msg = _call([s], decode=decode)
    assert rc == 1 and "share one dtype" in msg, msg
    rc, msg = _call([_stages(1, dtype=2), _stages(1, dtype=0)], decode=decode)
    assert rc == 1 and "share one dtype" in msg, msg


def test_python_stage_format():
    from hpdecode import _lib, ops
    a, b, t = object(), object(), object()
    s = ops.stage_scale({"hm_lo": a, "hm_hi": b, "tag": t})
    assert s["hm"] == [a, b] and s["hm_f"] == [] and s["tag"] is t and s["tag_f"] is None
    same = {"hm": [a], "hm_f": [], "tag": t, "tag_f": None}
    assert ops.stage_scale(same) is same
    with pytest.raises(_lib.HpdError, match="1 to 4 heatmap stages"):
        ops._stages_struct([{"hm": [], "tag": None}])
    with pytest.raises(_lib.HpdError, match="1 to 4 heatmap stages"):
        ops._stages_struct([{"hm": [torch.zeros(1)] * 5, "tag": None}])


def test_synthetic_network_stage_counts():
    from hpdecode import synth_net
    torch.manual_seed(0)
    x = torch.randn(1, 3, 64, 64)
    for nd, shapes in ((0, [(16, 16)]), (1, [(16, 16), (32, 32)]), (2, [(16, 16), (32, 32), (64, 64)])):
        net = synth_net.HigherHRNet(17, 8, num_deconvs=nd).eval()
        with torch.no_grad():
            hms, tag = net(x)
        assert [tuple(h.shape[-2:]) for h in hms] == shapes and tuple(tag.shape) == (1, 17, 16, 16)
        assert hms[0].stride(0) == 2 * 17 * 16 * 16                  # channel slice of the 2K-channel head
    with pytest.raises(ValueError):
        synth_net.HigherHRNet(17, 8, num_deconvs=3)
