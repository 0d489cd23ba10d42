"""CPU suite: ABI 6's dtype codes.  HPD_BF16 is accepted wherever HPD_F16 is, mixed dtypes and unknown codes are
refused, and hpd_resize_bilinear stays float32-only.  Every call below fails validation before any launch (the
message says which check it reached), so the pointers are never dereferenced and the tests need no GPU."""
import ctypes

import pytest

from hpdecode import _lib, ops

PTR = 1 << 20          # never dereferenced: every call fails validation before a launch


def _map(h, w, dtype):
    m = _lib.HpdMap()
    m.ptr, m.stride_c, m.h, m.w, m.dtype = PTR, h * w, h, w, dtype
    m.stride_b = 17 * m.stride_c
    return m


def _scale(dtype, flip, lh=64, lw=64, **dtypes):
    s = _lib.HpdScaleInputs()
    names = ("hm_lo", "hm_hi", "tag") + (("hm_lo_f", "hm_hi_f", "tag_f") if flip else ())
    for n in names:
        f = 2 if n.startswith("hm_hi") else 1
        setattr(s, n, _map(lh * f, lw * f, dtypes.get(n, dtype)))
    return s


def _aggregate(scales, E):
    L = _lib.lib()
    p = ops.make_params(1, 17, 256, 256, E, 30, 0.05, 0.5, num_scales=len(scales))
    arr = (_lib.HpdScaleInputs * len(scales))(*scales)
    b = _lib.HpdBuffers()
    for n in ("agg_hm", "nms_mask", "nms_wmax", "hm_wmax", "tag_bmin", "tag_bmax"):
        setattr(b, n, PTR)
    rc = L.hpd_aggregate_nms(ctypes.byref(p), arr, ctypes.byref(b), None)
    return rc, L.hpd_last_error_string().decode()


def test_abi_version_6_and_dtype_codes():
    assert _lib.HPD_ABI_VERSION == 6 and _lib.lib().hpd_abi_version() == 6
    assert (_lib.HPD_F32, _lib.HPD_F16, _lib.HPD_BF16) == (0, 1, 2)
    src = open(_lib.os.path.join(_lib.os.path.dirname(_lib._HERE), "..", "include", "hpdecode.h")).read()
    assert "HPD_BF16 = 2" in src and "#define HPD_ABI_VERSION 6" in src


@pytest.mark.parametrize("dtype", [0, 1, 2])
def test_aggregate_accepts_every_dtype_code(dtype):
    """A flip set with the flipped half-res map missing fails on the flip rule, which comes after the dtype checks."""
    s = _scale(dtype, True)
    s.hm_hi_f = _lib.HpdMap()
    rc, msg = _aggregate([s], 2)
    assert rc == 1 and "flip inputs" in msg, msg


@pytest.mark.parametrize("dtype", [3, 7, -1])
def test_aggregate_rejects_unknown_dtype_codes(dtype):
    rc, msg = _aggregate([_scale(dtype, True)], 2)
    assert rc == 1 and f"unsupported dtype code {dtype}" in msg, msg


@pytest.mark.parametrize("a,b,name", [(2, 1, "hm_hi"), (1, 2, "tag"), (2, 0, "tag_f"), (0, 2, "hm_lo_f")])
def test_aggregate_rejects_mixed_dtypes(a, b, name):
    rc, msg = _aggregate([_scale(a, True, **{name: b})], 2)
    assert rc == 1 and "share one dtype" in msg, msg


def test_aggregate_rejects_mixed_dtypes_across_scales():
    rc, msg = _aggregate([_scale(2, False, 32, 32), _scale(1, False)], 1)
    assert rc == 1 and "share one dtype" in msg, msg


def _tag_inputs(dtype, dtype_f=None):
    s = _lib.HpdScaleInputs()
    s.tag = _map(64, 64, dtype)
    if dtype_f is not None:
        s.tag_f = _map(64, 64, dtype_f)
    return s


@pytest.mark.parametrize("dtype,ok", [(0, True), (1, True), (2, True), (3, False), (7, False)])
def test_tag_stages_read_bf16_tags(dtype, ok):
    """hpd_aggregate_tags, hpd_topk and hpd_adjust_refine read tag-scale maps through one tag source: a known dtype
    gets past it (to the emb rule / the workspace check), an unknown one is refused there."""
    L = _lib.lib()
    p = ops.make_params(1, 17, 256, 256, 2, 30, 0.05, 0.5)
    arr = (_lib.HpdScaleInputs * 1)(_tag_inputs(dtype))           # emb = 2 but no flipped tag map
    rc = L.hpd_aggregate_tags(ctypes.byref(p), arr, ctypes.c_void_p(PTR), None)
    msg = L.hpd_last_error_string().decode()
    assert rc == 1 and (("emb must be 2" in msg) if ok else ("missing or malformed" in msg)), msg
    b = _lib.HpdBuffers()
    for n in ("agg_hm", "nms_mask", "nms_wmax", "hm_wmax", "scores_k", "idx_k", "coords_k", "tags_k", "poses",
              "person_scores", "n_person", "flags", "tag_bmin", "tag_bmax"):
        setattr(b, n, PTR)
    b.tag_inputs = _tag_inputs(dtype)
    assert L.hpd_topk(ctypes.byref(p), ctypes.byref(b), None) == 1
    msg = L.hpd_last_error_string().decode()
    assert ("emb must be 2" in msg) if ok else ("missing or malformed" in msg), msg
    b.tag_inputs = _tag_inputs(dtype, dtype)
    rc = L.hpd_adjust_refine(ctypes.byref(p), ctypes.byref(b), ctypes.c_void_p(PTR), 0, None)
    msg = L.hpd_last_error_string().decode()
    assert rc == (2 if ok else 1), msg                             # HPD_EWORKSPACE past the tag source
    assert ("workspace of" in msg) if ok else ("missing or malformed" in msg), msg


@pytest.mark.parametrize("dtype_f", [0, 1])
def test_tag_stages_reject_mixed_tag_dtypes(dtype_f):
    L = _lib.lib()
    p = ops.make_params(1, 17, 256, 256, 2, 30, 0.05, 0.5)
    arr = (_lib.HpdScaleInputs * 1)(_tag_inputs(2, dtype_f))
    assert L.hpd_aggregate_tags(ctypes.byref(p), arr, ctypes.c_void_p(PTR), None) == 1
    assert b"shape and dtype" in L.hpd_last_error_string()


@pytest.mark.parametrize("dtype", [1, 2])
def test_resize_stays_float32_only(dtype):
    L = _lib.lib()
    m = _map(4, 4, dtype)
    assert L.hpd_resize_bilinear(ctypes.byref(m), 1, 1, ctypes.c_void_p(PTR), 8, 8, None) == 1
    assert b"bad arguments" in L.hpd_last_error_string()


def test_python_maps_carry_the_dtype_code():
    """ops._map gives 16-bit CUDA tensors their code; without a device a CPU tensor of any dtype is refused."""
    import torch
    assert ops._DTYPE_CODES == {torch.float16: _lib.HPD_F16, torch.bfloat16: _lib.HPD_BF16}
    for dt in (torch.float16, torch.bfloat16, torch.float32):
        with pytest.raises(_lib.HpdError):
            ops._map(torch.zeros(1, 17, 8, 8, dtype=dt), "hm_lo", allow_16bit=True)
