"""CPU suite for the frame-stream path: argument validation of hpd_prepare_inputs (every rejection happens before a
launch), the layout of its ctypes struct, and FrameStream's batching / ordering logic with the device work stubbed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _args(batch=2, n_targets=2, flip=True):
    from hpdecode import _lib
    imgs = (_lib.HpdImage * (batch * n_targets))()
    for im in imgs:
        im.ptr, im.h, im.w, im.stride_row = 64, 10, 12, 36
        im.m[0] = im.m[4] = 1.0
    tg = (_lib.HpdPrepareTarget * max(n_targets, 1))()
    for t in range(n_targets):
        tg[t].out, tg[t].out_flipped, tg[t].out_h, tg[t].out_w = 4096 * (t + 1), (4096 * (t + 9)) if flip else None, 8, 16
    mean, std = (ctypes.c_float * 3)(0.5, 0.5, 0.5), (ctypes.c_float * 3)(0.2, 0.2, 0.2)
    return imgs, tg, mean, std


def _rejects(L, *a, what):
    rc = L.hpd_prepare_inputs(*a)
    msg = L.hpd_last_error_string()
    assert rc == 1, what
    assert msg.startswith(b"hpd_prepare_inputs"), (what, msg)
    assert L.hpd_last_launch_count() == 0, what
    return msg


def test_prepare_inputs_validates_before_any_launch():
    from hpdecode import _lib
    L = _lib.lib()
    imgs, tg, mean, std = _args()
    _rejects(L, None, 2, tg, 2, mean, std, None, what="no images")
    _rejects(L, imgs, 2, None, 2, mean, std, None, what="no targets")
    _rejects(L, imgs, 2, tg, 2, None, std, None, what="no mean")
    _rejects(L, imgs, 2, tg, 2, mean, None, None, what="no std")
    _rejects(L, imgs, 0, tg, 2, mean, std, None, what="batch 0")
    _rejects(L, imgs, 2, tg, 0, mean, std, None, what="no target")
    _rejects(L, imgs, 2, tg, _lib.HPD_MAX_SCALES + 1, mean, std, None, what="too many targets")
    for field, value, name in (("out", None, "no output"), ("out_h", 0, "height 0"), ("out_w", -3, "width < 0"),
                               ("out_h", 65535 * 16 + 1, "too tall")):
        imgs, tg, mean, std = _args()
        setattr(tg[1], field, value)
        assert b"target 1" in _rejects(L, imgs, 2, tg, 2, mean, std, None, what=name)
    imgs, tg, mean, std = _args()
    tg[0].out_flipped = tg[0].out
    assert b"out_flipped" in _rejects(L, imgs, 2, tg, 2, mean, std, None, what="out == out_flipped")
    # a bad image anywhere -- the last one included -- rejects the whole call, nothing is launched for the others
    for field, value in (("ptr", None), ("h", 0), ("w", 0), ("h", 40000), ("w", 40000), ("stride_row", 35)):
        imgs, tg, mean, std = _args()
        setattr(imgs[3], field, value)
        assert b"target 1 image 1" in _rejects(L, imgs, 2, tg, 2, mean, std, None, what=field)
    imgs, tg, mean, std = _args(batch=40, n_targets=1, flip=False)
    imgs[39].ptr = None                                     # past the first launch's 32 images
    assert b"image 39" in _rejects(L, imgs, 40, tg, 1, mean, std, None, what="second launch's image")


def test_prepare_target_struct_matches_c_layout(tmp_path):
    from hpdecode import _lib
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){printf("%zu %zu %zu %zu\\n",'
                     "sizeof(HpdPrepareTarget),offsetof(HpdPrepareTarget,out_flipped),offsetof(HpdPrepareTarget,out_h),"
                     "offsetof(HpdPrepareTarget,out_w));return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    T = _lib.HpdPrepareTarget
    assert got == [ctypes.sizeof(T), T.out_flipped.offset, T.out_h.offset, T.out_w.offset]


def test_multi_scale_geometry_matches_per_scale_calls():
    """geometry.multi_scale_geometry: one prepare_geometry per scale, the scale-1.0 frame returned for the decode."""
    from hpdecode import geometry
    shapes = [(480, 640), (481, 641)]
    sizes_hw, fwd, (centers, scales, inv) = geometry.multi_scale_geometry(shapes, 512, (0.5, 1.0, 1.5))
    assert fwd.shape == (3, 2, 6)
    for t, s in enumerate((0.5, 1.0, 1.5)):
        sz, c, sc, f, i = geometry.prepare_geometry(shapes, 512, s, 0.5)
        assert sizes_hw[2 * t:2 * t + 2] == [int(sz[0, 1]), int(sz[0, 0])] and np.array_equal(fwd[t], f)
        if s == 1.0:
            assert np.array_equal(inv, i) and np.array_equal(centers, c) and np.array_equal(scales, sc)
    with pytest.raises(ValueError):
        geometry.multi_scale_geometry(shapes, 512, (0.5, 1.5))
    with pytest.raises(Exception, match="share the resized size"):
        geometry.multi_scale_geometry([(480, 640), (100, 300)], 512, (1.0,))


class _Model:
    input_size, test_scales = 256, (1.0,)


def _stub_stream(batch_size, depth):
    """FrameStream with the device hooks replaced: a 'batch' is the list of frame ids it holds, and it finishes when
    the stream retires it; the geometry cache is the real one.  Records which batches were launched and how many were
    in flight at each launch."""
    import torch
    from hpdecode.stream import FrameStream

    class Stub(FrameStream):
        def _init_device(self):
            self.device = torch.device("cpu")           # the geometry cache's matrices stay on the host
            self.launched, self.peak, self.staged = [], 0, []

        def _stage(self, f, i):
            self.staged.append((int(f[0, 0, 0]), i))

        def _launch(self, frames, hw):
            sizes_hw, fwd, inv = self._geometry(hw, len(frames))
            assert fwd.shape == (1, len(frames), 6) and inv.shape == (len(frames), 6)
            ids = [int(f[0, 0, 0]) for f in frames]
            self.launched.append((hw, ids))
            self.peak = max(self.peak, len(self._inflight) + 1)
            return ids

        def _ready(self, batch):
            return len(batch) % 2 == 1      # some batches "still running": results(wait=False) must not pass them

        def _finish(self, batch):
            return list(batch)

    return Stub(_Model(), batch_size, depth)


def _frame(i, h=4, w=6):
    f = np.zeros((h, w, 3), np.uint8)
    f[0, 0, 0] = i
    return f


@pytest.mark.parametrize("batch_size,depth", [(1, 1), (5, 1), (5, 4), (8, 4), (30, 2)])
def test_stream_batches_in_order(batch_size, depth):
    fs = _stub_stream(batch_size, depth)
    got = []
    for i in range(23):
        fs.submit([_frame(i)])
        got += list(fs.results(wait=False))
        assert len(fs._inflight) <= depth
    got += list(fs.results())
    assert got == list(range(23))
    assert [ids for _, ids in fs.launched] == [list(range(b, min(b + batch_size, 23))) for b in range(0, 23, batch_size)]
    assert fs.peak <= depth and fs.geometry_calls == 1
    assert [i for _, i in fs.staged] == [i % batch_size for i in range(23)]     # slot within the batch
    assert list(fs.results()) == [] and not fs._inflight and not fs._open


def test_stream_size_change_closes_the_batch():
    fs = _stub_stream(4, 2)
    sizes = [(4, 6)] * 3 + [(6, 4)] * 2 + [(4, 6)] + [(6, 4)] * 6
    fs.submit(_frame(i, *hw) for i, hw in enumerate(sizes))
    assert list(fs) == list(range(len(sizes)))
    assert fs.launched == [((4, 6), [0, 1, 2]), ((6, 4), [3, 4]), ((4, 6), [5]), ((6, 4), [6, 7, 8, 9]),
                           ((6, 4), [10, 11])]
    assert fs.geometry_calls == 2


def test_stream_rejects_bad_frames():
    from hpdecode import _lib
    fs = _stub_stream(4, 2)
    for bad in (np.zeros((4, 6), np.uint8), np.zeros((4, 6, 4), np.uint8), np.zeros((4, 6, 3), np.float32), [[1, 2, 3]]):
        with pytest.raises(_lib.HpdError, match="uint8"):
            fs.submit([bad])
    with pytest.raises(ValueError):
        _stub_stream(0, 2)


def test_stream_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from hpdecode import FrameStream, _lib
    with pytest.raises(_lib.HpdError):
        FrameStream(_Model())
    with pytest.raises(_lib.HpdError):
        torch.ops.hpd.prepare_inputs([torch.zeros(4, 6, 3, dtype=torch.uint8)], torch.zeros(1, 1, 6, dtype=torch.float64),
                                     [8, 8], True, [0.5] * 3, [0.2] * 3)


def test_prepare_inputs_fake_shapes():
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    import hpdecode  # noqa: F401
    with FakeTensorMode():
        imgs = [torch.empty(10, 12, 3, dtype=torch.uint8) for _ in range(3)]
        xs, xs_f = torch.ops.hpd.prepare_inputs(imgs, torch.empty(2, 3, 6, dtype=torch.float64), [8, 16, 24, 32], True,
                                                [0.0] * 3, [1.0] * 3)
        assert [tuple(x.shape) for x in xs] == [(3, 3, 8, 16), (3, 3, 24, 32)] and len(xs_f) == 2
        assert xs[1].dtype == torch.float32 and tuple(xs_f[1].shape) == (3, 3, 24, 32)
        xs, xs_f = torch.ops.hpd.prepare_inputs(imgs, torch.empty(1, 3, 6, dtype=torch.float64), [8, 16], False,
                                                [0.0] * 3, [1.0] * 3)
        assert len(xs) == 1 and xs_f == []
