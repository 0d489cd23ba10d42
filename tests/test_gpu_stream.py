"""-m gpu: the frame-stream path.  hpd_prepare_inputs against hpd_prepare_input + torch.flip (bit for bit, launch
splitting, strided rows), and FrameStream / model.stream against predict_batch and the CPU oracle.

The network outputs are compared across runs, so cuDNN is pinned to deterministic algorithms here, and every
reference run uses the batch composition the stream used (an algorithm may depend on the batch size).
"""
import ctypes
import os

import numpy as np
import pytest
import torch
from torch import nn

from oracle import input_oracle
from oracle.gen_golden_input import CASES, image_of, sha

pytestmark = pytest.mark.gpu

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "input_cases.npz"))
MS = (0.5, 1.0, 1.5)


@pytest.fixture(autouse=True, scope="module")
def _deterministic():
    saved = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    yield
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = saved


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _call_prepare_inputs(imgs, fwd, sizes_hw, flip):
    """hpd_prepare_inputs through the C ABI into NaN-poisoned outputs -> (xs, xs_flipped, launches)."""
    from hpdecode import _lib, geometry, ops
    T, B = fwd.shape[:2]
    xs = [torch.full((B, 3, sizes_hw[2 * t], sizes_hw[2 * t + 1]), float("nan"), device="cuda:0") for t in range(T)]
    xs_f = [torch.full_like(x, float("nan")) for x in xs] if flip else []
    arr = ops._image_descriptors(imgs, fwd.reshape(-1, 6).tolist(), "test")
    tg = (_lib.HpdPrepareTarget * T)()
    for t in range(T):
        tg[t].out, tg[t].out_h, tg[t].out_w = xs[t].data_ptr(), sizes_hw[2 * t], sizes_hw[2 * t + 1]
        tg[t].out_flipped = xs_f[t].data_ptr() if flip else None
    L = _lib.lib()
    mean, std = (ctypes.c_float * 3)(*geometry.MEAN), (ctypes.c_float * 3)(*geometry.STD)
    _lib.check(L.hpd_prepare_inputs(arr, B, tg, T, mean, std, torch.cuda.current_stream().cuda_stream), "hpd_prepare_inputs")
    return xs, xs_f, L.hpd_last_launch_count()


def _single(imgs, fwd_t, h, w):
    from hpdecode import geometry
    return torch.ops.hpd.prepare_input(imgs, torch.from_numpy(np.ascontiguousarray(fwd_t)), h, w, list(geometry.MEAN),
                                       list(geometry.STD))


@pytest.mark.parametrize("i", range(len(CASES)))
def test_prepare_inputs_matches_goldens(i):
    """Scale 1.0 of every golden case: the reference's tensor (SHA-256), and its mirror."""
    from hpdecode import geometry
    h, w, input_size, seed = CASES[i]
    img = torch.from_numpy(image_of(h, w, seed)).cuda()
    sizes_hw, fwd, _ = geometry.multi_scale_geometry([(h, w)], input_size, (1.0,))
    xs, xs_f, launches = _call_prepare_inputs([img], fwd, sizes_hw, True)
    got = xs[0][0].cpu().numpy()
    assert launches == 1 and sha(got) == str(GOLD[f"c{i}_x_sha"])
    assert torch.equal(xs_f[0], torch.flip(xs[0], [3]))
    single = _single([img], fwd[0], *sizes_hw)
    assert np.array_equal(_bits(got), _bits(single[0].cpu().numpy()))


@pytest.mark.parametrize("batch", [1, 31, 32, 33, 70])
@pytest.mark.parametrize("flip", [False, True])
def test_prepare_inputs_equals_prepare_input_per_scale(batch, flip):
    """Scales 0.5 / 1.0 / 1.5 of a batch of odd-sized images whose rows are padded (stride > 3w): every target equal to
    hpd_prepare_input's output for the same descriptors, the mirrored copy to torch.flip; (scale, image) pairs are
    split 32 per launch."""
    from hpdecode import geometry
    rng = np.random.default_rng(batch)
    shapes = [(477, 641), (479, 639), (475, 643)]
    imgs = []
    for b in range(batch):
        h, w = shapes[b % 3]
        pad = int(rng.integers(1, 9))
        big = torch.from_numpy(rng.integers(0, 256, (h, w + pad, 3), dtype=np.uint8)).cuda()
        imgs.append(big[:, :w])
        assert imgs[-1].stride(0) == 3 * (w + pad)
    sizes_hw, fwd, _ = geometry.multi_scale_geometry([im.shape[:2] for im in imgs], 512, MS)
    xs, xs_f, launches = _call_prepare_inputs(imgs, fwd, sizes_hw, flip)
    assert launches == -(-3 * batch // 32)
    for t in range(3):
        want = _single(imgs, fwd[t], sizes_hw[2 * t], sizes_hw[2 * t + 1])
        assert not torch.isnan(xs[t]).any()
        assert torch.equal(xs[t].view(torch.int32), want.view(torch.int32)), t
        if flip:
            assert torch.equal(xs_f[t].view(torch.int32), torch.flip(want, [3]).view(torch.int32)), t
    if batch == 33:     # the oracle too, for an image of the second launch
        want = input_oracle.prepare_input(imgs[32].contiguous().cpu().numpy(), 512, 1.5, 0.5)[0]
        assert np.array_equal(_bits(xs[2][32].cpu().numpy()), _bits(want))


_KERNEL_PROBE = """
import json, sys, torch
sys.path[:0] = sys.argv[1:3]
from hpdecode import geometry, ops
img = torch.randint(0, 256, (480, 640, 3), dtype=torch.uint8, device="cuda:0")
torch.cuda.synchronize()
n0 = ops.launches_total()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    xs, xs_f, _, _ = geometry.prepare_inputs([img] * 11, 512, "cuda:0", (0.5, 1.0, 1.5), flip=True)
    torch.cuda.synchronize()
kernels = {}
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
        kernels[e.name] = kernels.get(e.name, 0) + 1
print(json.dumps({"kernels": kernels, "library_launches": ops.launches_total() - n0, "n_xs": len(xs), "n_xs_f": len(xs_f)}))
"""


def test_prepare_inputs_runs_its_own_kernel():
    """Which kernels a flip-test, three-scale prepare_inputs call runs on the device: the library's multi-target kernel,
    twice (33 (scale, image) pairs: 32 + 1), and nothing else -- no torch.flip, no copy, no per-scale kernel.  The
    profile is taken in a fresh process: in a long pytest process, earlier profiler sessions can leave CUPTI
    delivering the runtime calls but not the kernel records."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-s", "-c", _KERNEL_PROBE, root, os.path.join(root, "pytorch-human-pose_b200")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    got = json.loads(out.stdout.strip().splitlines()[-1])
    assert got["library_launches"] == 2 and got["n_xs"] == 3 and got["n_xs_f"] == 3, got
    names = got["kernels"]
    assert sum(c for k, c in names.items() if "warp_normalise_targets_kernel" in k) == 2, names
    assert sum(names.values()) == 2, names


def test_prepare_inputs_launch_count_in_process():
    """The same call in this process, through the Python op: the library reports two launches, and the mirrored
    outputs equal torch.flip of the others."""
    from hpdecode import geometry, ops
    img = torch.from_numpy(image_of(480, 640, 9)).cuda()
    n0 = ops.launches_total()
    xs, xs_f, _, _ = geometry.prepare_inputs([img] * 11, 512, "cuda:0", MS, flip=True)
    assert ops.launches_total() - n0 == 2
    assert len(xs) == 3 and len(xs_f) == 3 and xs[1].shape[:2] == (11, 3)
    for x, xf in zip(xs, xs_f):
        assert torch.equal(xf.view(torch.int32), torch.flip(x, [3]).view(torch.int32))


class CaptureNet(nn.Module):
    """Wraps a HigherHRNet and keeps every call's (input, outputs) on the host (when ``capture``)."""

    def __init__(self, net):
        super().__init__()
        self.net, self.calls, self.capture = net, [], False

    def forward(self, x):
        (lo, hi), tag = self.net(x)
        if self.capture:
            self.calls.append((x.detach().float().cpu().numpy(), lo.detach().float().cpu().numpy(),
                               hi.detach().float().cpu().numpy(), tag.detach().float().cpu().numpy()))
        return [lo, hi], tag


def _model(flip, scales, autocast=None, seed=0):
    from hpdecode import InferenceKeypointsModel, synth_net
    torch.manual_seed(seed)
    return InferenceKeypointsModel(CaptureNet(synth_net.HigherHRNet(17, 16)), use_flip=flip, input_size=128,
                                   device="cuda:0", test_scales=scales, autocast_dtype=autocast)


def _frames(n, shapes=((90, 120),), run=1):
    """n frames; the size cycles through ``shapes`` every ``run`` frames."""
    return [image_of(*shapes[(i // run) % len(shapes)], 100 + i) for i in range(n)]


def _batches(frames, batch_size):
    """The batches a FrameStream forms: runs of one size, cut every batch_size frames."""
    out, cur = [], []
    for i, f in enumerate(frames):
        if cur and (len(cur) == batch_size or f.shape != frames[cur[0]].shape):
            out.append(cur)
            cur = []
        cur.append(i)
    return out + [cur]


def _reference(model, frames, batch_size):
    """predict_batch and its records, batch by batch as the stream forms them."""
    from hpdecode import geometry
    results, raws = [], []
    mn = min(model.test_scales)
    for idx in _batches(frames, batch_size):
        imgs = [frames[i] for i in idx]
        results += model.predict_batch(imgs)
        x, _, _, minv = geometry.prepare_input(imgs, model.input_size, model.device, 1.0, mn, return_inverse=True)
        extra = [geometry.prepare_input(imgs, model.input_size, model.device, s, mn)[0] for s in model.test_scales if s != 1.0]
        raws.append(model.forward_decode(x, inv_affine=minv, extra_scales=extra).host().raw)
    return results, np.concatenate(raws)


def _same_result(a, b):
    for name in ("kpts_coords", "kpts_scores", "kpts_tags", "obj_scores"):
        x, y = np.ascontiguousarray(getattr(a, name)), np.ascontiguousarray(getattr(b, name))
        assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), name
    assert a.kpts_heatmaps is None and a.model_input_image is None and a.annot is None


CONFIGS = [  # flip, test scales, autocast, depth, batch_size, CUDA frames
    (False, (1.0,), None, 1, 1, False),
    (True, (1.0,), None, 4, 5, False),
    (True, MS, None, 4, 8, True),
    (False, MS, torch.bfloat16, 1, 5, False),
    (True, (1.0,), torch.bfloat16, 4, 8, False),
    (True, MS, torch.bfloat16, 4, 5, True),
    (False, (1.0,), None, 4, 8, True),
    (True, MS, None, 1, 8, False),
]


@pytest.mark.parametrize("flip,scales,autocast,depth,batch_size,on_device", CONFIGS)
def test_stream_equals_predict_batch(flip, scales, autocast, depth, batch_size, on_device):
    from hpdecode import FrameStream, Records
    model = _model(flip, scales, autocast)
    frames = _frames(23)
    want, want_raw = _reference(model, frames, batch_size)
    feed = [torch.from_numpy(f).cuda() for f in frames] if on_device else frames
    got = list(model.stream(iter(feed), batch_size, depth))
    assert len(got) == 23
    for g, w, f in zip(got, want, feed):
        assert g.raw_image is f
        _same_result(g, w)
    fs = FrameStream(model, batch_size, depth, records=True)
    fs.submit(feed[:11])
    fs.submit(feed[11:])
    recs = list(fs)
    assert len(recs) == 23 and all(isinstance(r, Records) and len(r) == 1 for r in recs)
    assert np.array_equal(np.concatenate([r.raw for r in recs]), want_raw)
    # nothing the stream used is left in a state that changes the model's other paths
    again, again_raw = _reference(model, frames, batch_size)
    assert np.array_equal(again_raw, want_raw)
    for a, w in zip(again, want):
        _same_result(a, w)


@pytest.mark.parametrize("run", [1, 3])
def test_stream_alternating_frame_sizes(run):
    """Two frame sizes alternating (every frame, or every 3 frames): each change closes a batch, results stay in
    submission order, geometry is computed once per size."""
    from hpdecode import FrameStream
    model = _model(True, MS)
    frames = _frames(17, shapes=((90, 120), (120, 90)), run=run)
    want, want_raw = _reference(model, frames, 4)
    fs = FrameStream(model, 4, 3)
    fs.submit(frames)
    got = list(fs)
    assert fs.geometry_calls == 2 and len(got) == 17
    for g, w in zip(got, want):
        _same_result(g, w)


def test_stream_matches_the_oracle(oracle):
    """The decoded fields of two frames against the CPU oracle on the network outputs the stream produced (flip test,
    scales 0.5 / 1.0 / 1.5): the network saw the reference's inputs, mirrored ones included."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_gpu_dropin import _oracle_result
    model = _model(True, MS, seed=4)
    frames = _frames(2, shapes=((100, 150),))
    model.net.capture = True
    got = list(model.stream(frames, batch_size=2, depth=2))
    calls = model.net.calls
    assert len(calls) == 6
    size, center, scale = input_oracle.get_multi_scale_size(100, 150, 128, 1.0, 0.5)
    for b in range(2):
        for t, s in enumerate(MS):
            want_x = input_oracle.prepare_input(frames[b], 128, s, 0.5)[0]
            assert np.array_equal(_bits(calls[2 * t][0][b]), _bits(want_x))
            assert np.array_equal(_bits(calls[2 * t + 1][0][b]), _bits(want_x[..., ::-1]))
        _, _, ref, coords = _oracle_result(oracle, calls, True, size, center, scale, b=b, tag_scale=1, n_scales=3)
        gj = ref["grouped_joints"]
        assert np.array_equal(_bits(got[b].kpts_coords), _bits(coords))
        assert np.array_equal(_bits(got[b].kpts_scores), _bits(gj[..., 2]))
        assert np.array_equal(_bits(got[b].obj_scores), _bits(ref["person_scores"]))
