"""Image <-> network-input geometry of the inference path, computed by libhpdecode.so (csrc/input.cu).

Python twins of /root/reference/src/base/transforms/utils.py:25-97 as far as the decode path uses them:
``get_multi_scale_size`` / ``get_affine_transform`` are float64 host code inside the library (the matrix comes
out bit-identical to cv2.getAffineTransform); ``resize_align_multi_scale`` + ToTensor + Normalize
(model.py:45-50,70-76) are ONE device kernel, ``prepare_input``, that replays cv2.warpAffine's fixed-point bilinear
arithmetic, so the tensor handed to the network is bit-identical to the reference's.  ``prepare_inputs`` runs the
same kernel body for every test scale and the flip-test copy in one launch.
"""
import ctypes
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops

COCO_FLIP_INDEX = list(ops.COCO_FLIP_INDEX)   # /root/reference/src/keypoints/transforms.py:11
MEAN = (0.485, 0.456, 0.406)                  # model.py:48
STD = (0.229, 0.224, 0.225)


def get_multi_scale_size(image, input_size: int, current_scale: float, min_scale: float):
    """utils.py:60-87.  ``image``: array [h,w,3] or an (h, w) pair.  -> ((w_resized, h_resized), center, scale)."""
    h, w = image.shape[:2] if hasattr(image, "shape") else image
    size, center, scale = (ctypes.c_int32 * 2)(), (ctypes.c_int32 * 2)(), (ctypes.c_double * 2)()
    _lib.check(_lib.lib().hpd_multi_scale_size(int(h), int(w), int(input_size), float(current_scale), float(min_scale),
                                               size, center, scale), "hpd_multi_scale_size")
    return (size[0], size[1]), (center[0], center[1]), (scale[0], scale[1])


def get_affine_transform(center, scale, rot: float, output_size, shift=(0, 0), inverse: bool = False) -> np.ndarray:
    """utils.py:25-57 for the call shapes of this path (rot = 0, shift = 0): float64 [2,3]."""
    if rot != 0 or tuple(shift) != (0, 0):
        raise _lib.HpdError("get_affine_transform: the decode path only uses rot = 0, shift = (0, 0)")
    c = (ctypes.c_double * 2)(float(center[0]), float(center[1]))
    s = (ctypes.c_double * 2)(float(scale[0]), float(scale[1]))
    o = (ctypes.c_int32 * 2)(int(output_size[0]), int(output_size[1]))
    m = (ctypes.c_double * 6)()
    _lib.check(_lib.lib().hpd_get_affine_transform(c, s, o, int(bool(inverse)), m), "hpd_get_affine_transform")
    return np.array(m[:], np.float64).reshape(2, 3)


def prepare_geometry(shapes_hw: Sequence[Tuple[int, int]], input_size: int, current_scale: float = 1, min_scale: float = 1):
    """get_multi_scale_size + both affine matrices for n images in ONE library call:
    (sizes int32 [n,2] (w,h), centers int32 [n,2], scales float64 [n,2], forward float64 [n,6], inverse float64 [n,6])."""
    n = len(shapes_hw)
    hs = np.ascontiguousarray([s[0] for s in shapes_hw], np.int32)
    ws = np.ascontiguousarray([s[1] for s in shapes_hw], np.int32)
    sizes, centers = np.empty((n, 2), np.int32), np.empty((n, 2), np.int32)
    scales, fwd, inv = np.empty((n, 2), np.float64), np.empty((n, 6), np.float64), np.empty((n, 6), np.float64)
    i32 = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    f64 = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    _lib.check(_lib.lib().hpd_prepare_geometry(n, i32(hs), i32(ws), int(input_size), float(current_scale), float(min_scale),
                                               i32(sizes), i32(centers), f64(scales), f64(fwd), f64(inv)), "hpd_prepare_geometry")
    return sizes, centers, scales, fwd, inv


def prepare_input(images: Sequence, input_size: int, device, current_scale: float = 1, min_scale: float = 1,
                  mean=MEAN, std=STD, return_inverse: bool = False):
    """Batched ``InferenceKeypointsModel.prepare_input`` (model.py:70-76) on the device.

    images: uint8 [h,w,3] arrays (host) or CUDA tensors, all mapping to the SAME resized size (group them with
    ``group_by_resized_size`` first).  Returns (x [B,3,H,W] float32 on ``device``, centers, scales) and, with
    ``return_inverse``, also the float64 [B,6] inverse matrices the decoder back-projects with."""
    device = torch.device(device)
    sizes, centers, scales, fwd, inv = prepare_geometry([im.shape[:2] for im in images], input_size, current_scale, min_scale)
    if (sizes != sizes[0]).any():
        raise _lib.HpdError("prepare_input: images of one call must share the resized size; got %s"
                            % sorted({(int(w), int(h)) for w, h in sizes}))
    x = torch.ops.hpd.prepare_input(device_images(images, device), torch.from_numpy(fwd), int(sizes[0, 1]), int(sizes[0, 0]), list(mean), list(std))
    out = (x, [(int(c[0]), int(c[1])) for c in centers], [(float(s[0]), float(s[1])) for s in scales])
    return out + (inv,) if return_inverse else out


def multi_scale_geometry(shapes_hw: Sequence[Tuple[int, int]], input_size: int, test_scales: Sequence[float],
                         min_scale: Optional[float] = None):
    """``prepare_geometry`` at every test scale, one library call per scale, for images that share their resized size
    at each scale.  -> (sizes_hw flat [h0, w0, h1, w1, ...] per scale, forward float64 [T,n,6], and the scale-1.0
    (centers int32 [n,2], scales float64 [n,2], inverse float64 [n,6]): the frame the decode projects back from)."""
    test_scales = [float(s) for s in test_scales]
    if 1.0 not in test_scales:
        raise ValueError("test_scales must contain 1.0 (the scale the tags and the output frame come from)")
    min_scale = min(test_scales) if min_scale is None else min_scale
    sizes_hw, fwd, base = [], [], None
    for s in test_scales:
        sizes, centers, scales, f, inv = prepare_geometry(shapes_hw, input_size, s, min_scale)
        if (sizes != sizes[0]).any():
            raise _lib.HpdError("prepare_inputs: images of one call must share the resized size; got %s at scale %g"
                                % (sorted({(int(w), int(h)) for w, h in sizes}), s))
        sizes_hw += [int(sizes[0, 1]), int(sizes[0, 0])]
        fwd.append(f)
        if s == 1.0:
            base = (centers, scales, inv)
    return sizes_hw, np.stack(fwd), base


def device_images(images: Sequence, device) -> list:
    """uint8 [h,w,3] host arrays or CUDA tensors -> CUDA tensors with packed pixels on ``device``."""
    out = []
    for im in images:
        t = im if isinstance(im, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(im))
        if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3:
            raise _lib.HpdError("prepare_input: images must be uint8 [h,w,3]")
        out.append(t.to(device, non_blocking=True).contiguous())
    return out


def prepare_inputs(images: Sequence, input_size: int, device, test_scales: Sequence[float] = (1.0,), flip: bool = False,
                   min_scale: Optional[float] = None, return_inverse: bool = False, mean=MEAN, std=STD):
    """``prepare_input`` at every test scale, and with ``flip`` the horizontally flipped copy of each, in ONE kernel
    launch (hpd_prepare_inputs; per 32 (scale, image) pairs).  The images are read once per scale and the flipped
    copy is a second store of the same values: xs_flipped[t] == torch.flip(xs[t], [3]) bit for bit.

    images: as for ``prepare_input`` (one resized size per scale).  min_scale defaults to min(test_scales), the
    multi-scale size rule of utils.py:60-87.  Returns (xs, xs_flipped, centers, scales): one [B,3,h,w] tensor per test
    scale in ``test_scales`` order, the flipped ones (empty list without ``flip``), and the scale-1.0 centers and scales;
    with ``return_inverse`` also the scale-1.0 inverse matrices float64 [B,6] the decoder back-projects with."""
    device = torch.device(device)
    sizes_hw, fwd, (centers, scales, inv) = multi_scale_geometry([im.shape[:2] for im in images], input_size,
                                                                 test_scales, min_scale)
    xs, xs_f = torch.ops.hpd.prepare_inputs(device_images(images, device), torch.from_numpy(fwd), sizes_hw, bool(flip),
                                            list(mean), list(std))
    out = (xs, xs_f, [(int(c[0]), int(c[1])) for c in centers], [(float(s[0]), float(s[1])) for s in scales])
    return out + (inv,) if return_inverse else out


def group_by_resized_size(shapes_hw: Sequence[Tuple[int, int]], input_size: int, current_scale: float = 1,
                          min_scale: float = 1) -> dict:
    """{(w_resized, h_resized): [indices]} -- images that can share one batched network call."""
    groups: dict = {}
    sizes = prepare_geometry(list(shapes_hw), input_size, current_scale, min_scale)[0]
    for i, (w, h) in enumerate(sizes):
        groups.setdefault((int(w), int(h)), []).append(i)
    return groups
