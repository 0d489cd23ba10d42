"""Drop-in for the decode part of /root/reference/src/keypoints/results.py.

Kept: ``BaseKeypointsResult.match_heatmaps_size / resize_heatmaps_list / resize_heatmaps`` (:46-67),
``InferenceKeypointsResult.from_preds`` (:203-263) with its fields and ``get_final_kpts_coords`` (:189-201),
``transform_coords`` (:158-171) and ``KeypointsResult.set_preds`` (:94-124).  Plotting and OKS (visualisation /
evaluation consumers) are out of scope.

``from_preds`` hands the already flip-averaged heatmaps and the list of tag maps to ONE fused device call
(aggregation + NMS + top-k + grouping + adjust + refine); the back-projection to raw-image coordinates
(:158-171,189-201,244) is the epilogue of that call's last kernel (csrc/refine.cu: refine_apply_kernel), fed with
the image's inverse affine matrix, so one device->host copy of the image's result record returns everything.
"""
from dataclasses import dataclass
from typing import Any, List, Optional

import numpy as np
import torch
from torch import Tensor

from . import geometry, ops
from .decoder import Records

MEAN = np.array(geometry.MEAN)
STD = np.array(geometry.STD)


def inverse_transform(image, mean=MEAN, std=STD) -> np.ndarray:
    """ImageTransform.inverse_transform (/root/reference/src/base/transforms/base.py:33-42): the normalised CHW
    tensor back to a uint8 HWC image (float64 arithmetic like the reference; a plotting aid, host side)."""
    npy = image.detach().cpu().numpy() if isinstance(image, Tensor) else np.asarray(image)
    return ((npy.transpose(1, 2, 0) * np.asarray(std) + np.asarray(mean)) * 255).astype(np.uint8)


class BaseKeypointsResult:
    @classmethod
    def match_heatmaps_size(cls, heatmaps: List[Tensor]) -> List[Tensor]:
        h, w = heatmaps[-1].shape[-2:]
        return [torch.ops.hpd.resize_bilinear(hm, h, w) for hm in heatmaps[:-1]] + [heatmaps[-1]]

    @classmethod
    def resize_heatmaps_list(cls, heatmaps: List[Tensor], h: int, w: int) -> List[Tensor]:
        return [torch.ops.hpd.resize_bilinear(hm, h, w) for hm in heatmaps]

    @classmethod
    def resize_heatmaps(cls, heatmaps: Tensor, h: int, w: int) -> Tensor:
        return torch.ops.hpd.resize_bilinear(heatmaps, h, w)


def _cuda_device(t: Tensor) -> torch.device:
    return t.device if t.is_cuda else torch.device("cuda:0")


def _decode_preaveraged(kpts_heatmaps: List[Tensor], tags_heatmaps: List[Tensor], img_h: int, img_w: int,
                        max_num_people: int, det_thr: float, tag_thr: float, inv_affine: Optional[np.ndarray] = None):
    """results.py:225-244 in one device call.  kpts_heatmaps = the head's 1..4 stages in the network's order, e.g.
    [stage1, stage2] for HigherHRNet (flip averaging already applied by the model, model.py:87-90); tags_heatmaps =
    [tag] or [tag, unflipped flip tag]; inv_affine: float64 [B,6]."""
    if not 1 <= len(kpts_heatmaps) <= ops._lib.HPD_MAX_STAGES:
        raise ops._lib.HpdError("hpdecode handles heads with 1 to %d heatmap stages (got %d)"
                                % (ops._lib.HPD_MAX_STAGES, len(kpts_heatmaps)))
    if len(tags_heatmaps) not in (1, 2):
        raise ops._lib.HpdError("1 or 2 tag maps expected")
    dev = _cuda_device(kpts_heatmaps[0])
    dtypes = {t.dtype for t in list(kpts_heatmaps) + list(tags_heatmaps)}
    # a uniform set of fp16 or bf16 network outputs (validation under autocast, module.py:78) goes to the kernel as it is
    same16 = len(dtypes) == 1 and dtypes <= {torch.float16, torch.bfloat16}
    f = lambda t: t.to(dev) if same16 else t.to(dev, torch.float32)
    scale = {"hm": [f(h) for h in kpts_heatmaps], "hm_f": [], "tag": f(tags_heatmaps[0]),
             "tag_f": f(tags_heatmaps[1]) if len(tags_heatmaps) == 2 else None}
    B, K = scale["hm"][0].shape[:2]
    E = len(tags_heatmaps)
    bufs = ops.DecodeBuffers(B, K, img_h, img_w, E, max_num_people, dev)
    if inv_affine is not None:
        bufs.inv_affine = torch.from_numpy(np.ascontiguousarray(inv_affine, np.float64).reshape(-1, 6)).to(dev)
    params = ops.make_params(B, K, img_h, img_w, E, max_num_people, det_thr, tag_thr, True, True,
                             tags_preflipped=True)
    ops.run_decode([scale], bufs, params)
    return bufs


def transform_coords(kpts_coords: np.ndarray, center, scale, output_size) -> np.ndarray:
    """results.py:158-171 for one person [K, >=2]: columns 0,1 mapped through the inverse affine transform on the
    device (same kernel arithmetic as the decode's epilogue), the dtype of the input array kept."""
    return InferenceKeypointsResult.get_final_kpts_coords(np.asarray(kpts_coords)[None], center, scale, output_size)[0]


@dataclass
class InferenceKeypointsResult(BaseKeypointsResult):
    raw_image: np.ndarray
    annot: Optional[list]
    model_input_image: np.ndarray
    kpts_heatmaps: np.ndarray
    tags_heatmaps: np.ndarray
    kpts_coords: np.ndarray
    kpts_scores: np.ndarray
    kpts_tags: np.ndarray
    obj_scores: np.ndarray
    limbs: list
    det_thr: float
    tag_thr: float
    track_ids: Optional[np.ndarray] = None   # int32 [P]: the persons' ids across frames (model.stream(track=True))
    smoothed_coords: Optional[np.ndarray] = None   # [P,K,2]: kpts_coords One-Euro filtered (model.stream(smooth=...))
    rendered: Optional[Any] = None   # uint8 [h,w,3]: the frame with its persons drawn (model.stream(render=...)); a
    #                                  NumPy array for a host frame, a CUDA tensor for a CUDA frame

    @classmethod
    def get_final_kpts_coords(cls, kpts_coords: np.ndarray, center, scale, hm_size) -> np.ndarray:
        """results.py:189-201 as a standalone call: [P,K,>=2] network-input coordinates -> raw-image coordinates.
        Runs the decode's back-projection epilogue on the given joints (hpd_adjust_refine with adjust and refine
        off); P is processed in chunks of HPD_MAX_PEOPLE."""
        kpts_coords = np.asarray(kpts_coords)
        if len(kpts_coords) == 0:
            return np.stack([])       # the reference's np.stack([]) raises too: an image always has >= 1 person
        P, K = kpts_coords.shape[:2]
        M = ops._lib.HPD_MAX_PEOPLE
        dev = torch.device("cuda:0")
        minv = geometry.get_affine_transform(center, scale, 0, hm_size, inverse=True)
        out = kpts_coords.copy()
        wide = kpts_coords.dtype == np.float64
        for p0 in range(0, P, M):
            n = min(M, P - p0)
            bufs = ops.DecodeBuffers(1, K, 64, 64, 1, M, dev)
            bufs.inv_affine = torch.from_numpy(minv.reshape(1, 6)).to(dev)
            poses = np.zeros((1, M, K, 4), np.float32)
            poses[0, :n, :, :2] = kpts_coords[p0:p0 + n, :, :2]
            bufs.poses.copy_(torch.from_numpy(poses))
            bufs.person_scores.zero_()
            bufs.n_person.fill_(n)
            bufs.flags.fill_(1 if wide else 0)      # float64 in -> float64 out (the fallback pseudo-person's path)
            params = ops.make_params(1, K, 64, 64, 1, M, 0.0, 0.0, adjust=False, refine=False)
            ops.run_stage("adjust_refine", bufs, params)
            rec = Records(bufs.records.cpu().numpy(), M, K, 1)
            out[p0:p0 + n, :, :2] = rec.coco[0, :n, : 3 * K].reshape(n, K, 3)[..., :2]
        return out

    @classmethod
    def from_preds(cls, raw_image: np.ndarray, annot, model_input_image, kpts_heatmaps: List[Tensor],
                   tags_heatmaps: List[Tensor], limbs, scale, center, det_thr: float = 0.05, tag_thr: float = 0.5,
                   max_num_people: int = 30) -> "InferenceKeypointsResult":
        """results.py:203-263.  ``model_input_image``: the normalised tensor [3,H,W] like in the reference."""
        model_input_image_npy = inverse_transform(model_input_image)
        img_h, img_w = model_input_image_npy.shape[:2]
        minv = geometry.get_affine_transform(center, scale, 0, (img_w, img_h), inverse=True)
        bufs = _decode_preaveraged(kpts_heatmaps, tags_heatmaps, img_h, img_w, max_num_people, det_thr, tag_thr, minv)
        rec = Records(bufs.records.cpu().numpy(), max_num_people, bufs.shape[1], bufs.shape[4])
        return cls.from_records(rec, 0, raw_image, annot, model_input_image_npy, limbs, det_thr, tag_thr,
                                kpts_heatmaps=bufs.agg_hm[0].cpu().numpy(),
                                tags_heatmaps=bufs.agg_tags[0, ..., 0].cpu().numpy())

    @classmethod
    def from_records(cls, rec: Records, b: int, raw_image, annot, model_input_image, limbs, det_thr, tag_thr,
                     kpts_heatmaps=None, tags_heatmaps=None, rendered=None) -> "InferenceKeypointsResult":
        """Image b of a batch's host records -> the reference's result object (results.py:240-263).  The batched
        callers pass no maps (they stay on the device); ``from_preds`` passes them like the reference.  Records that
        carry track ids give the image's persons theirs, and smoothed coordinates, with ``kpts_coords``' dtype."""
        grouped_joints, obj_scores = rec.image(b)
        return cls(raw_image=raw_image, annot=annot, model_input_image=model_input_image, kpts_heatmaps=kpts_heatmaps,
                   tags_heatmaps=tags_heatmaps, kpts_coords=rec.final_coords(b), kpts_scores=grouped_joints[..., 2],
                   kpts_tags=grouped_joints[..., 3:], obj_scores=obj_scores, limbs=limbs, det_thr=det_thr,
                   tag_thr=tag_thr,
                   track_ids=None if rec.track_ids is None else rec.track_ids[b, :len(obj_scores)].copy(),
                   smoothed_coords=None if rec.smoothed_coords is None else rec.smoothed_final_coords(b),
                   rendered=rendered)


class KeypointsResult(BaseKeypointsResult):
    """results.py:70-124 (validation-time caller): one tag map, E = 1.  The network runs under fp16 autocast there
    (module.py:78); a uniform set of float16 or bfloat16 inputs is accepted as it is and widened inside the kernels."""

    def __init__(self, model_input_image, kpts_heatmaps: List[Tensor], tags_heatmaps: Tensor, limbs,
                 max_num_people: int = 30, det_thr: float = 0.05, tag_thr: float = 0.5):
        self.model_input_image = inverse_transform(model_input_image)
        self._kpts_heatmaps = kpts_heatmaps
        self._tags_heatmaps = tags_heatmaps
        self.num_kpts = kpts_heatmaps[0].shape[1]
        self.limbs = limbs
        self.max_num_people = max_num_people
        self.det_thr = det_thr
        self.tag_thr = tag_thr

    def set_preds(self):
        img_h, img_w = self.model_input_image.shape[:2]
        hms = [h[:1] for h in self._kpts_heatmaps]
        bufs = _decode_preaveraged(hms, [self._tags_heatmaps[:1]], img_h, img_w, self.max_num_people,
                                   self.det_thr, self.tag_thr)
        rec = Records(bufs.records.cpu().numpy(), self.max_num_people, self.num_kpts, 1)
        grouped_joints, obj_scores = rec.image(0)
        self.kpts_coords = grouped_joints[..., :2]
        self.kpts_scores = grouped_joints[..., 2]
        self.kpts_tags = grouped_joints[..., 3:]
        self.obj_scores = obj_scores
        # results.py:121-124: per-stage heatmaps resized to the image, stages last
        dev = bufs.agg_hm.device
        stages = self.match_heatmaps_size([h.to(dev, torch.float32) for h in hms])
        stacked = torch.stack(stages, dim=1)[0]                       # [stages, K, h, w]
        resized = self.resize_heatmaps(stacked, img_h, img_w)
        self.kpts_heatmaps = resized.permute(1, 2, 3, 0).cpu().numpy()
        self.tags_heatmaps = bufs.agg_tags[0].cpu().numpy()
