"""Drop-in for /root/reference/src/keypoints/model.py:43-111: ``InferenceKeypointsModel``.

Same constructor, ``prepare_input(image) -> (x, center, scale)`` and
``__call__(raw_image, annot) -> InferenceKeypointsResult`` as the reference, so ``bin/inference.py:57`` and
``bin/eval.py:28`` run unchanged.  ``net`` is any stock-PyTorch network of the HigherHRNet family returning
``(list_of_stage_heatmaps, tag)`` with 1 to 4 heatmap stages -- ``([hm_lo, hm_hi], tag)`` for HigherHRNet, ``([hm], tag)``
for HRNet with the associative-embedding head; the convolutions are NOT part of this library.  What differs is where the work happens:

* ``prepare_input``: cv2.warpAffine + ToTensor + Normalize is one device kernel (csrc/input.cu) on the uint8
  image, bit-identical to the reference's tensor;
* the flip averaging (model.py:85-96) is not done with torch ops: the raw outputs of the normal and the flipped
  forward go straight into the fused aggregation kernel, which applies the W-flip and the COCO joint permutation
  while it loads its tiles;
* decode, back-projection and the COCO record layout are one chain of kernels; one device->host copy per batch.

Batched superset: ``predict_batch(raw_images)`` groups images by resized size, runs the network once per group
and decodes each group in one call.  ``test_scales`` enables real multi-scale inference (the reference has the size
logic, base/transforms/utils.py:60-97, but only ever calls it with scale 1): heatmaps are averaged over the scales,
tags come from scale 1.0, everything is projected to the scale-1.0 input frame.

``stream(frames)`` is the path for video and directory inference: frames are batched, uploaded through pinned
staging, prepared at every test scale (flip-test copy included) in one kernel launch, and several batches are kept in
flight (hpdecode.stream).

``autocast_dtype`` (torch.bfloat16 or torch.float16) runs every forward -- flipped run and test scales included --
under ``torch.autocast("cuda", dtype=...)`` and hands the 16-bit outputs to the decoder as they are: the kernels widen
them exactly on load, so the result is the float32 decode of the up-cast outputs, without a conversion pass.
"""
from typing import Iterable, Iterator, List, Optional, Sequence

import numpy as np
import torch
from torch import Tensor, nn

from . import geometry
from .decoder import BottomUpDecoder, DecodeResult
from .results import InferenceKeypointsResult, inverse_transform

# /root/reference/src/keypoints/datasets/coco.py:45-65 (the COCO skeleton: data, used by the plotting consumers)
COCO_LIMBS = [(9, 7), (7, 5), (5, 3), (3, 1), (1, 0), (0, 2), (1, 2), (2, 4), (4, 6), (6, 8), (8, 10), (5, 6), (5, 11),
              (6, 12), (11, 12), (11, 13), (13, 15), (12, 14), (14, 16)]


def _two_stage_dict(s: dict) -> dict:
    """A two-stage (HigherHRNet) scale in the {hm_lo, hm_hi, tag[, hm_lo_f, hm_hi_f, tag_f]} dict _net_outputs has
    always returned; other stage counts stay in the stage format."""
    if len(s["hm"]) != 2:
        return s
    out = {"hm_lo": s["hm"][0], "hm_hi": s["hm"][1], "tag": s["tag"]}
    if s["hm_f"]:
        out.update(hm_lo_f=s["hm_f"][0], hm_hi_f=s["hm_f"][1], tag_f=s["tag_f"])
    return out


class InferenceKeypointsModel:
    limbs = COCO_LIMBS
    model_input_shape: tuple

    def __init__(self, net: nn.Module, det_thr: float = 0.05, tag_thr: float = 0.5, use_flip: bool = False,
                 input_size: int = 512, max_num_people: int = 30, device: str = "cuda:0",
                 ckpt_path: Optional[str] = None, num_kpts: int = 17, test_scales: Sequence[float] = (1.0,),
                 autocast_dtype: Optional[torch.dtype] = None):
        if autocast_dtype not in (None, torch.bfloat16, torch.float16):
            raise ValueError(f"autocast_dtype must be None, torch.bfloat16 or torch.float16 (got {autocast_dtype})")
        self.autocast_dtype = autocast_dtype
        self.device = device
        self.input_size = input_size
        self.net = net.to(device)
        self.net.eval()
        if ckpt_path is not None:
            self.load_checkpoint(ckpt_path)
        self.det_thr, self.tag_thr = det_thr, tag_thr
        self.max_num_people = max_num_people
        self.use_flip = use_flip
        self.test_scales = tuple(float(s) for s in test_scales)
        if 1.0 not in self.test_scales:
            raise ValueError("test_scales must contain 1.0 (the scale the tags and the output frame come from)")
        self.decoder = BottomUpDecoder(num_kpts, max_num_people, det_thr, tag_thr, device)

    def load_checkpoint(self, ckpt_path: str):
        """base/model.py:166-172: accepts a raw state dict or the trainer's {"module": {"model": ...}} layout and
        strips the DDP / torch.compile prefixes."""
        ckpt = torch.load(ckpt_path, map_location=self.device)
        if "module" in ckpt.keys():
            ckpt = ckpt["module"]["model"]
        state = {}
        for key, value in ckpt.items():
            for prefix in ("module.", "_orig_mod.", "net."):
                key = key.replace(prefix, "")
            state[key] = value
        self.net.load_state_dict(state)

    # -- reference API ---------------------------------------------------------------------------------------------
    def prepare_input(self, image: np.ndarray):
        """model.py:70-76: (x [1,3,h,w] on the device, center, scale)."""
        x, centers, scales = geometry.prepare_input([image], self.input_size, self.device)
        return x, centers[0], scales[0]

    def __call__(self, raw_image: np.ndarray, annot: Optional[list] = None) -> InferenceKeypointsResult:
        """model.py:78-111 for one image; the maps and ``model_input_image`` are returned like in the reference."""
        return self.predict_batch([raw_image], [annot], keep_maps=True)[0]

    # -- batched superset -------------------------------------------------------------------------------------------
    @torch.no_grad()
    def _net_outputs(self, x: Tensor, x_flipped: Optional[Tensor] = None) -> dict:
        """x_flipped: torch.flip(x, [3]) when the caller already has it (prepare_inputs writes it with x)."""
        if self.autocast_dtype is not None:
            return _two_stage_dict(self._net_outputs_autocast(x, x_flipped))
        return _two_stage_dict(self._scale(x, x_flipped, lambda t: t.float()))

    def _scale(self, x: Tensor, x_flipped: Optional[Tensor], cast) -> dict:
        """The decoder's scale dict ({"hm": [stages], "tag", "hm_f", "tag_f"}, ops.stage_scale) from the net's
        ``(stage_heatmaps, tag)`` on x and, with the flip test (model.py:85-94, fused into the aggregation kernel),
        on the flipped input."""
        hms, tag = self.net(x)
        if not 1 <= len(hms) <= 4:
            raise ValueError(f"the net must return 1 to 4 heatmap stages (got {len(hms)})")
        scale = {"hm": [cast(h) for h in hms], "tag": cast(tag), "hm_f": [], "tag_f": None}
        if self.use_flip:
            fl_hms, fl_tag = self.net(torch.flip(x, [3]) if x_flipped is None else x_flipped)
            scale.update(hm_f=[cast(h) for h in fl_hms], tag_f=cast(fl_tag))
        return scale

    def _net_outputs_autocast(self, x: Tensor, x_flipped: Optional[Tensor] = None) -> dict:
        with torch.autocast("cuda", dtype=self.autocast_dtype):
            scale = self._scale(x, x_flipped, lambda t: t)
        # the decoder reads one dtype per call: a net whose head leaves some outputs in float32 under autocast has all
        # of them up-cast (exact), the usual all-16-bit set goes as it is
        tensors = scale["hm"] + scale["hm_f"] + [t for t in (scale["tag"], scale["tag_f"]) if t is not None]
        if len({t.dtype for t in tensors}) > 1:
            f = lambda t: None if t is None else t.float()
            scale = {"hm": [h.float() for h in scale["hm"]], "hm_f": [h.float() for h in scale["hm_f"]],
                     "tag": f(scale["tag"]), "tag_f": f(scale["tag_f"])}
        return scale

    @torch.no_grad()
    def forward_decode(self, x: Tensor, inv_affine=None, extra_scales: Sequence[Tensor] = ()) -> DecodeResult:
        """x: normalised input batch [B,3,H,W] on the device (the scale-1.0 input); extra_scales: the same images
        prepared at the other test scales, in ``test_scales`` order without the 1.0 entry."""
        h, w = x.shape[-2:]
        self.model_input_shape = (h, w)
        others = iter(extra_scales)
        ins = [self._net_outputs(x if s == 1.0 else next(others)) for s in self.test_scales]
        return self.decoder.decode(ins, (h, w), tag_scale=self.test_scales.index(1.0), inv_affine=inv_affine)

    def predict_batch(self, raw_images: Sequence[np.ndarray], annots: Optional[Sequence] = None,
                      keep_maps: bool = False) -> List[InferenceKeypointsResult]:
        """One result per image, in order.  Images sharing a resized size go through the network and the decoder
        together.  keep_maps=False leaves the aggregated maps and the un-normalised input on the device (the
        evaluation loop does not read them); keep_maps=True fills them like the reference."""
        annots = list(annots) if annots is not None else [None] * len(raw_images)
        results: List[Optional[InferenceKeypointsResult]] = [None] * len(raw_images)
        min_scale = min(self.test_scales)
        groups = geometry.group_by_resized_size([im.shape[:2] for im in raw_images], self.input_size, 1.0, min_scale)
        for size, idxs in groups.items():
            imgs = [raw_images[i] for i in idxs]
            x, centers, scales, minv = geometry.prepare_input(imgs, self.input_size, self.device, 1.0, min_scale,
                                                              return_inverse=True)
            extra = [geometry.prepare_input(imgs, self.input_size, self.device, s, min_scale)[0]
                     for s in self.test_scales if s != 1.0]
            res = self.forward_decode(x, inv_affine=minv, extra_scales=extra)
            rec = res.host()
            for j, i in enumerate(idxs):
                maps = {}
                if keep_maps:
                    maps = dict(kpts_heatmaps=res.agg_hm[j].cpu().numpy(), tags_heatmaps=res.agg_tags[j, ..., 0].cpu().numpy())
                results[i] = InferenceKeypointsResult.from_records(
                    rec, j, raw_images[i], annots[i], inverse_transform(x[j]) if keep_maps else None, self.limbs,
                    self.det_thr, self.tag_thr, **maps)
        return results

    def stream(self, frames: Iterable, batch_size: int = 8, depth: int = 4, records: bool = False,
               track: bool = False, smooth=None, render=None) -> Iterator:
        """Frame-stream inference (video, a directory of images): uint8 [h,w,3] frames (host arrays or CUDA tensors)
        in, one result per frame out, in input order -- an InferenceKeypointsResult (no maps), or the frame's
        Records with ``records=True``.  Up to ``batch_size`` frames of one size share a batch, ``depth`` batches are
        in flight (hpdecode.stream.FrameStream); results are yielded as their batches complete.  ``track=True``: the
        results' ``track_ids`` number the persons consistently across frames (hpdecode.track.PoseTracker);
        ``smooth=hpdecode.OneEuro(fps)`` (with ``track=True``) also gives them ``smoothed_coords``, the tracked joints
        One-Euro filtered.  ``render=hpdecode.PoseStyle(...)`` gives every result ``rendered``, the frame with its persons
        drawn on the device (coloured by track with ``track=True``, at the smoothed coordinates with ``smooth``)."""
        from .stream import FrameStream
        fs = FrameStream(self, batch_size, depth, records, track, smooth, render)
        for frame in frames:
            fs.submit([frame])
            yield from fs.results(wait=False)
        yield from fs.results()
