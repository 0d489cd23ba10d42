"""Person ids that persist across video frames, computed on the device from the decode's result records.

An associative-embedding tag separates people within one image only, so every frame's persons are numbered from
scratch.  ``PoseTracker`` links them over time with the greedy OKS tracker of mmpose's video demos
(include/hpdecode.h: hpd_track): per frame, persons in descending score take the live track whose last pose they
match best by OKS, if that OKS is above ``oks_thr``; the others start new tracks (when at least ``min_keypoints`` joints
are visible) and get ids never used before.  A track not matched for ``max_age`` frames is dropped.

The records are read where the decode wrote them and the state stays on the device, so tracking adds one kernel launch
per call and no host round trip.
"""
from typing import Optional, Sequence

import numpy as np
import torch
from torch import Tensor

from . import _lib, ops
from .cocoeval import COCO_KPT_OKS_SIGMAS


class PoseTracker:
    """Tracker state for one video.  ``update(records)`` takes consecutive frames' result records (a CUDA uint8
    [n, row_bytes] tensor, e.g. ``DecodeResult.packed()``) and returns their person ids, int32 [n, max_num_people] on
    the device, enqueued on the current stream; -1 marks persons without a track and slots past a frame's persons.
    ``sigmas``: one OKS sigma per joint (COCO's for 17 joints when None)."""

    def __init__(self, num_kpts: int = 17, max_num_people: int = 30, emb: int = 2, device="cuda:0",
                 oks_thr: float = 0.3, max_age: int = 1, min_keypoints: int = 3,
                 sigmas: Optional[Sequence[float]] = None):
        if not torch.cuda.is_available():
            raise _lib.HpdError("hpdecode needs a CUDA device (sm_100a); there is no CPU fallback")
        if sigmas is None:
            if num_kpts != len(COCO_KPT_OKS_SIGMAS):
                raise ValueError(f"sigmas are required for num_kpts={num_kpts} (COCO's are for 17 joints)")
            sigmas = COCO_KPT_OKS_SIGMAS
        self.kpt_vars = (np.asarray(sigmas, np.float64) * 2) ** 2      # cocoeval's computeOks: vars = (sigmas * 2)**2
        self.num_kpts, self.max_num_people, self.emb = num_kpts, max_num_people, emb
        self.oks_thr, self.max_age, self.min_keypoints = float(oks_thr), int(max_age), int(min_keypoints)
        self.params = ops.track_params(num_kpts, max_num_people, emb, self.max_age, self.min_keypoints, self.oks_thr,
                                       self.kpt_vars.tolist())
        self.device = torch.device(device)
        self.state = torch.empty((ops.track_state_bytes(self.params),), device=self.device, dtype=torch.uint8)
        ops.run_track_reset(self.params, self.state, clear_ids=True)

    def update(self, records: Tensor) -> Tensor:
        return torch.ops.hpd.track(records, self.state, self.num_kpts, self.max_num_people, self.emb, self.max_age,
                                   self.min_keypoints, self.oks_thr, self.kpt_vars.tolist())

    def reset(self):
        """Drops every track (on the current stream); ids keep counting from where they were."""
        ops.run_track_reset(self.params, self.state, clear_ids=False)
