"""Person ids that persist across video frames, computed on the device from the decode's result records.

An associative-embedding tag separates people within one image only, so every frame's persons are numbered from
scratch.  ``PoseTracker`` links them over time with the greedy OKS tracker of mmpose's video demos
(include/hpdecode.h: hpd_track): per frame, persons in descending score take the live track whose last pose they
match best by OKS, if that OKS is above ``oks_thr``; the others start new tracks (when at least ``min_keypoints`` joints
are visible) and get ids never used before.  A track not matched for ``max_age`` frames is dropped.

The records are read where the decode wrote them and the state stays on the device, so tracking adds one kernel launch
per call and no host round trip.

A per-frame pose jitters: joints snap to the network-input grid and the back-projection scales that grid up to the
frame.  ``PoseTracker(..., smoothing=OneEuro(fps))`` also runs the 1-Euro filter (Casiez, Roussel, Vogel, CHI 2012) on
every tracked joint in the same launch (include/hpdecode.h: hpd_track_smooth); its state lives and dies with the track.
"""
import math
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
from torch import Tensor

from . import _lib, ops
from .cocoeval import COCO_KPT_OKS_SIGMAS


@dataclass(frozen=True)
class OneEuro:
    """1-Euro filter settings: ``fps`` the video's constant frame rate, ``min_cutoff`` the cutoff (Hz) at rest,
    ``beta`` how fast the cutoff rises with the joint's speed (px/s), ``d_cutoff`` the cutoff (Hz) of that speed's
    estimate.  The defaults are the paper's starting point: 1 Hz, no speed term.  Ranges as hpd_track_smooth checks
    them: fps in [1e-3, 1e6], the cutoffs in (0, 1e6], beta in [0, 1e6], all finite."""
    fps: float
    min_cutoff: float = 1.0
    beta: float = 0.0
    d_cutoff: float = 1.0

    def __post_init__(self):
        for name, lo, lo_open in (("fps", 1e-3, False), ("min_cutoff", 0.0, True), ("beta", 0.0, False),
                                  ("d_cutoff", 0.0, True)):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float)):
                raise TypeError(f"OneEuro: {name} must be a number (got {v!r})")
            v = float(v)
            if not (math.isfinite(v) and (v > lo if lo_open else v >= lo) and v <= 1e6):
                raise ValueError(f"OneEuro: {name} must be finite and in {'(' if lo_open else '['}{lo:g}, 1e6] (got {v})")
            object.__setattr__(self, name, v)


class PoseTracker:
    """Tracker state for one video.  ``update(records)`` takes consecutive frames' result records (a CUDA uint8
    [n, row_bytes] tensor, e.g. ``DecodeResult.packed()``) and returns their person ids, int32 [n, max_num_people] on
    the device, enqueued on the current stream; -1 marks persons without a track and slots past a frame's persons.
    ``sigmas``: one OKS sigma per joint (COCO's for 17 joints when None).  ``smoothing``: a ``OneEuro`` to also filter
    the tracked joints; ``update_smoothed`` then returns their coordinates, and both methods advance the filter."""

    def __init__(self, num_kpts: int = 17, max_num_people: int = 30, emb: int = 2, device="cuda:0",
                 oks_thr: float = 0.3, max_age: int = 1, min_keypoints: int = 3,
                 sigmas: Optional[Sequence[float]] = None, smoothing: Optional[OneEuro] = None):
        if smoothing is not None and not isinstance(smoothing, OneEuro):
            raise TypeError(f"smoothing must be a hpdecode.OneEuro or None (got {type(smoothing).__name__})")
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
        self.smoothing = smoothing
        self.device = torch.device(device)
        nbytes = (ops.track_state_bytes if smoothing is None else ops.track_smooth_state_bytes)(self.params)
        self.state = torch.empty((nbytes,), device=self.device, dtype=torch.uint8)
        ops.run_track_reset(self.params, self.state, clear_ids=True)

    def update(self, records: Tensor) -> Tensor:
        if self.smoothing is not None:
            return self.update_smoothed(records)[0]
        return torch.ops.hpd.track(records, self.state, self.num_kpts, self.max_num_people, self.emb, self.max_age,
                                   self.min_keypoints, self.oks_thr, self.kpt_vars.tolist())

    def update_smoothed(self, records: Tensor) -> Tuple[Tensor, Tensor]:
        """Like ``update``, plus the COCO-section coordinates float64 [n, max_num_people, num_kpts, 2] on the device:
        tracked persons' visible joints filtered, other persons' joints raw, slots past a frame's persons 0."""
        sm = self.smoothing
        if sm is None:
            raise _lib.HpdError("update_smoothed: this PoseTracker was built without smoothing (pass smoothing=OneEuro(...))")
        return torch.ops.hpd.track_smooth(records, self.state, self.num_kpts, self.max_num_people, self.emb,
                                          self.max_age, self.min_keypoints, self.oks_thr, self.kpt_vars.tolist(),
                                          sm.fps, sm.min_cutoff, sm.beta, sm.d_cutoff)

    def reset(self):
        """Drops every track and its filters (on the current stream); ids keep counting from where they were."""
        ops.run_track_reset(self.params, self.state, clear_ids=False)
