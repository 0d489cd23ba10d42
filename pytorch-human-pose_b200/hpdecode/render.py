"""Decoded poses drawn onto frames on the device: every person's skeleton and joints painted into a copy of the frame
straight from the decode's result records (include/hpdecode.h: hpd_render_poses).

The rule is exact and stated in the header: a pixel is covered by a limb of width ``thickness`` or a joint disc of
radius ``joint_radius`` by a float64 test at the pixel's centre, and takes the colour of the last primitive that covers
it (per person: limbs in list order, then joints).  No anti-aliasing, no blending.  With track ids, each person's limbs
take the colour of its track, so a person keeps its colour across a video.
"""
import math
import numbers
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib, ops
from .model import COCO_LIMBS

Color = Tuple[int, int, int]

# 20 distinct colours (the "tab20" palette), in RGB; a frame in BGR order shows the same set in another assignment
DEFAULT_TRACK_COLORS = (
    (31, 119, 180), (255, 127, 14), (44, 160, 44), (214, 39, 40), (148, 103, 189), (140, 86, 75), (227, 119, 194),
    (127, 127, 127), (188, 189, 34), (23, 190, 207), (174, 199, 232), (255, 187, 120), (152, 223, 138),
    (255, 152, 150), (197, 176, 213), (196, 156, 148), (247, 182, 210), (199, 199, 199), (219, 219, 141),
    (158, 218, 229))


def _color(v, what: str) -> Color:
    try:
        c = tuple(v)
    except TypeError:
        raise TypeError(f"PoseStyle: {what} must be three integers in [0, 255] (got {v!r})") from None
    if len(c) != 3 or any(isinstance(x, bool) or not isinstance(x, numbers.Integral) for x in c):
        raise TypeError(f"PoseStyle: {what} must be three integers in [0, 255] (got {v!r})")
    if any(not 0 <= x <= 255 for x in c):
        raise ValueError(f"PoseStyle: {what} must be three integers in [0, 255] (got {v!r})")
    return tuple(int(x) for x in c)


@dataclass(frozen=True)
class PoseStyle:
    """How ``PoseRenderer`` and ``model.stream(render=...)`` draw poses.  ``limbs``: pairs of joint indices (distinct,
    up to 64); None is COCO's skeleton (``COCO_LIMBS``), which needs 17 joints.  ``limb_colors``: one colour per limb
    (None: ``track_colors`` in turn), used when there are no track ids; with ids, a tracked person's limbs take
    ``track_colors[id % len(track_colors)]`` (1 to 32 colours) and an untracked one's ``untracked_color``.  Joints take
    ``joint_color``.  Colours are three bytes in the frame's own channel order.  ``thickness`` (limb width) and
    ``joint_radius`` are pixels, finite and in [0, 1024]; 0 draws no limbs or no joints.  A joint is drawn when its
    score is above ``kpt_thr`` (finite)."""
    limbs: Optional[Sequence[Tuple[int, int]]] = None
    limb_colors: Optional[Sequence[Color]] = None
    joint_color: Color = (255, 255, 255)
    track_colors: Sequence[Color] = DEFAULT_TRACK_COLORS
    untracked_color: Color = (128, 128, 128)
    thickness: float = 3.0
    joint_radius: float = 4.0
    kpt_thr: float = 0.0

    def __post_init__(self):
        if self.limbs is not None:
            limbs = tuple(tuple(l) for l in self.limbs)
            if len(limbs) > _lib.HPD_RENDER_MAX_LIMBS:
                raise ValueError(f"PoseStyle: at most {_lib.HPD_RENDER_MAX_LIMBS} limbs (got {len(limbs)})")
            for l in limbs:
                if len(l) != 2 or any(isinstance(j, bool) or not isinstance(j, numbers.Integral) for j in l):
                    raise TypeError(f"PoseStyle: a limb is a pair of joint indices (got {l!r})")
                if l[0] < 0 or l[1] < 0 or l[0] == l[1]:
                    raise ValueError(f"PoseStyle: a limb joins two distinct joints >= 0 (got {l!r})")
            object.__setattr__(self, "limbs", tuple((int(a), int(b)) for a, b in limbs))
        n_limbs = len(COCO_LIMBS if self.limbs is None else self.limbs)
        if self.limb_colors is not None:
            colors = tuple(_color(c, "a limb colour") for c in self.limb_colors)
            if len(colors) != n_limbs:
                raise ValueError(f"PoseStyle: one limb colour per limb ({n_limbs}; got {len(colors)})")
            object.__setattr__(self, "limb_colors", colors)
        track = tuple(_color(c, "a track colour") for c in self.track_colors)
        if not 1 <= len(track) <= _lib.HPD_RENDER_MAX_COLORS:
            raise ValueError(f"PoseStyle: 1 to {_lib.HPD_RENDER_MAX_COLORS} track colours (got {len(track)})")
        object.__setattr__(self, "track_colors", track)
        object.__setattr__(self, "joint_color", _color(self.joint_color, "joint_color"))
        object.__setattr__(self, "untracked_color", _color(self.untracked_color, "untracked_color"))
        for name, hi in (("thickness", 1024.0), ("joint_radius", 1024.0), ("kpt_thr", None)):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, float)):
                raise TypeError(f"PoseStyle: {name} must be a number (got {v!r})")
            v = float(v)
            if not math.isfinite(v) or (hi is not None and not 0.0 <= v <= hi):
                raise ValueError(f"PoseStyle: {name} must be finite" + (f" and in [0, {hi:g}]" if hi else "")
                                 + f" (got {v})")
            object.__setattr__(self, name, v)

    def resolved_limbs(self, num_kpts: int) -> Tuple[Tuple[int, int], ...]:
        """The skeleton for ``num_kpts`` joints: ``limbs``, or COCO's for 17 joints."""
        if self.limbs is None:
            if num_kpts != 17:
                raise ValueError(f"PoseStyle: limbs are required for num_kpts={num_kpts} (COCO's are for 17 joints)")
            return tuple(COCO_LIMBS)
        for l in self.limbs:
            if max(l) >= num_kpts:
                raise ValueError(f"PoseStyle: limb {l} has a joint >= num_kpts={num_kpts}")
        return self.limbs

    def resolved_limb_colors(self, n_limbs: int) -> Tuple[Color, ...]:
        if self.limb_colors is not None:
            return self.limb_colors
        return tuple(self.track_colors[l % len(self.track_colors)] for l in range(n_limbs))


class PoseRenderer:
    """Draws result records onto frames for one record shape.  ``render(frames, records, track_ids=None,
    coords=None)``: ``frames`` uint8 [h,w,3] CUDA tensors (packed pixels, any row stride; left unchanged), ``records``
    their result records (CUDA uint8 [n, row_bytes], e.g. ``DecodeResult.packed()``), optional ``track_ids`` int32
    [n, max_num_people] (``PoseTracker.update``) and ``coords`` float64 [n, max_num_people, num_kpts, 2]
    (``PoseTracker.update_smoothed``) in place of the records' coordinates -> one new uint8 [h,w,3] CUDA tensor per
    frame, enqueued on the current stream.  Everything is on ``device``."""

    def __init__(self, num_kpts: int = 17, max_num_people: int = 30, emb: int = 2, style: Optional[PoseStyle] = None,
                 device="cuda:0"):
        if style is None:
            style = PoseStyle()
        if not isinstance(style, PoseStyle):
            raise TypeError(f"style must be a hpdecode.PoseStyle or None (got {type(style).__name__})")
        limbs = style.resolved_limbs(num_kpts)
        if not torch.cuda.is_available():
            raise _lib.HpdError("hpdecode needs a CUDA device (sm_100a); there is no CPU fallback")
        self.num_kpts, self.max_num_people, self.emb, self.style = num_kpts, max_num_people, emb, style
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        flat = lambda seq: [int(v) for item in seq for v in item]     # noqa: E731
        self._args = (num_kpts, max_num_people, emb, flat(limbs), flat(style.resolved_limb_colors(len(limbs))),
                      list(style.joint_color), flat(style.track_colors), list(style.untracked_color), style.thickness,
                      style.joint_radius, style.kpt_thr)
        self.params = ops.render_params(*self._args)

    def render(self, frames: Sequence[Tensor], records: Tensor, track_ids: Optional[Tensor] = None,
               coords: Optional[Tensor] = None):
        if records.device != self.device:
            raise _lib.HpdError(f"PoseRenderer: records on {records.device}, renderer on {self.device}")
        return torch.ops.hpd.render_poses(list(frames), records, track_ids, coords, *self._args)
