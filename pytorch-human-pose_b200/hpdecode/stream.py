"""Frame-stream inference: uint8 frames in, one result per frame out, several batches in flight on the device.

The reference's directory and video callers (bin/inference.py:49-114, base/datasets/video.py:142-176) run
``model(frame)`` once per frame, each call ending in a synchronising device->host copy.  ``FrameStream`` batches the
frames instead and keeps ``depth`` batches in flight (``DecodePipeline`` lanes); per batch, on the lane's stream:

1. host frames are copied into the lane's pinned staging slot at ``submit`` and uploaded on a stream of their own;
   an event orders the upload before the lane's work (CUDA frames are read where they are);
2. ``hpd_prepare_inputs``: the network input of every test scale and, with the flip test, its mirrored copy, in one
   launch (``prepare_input`` + ``torch.flip`` per scale, bit for bit);
3. the network, once per scale and run, under the model's autocast setting (``InferenceKeypointsModel._net_outputs``);
4. the decode with the scale-1.0 inverse matrices, so the records carry raw-frame coordinates;
5. one device->host copy of the batch's records into the lane's pinned records slot;
6. with ``track=True``, on the stream's own tracking stream and in submission order: it waits for the batch's records,
   runs ``PoseTracker.update`` on them in place (``hpd_track``) and copies the ids into the lane's pinned ids slot.  A
   change of frame size, which closes a batch, also resets the tracker (ids are not reused).  With ``smooth``, the
   tracker also filters the tracked joints (``PoseTracker.update_smoothed``, ``hpd_track_smooth``) and their coordinates
   go to the lane's pinned coordinates slot in the same way; the size-change reset drops the filters with the tracks;
7. with ``render=PoseStyle(...)``, the batch's frames are drawn with their persons (``hpd_render_poses``): on the
   tracking stream after the tracker, with its ids and, with ``smooth``, the smoothed coordinates; without ``track``
   on the lane's stream after the decode.  Host frames are drawn from the lane's staged copy into a per-lane device
   buffer and copied into the lane's pinned rendered slot; CUDA frames are drawn into new CUDA tensors (the caller's
   frames are not modified) and stay on the device.

A lane and its staging slot are reused only after the host has waited for that lane's records copy and, when
tracking, its ids (and coordinates) copy, and when rendering, its rendered copy (events, not a device synchronise), so a lane's records are tracked before they are overwritten.  A batch closes when it is full or when the frame size changes, so frames of mixed sizes work;
results come back in submission order either way.  Geometry is computed once per distinct frame size.

The stream decodes into the model decoder's buffer sets (slot = lane): do not call the model's other entry points
while a stream still has batches in flight (``results()`` drains it).
"""
from collections import OrderedDict, deque
from typing import Iterable, Iterator, List, Optional

import numpy as np
import torch

from . import _lib, geometry, ops
from .decoder import DecodePipeline, Records
from .results import InferenceKeypointsResult
from .render import PoseRenderer, PoseStyle
from .track import OneEuro, PoseTracker


class FrameStream:
    """``submit(frames)`` any number of times, then iterate ``results()`` (or the stream itself) for one result per
    frame in submission order: an InferenceKeypointsResult (no maps, like ``predict_batch``) or, with
    ``records=True``, the frame's ``Records`` (one row).  Frames are uint8 [h,w,3] NumPy arrays or CUDA tensors.
    ``track=True``: the stream owns a ``PoseTracker`` (``tracker``, default settings) and every result carries its
    persons' ids across frames (``track_ids``).  ``smooth=OneEuro(fps)`` (needs ``track=True``): the tracker also
    One-Euro filters the tracked joints, and every result carries ``smoothed_coords``.  ``render=PoseStyle(...)``: every
    result carries ``rendered``, the frame with its persons drawn (coloured by track with ``track=True``): an owned
    uint8 NumPy array for a host frame, a new CUDA tensor for a CUDA frame."""

    MAX_SIZES = 64    # distinct frame sizes whose geometry is kept

    def __init__(self, model, batch_size: int = 8, depth: int = 4, records: bool = False, track: bool = False,
                 smooth: Optional[OneEuro] = None, render: Optional[PoseStyle] = None):
        if batch_size < 1 or depth < 1:
            raise ValueError(f"batch_size and depth must be >= 1 (got {batch_size}, {depth})")
        if smooth is not None and not track:
            raise ValueError("smooth needs track=True: the filters follow the tracks")
        if smooth is not None and not isinstance(smooth, OneEuro):
            raise TypeError(f"smooth must be a hpdecode.OneEuro or None (got {type(smooth).__name__})")
        if render is not None and not isinstance(render, PoseStyle):
            raise TypeError(f"render must be a hpdecode.PoseStyle or None (got {type(render).__name__})")
        self.model, self.batch_size, self.depth, self.records = model, int(batch_size), int(depth), records
        self.track, self.smooth, self.render = bool(track), smooth, render
        self._open: list = []           # frames of the batch being filled
        self._open_hw = None
        self._inflight = deque()        # launched batches, oldest first
        self._done = deque()            # finished per-frame results not yet handed out
        self._geom = OrderedDict()      # (h, w) -> geometry of that frame size
        self.geometry_calls = 0
        self._init_device()

    # ---- batching -----------------------------------------------------------------------------------------------
    def submit(self, frames: Iterable):
        for f in frames:
            hw = self._frame_hw(f)
            if self._open and hw != self._open_hw:
                self._close()                            # one batch is one network input shape
            if not self._open:
                while len(self._inflight) >= self.depth:  # the lane this batch takes must have been consumed
                    self._retire()
                self._open_hw = hw
            self._stage(f, len(self._open))
            self._open.append(f)
            if len(self._open) == self.batch_size:
                self._close()

    def results(self, wait: bool = True) -> Iterator:
        """Finished results in submission order.  wait=True: closes the open batch and waits for everything
        submitted so far; wait=False: hands out only batches whose records have arrived, without blocking."""
        if wait and self._open:
            self._close()
        while self._inflight and (wait or self._ready(self._inflight[0])):
            self._retire()
        while self._done:
            yield self._done.popleft()

    __iter__ = results

    def _close(self):
        self._inflight.append(self._launch(self._open, self._open_hw))
        self._open = []

    def _retire(self):
        self._done.extend(self._finish(self._inflight.popleft()))

    @staticmethod
    def _frame_hw(f):
        if isinstance(f, torch.Tensor):
            ok = f.is_cuda and f.dtype == torch.uint8 and f.dim() == 3 and f.shape[2] == 3 and f.stride(2) == 1 and f.stride(1) == 3
        else:
            ok = isinstance(f, np.ndarray) and f.dtype == np.uint8 and f.ndim == 3 and f.shape[2] == 3
        if not ok:
            raise _lib.HpdError("FrameStream: a frame is a uint8 [h,w,3] NumPy array or CUDA tensor (packed pixels)")
        return int(f.shape[0]), int(f.shape[1])

    def _geometry(self, hw, n):
        """(sizes_hw per scale, host forward matrices [T,n,6], device scale-1.0 inverse matrices [n,6])."""
        g = self._geom.get(hw)
        if g is None:
            m = self.model
            sizes_hw, fwd, (_, _, inv) = geometry.multi_scale_geometry([hw], m.input_size, m.test_scales)
            self.geometry_calls += 1
            while len(self._geom) >= self.MAX_SIZES:
                self._geom.popitem(last=False)
            g = self._geom[hw] = {"sizes_hw": sizes_hw, "fwd": fwd, "inv": inv, "per_n": {}}
        else:
            self._geom.move_to_end(hw)
        per_n = g["per_n"].get(n)
        if per_n is None:
            per_n = g["per_n"][n] = (torch.from_numpy(np.repeat(g["fwd"], n, axis=1)),
                                     torch.from_numpy(np.repeat(g["inv"], n, axis=0)).to(self.device))
        return (g["sizes_hw"],) + per_n

    # ---- device work ----------------------------------------------------------------------------------------------
    def _init_device(self):
        if not torch.cuda.is_available():
            raise _lib.HpdError("hpdecode needs a CUDA device (sm_100a); there is no CPU fallback")
        m = self.model
        self.device = torch.device(m.device)
        self.pipe = DecodePipeline(m.decoder, self.depth)
        self._upload = torch.cuda.Stream(device=self.device)
        self._tag_scale = m.test_scales.index(1.0)
        K, M, E = m.decoder.num_kpts, m.decoder.max_num_people, 2 if m.use_flip else 1
        self._rec_shape = (M, K, E)
        row_bytes = ops.record_layout(K, M, E).row_bytes
        self._host_rec = torch.empty((self.depth, self.batch_size, row_bytes), dtype=torch.uint8, pin_memory=True)
        self._pinned: List = [None] * self.depth       # per lane: host frames of the batch, pinned
        self._staged: List = [None] * self.depth       # per lane: their device copy
        self._shape_only = {}
        self.tracker = None
        if self.track:
            self.tracker = PoseTracker(K, M, E, self.device, smoothing=self.smooth)
            self._track_stream = torch.cuda.Stream(device=self.device)
            self._track_stream.wait_stream(torch.cuda.current_stream(self.device))   # the tracker's initial reset
            self._host_ids = torch.empty((self.depth, self.batch_size, M), dtype=torch.int32, pin_memory=True)
            if self.smooth is not None:
                self._host_xy = torch.empty((self.depth, self.batch_size, M, K, 2), dtype=torch.float64,
                                            pin_memory=True)
            self._track_hw = None
        self.renderer = None
        if self.render is not None:
            self.renderer = PoseRenderer(K, M, E, self.render, self.device)
            self._rend_dev: List = [None] * self.depth    # per lane: host frames drawn, on the device
            self._rend_host: List = [None] * self.depth   # per lane: their pinned copy

    def _stage(self, f, i):
        lane = self.pipe._next          # the lane the open batch will be submitted on
        if isinstance(f, torch.Tensor):
            if f.device != self.device:
                raise _lib.HpdError(f"FrameStream: frame on {f.device}, model on {self.device}")
            return
        h, w = self._open_hw
        need = self.batch_size * h * w * 3
        if self._pinned[lane] is None or self._pinned[lane].numel() < need:
            self._pinned[lane] = torch.empty((need,), dtype=torch.uint8, pin_memory=True)
            self._staged[lane] = torch.empty((need,), dtype=torch.uint8, device=self.device)
        np.copyto(self._pinned[lane].numpy()[i * h * w * 3:(i + 1) * h * w * 3].reshape(h, w, 3), f)

    def _placeholders(self, n):
        """DecodePipeline.submit reads the batch size and the flip test from its ``scales`` argument; the network
        outputs themselves come from before_agg."""
        s = self._shape_only.get(n)
        if s is None:
            e = torch.empty((n, 0, 0, 0), device=self.device)
            one = {"hm_lo": e, "hm_hi": e, "tag": e}
            if self.model.use_flip:
                one.update(hm_lo_f=e, hm_hi_f=e, tag_f=e)
            s = self._shape_only[n] = [one] * len(self.model.test_scales)
        return s

    def _launch(self, frames, hw):
        m = self.model
        lane, n, (h, w) = self.pipe._next, len(frames), hw
        sizes_hw, fwd, inv = self._geometry(hw, n)
        upload_done = None
        if any(not isinstance(f, torch.Tensor) for f in frames):
            self._upload.wait_stream(torch.cuda.current_stream(self.device))   # staging memory may be fresh
            with torch.cuda.stream(self._upload):
                nb = n * h * w * 3
                self._staged[lane][:nb].copy_(self._pinned[lane][:nb], non_blocking=True)
                upload_done = torch.cuda.Event()
                upload_done.record()
        stage = self._staged[lane]
        imgs = [f if isinstance(f, torch.Tensor) else stage[i * h * w * 3:(i + 1) * h * w * 3].view(h, w, 3)
                for i, f in enumerate(frames)]

        def before_agg(ln):
            st = torch.cuda.current_stream(self.device)
            if upload_done is not None:
                st.wait_event(upload_done)
            for f in frames:
                if isinstance(f, torch.Tensor):
                    f.record_stream(st)
            xs, xs_f = torch.ops.hpd.prepare_inputs(imgs, fwd, sizes_hw, m.use_flip, list(geometry.MEAN),
                                                    list(geometry.STD))
            return [m._net_outputs(x, xs_f[t] if m.use_flip else None) for t, x in enumerate(xs)]

        written = torch.cuda.Event()
        outs = self._render_targets(lane, frames, hw) if self.render is not None else None

        def after_tail(ln, res):
            written.record()
            self._host_rec[lane][:n].copy_(res.records, non_blocking=True)
            if outs is not None and not self.track:
                self._draw(lane, imgs, frames, outs, res.records)

        ts = self._tag_scale
        res = self.pipe.submit(self._placeholders(n), (sizes_hw[2 * ts], sizes_hw[2 * ts + 1]), tag_scale=ts,
                               before_agg=before_agg, after_tail=after_tail, inv_affine=inv)
        tracked = self._track(lane, hw, res, written, imgs, frames, outs) if self.track else None
        return lane, frames, res, tracked, outs     # res keeps the lane's buffer set alive until the batch is retired

    def _render_targets(self, lane, frames, hw):
        """Where each frame is drawn: a slot of the lane's device buffer for a host frame, a new tensor (allocated on
        the caller's stream) for a CUDA frame."""
        h, w = hw
        nb = h * w * 3
        if any(not isinstance(f, torch.Tensor) for f in frames):
            need = len(frames) * nb
            if self._rend_dev[lane] is None or self._rend_dev[lane].numel() < need:
                self._rend_dev[lane] = torch.empty((need,), dtype=torch.uint8, device=self.device)
                self._rend_host[lane] = torch.empty((need,), dtype=torch.uint8, pin_memory=True)
        return [torch.empty((h, w, 3), dtype=torch.uint8, device=self.device) if isinstance(f, torch.Tensor)
                else self._rend_dev[lane][i * nb:(i + 1) * nb].view(h, w, 3) for i, f in enumerate(frames)]

    def _draw(self, lane, imgs, frames, outs, records, ids=None, xy=None):
        """Draws the batch on the current stream; host frames' drawings go on to the lane's pinned rendered slot."""
        st = torch.cuda.current_stream(self.device)
        for f, o in zip(frames, outs):
            if isinstance(f, torch.Tensor):
                f.record_stream(st)
                o.record_stream(st)
        ops.run_render(self.renderer.params, imgs, outs, records, ids, xy)
        if any(not isinstance(f, torch.Tensor) for f in frames):
            nb = len(frames) * outs[0].numel()
            self._rend_host[lane][:nb].copy_(self._rend_dev[lane][:nb], non_blocking=True)

    def _track(self, lane, hw, res, written, imgs, frames, outs):
        """Tracks the batch's records on the tracking stream once they are written; -> the event of the ids (and
        coordinates) copy."""
        st = self._track_stream
        st.wait_event(written)
        res.records.record_stream(st)
        with torch.cuda.stream(st):
            if self._track_hw is not None and hw != self._track_hw:
                self.tracker.reset()
            self._track_hw = hw
            xy = None
            if self.smooth is None:
                ids = self.tracker.update(res.records)
            else:
                ids, xy = self.tracker.update_smoothed(res.records)
                self._host_xy[lane][:xy.shape[0]].copy_(xy, non_blocking=True)
            self._host_ids[lane][:ids.shape[0]].copy_(ids, non_blocking=True)
            if outs is not None:
                self._draw(lane, imgs, frames, outs, res.records, ids, xy)
            done = torch.cuda.Event()
            done.record()
        return done

    def _ready(self, batch) -> bool:
        return batch[2].ready.query() and (batch[3] is None or batch[3].query())

    def _finish(self, batch) -> list:
        lane, frames, res, tracked, outs = batch
        res.ready.synchronize()
        raw = self._host_rec[lane][:len(frames)].numpy().copy()
        ids = xy = None
        if tracked is not None:
            tracked.synchronize()
            ids = self._host_ids[lane][:len(frames)].numpy().copy()
            if self.smooth is not None:
                xy = self._host_xy[lane][:len(frames)].numpy().copy()
        rendered = [None] * len(frames)
        if outs is not None:
            host = self._rend_host[lane]
            for b, (f, o) in enumerate(zip(frames, outs)):
                nb = o.numel()
                rendered[b] = o if isinstance(f, torch.Tensor) else host[b * nb:(b + 1) * nb].numpy().reshape(o.shape).copy()
        M, K, E = self._rec_shape
        if self.records:
            return [Records(raw[b:b + 1], M, K, E, None if ids is None else ids[b:b + 1],
                            None if xy is None else xy[b:b + 1], None if r is None else r[None])
                    for b, r in enumerate(rendered)]
        m, rec = self.model, Records(raw, M, K, E, ids, xy)
        return [InferenceKeypointsResult.from_records(rec, b, f, None, None, m.limbs, m.det_thr, m.tag_thr,
                                                      rendered=rendered[b])
                for b, f in enumerate(frames)]
