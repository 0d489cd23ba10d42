"""Batched bottom-up decoder: the public entry a pipeline calls once per batch.

``BottomUpDecoder.decode`` takes the raw HigherHRNet outputs of a batch (optionally of the flipped
run and of several test scales) as CUDA tensors and enqueues the whole path -- fused aggregation +
NMS, top-k, grouping, adjust, refine -- on the current stream through ``hpd_decode``.  Nothing is
copied to the host until ``DecodeResult.to_numpy()`` is called, and then only the pose lists.

The reference decodes one image per call (results.py:233-234 strips the batch dim); here the
batch is a superset: image b of a batch gives exactly what the reference returns for that image.
"""
from collections import OrderedDict
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops


class Records:
    """Host view of the per-image result records written by the decode's last kernel (HpdRecordLayout,
    include/hpdecode.h): ``raw`` is the uint8 [B,row_bytes] array of ONE device->host copy; the fields are
    zero-copy NumPy views into it.  ``track_ids``: optional int32 [B,M] person ids across frames (PoseTracker);
    ``smoothed_coords``: optional float64 [B,M,K,2] One-Euro-filtered COCO-section coordinates (PoseTracker with
    smoothing); ``rendered``: optional uint8 [B,h,w,3] frames with their persons drawn (PoseRenderer), a NumPy array
    or a CUDA tensor."""

    def __init__(self, raw: np.ndarray, M: int, K: int, E: int, track_ids: Optional[np.ndarray] = None,
                 smoothed_coords: Optional[np.ndarray] = None, rendered=None):
        L = ops.record_layout(K, M, E)
        self.track_ids, self.smoothed_coords, self.rendered = track_ids, smoothed_coords, rendered
        raw = np.ascontiguousarray(raw, np.uint8).reshape(-1, L.row_bytes)
        self.raw, self.M, self.K, self.E = raw, M, K, E
        B, D, C = raw.shape[0], 3 + E, L.coco_stride

        def view(off, dtype, shape, strides):
            return np.ndarray((B,) + shape, dtype, raw, offset=off, strides=(L.row_bytes,) + strides)

        self.coco = view(L.off_coco, np.float64, (M, C), (8 * C, 8))                       # (x, y, 1)*K, score
        self.poses = view(L.off_poses, np.float32, (M, K, D), (4 * K * D, 4 * D, 4))       # grouped joints
        self.person_scores = view(L.off_person_scores, np.float32, (M,), (4,))
        self.n_person = view(L.off_n_person, np.int32, (), ())
        self.flags = view(L.off_flags, np.int32, (), ())

    def __len__(self):
        return self.raw.shape[0]

    def image(self, b: int) -> Tuple[np.ndarray, np.ndarray]:
        """(grouped_joints [P,K,3+E], person_scores [P]) -- MPPEHeatmapParser.parse's return for image b."""
        P = int(self.n_person[b])
        return _finish(self.poses[b, :P].copy(), self.person_scores[b, :P].copy(), int(self.flags[b]) & 1)

    def final_coords(self, b: int) -> np.ndarray:
        """kpts_coords [P,K,2] back-projected to the raw image (results.py:244): float32 like the reference's
        array, float64 for the empty-scene fallback's pseudo-person."""
        P = int(self.n_person[b])
        xy = self.coco[b, :P, : 3 * self.K].reshape(P, self.K, 3)[..., :2]
        return xy.copy() if int(self.flags[b]) & 1 else xy.astype(np.float32)

    def smoothed_final_coords(self, b: int) -> np.ndarray:
        """``final_coords(b)`` with the tracked joints One-Euro filtered (``smoothed_coords``), in the same dtype."""
        P = int(self.n_person[b])
        xy = self.smoothed_coords[b, :P]
        return xy.copy() if int(self.flags[b]) & 1 else xy.astype(np.float32)

    def coco_records(self, b: int, image_id: int) -> List[dict]:
        """The COCO result dicts evaluate_dataset appends for image b (bin/eval.py:31-47)."""
        P = int(self.n_person[b])
        return [{"image_id": int(image_id), "category_id": 1, "keypoints": self.coco[b, p, : 3 * self.K].tolist(),
                 "score": float(self.coco[b, p, 3 * self.K])} for p in range(P)]


class DecodeResult:
    """Device-side result of one batch; ``to_numpy`` gives the reference's per-image return values."""

    def __init__(self, bufs: ops.DecodeBuffers):
        self.bufs = bufs
        self._generation = getattr(bufs, "generation", 0)   # a later decode into the same buffer set bumps it
        self.agg_hm = bufs.agg_hm          # [B,K,H,W]
        self.poses = bufs.poses            # [B,M,K,3+E]
        self.person_scores = bufs.person_scores
        self.n_person = bufs.n_person
        self.flags = bufs.flags
        self.records = bufs.records        # [B,row_bytes] uint8, written by the last kernel's epilogue

    def _check_live(self):
        if getattr(self.bufs, "generation", 0) != self._generation:
            raise ops._lib.HpdError("this DecodeResult was overwritten by a later decode into the same buffer set "
                                    "(same shape and slot): read or clone() a result before decoding again, or use "
                                    "distinct slots")

    @property
    def agg_tags(self) -> torch.Tensor:
        """The aggregated tags [B,K,H,W,E] (results.py:229-230).  A buffer set without a tag map (the decoder's
        default) did not write them: the first read computes the map from the network outputs of the decode (the
        buffer set keeps a reference to them), bit-identical to the one the aggregation would have written.  Those
        outputs must then be unchanged since the decode, and the result still live."""
        if self.bufs.tag_map is None:
            self._check_live()
        return self.bufs.agg_tags

    def packed(self) -> torch.Tensor:
        """The device tensor that holds everything a caller reads after a decode (one row per image):
        no ATen op runs here, the kernels wrote this layout themselves."""
        self._check_live()
        return self.records

    def host(self) -> "Records":
        self._check_live()
        B, M, K, D = self.poses.shape
        return Records(self.records.cpu().numpy(), M, K, D - 3)

    @staticmethod
    def unpack(packed: np.ndarray, M: int, K: int, E: int) -> List[Tuple[np.ndarray, np.ndarray]]:
        rec = Records(packed, M, K, E)
        return [rec.image(b) for b in range(len(rec))]

    def to_numpy(self) -> List[Tuple[np.ndarray, np.ndarray]]:
        """[(grouped_joints [P,K,3+E], person_scores [P]) per image] -- MPPEHeatmapParser.parse's return."""
        rec = self.host()
        return [rec.image(b) for b in range(len(rec))]


def _finish(poses: np.ndarray, scores: np.ndarray, fallback: int):
    if fallback:
        # grouping.py:262-269 builds this pseudo-person in float64 with score 0.01; the kernel wrote
        # the float32 image of it.  Coordinates and tags are exact in both; restore the dtype/score.
        poses = poses.astype(np.float64)
        poses[..., 2] = 0.01
        scores = poses[..., 2].mean(1)
    return poses, scores


class BottomUpDecoder:
    def __init__(self, num_kpts: int = 17, max_num_people: int = 30, det_thr: float = 0.05, tag_thr: float = 0.5,
                 device="cuda:0", adjust: bool = True, refine: bool = True, max_cached_shapes: int = 4,
                 keep_tag_map: bool = False):
        """keep_tag_map=False: the buffer sets hold no full-resolution tag map (the decode reads only a few thousand
        tags per map and interpolates them where it reads them); DecodeResult.agg_tags computes the map on demand.
        True: the aggregation writes it, as the reference computes it (4*K*H*W*E bytes per image of writes)."""
        if not torch.cuda.is_available():
            raise ops._lib.HpdError("hpdecode needs a CUDA device (sm_100a); there is no CPU fallback")
        ops._lib.lib()
        self.num_kpts, self.max_num_people = num_kpts, max_num_people
        self.det_thr, self.tag_thr = det_thr, tag_thr
        self.adjust, self.refine = adjust, refine
        self.device = torch.device(device)
        self._bufs = OrderedDict()
        self.max_cached_shapes = max_cached_shapes
        self.keep_tag_map = keep_tag_map

    def buffers(self, B, H, W, E, slot=0) -> ops.DecodeBuffers:
        """Buffer set for one (shape, slot), kept in a small LRU: bottom-up inference sees many padded
        (H, W) (resize_align_multi_scale keeps the aspect ratio) and a set is ~20 MB per image at 512 x 512 (~55 MB
        with the tag map), so at most ``max_cached_shapes`` distinct shapes stay resident (slots of one shape are evicted
        together; an evicted set is freed once the stream work that uses it has run, by the caching allocator)."""
        shape = (B, H, W, E)
        slots = self._bufs.get(shape)
        if slots is None:
            while len(self._bufs) >= self.max_cached_shapes:
                self._bufs.popitem(last=False)
            slots = self._bufs[shape] = {}
        else:
            self._bufs.move_to_end(shape)
        if slot not in slots:
            slots[slot] = ops.DecodeBuffers(B, self.num_kpts, H, W, E, self.max_num_people, self.device,
                                            tags=self.keep_tag_map)
        return slots[slot]

    def _set_inv_affine(self, bufs: ops.DecodeBuffers, inv_affine):
        if inv_affine is None:
            bufs.inv_affine = None
            return
        t = inv_affine if isinstance(inv_affine, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(inv_affine, np.float64))
        bufs.inv_affine = t.reshape(-1, 6).to(self.device, torch.float64, non_blocking=True).contiguous()

    def decode(self, scales: Sequence[dict], out_hw: Tuple[int, int], tag_scale: int = 0,
               tags_preflipped: bool = False, slot: int = 0, inv_affine=None) -> DecodeResult:
        """scales: one dict per test scale with CUDA float32 tensors hm_lo, hm_hi, tag [B,K,h,w] and,
        for the flip test, hm_lo_f, hm_hi_f, tag_f (raw outputs of the flipped forward) -- or, for a head with 1 to 4
        heatmap stages, ``{"hm": [stages], "tag", "hm_f": [stages], "tag_f"}`` (ops.stage_scale).  16-bit outputs
        (all maps float16 or all bfloat16) are read as they are.

        The returned DecodeResult VIEWS the decoder's cached buffer set for this (shape, slot): it is
        overwritten by the next decode of the same shape and slot.  Read it (``to_numpy()``), ``clone()``
        what must outlive that, or pass distinct ``slot`` values for results that are held together."""
        H, W = out_hw
        scales = [ops.stage_scale(s) for s in scales]
        B = scales[0]["hm"][0].shape[0]
        E = 2 if scales[tag_scale].get("tag_f") is not None else 1
        bufs = self.buffers(B, H, W, E, slot)
        self._set_inv_affine(bufs, inv_affine)     # float64 [B,6]: back-projection of the records' COCO section
        params = ops.make_params(B, self.num_kpts, H, W, E, self.max_num_people, self.det_thr, self.tag_thr,
                                 self.adjust, self.refine, len(scales), tag_scale, tags_preflipped=tags_preflipped)
        bufs.generation = getattr(bufs, "generation", 0) + 1
        ops.run_decode(scales, bufs, params)
        return DecodeResult(bufs)

    def decode_maps(self, agg_hm: torch.Tensor, agg_tags: torch.Tensor) -> DecodeResult:
        """Aggregated maps [B,K,H,W], [B,K,H,W,E] -> poses (the MPPEHeatmapParser.parse entry)."""
        B, K, H, W = agg_hm.shape
        E = agg_tags.shape[4]
        bufs = ops.DecodeBuffers(B, K, H, W, E, self.max_num_people, agg_hm.device, agg_hm.contiguous(),
                                 agg_tags.contiguous())
        params = ops.make_params(B, K, H, W, E, self.max_num_people, self.det_thr, self.tag_thr, self.adjust,
                                 self.refine)
        ops.run_decode(None, bufs, params)
        return DecodeResult(bufs)


class DecodePipeline:
    """Keeps ``depth`` batches in flight on one GPU.

    The path has one bandwidth-bound kernel (fused aggregation + NMS) followed by latency-bound ones (top-k,
    grouping, refine) that occupy a handful of SMs each.  Every lane owns a buffer set and a stream, so batch i+1's
    aggregation overlaps batch i's tail.  ``submit`` returns the lane's DecodeResult; it stays valid until the lane
    is reused ``depth`` submits later (call ``result.ready.synchronize()`` or ``drain()`` before reading).
    Lifetime contract for the inputs: ``submit`` records their use on the lane's stream (``Tensor.record_stream``),
    so the caller may drop them as soon as it returns.  The lanes' buffer sets hold no tag map unless the decoder keeps
    one: the lane's buffer set then keeps a reference to the inputs (those ``before_agg`` returned, if any), and ``agg_tags``
    computes the map from them -- so they must be unchanged when ``agg_tags`` is first read.

    ``records_ring``: an optional uint8 tensor [depth, B, row_bytes]; lane i's result records are then written
    straight into ``records_ring[i]`` by the decode's last kernel, so consecutive lanes form one contiguous block
    (one gather / one device->host copy for several batches).
    ``use_graphs``: the launches of a lane are captured in a CUDA graph per (input pointers, shape) and replayed --
    for small per-GPU batches, where seven launches plus their ctypes marshalling would cost more host time than
    the kernels take.  The inputs must then stay at the same addresses between submits.
    """

    STAGES = ("aggregate_nms", "topk", "group", "adjust_refine")

    def __init__(self, decoder: "BottomUpDecoder", depth: int = 3, records_ring: Optional[torch.Tensor] = None,
                 use_graphs: bool = False):
        self.dec = decoder
        self.depth = max(1, depth)
        self.records_ring = records_ring
        self.use_graphs = use_graphs
        self.graph_replays = 0
        self.lanes = [{"slot": i, "stream": torch.cuda.Stream(device=decoder.device), "ready": torch.cuda.Event(),
                       "used": False, "graphs": {}, "gate": None} for i in range(self.depth)]
        self._next = 0

    def _launch(self, ln, bufs, params, scales):
        ops.run_decode(scales, bufs, params)      # one C-ABI call: all eight launches on the lane's stream

    def submit(self, scales: Sequence[dict], out_hw: Tuple[int, int], tag_scale: int = 0, before_agg=None,
               after_tail=None, inv_affine=None) -> DecodeResult:
        """Enqueue one batch.  ``before_agg(lane)`` / ``after_tail(lane, result)`` run on the lane's stream
        (e.g. the H2D copies of the inputs and the D2H copy of the records).  A lane's ``gate`` event, if a
        callback set one (say, a gather that still reads the lane's records), is waited for before reuse."""
        ln = self.lanes[self._next]
        self._next = (self._next + 1) % self.depth
        H, W = out_hw
        first = ops.stage_scale(scales[0])["hm"][0]
        B = first.shape[0]
        E = 2 if scales[tag_scale].get("tag_f") is not None else 1
        d = self.dec
        bufs = d.buffers(B, H, W, E, slot=ln["slot"])
        if self.records_ring is not None:
            bufs.records = self.records_ring[ln["slot"]]
        params = ops.make_params(B, d.num_kpts, H, W, E, d.max_num_people, d.det_thr, d.tag_thr, d.adjust, d.refine,
                                 len(scales), tag_scale)
        params.batches_in_flight = self.depth       # >= 8: small batches take the throughput-oriented top-k launch
        cur = torch.cuda.current_stream(d.device)
        st = ln["stream"]
        if inv_affine is not None or bufs.inv_affine is not None:
            d._set_inv_affine(bufs, inv_affine)
            if bufs.inv_affine is not None:
                bufs.inv_affine.record_stream(st)
        st.wait_stream(cur)
        # The inputs were allocated on the caller's stream but are read on the lane's: tell the caching
        # allocator, or a caller that drops them right after submit() (net outputs -> submit -> next forward)
        # could get their memory back while the aggregation kernel is still reading it.
        tensors = [t for s in scales for t in ops.scale_tensors(s)]
        for t in tensors:
            if t.is_cuda:
                t.record_stream(st)
        bufs.generation = getattr(bufs, "generation", 0) + 1
        res = DecodeResult(bufs)
        with torch.cuda.stream(st):
            if ln["used"]:
                st.wait_event(ln["ready"])             # the lane's previous batch has been consumed
            if ln["gate"] is not None:
                st.wait_event(ln["gate"])
            if before_agg is not None:
                scales = before_agg(ln) or scales      # tensors made here belong to the lane's stream already
            if self.use_graphs:
                if before_agg is not None:
                    tensors = [t for s in scales for t in ops.scale_tensors(s)]
                key = (tuple(t.data_ptr() for t in tensors), B, H, W, tag_scale,
                       bufs.records.data_ptr(), 0 if bufs.inv_affine is None else bufs.inv_affine.data_ptr())
                g = ln["graphs"].get(key)
                if g is None:
                    self._launch(ln, bufs, params, scales)      # eager once: workspace, shared-memory opt-ins
                    st.synchronize()
                    g = torch.cuda.CUDAGraph()
                    ops.launches_in_last_capture()
                    with torch.cuda.graph(g, stream=st):
                        self._launch(ln, bufs, params, scales)
                    n_captured = ops.launches_in_last_capture()
                    ops.add_launches(-n_captured)              # captured, not executed
                    g = ln["graphs"][key] = (g, n_captured)
                g[0].replay()
                ops.add_launches(g[1])
                self.graph_replays += 1
            else:
                self._launch(ln, bufs, params, scales)
            bufs.note_inputs(scales, params)           # a replay does not pass through run_decode
            if after_tail is not None:
                after_tail(ln, res)
            ln["ready"].record()
        ln["used"] = True
        res.ready = ln["ready"]
        return res

    def drain(self):
        """Make the current stream wait for everything submitted so far."""
        cur = torch.cuda.current_stream(self.dec.device)
        for ln in self.lanes:
            if ln["used"]:
                cur.wait_event(ln["ready"])
            if ln["gate"] is not None:
                cur.wait_event(ln["gate"])
