"""PyTorch custom ops over the C ABI: device pointers in, device tensors out, no host round trip.

``torch.ops.hpd.*`` are registered with ``torch.library.custom_op``; each one fills ctypes structs
with ``tensor.data_ptr()`` / strides and the current CUDA stream and calls libhpdecode.so.  PyTorch is
plumbing here (memory, streams); all arithmetic happens in the library's sm_100a kernels.

Stage ops mirror the reference methods one to one (paths relative to /root/reference):
  hpd::aggregate_nms  model.py:85-96 + results.py:225-230 (+ grouping.py:80-83 fused)
  hpd::nms            MPPEHeatmapParser.nms          grouping.py:80-83
  hpd::topk           MPPEHeatmapParser.top_k        grouping.py:147-170
  hpd::group          MPPEHeatmapParser.match_by_tag grouping.py:85-145 (+ fallback :262-269)
  hpd::adjust_refine  adjust / person score / refine grouping.py:172-191,276,193-250
  hpd::decode         all of the above in one call   (from_preds, results.py:225-238)
  hpd::decode_stages  the same for heads with 1..4 heatmap stages per scale (results.py:46-54,226 take stage lists)
  hpd::prepare_input  resize_align_multi_scale + ToTensor + Normalize  utils.py:89-97, model.py:45-50
  hpd::prepare_inputs the same for every test scale, plus the flip-test input (model.py:86), in one call
  hpd::coco_eval      pycocotools COCOeval(..., "keypoints").evaluate() + accumulate() (bin/eval.py:52-65)
  hpd::track          person ids across consecutive frames' result records (greedy OKS tracking; hpdecode.track)
  hpd::track_smooth   the same ids plus the tracked joints' One-Euro-filtered coordinates (hpdecode.track.OneEuro)
  hpd::render_poses   skeletons and joints drawn into copies of frames from their result records (hpdecode.render)
"""
import ctypes
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import (HpdBuffers, HpdCocoDets, HpdCocoEvalOutputs, HpdCocoEvalParams, HpdCocoGts, HpdImage, HpdMap,
                   HpdParams, HpdRecordLayout, HpdRenderFrame, HpdRenderParams, HpdScaleInputs, HpdSmoothParams,
                   HpdStageInputs, HpdTrackParams)

COCO_FLIP_INDEX = [0, 2, 1, 4, 3, 6, 5, 8, 7, 10, 9, 12, 11, 14, 13, 16, 15]  # transforms.py:11
JOINTS_ORDER_17 = [0, 1, 2, 3, 4, 5, 6, 11, 12, 7, 8, 9, 10, 13, 14, 15, 16]   # grouping.py:63-65

_launches = 0


def launches_total() -> int:
    """Kernel launches enqueued through this module since import (bench accounting)."""
    return _launches


def _require_cuda(t: Tensor, name: str):
    if not t.is_cuda:
        raise _lib.HpdError(f"{name} must be a CUDA tensor: hpdecode has no CPU path")
    if t.dtype != torch.float32:
        raise _lib.HpdError(f"{name} must be float32 (got {t.dtype})")


# network outputs under fp16 / bf16 autocast (module.py:78): read as they are, widened exactly inside the kernels
_DTYPE_CODES = {torch.float16: _lib.HPD_F16, torch.bfloat16: _lib.HPD_BF16}


def _map(t: Optional[Tensor], name: str, allow_16bit: bool = False) -> HpdMap:
    m = HpdMap()
    if t is None:
        return m
    if allow_16bit and t.is_cuda and t.dtype in _DTYPE_CODES:
        m.dtype = _DTYPE_CODES[t.dtype]
    else:
        _require_cuda(t, name)
    if t.dim() != 4:
        raise _lib.HpdError(f"{name} must be [B,K,h,w]")
    if t.stride(3) != 1 or t.stride(2) != t.shape[3]:
        raise _lib.HpdError(f"{name}: rows must be contiguous (strides {t.stride()}); call .contiguous()")
    m.ptr = t.data_ptr()
    m.stride_b, m.stride_c = t.stride(0), t.stride(1)
    m.h, m.w = t.shape[2], t.shape[3]
    return m


def make_params(B: int, K: int, H: int, W: int, E: int, M: int, det_thr: float, tag_thr: float, adjust: bool = True,
                refine: bool = True, num_scales: int = 1, tag_scale: int = 0, flip_index=None,
                joints_order=None, tags_preflipped: bool = False) -> HpdParams:
    p = HpdParams()
    p.batch, p.num_kpts, p.out_h, p.out_w, p.emb, p.max_people = B, K, H, W, E, M
    p.num_scales, p.tag_scale = num_scales, tag_scale
    p.do_adjust, p.do_refine = int(adjust), int(refine)
    p.tags_preflipped = int(tags_preflipped)
    p.det_thr, p.tag_thr = float(det_thr), float(tag_thr)
    if flip_index is None:
        flip_index = COCO_FLIP_INDEX if K == 17 else list(range(K))
    if joints_order is None:
        joints_order = JOINTS_ORDER_17 if K == 17 else list(range(K))
    for k in range(min(K, _lib.HPD_MAX_KPTS)):
        p.flip_index[k] = flip_index[k]
        p.joints_order[k] = joints_order[k]
    return p


_layouts = {}


def record_layout(K: int, M: int, E: int) -> HpdRecordLayout:
    """hpd_record_layout for (num_kpts, max_people, emb): byte offsets of one image's result record."""
    key = (K, M, E)
    if key not in _layouts:
        p = HpdParams()
        p.num_kpts, p.max_people, p.emb = K, M, E
        L = HpdRecordLayout()
        _lib.check(_lib.lib().hpd_record_layout(ctypes.byref(p), ctypes.byref(L)), "hpd_record_layout")
        _layouts[key] = L
    return _layouts[key]


class DecodeBuffers:
    """Device buffers of one decode call (HpdBuffers).  Re-usable across calls of the same shape.

    ``records`` [B,row_bytes] uint8 receives one result record per image (HpdRecordLayout) from the epilogue of
    the last kernel; ``inv_affine`` (optional float64 [B,6] on the device) is the per-image matrix the COCO
    section's coordinates are back-projected with (None = network-input coordinates).

    ``tags=False`` allocates no full-resolution tag map (``tag_map`` is None, 4*K*H*W*E bytes per image less): the
    aggregation stage then writes none and the tag stages interpolate the few tags they read from the network outputs,
    which ``run_stage`` hands them from its ``scales``.  ``agg_tags`` is then computed on first read from the network
    outputs of the last decode into the set (``run_aggregate_tags``), which must be unchanged by then."""

    def __init__(self, B: int, K: int, H: int, W: int, E: int, M: int, device, agg_hm: Optional[Tensor] = None,
                 agg_tags: Optional[Tensor] = None, tags: bool = True):
        self.shape = (B, K, H, W, E, M)
        wpr = (W + 31) // 32
        f32 = dict(device=device, dtype=torch.float32)
        i32 = dict(device=device, dtype=torch.int32)
        self.agg_hm = agg_hm if agg_hm is not None else torch.empty((B, K, H, W), **f32)
        self.tag_map = agg_tags if agg_tags is not None else (torch.empty((B, K, H, W, E), **f32) if tags else None)
        self._tag_inputs = self._tag_lazy = None
        self.nms_mask = torch.empty((B, K, H, wpr), **i32)
        self.nms_wmax = torch.empty((B, K, H, wpr), **f32)
        self.hm_wmax = torch.empty((B, K, H, wpr), **f32)
        self.tag_bmin = torch.empty((B, K, (H + 3) // 4, wpr), **f32)
        self.tag_bmax = torch.empty((B, K, (H + 3) // 4, wpr), **f32)
        self.scores_k = torch.empty((B, K, M), **f32)
        self.idx_k = torch.empty((B, K, M), **i32)
        self.coords_k = torch.empty((B, K, M, 2), **i32)
        self.tags_k = torch.empty((B, K, M, E), **f32)
        self.poses = torch.empty((B, M, K, 3 + E), **f32)
        self.person_scores = torch.empty((B, M), **f32)
        self.n_person = torch.empty((B,), **i32)
        self.flags = torch.empty((B,), **i32)
        self.records = torch.empty((B, record_layout(K, M, E).row_bytes), device=device, dtype=torch.uint8)
        self.inv_affine = None
        self.workspace = None

    @classmethod
    def for_grouping(cls, scores_k: Tensor, coords_k: Tensor, tags_k: Tensor) -> "DecodeBuffers":
        """Only what hpd_group touches (top-k inputs, pose outputs); the map-sized buffers stay empty."""
        B, K, M, E = tags_k.shape
        dev = tags_k.device
        self = cls.__new__(cls)
        self.shape = (B, K, 0, 0, E, M)
        zf = torch.empty((0,), device=dev, dtype=torch.float32)
        zi = torch.empty((0,), device=dev, dtype=torch.int32)
        self.agg_hm = self.tag_map = self.nms_wmax = self.hm_wmax = self.tag_bmin = self.tag_bmax = zf
        self._tag_inputs = self._tag_lazy = None
        self.person_scores = zf
        self.nms_mask = self.idx_k = zi
        self.scores_k, self.coords_k, self.tags_k = scores_k, coords_k, tags_k
        self.poses = torch.empty((B, M, K, 3 + E), device=dev, dtype=torch.float32)
        self.n_person = torch.empty((B,), device=dev, dtype=torch.int32)
        self.flags = torch.empty((B,), device=dev, dtype=torch.int32)
        self.records = self.inv_affine = None
        self.workspace = None
        return self

    @property
    def agg_tags(self) -> Optional[Tensor]:
        """[B,K,H,W,E] aggregated tags: the tag map, or for a set without one the map computed (once per decode, on
        the current stream, after the decode's stream) from the network outputs of the last decode into the set."""
        if self.tag_map is not None or self._tag_inputs is None:
            return self.tag_map
        if self._tag_lazy is None:
            scales, params, stream = self._tag_inputs
            B, K, H, W, E, _ = self.shape
            dev = self.agg_hm.device
            torch.cuda.current_stream(dev).wait_stream(stream)
            self._tag_lazy = run_aggregate_tags(scales, params, torch.empty((B, K, H, W, E), device=dev, dtype=torch.float32))
        return self._tag_lazy

    def note_inputs(self, scales: Sequence[dict], params: HpdParams):
        """A decode into this set from these network outputs was enqueued on the current stream (agg_tags)."""
        if self.tag_map is None:
            self._tag_inputs = (scales, params, torch.cuda.current_stream(self.agg_hm.device))
            self._tag_lazy = None

    def struct(self) -> HpdBuffers:
        s = HpdBuffers()
        for name, _ in HpdBuffers._fields_:
            if name == "tag_inputs":        # not a buffer: run_stage / hpd_decode fill it from the scales
                continue
            t = self.tag_map if name == "agg_tags" else getattr(self, name)
            if t is None:
                continue
            if name == "inv_affine" and (t.dtype != torch.float64 or t.numel() != 6 * self.shape[0] or not t.is_cuda):
                raise _lib.HpdError("inv_affine must be a CUDA float64 tensor [B,6]")
            if not t.is_contiguous():
                raise _lib.HpdError(f"buffer {name} must be contiguous")
            setattr(s, name, t.data_ptr())
        return s

    def ensure_workspace(self, params: HpdParams):
        n = ctypes.c_size_t(0)
        _lib.check(_lib.lib().hpd_workspace_bytes(ctypes.byref(params), ctypes.byref(n)), "hpd_workspace_bytes")
        if self.workspace is None or self.workspace.numel() < n.value:
            self.workspace = torch.empty((max(n.value, 8),), device=self.agg_hm.device, dtype=torch.uint8)
        return self.workspace


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def stage_scale(s: dict) -> dict:
    """One test scale's network outputs in the library's scale format {"hm": [stages], "hm_f": [stages] or [],
    "tag", "tag_f"}: heatmap stages in the network's order (1..HPD_MAX_STAGES; the stage mean is taken at the last
    one's size).  The two-stage HigherHRNet dicts {"hm_lo", "hm_hi", "tag"[, "hm_lo_f", "hm_hi_f", "tag_f"]} are
    converted; a dict already in this format is returned as it is."""
    if "hm" in s:
        return s
    flip = s.get("hm_lo_f") is not None
    return {"hm": [s["hm_lo"], s["hm_hi"]], "hm_f": [s["hm_lo_f"], s["hm_hi_f"]] if flip else [],
            "tag": s.get("tag"), "tag_f": s.get("tag_f")}


def scale_tensors(s: dict) -> List[Tensor]:
    """Every tensor of a scale dict (either format)."""
    if "hm" not in s:
        return [t for t in s.values() if t is not None]
    return [t for t in list(s["hm"]) + list(s.get("hm_f") or []) + [s.get("tag"), s.get("tag_f")] if t is not None]


def _stages_struct(scales: Sequence[dict]):
    arr = (HpdStageInputs * len(scales))()
    keep = []
    for i, s in enumerate(scales):
        s = stage_scale(s)
        hm, hm_f = list(s["hm"]), list(s.get("hm_f") or [])
        if not 1 <= len(hm) <= _lib.HPD_MAX_STAGES:
            raise _lib.HpdError(f"a scale has 1 to {_lib.HPD_MAX_STAGES} heatmap stages (got {len(hm)})")
        if hm_f and len(hm_f) != len(hm):
            raise _lib.HpdError(f"flipped-run stages: {len(hm_f)} for {len(hm)} stages")
        arr[i].num_stages = len(hm)
        for j, t in enumerate(hm):
            arr[i].hm[j] = _map(t, f"hm[{j}]", allow_16bit=True)
        for j, t in enumerate(hm_f):
            arr[i].hm_f[j] = _map(t, f"hm_f[{j}]", allow_16bit=True)
        arr[i].tag = _map(s.get("tag"), "tag", allow_16bit=True)
        arr[i].tag_f = _map(s.get("tag_f"), "tag_f", allow_16bit=True)
        keep.append(s)
    return arr, keep


def _scales_struct(scales: Sequence[dict]):
    """HpdScaleInputs of two-stage scale dicts; of the library's scale format only the tag maps are filled (what the
    tag entry points read)."""
    arr = (HpdScaleInputs * len(scales))()
    keep = []
    for i, s in enumerate(scales):
        for name in ("hm_lo", "hm_hi", "tag", "hm_lo_f", "hm_hi_f", "tag_f"):
            t = s.get(name)
            setattr(arr[i], name, _map(t, name, allow_16bit=True))
            keep.append(t)
    return arr, keep


_capture_launches = 0


def _count(L):
    global _launches, _capture_launches
    n = L.hpd_last_launch_count()
    _launches += n
    _capture_launches += n


def launches_in_last_capture() -> int:
    """Launches enqueued since the previous call of this function (DecodePipeline brackets a graph capture with
    two calls and books that many launches per replay)."""
    global _capture_launches
    n, _capture_launches = _capture_launches, 0
    return n


def add_launches(n: int):
    global _launches
    _launches += n


# ------------------------------------------------------------------------------------------------
# functional core (used by the custom ops below and by hpdecode.decoder)
# ------------------------------------------------------------------------------------------------
def run_decode(scales: Optional[Sequence[dict]], bufs: DecodeBuffers, params: HpdParams):
    """hpd_decode on the current stream.  scales=None -> bufs.agg_hm / agg_tags are the inputs."""
    L = _lib.lib()
    dev = bufs.agg_hm.device
    ws = bufs.ensure_workspace(params)
    with torch.cuda.device(dev):
        if scales is not None:
            bufs.note_inputs(scales, params)
            arr, _keep = _stages_struct(scales)
            rc = L.hpd_decode_stages(ctypes.byref(params), arr, ctypes.byref(bufs.struct()), ws.data_ptr(), ws.numel(),
                                     _stream_ptr(dev))
        else:
            rc = L.hpd_decode(ctypes.byref(params), None, ctypes.byref(bufs.struct()), ws.data_ptr(), ws.numel(),
                              _stream_ptr(dev))
    _lib.check(rc, "hpd_decode")
    _count(L)
    return bufs


def run_aggregate_tags(scales: Sequence[dict], params: HpdParams, out: Tensor):
    """hpd_aggregate_tags on the current stream: the full-resolution tag map [B,K,H,W,E] of scales[tag_scale] into
    ``out``: the kernel hpd_aggregate_nms runs to fill a tag map."""
    B, K, H, W, E = params.batch, params.num_kpts, params.out_h, params.out_w, params.emb
    if tuple(out.shape) != (B, K, H, W, E) or not out.is_contiguous() or not out.is_cuda or out.dtype != torch.float32:
        raise _lib.HpdError(f"aggregate_tags: out must be a contiguous CUDA float32 tensor {(B, K, H, W, E)}")
    L = _lib.lib()
    with torch.cuda.device(out.device):
        arr, _keep = _scales_struct(scales)
        rc = L.hpd_aggregate_tags(ctypes.byref(params), arr, out.data_ptr(), _stream_ptr(out.device))
    _lib.check(rc, "hpd_aggregate_tags")
    _count(L)
    return out


def run_stage(stage: str, bufs: DecodeBuffers, params: HpdParams, scales=None, nms_out: Optional[Tensor] = None):
    """One stage on the current stream.  Buffers without a tag map (``tags=False``) need ``scales`` for the tag
    stages (topk, adjust_refine): they interpolate from scales[params.tag_scale]."""
    L = _lib.lib()
    dev = bufs.agg_hm.device
    st = _stream_ptr(dev)
    b = bufs.struct()
    if bufs.tag_map is None and scales is not None and stage in ("topk", "adjust_refine"):
        tag_arr, _keep_tag = _scales_struct([scales[params.tag_scale]])
        b.tag_inputs = tag_arr[0]
    with torch.cuda.device(dev):
        if stage == "aggregate_nms":
            bufs.note_inputs(scales, params)
            arr, _keep = _stages_struct(scales)
            rc = L.hpd_aggregate_nms_stages(ctypes.byref(params), arr, ctypes.byref(b), st)
        elif stage == "nms":
            rc = L.hpd_nms(ctypes.byref(params), ctypes.byref(b), nms_out.data_ptr() if nms_out is not None else None, st)
        elif stage == "topk":
            rc = L.hpd_topk(ctypes.byref(params), ctypes.byref(b), st)
        elif stage == "group":
            rc = L.hpd_group(ctypes.byref(params), ctypes.byref(b), st)
        elif stage == "adjust_refine":
            ws = bufs.ensure_workspace(params)
            rc = L.hpd_adjust_refine(ctypes.byref(params), ctypes.byref(b), ws.data_ptr(), ws.numel(), st)
        else:
            raise ValueError(stage)
    _lib.check(rc, f"hpd_{stage}")
    _count(L)
    return bufs


def coco_eval_params(num_images: int, num_kpts: int, max_dets: int, max_gts: int, iou_thrs: Sequence[float],
                     rec_thrs: Sequence[float], area_rng: Sequence[float], kpt_vars: Sequence[float]) -> HpdCocoEvalParams:
    """HpdCocoEvalParams; the thresholds and variances are taken as given (float64, computed by NumPy upstream).
    area_rng is flat: [lo0, hi0, lo1, hi1, ...]."""
    p = HpdCocoEvalParams()
    p.num_images, p.num_kpts, p.max_dets, p.max_gts = num_images, num_kpts, max_dets, max_gts
    p.num_iou_thrs, p.num_rec_thrs, p.num_areas = len(iou_thrs), len(rec_thrs), len(area_rng) // 2
    if (len(iou_thrs) > _lib.HPD_COCO_MAX_IOU_THRS or len(rec_thrs) > _lib.HPD_COCO_MAX_REC_THRS
            or len(area_rng) > 2 * _lib.HPD_COCO_MAX_AREAS or len(area_rng) % 2 or len(kpt_vars) != num_kpts
            or num_kpts > _lib.HPD_MAX_KPTS):
        raise _lib.HpdError(f"coco_eval: at most {_lib.HPD_COCO_MAX_IOU_THRS} OKS thresholds, {_lib.HPD_COCO_MAX_REC_THRS} "
                            f"recall thresholds, {_lib.HPD_COCO_MAX_AREAS} [lo, hi] area ranges and one variance per "
                            f"joint (<= {_lib.HPD_MAX_KPTS})")
    for j, v in enumerate(iou_thrs):
        p.iou_thrs[j] = v
    for j, v in enumerate(rec_thrs):
        p.rec_thrs[j] = v
    for j, v in enumerate(area_rng):
        p.area_rng[j // 2][j % 2] = v
    for j, v in enumerate(kpt_vars):
        p.kpt_vars[j] = v
    return p


def run_coco_eval(params: HpdCocoEvalParams, records: Sequence[Tensor], row_of_image, off_coco: int, off_count: int,
                  person_stride: int, max_per_row: int, gt: Sequence[Tensor], outs: Sequence[Optional[Tensor]]):
    """hpd_coco_eval on the current stream.  records: uint8 CUDA tensors [rows, >= row bytes] whose rows are read in
    place; row_of_image: host int64 [I], the row of image i counted across ``records`` in order (-1: none).
    gt: (kpts, area, bbox, iscrowd, ignore, n_gt); outs: (precision, recall, scores, oks, codes, npig), the last three
    optional (None)."""
    dev = gt[0].device
    rows = torch.as_tensor(row_of_image, dtype=torch.int64).cpu()
    if rows.numel() != params.num_images:
        raise _lib.HpdError("coco_eval: row_of_image needs one entry per image")
    for t in records:
        if not t.is_cuda or t.dtype != torch.uint8 or t.dim() != 2 or t.stride(1) != 1 or t.device != dev:
            raise _lib.HpdError("coco_eval: detection rows must be 2-D uint8 CUDA tensors with packed bytes, on the "
                                "ground truth's device")
    if not records:
        records = [torch.zeros((0, 8), device=dev, dtype=torch.uint8)]
    base = min(t.data_ptr() for t in records)
    starts = torch.tensor([0] + [t.shape[0] for t in records], dtype=torch.int64).cumsum(0)
    if int(rows.max()) >= int(starts[-1]):
        raise _lib.HpdError("coco_eval: row_of_image points past the last detection row")
    which = torch.searchsorted(starts[1:], rows, right=True).clamp(max=len(records) - 1)
    tbase = torch.tensor([t.data_ptr() - base for t in records], dtype=torch.int64)
    pitch = torch.tensor([t.stride(0) for t in records], dtype=torch.int64)
    offsets = torch.where(rows >= 0, tbase[which] + (rows - starts[which]) * pitch[which], torch.full_like(rows, -1))
    offsets = offsets.to(dev)
    d = HpdCocoDets()
    d.base, d.row_offset, d.off_coco, d.off_count = base, offsets.data_ptr(), off_coco, off_count
    d.person_stride, d.max_per_row = person_stride, max_per_row
    g = HpdCocoGts()
    for (name, dtype), t in zip((("kpts", torch.float64), ("area", torch.float64), ("bbox", torch.float64),
                                 ("iscrowd", torch.uint8), ("ignore", torch.uint8), ("n_gt", torch.int32)), gt):
        if not t.is_cuda or t.dtype != dtype or not t.is_contiguous() or t.device != dev:
            raise _lib.HpdError(f"coco_eval: gt {name} must be a contiguous CUDA {dtype} tensor")
        setattr(g, name, t.data_ptr())
    o = HpdCocoEvalOutputs()
    for name, t in zip(("precision", "recall", "scores", "oks", "codes", "npig"), outs):
        if t is not None:
            if not t.is_cuda or not t.is_contiguous() or t.device != dev:
                raise _lib.HpdError(f"coco_eval: output {name} must be a contiguous CUDA tensor")
            setattr(o, name, t.data_ptr())
    L = _lib.lib()
    n = ctypes.c_size_t(0)
    _lib.check(L.hpd_coco_eval_workspace_bytes(ctypes.byref(params), ctypes.byref(n)), "hpd_coco_eval_workspace_bytes")
    ws = torch.empty((max(n.value, 8),), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        rc = L.hpd_coco_eval(ctypes.byref(params), ctypes.byref(d), ctypes.byref(g), ctypes.byref(o), ws.data_ptr(),
                             ws.numel(), _stream_ptr(dev))
    _lib.check(rc, "hpd_coco_eval")
    _count(L)
    return outs


def track_params(K: int, M: int, E: int, max_age: int, min_keypoints: int, oks_thr: float,
                 kpt_vars: Sequence[float]) -> HpdTrackParams:
    """HpdTrackParams; kpt_vars = (2 sigma)**2 per joint, float64 as NumPy computed them.  The library checks ranges."""
    if len(kpt_vars) != K or K > _lib.HPD_MAX_KPTS:
        raise _lib.HpdError(f"track: one variance per joint (got {len(kpt_vars)} for K={K}, K <= {_lib.HPD_MAX_KPTS})")
    p = HpdTrackParams()
    p.num_kpts, p.max_people, p.emb, p.max_age, p.min_keypoints = K, M, E, max_age, min_keypoints
    p.oks_thr = float(oks_thr)
    for k, v in enumerate(kpt_vars):
        p.kpt_vars[k] = float(v)
    return p


def track_state_bytes(params: HpdTrackParams) -> int:
    n = ctypes.c_size_t(0)
    _lib.check(_lib.lib().hpd_track_state_bytes(ctypes.byref(params), ctypes.byref(n)), "hpd_track_state_bytes")
    return n.value


def _check_state(state: Tensor, device):
    if not state.is_cuda or state.dtype != torch.uint8 or not state.is_contiguous() or state.device != device:
        raise _lib.HpdError("track: the state must be a contiguous uint8 CUDA tensor on the records' device")


def run_track_reset(params: HpdTrackParams, state: Tensor, clear_ids: bool):
    """hpd_track_reset on the current stream: drop every track; clear_ids also restarts the ids at 0."""
    _check_state(state, state.device)
    with torch.cuda.device(state.device):
        rc = _lib.lib().hpd_track_reset(ctypes.byref(params), state.data_ptr(), state.numel(), int(clear_ids),
                                        _stream_ptr(state.device))
    _lib.check(rc, "hpd_track_reset")


def _check_track_args(params: HpdTrackParams, records: Tensor, state: Tensor, out: Tensor):
    row_bytes = record_layout(params.num_kpts, params.max_people, params.emb).row_bytes
    if (not records.is_cuda or records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != row_bytes
            or records.stride(1) != 1 or (records.shape[0] > 1 and records.stride(0) != row_bytes)):
        raise _lib.HpdError(f"track: records must be a uint8 CUDA tensor [n, {row_bytes}] with packed rows")
    _check_state(state, records.device)
    n, M = records.shape[0], params.max_people
    if tuple(out.shape) != (n, M) or out.dtype != torch.int32 or not out.is_contiguous() or out.device != records.device:
        raise _lib.HpdError(f"track: out must be a contiguous int32 tensor {(n, M)} on the records' device")


def run_track(params: HpdTrackParams, records: Tensor, state: Tensor, out: Tensor) -> Tensor:
    """hpd_track on the current stream: records uint8 [n, row_bytes] (rows packed, read in place) -> out int32 [n, M]."""
    _check_track_args(params, records, state, out)
    n = records.shape[0]
    if n == 0:
        return out
    L = _lib.lib()
    with torch.cuda.device(records.device):
        rc = L.hpd_track(ctypes.byref(params), records.data_ptr(), n, state.data_ptr(), state.numel(), out.data_ptr(),
                         _stream_ptr(records.device))
    _lib.check(rc, "hpd_track")
    _count(L)
    return out


def smooth_params(fps: float, min_cutoff: float, beta: float, d_cutoff: float) -> HpdSmoothParams:
    """HpdSmoothParams; the library checks ranges."""
    sp = HpdSmoothParams()
    sp.min_cutoff, sp.beta, sp.d_cutoff, sp.fps = float(min_cutoff), float(beta), float(d_cutoff), float(fps)
    return sp


def track_smooth_state_bytes(params: HpdTrackParams) -> int:
    n = ctypes.c_size_t(0)
    _lib.check(_lib.lib().hpd_track_smooth_state_bytes(ctypes.byref(params), ctypes.byref(n)),
               "hpd_track_smooth_state_bytes")
    return n.value


def run_track_smooth(params: HpdTrackParams, sparams: HpdSmoothParams, records: Tensor, state: Tensor, out: Tensor,
                     coords: Tensor) -> Tuple[Tensor, Tensor]:
    """hpd_track_smooth on the current stream: records uint8 [n, row_bytes] -> out int32 [n, M] and coords float64
    [n, M, K, 2]."""
    _check_track_args(params, records, state, out)
    n, M, K = records.shape[0], params.max_people, params.num_kpts
    if (tuple(coords.shape) != (n, M, K, 2) or coords.dtype != torch.float64 or not coords.is_contiguous()
            or coords.device != records.device):
        raise _lib.HpdError(f"track_smooth: coords must be a contiguous float64 tensor {(n, M, K, 2)} on the records' "
                            "device")
    if n == 0:
        return out, coords
    L = _lib.lib()
    with torch.cuda.device(records.device):
        rc = L.hpd_track_smooth(ctypes.byref(params), ctypes.byref(sparams), records.data_ptr(), n, state.data_ptr(),
                                state.numel(), out.data_ptr(), coords.data_ptr(), _stream_ptr(records.device))
    _lib.check(rc, "hpd_track_smooth")
    _count(L)
    return out, coords


def render_params(K: int, M: int, E: int, limbs: Sequence[int], limb_colors: Sequence[int], joint_color: Sequence[int],
                  track_colors: Sequence[int], untracked_color: Sequence[int], thickness: float, joint_radius: float,
                  kpt_thr: float) -> HpdRenderParams:
    """HpdRenderParams; limbs and colour lists are flat ([a0, b0, a1, b1, ...], [r, g, b, r, g, b, ...]).  The library
    checks ranges."""
    L = len(limbs) // 2
    C = len(track_colors) // 3
    if (len(limbs) % 2 or L > _lib.HPD_RENDER_MAX_LIMBS or len(limb_colors) != 3 * L or len(track_colors) % 3
            or C > _lib.HPD_RENDER_MAX_COLORS or len(joint_color) != 3 or len(untracked_color) != 3):
        raise _lib.HpdError(f"render: up to {_lib.HPD_RENDER_MAX_LIMBS} limbs with one colour each, up to "
                            f"{_lib.HPD_RENDER_MAX_COLORS} track colours, colours of 3 bytes")
    p = HpdRenderParams()
    p.num_kpts, p.max_people, p.emb, p.num_limbs, p.num_track_colors = K, M, E, L, C
    for l in range(L):
        p.limbs[l][0], p.limbs[l][1] = limbs[2 * l], limbs[2 * l + 1]
        for c in range(3):
            p.limb_rgb[l][c] = limb_colors[3 * l + c]
    for i in range(C):
        for c in range(3):
            p.track_rgb[i][c] = track_colors[3 * i + c]
    for c in range(3):
        p.joint_rgb[c], p.untracked_rgb[c] = joint_color[c], untracked_color[c]
    p.thickness, p.joint_radius, p.kpt_thr = float(thickness), float(joint_radius), float(kpt_thr)
    return p


def _check_frame(t: Tensor, what: str):
    if not t.is_cuda or t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
        raise _lib.HpdError(f"render: {what} must be a CUDA uint8 [h,w,3] tensor with packed pixels")


def run_render(params: HpdRenderParams, frames: Sequence[Tensor], out: Sequence[Tensor], records: Tensor,
               track_ids: Optional[Tensor] = None, coords: Optional[Tensor] = None) -> Sequence[Tensor]:
    """hpd_render_poses on the current stream: frames[i] drawn with the persons of records[i] (uint8 [n, row_bytes],
    rows packed) into out[i] (same size; any row stride).  track_ids: int32 [n, M]; coords: float64 [n, M, K, 2]."""
    n, M, K = len(frames), params.max_people, params.num_kpts
    row_bytes = record_layout(K, M, params.emb).row_bytes
    if (not records.is_cuda or records.dtype != torch.uint8 or records.dim() != 2 or records.shape != (n, row_bytes)
            or records.stride(1) != 1 or (n > 1 and records.stride(0) != row_bytes)):
        raise _lib.HpdError(f"render: records must be a uint8 CUDA tensor [{n}, {row_bytes}] with packed rows")
    dev = records.device
    for name, t, dtype, shape in (("track_ids", track_ids, torch.int32, (n, M)),
                                  ("coords", coords, torch.float64, (n, M, K, 2))):
        if t is not None and (tuple(t.shape) != shape or t.dtype != dtype or not t.is_contiguous() or t.device != dev):
            raise _lib.HpdError(f"render: {name} must be a contiguous {dtype} tensor {shape} on the records' device")
    if len(out) != n:
        raise _lib.HpdError("render: one output per frame")
    if n == 0:
        return out
    arr = (HpdRenderFrame * n)()
    for i, (f, o) in enumerate(zip(frames, out)):
        _check_frame(f, "frame %d" % i)
        _check_frame(o, "output %d" % i)
        if f.device != dev or o.device != dev or f.shape != o.shape:
            raise _lib.HpdError("render: frame %d and its output must have one size, on the records' device" % i)
        setattr(arr[i], "in", f.data_ptr())
        arr[i].out, arr[i].in_stride_row, arr[i].out_stride_row = o.data_ptr(), f.stride(0), o.stride(0)
        arr[i].h, arr[i].w = f.shape[0], f.shape[1]
    L = _lib.lib()
    with torch.cuda.device(dev):
        rc = L.hpd_render_poses(ctypes.byref(params), arr, n, records.data_ptr(),
                                None if track_ids is None else track_ids.data_ptr(),
                                None if coords is None else coords.data_ptr(), _stream_ptr(dev))
    _lib.check(rc, "hpd_render_poses")
    _count(L)
    return out


def _scales_from_lists(hm_lo, hm_hi, tag, hm_lo_f, hm_hi_f, tag_f):
    n = len(hm_lo)
    flip = len(hm_lo_f) > 0
    out = []
    for i in range(n):
        d = {"hm_lo": hm_lo[i], "hm_hi": hm_hi[i], "tag": tag[i] if i < len(tag) else None}
        if flip:
            d.update(hm_lo_f=hm_lo_f[i], hm_hi_f=hm_hi_f[i], tag_f=tag_f[i] if i < len(tag_f) else None)
        out.append(d)
    return out


def _decode_scales(scales: Sequence[dict], out_h: int, out_w: int, max_people: int, det_thr: float, tag_thr: float,
                   adjust: bool, refine: bool, tag_scale: int) -> List[Tensor]:
    for s in scales:
        for t in scale_tensors(s):
            if not (t.is_cuda and t.dtype in _DTYPE_CODES):
                _require_cuda(t, "network output")
    first = stage_scale(scales[0])["hm"][0]
    B, K = first.shape[:2]
    E = 2 if stage_scale(scales[tag_scale]).get("tag_f") is not None else 1
    bufs = DecodeBuffers(B, K, out_h, out_w, E, max_people, first.device)
    params = make_params(B, K, out_h, out_w, E, max_people, det_thr, tag_thr, adjust, refine, len(scales), tag_scale)
    run_decode(scales, bufs, params)
    return [bufs.agg_hm, bufs.agg_tags, bufs.poses, bufs.person_scores, bufs.n_person, bufs.flags, bufs.scores_k,
            bufs.idx_k, bufs.coords_k, bufs.tags_k]


def _decode_fake(first: Tensor, out_h: int, out_w: int, max_people: int, E: int) -> List[Tensor]:
    B, K = first.shape[:2]
    M = max_people
    f = lambda *s: first.new_empty(s, dtype=torch.float32)
    i = lambda *s: first.new_empty(s, dtype=torch.int32)
    return [f(B, K, out_h, out_w), f(B, K, out_h, out_w, E), f(B, M, K, 3 + E), f(B, M), i(B), i(B), f(B, K, M),
            i(B, K, M), i(B, K, M, 2), f(B, K, M, E)]


# ------------------------------------------------------------------------------------------------
# torch.library custom ops
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("hpd::decode_stages", mutates_args=())
def decode_stages_op(hm: Sequence[Tensor], hm_f: Sequence[Tensor], tag: Sequence[Tensor], tag_f: Sequence[Tensor],
                     num_stages: int, out_h: int, out_w: int, max_people: int, det_thr: float, tag_thr: float,
                     adjust: bool, refine: bool, tag_scale: int) -> List[Tensor]:
    """``hpd::decode`` for heads with ``num_stages`` (1..4) heatmap stages per scale.  ``hm``: the stages of every
    scale, scale-major (scale s, stage i at s * num_stages + i); ``hm_f`` the same for the flipped run, or empty;
    ``tag`` / ``tag_f``: one entry per scale (``tag_f`` empty without the flip test).  -> [agg_hm, agg_tags, poses,
    person_scores, n_person, flags, scores_k, idx_k, coords_k, tags_k]."""
    if num_stages < 1 or len(hm) == 0 or len(hm) % num_stages or (len(hm_f) and len(hm_f) != len(hm)):
        raise _lib.HpdError("decode_stages: hm (and hm_f) must hold num_stages maps per scale")
    n = num_stages
    scales = [{"hm": list(hm[s * n:(s + 1) * n]), "hm_f": list(hm_f[s * n:(s + 1) * n]) if len(hm_f) else [],
               "tag": tag[s] if s < len(tag) else None, "tag_f": tag_f[s] if s < len(tag_f) else None}
              for s in range(len(hm) // n)]
    return _decode_scales(scales, out_h, out_w, max_people, det_thr, tag_thr, adjust, refine, tag_scale)


@decode_stages_op.register_fake
def _(hm, hm_f, tag, tag_f, num_stages, out_h, out_w, max_people, det_thr, tag_thr, adjust, refine, tag_scale):
    return _decode_fake(hm[0], out_h, out_w, max_people, 2 if len(tag_f) > 0 else 1)


@torch.library.custom_op("hpd::decode", mutates_args=())
def decode_op(hm_lo: Sequence[Tensor], hm_hi: Sequence[Tensor], tag: Sequence[Tensor], hm_lo_f: Sequence[Tensor],
              hm_hi_f: Sequence[Tensor], tag_f: Sequence[Tensor], out_h: int, out_w: int, max_people: int,
              det_thr: float, tag_thr: float, adjust: bool, refine: bool, tag_scale: int) -> List[Tensor]:
    """Network outputs (one list entry per test scale; float32, or all float16 or all bfloat16) -> [agg_hm, agg_tags,
    poses, person_scores, n_person, flags, scores_k, idx_k, coords_k, tags_k]."""
    for name, ts in (("hm_lo", hm_lo), ("hm_hi", hm_hi), ("tag", tag), ("hm_lo_f", hm_lo_f), ("hm_hi_f", hm_hi_f),
                     ("tag_f", tag_f)):
        for t in ts:
            if not (t.is_cuda and t.dtype in _DTYPE_CODES):
                _require_cuda(t, name)
    scales = _scales_from_lists(hm_lo, hm_hi, tag, hm_lo_f, hm_hi_f, tag_f)
    return _decode_scales(scales, out_h, out_w, max_people, det_thr, tag_thr, adjust, refine, tag_scale)


@torch.library.custom_op("hpd::parse", mutates_args=())
def parse_op(agg_hm: Tensor, agg_tags: Tensor, max_people: int, det_thr: float, tag_thr: float, adjust: bool,
             refine: bool) -> List[Tensor]:
    """Aggregated maps [B,K,H,W] / [B,K,H,W,E] -> [poses, person_scores, n_person, flags, scores_k, idx_k,
    coords_k, tags_k]   (MPPEHeatmapParser.parse, grouping.py:252-283)."""
    _require_cuda(agg_hm, "agg_hm")
    _require_cuda(agg_tags, "agg_tags")
    B, K, H, W = agg_hm.shape
    E = agg_tags.shape[4]
    bufs = DecodeBuffers(B, K, H, W, E, max_people, agg_hm.device, agg_hm.contiguous(), agg_tags.contiguous())
    params = make_params(B, K, H, W, E, max_people, det_thr, tag_thr, adjust, refine)
    run_decode(None, bufs, params)
    return [bufs.poses, bufs.person_scores, bufs.n_person, bufs.flags, bufs.scores_k, bufs.idx_k, bufs.coords_k,
            bufs.tags_k]


@torch.library.custom_op("hpd::nms", mutates_args=())
def nms_op(hm: Tensor) -> Tensor:
    """MPPEHeatmapParser.nms on [B,K,H,W] (grouping.py:80-83): x where it equals its 5x5 max, else x*0."""
    _require_cuda(hm, "hm")
    B, K, H, W = hm.shape
    bufs = DecodeBuffers(B, K, H, W, 1, 1, hm.device, hm.contiguous(), torch.empty((0,), device=hm.device))
    params = make_params(B, K, H, W, 1, 1, 0.0, 0.0)
    out = torch.empty_like(bufs.agg_hm)
    run_stage("nms", bufs, params, nms_out=out)
    return out


@torch.library.custom_op("hpd::topk", mutates_args=())
def topk_op(agg_hm: Tensor, agg_tags: Tensor, max_people: int) -> List[Tensor]:
    """MPPEHeatmapParser.top_k on [B,K,H,W] / [B,K,H,W,E] (grouping.py:147-170):
    [tags_k, coords_k, scores_k, idx_k]."""
    _require_cuda(agg_hm, "agg_hm")
    _require_cuda(agg_tags, "agg_tags")
    B, K, H, W = agg_hm.shape
    E = agg_tags.shape[4]
    bufs = DecodeBuffers(B, K, H, W, E, max_people, agg_hm.device, agg_hm.contiguous(), agg_tags.contiguous())
    params = make_params(B, K, H, W, E, max_people, 0.0, 0.0)
    run_stage("nms", bufs, params)
    run_stage("topk", bufs, params)
    return [bufs.tags_k, bufs.coords_k, bufs.scores_k, bufs.idx_k]


@torch.library.custom_op("hpd::group", mutates_args=())
def group_op(tags_k: Tensor, coords_k: Tensor, scores_k: Tensor, det_thr: float, tag_thr: float,
             out_h: int, out_w: int) -> List[Tensor]:
    """MPPEHeatmapParser.match_by_tag on [B,K,M,E] / [B,K,M,2] / [B,K,M] (grouping.py:85-145):
    [poses [B,M,K,3+E], n_person [B], flags [B]]."""
    _require_cuda(tags_k, "tags_k")
    _require_cuda(scores_k, "scores_k")
    B, K, M, E = tags_k.shape
    dev = tags_k.device
    params = make_params(B, K, out_h, out_w, E, M, det_thr, tag_thr)
    bufs = DecodeBuffers.for_grouping(scores_k.contiguous(), coords_k.contiguous().int(), tags_k.contiguous())
    run_stage("group", bufs, params)
    return [bufs.poses, bufs.n_person, bufs.flags]


@torch.library.custom_op("hpd::resize_bilinear", mutates_args=())
def resize_bilinear_op(x: Tensor, out_h: int, out_w: int) -> Tensor:
    """F.interpolate(x, size=[out_h, out_w], mode='bilinear', align_corners=False) with torch's CPU
    arithmetic (results.py:46-67) on a [B,C,h,w] CUDA tensor."""
    m = _map(x, "x")
    B, C = x.shape[:2]
    out = torch.empty((B, C, out_h, out_w), device=x.device, dtype=torch.float32)
    L = _lib.lib()
    with torch.cuda.device(x.device):
        rc = L.hpd_resize_bilinear(ctypes.byref(m), B, C, out.data_ptr(), out_h, out_w, _stream_ptr(x.device))
    _lib.check(rc, "hpd_resize_bilinear")
    _count(L)
    return out


@torch.library.custom_op("hpd::prepare_input", mutates_args=())
def prepare_input_op(images: Sequence[Tensor], matrices: Tensor, out_h: int, out_w: int, mean: Sequence[float],
                     std: Sequence[float]) -> Tensor:
    """cv2.warpAffine(image, M, (out_w, out_h)) + ToTensor + Normalize (utils.py:96, model.py:45-50) for a batch of
    uint8 [h,w,3] CUDA images; ``matrices``: float64 [B,6] on the HOST (the forward 2x3 matrices).  -> [B,3,out_h,out_w]."""
    if len(images) == 0 or matrices.is_cuda or matrices.dtype != torch.float64 or matrices.numel() != 6 * len(images):
        raise _lib.HpdError("prepare_input: need >= 1 image and a host float64 [B,6] matrix tensor")
    dev = images[0].device
    arr = (HpdImage * len(images))()
    mats = matrices.reshape(-1, 6).tolist()
    for i, t in enumerate(images):
        if not t.is_cuda or t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
            raise _lib.HpdError("prepare_input: image %d must be a CUDA uint8 [h,w,3] tensor with packed pixels" % i)
        arr[i].ptr, arr[i].stride_row, arr[i].h, arr[i].w = t.data_ptr(), t.stride(0), t.shape[0], t.shape[1]
        for j in range(6):
            arr[i].m[j] = mats[i][j]
    out = torch.empty((len(images), 3, out_h, out_w), device=dev, dtype=torch.float32)
    mean_c, std_c = (ctypes.c_float * 3)(*mean), (ctypes.c_float * 3)(*std)
    L = _lib.lib()
    with torch.cuda.device(dev):
        rc = L.hpd_prepare_input(arr, len(images), out.data_ptr(), out_h, out_w, mean_c, std_c, _stream_ptr(dev))
    _lib.check(rc, "hpd_prepare_input")
    _count(L)
    return out


def _image_descriptors(images: Sequence[Tensor], mats, who: str):
    """HpdImage array: entry e = images[e % len(images)] with the 2x3 matrix mats[e]."""
    arr = (HpdImage * len(mats))()
    for i, t in enumerate(images):
        if not t.is_cuda or t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
            raise _lib.HpdError("%s: image %d must be a CUDA uint8 [h,w,3] tensor with packed pixels" % (who, i))
    for e, m in enumerate(mats):
        t = images[e % len(images)]
        arr[e].ptr, arr[e].stride_row, arr[e].h, arr[e].w = t.data_ptr(), t.stride(0), t.shape[0], t.shape[1]
        for j in range(6):
            arr[e].m[j] = m[j]
    return arr


@torch.library.custom_op("hpd::prepare_inputs", mutates_args=())
def prepare_inputs_op(images: Sequence[Tensor], matrices: Tensor, sizes_hw: Sequence[int], flip: bool,
                      mean: Sequence[float], std: Sequence[float]) -> Tuple[List[Tensor], List[Tensor]]:
    """``prepare_input`` for every test scale of a batch in ONE library call (hpd_prepare_inputs): uint8 [h,w,3] CUDA
    images; ``matrices``: float64 [T,B,6] on the HOST (the forward matrix of image b at scale t); ``sizes_hw``: the
    output (h, w) of each scale, flat [h0, w0, h1, w1, ...].  -> (xs, xs_flipped): T tensors [B,3,h_t,w_t] and, with
    ``flip``, their mirrored copies (torch.flip(x, [3]), bit for bit), else an empty list."""
    B = len(images)
    T = len(sizes_hw) // 2
    if (B == 0 or T == 0 or len(sizes_hw) % 2 or matrices.is_cuda or matrices.dtype != torch.float64
            or matrices.numel() != 6 * T * B):
        raise _lib.HpdError("prepare_inputs: need >= 1 image, (h, w) per scale and a host float64 [T,B,6] matrix tensor")
    dev = images[0].device
    arr = _image_descriptors(images, matrices.reshape(-1, 6).tolist(), "prepare_inputs")
    xs = [torch.empty((B, 3, sizes_hw[2 * t], sizes_hw[2 * t + 1]), device=dev, dtype=torch.float32) for t in range(T)]
    xs_f = [torch.empty_like(x) for x in xs] if flip else []
    targets = (_lib.HpdPrepareTarget * T)()
    for t in range(T):
        targets[t].out, targets[t].out_h, targets[t].out_w = xs[t].data_ptr(), sizes_hw[2 * t], sizes_hw[2 * t + 1]
        targets[t].out_flipped = xs_f[t].data_ptr() if flip else None
    mean_c, std_c = (ctypes.c_float * 3)(*mean), (ctypes.c_float * 3)(*std)
    L = _lib.lib()
    with torch.cuda.device(dev):
        rc = L.hpd_prepare_inputs(arr, B, targets, T, mean_c, std_c, _stream_ptr(dev))
    _lib.check(rc, "hpd_prepare_inputs")
    _count(L)
    return xs, xs_f


@prepare_inputs_op.register_fake
def _(images, matrices, sizes_hw, flip, mean, std):
    B = len(images)
    xs = [images[0].new_empty((B, 3, sizes_hw[2 * t], sizes_hw[2 * t + 1]), dtype=torch.float32)
          for t in range(len(sizes_hw) // 2)]
    return xs, ([torch.empty_like(x) for x in xs] if flip else [])


@torch.library.custom_op("hpd::coco_eval", mutates_args=())
def coco_eval_op(records: Sequence[Tensor], row_of_image: Tensor, off_coco: int, off_count: int, person_stride: int,
                 max_per_row: int, gt_kpts: Tensor, gt_area: Tensor, gt_bbox: Tensor, gt_iscrowd: Tensor,
                 gt_ignore: Tensor, n_gt: Tensor, iou_thrs: Sequence[float], rec_thrs: Sequence[float],
                 area_rng: Sequence[float], kpt_vars: Sequence[float], max_dets: int, debug: bool) -> List[Tensor]:
    """COCOeval(gt, dt, "keypoints").evaluate() + accumulate() for category 1 (pycocotools cocoeval.py):
    detections read in place from ``records`` (see run_coco_eval), ground truth padded [I,G,...].
    -> [precision [T,R,A], recall [T,A], scores [T,R,A], oks [I,max_dets,G], codes [A,T,I,max_dets] uint8,
    npig [A] int64]; the last three are empty unless ``debug``."""
    I, G, K = gt_kpts.shape[:3]
    params = coco_eval_params(I, K, max_dets, G, iou_thrs, rec_thrs, area_rng, kpt_vars)
    T, R, A = params.num_iou_thrs, params.num_rec_thrs, params.num_areas
    f64 = dict(device=gt_kpts.device, dtype=torch.float64)
    outs = [torch.empty((T, R, A), **f64), torch.empty((T, A), **f64), torch.empty((T, R, A), **f64)]
    if debug:
        outs += [torch.empty((I, max_dets, G), **f64), torch.empty((A, T, I, max_dets), device=gt_kpts.device,
                 dtype=torch.uint8), torch.empty((A,), device=gt_kpts.device, dtype=torch.int64)]
    else:
        outs += [None, None, None]
    run_coco_eval(params, records, row_of_image, off_coco, off_count, person_stride, max_per_row,
                  (gt_kpts, gt_area, gt_bbox, gt_iscrowd, gt_ignore, n_gt), outs)
    return [t if t is not None else gt_kpts.new_empty((0,)) for t in outs]


@coco_eval_op.register_fake
def _(records, row_of_image, off_coco, off_count, person_stride, max_per_row, gt_kpts, gt_area, gt_bbox, gt_iscrowd,
      gt_ignore, n_gt, iou_thrs, rec_thrs, area_rng, kpt_vars, max_dets, debug):
    I, G = gt_kpts.shape[:2]
    T, R, A = len(iou_thrs), len(rec_thrs), len(area_rng) // 2
    f = lambda *s: gt_kpts.new_empty(s)
    if debug:
        tail = [f(I, max_dets, G), gt_kpts.new_empty((A, T, I, max_dets), dtype=torch.uint8),
                gt_kpts.new_empty((A,), dtype=torch.int64)]
    else:
        tail = [f(0), f(0), f(0)]
    return [f(T, R, A), f(T, A), f(T, R, A)] + tail


@torch.library.custom_op("hpd::track", mutates_args=("state",))
def track_op(records: Tensor, state: Tensor, num_kpts: int, max_people: int, emb: int, max_age: int,
             min_keypoints: int, oks_thr: float, kpt_vars: Sequence[float]) -> Tensor:
    """Person ids of consecutive frames (hpd_track): ``records`` uint8 [n, row_bytes] result records in time order,
    ``state`` the tracker state (updated in place) -> int32 [n, max_people], -1 for persons without a track and for
    slots past the frame's persons."""
    params = track_params(num_kpts, max_people, emb, max_age, min_keypoints, oks_thr, kpt_vars)
    out = torch.empty((records.shape[0], max_people), device=records.device, dtype=torch.int32)
    return run_track(params, records, state, out)


@track_op.register_fake
def _(records, state, num_kpts, max_people, emb, max_age, min_keypoints, oks_thr, kpt_vars):
    return records.new_empty((records.shape[0], max_people), dtype=torch.int32)


@torch.library.custom_op("hpd::track_smooth", mutates_args=("state",))
def track_smooth_op(records: Tensor, state: Tensor, num_kpts: int, max_people: int, emb: int, max_age: int,
                    min_keypoints: int, oks_thr: float, kpt_vars: Sequence[float], fps: float, min_cutoff: float,
                    beta: float, d_cutoff: float) -> Tuple[Tensor, Tensor]:
    """hpd::track's ids plus the tracked joints' One-Euro-filtered COCO-section coordinates (hpd_track_smooth):
    -> (int32 [n, max_people], float64 [n, max_people, num_kpts, 2]); ``state`` is a smoothing tracker state."""
    params = track_params(num_kpts, max_people, emb, max_age, min_keypoints, oks_thr, kpt_vars)
    n = records.shape[0]
    out = torch.empty((n, max_people), device=records.device, dtype=torch.int32)
    coords = torch.empty((n, max_people, num_kpts, 2), device=records.device, dtype=torch.float64)
    return run_track_smooth(params, smooth_params(fps, min_cutoff, beta, d_cutoff), records, state, out, coords)


@track_smooth_op.register_fake
def _(records, state, num_kpts, max_people, emb, max_age, min_keypoints, oks_thr, kpt_vars, fps, min_cutoff, beta,
      d_cutoff):
    n = records.shape[0]
    return (records.new_empty((n, max_people), dtype=torch.int32),
            records.new_empty((n, max_people, num_kpts, 2), dtype=torch.float64))


@torch.library.custom_op("hpd::render_poses", mutates_args=())
def render_poses_op(frames: Sequence[Tensor], records: Tensor, track_ids: Optional[Tensor], coords: Optional[Tensor],
                    num_kpts: int, max_people: int, emb: int, limbs: Sequence[int], limb_colors: Sequence[int],
                    joint_color: Sequence[int], track_colors: Sequence[int], untracked_color: Sequence[int],
                    thickness: float, joint_radius: float, kpt_thr: float) -> List[Tensor]:
    """Skeletons and joints of the persons of records[i] drawn into a new copy of frames[i] (hpd_render_poses; uint8
    [h,w,3] CUDA frames, left unchanged): -> one new contiguous uint8 [h,w,3] tensor per frame.  ``limbs`` and the
    colours are flat lists (pairs, RGB triples); ``track_ids`` int32 [n, max_people] and ``coords`` float64
    [n, max_people, num_kpts, 2] are optional."""
    params = render_params(num_kpts, max_people, emb, limbs, limb_colors, joint_color, track_colors, untracked_color,
                           thickness, joint_radius, kpt_thr)
    out = [torch.empty((f.shape[0], f.shape[1], 3), device=f.device, dtype=torch.uint8) for f in frames]
    run_render(params, frames, out, records, track_ids, coords)
    return out


@render_poses_op.register_fake
def _(frames, records, track_ids, coords, num_kpts, max_people, emb, limbs, limb_colors, joint_color, track_colors,
      untracked_color, thickness, joint_radius, kpt_thr):
    return [f.new_empty((f.shape[0], f.shape[1], 3), dtype=torch.uint8) for f in frames]


@prepare_input_op.register_fake
def _(images, matrices, out_h, out_w, mean, std):
    return images[0].new_empty((len(images), 3, out_h, out_w), dtype=torch.float32)


@resize_bilinear_op.register_fake
def _(x, out_h, out_w):
    return x.new_empty((x.shape[0], x.shape[1], out_h, out_w))


@decode_op.register_fake
def _(hm_lo, hm_hi, tag, hm_lo_f, hm_hi_f, tag_f, out_h, out_w, max_people, det_thr, tag_thr, adjust, refine,
      tag_scale):
    return _decode_fake(hm_lo[0], out_h, out_w, max_people, 2 if len(tag_f) > 0 else 1)


@parse_op.register_fake
def _(agg_hm, agg_tags, max_people, det_thr, tag_thr, adjust, refine):
    B, K = agg_hm.shape[:2]
    E, M = agg_tags.shape[4], max_people
    f = lambda *s: agg_hm.new_empty(s)
    i = lambda *s: agg_hm.new_empty(s, dtype=torch.int32)
    return [f(B, M, K, 3 + E), f(B, M), i(B), i(B), f(B, K, M), i(B, K, M), i(B, K, M, 2), f(B, K, M, E)]


@nms_op.register_fake
def _(hm):
    return torch.empty_like(hm)


@topk_op.register_fake
def _(agg_hm, agg_tags, max_people):
    B, K = agg_hm.shape[:2]
    E, M = agg_tags.shape[4], max_people
    return [agg_hm.new_empty((B, K, M, E)), agg_hm.new_empty((B, K, M, 2), dtype=torch.int32), agg_hm.new_empty((B, K, M)),
            agg_hm.new_empty((B, K, M), dtype=torch.int32)]


@group_op.register_fake
def _(tags_k, coords_k, scores_k, det_thr, tag_thr, out_h, out_w):
    B, K, M, E = tags_k.shape
    return [tags_k.new_empty((B, M, K, 3 + E)), tags_k.new_empty((B,), dtype=torch.int32),
            tags_k.new_empty((B,), dtype=torch.int32)]
