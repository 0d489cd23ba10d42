"""ctypes binding of libhpdecode.so (include/hpdecode.h).

The library is the product: there is NO CPU or eager-PyTorch fallback.  ``lib()`` raises if the
shared object is missing; every op raises if it is handed non-CUDA tensors.
"""
import ctypes
import os

HPD_MAX_KPTS = 32
HPD_MAX_PEOPLE = 32
HPD_MAX_EMB = 2
HPD_MAX_SCALES = 4
HPD_MAX_STAGES = 4
HPD_ABI_VERSION = 6
HPD_COCO_MAX_IOU_THRS, HPD_COCO_MAX_REC_THRS, HPD_COCO_MAX_AREAS, HPD_COCO_MAX_PER_IMAGE = 16, 128, 4, 1024
HPD_F32, HPD_F16, HPD_BF16 = 0, 1, 2
HPD_TRACK_MAX_AGE = 8
HPD_RENDER_MAX_LIMBS, HPD_RENDER_MAX_COLORS = 64, 32

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhpdecode.so")

EXPORTS = (
    "hpd_abi_version", "hpd_last_error_string", "hpd_workspace_bytes", "hpd_aggregate_nms", "hpd_nms",
    "hpd_topk", "hpd_group", "hpd_adjust_refine", "hpd_decode", "hpd_last_launch_count", "hpd_resize_bilinear",
    "hpd_record_layout", "hpd_multi_scale_size", "hpd_get_affine_transform", "hpd_prepare_input", "hpd_prepare_geometry",
    "hpd_aggregate_tags", "hpd_coco_eval_workspace_bytes", "hpd_coco_eval", "hpd_prepare_inputs",
    "hpd_aggregate_nms_stages", "hpd_decode_stages", "hpd_track_state_bytes", "hpd_track_reset", "hpd_track",
    "hpd_track_smooth_state_bytes", "hpd_track_smooth", "hpd_render_poses",
)


class HpdMap(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("stride_b", ctypes.c_int64), ("stride_c", ctypes.c_int64),
                ("h", ctypes.c_int32), ("w", ctypes.c_int32), ("dtype", ctypes.c_int32), ("reserved_", ctypes.c_int32)]


class HpdScaleInputs(ctypes.Structure):
    _fields_ = [("hm_lo", HpdMap), ("hm_hi", HpdMap), ("tag", HpdMap),
                ("hm_lo_f", HpdMap), ("hm_hi_f", HpdMap), ("tag_f", HpdMap)]


class HpdStageInputs(ctypes.Structure):
    _fields_ = [("hm", HpdMap * HPD_MAX_STAGES), ("hm_f", HpdMap * HPD_MAX_STAGES), ("tag", HpdMap), ("tag_f", HpdMap),
                ("num_stages", ctypes.c_int32), ("reserved_", ctypes.c_int32)]


class HpdParams(ctypes.Structure):
    _fields_ = [("batch", ctypes.c_int32), ("num_kpts", ctypes.c_int32), ("out_h", ctypes.c_int32),
                ("out_w", ctypes.c_int32), ("emb", ctypes.c_int32), ("max_people", ctypes.c_int32),
                ("num_scales", ctypes.c_int32), ("tag_scale", ctypes.c_int32), ("do_adjust", ctypes.c_int32),
                ("do_refine", ctypes.c_int32), ("tags_preflipped", ctypes.c_int32), ("force_generic", ctypes.c_int32),
                ("batches_in_flight", ctypes.c_int32), ("reserved_", ctypes.c_int32),
                ("det_thr", ctypes.c_double), ("tag_thr", ctypes.c_double),
                ("flip_index", ctypes.c_int32 * HPD_MAX_KPTS), ("joints_order", ctypes.c_int32 * HPD_MAX_KPTS)]


class HpdBuffers(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in (
        "agg_hm", "agg_tags", "nms_mask", "nms_wmax", "hm_wmax", "scores_k", "idx_k", "coords_k", "tags_k",
        "poses", "person_scores", "n_person", "flags", "tag_bmin", "tag_bmax", "records", "inv_affine")] + [
        ("tag_inputs", HpdScaleInputs)]


class HpdRecordLayout(ctypes.Structure):
    _fields_ = [("row_bytes", ctypes.c_int64), ("off_coco", ctypes.c_int64), ("off_poses", ctypes.c_int64),
                ("off_person_scores", ctypes.c_int64), ("off_n_person", ctypes.c_int64), ("off_flags", ctypes.c_int64),
                ("coco_stride", ctypes.c_int32), ("reserved_", ctypes.c_int32)]


class HpdImage(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("stride_row", ctypes.c_int64), ("h", ctypes.c_int32), ("w", ctypes.c_int32),
                ("m", ctypes.c_double * 6)]


class HpdPrepareTarget(ctypes.Structure):
    _fields_ = [("out", ctypes.c_void_p), ("out_flipped", ctypes.c_void_p), ("out_h", ctypes.c_int32),
                ("out_w", ctypes.c_int32)]


class HpdCocoEvalParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("num_images", "num_kpts", "max_dets", "max_gts", "num_iou_thrs",
                                              "num_rec_thrs", "num_areas", "reserved_")] + [
        ("iou_thrs", ctypes.c_double * HPD_COCO_MAX_IOU_THRS), ("rec_thrs", ctypes.c_double * HPD_COCO_MAX_REC_THRS),
        ("area_rng", (ctypes.c_double * 2) * HPD_COCO_MAX_AREAS), ("kpt_vars", ctypes.c_double * HPD_MAX_KPTS)]


class HpdCocoDets(ctypes.Structure):
    _fields_ = [("base", ctypes.c_void_p), ("row_offset", ctypes.c_void_p), ("off_coco", ctypes.c_int64),
                ("off_count", ctypes.c_int64), ("person_stride", ctypes.c_int32), ("max_per_row", ctypes.c_int32)]


class HpdCocoGts(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("kpts", "area", "bbox", "iscrowd", "ignore", "n_gt")]


class HpdCocoEvalOutputs(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("precision", "recall", "scores", "oks", "codes", "npig")]


class HpdTrackParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("num_kpts", "max_people", "emb", "max_age", "min_keypoints",
                                              "reserved_")] + [
        ("oks_thr", ctypes.c_double), ("kpt_vars", ctypes.c_double * HPD_MAX_KPTS)]


class HpdSmoothParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in ("min_cutoff", "beta", "d_cutoff", "fps")]


class HpdRenderParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("num_kpts", "max_people", "emb", "num_limbs")] + [
        ("limbs", (ctypes.c_int32 * 2) * HPD_RENDER_MAX_LIMBS), ("limb_rgb", (ctypes.c_uint8 * 3) * HPD_RENDER_MAX_LIMBS),
        ("joint_rgb", ctypes.c_uint8 * 3), ("untracked_rgb", ctypes.c_uint8 * 3), ("reserved0_", ctypes.c_uint8 * 2),
        ("num_track_colors", ctypes.c_int32), ("reserved1_", ctypes.c_int32),
        ("track_rgb", (ctypes.c_uint8 * 3) * HPD_RENDER_MAX_COLORS)] + [
        (n, ctypes.c_double) for n in ("thickness", "joint_radius", "kpt_thr")]


class HpdRenderFrame(ctypes.Structure):
    _fields_ = [("in", ctypes.c_void_p), ("out", ctypes.c_void_p), ("in_stride_row", ctypes.c_int64),
                ("out_stride_row", ctypes.c_int64), ("h", ctypes.c_int32), ("w", ctypes.c_int32)]


class HpdError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libhpdecode.so or fail loudly (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise HpdError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  hpdecode has no CPU / eager fallback.")
    L = ctypes.CDLL(LIB_PATH)
    L.hpd_abi_version.restype = ctypes.c_int
    L.hpd_last_error_string.restype = ctypes.c_char_p
    L.hpd_last_launch_count.restype = ctypes.c_int
    P, S, B, V = ctypes.POINTER(HpdParams), ctypes.POINTER(HpdScaleInputs), ctypes.POINTER(HpdBuffers), ctypes.c_void_p
    L.hpd_workspace_bytes.argtypes = [P, ctypes.POINTER(ctypes.c_size_t)]
    L.hpd_aggregate_nms.argtypes = [P, S, B, V]
    L.hpd_aggregate_tags.argtypes = [P, S, V, V]
    L.hpd_nms.argtypes = [P, B, V, V]
    L.hpd_topk.argtypes = [P, B, V]
    L.hpd_group.argtypes = [P, B, V]
    L.hpd_adjust_refine.argtypes = [P, B, V, ctypes.c_size_t, V]
    L.hpd_decode.argtypes = [P, S, B, V, ctypes.c_size_t, V]
    SS = ctypes.POINTER(HpdStageInputs)
    L.hpd_aggregate_nms_stages.argtypes = [P, SS, B, V]
    L.hpd_decode_stages.argtypes = [P, SS, B, V, ctypes.c_size_t, V]
    L.hpd_resize_bilinear.argtypes = [ctypes.POINTER(HpdMap), ctypes.c_int, ctypes.c_int, V, ctypes.c_int,
                                      ctypes.c_int, V]
    I32P, F64P, F32P = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float)
    L.hpd_record_layout.argtypes = [P, ctypes.POINTER(HpdRecordLayout)]
    L.hpd_multi_scale_size.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, I32P,
                                       I32P, F64P]
    L.hpd_get_affine_transform.argtypes = [F64P, F64P, I32P, ctypes.c_int, F64P]
    L.hpd_prepare_geometry.argtypes = [ctypes.c_int, I32P, I32P, ctypes.c_int, ctypes.c_double, ctypes.c_double, I32P, I32P, F64P,
                                       F64P, F64P]
    L.hpd_prepare_input.argtypes = [ctypes.POINTER(HpdImage), ctypes.c_int, V, ctypes.c_int, ctypes.c_int, F32P, F32P, V]
    L.hpd_prepare_inputs.argtypes = [ctypes.POINTER(HpdImage), ctypes.c_int, ctypes.POINTER(HpdPrepareTarget), ctypes.c_int,
                                     F32P, F32P, V]
    CP = ctypes.POINTER(HpdCocoEvalParams)
    L.hpd_coco_eval_workspace_bytes.argtypes = [CP, ctypes.POINTER(ctypes.c_size_t)]
    L.hpd_coco_eval.argtypes = [CP, ctypes.POINTER(HpdCocoDets), ctypes.POINTER(HpdCocoGts),
                                ctypes.POINTER(HpdCocoEvalOutputs), V, ctypes.c_size_t, V]
    TP = ctypes.POINTER(HpdTrackParams)
    L.hpd_track_state_bytes.argtypes = [TP, ctypes.POINTER(ctypes.c_size_t)]
    L.hpd_track_reset.argtypes = [TP, V, ctypes.c_size_t, ctypes.c_int, V]
    L.hpd_track.argtypes = [TP, V, ctypes.c_int, V, ctypes.c_size_t, V, V]
    L.hpd_track_smooth_state_bytes.argtypes = [TP, ctypes.POINTER(ctypes.c_size_t)]
    L.hpd_track_smooth.argtypes = [TP, ctypes.POINTER(HpdSmoothParams), V, ctypes.c_int, V, ctypes.c_size_t, V, V, V]
    L.hpd_render_poses.argtypes = [ctypes.POINTER(HpdRenderParams), ctypes.POINTER(HpdRenderFrame), ctypes.c_int, V, V, V,
                                   V]
    for n in EXPORTS:
        if n not in ("hpd_last_error_string",):
            getattr(L, n).restype = ctypes.c_int
    if L.hpd_abi_version() != HPD_ABI_VERSION:
        raise HpdError(f"libhpdecode ABI {L.hpd_abi_version()} != binding {HPD_ABI_VERSION}")
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise HpdError(f"{what} failed (code {rc}): {lib().hpd_last_error_string().decode()}")
