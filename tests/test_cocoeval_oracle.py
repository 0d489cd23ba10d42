"""CPU suite for the COCO keypoint evaluation: known answers of the pycocotools restatement
(oracle/coco_eval_oracle.py), the oracle against the real pycocotools when it is importable, the C layout of the new
ABI structs, and argument validation before any launch."""
import copy
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import coco_eval_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 17


def _gt(img, ann_id, xy, area, vis=2.0, iscrowd=0, bbox=None):
    xy = np.asarray(xy, np.float64).reshape(K, 2)
    v = np.full(K, vis)
    if bbox is None:
        x0, y0 = xy.min(0)
        w, h = xy.max(0) - xy.min(0)
        bbox = [x0, y0, w, h]
    return {"id": ann_id, "image_id": img, "category_id": 1, "keypoints": np.column_stack([xy, v]).ravel().tolist(),
            "num_keypoints": int(np.count_nonzero(v > 0)), "area": float(area), "bbox": list(bbox), "iscrowd": iscrowd}


def _dt(img, xy, score):
    xy = np.asarray(xy, np.float64).reshape(K, 2)
    return {"image_id": img, "category_id": 1, "keypoints": np.column_stack([xy, np.ones(K)]).ravel().tolist(),
            "score": score}


def _person(cx, cy, s):
    k = np.arange(K)
    return np.column_stack([cx + s * np.cos(k), cy + s * np.sin(k)])


def _run(images, anns, results, **kw):
    return O.COCOevalKeypoints({"images": [{"id": i} for i in images], "annotations": anns}, results, **kw).run()


def test_perfect_detections_give_ap_and_ar_one():
    p = [_person(100 + 50 * i, 200, 60) for i in range(3)]
    anns = [_gt(1, 1, p[0], 150 ** 2), _gt(1, 2, p[1], 150 ** 2), _gt(2, 3, p[2], 150 ** 2)]
    res = [_dt(1, p[0], 0.9), _dt(1, p[1], 0.8), _dt(2, p[2], 0.7)]
    ev = _run([1, 2], anns, res)
    assert ev.stats[0] == 1.0 and ev.stats[5] == 1.0 and ev.stats[4] == 1.0
    assert ev.stats[3] == -1 and ev.stats[8] == -1           # no medium gt: npig == 0 leaves -1
    assert np.all(ev.codes()[0, :, :, :2][:, 0] == O.TP)


def test_one_pair_closed_form_oks():
    g = _person(300, 300, 40)
    vis = np.zeros(K)
    vis[[0, 5, 11]] = 2
    ann = _gt(1, 1, g, 5000.0)
    ann["keypoints"] = np.column_stack([g, vis]).ravel().tolist()
    ann["num_keypoints"] = 3
    d = g + np.array([3.0, -4.0])
    ev = _run([1], [ann], [_dt(1, d, 0.5)])
    var = (O.KPT_OKS_SIGMAS * 2) ** 2
    e = 25.0 / var[[0, 5, 11]] / (5000.0 + np.spacing(1)) / 2
    assert ev.oks_matrix(1)[0, 0] == (np.exp(-e[0]) + np.exp(-e[1]) + np.exp(-e[2])) / 3


def test_crowd_gt_absorbs_detections_which_are_ignored():
    p, q = _person(100, 100, 60), _person(400, 300, 60)
    anns = [_gt(1, 1, p, 150 ** 2), _gt(1, 2, q, 150 ** 2, iscrowd=1)]
    res = [_dt(1, p, 0.9)] + [_dt(1, q + 0.5 * j, 0.8 - 0.1 * j) for j in range(3)]
    ev = _run([1], anns, res)
    codes = ev.codes()[0, 0, 0, :4]
    assert list(codes) == [O.TP, O.IGNORED, O.IGNORED, O.IGNORED]
    assert ev.npig()[0] == 1 and ev.stats[0] == 1.0 / (1.0 + 2.0 ** -52)   # one tp: fp + tp + eps


def test_gt_without_labelled_joints_is_ignored():
    p, q = _person(100, 100, 60), _person(400, 300, 60)
    anns = [_gt(1, 1, p, 150 ** 2), _gt(1, 2, q, 150 ** 2, vis=0.0, bbox=[340, 240, 120, 120])]
    assert anns[1]["num_keypoints"] == 0
    ev = _run([1], anns, [_dt(1, p, 0.9)])
    assert ev.npig()[0] == 1 and ev.stats[5] == 1.0


def test_area_bands_classify_gts_and_detections():
    small, medium, large = _person(50, 50, 5), _person(200, 200, 20), _person(400, 400, 60)
    anns = [_gt(1, 1, small, 20 ** 2), _gt(1, 2, medium, 50 ** 2), _gt(1, 3, large, 150 ** 2)]
    far = _person(600, 50, 80)                                   # an unmatched detection with a large area
    res = [_dt(1, large, 0.9), _dt(1, medium, 0.8), _dt(1, small, 0.7), _dt(1, far, 0.6)]
    ev = _run([1], anns, res)
    assert list(ev.npig()) == [3, 1, 1]
    codes = ev.codes()[:, 0, 0, :4]                              # [area][rank] at threshold 0.5
    assert list(codes[0]) == [O.TP, O.TP, O.TP, O.FP]
    assert list(codes[1]) == [O.IGNORED, O.TP, O.IGNORED, O.IGNORED]   # medium: the large / far ones are out of range
    assert list(codes[2]) == [O.TP, O.IGNORED, O.IGNORED, O.FP]


def test_max_dets_cut_keeps_the_best_scored():
    p = _person(200, 200, 60)
    fp = [_dt(1, _person(600, 600, 10) + j, 0.5 + 0.01 * j) for j in range(19)]
    res = fp[:10] + [_dt(1, p, 0.3)] + fp[10:] + [_dt(1, _person(50, 600, 10) + j, 0.1) for j in range(6)]
    ev = _run([1], [_gt(1, 1, p, 150 ** 2)], res, max_dets=20)
    e = ev.evalImgs[0]
    assert len(e['dtIds']) == 20 and min(e['dtScores']) == 0.3      # the six 0.1 ones are cut
    ev5 = _run([1], [_gt(1, 1, p, 150 ** 2)], res, max_dets=5)
    assert ev5.stats[5] == 0.0 and ev.stats[5] == 1.0


def test_cross_image_score_tie_order_changes_ap():
    p, q = _person(200, 200, 60), _person(500, 200, 60)

    def scene(tp_image, fp_image):
        anns = [_gt(tp_image, 1, p, 150 ** 2), _gt(fp_image, 2, q, 150 ** 2)]
        return _run([tp_image, fp_image], anns, [_dt(tp_image, p, 0.5), _dt(fp_image, _person(50, 50, 10), 0.5)])

    first, second = scene(1, 2), scene(2, 1)     # the tp's image comes first / second in p.imgIds order
    assert first.eval['precision'][0, 0, 0, 0, 0] == 1.0 / (1.0 + np.spacing(1))
    assert second.eval['precision'][0, 0, 0, 0, 0] == 0.5
    assert first.stats[0] != second.stats[0]


def test_fp_plus_tp_equal_one_keeps_the_spacing():
    p = _person(200, 200, 60)
    ev = _run([1], [_gt(1, 1, p, 150 ** 2)], [_dt(1, p, 0.9)])
    v = ev.eval['precision'][0, 0, 0, 0, 0]
    assert v == 1.0 / (1.0 + 2.0 ** -52) and v < 1.0


def test_unreachable_recall_leaves_the_tail_zero():
    p, q = _person(200, 200, 60), _person(500, 200, 60)
    ev = _run([1], [_gt(1, 1, p, 150 ** 2), _gt(1, 2, q, 150 ** 2)], [_dt(1, p, 0.9)])
    prec, sc = ev.eval['precision'][0, :, 0, 0, 0], ev.eval['scores'][0, :, 0, 0, 0]
    assert ev.eval['recall'][0, 0, 0, 0] == 0.5
    assert np.all(prec[:51] > 0) and np.all(prec[51:] == 0) and np.all(sc[51:] == 0) and np.all(sc[:51] == 0.9)


def test_oracle_matches_pycocotools():
    pytest.importorskip("pycocotools")
    from pycocotools.coco import COCO
    from pycocotools.cocoeval import COCOeval
    from hpdecode import synth
    for seed, kw in ((0, {}), (1, dict(score_levels=5)), (2, dict(max_gts=30, crowd_frac=0.3, no_kpt_frac=0.3))):
        dataset, results = synth.coco_eval_set(40, seed=seed, **kw)
        gt = COCO()
        gt.dataset = copy.deepcopy(dataset)
        gt.createIndex()
        ce = COCOeval(gt, gt.loadRes(copy.deepcopy(results)), "keypoints")
        ce.evaluate()
        ce.accumulate()
        ce.summarize()
        ev = O.COCOevalKeypoints(dataset, results).run()
        for name in ("precision", "recall", "scores"):
            np.testing.assert_array_equal(ce.eval[name], ev.eval[name])
        np.testing.assert_array_equal(ce.stats, ev.stats)


def test_generator_covers_the_edges():
    from hpdecode import synth
    dataset, results = synth.coco_eval_set(60, seed=3, score_levels=10)
    anns = dataset["annotations"]
    assert any(a["iscrowd"] for a in anns) and any(a["num_keypoints"] == 0 for a in anns)
    areas = np.array([a["area"] for a in anns])
    assert (areas < 32 ** 2).any() and ((areas > 32 ** 2) & (areas < 96 ** 2)).any() and (areas > 96 ** 2).any()
    ids = {img["id"] for img in dataset["images"]}
    with_gt, with_dt = {a["image_id"] for a in anns}, {r["image_id"] for r in results}
    assert ids - with_gt and ids - with_dt
    per = {}
    for r in results:
        per.setdefault(r["image_id"], []).append(r["score"])
    assert max(len(v) for v in per.values()) > 20
    assert any(len(set(v)) < len(v) for v in per.values())
    assert synth.coco_eval_set(60, seed=3, score_levels=10) == (dataset, results)
    ev = O.COCOevalKeypoints(dataset, results).run()
    assert ev.oks_margin() >= 1e-9 and 0 < ev.stats[0] < 1


def test_coco_eval_structs_match_c_layout(tmp_path):
    from hpdecode import _lib
    probe = tmp_path / "probe.c"
    fields = ("sizeof(HpdCocoEvalParams)", "offsetof(HpdCocoEvalParams,iou_thrs)", "offsetof(HpdCocoEvalParams,rec_thrs)",
              "offsetof(HpdCocoEvalParams,area_rng)", "offsetof(HpdCocoEvalParams,kpt_vars)", "sizeof(HpdCocoDets)",
              "offsetof(HpdCocoDets,person_stride)", "sizeof(HpdCocoGts)", "sizeof(HpdCocoEvalOutputs)",
              "offsetof(HpdCocoEvalOutputs,npig)")
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "hpdecode.h"\nint main(){printf("'
                     + " ".join(["%zu"] * len(fields)) + '\\n",' + ",".join(fields) + ");return 0;}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    P, D, G, Ou = _lib.HpdCocoEvalParams, _lib.HpdCocoDets, _lib.HpdCocoGts, _lib.HpdCocoEvalOutputs
    want = [ctypes.sizeof(P), P.iou_thrs.offset, P.rec_thrs.offset, P.area_rng.offset, P.kpt_vars.offset,
            ctypes.sizeof(D), D.person_stride.offset, ctypes.sizeof(G), ctypes.sizeof(Ou), Ou.npig.offset]
    assert got == want


def test_coco_eval_validates_before_any_launch():
    from hpdecode import _lib, ops
    from hpdecode.cocoeval import IOU_THRS, REC_THRS
    L = _lib.lib()
    area = [0.0, 1e10, 1024.0, 9216.0, 9216.0, 1e10]
    good = dict(num_images=4, num_kpts=17, max_dets=20, max_gts=8)

    def params(**over):
        a = dict(good, **over)
        return ops.coco_eval_params(a["num_images"], a["num_kpts"], a["max_dets"], a["max_gts"], IOU_THRS.tolist(),
                                    REC_THRS.tolist(), area, [0.01] * a["num_kpts"])

    n = ctypes.c_size_t(0)
    for over, msg in ((dict(max_dets=33), b"max_dets"), (dict(max_gts=1025), b"max_gts"), (dict(num_kpts=33), None),
                      (dict(num_images=0), b"num_images"), (dict(max_dets=0), b"max_dets")):
        if msg is None:
            with pytest.raises(_lib.HpdError):
                params(**over)
            continue
        p = params(**over)
        assert L.hpd_coco_eval_workspace_bytes(ctypes.byref(p), ctypes.byref(n)) == 1
        assert msg in L.hpd_last_error_string()
        assert L.hpd_coco_eval(ctypes.byref(p), None, None, None, None, 0, None) == 1
    p = params()
    p.num_iou_thrs = 17
    assert L.hpd_coco_eval(ctypes.byref(p), None, None, None, None, 0, None) == 1
    assert b"num_iou_thrs" in L.hpd_last_error_string()
    p = params()
    p.num_rec_thrs = 129
    assert L.hpd_coco_eval(ctypes.byref(p), None, None, None, None, 0, None) == 1
    assert b"num_rec_thrs" in L.hpd_last_error_string()
    p = params()
    d, g, o = _lib.HpdCocoDets(), _lib.HpdCocoGts(), _lib.HpdCocoEvalOutputs()
    assert L.hpd_coco_eval(ctypes.byref(p), ctypes.byref(d), ctypes.byref(g), ctypes.byref(o), None, 0, None) == 1
    d.base, d.row_offset, d.person_stride, d.max_per_row = 8, 8, 3 * 17, 30
    assert L.hpd_coco_eval(ctypes.byref(p), ctypes.byref(d), ctypes.byref(g), ctypes.byref(o), None, 0, None) == 1
    assert b"person_stride" in L.hpd_last_error_string()
    d.person_stride, d.max_per_row = 3 * 17 + 1, 1025
    assert L.hpd_coco_eval(ctypes.byref(p), ctypes.byref(d), ctypes.byref(g), ctypes.byref(o), None, 0, None) == 1
    assert b"max_per_row" in L.hpd_last_error_string()
    with pytest.raises(_lib.HpdError):
        ops.coco_eval_params(4, 17, 20, 8, [0.5] * 17, REC_THRS.tolist(), area, [0.01] * 17)
