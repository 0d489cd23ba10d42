"""COCO keypoint evaluation on the device (hpd_coco_eval) against the NumPy restatement of pycocotools
(oracle/coco_eval_oracle.py).

OKS values agree within a few ulp (the oracle's np.exp and CUDA's exp differ in the last bits); every later step is
compared exactly, on seeded scenes whose OKS values all sit at least 1e-9 from every decision (asserted).  Outputs are
NaN-poisoned first, so every entry the device must write is checked."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

K14_SIGMAS = np.array([.79, .79, .72, .72, .62, .62, 1.07, 1.07, .87, .87, .89, .89, .26, .35]) / 10.0

# (seed, generator kwargs, sigmas, max_dets)
CASES = [(s, {}, None, 20) for s in range(8)] + [
    (8, dict(score_levels=10), None, 20),
    (9, dict(score_levels=4, num_images=40), None, 20),
    (10, dict(dets_per_image=60), None, 20),
    (11, dict(max_gts=40, crowd_frac=0.3), None, 20),
    (12, dict(no_kpt_frac=0.4, no_gt_frac=0.4, no_det_frac=0.4), None, 20),
    (13, dict(spread=0.3), None, 20),
    (14, dict(spread=3.0, score_levels=20), None, 20),
    (15, dict(num_kpts=14, score_levels=8), K14_SIGMAS, 20),
    (16, dict(num_kpts=14), K14_SIGMAS, 7),
    (17, dict(num_kpts=14, dets_per_image=5), K14_SIGMAS, 32),
    (18, {}, None, 5),
    (19, dict(score_levels=6), None, 1),
    (20, dict(num_images=3, max_gts=2, dets_per_image=3), None, 20),
    (21, dict(max_gts=200, dets_per_image=200, num_images=6), None, 32),
]


def _oracle(dataset, results, sigmas, max_dets):
    from oracle import coco_eval_oracle as O
    ev = O.COCOevalKeypoints(dataset, results, sigmas=sigmas, max_dets=max_dets).run()
    assert ev.oks_margin() >= 1e-9, "scene has an OKS too close to a decision for an exact comparison"
    return ev


def _assert_oks_close(dev_oks, ev, img_ids):
    """[I, max_dets, G] device OKS within 4 ulp of the oracle's, zeros outside each image's matrix."""
    for i, img in enumerate(img_ids):
        m = ev.oks_matrix(img)
        ref = np.asarray(m, np.float64) if len(m) else np.zeros((0, 0))
        nd, ng = ref.shape
        got = dev_oks[i]
        if ref.size:
            tol = 4 * np.spacing(np.abs(ref))
            assert np.all(np.abs(got[:nd, :ng] - ref) <= tol), f"OKS of image {img}"
        mask = np.ones(got.shape, bool)
        mask[:nd, :ng] = False
        assert np.all(got[mask] == 0), f"OKS padding of image {img}"


def _assert_same(res, ev):
    np.testing.assert_array_equal(res.precision, ev.eval['precision'])
    np.testing.assert_array_equal(res.recall, ev.eval['recall'])
    np.testing.assert_array_equal(res.scores, ev.eval['scores'])
    np.testing.assert_array_equal(res.stats, ev.stats)
    assert res.summary() == ev.summary_lines


@pytest.mark.parametrize("seed,kw,sigmas,max_dets", CASES)
def test_device_matches_oracle(seed, kw, sigmas, max_dets):
    from hpdecode import KeypointEvaluator, KeypointGroundTruth, ops, synth
    kw = dict(kw)
    n = kw.pop("num_images", 24)
    dataset, results = synth.coco_eval_set(n, seed=seed, sigmas=sigmas, **kw)
    ev = _oracle(dataset, results, sigmas, max_dets)
    gt = KeypointGroundTruth.from_coco(dataset, "cuda:0")
    E = KeypointEvaluator(gt, sigmas=ev.params.kpt_oks_sigmas, max_dets=max_dets)
    p = E.params()
    I, G, T, R, A = p.num_images, p.max_gts, p.num_iou_thrs, p.num_rec_thrs, p.num_areas
    nan = dict(device="cuda:0", dtype=torch.float64)
    outs = [torch.full((T, R, A), np.nan, **nan), torch.full((T, A), np.nan, **nan), torch.full((T, R, A), np.nan, **nan),
            torch.full((I, max_dets, G), np.nan, **nan),
            torch.full((A, T, I, max_dets), 255, device="cuda:0", dtype=torch.uint8),
            torch.full((A,), -7, device="cuda:0", dtype=torch.int64)]
    records, rows, off_coco, off_count, stride, D = E.results_view(results)
    ops.run_coco_eval(p, records, rows, off_coco, off_count, stride, D, E.gt_tensors(), outs)
    prec, rec, sc, oks, codes, npig = [t.cpu().numpy() for t in outs]
    _assert_oks_close(oks, ev, gt.image_ids)
    np.testing.assert_array_equal(codes, ev.codes())
    np.testing.assert_array_equal(npig, ev.npig())
    np.testing.assert_array_equal(prec, ev.eval['precision'][:, :, 0, :, 0])
    np.testing.assert_array_equal(rec, ev.eval['recall'][:, 0, :, 0])
    np.testing.assert_array_equal(sc, ev.eval['scores'][:, :, 0, :, 0])
    _assert_same(E.evaluate_results(results), ev)


def test_gt_subset_and_foreign_results():
    """p.imgIds narrower than the dataset: results of the other images are dropped, results of unknown images and
    duplicated record rows are errors."""
    from hpdecode import KeypointEvaluator, KeypointGroundTruth, _lib, ops, synth
    from oracle import coco_eval_oracle as O
    dataset, results = synth.coco_eval_set(30, seed=5)
    ids = sorted(img['id'] for img in dataset['images'])[::2]
    ev = O.COCOevalKeypoints(dataset, results, img_ids=ids).run()
    assert ev.oks_margin() >= 1e-9
    E = KeypointEvaluator(KeypointGroundTruth.from_coco(dataset, "cuda:0", image_ids=ids[::-1]))
    _assert_same(E.evaluate_results(results), ev)
    with pytest.raises(_lib.HpdError, match="not in the ground truth"):
        E.evaluate_results(results + [dict(results[0], image_id=10 ** 9)])
    rec = torch.zeros((2, ops.record_layout(17, 30, 2).row_bytes), device="cuda:0", dtype=torch.uint8)
    with pytest.raises(_lib.HpdError, match="two places"):
        E.evaluate_records([(rec, [ids[0], ids[0]])], 30, 17, 2)
    with pytest.raises(_lib.HpdError, match="records must be"):
        E.evaluate_records([(rec[:, :1024], [ids[0]])], 30, 17, 2)


def test_records_path_equals_dict_path_end_to_end():
    """Two decoded crowd batches with a non-trivial inv_affine; gts from the oracle's decode of the same inputs,
    jittered, with persons dropped and extras added.  Records of both batches (rows shuffled, batches reversed) read
    in place == the result dicts (batch_to_coco) == the oracle on those dicts."""
    from hpdecode import BottomUpDecoder, KeypointEvaluator, KeypointGroundTruth, batch_to_coco, geometry, synth
    from oracle import cpu_oracle, input_oracle
    cpu_oracle.build()
    size, B, M, K = 192, 3, 30, 17
    dec = BottomUpDecoder(K, M, 0.05, 0.5, "cuda:0")
    center, scale = (150, 100), (300.0, 200.0)
    minv = geometry.get_affine_transform(center, scale, 0, (size, size), inverse=True)
    inv = np.stack([minv.ravel()] * B)
    batches, images, anns = [], [], []
    rnd = synth._Draws(99)
    for bi, seed in enumerate((21, 22)):
        scales = synth.crowd(B, size, persons=6 + 2 * bi, flip=True, seed=seed)
        dev = [{k: torch.from_numpy(v).cuda() for k, v in s.items()} for s in scales]
        res = dec.decode(dev, (size, size), inv_affine=inv, slot=bi)
        ids = [100 + 10 * b + bi for b in range(B)]
        batches.append((res.packed().clone(), ids, res.host()))
        for b, img in enumerate(ids):
            images.append({"id": img})
            hm, tags = cpu_oracle.aggregate(synth.image_slice(scales, b), (size, size))
            ref = cpu_oracle.parse(hm, tags, M, 0.05, 0.5)
            xy = input_oracle.affine_points(ref["grouped_joints"][..., :2].reshape(-1, 2), minv).reshape(-1, K, 2)
            persons = [xy[p].astype(np.float64) for p in range(len(xy)) if p % 4 != 1]          # drop some
            persons += [np.array([[40 + 200 * rnd.one(), 30 + 150 * rnd.one()] for _ in range(K)])]  # an extra
            for p in persons:
                j = p + (rnd.take(2 * K).reshape(K, 2) - 0.5) * 6.0
                x0, y0 = j.min(0)
                w, h = j.max(0) - j.min(0)
                kp = np.concatenate([j, np.full((K, 1), 2.0)], 1).ravel()
                anns.append({"id": len(anns) + 1, "image_id": img, "category_id": 1, "keypoints": kp.tolist(),
                             "num_keypoints": K, "area": float(w * h * 0.5), "bbox": [x0, y0, w, h], "iscrowd": 0})
    images.append({"id": 999})            # an image no batch holds
    dataset = {"images": images, "annotations": anns}
    results = [r for rec, ids, host in batches for r in batch_to_coco(ids, host)]
    ev = _oracle(dataset, results, None, 20)
    E = KeypointEvaluator(KeypointGroundTruth.from_coco(dataset, "cuda:0"))
    by_dicts = E.evaluate_results(results)
    _assert_same(by_dicts, ev)
    perm = [2, 0, 1]
    shuffled = [(rec[perm], [ids[p] for p in perm]) for rec, ids, _ in batches[::-1]]
    by_records = E.evaluate_records(shuffled, M, K, 2)
    _assert_same(by_records, ev)
    in_place = E.evaluate_records([(rec, ids) for rec, ids, _ in batches], M, K, 2)
    _assert_same(in_place, ev)
    assert ev.stats[0] > 0.05, "the scene should match some persons"


def test_fake_impl_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    import hpdecode  # noqa: F401
    with FakeTensorMode():
        I, G, K = 5, 3, 17
        f = lambda *s, dt=torch.float64: torch.empty(s, dtype=dt, device="cuda:0")
        args = ([f(2, 64, dt=torch.uint8)], torch.full((I,), -1, dtype=torch.int64), 0, 8, 52, 4, f(I, G, K, 3),
                f(I, G), f(I, G, 4), f(I, G, dt=torch.uint8), f(I, G, dt=torch.uint8), f(I, dt=torch.int32),
                [0.5] * 10, [0.0] * 101, [0.0, 1.0] * 3, [0.01] * K, 20)
        out = torch.ops.hpd.coco_eval(*args, True)
        assert [tuple(t.shape) for t in out] == [(10, 101, 3), (10, 3), (10, 101, 3), (I, 20, G), (3, 10, I, 20), (3,)]
        assert out[4].dtype == torch.uint8 and out[5].dtype == torch.int64
        out = torch.ops.hpd.coco_eval(*args, False)
        assert [tuple(t.shape) for t in out[:3]] == [(10, 101, 3), (10, 3), (10, 101, 3)]
