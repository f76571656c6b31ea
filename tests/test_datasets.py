"""Detection consumers on the far side of test_net (SURVEY.md 8(f) rank 3): VOC / COCO image databases, result
files and scoring.  voc_eval is pinned to vectors produced by the reference's own voc_eval
(tests/golden/make_voc_golden.py); the COCO bbox scorer has hand-computed cases only (pycocotools absent: unpinned)."""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from tf_faster_rcnn_b200 import paths  # noqa: E402
paths.add_lib_path()
import voc_fixture  # noqa: E402
from model.config import cfg  # noqa: E402
from datasets import voc_eval as ve  # noqa: E402
from datasets.factory import get_imdb, list_imdbs  # noqa: E402

G = np.load(os.path.join(HERE, "golden", "voc_eval_vectors.npz"))


@pytest.fixture()
def data_dir(tmp_path):
    old = cfg.DATA_DIR
    cfg.DATA_DIR = str(tmp_path / "data")
    os.makedirs(cfg.DATA_DIR)
    yield cfg.DATA_DIR
    cfg.DATA_DIR = old


def test_voc_eval_matches_reference_vectors(tmp_path):
    root = str(tmp_path)
    ids, dets = voc_fixture.build(root)
    detpath = voc_fixture.write_det_files(os.path.join(root, "dets"), dets)
    annopath = os.path.join(root, "VOC2007", "Annotations", "{:s}.xml")
    imageset = os.path.join(root, "VOC2007", "ImageSets", "Main", "test.txt")
    got = np.array([[o["truncated"], o["difficult"]] + o["bbox"] for o in ve.parse_rec(annopath.format(ids[0]))]).reshape(-1, 6)
    assert np.array_equal(got, G["parse_000001"])
    for cls in ("car", "person", "dog"):
        for m07 in (False, True):
            for diff in (False, True):
                rec, prec, ap = ve.voc_eval(detpath, annopath, imageset, cls, os.path.join(root, "cache"), ovthresh=0.5,
                                            use_07_metric=m07, use_diff=diff)
                tag = "%s_%d_%d" % (cls, m07, diff)
                assert np.array_equal(rec, G["rec_" + tag]), tag
                assert np.array_equal(prec, G["prec_" + tag]), tag
                assert abs(ap - float(G["ap_" + tag])) < 1e-15, tag
    assert os.path.isfile(imageset + "_annots.pkl")          # cache lands where the reference puts it


def test_voc_ap_hand_cases():
    rec = np.array([0.5, 0.5, 1.0])
    prec = np.array([1.0, 0.5, 2.0 / 3])
    assert abs(ve.voc_ap(rec, prec) - (0.5 * 1.0 + 0.5 * 2.0 / 3)) < 1e-12
    assert abs(ve.voc_ap(rec, prec, use_07_metric=True) - (6 * 1.0 + 5 * 2.0 / 3) / 11) < 1e-12
    assert ve.voc_ap(np.array([]), np.array([])) == 0.0


def test_pascal_voc_imdb_end_to_end(tmp_path, data_dir, capsys):
    devkit = os.path.join(data_dir, "VOCdevkit2007")
    ids, dets = voc_fixture.build(devkit, with_images=True)
    imdb = get_imdb("voc_2007_test")
    assert imdb.name == "voc_2007_test" and imdb.num_classes == 21 and imdb.classes[15] == "person"
    assert imdb.image_index == ids and imdb.num_images == len(ids)
    assert imdb.image_path_at(2) == os.path.join(devkit, "VOC2007", "JPEGImages", ids[2] + ".jpg")
    roidb = imdb.roidb
    recs = [ve.parse_rec(os.path.join(devkit, "VOC2007", "Annotations", i + ".xml")) for i in ids]
    for entry, objs in zip(roidb, recs):
        keep = [o for o in objs if not o["difficult"]]
        assert entry["boxes"].dtype == np.uint16 and entry["boxes"].shape == (len(keep), 4)
        assert np.array_equal(entry["boxes"], np.array([o["bbox"] for o in keep], dtype=np.int64).reshape(-1, 4) - 1)
        assert [imdb.classes[c] for c in entry["gt_classes"]] == [o["name"] for o in keep]
        assert entry["gt_overlaps"].shape == (len(keep), 21) and entry["flipped"] is False
    assert len(get_imdb("voc_2007_test_diff").gt_roidb()[0]["boxes"]) == len(recs[0])      # *_diff keeps difficult objects
    assert os.path.isfile(os.path.join(data_dir, "cache", "voc_2007_test_gt_roidb.pkl"))

    # all_boxes as test_net builds it (0-based), from the fixture's devkit-coordinate rows
    all_boxes = [[np.zeros((0, 5), np.float32) for _ in ids] for _ in imdb.classes]
    for c, cls in enumerate(imdb.classes):
        for row in dets.get(cls, []):
            i = ids.index(row[0])
            all_boxes[c][i] = np.vstack([all_boxes[c][i], np.array([[row[2] - 1, row[3] - 1, row[4] - 1, row[5] - 1, row[1]]], np.float32)])
    imdb.competition_mode(True)
    out_dir = str(tmp_path / "out")
    aps = imdb.evaluate_detections(all_boxes, out_dir)
    results = os.path.join(devkit, "results", "VOC2007", "Main")
    assert sorted(os.listdir(results))[0] == "comp4_det_test_aeroplane.txt" and len(os.listdir(results)) == 20
    with open(os.path.join(results, "comp4_det_test_car.txt")) as f:
        first = f.readline().split()
    assert first[0] in ids and len(first) == 6 and len(first[1].split(".")[1]) == 3 and len(first[2].split(".")[1]) == 1
    assert len(aps) == 20 and os.path.isfile(os.path.join(out_dir, "car_pr.pkl"))
    # float32 round trip of the fixture rows can move a %.1f digit; AP of the file-based golden run is reproduced closely
    assert abs(aps[imdb.classes.index("person") - 1] - float(G["ap_person_1_0"])) < 0.05
    assert "Mean AP" in capsys.readouterr().out
    imdb.competition_mode(False)
    imdb.evaluate_detections(all_boxes, out_dir)
    assert [f for f in os.listdir(results) if not f.startswith("comp4_det_")] == []      # salted files were cleaned up
    with pytest.raises(AssertionError):
        get_imdb("voc_2012_val")
    assert {"voc_2007_trainval", "voc_2012_test_diff", "coco_2014_minival", "coco_2015_test-dev"} <= set(list_imdbs())


# ---- COCO -----------------------------------------------------------------------------------------------------------
def _coco_tree(data_dir, images, anns, cats=((1, "person"), (3, "car"))):
    base = os.path.join(data_dir, "coco")
    os.makedirs(os.path.join(base, "annotations"), exist_ok=True)
    os.makedirs(os.path.join(base, "images", "val2014"), exist_ok=True)
    doc = {"images": [{"id": i, "width": w, "height": h, "file_name": "COCO_val2014_%012d.jpg" % i} for i, w, h in images],
           "categories": [{"id": c, "name": n, "supercategory": "x"} for c, n in cats],
           "annotations": [dict(a, id=k + 1) for k, a in enumerate(anns)]}
    for name in ("instances_val2014.json", "instances_minival2014.json"):
        with open(os.path.join(base, "annotations", name), "w") as f:
            json.dump(doc, f)
    for i, _, _ in images:
        open(os.path.join(base, "images", "val2014", "COCO_val2014_%012d.jpg" % i), "wb").close()


def _ann(img, cat, box, crowd=0, area=None):
    return {"image_id": img, "category_id": cat, "bbox": list(box), "iscrowd": crowd,
            "area": float(box[2] * box[3] if area is None else area)}


def test_coco_imdb_roidb_and_results(data_dir, tmp_path):
    _coco_tree(data_dir, [(42, 100, 80), (7, 64, 64)],
               [_ann(42, 3, (10, 20, 30, 40)), _ann(42, 1, (90, 70, 30, 30)), _ann(42, 1, (5, 5, 10, 10), crowd=1),
                _ann(7, 1, (1, 1, 5, 5), area=0)])
    imdb = get_imdb("coco_2014_minival")
    assert imdb.classes == ("__background__", "person", "car") and imdb.image_index == [42, 7]
    assert imdb.image_path_at(0).endswith("images/val2014/COCO_val2014_000000000042.jpg")     # minival is a view of val2014
    r0, r1 = imdb.roidb
    assert r0["boxes"].tolist() == [[10, 20, 39, 59], [90, 70, 99, 79], [5, 5, 14, 14]]       # clipped to W-1/H-1
    assert r0["gt_classes"].tolist() == [2, 1, 1] and (r0["width"], r0["height"]) == (100, 80)
    ov = r0["gt_overlaps"].toarray()
    assert ov[0].tolist() == [0, 0, 1] and ov[2].tolist() == [-1, -1, -1]                     # crowd row
    assert len(r1["boxes"]) == 0                                                               # zero-area annotation dropped
    all_boxes = [[np.zeros((0, 5), np.float32)] * 2 for _ in range(3)]
    all_boxes[2][0] = np.array([[10, 20, 39, 59, 0.9]], np.float32)
    res = imdb._write_coco_results_file(all_boxes, str(tmp_path / "r.json"))
    assert res == [{"image_id": 42, "category_id": 3, "bbox": [10.0, 20.0, 30.0, 40.0], "score": pytest.approx(0.9)}]


def _eval(gt_anns, dts, cats=(1,), imgs=(1,)):
    from datasets.coco_eval import BboxEval
    gt = {}
    for a in gt_anns:
        gt.setdefault(a["image_id"], []).append(a)
    return BboxEval(gt, dts, cats, imgs).evaluate()


def _dt(img, cat, box, score):
    return {"image_id": img, "category_id": cat, "bbox": list(box), "score": score}


def test_coco_bbox_eval_hand_cases():
    from datasets.coco_eval import box_iou
    assert box_iou([[0, 0, 10, 10]], [[5, 0, 10, 10], [0, 0, 20, 20]], [0, 1]).tolist() == [[50 / 150, 1.0]]
    # A: two medium ground truths, both found exactly -> AP 1, AR@1 0.5
    gts = [_ann(1, 1, (10, 10, 50, 50)), _ann(1, 1, (100, 100, 40, 60))]
    ev = _eval(gts, [_dt(1, 1, (10, 10, 50, 50), 0.9), _dt(1, 1, (100, 100, 40, 60), 0.8)])
    s = ev.summarize(verbose=False)
    assert s[0] == pytest.approx(1.0) and s[1] == pytest.approx(1.0) and s[4] == pytest.approx(1.0) and s[3] == -1.0 and s[5] == -1.0
    assert s[6] == pytest.approx(0.5) and s[7] == pytest.approx(1.0) and s[8] == pytest.approx(1.0)
    # B: a higher-scoring miss in front of the hit -> precision 0.5 at every recall point, every threshold
    ev = _eval(gts[:1], [_dt(1, 1, (200, 200, 50, 50), 0.9), _dt(1, 1, (10, 10, 50, 50), 0.8)])
    assert np.allclose(ev.precision[:, :, 0, 0, 2], 0.5) and ev.summarize(verbose=False)[0] == pytest.approx(0.5)
    # C: IoU 0.82 (41 of 50 rows) -> true positive at thresholds 0.50 .. 0.80 (7 of 10), missed above
    assert box_iou([[10, 10, 50, 41]], [[10, 10, 50, 50]], [0])[0, 0] == pytest.approx(0.82)
    ev = _eval(gts[:1], [_dt(1, 1, (10, 10, 50, 41), 0.9)])
    s = ev.summarize(verbose=False)
    assert s[0] == pytest.approx(0.7) and s[1] == pytest.approx(1.0) and s[2] == pytest.approx(1.0)
    # D: detections on a crowd region are ignored, not false positives; the crowd itself is not a positive
    ev = _eval([gts[0], _ann(1, 1, (200, 200, 100, 100), crowd=1)],
               [_dt(1, 1, (10, 10, 50, 50), 0.5), _dt(1, 1, (210, 210, 30, 30), 0.9), _dt(1, 1, (250, 250, 30, 30), 0.8)])
    assert ev.summarize(verbose=False)[0] == pytest.approx(1.0)
    # E: second detection of an already matched box is a false positive; a category without gt or dt stays -1
    ev = _eval(gts[:1], [_dt(1, 1, (10, 10, 50, 50), 0.9), _dt(1, 1, (11, 10, 50, 50), 0.8)], cats=(1, 2))
    assert np.all(ev.precision[:, :, 1] == -1) and ev.summarize(verbose=False)[0] == pytest.approx(1.0)
    ev = _eval(gts[:1], [_dt(1, 1, (11, 10, 50, 50), 0.9), _dt(1, 1, (10, 10, 50, 50), 0.8)])
    # IoU of the first = 49/51 = 0.961 >= every threshold: it takes the box, the exact one becomes the false positive
    assert ev.summarize(verbose=False)[0] == pytest.approx(1.0)
    # F: max detections: with only one detection allowed the lower-scoring true positive is cut
    ev = _eval(gts, [_dt(1, 1, (300, 300, 50, 50), 0.9), _dt(1, 1, (10, 10, 50, 50), 0.8)])
    assert ev.recall[0, 0, 0, 0] == 0.0 and ev.recall[0, 0, 0, 1] == 0.5
    # G: small object counted under 'small' and 'all' only
    ev = _eval([_ann(1, 1, (10, 10, 20, 20))], [_dt(1, 1, (10, 10, 20, 20), 0.9)])
    s = ev.summarize(verbose=False)
    assert s[0] == pytest.approx(1.0) and s[3] == pytest.approx(1.0) and s[4] == -1.0 and s[5] == -1.0


def test_coco_evaluate_detections_end_to_end(data_dir, tmp_path, capsys):
    _coco_tree(data_dir, [(1, 400, 400), (2, 400, 400)],
               [_ann(1, 1, (10, 10, 50, 50)), _ann(1, 3, (100, 100, 120, 120)), _ann(2, 1, (30, 30, 60, 60))])
    imdb = get_imdb("coco_2014_val")
    all_boxes = [[np.zeros((0, 5), np.float32)] * 2 for _ in range(3)]
    all_boxes[1][0] = np.array([[10, 10, 59, 59, 0.9]], np.float32)            # x2 = x1 + w - 1
    all_boxes[1][1] = np.array([[30, 30, 89, 89, 0.7], [300, 300, 350, 350, 0.2]], np.float32)
    all_boxes[2][0] = np.array([[100, 100, 219, 219, 0.8]], np.float32)
    out = str(tmp_path / "o")
    stats = imdb.evaluate_detections(all_boxes, out)
    assert stats[0] == pytest.approx(1.0) and os.path.isfile(os.path.join(out, "detection_results.pkl"))
    assert [f for f in os.listdir(out) if f.endswith(".json")] == []            # salted results json removed
    text = capsys.readouterr().out
    assert "Mean and per-category AP" in text and "Average Precision" in text
    imdb.competition_mode(True)
    imdb.evaluate_detections(all_boxes, out)
    assert os.path.isfile(os.path.join(out, "detections_val2014_results.json"))


def test_reval_tool_rescoring_from_detections_pkl(tmp_path):
    """tools/reval.py on a pickled all_boxes (what test_net leaves behind), as a subprocess like a user would run it."""
    import pickle
    import subprocess
    data = str(tmp_path / "data")
    devkit = os.path.join(data, "VOCdevkit2007")
    ids, dets = voc_fixture.build(devkit, with_images=True)
    all_boxes = [[np.zeros((0, 5), np.float32) for _ in ids] for _ in range(21)]
    from datasets.pascal_voc import VOC_CLASSES
    for c, cls in enumerate(VOC_CLASSES):
        for row in dets.get(cls, []):
            i = ids.index(row[0])
            all_boxes[c][i] = np.vstack([all_boxes[c][i], np.array([[row[2] - 1, row[3] - 1, row[4] - 1, row[5] - 1, row[1]]], np.float32)])
    out = str(tmp_path / "run")
    os.makedirs(out)
    with open(os.path.join(out, "detections.pkl"), "wb") as f:
        pickle.dump(all_boxes, f)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "reval.py"), out, "--imdb", "voc_2007_test", "--comp",
                        "--set", "DATA_DIR", data], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "Mean AP = " in r.stdout and "AP for person = " in r.stdout
    assert os.path.isfile(os.path.join(devkit, "results", "VOC2007", "Main", "comp4_det_test_dog.txt"))


def test_coco_bbox_eval_against_a_plain_loop_implementation():
    """Randomised cross-check of the vectorised scorer against a deliberately naive re-statement (python loops, one IoU
    threshold at a time, no crowds / area filters): same protocol, independent code."""
    from datasets.coco_eval import BboxEval, IOU_THRS, REC_THRS

    def iou(a, b):
        iw = min(a[0] + a[2], b[0] + b[2]) - max(a[0], b[0])
        ih = min(a[1] + a[3], b[1] + b[3]) - max(a[1], b[1])
        inter = max(iw, 0.0) * max(ih, 0.0)
        return inter / (a[2] * a[3] + b[2] * b[3] - inter)

    def naive_ap(gt, dt, imgs, thr):
        rows, npos = [], 0                                     # (score, is_tp) over all images
        for img in imgs:
            g = [a["bbox"] for a in gt.get(img, [])]
            d = sorted([x for x in dt if x["image_id"] == img], key=lambda x: -x["score"])[:100]
            npos += len(g)
            taken = [False] * len(g)
            for x in d:
                best, m = min(thr, 1 - 1e-10), -1
                for j, gb in enumerate(g):
                    if taken[j]:
                        continue
                    v = iou(x["bbox"], gb)
                    if v >= best:
                        best, m = v, j
                if m >= 0:
                    taken[m] = True
                rows.append((x["score"], m >= 0))
        order = sorted(range(len(rows)), key=lambda i: -rows[i][0])       # python's sort is stable, like mergesort
        tp = fp = 0
        rc, pr = [], []
        for i in order:
            tp += rows[i][1]
            fp += not rows[i][1]
            rc.append(tp / npos)
            pr.append(tp / (tp + fp + np.spacing(1)))
        for i in range(len(pr) - 1, 0, -1):
            pr[i - 1] = max(pr[i - 1], pr[i])
        q = []
        for r in REC_THRS:
            idx = next((i for i, v in enumerate(rc) if v >= r), None)
            q.append(pr[idx] if idx is not None else 0.0)
        return float(np.mean(q))

    rng = np.random.default_rng(11)
    for trial in range(3):
        imgs = list(range(1, 7))
        gt, dt = {}, []
        for img in imgs:
            for _ in range(int(rng.integers(0, 5))):
                x, y = rng.uniform(0, 300, 2)
                w, h = rng.uniform(40, 120, 2)                 # all 'medium'/'large': inside the 'all' range either way
                gt.setdefault(img, []).append({"image_id": img, "category_id": 1, "bbox": [x, y, w, h], "area": w * h, "iscrowd": 0})
                for _ in range(int(rng.integers(0, 3))):       # detections scattered around the object
                    j = rng.normal(0, 14, 4)
                    dt.append({"image_id": img, "category_id": 1, "bbox": [x + j[0], y + j[1], max(w + j[2], 5), max(h + j[3], 5)],
                               "score": float(rng.random())})
            for _ in range(int(rng.integers(0, 3))):
                x, y = rng.uniform(0, 300, 2)
                dt.append({"image_id": img, "category_id": 1, "bbox": [x, y, 60.0, 60.0], "score": float(rng.random())})
        ev = BboxEval(gt, dt, [1], imgs).evaluate()
        for t, thr in enumerate(IOU_THRS):
            got = float(np.mean(ev.precision[t, :, 0, 0, 2]))
            assert got == pytest.approx(naive_ap(gt, dt, imgs, thr), abs=1e-12), (trial, thr)


def test_ds_utils_helpers():
    from datasets import ds_utils as du
    boxes = np.array([[10, 20, 30, 40], [10, 20, 30, 40], [0, 0, 5, 9], [10.2, 20.4, 30.1, 39.6]], np.float32)
    assert du.unique_boxes(boxes).tolist() == [0, 2] and du.unique_boxes(boxes, scale=10).tolist() == [0, 2, 3]
    assert du.xywh_to_xyxy(np.array([[2, 3, 4, 5]])).tolist() == [[2, 3, 5, 7]]
    assert du.xyxy_to_xywh(du.xywh_to_xyxy(np.array([[2, 3, 4, 5]]))).tolist() == [[2, 3, 4, 5]]
    assert du.filter_small_boxes(boxes, 9).tolist() == [0, 1, 3]           # w >= 9 and h > 9 (the reference's asymmetry)
    du.validate_boxes(np.array([[0, 0, 4, 4]]), width=5, height=5)
    with pytest.raises(AssertionError):
        du.validate_boxes(np.array([[0, 0, 5, 4]]), width=5, height=5)
    # differential check against the original project's ds_utils outputs (golden/make_ds_utils_golden.py)
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "ds_utils_vectors.npz"))
    b = ref["boxes"]
    assert np.array_equal(du.unique_boxes(b), ref["unique"])
    assert np.array_equal(du.unique_boxes(b, 0.25), ref["unique_0.25"])
    assert np.array_equal(du.xywh_to_xyxy(b), ref["xywh_to_xyxy"]) and np.array_equal(du.xyxy_to_xywh(b), ref["xyxy_to_xywh"])
    assert np.array_equal(du.filter_small_boxes(b, 12), ref["filter_small_12"])
