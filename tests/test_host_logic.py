"""Host-side logic of the reference-facing surface (no GPU): config tree, blobs, anchors, thresholds, imdb,
tensorflow shim, the N>1 record gather over gloo, and tools/demo.py driven up to the (loud) device check."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))


def test_config_defaults_merge_and_set(tmp_path):
    from model import config as C
    cfg = C.cfg
    assert cfg.TEST.SCALES == (600,) and cfg.TEST.MAX_SIZE == 1000 and cfg.TEST.NMS == 0.3
    assert cfg.TEST.RPN_POST_NMS_TOP_N == 300 and cfg.TEST.RPN_NMS_THRESH == 0.7 and cfg.POOLING_SIZE == 7
    assert cfg.USE_E2E_TF is True and cfg.USE_GPU_NMS is True and cfg.RPN_CHANNELS == 512
    assert np.allclose(cfg.PIXEL_MEANS, [[[102.9801, 115.9465, 122.7717]]])
    y = tmp_path / "x.yml"
    y.write_text("EXP_DIR: t\nTEST:\n  HAS_RPN: True\n  SCALES: [800]\n  MAX_SIZE: 1333\nANCHOR_SCALES: [2,4,8,16,32]\n")
    saved = (cfg.TEST.SCALES, cfg.TEST.MAX_SIZE, list(cfg.ANCHOR_SCALES), cfg.EXP_DIR, cfg.TEST.HAS_RPN)
    try:
        C.cfg_from_file(str(y))
        assert cfg.TEST.SCALES == (800,) and cfg.TEST.MAX_SIZE == 1333 and cfg.ANCHOR_SCALES == [2, 4, 8, 16, 32]
        C.cfg_from_list(["TEST.MODE", "top", "TEST.RPN_TOP_N", "1000"])
        assert cfg.TEST.MODE == "top" and cfg.TEST.RPN_TOP_N == 1000
        with pytest.raises(KeyError):
            C._merge({"NOPE": 1}, cfg)
        with pytest.raises(ValueError):
            C._merge({"TEST": {"NMS": "x"}}, cfg)
        with pytest.raises(AssertionError):
            C.cfg_from_list(["TEST.NMS", "'str'"])

        class Imdb:
            name = "unit"
        old_root = cfg.ROOT_DIR
        cfg.ROOT_DIR = str(tmp_path)
        d = C.get_output_dir(Imdb(), None)
        assert d.endswith(os.path.join("output", "t", "unit", "default")) and os.path.isdir(d)
        cfg.ROOT_DIR = old_root
    finally:
        cfg.TEST.SCALES, cfg.TEST.MAX_SIZE, cfg.ANCHOR_SCALES, cfg.EXP_DIR, cfg.TEST.HAS_RPN = saved
        cfg.TEST.MODE, cfg.TEST.RPN_TOP_N = "nms", 5000


def test_im_list_to_blob_matches_reference_vector():
    from utils.blob import im_list_to_blob
    out = im_list_to_blob([G["blob_in0"], G["blob_in1"]])
    assert out.dtype == np.float32 and np.array_equal(out, G["blob_out"])


@pytest.mark.parametrize("tag,scales", [("s3", (8, 16, 32)), ("s4", (4, 8, 16, 32)), ("s5", (2, 4, 8, 16, 32))])
def test_product_anchors_match_reference(tag, scales):
    from layer_utils.generate_anchors import generate_anchors
    from layer_utils.snippets import generate_anchors_pre
    from oracle import anchors as OA
    assert np.array_equal(generate_anchors(scales=np.array(scales)), G["anchors_" + tag])
    tab, n = generate_anchors_pre(5, 7, 16, scales, (0.5, 1, 2))
    assert n == 5 * 7 * 3 * len(scales) and np.array_equal(tab, OA.tiled_anchors(5, 7, 16, scales, (0.5, 1, 2)))


def test_image_blob_scaling_rule_matches_oracle():
    from model.test import _get_image_blob
    from oracle import pipeline as P
    rng = np.random.default_rng(0)
    for hw in ((375, 500), (480, 640), (300, 1200), (1000, 200)):
        im = rng.integers(0, 256, hw + (3,), dtype=np.uint8)
        blob, scales = _get_image_blob(im)
        want, s = P.get_image_blob(im)
        assert scales.shape == (1,) and scales[0] == s and np.array_equal(blob, want)
        assert max(blob.shape[1:3]) <= 1000 + 1


def test_blob_geometry_predicts_opencv_output_size():
    """blob_geometry (used by the device preprocess path) == the size cv2.resize(fx, fy) actually produces."""
    from model.test import _get_image_blob, blob_geometry
    rng = np.random.default_rng(1)
    for _ in range(40):
        h, w = int(rng.integers(120, 1400)), int(rng.integers(120, 1400))
        blob, scales = _get_image_blob(np.zeros((h, w, 3), np.uint8))
        H, W, f = blob_geometry((h, w, 3))
        assert (H, W) == blob.shape[1:3] and f == scales[0], (h, w)


def test_nms_threshold_rule_and_empty_input():
    from tf_faster_rcnn_b200 import engine, _native as N
    from model.nms_wrapper import nms
    t, f = engine.nms_threshold(0.3, use_gpu_nms=False)
    assert f == N.NMS_MODE_CPU_NMS and t >= 0.3 and np.float32(t) == np.nextafter(np.float32(0.3), np.float32(0)) or t >= 0.3
    t2, f2 = engine.nms_threshold(0.3, use_gpu_nms=True)
    assert f2 == N.NMS_MODE_GPU_NMS and t2 == float(np.float32(0.3))
    assert engine.nms_threshold(0.5, False)[0] == 0.5
    assert nms(np.zeros((0, 5), np.float32), 0.3) == []          # nms_wrapper.py:18-19, no device needed


def test_conv_geometry_helpers():
    from tf_faster_rcnn_b200 import ops
    assert ops.same_pads(600, 3, 1) == (1, 1) and ops.same_pads(75, 2, 2) == (0, 1) and ops.same_pads(38, 2, 2) == (0, 0)
    assert ops.conv_out_hw(600, 800, 7, 2, "EXPLICIT") == (300, 400, 3, 3)
    assert ops.conv_out_hw(75, 100, 3, 2, "EXPLICIT") == (38, 50, 1, 1)
    assert ops.conv_out_hw(38, 50, 3, 1, "SAME") == (38, 50, 1, 1)


def test_synthetic_imdb_and_tf_shim(tmp_path):
    from datasets.factory import get_imdb
    imdb = get_imdb("synthetic_3_5")
    assert imdb.num_classes == 5 and len(imdb.image_index) == 3 and os.path.isfile(imdb.image_path_at(2))
    with pytest.raises(KeyError):
        get_imdb("imagenet_2012_val")
    from tf_faster_rcnn_b200 import paths
    sys.path.append(paths.SHIMS)
    try:
        import importlib
        tf = importlib.import_module("tensorflow")
        c = tf.ConfigProto(allow_soft_placement=True)
        c.gpu_options.allow_growth = True
        s = tf.Session(config=c)
        with pytest.raises(IOError):
            tf.train.Saver().restore(s, str(tmp_path / "missing.ckpt"))
        s.close()
    finally:
        sys.path.remove(paths.SHIMS)
        sys.modules.pop("tensorflow", None)


def test_result_file_formats(tmp_path):
    """VOC text lines (+1 pixel shift, %.3f/%.1f) and COCO json (xywh with +1 extents), as the reference writes them."""
    import json
    from datasets.factory import SimpleImdb
    imdb = SimpleImdb("fmt", ["/x/000012.jpg", "/x/000034.png"], 3)
    e = np.zeros((0, 5), np.float32)
    all_boxes = [[e, e], [np.array([[10.26, 20.0, 110.5, 220.04, 0.98765]], np.float32), e],
                 [e, np.array([[0.0, 1.0, 2.0, 3.0, 0.5], [5.5, 6.5, 7.5, 8.5, 0.25]], np.float32)]]
    files = imdb.write_voc_results(all_boxes, str(tmp_path))
    assert open(files[0]).read() == "000012 0.988 11.3 21.0 111.5 221.0\n"
    assert open(files[1]).read() == "000034 0.500 1.0 2.0 3.0 4.0\n000034 0.250 6.5 7.5 8.5 9.5\n"
    res = imdb.write_coco_results(all_boxes, str(tmp_path / "r.json"))
    assert json.load(open(tmp_path / "r.json")) == res and len(res) == 3
    assert res[1] == {"image_id": "000034", "category_id": 2, "bbox": [0.0, 1.0, 3.0, 3.0], "score": 0.5}
    assert imdb.evaluate_detections(all_boxes, str(tmp_path)) == [0, 1, 2]


GLOO_WORKER = textwrap.dedent("""
    import os, sys
    sys.path.insert(0, %r)
    import numpy as np, torch, torch.distributed as dist
    from tf_faster_rcnn_b200 import parallel as PP
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", rank=rank, world_size=world)
    num_images, C, max_det = 5, 4, 8
    H = PP.REC_HEADER
    all_boxes = [[[] for _ in range(num_images)] for _ in range(C)]
    recs = [torch.zeros(H + max_det * 6), torch.zeros(H + max_det * 6)]      # the producer alternates between two record buffers
    g = PP.RecordGather(recs[0], world)
    mine = PP.shard_indices(num_images, rank, world)
    nsteps = PP.steps_for(num_images, world)
    for step in range(nsteps):
        slot = step & 1
        g.before_overwrite(slot)
        rec = recs[slot]
        rec.zero_()
        if step < len(mine):
            img = mine[step]
            n = 1 + img %% 3
            rows = rec[H:].view(max_det, 6)
            for k in range(n):
                rows[k] = torch.tensor([img, k, img + 10, k + 10, 0.9 - 0.1 * k, 1 + (img + k) %% (C - 1)], dtype=torch.float32)
            rec.view(torch.int32)[0] = n
        g.issue(slot, rec)                                   # ONE collective per step, asynchronous
        if step > 0:
            PP.records_to_all_boxes(all_boxes, step - 1, world, g.result(slot ^ 1), num_images)
    PP.records_to_all_boxes(all_boxes, nsteps - 1, world, g.result((nsteps - 1) & 1), num_images)
    assert g.collectives == nsteps, g.collectives
    tot = sum(len(all_boxes[j][i]) for j in range(1, C) for i in range(num_images))
    assert tot == sum(1 + i %% 3 for i in range(num_images)), tot
    for i in range(num_images):
        for j in range(1, C):
            for row in all_boxes[j][i]:
                assert row[0] == i
    dist.destroy_process_group()
    print("rank", rank, "ok")
""")


def test_two_rank_record_gather_over_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER % ROOT)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29611", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("ok" in o for o in outs)


SHARDED_WORKER = textwrap.dedent("""
    import os, sys, pickle
    sys.path.insert(0, %r)
    import numpy as np, torch, torch.distributed as dist
    from tf_faster_rcnn_b200 import paths
    paths.add_lib_path()
    from model import test as T
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dist.init_process_group("gloo", rank=rank, world_size=world)

    class Imdb:
        num_classes = 4
        def __init__(self, n): self.image_index = list(range(n))

    from tf_faster_rcnn_b200.parallel import REC_HEADER as H
    bufs = [torch.zeros(H + 12 * 6), torch.zeros(H + 12 * 6)]
    turn = [0]

    def fake(i, cap=12):            # a deterministic stand-in for the device path: records depend on the image only
        n = (i * 5) %% 7
        rec = bufs[turn[0] & 1]; turn[0] += 1        # like ShapePlan: consecutive records alternate between two buffers
        rec.zero_()
        rows = rec[H:].view(cap, 6)
        for k in range(n):
            rows[k] = torch.tensor([i, k, i + 20, k + 20, 1.0 - 0.1 * k, 1 + (i + k) %% 3], dtype=torch.float32)
        rec.view(torch.int32)[0] = n
        return rec

    out = {}
    for n_images in (5, 1, 0, 4):
        calls = []
        boxes = T._test_net_sharded(Imdb(n_images), lambda i: (calls.append(i), fake(i))[1], verbose=False)
        assert calls == list(range(rank, n_images, world)), calls           # each rank ran only its shard
        out[n_images] = boxes
    if rank == 0:
        with open(os.environ["OUT"], "wb") as f:
            pickle.dump(out, f)
    dist.barrier()
    dist.destroy_process_group()
    print("rank", rank, "ok")
""")


def test_sharded_test_net_matches_single_process(tmp_path):
    """model.test._test_net_sharded over 2 gloo ranks (5 / 1 / 0 / 4 images: ragged last step, an idle rank, empty set)
    assembles the same all_boxes on every rank as a single-process pass over the same per-image records."""
    import pickle
    script = tmp_path / "s.py"
    script.write_text(SHARDED_WORKER % ROOT)
    out = str(tmp_path / "boxes.pkl")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29613", WORLD_SIZE="2", OUT=out)
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    got = pickle.load(open(out, "rb"))
    for n_images, boxes in got.items():
        assert len(boxes) == 4 and all(len(per_image) == n_images for per_image in boxes)
        for i in range(n_images):
            n = (i * 5) % 7
            rows = np.array([[i, k, i + 20, k + 20, np.float32(1.0 - 0.1 * k), 1 + (i + k) % 3] for k in range(n)], np.float32).reshape(-1, 6)
            for j in range(1, 4):
                want = rows[rows[:, 5] == j, :5]
                assert np.array_equal(np.asarray(boxes[j][i], np.float32).reshape(-1, 5), want), (n_images, i, j)


def test_demo_script_stops_loudly_without_a_device(tmp_path):
    """tools/demo.py with a TensorFlow V2 checkpoint and a directory of images.  Without a GPU it must get through argument
    parsing, cfg, create_architecture, the strict checkpoint restore and cv2.imread, and stop at the first image with the
    loud 'no CUDA device' error -- there is no CPU fallback to fall into."""
    import cv2
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the behaviour without a CUDA device")
    pre = str(tmp_path / "res50_faster_rcnn.ckpt")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_synthetic_ckpt.py"), "--net", "res50", "--classes", "21",
                           "--anchors", "9", "--format", "bundle", "--out", pre], cwd=ROOT)
    images = tmp_path / "images"
    images.mkdir()
    cv2.imwrite(str(images / "000456.jpg"), np.random.default_rng(0).integers(0, 256, (240, 320, 3), dtype=np.uint8))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "demo.py"), "--net", "res50", "--images", str(images),
                        "--model", pre], cwd=str(tmp_path), capture_output=True, text=True, timeout=300)
    out = r.stdout + r.stderr
    assert r.returncode != 0
    assert "in im_detect" in out, out[-2000:]
    assert "check_device failed" in out and "no CUDA device" in out, out[-2000:]


def test_nms_module_surface_routes_to_the_device_entry(monkeypatch):
    """nms.gpu_nms / nms.cpu_nms / nms.py_cpu_nms (the reference's import surface) sort on the host, call the
    `_nms`-compatible device entry with the right predicate flags, and map kept positions back to input indices."""
    from tf_faster_rcnn_b200 import ops, _native as N
    from nms.gpu_nms import gpu_nms
    from nms.cpu_nms import cpu_nms
    from nms.py_cpu_nms import py_cpu_nms
    calls = []

    def fake(sorted_dets, thresh, flags, device_id=0):
        calls.append((np.array(sorted_dets), thresh, flags, device_id))
        return np.array([0, 2], dtype=np.int32)              # keep the best and the third best
    monkeypatch.setattr(ops, "nms_host", fake)
    dets = np.array([[0, 0, 9, 9, 0.2], [1, 1, 8, 8, 0.9], [2, 2, 7, 7, 0.5], [3, 3, 6, 6, 0.9]], np.float32)
    assert gpu_nms(dets, 0.3, device_id=0) == [1, 2]          # order = [1, 3, 2, 0] (tie 0.9: lower index first)
    assert calls[-1][0][:, 4].tolist() == pytest.approx([0.9, 0.9, 0.5, 0.2]) and calls[-1][2] == N.NMS_MODE_GPU_NMS
    assert calls[-1][1] == float(np.float32(0.3))
    assert cpu_nms(dets, 0.3) == [1, 2] and calls[-1][2] == N.NMS_MODE_CPU_NMS
    assert calls[-1][1] == float(np.float32(0.3))             # f32(0.3) > 0.3: '>= 0.3 (double)' == '>= f32(0.3)'
    cpu_nms(dets, 0.7)
    assert calls[-1][1] == float(np.nextafter(np.float32(0.7), np.float32(1)))    # f32(0.7) < 0.7: next fp32 up
    assert py_cpu_nms(dets, 0.3) == [1, 2] and calls[-1][2] == N.NMS_MODE_GPU_NMS
    assert gpu_nms(np.zeros((0, 5), np.float32), 0.3) == [] and cpu_nms(np.zeros((0, 5), np.float32), 0.3) == []


def test_bbox_transform_module_matches_oracle_codec():
    """model.bbox_transform (reference module surface): decode / clip equal the oracle codec on fp32 inputs up to exp's last ulp,
    the regression targets invert the decode."""
    from model import bbox_transform as BT
    from oracle import boxes as OB
    rng = np.random.default_rng(4)
    b = np.sort(rng.uniform(0, 500, (50, 2, 2)), axis=1).transpose(0, 2, 1).reshape(50, 4).astype(np.float32)[:, [0, 2, 1, 3]]
    b = np.stack([b[:, 0], b[:, 1], b[:, 0] + rng.uniform(5, 200, 50), b[:, 1] + rng.uniform(5, 200, 50)], axis=1).astype(np.float32)
    d = (rng.standard_normal((50, 12)) * 0.3).astype(np.float32)
    got = BT.bbox_transform_inv(b, d)
    want = OB.decode(b, d)
    assert got.dtype == np.float32 and np.abs(got - want).max() < 1e-3 * 1.0 and np.abs(got - want).max() / np.abs(want).max() < 1e-6
    assert np.array_equal(BT.clip_boxes(got.copy(), (375, 500)), OB.clip_two_sided(got, 375, 500))
    assert BT.bbox_transform_inv(np.zeros((0, 4), np.float32), np.zeros((0, 8), np.float32)).shape == (0, 8)
    # targets: '+1' widths, centre offsets in units of the example box, log size ratios (hand-computed case)
    t = BT.bbox_transform(np.array([[0., 0., 9., 9.]]), np.array([[5., 5., 24., 24.]]))
    assert np.allclose(t, [[1.0, 1.0, np.log(2.0), np.log(2.0)]])
