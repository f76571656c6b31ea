"""End-to-end parity: Network.test_image / im_detect / fused detect on the GPU against the oracle's whole
TEST-mode graph on identical seeded weights and inputs.

Stage-isolated tests (test_conv_gpu.py, test_stages_gpu.py) carry the bit-exact / 1e-4 claims.  End to end,
two different fp32 summation orders (oneDNN on the CPU, tcgen05 FP16x3 on the GPU) feed a sort + greedy NMS,
so a near-tie may legitimately flip; the assertions below therefore check (a) every dense tensor to a
relative bound, (b) the RoI set, (c) final scores/boxes to 1e-4 on the RoIs both sides selected."""
import numpy as np
import pytest
import torch

from oracle import pipeline as P
from tf_faster_rcnn_b200 import synth

pytestmark = pytest.mark.gpu
F = np.float32


def build(net_name, num_classes, scales):
    from model.config import cfg
    from nets.vgg16 import vgg16
    from nets.resnet_v1 import resnetv1
    from nets.mobilenet_v1 import mobilenetv1
    cfg.TEST.HAS_RPN = True
    if net_name == "vgg16":
        net = vgg16()
    elif net_name == "mobile":
        net = mobilenetv1()
    else:
        net = resnetv1(num_layers=int(net_name[3:]))
    net.create_architecture("TEST", num_classes, tag="default", anchor_scales=scales, anchor_ratios=(0.5, 1, 2))
    w = synth.make(net_name, num_classes, 3 * len(scales))
    net.load_weights(w)
    return net, w


def relerr(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def compare_detections(det, want_per_class, tol=0.05):
    """Match final detections (rows x1,y1,x2,y2,score,class) with the oracle's per-class lists: a detection is matched to the
    closest oracle box of its class when every coordinate agrees within `tol` px.  Unmatched rows on either side are near-tie
    flips of the two sorts / greedy NMS passes upstream (different fp32 summation orders), counted, not hidden."""
    n_want = int(sum(d.shape[0] for d in want_per_class))
    matched, box_err, score_err = 0, 0.0, 0.0
    cls = det[:, 5].astype(np.int64) if det.shape[0] else np.zeros(0, np.int64)
    for j, w in enumerate(want_per_class):
        g = det[cls == j]
        if not g.shape[0] or not w.shape[0]:
            continue
        d = np.abs(g[:, None, :4] - w[None, :, :4]).max(axis=2)
        used = set()
        for i in range(g.shape[0]):
            k = int(np.argmin(d[i]))
            if d[i, k] <= tol and k not in used:
                used.add(k); matched += 1
                box_err = max(box_err, float(d[i, k])); score_err = max(score_err, float(abs(g[i, 4] - w[k, 4])))
    return dict(n_got=int(det.shape[0]), n_want=n_want, matched=matched, box_err=box_err, score_err=score_err)


def fmt_report(r):
    return "detections gpu %d oracle %d matched %d (flips: %d gpu-only, %d oracle-only) | matched: box max %.2e px, score max %.2e" % (
        r["n_got"], r["n_want"], r["matched"], r["n_got"] - r["matched"], r["n_want"] - r["matched"], r["box_err"], r["score_err"])


def parity_log(line):
    """Append to gpurun_out/r02_parity.log when run on the GPU box (copied into profiles/r02_parity.md afterwards)."""
    import os
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, "r02_parity.log"), "a") as f:
            f.write(line.rstrip() + "\n")


@pytest.mark.parametrize("net_name,C,scales,hw", [
    ("vgg16", 21, (8, 16, 32), (300, 400)),
    ("res101", 81, (4, 8, 16, 32), (600, 800)),
    ("mobile", 81, (4, 8, 16, 32), (304, 400)),
    ("res50", 21, (8, 16, 32), (210, 333)),
])
def test_test_image_matches_oracle(cuda, net_name, C, scales, hw):
    net, w = build(net_name, C, scales)
    blob = synth.synthetic_blob(*hw)
    im_info = np.array([hw[0], hw[1], 1.0], F)
    o = P.opts(anchor_scales=scales)
    st = P.test_image(net_name, w, blob, im_info, C, o)
    cls_score, cls_prob, bbox_pred, rois = net.test_image(None, blob, im_info)
    plan = net.plan_for(*hw)
    feat = plan.feat.cpu().numpy()
    e_feat = relerr(feat, st["feat"])
    A = 3 * len(scales)
    rpn = plan.rpn_out.cpu().numpy().reshape(-1, plan.rpn_out.shape[-1])
    e_rpn_cls = relerr(rpn[:, :2 * A], st["rpn_cls_score"].reshape(-1, 2 * A))
    e_rpn_box = relerr(rpn[:, plan.rpn_dcol:plan.rpn_dcol + 4 * A], st["rpn_bbox_pred"].reshape(-1, 4 * A))
    e_scores = float(np.abs(plan.rpn_scores.cpu().numpy() - st["rpn_scores"]).max())
    e_props = float(np.abs(plan.rpn_props.cpu().numpy() - st["rpn_props"]).max())
    keep = plan.roi_keep.cpu().numpy()[:rois.shape[0]]
    same_set = np.array_equal(keep, st["roi_keep"])
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    e_prob = float(np.abs(cls_prob[ia] - st["cls_prob"][ib]).max())
    e_bbox = float(np.abs(bbox_pred[ia] - st["bbox_pred"][ib]).max())
    e_rois = float(np.abs(rois[ia] - st["rois"][ib]).max())
    print("\n[%s %dx%d] feat rel %.2e | rpn cls rel %.2e box rel %.2e | fg-score abs %.2e props abs %.2e | rois identical=%s "
          "common=%d/%d | cls_prob abs %.2e bbox_pred abs %.2e rois abs %.2e | GFLOP %.1f" %
          (net_name, hw[0], hw[1], e_feat, e_rpn_cls, e_rpn_box, e_scores, e_props, same_set, len(common), len(st["roi_keep"]),
           e_prob, e_bbox, e_rois, plan.tape.flops / 1e9))
    assert e_feat < 2e-5 and e_rpn_cls < 2e-5 and e_rpn_box < 5e-5
    assert e_scores < 2e-5 and e_props < 5e-3        # end-to-end drift: exp(dw)*w amplifies a 1e-5 delta error by the box size
    assert len(common) >= 0.97 * len(st["roi_keep"])
    assert e_prob < 1e-4 and e_bbox < 1e-4 and e_rois < 5e-3


def test_im_detect_and_fused_detect(cuda, monkeypatch):
    """im_detect surface + fused post-processing vs the oracle fed with the GPU's own head outputs
    (isolates the tail: decode, clip, per-class NMS, cap -> must be bit-exact)."""
    from model.test import im_detect, detect_image, _detections_python_loop
    from model.config import cfg
    net, w = build("res50", 21, (8, 16, 32))
    rng = np.random.default_rng(0)
    im = rng.integers(0, 256, (240, 320, 3), dtype=np.uint8)
    import cv2
    im = cv2.blur(im, (5, 5))
    monkeypatch.setattr(cfg, "USE_GPU_NMS", False)     # restored afterwards: the config is global to the session
    scores, boxes = im_detect(None, net, im)
    blob, scale = P.get_image_blob(im)
    plan = net.plan_for(blob.shape[1], blob.shape[2])
    r = scores.shape[0]
    rois = plan.rois[:r].cpu().numpy(); bbox_pred = plan.bbox_pred[:r].cpu().numpy()
    want_scores, want_boxes = P.im_detect_post(rois, scores, bbox_pred, scale, im.shape[0], im.shape[1])
    assert np.abs(boxes - want_boxes).max() < 1e-4
    net.options["use_gpu_nms"] = False
    per_class = detect_image(net, im, 0.0, 100)
    want = P.test_net_post(scores, boxes, P.opts(use_gpu_nms=False))
    loop = _detections_python_loop(scores, boxes, 21, 0.0, 100)
    for j in range(1, 21):
        assert np.array_equal(per_class[j], want[j]), j
        assert np.array_equal(loop[j], want[j]), j


def _run_modes(net_name, C, scales, hw, cfg_updates, oracle_opts):
    from model.config import cfg
    saved = {}
    try:
        for k, v in cfg_updates.items():
            node = cfg
            *parents, leaf = k.split(".")
            for p_ in parents:
                node = node[p_]
            saved[k] = node[leaf]
            node[leaf] = v
        net, w = build(net_name, C, scales)
        blob = synth.synthetic_blob(*hw)
        im_info = np.array([hw[0], hw[1], 1.0], F)
        st = P.test_image(net_name, w, blob, im_info, C, P.opts(anchor_scales=scales, **oracle_opts))
        out = net.test_image(None, blob, im_info)
        return net, st, out
    finally:
        for k, v in saved.items():
            node = cfg
            *parents, leaf = k.split(".")
            for p_ in parents:
                node = node[p_]
            node[leaf] = v


def test_top_mode_end_to_end(cuda):
    """TEST.MODE='top' (proposal_top_layer_tf): 5000 RoIs by score, no NMS -- through the whole net."""
    net, st, (cls_score, cls_prob, bbox_pred, rois) = _run_modes(
        "mobile", 21, (8, 16, 32), (320, 480), {"TEST.MODE": "top"}, dict(test_mode="top"))      # RPN_TOP_N = 5000 (config.py:208)
    assert rois.shape == (5000, 5) and st["rois"].shape == (5000, 5)
    plan = net.plan_for(320, 480)
    keep = plan.roi_keep.cpu().numpy()
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    assert len(common) >= 4950
    assert np.abs(cls_prob[ia] - st["cls_prob"][ib]).max() < 1e-4 and np.abs(bbox_pred[ia] - st["bbox_pred"][ib]).max() < 1e-4
    # ... and through the fused test_net tail (5000 RoIs per class list: kept sets in the global workspace)
    blob = synth.synthetic_blob(320, 480)
    det, _ = net.detect(blob, np.array([320, 480, 1.0], F), (320, 480))
    scores, boxes = P.im_detect_post(st["rois"], st["cls_prob"], st["bbox_pred"], 1.0, 320, 480)
    want = P.test_net_post(scores, boxes, P.opts())
    rep = compare_detections(det, want)
    print("\n[top-mode 5000] " + fmt_report(rep))
    assert rep["matched"] >= 0.9 * rep["n_want"] and rep["box_err"] < 2e-2 and rep["score_err"] < 1e-4


@pytest.mark.parametrize("gpu_pred", [False, True])
def test_non_e2e_proposal_mode_end_to_end(cuda, gpu_pred):
    """USE_E2E_TF=False (proposal_layer: pre-NMS top 6000 + '+1' NMS with the cpu_nms / gpu_nms predicate)."""
    net, st, (cls_score, cls_prob, bbox_pred, rois) = _run_modes(
        "res50", 21, (8, 16, 32), (210, 333), {"USE_E2E_TF": False, "USE_GPU_NMS": gpu_pred}, dict(use_e2e_tf=False, use_gpu_nms=gpu_pred))
    plan = net.plan_for(210, 333)
    keep = plan.roi_keep.cpu().numpy()[:rois.shape[0]]
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    assert abs(rois.shape[0] - st["rois"].shape[0]) <= 3 and len(common) >= 0.97 * len(st["roi_keep"])
    assert np.abs(cls_prob[ia] - st["cls_prob"][ib]).max() < 1e-4 and np.abs(bbox_pred[ia] - st["bbox_pred"][ib]).max() < 1e-4


def test_cfg5_shape_resnet152_1000_proposals(cuda):
    """config 5 geometry at a reduced image size: ResNet-152, anchor scales (2,4,8,16,32) (A=15), 1000 proposals."""
    net, st, (cls_score, cls_prob, bbox_pred, rois) = _run_modes(
        "res152", 81, (2, 4, 8, 16, 32), (256, 352), {"TEST.RPN_POST_NMS_TOP_N": 1000}, dict(rpn_post_nms_top_n=1000))
    plan = net.plan_for(256, 352)
    keep = plan.roi_keep.cpu().numpy()[:rois.shape[0]]
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    print("\n[cfg5-shape] rois gpu %d oracle %d common %d" % (rois.shape[0], st["rois"].shape[0], len(common)))
    assert len(common) >= 0.97 * len(st["roi_keep"])
    assert np.abs(cls_prob[ia] - st["cls_prob"][ib]).max() < 1e-4 and np.abs(bbox_pred[ia] - st["bbox_pred"][ib]).max() < 1e-4


def test_shape_cache_and_repeatability(cuda):
    """Two blob shapes through one network (plan cache) and bit-identical repeated runs (CUDA graph replay, split-K)."""
    net, w = build("res50", 21, (8, 16, 32))
    a = synth.synthetic_blob(208, 320, 1); b = synth.synthetic_blob(240, 272, 2)
    r1 = net.test_image(None, a, np.array([208, 320, 1.0], F))
    r2 = net.test_image(None, b, np.array([240, 272, 1.0], F))
    r3 = net.test_image(None, a, np.array([208, 320, 1.0], F))
    assert len(net._plans) == 2
    assert list(net._plans)[-1] == (208, 320, 1)      # most recently used last
    for x, y in zip(r1, r3):
        assert np.array_equal(x, y)
    assert r2[3].shape[1] == 5


def test_im_detect_with_device_preprocess(cuda):
    """Opt-in device blob (frcnn_preprocess) gives the same detections as the host OpenCV blob (inputs differ <= 1e-4)."""
    import cv2
    import model.test as MT
    net, w = build("res50", 21, (8, 16, 32))
    im = cv2.blur(np.random.default_rng(5).integers(0, 256, (240, 320, 3), dtype=np.uint8), (5, 5))
    s0, b0 = MT.im_detect(None, net, im)
    MT.DEVICE_PREPROCESS = True
    try:
        s1, b1 = MT.im_detect(None, net, im)
    finally:
        MT.DEVICE_PREPROCESS = False
    assert s0.shape == s1.shape and np.abs(s0 - s1).max() < 1e-3 and np.abs(b0 - b1).max() < 0.5


FULL_CONFIGS = [
    # (label, net, classes, anchor scales, blob H x W, cfg updates, oracle option updates, end-to-end box bound in px)
    # The box bound is 2x the measured end-to-end drift (profiles/r02_parity.md): two fp32 summation orders upstream, amplified by
    # exp(dw) * w -- it grows with the largest anchor (724 px wide at scale 32, 1448 px with the 800 px config's anchors).
    ("cfg2 ResNet-101 COCO 600x800, 300 proposals", "res101", 81, (4, 8, 16, 32), (600, 800), {}, {}, 5e-3),
    ("cfg1/3 VGG16 VOC 600x800, 300 proposals", "vgg16", 21, (8, 16, 32), (600, 800), {}, {}, 9e-3),
    ("cfg4 MobileNet-v1 COCO 600x800", "mobile", 81, (4, 8, 16, 32), (600, 800), {}, {}, 4e-3),
    ("cfg5 ResNet-152 800x1067, A=15, 1000 proposals", "res152", 81, (2, 4, 8, 16, 32), (800, 1067),
     {"TEST.RPN_POST_NMS_TOP_N": 1000}, dict(rpn_post_nms_top_n=1000), 2.6e-2),
]


@pytest.mark.parametrize("label,net_name,C,scales,hw,cfg_updates,oo,box_tol", FULL_CONFIGS, ids=[c[1] for c in FULL_CONFIGS])
def test_full_size_detections_match_oracle(cuda, label, net_name, C, scales, hw, cfg_updates, oo, box_tol):
    """BASELINE.json configs at their FULL shapes: Network.detect() (one graph replay: backbone .. per-class NMS .. cap) against
    the oracle's OWN chain test_image -> im_detect_post -> test_net_post -- nothing of the GPU run is fed to the oracle."""
    net, st, (cls_score, cls_prob, bbox_pred, rois) = _run_modes(net_name, C, scales, hw, cfg_updates, oo)
    plan = net.plan_for(*hw)
    keep = plan.roi_keep.cpu().numpy()[:rois.shape[0]]
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    e_props = float(np.abs(plan.rpn_props.cpu().numpy() - st["rpn_props"]).max())
    e_rois = float(np.abs(rois[ia] - st["rois"][ib]).max())
    e_prob = float(np.abs(cls_prob[ia] - st["cls_prob"][ib]).max())
    e_bbox = float(np.abs(bbox_pred[ia] - st["bbox_pred"][ib]).max())
    same_order = np.array_equal(keep, st["roi_keep"])
    blob = synth.synthetic_blob(*hw)
    det, _ = net.detect(blob, np.array([hw[0], hw[1], 1.0], F), hw)
    scores, boxes = P.im_detect_post(st["rois"], st["cls_prob"], st["bbox_pred"], 1.0, hw[0], hw[1])
    want = P.test_net_post(scores, boxes, P.opts(anchor_scales=scales, **oo))
    rep = compare_detections(det, want)
    line = ("[%s] RoIs: gpu %d oracle %d common %d identical-order=%s | proposals abs %.2e px, common RoIs abs %.2e px, cls_prob abs %.2e, "
            "bbox_pred abs %.2e | %s" % (label, rois.shape[0], st["rois"].shape[0], len(common), same_order, e_props, e_rois, e_prob, e_bbox,
                                       fmt_report(rep)))
    print("\n" + line)
    parity_log(line)
    assert len(common) >= 0.97 * len(st["roi_keep"])
    assert e_prob < 1e-4 and e_bbox < 1e-4                       # north-star tolerance on the RoIs both sides selected
    assert e_rois < box_tol and e_props < box_tol
    assert rep["matched"] >= 0.95 * rep["n_want"] and rep["score_err"] < 1e-4 and rep["box_err"] < box_tol


def test_detect_batch_matches_oracle_per_image(cuda):
    """Batch of 3 different images of one blob shape through ONE graph replay: every image's records match the oracle run on
    that image alone (per-image scale / original size are read from the device meta rows)."""
    net, w = build("res50", 21, (8, 16, 32))
    hw = (224, 304)
    blobs = np.concatenate([synth.synthetic_blob(hw[0], hw[1], seed) for seed in (1, 2, 3)], axis=0)
    scales = [1.0, 1.25, 0.8]
    orig = [(224, 304), (179, 243), (280, 380)]
    dets, plan = net.detect_batch(blobs, scales, orig)
    assert plan.batch == 3 and len(dets) == 3
    o = P.opts()
    for b in range(3):
        st = P.test_image("res50", w, blobs[b:b + 1], np.array([hw[0], hw[1], scales[b]], F), 21, o)
        scores, boxes = P.im_detect_post(st["rois"], st["cls_prob"], st["bbox_pred"], scales[b], orig[b][0], orig[b][1])
        want = P.test_net_post(scores, boxes, o)
        rep = compare_detections(dets[b], want)
        line = "[batch-of-3 image %d, res50 224x304] %s" % (b, fmt_report(rep))
        print("\n" + line); parity_log(line)
        assert rep["matched"] >= 0.9 * rep["n_want"] and rep["score_err"] < 1e-4 and rep["box_err"] < 5e-3
    # the same images one at a time give the same records up to the summation order of the split-K layers
    for b in range(3):
        single, _ = net.detect(blobs[b:b + 1], np.array([hw[0], hw[1], scales[b]], F), orig[b])
        rep = compare_detections(dets[b], [single[single[:, 5] == j, :5] for j in range(21)])
        assert rep["matched"] >= 0.95 * max(single.shape[0], 1) and rep["score_err"] < 1e-4


def test_submit_collect_pipeline_equals_detect_batch(cuda):
    """The pipelined throughput API (two batches in flight, copy stream + staging buffers) returns exactly detect_batch()'s records."""
    import torch
    net, w = build("res50", 21, (8, 16, 32))
    hw = (208, 320)
    batches = [np.concatenate([synth.synthetic_blob(hw[0], hw[1], 10 * i + b) for b in range(2)], axis=0) for i in range(5)]
    metas = [([1.0 + 0.1 * i, 0.9], [(208, 320), (231, 355)]) for i in range(5)]
    want = [net.detect_batch(x, m[0], m[1])[0] for x, m in zip(batches, metas)]
    pinned = [torch.from_numpy(x).pin_memory() for x in batches]
    tickets, got = [], []
    for x, m in zip(pinned, metas):
        tickets.append(net.submit_batch(x, m[0], m[1]))
        if len(tickets) > 1:
            got.append(net.collect_batch(tickets.pop(0)))
    got.append(net.collect_batch(tickets.pop(0)))
    for g, wnt in zip(got, want):
        for a, b in zip(g, wnt):
            assert np.array_equal(a, b)


def test_plan_cache_is_bounded(cuda):
    """ADVICE r01: the per-shape plan cache is an LRU (hundreds of distinct blob shapes in a dataset must not exhaust HBM)."""
    net, w = build("res50", 21, (8, 16, 32))
    net.MAX_PLANS = 2
    shapes = [(208, 320), (224, 272), (240, 256), (208, 320)]
    outs = []
    for i, (h, wd) in enumerate(shapes):
        outs.append(net.test_image(None, synth.synthetic_blob(h, wd, 1), np.array([h, wd, 1.0], F)))
        assert len(net._plans) <= 2
    for x, y in zip(outs[0], outs[3]):           # evicted and rebuilt: same results
        assert np.array_equal(x, y)


def test_throughput_mode_end_to_end_deviation(cuda, monkeypatch):
    """Opt-in throughput mode (FRCNN_CONV_IMPL=f16x1: plain fp16 operands, NOT fp32-grade) through the whole net: the deviation
    from the oracle is REPORTED (profiles/r02_parity.md), bounded loosely here; the default path's 1e-4 bounds do not apply."""
    monkeypatch.setenv("FRCNN_CONV_IMPL", "f16x1")
    net, w = build("res50", 21, (8, 16, 32))
    hw = (320, 480)
    blob = synth.synthetic_blob(*hw)
    im_info = np.array([hw[0], hw[1], 1.0], F)
    st = P.test_image("res50", w, blob, im_info, 21, P.opts())
    cls_score, cls_prob, bbox_pred, rois = net.test_image(None, blob, im_info)
    plan = net.plan_for(*hw)
    e_feat = relerr(plan.feat.cpu().numpy(), st["feat"])
    keep = plan.roi_keep.cpu().numpy()[:rois.shape[0]]
    common, ia, ib = np.intersect1d(keep, st["roi_keep"], return_indices=True)
    e_prob = float(np.abs(cls_prob[ia] - st["cls_prob"][ib]).max()) if len(common) else float("nan")
    det, _ = net.detect(blob, im_info, hw)
    scores, boxes = P.im_detect_post(st["rois"], st["cls_prob"], st["bbox_pred"], 1.0, hw[0], hw[1])
    rep = compare_detections(det, P.test_net_post(scores, boxes, P.opts()), tol=2.0)
    line = ("[THROUGHPUT MODE f16x1 (not fp32-grade), res50 320x480] feature map rel err %.2e | RoIs common %d/%d | cls_prob abs %.2e | %s"
            % (e_feat, len(common), len(st["roi_keep"]), e_prob, fmt_report(rep)))
    print("\n" + line); parity_log(line)
    assert 1e-5 < e_feat < 2e-2                       # visibly NOT the fp32-grade path, but sane
    assert len(common) >= 0.7 * len(st["roi_keep"]) and rep["matched"] >= 0.6 * rep["n_want"]
