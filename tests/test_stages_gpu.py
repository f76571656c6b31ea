"""Stage-isolated parity of the bandwidth kernels against the oracle (same seeded inputs).
Integer / index outputs (sort order, NMS survivors, keep lists) must be bit-exact; float outputs are
checked with the tolerance written at each assert (1e-4 absolute on boxes/scores is the north-star bound)."""
import os

import numpy as np
import pytest
import torch

from oracle import anchors as OA
from oracle import boxes as OB
from oracle import layers as L
from oracle import nms as ONMS
from oracle import pipeline as P

pytestmark = pytest.mark.gpu
F = np.float32


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rand_boxes(rng, n, size=600.0, wh=(8, 200)):
    xy = rng.uniform(0, size, (n, 2))
    s = rng.uniform(wh[0], wh[1], (n, 2))
    return np.hstack([xy, np.minimum(xy + s, size - 1)]).astype(F)


# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,stride,cout,act,bn", [(3, 1, 64, 1, False), (7, 2, 64, 1, True), (3, 2, 32, 2, True)])
def test_conv_first(cuda, k, stride, cout, act, bn):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(k * 10 + stride)
    x = (rng.standard_normal((1, 61, 83, 3)) * 50).astype(F)
    w = (rng.standard_normal((k, k, 3, cout)) * 0.01).astype(F)
    if stride == 1:
        conv = L.conv2d(x, w, 1, "SAME"); mode = "SAME"
    else:
        conv = L.conv2d_same(x, w, stride); mode = "EXPLICIT"
    if bn:
        y, scale, shift = L.batch_norm(conv, rng.uniform(.5, 1.5, cout).astype(F), rng.standard_normal(cout).astype(F),
                                       rng.standard_normal(cout).astype(F), rng.uniform(.5, 1.5, cout).astype(F), 1e-5)
    else:
        scale, shift = None, rng.standard_normal(cout).astype(F)
        y = conv + shift
    want = L.relu(y) if act == 1 else L.relu6(y)
    ho, wo, pt, pl = ops.conv_out_hw(61, 83, k, stride, mode)
    out = torch.empty((1, ho, wo, cout), dtype=torch.float32, device="cuda")
    ops.conv_first(dev(x), dev(w), None if scale is None else dev(scale), dev(shift), out, k, stride, pt, pl, act)
    got = out.cpu().numpy()
    assert got.shape == want.shape
    assert np.abs(got - want).max() < 1e-4 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("stride", [1, 2])
def test_depthwise(cuda, stride):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(stride)
    c = 64
    x = rng.standard_normal((1, 37, 50, c)).astype(F)
    w = rng.standard_normal((3, 3, c, 1)).astype(F)
    conv = L.conv2d_same(x, w, stride, groups=c)
    y, scale, shift = L.batch_norm(conv, rng.uniform(.5, 1.5, c).astype(F), rng.standard_normal(c).astype(F),
                                   rng.standard_normal(c).astype(F), rng.uniform(.5, 1.5, c).astype(F), 1e-3)
    want = L.relu6(y)
    ho, wo, pt, pl = ops.conv_out_hw(37, 50, 3, stride, "SAME" if stride == 1 else "EXPLICIT")
    out = torch.empty((1, ho, wo, c), dtype=torch.float32, device="cuda")
    ops.depthwise3x3(dev(x), dev(w.reshape(3, 3, c)), dev(scale), dev(shift), out, stride, pt, pl, 2)
    got = out.cpu().numpy()
    assert got.shape == want.shape
    assert np.abs(got - want).max() < 2e-5


def test_max_pools(cuda):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 75, 101, 64)).astype(F)
    # VGG 2x2/2 SAME (odd dims -> pad after, ignored)
    want = L.max_pool(x, 2, 2, "SAME")
    out = torch.empty(want.shape, dtype=torch.float32, device="cuda")
    ops.max_pool(dev(x), out, 2, 2, 0, 0, True)
    assert np.array_equal(out.cpu().numpy(), want)
    # ResNet pool1: zero pad 1 then 3x3/2 VALID
    want = L.max_pool(np.pad(x, ((0, 0), (1, 1), (1, 1), (0, 0))), 3, 2, "VALID")
    out = torch.empty(want.shape, dtype=torch.float32, device="cuda")
    ops.max_pool(dev(x), out, 3, 2, 1, 1, False)
    assert np.array_equal(out.cpu().numpy(), want)
    # shortcut subsample: 1x1/2
    want = L.max_pool(x, 1, 2, "VALID")
    out = torch.empty(want.shape, dtype=torch.float32, device="cuda")
    ops.max_pool(dev(x), out, 1, 2, 0, 0, True)
    assert np.array_equal(out.cpu().numpy(), want)


def test_spatial_mean(cuda):
    from tf_faster_rcnn_b200 import ops
    x = np.random.default_rng(1).standard_normal((33, 7, 7, 256)).astype(F)
    out = torch.empty((33, 256), dtype=torch.float32, device="cuda")
    ops.spatial_mean(dev(x), out)
    assert np.abs(out.cpu().numpy() - x.mean(axis=(1, 2), dtype=F)).max() < 1e-6


@pytest.mark.parametrize("pre_pool", [0, 1])
def test_crop_pool(cuda, pre_pool):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(7 + pre_pool)
    feat = rng.standard_normal((1, 38, 50, 64)).astype(F)
    b = rand_boxes(rng, 97, 800.0)
    b[:, [1, 3]] = np.minimum(b[:, [1, 3]], 599)
    b[0] = [0, 0, 799, 599]; b[1] = [790, 590, 799, 599]; b[2] = [5, 5, 5, 5]   # full image, corner, degenerate
    rois = np.hstack([np.zeros((97, 1), F), b]).astype(F)
    nb = P.roi_norm_boxes(feat.shape, rois)
    want = L.max_pool(L.crop_and_resize(feat, nb, 14), 2, 2, "SAME") if pre_pool else L.crop_and_resize(feat, nb, 7)
    out = torch.empty((97, 7, 7, 64), dtype=torch.float32, device="cuda")
    ops.crop_pool(dev(feat), dev(rois), 7, pre_pool, out)
    got = out.cpu().numpy()
    assert np.array_equal(got, want), "crop_and_resize must be bit-exact (same fp32 op order); max diff %g" % np.abs(got - want).max()


@pytest.mark.parametrize("scales", [(8, 16, 32), (4, 8, 16, 32), (2, 4, 8, 16, 32)])
def test_rpn_decode(cuda, scales):
    from tf_faster_rcnn_b200 import ops
    A = 3 * len(scales)
    fh, fw = 38, 50
    rng = np.random.default_rng(A)
    cls = (rng.standard_normal((1, fh, fw, 2 * A)) * 2).astype(F)
    box = (rng.standard_normal((1, fh, fw, 4 * A)) * 0.3).astype(F)
    o = P.opts(anchor_scales=scales)
    s_want, p_want, _ = P.rpn_decode(cls, box, np.array([600, 800, 1.0], F), o)
    dcol = (2 * A + 3) // 4 * 4
    ld = (dcol + 4 * A + 3) // 4 * 4
    fused = np.zeros((fh * fw, ld), F)
    fused[:, :2 * A] = cls.reshape(-1, 2 * A)
    fused[:, dcol:dcol + 4 * A] = box.reshape(-1, 4 * A)
    scores = torch.empty(fh * fw * A, dtype=torch.float32, device="cuda")
    props = torch.empty((fh * fw * A, 4), dtype=torch.float32, device="cuda")
    base = OA.base_anchors(ratios=(0.5, 1, 2), scales=scales).astype(F)
    ops.rpn_decode(dev(fused), dcol, dev(base), A, fh, fw, 600.0, 800.0, scores, props)
    assert np.abs(scores.cpu().numpy() - s_want).max() < 1e-6          # 2-way softmax, expf vs np.exp
    assert np.abs(props.cpu().numpy() - p_want).max() < 1e-4           # north-star box tolerance


def test_sort_desc_stable(cuda):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(3)
    for n in (1, 2, 7, 8, 9, 255, 256, 257, 8191, 8192, 8193, 22800, 50250, 90112):
        keys = rng.random(n).astype(F)
        keys[rng.integers(0, n, n // 3)] = F(0.5)      # many exact ties
        if n > 100:
            keys[:40] = (rng.standard_normal(40) * 1e3).astype(F)       # negative / large keys, +-0, denormals: the total order
            keys[40:44] = [0.0, -0.0, 1e-40, -1e-40]
        order = torch.empty(n, dtype=torch.int32, device="cuda")
        sk = torch.empty(n, dtype=torch.float32, device="cuda")
        ops.sort_desc(dev(keys), order, sk)
        assert np.array_equal(order.cpu().numpy(), ONMS.argsort_desc(keys)), n


def _proposal_case(rng, n):
    props = rand_boxes(rng, n, 800.0, (16, 400))
    # clusters of near-duplicates so NMS has work to do
    props[n // 2:] = props[: n - n // 2] + rng.uniform(-6, 6, (n - n // 2, 4)).astype(F)
    scores = rng.random(n).astype(F)
    return np.ascontiguousarray(props, F), scores


@pytest.mark.parametrize("n,post", [(1, 300), (63, 300), (64, 300), (65, 300), (300, 300), (6000, 300), (22800, 300), (50250, 1000)])
def test_proposals_tf_mode(cuda, n, post):
    from tf_faster_rcnn_b200 import ops, _native as N
    rng = np.random.default_rng(n)
    props, scores = _proposal_case(rng, n)
    if n > 100:
        props[5] = [10, 10, 10, 50]; props[6] = [30, 30, 20, 20]      # zero-area and inverted boxes (TF rule)
        scores[[5, 6]] = [0.999, 0.998]
    want_rois, want_sc, want_keep = P.proposals_e2e_tf(scores, props, P.opts(rpn_post_nms_top_n=post))
    order = torch.empty(n, dtype=torch.int32, device="cuda"); sk = torch.empty(n, dtype=torch.float32, device="cuda")
    pd, sd = dev(props), dev(scores)
    ops.sort_desc(sd, order, sk)
    rois = torch.empty((post, 5), dtype=torch.float32, device="cuda"); rs = torch.empty(post, dtype=torch.float32, device="cuda")
    keep = torch.empty(post, dtype=torch.int32, device="cuda"); num = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.proposals(pd, sd, order, 0, post, 0.7, N.NMS_MODE_TF, rois, rs, keep, num)
    k = int(num.item())
    assert k == want_keep.shape[0]
    assert np.array_equal(keep.cpu().numpy()[:k], want_keep)                     # survivor indices bit-exact
    assert np.array_equal(rois.cpu().numpy()[:k], want_rois)
    assert np.array_equal(rs.cpu().numpy()[:k], want_sc.ravel())
    assert not rois.cpu().numpy()[k:].any()


@pytest.mark.parametrize("gpu_pred", [False, True])
def test_proposals_numpy_mode_and_top(cuda, gpu_pred):
    from tf_faster_rcnn_b200 import ops, _native as N
    n = 22800
    rng = np.random.default_rng(11)
    props, scores = _proposal_case(rng, n)
    props = np.round(props)                                       # integer coords: exact-threshold IoUs do occur
    o = P.opts(use_e2e_tf=False, use_gpu_nms=gpu_pred)
    want_rois, _, want_keep = P.proposals_numpy(scores, props, o)
    order = torch.empty(n, dtype=torch.int32, device="cuda"); sk = torch.empty(n, dtype=torch.float32, device="cuda")
    pd, sd = dev(props), dev(scores)
    ops.sort_desc(sd, order, sk)
    rois = torch.empty((300, 5), dtype=torch.float32, device="cuda"); rs = torch.empty(300, dtype=torch.float32, device="cuda")
    keep = torch.empty(300, dtype=torch.int32, device="cuda"); num = torch.zeros(1, dtype=torch.int32, device="cuda")
    flags = N.NMS_MODE_GPU_NMS if gpu_pred else N.NMS_MODE_CPU_NMS
    thr = float(ONMS.thresh_f32(0.7, inclusive=not gpu_pred))
    ops.proposals(pd, sd, order, 6000, 300, thr, flags, rois, rs, keep, num)
    k = int(num.item())
    assert k == want_keep.shape[0] and np.array_equal(keep.cpu().numpy()[:k], want_keep)
    assert np.array_equal(rois.cpu().numpy()[:k], want_rois)
    # TEST.MODE='top': first 5000 by score, no NMS
    want_rois, _, want_keep = P.proposals_top(scores, props, P.opts(test_mode="top"))
    rois = torch.empty((5000, 5), dtype=torch.float32, device="cuda"); rs = torch.empty(5000, dtype=torch.float32, device="cuda")
    keep = torch.empty(5000, dtype=torch.int32, device="cuda")
    ops.proposals(pd, sd, order, 0, 5000, -1.0, 0, rois, rs, keep, num)
    assert int(num.item()) == 5000 and np.array_equal(keep.cpu().numpy(), want_keep)
    assert np.array_equal(rois.cpu().numpy(), want_rois)


def test_cls_finish_and_bbox_decode(cuda):
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(21)
    R, Cc = 300, 81
    logits = (rng.standard_normal((R, Cc)) * 3).astype(F)
    deltas = (rng.standard_normal((R, 4 * Cc)) * 0.5).astype(F)
    head = np.hstack([logits, deltas]).astype(F)
    stds, means = (0.1, 0.1, 0.2, 0.2), (0.0, 0.0, 0.0, 0.0)
    cs = torch.empty((R, Cc), dtype=torch.float32, device="cuda"); cp = torch.empty_like(cs)
    bp = torch.empty((R, 4 * Cc), dtype=torch.float32, device="cuda")
    ops.cls_finish(dev(head), Cc, stds, means, cs, cp, bp)
    want_prob = L.softmax_lastdim(logits)
    want_bbox = (deltas * np.tile(np.asarray(stds), Cc).astype(F) + np.tile(np.asarray(means), Cc).astype(F)).astype(F)
    assert np.array_equal(cs.cpu().numpy(), logits)
    assert np.abs(cp.cpu().numpy() - want_prob).max() < 1e-6
    assert np.array_equal(bp.cpu().numpy(), want_bbox)
    b = rand_boxes(rng, R, 800.0)
    rois = np.hstack([np.zeros((R, 1), F), b]).astype(F)
    scale = 1.6
    _, want_pred = P.im_detect_post(rois, want_prob, want_bbox, scale, 375, 500)
    pred = torch.empty((R, 4 * Cc), dtype=torch.float32, device="cuda")
    ops.bbox_decode(dev(rois), dev(want_bbox), Cc, ops.im_meta_tensor([(scale, 375, 500)]), pred)
    assert np.abs(pred.cpu().numpy() - want_pred).max() < 1e-4      # north-star box tolerance


@pytest.mark.parametrize("R,Cc,gpu_pred", [(300, 21, False), (300, 81, False), (300, 81, True), (1000, 81, False), (17, 5, False)])
def test_detect_post(cuda, R, Cc, gpu_pred):
    from tf_faster_rcnn_b200 import ops, _native as N
    rng = np.random.default_rng(R + Cc)
    probs = L.softmax_lastdim((rng.standard_normal((R, Cc)) * 2).astype(F))
    probs[rng.integers(0, R, 5), rng.integers(1, Cc, 5)] = 0.0      # exact zeros are dropped by `> 0.`
    centers = rand_boxes(rng, R, 500.0, (20, 200))
    pred = np.repeat(centers[:, None, :], Cc, axis=1) + rng.uniform(-15, 15, (R, Cc, 4)).astype(F)
    pred = np.round(pred.reshape(R, 4 * Cc)).astype(F)
    o = P.opts(use_gpu_nms=gpu_pred)
    want = P.test_net_post(probs, pred, o)
    det = torch.zeros((2048, 6), dtype=torch.float32, device="cuda"); ndet = torch.zeros(1, dtype=torch.int32, device="cuda")
    keep = torch.empty((Cc, R), dtype=torch.int32, device="cuda"); cnt = torch.empty(Cc, dtype=torch.int32, device="cuda")
    ks = torch.empty((Cc, R), dtype=torch.float32, device="cuda")
    nr = torch.tensor([R], dtype=torch.int32, device="cuda")
    flags = N.NMS_MODE_GPU_NMS if gpu_pred else N.NMS_MODE_CPU_NMS
    thr = float(ONMS.thresh_f32(0.3, inclusive=not gpu_pred))
    ops.detect_post(dev(probs), dev(pred), nr, Cc, 0.0, thr, flags, 100, det, ndet, keep, cnt, ks)
    nd = int(ndet.item())
    got = det.cpu().numpy()[:nd]
    want_flat = np.vstack([np.hstack([d, np.full((d.shape[0], 1), j, F)]) for j, d in enumerate(want) if d.shape[0]])
    assert nd == want_flat.shape[0], (nd, want_flat.shape)
    assert np.array_equal(got, want_flat)          # boxes, scores, classes and order all bit-exact
    cn = cnt.cpu().numpy()
    assert [int(c) for c in cn] == [d.shape[0] for d in want]


@pytest.mark.parametrize("n", [0, 1, 63, 64, 65, 300, 6000])
@pytest.mark.parametrize("mode", ["cpu_nms", "gpu_nms", "tf"])
def test_nms_host_matches_oracle(cuda, n, mode):
    from tf_faster_rcnn_b200 import ops, _native as N
    rng = np.random.default_rng(n + 1)
    if n == 0:
        assert ops.nms_host(np.zeros((0, 5), F), 0.3, N.NMS_MODE_CPU_NMS).shape[0] == 0
        return
    props, scores = _proposal_case(rng, n)
    props = np.round(props)
    dets = np.hstack([props, scores[:, None]]).astype(F)
    order = ONMS.argsort_desc(scores)
    sd = dets[order]
    for thr in (0.3, 0.7):
        if mode == "tf":
            want = ONMS.nms_tf_c(props, scores, n, thr)
            got = order[ops.nms_host(sd, float(F(thr)), N.NMS_MODE_TF)]
        else:
            inc = mode == "cpu_nms"
            want = ONMS.nms_plus1_c(dets, thr, inc)
            got = order[ops.nms_host(sd, float(ONMS.thresh_f32(thr, inc)), N.NMS_MODE_CPU_NMS if inc else N.NMS_MODE_GPU_NMS)]
        assert np.array_equal(got, want), (n, mode, thr)


def test_nms_corner_cases(cuda):
    """exact-threshold IoU separates > from >=; zero-area boxes follow the TF rule; ties follow index order."""
    from tf_faster_rcnn_b200 import ops, _native as N
    # two 10x10(+1) boxes overlapping so that IoU(+1) == 0.5 exactly: inter 11*... use integer construction
    a = [0, 0, 9, 9, 0.9]; b = [0, 5, 9, 14, 0.8]           # +1: areas 100,100, inter 10*5=50 -> 50/150 = 1/3
    dets = np.array([a, b], F)
    third = float(F(50.0) / F(150.0))
    assert list(ops.nms_host(dets, third, N.NMS_MODE_GPU_NMS)) == [0, 1]       # strict: equal is kept
    assert list(ops.nms_host(dets, third, N.NMS_MODE_CPU_NMS)) == [0]          # inclusive: equal is suppressed
    z = np.array([[0, 0, 10, 10, 0.9], [5, 5, 5, 9, 0.8], [0, 0, 10, 10, 0.7]], F)
    assert list(ops.nms_host(z, 0.5, N.NMS_MODE_TF)) == [0, 1]                 # zero-area never suppressed; dup suppressed


def test_nms_host_vs_reference_kernel(cuda):
    """Differential check against the keep lists of the reference's own nms_kernel.cu, compiled as-is and run on a B200
    (golden/make_nms_kernel_golden.py)."""
    from tf_faster_rcnn_b200 import ops, _native as N
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "nms_kernel_vectors.npz"))
    for n in (1, 64, 65, 300, 2000, 6000):
        sd = ref["dets_%d" % n]
        for thr in (0.3, 0.7):
            got = ops.nms_host(sd, thr, N.NMS_MODE_GPU_NMS)
            assert np.array_equal(got, ref["keep_%d_%g" % (n, thr)]), (n, thr)


@pytest.mark.parametrize("hw", [(375, 500), (480, 640), (333, 1200), (601, 799)])
def test_device_preprocess_matches_opencv(cuda, hw):
    """frcnn_preprocess vs the host path (float32(im) - PIXEL_MEANS, cv2.resize INTER_LINEAR): same blob size, <= 1e-4."""
    from tf_faster_rcnn_b200 import ops
    from model.test import _get_image_blob, blob_geometry
    from model.config import cfg
    rng = np.random.default_rng(hw[0])
    im = rng.integers(0, 256, hw + (3,), dtype=np.uint8)
    want, scales = _get_image_blob(im)
    H, W, f = blob_geometry(im.shape)
    assert (H, W) == want.shape[1:3] and f == scales[0]
    blob = torch.empty((1, H, W, 3), dtype=torch.float32, device="cuda")
    ops.preprocess(dev(im), np.asarray(cfg.PIXEL_MEANS).ravel(), f, f, blob)
    err = np.abs(blob.cpu().numpy() - want).max()
    print("\n[preprocess %dx%d -> %dx%d] max abs diff vs OpenCV %.2e" % (hw[0], hw[1], H, W, err))
    assert err < 1e-4


def test_sort_desc_segments(cuda):
    """batch > 1: every segment is sorted on its own cluster, indices are segment-local."""
    from tf_faster_rcnn_b200 import ops
    rng = np.random.default_rng(5)
    B, n = 3, 17100
    keys = rng.random((B, n)).astype(F)
    keys[1, ::3] = F(0.25)
    order = torch.empty(B * n, dtype=torch.int32, device="cuda"); sk = torch.empty(B * n, dtype=torch.float32, device="cuda")
    ops.sort_desc(dev(keys.reshape(-1)), order, sk, batch=B)
    o = order.cpu().numpy().reshape(B, n); k = sk.cpu().numpy().reshape(B, n)
    for b in range(B):
        want = ONMS.argsort_desc(keys[b])
        assert np.array_equal(o[b], want)
        assert np.array_equal(k[b], keys[b][want])


def test_batched_proposal_stages_match_per_image(cuda):
    """rpn_decode -> sort -> proposals -> crop_pool -> bbox_decode -> detect_post on a batch of 3 images equal, bit for bit,
    the same stages run image by image (the per-image arrays are only concatenated; RoI column 0 selects the image)."""
    from tf_faster_rcnn_b200 import ops, _native as N
    rng = np.random.default_rng(77)
    B, A, fh, fw, Cc, R = 3, 9, 38, 50, 21, 300
    n = fh * fw * A
    dcol = (2 * A + 3) // 4 * 4; ld = (dcol + 4 * A + 3) // 4 * 4
    fused = np.zeros((B, fh * fw, ld), F)
    fused[..., :2 * A] = (rng.standard_normal((B, fh * fw, 2 * A)) * 2).astype(F)
    fused[..., dcol:dcol + 4 * A] = (rng.standard_normal((B, fh * fw, 4 * A)) * 0.3).astype(F)
    base = dev(OA.base_anchors(ratios=(0.5, 1, 2), scales=(8, 16, 32)).astype(F))
    feat = rng.standard_normal((B, fh, fw, 64)).astype(F)
    meta = [(1.6, 375, 500), (1.2, 500, 667), (2.0, 300, 400)]
    probs = L.softmax_lastdim((rng.standard_normal((B * R, Cc)) * 2).astype(F))
    deltas = (rng.standard_normal((B * R, 4 * Cc)) * 0.2).astype(F)

    def run(b_lo, b_hi):
        nb = b_hi - b_lo
        scores = torch.empty(nb * n, dtype=torch.float32, device="cuda"); props = torch.empty((nb * n, 4), dtype=torch.float32, device="cuda")
        ops.rpn_decode(dev(fused[b_lo:b_hi].reshape(nb * fh * fw, ld)), dcol, base, A, fh, fw, 600.0, 800.0, scores, props, batch=nb)
        order = torch.empty(nb * n, dtype=torch.int32, device="cuda"); sk = torch.empty(nb * n, dtype=torch.float32, device="cuda")
        ops.sort_desc(scores, order, sk, batch=nb)
        rois = torch.empty((nb * R, 5), dtype=torch.float32, device="cuda"); rs = torch.empty(nb * R, dtype=torch.float32, device="cuda")
        keep = torch.empty(nb * R, dtype=torch.int32, device="cuda"); num = torch.zeros(nb, dtype=torch.int32, device="cuda")
        ops.proposals(props, scores, order, 0, R, 0.7, N.NMS_MODE_TF, rois, rs, keep, num, batch=nb)
        pool = torch.empty((nb * R, 7, 7, 64), dtype=torch.float32, device="cuda")
        ops.crop_pool(dev(feat[b_lo:b_hi]), rois, 7, 0, pool)
        pred = torch.empty((nb * R, 4 * Cc), dtype=torch.float32, device="cuda")
        ops.bbox_decode(rois, dev(deltas[b_lo * R:b_hi * R]), Cc, ops.im_meta_tensor(meta[b_lo:b_hi]), pred)
        det = torch.zeros((nb, 256, 6), dtype=torch.float32, device="cuda"); ndet = torch.zeros(nb, dtype=torch.int32, device="cuda")
        kp = torch.empty((nb, Cc, R), dtype=torch.int32, device="cuda"); cnt = torch.empty((nb, Cc), dtype=torch.int32, device="cuda")
        ks = torch.empty((nb, Cc, R), dtype=torch.float32, device="cuda")
        ops.detect_post(dev(probs[b_lo * R:b_hi * R]), pred, num, Cc, 0.0, float(ONMS.thresh_f32(0.3, True)), N.NMS_MODE_CPU_NMS, 100,
                        det, ndet, kp, cnt, ks, batch=nb)
        torch.cuda.synchronize()
        r = rois.cpu().numpy().reshape(nb, R, 5).copy()
        r[:, :, 0] = 0
        return (r, num.cpu().numpy(), pool.cpu().numpy().reshape(nb, R, 7, 7, 64), pred.cpu().numpy().reshape(nb, R, -1),
                det.cpu().numpy(), ndet.cpu().numpy(), rois.cpu().numpy().reshape(nb, R, 5)[:, :, 0])
    whole = run(0, B)
    for b in range(B):
        one = run(b, b + 1)
        for i in range(6):
            assert np.array_equal(whole[i][b], one[i][0]), (b, i)
        k = int(whole[1][b])
        assert k > 50 and (whole[6][b][:k] == b).all()          # the RoI rows carry their image index
        nd = int(whole[5][b])
        assert 0 < nd <= 256


def test_detect_post_top_mode_5000_rois(cuda):
    """TEST.MODE='top': RPN_TOP_N = 5000 RoIs per image (lib/model/config.py:208) through the fused post path -- the kept
    sets live in the global-memory workspace; records bit-exact against the oracle."""
    from tf_faster_rcnn_b200 import ops, _native as N
    rng = np.random.default_rng(5000)
    R, Cc = 5000, 21
    probs = L.softmax_lastdim((rng.standard_normal((R, Cc)) * 2).astype(F))
    centers = rand_boxes(rng, R, 500.0, (20, 200))
    pred = np.repeat(centers[:, None, :], Cc, axis=1) + rng.uniform(-15, 15, (R, Cc, 4)).astype(F)
    pred = np.round(pred.reshape(R, 4 * Cc)).astype(F)
    want = P.test_net_post(probs, pred, P.opts())
    det = torch.zeros((2048, 6), dtype=torch.float32, device="cuda"); ndet = torch.zeros(1, dtype=torch.int32, device="cuda")
    keep = torch.empty((Cc, R), dtype=torch.int32, device="cuda"); cnt = torch.empty(Cc, dtype=torch.int32, device="cuda")
    ks = torch.empty((Cc, R), dtype=torch.float32, device="cuda")
    nr = torch.tensor([R], dtype=torch.int32, device="cuda")
    ops.detect_post(dev(probs), dev(pred), nr, Cc, 0.0, float(ONMS.thresh_f32(0.3, True)), N.NMS_MODE_CPU_NMS, 100, det, ndet, keep, cnt, ks,
                    workspace=ops.detect_post_workspace(R, Cc))
    nd = int(ndet.item())
    want_flat = np.vstack([np.hstack([d, np.full((d.shape[0], 1), j, F)]) for j, d in enumerate(want) if d.shape[0]])
    assert nd == want_flat.shape[0]
    assert np.array_equal(det.cpu().numpy()[:nd], want_flat)


def test_reference_proposal_layer_modules(cuda):
    """layer_utils.proposal_layer / proposal_layer_tf / proposal_top_layer(_tf): the reference's array-in / array-out entry points,
    device sort + NMS underneath, against the oracle's three proposal modes."""
    from model.config import cfg
    from layer_utils.proposal_layer import proposal_layer, proposal_layer_tf
    from layer_utils.proposal_top_layer import proposal_top_layer, proposal_top_layer_tf
    A, fh, fw = 9, 20, 30
    rng = np.random.default_rng(9)
    cls = (rng.standard_normal((1, fh, fw, 2 * A)) * 2).astype(F)
    box = (rng.standard_normal((1, fh, fw, 4 * A)) * 0.3).astype(F)
    im_info = np.array([320, 480, 1.0], F)
    o = P.opts()
    prob = np.concatenate([1 - P.rpn_fg_prob(cls).reshape(1, fh, fw, A), P.rpn_fg_prob(cls).reshape(1, fh, fw, A)], axis=3).astype(F)
    scores, props, anchors = P.rpn_decode(cls, box, im_info, o)
    saved = (cfg.USE_GPU_NMS, cfg.TEST.RPN_TOP_N)
    try:
        cfg.USE_GPU_NMS = False
        blob, sc = proposal_layer(prob, box, im_info, "TEST", 16, anchors, A)
        want_rois, want_sc, _ = P.proposals_numpy(scores, props, P.opts(use_e2e_tf=False, use_gpu_nms=False))
        assert blob.shape == want_rois.shape and np.abs(blob - want_rois).max() < 1e-3 and np.abs(sc - want_sc).max() < 1e-6
        blob, sc = proposal_layer_tf(prob, box, im_info, "TEST", 16, anchors, A)
        want_rois, want_sc, _ = P.proposals_e2e_tf(scores, props, o)
        assert blob.shape == want_rois.shape and np.abs(blob - want_rois).max() < 1e-3 and np.abs(sc - want_sc).max() < 1e-6
        cfg.TEST.RPN_TOP_N = 2000
        blob, sc = proposal_top_layer_tf(prob, box, im_info, 16, anchors, A)
        want_rois, want_sc, _ = P.proposals_top(scores, props, P.opts(test_mode="top", rpn_top_n=2000))
        assert blob.shape == (2000, 5) and np.abs(blob - want_rois).max() < 1e-3
        blob2, _ = proposal_top_layer(prob, box, im_info, 16, anchors, A)
        assert np.array_equal(blob, blob2)
        cfg.TEST.RPN_TOP_N = 6000                      # more than the 5400 anchors: random fill with replacement, as the reference
        blob3, sc3 = proposal_top_layer(prob, box, im_info, 16, anchors, A)
        assert blob3.shape == (6000, 5) and sc3.shape == (6000, 1)
    finally:
        cfg.USE_GPU_NMS, cfg.TEST.RPN_TOP_N = saved
