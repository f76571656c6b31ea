"""Element-by-element contract of the tcgen05 conv / FC kernel (FP16x3, and the TF32x3 kernel behind impl=CONV_TF32X3).

Every output is checked against a float64 reference with a per-element error bound derived from the kernel's own
arithmetic, instead of one tolerance normalised by the largest output (which lets a small output be wrong by a large
relative amount).  For one output, S = sum |x| |w| over its window (float64, same padding), K = kh*kw*cin.

Raw sum (before the epilogue), for both split kernels (u = 2^-11 is the unit roundoff of an 11-bit significand, fp16 or
tf32):
  * operand split: x = hi + lo*2^-11 + dx with |x - hi| <= u|x| and |dx| <= u|x - hi| <= 2^-22 |x|, the same for w; the
    kernel forms hi*hi + lo*hi + hi*lo and drops lo*lo (<= 2^-22 |x||w|).  Per product at most 3 * 2^-22 |x||w|, so
    3 * 2^-22 * S.  Floor (FP16x3 only): an activation below fp16's normal range has a subnormal hi and lo plane, whose
    spacing 2^-24 leaves 2^-25 * 2^-11 = 2^-36 absolute per activation, i.e. 2^-36 * sum |w| over the window (bounded here
    by the sum over the whole filter).  Weights are scaled by 2^wexp before the split (max|w| * 2^wexp in [2^13, 2^14)),
    which gives the symmetric floor 2^-36 * 2^-wexp * sum |x| over the window.
  * truncating adds in tensor memory: each tcgen05.mma adds into its fp32 accumulator with an error below one ulp, at most
    2^-23 of the partial sum, and a partial sum is at most the S of the terms it holds.  The chunk accumulator D_main takes
    4 MMAs per k-block (64-wide k-blocks of 4 x k16 for FP16x3, 32-wide of 4 x k8 for TF32x3) over kb_per_chunk k-blocks,
    and the chunks partition the sum: 4 * kb_per_chunk * 2^-23 * S.  The cross-term accumulator D_small (magnitude at most
    2u * S = 2^-10 S) takes 8 MMAs per k-block over the whole k range of the unit: 8 * k_blocks_of_unit * 2^-33 * S.
  * round-to-nearest chunk promotion into registers: num_chunks adds of at most 2^-24 * S each, plus one rounding that
    folds D_small in: (num_chunks + 1) * 2^-24 * S.
  * split-K: tail_reduce_kernel adds the split partials in index order, splits - 1 more roundings: (splits - 1) * 2^-24 * S.

Epilogue y = act(raw*scale + shift (+ res)): the raw bound times |scale|, plus one rounding (2^-24 of the running
magnitude, itself inflated by the error so far) per operation.  ReLU / ReLU6 are 1-Lipschitz and add nothing.  The
constants follow from the arithmetic above and are not fitted to any data; each case prints its worst err / bound.

Mutation check: the same cases run with impl = CONV_F16X1, which is the FP16x3 kernel without the lo planes -- an
fp32-claiming kernel that is subtly wrong.  Its error per element is a sum of independent roundings of both operands,
modelled as sigma = 2^-12 / sqrt(3) * sqrt(2 * sum x^2 w^2) (a lower estimate of the rounding-error spread).  Where the
median over all elements of sigma / bound is at least 4 the model predicts a clear violation, and the bound must reject
X1 there.  Those are the cases in MUTATION_CASES (the short-K layers); for long K, X1's error averages down toward the
bound (it grows like sqrt(K) while S grows like K) and the check does not apply.

Activation range: the FP16x3 splitter converts activations to fp16 with round-to-nearest, so the kernel is fp32-grade for
|x| < 65520 and a larger magnitude turns the outputs it feeds into Inf / NaN -- like fp32 arithmetic does for NaN and Inf
inputs.  test_nonfinite_footprint checks that the set of non-finite outputs is exactly the receptive-field footprint of
the poisoned inputs.

The branch table below names the work-decomposition branch each layer exists for; test_branch_table_at_148_sms pins those
branches on the host (no GPU) so that the sweep keeps covering them if decide_geometry's heuristics change.
"""
import ctypes as C
import zlib
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tf_faster_rcnn_b200 import _native as N
from tf_faster_rcnn_b200 import ops

F = np.float32
SMS = 148
GEOM_KEYS = ["block_n", "tile_n", "tile_h", "tile_w", "m_tiles", "n_tiles", "tiles", "split_tiles", "splits", "kb_per_split",
             "units", "grid", "k_blocks", "kb_per_chunk", "tiles_h", "tiles_w"]
IMPL_NAMES = {N.CONV_F16X3: "f16x3", N.CONV_TF32X3: "tf32x3", N.CONV_F16X1: "f16x1"}


def cdiv(a, b):
    return -(-a // b)


def seed(name):
    return zlib.crc32(name.encode())


# ---------------------------------------------------------------------------------------------------------------------
# branch table: name, branch, (n, h, w, cin, cout, k, stride, mode), options, predicate on the 148-SM geometry
def _half_empty_last_split(g, cin, k):
    """odd count of 32-channel blocks (last 64-wide k-block half empty), every tile split, the last split holds that block,
    and a split ends on a chunk shorter than kb_per_chunk"""
    last = g["k_blocks"] - (g["splits"] - 1) * g["kb_per_split"]
    return ((k * k * cin // 32) % 2 == 1 and g["split_tiles"] == g["tiles"] > 0 and g["splits"] > 1 and 0 < last and
            (g["kb_per_split"] % g["kb_per_chunk"] != 0 or last % g["kb_per_chunk"] != 0))


BRANCHES = [
    ("pw_cin32_persistent", "whole tiles, more units than SMs (persistent), single half-empty k-block, BN 64",
     (1, 150, 200, 32, 64, 1, 1, "SAME"), {},
     lambda g: g["split_tiles"] == 0 and g["units"] > SMS and g["k_blocks"] == 1 and g["block_n"] == 64),
    ("c3_halfblock_split", "small layer: every tile split, half-empty k-block in the last split, short last chunk",
     (1, 38, 50, 96, 64, 3, 1, "SAME"), {},
     lambda g: _half_empty_last_split(g, 96, 3) and g["tiles"] <= SMS // 2),
    ("c3_halfblock_split_k3c3", "as above with split_k=3, kb_per_chunk=3 forced",
     (1, 38, 50, 96, 64, 3, 1, "SAME"), {"split_k": 3, "kb_per_chunk": 3},
     lambda g: _half_empty_last_split(g, 96, 3) and g["splits"] == 3 and g["kb_per_chunk"] == 3),
    ("ragged_round", "ragged last round: whole tiles and split tiles in one launch",
     (300, 7, 7, 2048, 512, 1, 1, "SAME"), {"res": True},
     lambda g: g["tiles"] > SMS and 0 < g["split_tiles"] < g["tiles"] and g["units"] > SMS),
    ("tile_n_partial", "tile spans several images, last image group partial, split",
     (19, 7, 7, 512, 512, 3, 1, "SAME"), {},
     lambda g: g["tile_n"] > 1 and 19 % g["tile_n"] != 0 and g["split_tiles"] == g["tiles"]),
    ("s2_explicit_odd", "stride 2, EXPLICIT padding, odd input sizes, odd tile width",
     (1, 75, 101, 32, 64, 3, 2, "EXPLICIT"), {"act": N.ACT_RELU},
     lambda g: g["tile_w"] % 2 == 1 and g["tiles_w"] * g["tile_w"] >= 51 and g["tiles_h"] * g["tile_h"] >= 38),
    ("s2_same_even", "stride 2, SAME padding, even input sizes",
     (1, 76, 100, 32, 64, 3, 2, "SAME"), {},
     lambda g: g["tiles_w"] * g["tile_w"] >= 50 and g["tiles_h"] * g["tile_h"] >= 38 and g["tile_h"] > 1),
    ("pw_s2", "pointwise stride 2 (spatial tiles, not flattened), several N-blocks",
     (1, 38, 50, 256, 512, 1, 2, "SAME"), {"res": True},
     lambda g: g["tile_h"] * g["tiles_h"] >= 19 and g["tiles_h"] > 1 and g["n_tiles"] > 1 and g["split_tiles"] == 0),
    ("generic_epi_105", "cout % 4 != 0 with n_tiles > 1: scalar-tail epilogue, residual + ReLU6",
     (1, 1, 300, 2048, 105, 1, 1, "SAME"), {"block_n": 64, "res": True, "act": N.ACT_RELU6},
     lambda g: g["n_tiles"] > 1 and g["split_tiles"] == 0 and g["block_n"] == 64),
    ("generic_epi_21", "cout % 4 != 0 inside one N-block: scalar-tail epilogue, residual + ReLU6",
     (1, 1, 300, 2048, 21, 1, 1, "SAME"), {"res": True, "act": N.ACT_RELU6},
     lambda g: g["n_tiles"] == 1 and g["split_tiles"] == 0),
    ("cout36", "cout % 4 == 0, not a multiple of 32: partial N-block through the split reduce",
     (1, 38, 50, 128, 36, 3, 1, "SAME"), {"res": True},
     lambda g: g["split_tiles"] == g["tiles"] and g["n_tiles"] * g["block_n"] > 36),
    ("cout72", "cout % 4 == 0, not a multiple of 32, flattened pointwise, split",
     (1, 19, 25, 512, 72, 1, 1, "SAME"), {"act": N.ACT_RELU},
     lambda g: g["split_tiles"] == g["tiles"] and g["tile_h"] == 1 and g["n_tiles"] * g["block_n"] > 72),
    ("cout324", "cout % 4 == 0, not a multiple of 32, three N-blocks, split",
     (1, 1, 300, 1024, 324, 1, 1, "SAME"), {"res": True},
     lambda g: g["n_tiles"] == 3 and g["split_tiles"] == g["tiles"]),
    ("k5", "5x5 filter",
     (2, 20, 30, 64, 96, 5, 1, "SAME"), {},
     lambda g: g["k_blocks"] == 25),
    ("raster_split", "several N- and M-blocks, every tile split (raster order matters)",
     (1, 38, 50, 64, 256, 3, 1, "SAME"), {},
     lambda g: g["n_tiles"] > 1 and g["m_tiles"] > 1 and g["split_tiles"] == g["tiles"]),
]
BY_NAME = {b[0]: b for b in BRANCHES}
# the cases where the X1 error model predicts >= 4x the bound (median over elements), see the module docstring
MUTATION_CASES = {"pw_cin32_persistent", "c3_halfblock_split_k3c3", "s2_explicit_odd", "s2_same_even", "pw_s2", "cout72",
                  "raster_split"}
RASTER_CASES = ["pw_s2", "raster_split"]


def layer_geom(shape):
    n, h, w, cin, cout, k, stride, mode = shape
    ho, wo, pt, pl = ops.conv_out_hw(h, w, k, stride, mode)
    return ho, wo, pt, pl


def geometry(shape, impl, opts, sms=SMS):
    n, h, w, cin, cout, k, stride, mode = shape
    ho, wo, pt, pl = layer_geom(shape)
    d = N.ConvDesc(None, None, None, None, None, None, None, n, h, w, cin, cout, k, k, stride, pt, pl, ho, wo, opts.get("act", 0),
                   opts.get("block_n", 0), opts.get("kb_per_chunk", 0), opts.get("split_k", 0), impl, 1.0)
    out = (C.c_int * 16)()
    N.check(N.lib().frcnn_conv_plan_geometry(C.byref(d), sms, out), "geometry")
    return dict(zip(GEOM_KEYS, list(out)))


def test_branch_table_at_148_sms():
    """CPU: every row of the branch table hits the branch it names on a 148-SM B200."""
    for name, branch, shape, opts, pred in BRANCHES:
        g = geometry(shape, N.CONV_F16X3, opts)
        assert pred(g), "%s no longer covers '%s': %s" % (name, branch, g)
    cout = [BY_NAME[c][2][4] for c in ("generic_epi_105", "generic_epi_21", "cout36", "cout72", "cout324")]
    assert [c % 4 != 0 for c in cout] == [True, True, False, False, False] and all(c % 32 for c in cout)


# ---------------------------------------------------------------------------------------------------------------------
# float64 references and the bound
def conv64(x, w, stride, pt, pl, ho, wo):
    xt = torch.from_numpy(np.asarray(x, np.float64)).permute(0, 3, 1, 2)
    wt = torch.from_numpy(np.asarray(w, np.float64)).permute(3, 2, 0, 1)
    kh, kw = w.shape[:2]
    h, wd = x.shape[1:3]
    pb = max((ho - 1) * stride + kh - h - pt, 0)
    pr = max((wo - 1) * stride + kw - wd - pl, 0)
    xt = torch.nn.functional.pad(xt, (pl, pr, pt, pb))
    return torch.nn.functional.conv2d(xt, wt, None, stride=stride).permute(0, 2, 3, 1).numpy()[:, :ho, :wo]


class Ref:
    """float64 raw sums of one layer and what the bound needs: S = conv(|x|, |w|), the activation and weight floors."""

    def __init__(self, x, w, stride, pt, pl, ho, wo, want_q=False):
        self.geo = (stride, pt, pl, ho, wo)
        ax, aw = np.abs(x.astype(np.float64)), np.abs(w.astype(np.float64))
        self.raw = conv64(x, w, *self.geo)
        self.S = conv64(ax, aw, *self.geo)
        self.xsum = conv64(ax, np.ones(w.shape[:3] + (1,)), *self.geo)          # sum |x| over the window
        self.wsum = aw.sum(axis=(0, 1, 2))                                        # sum |w| over the filter, per cout
        self.wexp = ops.weight_exponent(w)
        self.Q = conv64(x.astype(np.float64) ** 2, w.astype(np.float64) ** 2, *self.geo) if want_q else None


def raw_bound(ref, g, impl):
    kpc, nkb, splits = g["kb_per_chunk"], g["k_blocks"], g["splits"]
    kb_unit = nkb if g["split_tiles"] < g["tiles"] else g["kb_per_split"]   # longest k range of one unit
    chunks = cdiv(kb_unit, kpc)
    rel = 3 * 2.0 ** -22 + 4 * kpc * 2.0 ** -23 + 8 * kb_unit * 2.0 ** -33 + (chunks + 1 + splits - 1) * 2.0 ** -24
    b = rel * ref.S
    if impl != N.CONV_TF32X3:
        b = b + 2.0 ** -36 * ref.wsum + 2.0 ** -36 * 2.0 ** -ref.wexp * ref.xsum
    return b


def act64(a, act):
    if act == N.ACT_RELU:
        return np.maximum(a, 0.0)
    if act == N.ACT_RELU6:
        return np.minimum(np.maximum(a, 0.0), 6.0)
    return a


def epilogue64(raw, rb, scale, shift, res, act):
    """exact y and its bound: raw bound times |scale|, then one fp32 rounding per epilogue operation"""
    u = 2.0 ** -24
    sc = np.ones(raw.shape[-1]) if scale is None else scale.astype(np.float64)
    a = raw * sc
    e = np.abs(sc) * rb
    e = e + u * (np.abs(a) + e)
    if shift is not None:
        a = a + shift.astype(np.float64)
        e = e + u * (np.abs(a) + e)
    if res is not None:
        a = a + res.astype(np.float64)
        e = e + u * (np.abs(a) + e)
    return act64(a, act), e


def ratio(got, want, bound):
    err = np.abs(got.astype(np.float64) - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(bound > 0, err / bound, np.where(err > 0, np.inf, 0.0))
    r[~np.isfinite(got)] = np.inf
    return r


def run_plan(x, w, impl, shape, scale=None, shift=None, res=None, act=0, block_n=0, kb_per_chunk=0, split_k=0):
    n, h, wd, cin, cout, k, stride, mode = shape
    ho, wo, pt, pl = layer_geom(shape)
    pc = ops.PackedConv(w, scale, shift, impl=impl)
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    out = torch.full((n, ho, wo, cout), float("nan"), dtype=torch.float32, device="cuda")
    rd = None if res is None else torch.from_numpy(np.ascontiguousarray(res)).cuda()
    plan = ops.ConvPlan(xd, pc, out, stride, pt, pl, act, rd, block_n, kb_per_chunk, split_k)
    plan.run()
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.fixture(scope="module")
def b200(cuda):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != SMS:
        pytest.skip("the branch table is laid out for %d SMs, this device has %d" % (SMS, sms))
    return sms


def make_layer(name, shape, opts):
    n, h, w, cin, cout, k, stride, mode = shape
    ho, wo, pt, pl = layer_geom(shape)
    rng = np.random.default_rng(seed(name))
    x = rng.standard_normal((n, h, w, cin)).astype(F)
    wt = (rng.standard_normal((k, k, cin, cout)) * np.sqrt(2.0 / (k * k * cin))).astype(F)
    scale = np.exp(rng.uniform(np.log(1e-3), np.log(1e3), cout)).astype(F)
    shift = rng.standard_normal(cout).astype(F)
    res = rng.standard_normal((n, ho, wo, cout)).astype(F) if opts.get("res") else None
    return x, wt, scale, shift, res


# ---------------------------------------------------------------------------------------------------------------------
# (c) branch sweep, F16X3 and TF32X3, with the X1 mutation check
@pytest.mark.gpu
@pytest.mark.parametrize("name", [b[0] for b in BRANCHES])
def test_branch_sweep(b200, name):
    _, branch, shape, opts, pred = BY_NAME[name]
    x, wt, scale, shift, res = make_layer(name, shape, opts)
    ho, wo, pt, pl = layer_geom(shape)
    ref = Ref(x, wt, shape[6], pt, pl, ho, wo, want_q=True)
    act = opts.get("act", 0)
    kw = dict(block_n=opts.get("block_n", 0), kb_per_chunk=opts.get("kb_per_chunk", 0), split_k=opts.get("split_k", 0))
    g16 = geometry(shape, N.CONV_F16X3, opts)
    assert pred(g16), "%s: plan %s is not the branch '%s'" % (name, g16, branch)
    for impl in (N.CONV_F16X3, N.CONV_TF32X3):
        g = geometry(shape, impl, opts)
        want, bound = epilogue64(ref.raw, raw_bound(ref, g, impl), scale, shift, res, act)
        got = run_plan(x, wt, impl, shape, scale, shift, res, act, **kw)
        r = ratio(got, want, bound)
        worst = np.unravel_index(np.argmax(r), r.shape)
        print("\n[%s %s] %s  worst err/bound %.3f at %s" % (name, IMPL_NAMES[impl], branch, r.max(), worst))
        assert r.max() <= 1.0, (name, IMPL_NAMES[impl], g, float(r.max()), worst)
    # mutation: X1 drops the lo planes; the bound must reject it wherever the model predicts a clear violation
    want, bound = epilogue64(ref.raw, raw_bound(ref, g16, N.CONV_F16X3), scale, shift, res, act)
    sigma = 2.0 ** -12 / np.sqrt(3.0) * np.sqrt(2.0 * ref.Q) * np.abs(scale.astype(np.float64))
    predicted = float(np.median(sigma / bound))
    got = run_plan(x, wt, N.CONV_F16X1, shape, scale, shift, res, act, **kw)
    r = ratio(got, want, bound)
    print("[%s f16x1] predicted sigma/bound (median) %.2f  worst err/bound %.2f" % (name, predicted, r.max()))
    assert (predicted >= 4.0) == (name in MUTATION_CASES), (name, predicted)
    if name in MUTATION_CASES:
        assert r.max() > 1.0, "the bound accepts the lo-plane-free kernel on %s (worst %.2f)" % (name, r.max())


# ---------------------------------------------------------------------------------------------------------------------
# (d) operand range, FP16x3
RANGE_SHAPE = (1, 20, 30, 64, 64, 3, 1, "SAME")


def _range_inputs(kind, rng):
    n, h, w, cin, cout, k = RANGE_SHAPE[:6]
    x = rng.standard_normal((n, h, w, cin))
    wt = rng.standard_normal((k, k, cin, cout)) * np.sqrt(2.0 / (k * k * cin))
    if kind.startswith("x_2^"):
        x = np.clip(x * 2.0 ** int(kind[4:]), -65504.0, 65504.0)
    elif kind == "x_channels_2^-12..2^12":
        x = x * 2.0 ** np.linspace(-12, 12, cin)
    elif kind == "x_65504_65519":
        flat = x.reshape(-1)
        idx = rng.choice(flat.size, 64, replace=False)
        flat[idx] = np.tile([65504.0, -65504.0, 65519.0, -65519.0], 16)
    elif kind == "w_max_pow2":
        wt = np.clip(wt, -0.49, 0.49)
        wt.reshape(-1)[7] = -0.5
    elif kind == "w_max_below_pow2":
        wt = np.clip(wt, -0.49, 0.49)
        wt.reshape(-1)[7] = np.nextafter(F(0.5), F(0))
    elif kind == "w_one_large":
        wt = wt * 1e-6
        wt.reshape(-1)[123] = 1.0
    return x.astype(F), wt.astype(F)


RANGE_KINDS = ["x_2^-16", "x_2^-8", "x_2^0", "x_2^8", "x_2^14", "x_channels_2^-12..2^12", "x_65504_65519",
               "w_max_pow2", "w_max_below_pow2", "w_one_large"]


def test_range_inputs_are_what_they_claim():
    """CPU: the operand-range fixtures hit their edges (fp16 range of x, power-of-two edges of weight_exponent)."""
    for kind in RANGE_KINDS:
        x, wt = _range_inputs(kind, np.random.default_rng(seed(kind)))
        assert np.abs(x).max() <= 65519.0
        m = float(np.abs(wt).max())
        assert 2 ** 13 <= m * 2.0 ** ops.weight_exponent(wt) < 2 ** 14
        if kind == "x_2^14":
            assert 2.0 ** 15 < np.abs(x).max() <= 65504.0    # the top binade of fp16
        if kind == "x_2^-16":
            assert (np.abs(x) < 2.0 ** -14).mean() > 0.99  # activations below fp16's normal range
        if kind == "w_max_pow2":
            assert m == 0.5
        if kind == "w_max_below_pow2":
            assert m == np.nextafter(F(0.5), F(0)) and ops.weight_exponent(wt) == 15


@pytest.mark.gpu
@pytest.mark.parametrize("kind", RANGE_KINDS)
def test_operand_range(b200, kind):
    rng = np.random.default_rng(seed(kind))
    x, wt = _range_inputs(kind, rng)
    shape = RANGE_SHAPE
    ho, wo, pt, pl = layer_geom(shape)
    cout = shape[4]
    scale = np.exp(rng.uniform(np.log(1e-3), np.log(1e3), cout)).astype(F)
    shift = rng.standard_normal(cout).astype(F)
    ref = Ref(x, wt, 1, pt, pl, ho, wo)
    g = geometry(shape, N.CONV_F16X3, {})
    want, bound = epilogue64(ref.raw, raw_bound(ref, g, N.CONV_F16X3), scale, shift, None, 0)
    got = run_plan(x, wt, N.CONV_F16X3, shape, scale, shift)
    r = ratio(got, want, bound)
    print("\n[range %s] max|x| %.3g max|w| %.9g  worst err/bound %.3f" % (kind, np.abs(x).max(), np.abs(wt).max(), r.max()))
    assert r.max() <= 1.0, (kind, float(r.max()))


# ---------------------------------------------------------------------------------------------------------------------
# (e) non-finite footprint, FP16x3
# (n, h, w, c) input positions per layer: corners, tile seams (spatial, and between the images of a tile_n > 1 tile), the
# last channel of the half-empty k-block, pixels that no output reads (odd rows / columns of the 1x1 stride-2 layer).  On
# the persistent layer, pixel 0 lies in unit 0: CTA 0 runs unit 148 afterwards, which must stay clean.
POISON = {
    "pw_cin32_persistent": [(0, 0, 0, 3), (0, 0, 199, 31), (0, 149, 0, 0), (0, 149, 199, 17), (0, 0, 127, 5), (0, 0, 128, 6),
                            (0, 75, 100, 31)],
    "c3_halfblock_split": [(0, 0, 0, 95), (0, 37, 49, 0), (0, 4, 24, 64), (0, 5, 25, 95), (0, 20, 30, 95)],
    "tile_n_partial": [(0, 3, 3, 0), (1, 0, 0, 511), (17, 6, 6, 100), (18, 6, 6, 7), (18, 0, 0, 255)],
    "s2_explicit_odd": [(0, 0, 0, 0), (0, 74, 100, 31), (0, 1, 1, 16), (0, 37, 50, 2)],
    "pw_s2": [(0, 1, 1, 5), (0, 37, 49, 255), (0, 2, 4, 0), (0, 36, 48, 255)],
}
POISON_VALUES = [("nan", np.nan), ("+inf", np.inf), ("-inf", -np.inf), ("7e4", 7e4), ("-65520", -65520.0)]
_clean_cache = {}


def _clean(name):
    if name not in _clean_cache:
        shape = BY_NAME[name][2]
        x, wt, scale, shift, _ = make_layer(name, shape, {})
        ho, wo, pt, pl = layer_geom(shape)
        _clean_cache[name] = (x, wt, scale, shift, Ref(x, wt, shape[6], pt, pl, ho, wo))
    return _clean_cache[name]


def _footprint(shape, pos):
    """outputs whose window covers any poisoned pixel (all output channels): a float64 conv of the indicator"""
    n, h, w, cin, cout, k, stride, mode = shape
    ho, wo, pt, pl = layer_geom(shape)
    m = np.zeros((n, h, w, 1))
    for (i, y, xx, c) in pos:
        m[i, y, xx, 0] = 1.0
    return conv64(m, np.ones((k, k, 1, 1)), stride, pt, pl, ho, wo)[..., 0] > 0


def _add_pixel(out, shape, wt, i, y, xx, c, dv):
    """out += contribution dv * w of one input pixel / channel (exact loop over the taps that read it)"""
    k, stride = shape[5], shape[6]
    ho, wo, pt, pl = layer_geom(shape)
    for r in range(k):
        for s in range(k):
            oy, ox = y + pt - r, xx + pl - s
            if oy % stride or ox % stride:
                continue
            oy //= stride; ox //= stride
            if 0 <= oy < ho and 0 <= ox < wo:
                out[i, oy, ox] += dv * wt[r, s, c].astype(np.float64)


@pytest.mark.gpu
@pytest.mark.parametrize("value", [v[0] for v in POISON_VALUES])
@pytest.mark.parametrize("name", list(POISON))
def test_nonfinite_footprint(b200, name, value):
    val = dict(POISON_VALUES)[value]
    shape = BY_NAME[name][2]
    x, wt, scale, shift, ref = _clean(name)
    pos = POISON[name]
    xp = x.copy()
    for p in pos:
        xp[p] = val
    fp = _footprint(shape, pos)
    fp_all = np.broadcast_to(fp[..., None], ref.raw.shape)
    g = geometry(shape, N.CONV_F16X3, {})
    raw, S, xsum = ref.raw.copy(), ref.S.copy(), ref.xsum.copy()
    if np.isfinite(val):                      # the exact sums with the finite out-of-range value in place
        for (i, y, xx, c) in pos:
            _add_pixel(raw, shape, wt, i, y, xx, c, float(val) - float(x[i, y, xx, c]))
            _add_pixel(S, shape, np.abs(wt), i, y, xx, c, abs(float(val)) - abs(float(x[i, y, xx, c])))
            _add_pixel(xsum, shape, np.ones(wt.shape[:3] + (1,)), i, y, xx, c, abs(float(val)) - abs(float(x[i, y, xx, c])))
    ref_p = SimpleNamespace(raw=raw, S=S, xsum=xsum, wsum=ref.wsum, wexp=ref.wexp)
    want, bound = epilogue64(raw, raw_bound(ref_p, g, N.CONV_F16X3), scale, shift, None, 0)
    got = run_plan(xp, wt, N.CONV_F16X3, shape, scale, shift)
    bad = ~np.isfinite(got)
    r = ratio(got, want, bound)
    inside_finite_ok = np.isfinite(got) & (r <= 1.0)
    print("\n[%s %s] footprint %d outputs, non-finite %d (%d outside the footprint), finite in the footprint %d "
          "(%d beyond the bound, worst err/bound %.3g), worst err/bound outside %.3f" %
          (name, value, int(fp_all.sum()), int(bad.sum()), int((bad & ~fp_all).sum()), int((~bad & fp_all).sum()),
           int((~bad & fp_all & ~inside_finite_ok).sum()), float(np.where(fp_all & ~bad, r, 0).max()),
           float(np.where(fp_all, 0, r).max())))
    assert not (bad & ~fp_all).any(), "non-finite outputs outside the receptive-field footprint"
    assert np.where(fp_all, 0, r).max() <= 1.0, "outputs outside the footprint beyond the bound"
    if not np.isfinite(val):
        assert np.array_equal(bad, fp_all), "a NaN / Inf input must make every output of its footprint non-finite"
    else:
        assert (bad | inside_finite_ok)[fp_all].all(), "finite but wrong outputs from an out-of-range activation"


# ---------------------------------------------------------------------------------------------------------------------
# forced raster order, and chained plans on one stream
@pytest.mark.gpu
@pytest.mark.parametrize("name", RASTER_CASES)
def test_raster_forced_m_vs_n(b200, name, monkeypatch):
    """FRCNN_CONV_RASTER (read at plan creation) only reorders the tiles over the CTAs: the results are bit-identical."""
    _, branch, shape, opts, pred = BY_NAME[name]
    assert geometry(shape, N.CONV_F16X3, opts)["n_tiles"] > 1
    x, wt, scale, shift, res = make_layer(name, shape, opts)
    outs = {}
    for order in ("m", "n"):
        monkeypatch.setenv("FRCNN_CONV_RASTER", order)
        outs[order] = run_plan(x, wt, N.CONV_F16X3, shape, scale, shift, res)
    monkeypatch.delenv("FRCNN_CONV_RASTER")
    ho, wo, pt, pl = layer_geom(shape)
    ref = Ref(x, wt, shape[6], pt, pl, ho, wo)
    want, bound = epilogue64(ref.raw, raw_bound(ref, geometry(shape, N.CONV_F16X3, opts), N.CONV_F16X3), scale, shift, res, 0)
    print("\n[raster %s] worst err/bound %.3f" % (name, ratio(outs["m"], want, bound).max()))
    assert ratio(outs["m"], want, bound).max() <= 1.0
    assert np.array_equal(outs["m"], outs["n"], equal_nan=True)


@pytest.mark.gpu
def test_chained_bottleneck_pdl(b200):
    """A ResNet bottleneck (1x1 -> 3x3 -> 1x1 + shortcut, BN + ReLU) enqueued back to back on one stream (programmatic
    dependent launch: each kernel starts before its producer finished) equals the same plans with a synchronize between
    them, bit for bit; every stage meets the bound against float64 of its own input."""
    rng = np.random.default_rng(7)
    n, h, w, c, m = 1, 38, 50, 256, 64
    x = rng.standard_normal((n, h, w, c)).astype(F)
    specs = [(1, c, m), (3, m, m), (1, m, c)]
    layers = []
    for k, ci, co in specs:
        wt = (rng.standard_normal((k, k, ci, co)) * np.sqrt(2.0 / (k * k * ci))).astype(F)
        layers.append((k, wt, rng.uniform(0.5, 2.0, co).astype(F), rng.standard_normal(co).astype(F)))
    xd = torch.from_numpy(x).cuda()
    t1 = torch.empty((n, h, w, m), device="cuda")
    t2 = torch.empty((n, h, w, m), device="cuda")
    out = torch.empty((n, h, w, c), device="cuda")
    bufs = [(xd, t1, None), (t1, t2, None), (t2, out, xd)]
    plans = []
    for (k, wt, sc, sh), (src, dst, res) in zip(layers, bufs):
        pc = ops.PackedConv(wt, sc, sh, impl=N.CONV_F16X3)
        plans.append(ops.ConvPlan(src, pc, dst, 1, k // 2, k // 2, N.ACT_RELU, res))
    results = []
    for sync_between in (False, True):
        for t in (t1, t2, out):
            t.fill_(float("nan"))
        torch.cuda.synchronize()
        for p in plans:
            p.run()
            if sync_between:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        results.append([t.cpu().numpy() for t in (t1, t2, out)])
    for a, b in zip(*results):
        assert np.isfinite(a).all() and np.array_equal(a, b)
    ins = [x, results[1][0], results[1][1]]
    for i, ((k, wt, sc, sh), src) in enumerate(zip(layers, ins)):
        shape = (n, h, w, wt.shape[2], wt.shape[3], k, 1, "SAME")
        ref = Ref(src, wt, 1, k // 2, k // 2, h, w)
        want, bound = epilogue64(ref.raw, raw_bound(ref, geometry(shape, N.CONV_F16X3, {}), N.CONV_F16X3), sc, sh,
                                 x if i == 2 else None, N.ACT_RELU)
        r = ratio(results[1][i], want, bound)
        print("\n[bottleneck stage %d] worst err/bound %.3f" % (i, r.max()))
        assert r.max() <= 1.0
