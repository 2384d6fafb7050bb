"""Generic layer kernels and CUDA-core fallbacks at cfg shapes the shipped models never reach.

Every GPU case builds one tiny cfg: a [net] block, producer layers that give the layer under test its input shapes, then the
layer under test, with seeded weights (synth.write_weights, damp_heads=False).  The batch is 3.  The producers' outputs are
teacher-forced with set_layer_output (values of both signs, plus an all-negative plane; rounded to bf16 first when the
buffer is bf16), only the layer under test runs (run_layers(i, i + 1)), and every image of its output is compared with the
float64 restatements of tests/np_layers.py.  Each case asserts the kernel the planner chose (net.kernel), and where a sub-branch
is invisible there, the dispatch predicate it mirrors.

Comparison rules:
  * copy, max, select and permutation kernels (maxpool, upsample, route, reorg, and shortcut in fp32 mode): bit-exact against
    the fp32 restatement.  In bf16 mode the expected value is the bf16 rounding of the restatement computed in the kernel's
    operation order, leaky as 0.1f * x (common.cuh apply_act with EXACT = false).
  * sums (convolution, local, connected): per element
        |got - ref64| <= slope(act) * (K + 2) * 2^-24 * (sum_k |w_k x_k| * |scale| + |shift|)
                         + 2^-23 * |ref64| + half an ulp of the output dtype at ref64 + 2^-126,
    with the weights and inputs as the device holds them (bf16-rounded in bf16 mode).  A missing or wrong tap moves an element
    by about sum / K, far outside this bound.
  * avgpool: hw * 2^-24 * mean|x| + 2^-24 * |ref64| + the output rounding.
  * logistic, softmax: at most 2 fp32 ulp from the float64 restatement, plus, for a softmax, the worst-case rounding of its
    fp32 sum (2^-24 per level of the kernel's reduction: the values one thread adds serially, then the shuffle / CTA tree).
    Probabilities are zero in exactly the places where the restatement rounds to zero in fp32.
"""

import numpy as np
import pytest

import np_classifier as C
import np_layers as NL
from yolo_tensorflow_b200 import synth

gpu = pytest.mark.gpu
BATCH = 3
F32, F64 = np.float32, np.float64


# ---------------------------------------------------------------------------------------------------
# harness
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dn():
    from yolo_tensorflow_b200 import darknet
    return darknet


def cfg_text(h, w, c, body, batch=BATCH):
    return "[net]\nbatch=%d\nheight=%d\nwidth=%d\nchannels=%d\n%s" % (batch, h, w, c, body)


def write_case(tmp_path, text, seed=11):
    cfg = tmp_path / "case.cfg"
    cfg.write_text(text)
    w = str(tmp_path / "case.weights")
    synth.write_weights(str(cfg), w, seed=seed, damp_heads=False)
    return str(cfg), w


def open_case(dn, cfg, w, prec):
    return dn.Network(cfg, w, precision=dn.PREC_BF16 if prec == "bf16" else dn.PREC_FP32, fuse=False)


def sources(L, i):
    if L.type == "route":
        return L.src
    if L.type == "shortcut":
        return [i - 1, L.src]
    return [i - 1]


def out_shape(L, batch):
    if L.out_h and L.out_w and L.type not in ("connected", "softmax", "yolo", "region", "detection"):
        return (batch, L.out_c, L.out_h, L.out_w)
    return (batch, L.outputs)


def fp32_buffer(port, j):
    """does layer j's device buffer hold fp32 in bf16 mode (heads, [connected], [softmax], and what aliases them)?"""
    L = port.layers[j]
    if L.type == "dropout":
        return fp32_buffer(port, j - 1)
    return L.type in ("connected", "softmax", "yolo", "region", "detection")


def sample(rng, shape, scale=1.):
    """both signs; in every image the first channel plane is all negative"""
    x = (rng.standard_normal(shape) * scale).astype(F32)
    if len(shape) == 4:
        x[:, 0] = -np.abs(x[:, 0]) - F32(.25)
    return x


def force(net, port, i, prec, rng, make=None):
    """teacher-force the sources of layer i, run it alone; returns ({source: input}, output [batch, outputs])"""
    xs = {}
    for j in sources(port.layers[i], i):
        shape = out_shape(port.layers[j], net.batch)
        x = make(shape) if make else sample(rng, shape)
        if prec == "bf16" and not fp32_buffer(port, j):
            x = NL.bf16(x)
        net.set_layer_output(j, x.reshape(net.batch, -1))
        xs[j] = x
    net.run_layers(i, i + 1)
    return xs, net.layer_output(i)


def case(dn, tmp_path, prec, h, w, c, body, batch=BATCH, seed=11):
    cfg, wpath = write_case(tmp_path, cfg_text(h, w, c, body, batch), seed)
    port = C.Net(cfg, wpath)
    return open_case(dn, cfg, wpath, prec), port


def expect_exact(got, want, prec, what=""):
    want = NL.bf16(want) if prec == "bf16" else np.asarray(want, F32)
    want = want.reshape(got.shape)
    bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32)) if got.dtype == F32 else []
    assert np.array_equal(got, want), (what, len(bad), bad[:4], got.flat[0], want.flat[0])


def expect_sum(got, y64, mag, K, act, bf_out, what=""):
    ref = NL.act64(y64, act).reshape(got.shape)
    pre = NL.act_slope(act) * (K + 2) * NL.U * mag.reshape(got.shape)
    bound = pre + 2 * NL.U * np.abs(ref) + NL.half_ulp(np.abs(ref) + pre, bf_out) + 2.0 ** -126
    err = np.abs(got.astype(F64) - ref)
    k = np.unravel_index(np.argmax(err - bound), err.shape)
    assert (err <= bound).all(), (what, k, float(got[k]), float(ref[k]), float(err[k]), float(bound[k]))
    return err


def expect_probs(got, p64, depth, what=""):
    p64 = p64.reshape(got.shape)
    bound = 4 * NL.half_ulp(p64, False) + depth * NL.U * np.abs(p64)
    err = np.abs(got.astype(F64) - p64)
    k = np.unravel_index(np.argmax(err - bound), err.shape)
    assert (err <= bound).all(), (what, k, float(got[k]), float(p64[k]), float(err[k]))
    assert np.array_equal(got == 0, p64.astype(F32) == 0), what


def weights_of(L, prec):
    """the layer's weights as the device holds them, and its folded (scale, shift) in float64"""
    w = NL.bf16(L.weights) if prec == "bf16" else L.weights
    if L.get("bn"):
        return w, NL.fold64(L.biases, L.scales, L.mean, L.var)
    return w, NL.fold64(L.biases)


PRECS = ["fp32", "bf16"]
MP1 = "[maxpool]\nsize=1\nstride=1\n"                   # a producer that keeps the [net] shape
# convolutional producers read 8 input channels, so they plan on CUDA cores: only the layer under test uses tcgen05


# ---------------------------------------------------------------------------------------------------
# maxpool: general maxpool_kernel, VEC and VEC = 1 (layers.cu:154-166)
# ---------------------------------------------------------------------------------------------------
MAXPOOL = {
    "2s2_odd_13x27": (13, 27, 16, "size=2\nstride=2\n"),
    "3s2_15x15": (15, 15, 16, "size=3\nstride=2\n"),
    "3s2_16x16": (16, 16, 16, "size=3\nstride=2\n"),
    "5s1_13x13x512": (13, 13, 512, "size=5\nstride=1\n"),
    "9s1_13x13x512": (13, 13, 512, "size=9\nstride=1\n"),
    "13s1_13x13x512": (13, 13, 512, "size=13\nstride=1\n"),
    "3s1_pad0": (9, 11, 16, "size=3\nstride=1\npadding=0\n"),
    "c6": (10, 10, 6, "size=3\nstride=2\n"),
    "c20": (11, 11, 20, "size=2\nstride=2\n"),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(MAXPOOL))
def test_maxpool(dn, tmp_path, prec, name):
    h, w, c, opts = MAXPOOL[name]
    net, port = case(dn, tmp_path, prec, h, w, c, MP1 + "[maxpool]\n" + opts)
    L = port.layers[1]
    assert net.kernel(1) == "maxpool"
    V = 8 if prec == "bf16" else 4
    fast = c % V == 0 and L.size == 2 and L.stride == 2 and L.pad == 0 and h == 2 * L.out_h and w == 2 * L.out_w
    assert not fast                                                   # maxpool_dispatch, layers.cu:154: not the 2x2 kernel
    xs, got = force(net, port, 1, prec, np.random.default_rng(1))
    if name.startswith(("5s1", "9s1", "13s1")):
        assert (L.out_h, L.out_w) == {5: (17, 17), 9: (21, 21), 13: (25, 25)}[L.size]
    want = NL.maxpool(xs[0], L.size, L.stride, L.pad, L.out_h, L.out_w)
    expect_exact(got, want.reshape(BATCH, -1), prec, name)
    net.close()


# ---------------------------------------------------------------------------------------------------
# upsample: vector and scalar upsample_kernel (layers.cu:206)
# ---------------------------------------------------------------------------------------------------
UPSAMPLE = {
    "s2_c16": (5, 7, 16, "stride=2\n"),
    "s3_c6": (5, 4, 6, "stride=3\n"),
    "s4_half_c24": (3, 5, 24, "stride=4\nscale=0.5\n"),
    "s2_x3_c24": (4, 4, 24, "stride=2\nscale=3\n"),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(UPSAMPLE))
def test_upsample(dn, tmp_path, prec, name):
    h, w, c, opts = UPSAMPLE[name]
    net, port = case(dn, tmp_path, prec, h, w, c, MP1 + "[upsample]\n" + opts)
    L = port.layers[1]
    assert net.kernel(1) == "upsample"
    xs, got = force(net, port, 1, prec, np.random.default_rng(2))
    expect_exact(got, NL.upsample(xs[0], L.stride, L.scale).reshape(BATCH, -1), prec, name)
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
def test_upsample_into_a_concat_slice(dn, tmp_path, prec):
    """the upsample writes its channel slice of the route's buffer (row pitch 32, first channel 0)"""
    body = MP1 + "[maxpool]\nsize=2\nstride=2\n[upsample]\nstride=2\n[route]\nlayers=-1,-3\n"
    net, port = case(dn, tmp_path, prec, 8, 8, 16, body)
    assert net.kernel(2) == "upsample" and net.kernel(3) == "concat_in_place"
    xs, got = force(net, port, 2, prec, np.random.default_rng(3))
    expect_exact(got, NL.upsample(xs[1], 2, 1.).reshape(BATCH, -1), prec)
    net.close()


# ---------------------------------------------------------------------------------------------------
# shortcut: shortcut_same_kernel (VEC and VEC = 1), shortcut_general_kernel (layers.cu:243-287)
# ---------------------------------------------------------------------------------------------------
SHORTCUT = {
    # name: (h, w, c, producers, shortcut options, index of the layer under test)
    "same_leaky": (8, 8, 16, MP1 + MP1, "from=-2\nalpha=.5\nbeta=2\nactivation=leaky\n", 2),
    "same_relu": (8, 8, 16, MP1 + MP1, "from=-2\nalpha=.5\nbeta=2\nactivation=relu\n", 2),
    "same_logistic": (8, 8, 16, MP1 + MP1, "from=-2\nalpha=.5\nbeta=2\nactivation=logistic\n", 2),
    "same_c6": (7, 5, 6, MP1 + MP1, "from=-2\nalpha=.5\nbeta=2\nactivation=leaky\n", 2),
    "add_larger": (16, 16, 16, MP1 + "[maxpool]\nsize=2\nstride=2\n", "from=-2\nactivation=leaky\n", 2),
    "add_smaller": (8, 8, 16, MP1 + "[maxpool]\nsize=2\nstride=2\n[upsample]\nstride=2\n", "from=-2\nactivation=linear\n", 3),
    "add_fewer_channels": (6, 6, 8, "[convolutional]\nfilters=8\nsize=1\nactivation=linear\n"
                                     "[convolutional]\nfilters=16\nsize=1\nactivation=linear\n", "from=-2\nalpha=.5\n", 2),
    "add_more_channels": (6, 6, 8, "[convolutional]\nfilters=24\nsize=1\nactivation=linear\n"
                                    "[convolutional]\nfilters=16\nsize=1\nactivation=linear\n", "from=-2\nbeta=-1\n", 2),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(SHORTCUT))
def test_shortcut(dn, tmp_path, prec, name):
    h, w, c, producers, opts, i = SHORTCUT[name]
    net, port = case(dn, tmp_path, prec, h, w, c, producers + "[shortcut]\n" + opts)
    L = port.layers[i]
    assert net.kernel(i) == "shortcut"
    xs, got = force(net, port, i, prec, np.random.default_rng(4))
    x, add = xs[i - 1], xs[L.src]
    same = add.shape == x.shape
    assert same == name.startswith("same")                            # shortcut_dispatch, layers.cu:273
    y = NL.act_f32(NL.shortcut(x, add, L.alpha, L.beta), L.act, exact=prec == "fp32")
    expect_exact(got, y.reshape(BATCH, -1), prec, name)
    net.close()


# ---------------------------------------------------------------------------------------------------
# route: route_copy with vector and scalar copy_channels_kernel; a one-input alias
# ---------------------------------------------------------------------------------------------------
ROUTE = {
    "24_40_8": ("[convolutional]\nfilters=24\nsize=1\nactivation=linear\n[convolutional]\nfilters=40\nsize=1\nactivation=linear\n"
                "[convolutional]\nfilters=8\nsize=1\nactivation=linear\n[route]\nlayers=-3,-2,-1\n", 3),
    "padded_ld_10": ("[convolutional]\nfilters=10\nsize=1\nactivation=linear\n[convolutional]\nfilters=16\nsize=1\nactivation=linear\n"
                     "[route]\nlayers=-2,-1\n", 2),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(ROUTE))
def test_route_copy(dn, tmp_path, prec, name):
    body, i = ROUTE[name]
    net, port = case(dn, tmp_path, prec, 5, 6, 8, body)
    assert net.kernel(i) == "route_copy"
    xs, got = force(net, port, i, prec, np.random.default_rng(5))
    expect_exact(got, NL.route([xs[j] for j in port.layers[i].src]), prec, name)
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
def test_route_alias_feeds_its_consumer(dn, tmp_path, prec):
    body = "[convolutional]\nfilters=16\nsize=1\nactivation=linear\n[route]\nlayers=-1\n[maxpool]\nsize=3\nstride=2\n"
    net, port = case(dn, tmp_path, prec, 9, 9, 8, body)
    assert net.kernel(1) == "alias" and net.kernel(2) == "maxpool"
    xs, got = force(net, port, 2, prec, np.random.default_rng(6))
    L = port.layers[2]
    expect_exact(got, NL.maxpool(xs[1], L.size, L.stride, L.pad, L.out_h, L.out_w).reshape(BATCH, -1), prec)
    net.close()


# ---------------------------------------------------------------------------------------------------
# reorg: formula reorg_kernel; table kernel with dense and non-dense staging (layers.cu:373-379, 411)
# ---------------------------------------------------------------------------------------------------
REORG = {
    # name: (precisions, h, w, c, producer, stride, table kernel?)
    "s2_38x38x64": ("fp32", 38, 38, 64, MP1, 2, False),
    "s2_64x64x64": ("bf16", 64, 64, 64, MP1, 2, False),
    "s3_12x12x18": (None, 12, 12, 18, MP1, 3, True),
    "s2_padded_ld_40": (None, 8, 8, 8, "[convolutional]\nfilters=40\nsize=1\nactivation=linear\n", 2, True),
}
REORG_CASES = [(n, p) for n, v in sorted(REORG.items()) for p in PRECS if v[0] in (None, p)]


@gpu
@pytest.mark.parametrize("name,prec", REORG_CASES)
def test_reorg(dn, tmp_path, name, prec):
    _, h, w, c, producer, stride, table = REORG[name]
    net, port = case(dn, tmp_path, prec, h, w, c, producer + "[reorg]\nstride=%d\n" % stride)
    L = port.layers[1]
    assert net.kernel(1) == "reorg"
    assert (L.h * L.w * L.c * (2 if prec == "bf16" else 4) <= 200 * 1024) == table       # engine.cu select_kernels, layers.cu:411
    xs, got = force(net, port, 1, prec, np.random.default_rng(7))
    expect_exact(got, NL.reorg(xs[0], stride).reshape(BATCH, -1), prec, name)
    net.close()


# ---------------------------------------------------------------------------------------------------
# avgpool: avgpool_kernel<T, U, VEC> for every reachable (T, U) pair (classify.cu:78-91)
# ---------------------------------------------------------------------------------------------------
AVGPOOL = {
    # name: (h, w, c, consumer)
    "c20_7x7_softmax": (7, 7, 20, "[softmax]\n"),
    "c6_17x13_softmax": (17, 13, 6, "[softmax]\n"),
    "c20_1x1_conv": (1, 1, 20, "[convolutional]\nfilters=16\nsize=1\nactivation=linear\n"),
    "c6_17x13_conv": (17, 13, 6, "[convolutional]\nfilters=16\nsize=1\nactivation=linear\n"),
    "c24_7x7_connected": (7, 7, 24, "[connected]\noutput=8\nactivation=linear\n"),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(AVGPOOL))
def test_avgpool(dn, tmp_path, prec, name):
    h, w, c, consumer = AVGPOOL[name]
    net, port = case(dn, tmp_path, prec, h, w, c, MP1 + "[avgpool]\n" + consumer)
    assert net.kernel(1) == "avgpool"
    xs, got = force(net, port, 1, prec, np.random.default_rng(8))
    mean, mean_abs = NL.avgpool64(xs[0])
    bf_out = prec == "bf16" and "softmax" not in name                 # engine.cu plan_outputs: fp32 up to a [softmax]
    bound = h * w * NL.U * mean_abs + NL.U * np.abs(mean) + NL.half_ulp(np.abs(mean), bf_out) + 2.0 ** -126
    err = np.abs(got.astype(F64) - mean)
    assert (err <= bound).all(), (name, float((err / bound).max()))
    net.close()


# ---------------------------------------------------------------------------------------------------
# softmax: softmax_kernel with groups, temperature, group sizes past the CTA's 256 threads
# ---------------------------------------------------------------------------------------------------
def logits(shape, rng, scale=3.):
    """image 0 random, image 1 one constant per row (all equal), image 2 +-80"""
    x = (rng.standard_normal(shape) * scale).astype(F32)
    x[1] = F32(.375)
    x[2] = np.where(rng.random(shape[1:]) < .5, F32(-80), F32(80))
    return x


SOFTMAX = [(g, t, n) for g in (1, 2, 4, 8) for t in (1., 2.5, .5) for n in (7,)] + \
          [(1, 1., 1), (4, 1., 1), (1, .5, 32), (4, 2.5, 33), (1, 1., 1000), (2, .5, 1000), (1, 2.5, 2000)]


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("groups,temp,n", SOFTMAX)
def test_softmax_after_avgpool(dn, tmp_path, prec, groups, temp, n):
    net, port = case(dn, tmp_path, prec, 2, 2, groups * n, MP1 + "[avgpool]\n[softmax]\ngroups=%d\ntemperature=%g\n" % (groups, temp))
    assert net.kernel(2) == "softmax"
    rng = np.random.default_rng(9)
    x = logits((BATCH, groups * n), rng)
    net.set_layer_output(1, x)                                        # avgpool -> softmax keeps fp32
    net.run_layers(2, 3)
    got = net.layer_output(2).reshape(BATCH, groups, n)
    p64 = NL.softmax64(x.reshape(BATCH, groups, n), temp)
    expect_probs(got, p64, -(-n // 256) + 8, (groups, temp, n))      # 256 threads: serial, 5 shuffle levels, 3 CTA levels
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("source", ["classifier_conv", "connected"])
def test_softmax_after_conv_or_connected(dn, tmp_path, prec, source):
    producer = ("[convolutional]\nfilters=1000\nsize=1\nactivation=linear\n" if source == "classifier_conv"
                else "[connected]\noutput=33\nactivation=linear\n")
    net, port = case(dn, tmp_path, prec, 1, 1, 8, MP1 + producer + "[softmax]\ntemperature=.5\n")
    assert net.kernel(2) == "softmax"
    n = port.layers[1].outputs
    x = logits((BATCH, n), np.random.default_rng(10))
    net.set_layer_output(1, x)                                        # fp32: classifier logits (row pitch 1024) or [connected]
    net.run_layers(2, 3)
    expect_probs(net.layer_output(2), NL.softmax64(x, .5), -(-n // 256) + 8, source)
    net.close()


# ---------------------------------------------------------------------------------------------------
# heads: region_forward (tiled and direct-store), detection softmax pass, yolo with 1 and 200 classes
# ---------------------------------------------------------------------------------------------------
ANCH = "anchors=1.08,1.19,3.42,4.41,6.63,11.38,9.42,5.11,16.62,10.52\n"
HEADS = {
    # name: (h, w, body, classes, depth of the class softmax's fp32 sum)
    "region_logistic": (5, 5, "[convolutional]\nfilters=125\nsize=1\nactivation=linear\n"
                              "[region]\n" + ANCH + "classes=20\ncoords=4\nnum=5\nsoftmax=0\n", 20, 0),
    "region_softmax_400": (3, 4, "[convolutional]\nfilters=810\nsize=1\nactivation=linear\n"
                                 "[region]\nanchors=1,1,2,2\nclasses=400\ncoords=4\nnum=2\nsoftmax=1\n", 400, 13 + 5),
    "yolo_1_class": (6, 5, "[convolutional]\nfilters=12\nsize=1\nactivation=linear\n"
                           "[yolo]\nmask=0,1\nanchors=10,13,16,30,33,23\nclasses=1\nnum=3\n", 1, 0),
    "yolo_200_classes": (4, 4, "[convolutional]\nfilters=410\nsize=1\nactivation=linear\n"
                               "[yolo]\nmask=1,2\nanchors=10,13,16,30,33,23\nclasses=200\nnum=3\n", 200, 0),
}


DECODE_TOL = 2e-6          # decode is fp32 on both sides: libm exp vs the device's, one or two ulp


def expect_boxes(dn, net, port, i, head, w, h, thresh):
    """get_network_boxes_batch on the head output the device computed (its host copy set from it, as a driver that rewrites
    l.output would) against the port's get_network_boxes on the same values: count, boxes, objectness and probabilities"""
    from oracle import np_darknet as P
    net.set_layer_output(i, head)
    outs = [None] * i + [head]
    classes = port.layers[i].classes
    decoded = 0
    for b in range(net.batch):
        dets, n = net.boxes(b, w, h, thresh)
        boxes, obj, probs = dn.dets_to_arrays(dets, n, classes)
        dn.free_detections(dets, n)
        pb, po, pp, _ = P.get_network_boxes(port, outs, b, w, h, thresh)
        assert n == len(po), (b, n, len(po))
        if n:
            np.testing.assert_allclose(boxes, np.asarray(pb, F32), rtol=DECODE_TOL, atol=1e-9)
            assert np.array_equal(obj, np.asarray(po, F32)), b
            assert np.array_equal(probs == 0, np.asarray(pp) == 0), b
            np.testing.assert_allclose(probs, np.asarray(pp, F32), rtol=DECODE_TOL, atol=0)
        decoded += int((probs > 0).sum())
    assert decoded > 0                                                # some (box, class) pair passed the threshold


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(HEADS))
def test_region_and_yolo_heads(dn, tmp_path, prec, name):
    h, w, body, classes, depth = HEADS[name]
    net, port = case(dn, tmp_path, prec, h, w, 8, MP1 + body)
    L = port.layers[2]
    assert net.kernel(2) == ("yolo_forward" if L.type == "yolo" else "region_forward")
    if L.type == "region":
        assert ((L.coords + 1 + classes) * 33 * 4 > 48 * 1024) == (classes == 400)      # heads.cu:215: direct-store kernel
    x = (np.random.default_rng(12).standard_normal((BATCH, port.layers[1].out_c, h, w)) * 4).astype(F32)
    x[2] *= 4                                                         # saturating logistics and a peaked softmax
    x = NL.bf16(x) if prec == "bf16" else x                           # bf16-representable: the same values in either buffer
    net.set_layer_output(1, x.reshape(BATCH, -1))
    net.run_layers(2, 3)
    got = net.layer_output(2)
    if L.type == "yolo":
        want = NL.yolo64(x, L.n, classes)
        expect_probs(got, want, 0, name)
    else:
        want = NL.region64(x, L.n, L.coords, classes, L.softmax)
        expect_probs(got, want, depth, name)
    expect_boxes(dn, net, port, 2, got, w * 32, h * 32, .2 if classes < 400 else .005)
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("softmax", [0, 1])
def test_detection_head(dn, tmp_path, prec, softmax):
    body = MP1 + "[connected]\noutput=325\nactivation=linear\n[detection]\nclasses=3\ncoords=4\nrescore=1\nside=5\nnum=2\nsoftmax=%d\n" % softmax
    net, port = case(dn, tmp_path, prec, 1, 1, 16, body)
    assert net.kernel(2) == "detection_forward"
    x = (np.random.default_rng(13).standard_normal((BATCH, 325)) * 4).astype(F32)
    x[2] = np.where(x[2] > 0, F32(100), F32(-100))                   # exp(100) overflows fp32 without the max subtraction
    net.set_layer_output(1, x)
    net.run_layers(2, 3)
    got = net.layer_output(2)
    expect_probs(got, NL.detection64(x, 5, 3, softmax), 3, softmax)
    expect_boxes(dn, net, port, 2, got, 1, 1, .2)
    net.close()


# ---------------------------------------------------------------------------------------------------
# stem: conv_stem_kernel, try_stem_fast, try_stem_const, the tcgen05 stem's LDG fallback
# ---------------------------------------------------------------------------------------------------
def stem_branch(prec, c, size, stride, filters, w, act):
    """mirror of launch_conv_stem's dispatch (conv_stem_tc.cu:700-731, conv_simt.cu:227-303) for a cfg with pad=1"""
    V = 8 if prec == "bf16" else 4
    if prec == "bf16" and c == 3 and size == 7 and stride == 2 and filters == 64 and w % 4 == 0 and act in ("leaky", "linear"):
        return "tc7x7"
    if prec == "bf16" and c == 3 and size == 3 and stride == 1 and filters in (16, 32) and act in ("leaky", "linear"):
        return "tc_tma" if w % 4 == 0 else "tc_ldg"
    if c == 3 and size == 3 and stride in (1, 2) and filters in (16, 32, 64):
        return "const"
    if c == 3 and size in (3, 7) and filters % V == 0:
        return "fast"
    return "generic"


STEM = {
    # name: (channels, size, stride, filters, h, w, activation, branch in fp32, branch in bf16)
    "c1_3x3": (1, 3, 1, 16, 9, 10, "leaky", "generic", "generic"),
    "c2_3x3": (2, 3, 1, 8, 9, 10, "leaky", "generic", "generic"),
    "c4_3x3_s2": (4, 3, 2, 16, 9, 10, "leaky", "generic", "generic"),
    "c3_5x5": (3, 5, 1, 16, 9, 10, "leaky", "generic", "generic"),
    "c3_1x1": (3, 1, 1, 16, 9, 10, "linear", "generic", "generic"),
    "c3_3x3_s2_16": (3, 3, 2, 16, 11, 13, "leaky", "const", "const"),
    "c3_3x3_s2_32": (3, 3, 2, 32, 11, 13, "leaky", "const", "const"),
    "c3_3x3_s2_64": (3, 3, 2, 64, 11, 13, "leaky", "const", "const"),
    "c3_3x3_f24": (3, 3, 1, 24, 9, 10, "leaky", "fast", "fast"),
    "c3_3x3_f20": (3, 3, 1, 20, 9, 10, "leaky", "fast", "generic"),
    "c3_7x7_s2_w_odd": (3, 7, 2, 64, 15, 21, "leaky", "fast", "fast"),
    "c3_3x3_s1_16_w_odd": (3, 3, 1, 16, 10, 15, "leaky", "const", "tc_ldg"),
    "c3_3x3_s1_32_w_odd": (3, 3, 1, 32, 10, 13, "leaky", "const", "tc_ldg"),
    "c3_3x3_relu": (3, 3, 1, 16, 8, 8, "relu", "const", "const"),
    "c3_3x3_logistic": (3, 3, 1, 32, 8, 8, "logistic", "const", "const"),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(STEM))
def test_stem(dn, tmp_path, prec, name):
    c, size, stride, filters, h, w, act, b32, b16 = STEM[name]
    assert stem_branch(prec, c, size, stride, filters, w, act) == (b16 if prec == "bf16" else b32)
    body = "[convolutional]\nbatch_normalize=1\nfilters=%d\nsize=%d\nstride=%d\npad=1\nactivation=%s\n" % (filters, size, stride, act)
    net, port = case(dn, tmp_path, prec, h, w, c, body)
    assert net.kernel(0) == "conv_stem"
    x = NL.bf16(sample(np.random.default_rng(14), (BATCH, c, h, w)))   # the stem reads the fp32 image: bf16-representable
    net.predict(x)
    got = net.layer_output(0)
    L = port.layers[0]
    wt, (scale, shift) = weights_of(L, prec)
    y, mag = NL.conv64(x, wt, scale, shift, L.size, L.stride, L.pad)
    expect_sum(got, y.reshape(BATCH, -1), mag.reshape(BATCH, -1), L.size * L.size * c, act, prec == "bf16", name)
    net.close()


# ---------------------------------------------------------------------------------------------------
# convolution on CUDA cores (conv_simt_kernel, all three dtype pairs, conv_simt.cu:391-393) and tcgen05 padding cases
# ---------------------------------------------------------------------------------------------------
CONV = {
    # name: (cin, h, w, conv options, consumer, kernel in bf16 mode)
    "cin8": (8, 9, 11, "filters=16\nsize=3\nstride=1\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "cin24": (24, 9, 11, "filters=32\nsize=3\nstride=1\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "stride3": (16, 13, 11, "filters=16\nsize=3\nstride=3\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "5x5_s2": (8, 13, 12, "filters=16\nsize=5\nstride=2\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "relu_cin64": (64, 7, 9, "filters=32\nsize=3\nstride=1\npad=1\nactivation=relu\n", "", "conv_simt"),
    "logistic_cin64": (64, 7, 9, "batch_normalize=1\nfilters=32\nsize=3\nstride=1\npad=1\nactivation=logistic\n", "", "conv_simt"),
    "filters10": (8, 8, 9, "filters=10\nsize=3\nstride=1\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "filters33": (8, 8, 9, "batch_normalize=1\nfilters=33\nsize=3\nstride=1\npad=1\nactivation=leaky\n", "", "conv_simt"),
    "cin24_to_yolo": (24, 6, 6, "filters=18\nsize=3\nstride=1\npad=1\nactivation=linear\n",
                      "[yolo]\nmask=0,1,2\nanchors=10,13,16,30,33,23\nclasses=1\nnum=3\n", "conv_simt"),
    "tc_3x3_valid": (32, 10, 12, "batch_normalize=1\nfilters=32\nsize=3\nstride=1\npadding=0\nactivation=leaky\n", "", "conv_tc"),
    "tc_3x3_pad2": (32, 9, 10, "batch_normalize=1\nfilters=32\nsize=3\nstride=1\npadding=2\nactivation=leaky\n", "", "conv_tc"),
    "tc_7x7_cin32": (32, 11, 12, "batch_normalize=1\nfilters=32\nsize=7\nstride=1\npad=1\nactivation=leaky\n", "", "conv_tc"),
    "tc_7x7_cin64": (64, 11, 12, "batch_normalize=1\nfilters=64\nsize=7\nstride=1\npad=1\nactivation=leaky\n", "", "conv_tc"),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(CONV))
def test_conv(dn, tmp_path, prec, name):
    cin, h, w, opts, consumer, bf16_kernel = CONV[name]
    net, port = case(dn, tmp_path, prec, h, w, cin, MP1 + "[convolutional]\n" + opts + consumer)
    L = port.layers[1]
    kernel = net.kernel(1)
    assert kernel == ("conv_simt" if prec == "fp32" else bf16_kernel)
    xs, got = force(net, port, 1, prec, np.random.default_rng(15))
    wt, (scale, shift) = weights_of(L, prec)
    y, mag = NL.conv64(xs[0], wt, scale, shift, L.size, L.stride, L.pad)
    bf_out = prec == "bf16" and not consumer                          # logits feeding a [yolo] stay fp32
    expect_sum(got, y.reshape(BATCH, -1), mag.reshape(BATCH, -1), L.size * L.size * cin, L.act, bf_out, (name, kernel))
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
def test_first_layer_conv_reads_the_image(dn, tmp_path, prec):
    """a first convolution with more than 4 input channels is no stem: it is planned on the converted image"""
    net, port = case(dn, tmp_path, prec, 8, 9, 16, "[convolutional]\nfilters=16\nsize=3\nstride=1\npad=1\nactivation=leaky\n")
    assert net.kernel(0) == ("conv_tc" if prec == "bf16" else "conv_simt")
    x = sample(np.random.default_rng(18), (BATCH, 16, 8, 9))
    net.predict(x)
    L = port.layers[0]
    wt, (scale, shift) = weights_of(L, prec)
    y, mag = NL.conv64(NL.bf16(x) if prec == "bf16" else x, wt, scale, shift, 3, 1, 1)
    expect_sum(net.layer_output(0), y.reshape(BATCH, -1), mag.reshape(BATCH, -1), 9 * 16, "leaky", prec == "bf16")
    net.close()


@gpu
@pytest.mark.parametrize("prec", PRECS)
def test_conv_feeding_connected_keeps_a_dense_pitch(dn, tmp_path, prec):
    """24 filters from 32 input channels: the tcgen05 plan would take the shape, but a [connected] reads the output, whose
    row pitch then stays 24 (below the 32 padded filters conv_tc_plan_create needs), so it runs on CUDA cores; the
    [connected] reads the dense rows it wrote"""
    body = MP1 + "[convolutional]\nfilters=24\nsize=3\nstride=1\npad=1\nactivation=leaky\n[connected]\noutput=16\nactivation=linear\n"
    net, port = case(dn, tmp_path, prec, 5, 5, 32, body)
    assert net.kernel(1) == "conv_simt" and net.kernel(2) == "connected"
    xs, _ = force(net, port, 1, prec, np.random.default_rng(19))
    net.run_layers(2, 3)
    conv = net.layer_output(1)
    L = port.layers[1]
    wt, (scale, shift) = weights_of(L, prec)
    y, mag = NL.conv64(xs[0], wt, scale, shift, 3, 1, 1)
    expect_sum(conv, y.reshape(BATCH, -1), mag.reshape(BATCH, -1), 9 * 32, "leaky", prec == "bf16")
    F = port.layers[2]
    wt, (scale, shift) = weights_of(F, prec)
    y, mag = NL.connected64(conv, wt, scale, shift)
    expect_sum(net.layer_output(2), y, mag, F.inputs, "linear", False)
    net.close()


# ---------------------------------------------------------------------------------------------------
# local: local_kernel
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("prec", PRECS)
def test_local(dn, tmp_path, prec):
    net, port = case(dn, tmp_path, prec, 11, 11, 16, MP1 + "[local]\nfilters=32\nsize=5\nstride=2\npad=0\nactivation=leaky\n")
    L = port.layers[1]
    assert net.kernel(1) == "local"
    xs, got = force(net, port, 1, prec, np.random.default_rng(16))
    wt = NL.bf16(L.weights) if prec == "bf16" else L.weights
    y, mag = NL.local64(xs[0], wt, L.biases, L.size, L.stride, L.pad, L.out_h, L.out_w)
    expect_sum(got, y.reshape(BATCH, -1), mag.reshape(BATCH, -1), L.size * L.size * L.c, L.act, prec == "bf16")
    net.close()


# ---------------------------------------------------------------------------------------------------
# connected: connected_kernel (bf16 weights on bf16 or fp32 inputs, fp32), batch-norm fold (engine.cu fold_bn)
# ---------------------------------------------------------------------------------------------------
CONNECTED = {
    # name: (h, w, c, producers, connected options, index, batch)
    "in200_leaky": (5, 5, 8, MP1, "output=24\nactivation=leaky\n", 1, BATCH),
    "in200_relu": (5, 5, 8, MP1, "output=24\nactivation=relu\n", 1, BATCH),
    "in200_logistic": (5, 5, 8, MP1, "output=24\nactivation=logistic\n", 1, BATCH),
    "batch_normalize": (5, 5, 8, MP1, "output=40\nbatch_normalize=1\nactivation=leaky\n", 1, BATCH),
    "batch9": (5, 5, 8, MP1, "output=24\nactivation=leaky\n", 1, 9),
    "after_connected": (4, 4, 8, MP1 + "[connected]\noutput=48\nactivation=leaky\n", "output=20\nactivation=leaky\n", 2, BATCH),
    "after_dropout": (4, 4, 8, MP1 + "[connected]\noutput=48\nactivation=leaky\n[dropout]\nprobability=.5\n",
                      "output=20\nactivation=linear\n", 3, BATCH),
    "after_conv_filters10": (4, 4, 8, "[convolutional]\nfilters=10\nsize=3\nstride=1\npad=1\nactivation=leaky\n",
                             "output=24\nactivation=leaky\n", 1, BATCH),
}


@gpu
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("name", sorted(CONNECTED))
def test_connected(dn, tmp_path, prec, name):
    h, w, c, producers, opts, i, batch = CONNECTED[name]
    net, port = case(dn, tmp_path, prec, h, w, c, producers + "[connected]\n" + opts, batch=batch)
    L = port.layers[i]
    assert net.kernel(i) == "connected"
    assert L.inputs % 8 == 0 and (name != "in200_leaky" or L.inputs == 200)
    xs, got = force(net, port, i, prec, np.random.default_rng(17))
    wt, (scale, shift) = weights_of(L, prec)
    y, mag = NL.connected64(xs[i - 1], wt, scale, shift)
    expect_sum(got, y, mag, L.inputs, L.act, False, name)
    net.close()


# ---------------------------------------------------------------------------------------------------
# CPU: the restatements against the port and against the literal loops
# ---------------------------------------------------------------------------------------------------
def port_layer(**kw):
    from oracle import np_darknet as P
    return P, P.Layer(**kw)


def test_shortcut_restatement_is_shortcut_cpu():
    rng = np.random.default_rng(20)
    for xs, adds in [((2, 6, 4, 4), (2, 6, 4, 4)), ((2, 6, 4, 4), (2, 6, 8, 8)), ((2, 6, 8, 8), (2, 6, 4, 4)),
                     ((2, 6, 4, 4), (2, 3, 4, 4)), ((2, 3, 4, 4), (2, 6, 4, 4)), ((1, 5, 6, 6), (1, 7, 3, 3))]:
        x, add = sample(rng, xs), sample(rng, adds)
        for alpha, beta in ((1., 1.), (.5, 2.), (-.3, 1.7)):
            assert np.array_equal(NL.shortcut(x, add, alpha, beta), NL.shortcut_loop(x, add, alpha, beta)), (xs, adds, alpha)


def test_shortcut_restatement_matches_the_port_on_equal_shapes():
    P, L = port_layer(src=0, alpha=.5, beta=2., act="leaky")
    rng = np.random.default_rng(21)
    x, add = sample(rng, (2, 5, 3, 4)), sample(rng, (2, 5, 3, 4))
    want = P.fwd_shortcut(None, L, x, [add])
    assert np.array_equal(NL.act_f32(NL.shortcut(x, add, .5, 2.), "leaky", True), want)


@pytest.mark.parametrize("size,stride,pad,h,w", [(2, 2, 0, 13, 27), (3, 2, 1, 15, 15), (5, 1, 2, 13, 13), (13, 1, 6, 13, 13),
                                                 (3, 1, 0, 9, 11)])
def test_maxpool_restatement_matches_the_port(size, stride, pad, h, w):
    oh, ow = (h + 2 * pad) // stride, (w + 2 * pad) // stride
    P, L = port_layer(size=size, stride=stride, pad=pad, out_h=oh, out_w=ow)
    x = sample(np.random.default_rng(22), (2, 3, h, w))
    assert np.array_equal(NL.maxpool(x, size, stride, pad, oh, ow), P.fwd_maxpool(None, L, x, []))


@pytest.mark.parametrize("stride,c,h,w", [(2, 8, 6, 6), (3, 18, 12, 12), (2, 40, 8, 4)])
def test_reorg_restatement_matches_the_port(stride, c, h, w):
    P, L = port_layer(w=w, h=h, c=c, stride=stride, out_c=c * stride * stride, out_h=h // stride, out_w=w // stride)
    x = sample(np.random.default_rng(23), (2, c, h, w))
    assert np.array_equal(NL.reorg(x, stride), P.fwd_reorg(None, L, x, []))


@pytest.mark.parametrize("stride,scale", [(2, 1.), (3, 1.), (4, .5), (2, 3.)])
def test_upsample_restatement_matches_the_port(stride, scale):
    P, L = port_layer(stride=stride, scale=scale)
    x = sample(np.random.default_rng(24), (2, 3, 4, 5))
    assert np.array_equal(NL.upsample(x, stride, scale), P.fwd_upsample(None, L, x, []))


@pytest.mark.parametrize("softmax,classes", [(0, 20), (1, 20), (1, 400)])
def test_region_restatement_matches_the_port(softmax, classes):
    P, L = port_layer(n=2, coords=4, classes=classes, softmax=softmax, h=3, w=4)
    x = (np.random.default_rng(25).standard_normal((2, 2 * (5 + classes), 3, 4)) * 4).astype(F32)
    want = P.fwd_region(None, L, x, [])
    got = NL.region64(x, 2, 4, classes, softmax)
    assert (np.abs(got - want) <= 4 * NL.half_ulp(got, False) + classes * NL.U * np.abs(got)).all()   # the port sums serially in fp32


@pytest.mark.parametrize("softmax", [0, 1])
def test_detection_restatement_matches_the_port(softmax):
    P, L = port_layer(side=5, classes=3, softmax=softmax)
    x = (np.random.default_rng(26).standard_normal((2, 325)) * 4).astype(F32)
    want = P.fwd_detection(None, L, x, [])
    assert (np.abs(NL.detection64(x, 5, 3, softmax) - want) <= 4 * NL.half_ulp(want, False) + 3 * NL.U * np.abs(want)).all()


def test_conv_restatement_matches_the_port():
    from oracle import np_darknet as P
    rng = np.random.default_rng(27)
    L = P.Layer(n=10, size=3, stride=2, pad=1, bn=1, act="leaky", out_h=4, out_w=5, c=6, h=7, w=9)
    L.weights = rng.standard_normal((10, 54)).astype(F32)
    L.biases, L.scales = rng.standard_normal(10).astype(F32), rng.uniform(.5, 1.5, 10).astype(F32)
    L.mean, L.var = (rng.standard_normal(10) * .1).astype(F32), rng.uniform(.5, 1.5, 10).astype(F32)
    x = sample(rng, (2, 6, 7, 9))
    want = P.fwd_conv(None, L, x, [])
    y, mag = NL.conv64(x, L.weights, *NL.fold64(L.biases, L.scales, L.mean, L.var), 3, 2, 1)
    expect_sum(want.reshape(2, -1), y.reshape(2, -1), mag.reshape(2, -1), 54, "leaky", False)


def test_bf16_rounding_is_nearest_even():
    v = np.array([1., 1 + 2 ** -8, 1 + 3 * 2 ** -8, 1 + 2 ** -9, -np.finfo(F32).max, -0.], F32)
    want = np.array([1., 1., 1 + 4 * 2 ** -8, 1., -np.inf, -0.], F32)
    assert np.array_equal(NL.bf16(v), want)
