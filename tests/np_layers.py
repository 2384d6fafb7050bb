"""TEST INFRASTRUCTURE — float64 (and, for the copy / select / permute layers, exact fp32) restatements of darknet's layers for
tests/test_layer_zoo.py.  Same conventions as oracle/np_darknet.py: NCHW arrays, heads as [batch, outputs], and every function
cites the reference function it restates.  Unlike the port, the summing layers return the float64 result together with the
magnitude sum_k |w_k x_k| that bounds the rounding error of any fp32 summation order.  The product never imports it.
"""
import numpy as np

F32 = np.float32
F64 = np.float64
U = 2.0 ** -24                                                                     # unit roundoff of fp32


def bf16(x):
    """round fp32 to the nearest bf16, ties to even (__float2bfloat16_rn), returned as fp32"""
    u = np.ascontiguousarray(x, dtype=F32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    nan = np.isnan(np.asarray(x, dtype=F32))
    return np.where(nan, np.float32(np.nan), r.astype(np.uint32).view(F32)).astype(F32)


def half_ulp(v, bf):
    """half a unit in the last place of fp32 (bf=False) or bf16 (bf=True) at |v| (normal range; a floor below it)"""
    a = np.maximum(np.abs(np.asarray(v, dtype=F64)), 2.0 ** -126)
    return np.exp2(np.floor(np.log2(a)) - (8 if bf else 24))


# ---------------------------------------------------------------------------------------------------
# activations (activations.h:32,38; common.cuh apply_act)
# ---------------------------------------------------------------------------------------------------
def act64(y, act):
    y = np.asarray(y, dtype=F64)
    if act == "leaky":
        return np.where(y > 0, y, .1 * y)
    if act == "logistic":
        return 1. / (1. + np.exp(-y))
    if act == "relu":
        return np.where(y > 0, y, 0.)
    if act == "linear":
        return y
    raise ValueError(act)


def act_slope(act):
    """largest |d act / dy|: how far an error before the activation can move its result"""
    return {"leaky": 1., "relu": 1., "linear": 1., "logistic": .25}[act]


def act_f32(y, act, exact):
    """the activation in fp32 as the kernels apply it: EXACT (fp32 mode) takes leaky as (float)(.1 * (double)x), the bf16 mode
    as 0.1f * x; logistic is (float)(1 / (1 + exp(-(double)x))) in both"""
    y = np.asarray(y, dtype=F32)
    if act == "leaky":
        neg = (F64(.1) * y.astype(F64)).astype(F32) if exact else (F32(.1) * y).astype(F32)
        return np.where(y > 0, y, neg).astype(F32)
    if act == "logistic":
        return (1. / (1. + np.exp(-y.astype(F64)))).astype(F32)
    if act == "relu":
        return np.where(y > 0, y, F32(0)).astype(F32)
    return y


# ---------------------------------------------------------------------------------------------------
# copy / select / permute layers: exact in fp32
# ---------------------------------------------------------------------------------------------------
def maxpool(x, size, stride, pad, oh, ow):                                         # maxpool_layer.c:79-114
    """window origin -pad; taps outside the image count as -FLT_MAX; a tap replaces the maximum when strictly greater"""
    B, C, H, W = x.shape
    y = np.full((B, C, oh, ow), -np.finfo(F32).max, dtype=F32)
    for i in range(oh):
        for j in range(ow):
            for n in range(size):
                for m in range(size):
                    cur_h, cur_w = i * stride + n - pad, j * stride + m - pad
                    if 0 <= cur_h < H and 0 <= cur_w < W:
                        v = x[:, :, cur_h, cur_w]
                        y[:, :, i, j] = np.where(v > y[:, :, i, j], v, y[:, :, i, j])
    return y


def upsample(x, stride, scale):                                                    # blas.c:334-349 upsample_cpu (forward)
    B, C, H, W = x.shape
    y = np.empty((B, C, H * stride, W * stride), dtype=F32)
    for j in range(H * stride):
        for i in range(W * stride):
            y[:, :, j, i] = (F32(scale) * x[:, :, j // stride, i // stride]).astype(F32)
    return y


def shortcut(x, add, alpha, beta):                                                 # blas.c:68-92 shortcut_cpu on a copy of x
    """out = x, then out[over the overlap] = s1*out + s2*add with the stride / sample indexing; shapes (B, c, h, w)"""
    B, c2, h2, w2 = x.shape
    _, c1, h1, w1 = add.shape
    stride, sample = max(w1 // w2, 1), max(w2 // w1, 1)
    minw, minh, minc = min(w1, w2), min(h1, h2), min(c1, c2)
    out = x.astype(F32).copy()
    o = out[:, :minc, 0:minh * sample:sample, 0:minw * sample:sample]
    a = add[:, :minc, 0:minh * stride:stride, 0:minw * stride:stride]
    out[:, :minc, 0:minh * sample:sample, 0:minw * sample:sample] = (F32(alpha) * o).astype(F32) + (F32(beta) * a).astype(F32)
    return out


def shortcut_loop(x, add, alpha, beta):                                            # blas.c:68-92, literally
    B, c2, h2, w2 = x.shape
    _, c1, h1, w1 = add.shape
    stride, sample = w1 // w2, w2 // w1
    stride, sample = max(stride, 1), max(sample, 1)
    minw, minh, minc = min(w1, w2), min(h1, h2), min(c1, c2)
    out = x.astype(F32).reshape(-1).copy()
    addf = add.astype(F32).reshape(-1)
    for b in range(B):
        for k in range(minc):
            for j in range(minh):
                for i in range(minw):
                    out_index = i * sample + w2 * (j * sample + h2 * (k + c2 * b))
                    add_index = i * stride + w1 * (j * stride + h1 * (k + c1 * b))
                    out[out_index] = F32(F32(alpha) * out[out_index]) + F32(F32(beta) * addf[add_index])
    return out.reshape(x.shape)


def route(xs):                                                                     # route_layer.c:74-87
    return np.concatenate([x.reshape(x.shape[0], -1) for x in xs], axis=1)


def reorg(x, stride):                                                              # blas.c:9-30 reorg_cpu(forward=0), reorg_layer.c:107-109
    """with (w, h, c) the INPUT dims: out[in_index] = x[out_index] for every (b, k, j, i) of the input"""
    B, c, h, w = x.shape
    flat = x.reshape(B, -1)
    out = np.empty_like(flat)
    out_c = c // (stride * stride)
    for k in range(c):
        for j in range(h):
            for i in range(w):
                in_index = i + w * (j + h * k)
                c2, offset = k % out_c, k // out_c
                w2, h2 = i * stride + offset % stride, j * stride + offset // stride
                out_index = w2 + w * stride * (h2 + h * stride * c2)
                out[:, in_index] = flat[:, out_index]
    return out.reshape(B, c * stride * stride, h // stride, w // stride)


# ---------------------------------------------------------------------------------------------------
# summing layers: (float64 result before the activation, sum |terms| after the scale)
# ---------------------------------------------------------------------------------------------------
def fold64(biases, scales=None, mean=None, var=None):                              # batchnorm_layer.c:150-154, blas.c:147-158
    """per-output (scale, shift) of the inference batch-norm, or (1, bias) without one"""
    if scales is None:
        return np.ones(len(biases)), np.asarray(biases, F64)
    s = np.asarray(scales, F64) / (np.sqrt(np.asarray(var, F64)) + F64(F32(.000001)))
    return s, np.asarray(biases, F64) - np.asarray(mean, F64) * s


def im2col64(x, size, stride, pad):                                                # im2col.c:16-39, zero padding
    B, C, H, W = x.shape
    oh, ow = (H + 2 * pad - size) // stride + 1, (W + 2 * pad - size) // stride + 1
    xp = np.zeros((B, C, H + 2 * pad, W + 2 * pad))
    xp[:, :, pad:pad + H, pad:pad + W] = x
    cols = np.empty((B, C, size, size, oh, ow))
    for ky in range(size):
        for kx in range(size):
            cols[:, :, ky, kx] = xp[:, :, ky:ky + stride * oh:stride, kx:kx + stride * ow:stride]
    return cols.reshape(B, C * size * size, oh * ow), oh, ow


def conv64(x, weights, scale, shift, size, stride, pad):                           # convolutional_layer.c:445-485
    """weights [n][c*size*size]; returns (y, mag) of shape [B, n, oh, ow]"""
    B = x.shape[0]
    cols, oh, ow = im2col64(np.asarray(x, F64), size, stride, pad)
    w = np.asarray(weights, F64)
    y = np.matmul(w[None], cols) * scale[None, :, None] + shift[None, :, None]
    mag = np.matmul(np.abs(w)[None], np.abs(cols)) * np.abs(scale)[None, :, None] + np.abs(shift)[None, :, None]
    return y.reshape(B, -1, oh, ow), mag.reshape(B, -1, oh, ow)


def local64(x, weights, biases, size, stride, pad, oh, ow):                        # local_layer.c:91-120
    """weights [loc][n][c*size*size], biases [n][loc]; local_layer pads by `pad` on each side"""
    B = x.shape[0]
    cols, _, _ = im2col64(np.asarray(x, F64), size, stride, pad)
    cols = cols[:, :, :oh * ow]
    w = np.asarray(weights, F64)
    y = np.einsum("lnk,bkl->bnl", w, cols) + np.asarray(biases, F64).reshape(1, -1, oh * ow)
    mag = np.einsum("lnk,bkl->bnl", np.abs(w), np.abs(cols)) + np.abs(np.asarray(biases, F64)).reshape(1, -1, oh * ow)
    return y.reshape(B, -1, oh, ow), mag.reshape(B, -1, oh, ow)


def connected64(x, weights, scale, shift):                                         # connected_layer.c:151-167
    x = np.asarray(x, F64).reshape(x.shape[0], -1)
    w = np.asarray(weights, F64)
    return x @ w.T * scale + shift, np.abs(x) @ np.abs(w).T * np.abs(scale) + np.abs(shift)


def avgpool64(x):                                                                  # avgpool_layer.c forward_avgpool_layer
    B, C = x.shape[:2]
    v = np.asarray(x, F64).reshape(B, C, -1)
    return v.mean(axis=2), np.abs(v).mean(axis=2)


# ---------------------------------------------------------------------------------------------------
# softmax and the detection heads
# ---------------------------------------------------------------------------------------------------
def softmax64(x, temp=1.):                                                         # blas.c:305-321 softmax(), along the last axis
    """exp(x/temp - largest/temp) with the quotients and the difference rounded to fp32 as in the C code, the rest in float64"""
    x = np.asarray(x, F32)
    largest = x.max(axis=-1, keepdims=True)
    arg = ((x / F32(temp)).astype(F32) - (largest / F32(temp)).astype(F32)).astype(F32)
    e = np.exp(arg.astype(F64))
    return e / e.sum(axis=-1, keepdims=True)


def logistic64(x):                                                                 # activations.h:32
    return 1. / (1. + np.exp(-np.asarray(x, F64)))


def region64(x, n, coords, classes, softmax):                                      # region_layer.c:158-189 (no tree)
    """x: the head input [B, n*(coords+1+classes), h, w]; returns [B, outputs] float64"""
    B, _, h, w = x.shape
    y = np.asarray(x, F64).reshape(B, n, coords + 1 + classes, h * w).copy()
    y[:, :, 0:2] = logistic64(y[:, :, 0:2])
    y[:, :, coords] = logistic64(y[:, :, coords])
    cls = x.reshape(B, n, coords + 1 + classes, h * w)[:, :, coords + 1:]
    y[:, :, coords + 1:] = np.moveaxis(softmax64(np.moveaxis(cls, 2, 3)), 3, 2) if softmax else logistic64(cls)
    return y.reshape(B, -1)


def yolo64(x, n, classes):                                                         # yolo_layer.c:132-149
    B, _, h, w = x.shape
    y = np.asarray(x, F64).reshape(B, n, classes + 5, h * w).copy()
    y[:, :, 0:2] = logistic64(y[:, :, 0:2])
    y[:, :, 4:] = logistic64(y[:, :, 4:])
    return y.reshape(B, -1)


def detection64(x, side, classes, softmax):                                        # detection_layer.c:50-66
    B = x.shape[0]
    y = np.asarray(x, F64).reshape(B, -1).copy()
    if softmax:
        loc = side * side
        y[:, :loc * classes] = softmax64(x.reshape(B, -1)[:, :loc * classes].reshape(B, loc, classes)).reshape(B, -1)
    return y
