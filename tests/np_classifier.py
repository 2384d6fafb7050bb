"""TEST INFRASTRUCTURE — the numpy port of oracle/np_darknet.py extended with the layers of darknet's ImageNet classifiers
([avgpool], [softmax], [cost]) and top_k of utils.c, for tests/test_classifier.py.  Same conventions as the port: fp32 NCHW,
every function cites the reference function it restates.  The product never imports it.

    python tests/np_classifier.py --calibrate darknet53     prints the logit std that yolo_tensorflow_b200/synth.py damps by
"""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from oracle import np_darknet as P  # noqa: E402

F32 = P.F32


def fwd_avgpool(net, L, x, outs):                                                  # avgpool_layer.c forward_avgpool_layer
    B = x.shape[0]
    v = x.reshape(B, L.c, L.h * L.w)
    s = np.zeros((B, L.c), dtype=F32)
    for i in range(L.h * L.w):                                                     # float accumulation in pixel order
        s = (s + v[:, :, i]).astype(F32)
    return (s / F32(L.h * L.w)).astype(F32).reshape(B, L.c, 1, 1)


def fwd_softmax(net, L, x, outs):                                                  # softmax_layer.c forward_softmax_layer -> softmax_cpu
    # softmax() of blas.c: exp(x/temp - largest/temp).  For temp > 0 the largest of x/temp is largest/temp, so this is the
    # port's softmax_strided (the [region] head's arithmetic) applied to x/temp, one group per row
    B = x.shape[0]
    v = (x.reshape(B, L.groups, L.inputs // L.groups, 1) / F32(L.temperature)).astype(F32)
    return P.softmax_strided(v).reshape(B, -1)


def fwd_cost(net, L, x, outs):                                                     # cost_layer.c forward_cost_layer: no truth, no work
    return x.reshape(x.shape[0], -1)


def top_k(a, k):                                                                   # utils.c top_k, literally
    """indices of the k largest of a[n], descending, by insertion with a strict `>`: equal values do not always keep index
    order (an entry displaced from its slot moves on only past strictly smaller ones)"""
    index = [-1] * k
    for i in range(len(a)):
        curr = i
        for j in range(k):
            if index[j] < 0 or a[curr] > a[index[j]]:
                curr, index[j] = index[j], curr
    return np.array(index)


FORWARD = dict(P.FORWARD, avgpool=fwd_avgpool, avg=fwd_avgpool, softmax=fwd_softmax, soft=fwd_softmax, cost=fwd_cost)


class Net(P.Net):
    """P.Net that also builds and runs the classifier layers"""

    def _make(self, t, o, i, h, w, c, inputs):
        if t not in ("avgpool", "avg", "softmax", "soft", "cost"):
            return super()._make(t, o, i, h, w, c, inputs)
        L = P.Layer(type=t, index=i, h=h, w=w, c=c, inputs=inputs, act=None)
        if t in ("avgpool", "avg"):                                                # avgpool_layer.c make_avgpool_layer
            L.out_w, L.out_h, L.out_c = 1, 1, c
            L.outputs = c
        else:                                                                      # parser.c parse_softmax / parse_cost
            if t in ("softmax", "soft"):
                L.groups, L.temperature = int(o.get("groups", 1)), float(o.get("temperature", 1))
            L.out_w = L.out_h = L.out_c = 0
            L.outputs = inputs
        return L

    def forward(self, x, keep=True):                                               # network.c forward_network
        cur = np.ascontiguousarray(x, dtype=F32)
        outs = []
        for L in self.layers:
            cur = FORWARD[L.type](self, L, cur, outs)
            outs.append(cur)
        return outs


def calibrate(model, seed_image=1000):
    """std of the [softmax] input (the logits) with the UNDAMPED seed-0 file on one seed image at the cfg's size: the
    numbers synth.HEAD_RAW_STD holds for the classifiers"""
    import tempfile
    from yolo_tensorflow_b200 import synth
    with tempfile.TemporaryDirectory() as tmp:
        cfg = os.path.join(synth.CFG_DIR, model + ".cfg")
        w = os.path.join(tmp, "raw.weights")
        synth.write_weights(cfg, w, seed=0, damp_heads=False)
        net = Net(cfg, w)
        outs = net.forward(synth.make_images(1, net.c, net.h, net.w, seed_image))
        return [float(outs[L.index - 1].std()) for L in net.layers if L.type in ("softmax", "soft")]


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--calibrate":
        print(sys.argv[2], ["%.4g" % v for v in calibrate(sys.argv[2])])
