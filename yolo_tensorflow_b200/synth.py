"""Synthetic workloads for parity tests and bench.py (SURVEY.md §8d): cfg variants, seeded `.weights`
files in the reference's on-disk order, and seeded images.  There is no network access for real
datasets or checkpoints, so both the reference and this engine always load the SAME synthetic file.

Distributions (seed 0): conv/local/connected weights N(0, sqrt(2/fan_in)) — the scale
make_convolutional_layer itself uses (convolutional_layer.c:205-209); biases N(0,0.1); BN scales
U(0.5,1.5), rolling_mean N(0,0.1), rolling_variance U(0.5,1.5).  `damp_heads=True` rescales the
convolution (or connected layer) that feeds each detection head so that logits have std 1.5 and sets the
objectness biases so that 10^1-10^2 candidates per image pass the threshold instead of thousands (the
undamped file is the NMS stress configuration).
"""
import os
import re
import struct

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG_DIR = os.path.join(REPO, "cfg")


# --------------------------------------------------------------------------------------------------
# cfg handling
# --------------------------------------------------------------------------------------------------
def read_cfg(path):
    """-> list of (section_name, dict) with darknet's whitespace stripping"""
    sections = []
    for raw in open(path):
        line = re.sub(r"[ \t\r\n]", "", raw)
        if not line or line[0] in "#;":
            continue
        if line[0] == "[":
            sections.append((line, {}))
        elif "=" in line:
            k, v = line.split("=", 1)
            sections[-1][1][k] = v
    return sections


def make_cfg(model, out_dir, batch=1, width=None, height=None):
    """writes cfg/<model>.cfg with batch/width/height replaced; returns the new path"""
    src = os.path.join(CFG_DIR, model + ".cfg")
    text = open(src).read()
    text = re.sub(r"(?m)^batch=\d+", f"batch={batch}", text, count=1)
    if width:
        text = re.sub(r"(?m)^width=\d+", f"width={width}", text, count=1)
    if height:
        text = re.sub(r"(?m)^height=\d+", f"height={height}", text, count=1)
    os.makedirs(out_dir, exist_ok=True)
    tag = f"{model}_b{batch}" + (f"_{width}x{height}" if width else "")
    dst = os.path.join(out_dir, tag + ".cfg")
    # several ranks of one job derive the same file at the same time while others already parse it: never truncate in place
    if os.path.exists(dst) and open(dst).read() == text:
        return dst
    tmp = dst + ".%d.tmp" % os.getpid()
    with open(tmp, "w") as f:
        f.write(text)
    os.replace(tmp, dst)
    return dst


def make_tree_cfg(out_dir, tree_path, batch=1, size=64, classes=240, num=3):
    """a small YOLO9000-style network: two conv/maxpool stages and a [region] head with a class WordTree (`tree=`, SURVEY §8f-4)"""
    text = (f"[net]\nbatch={batch}\nsubdivisions=1\nheight={size}\nwidth={size}\nchannels=3\nmomentum=0.9\ndecay=0.0005\n"
            "learning_rate=0.001\nmax_batches=1\npolicy=constant\n"
            "[convolutional]\nbatch_normalize=1\nfilters=16\nsize=3\nstride=1\npad=1\nactivation=leaky\n[maxpool]\nsize=2\nstride=2\n"
            "[convolutional]\nbatch_normalize=1\nfilters=64\nsize=3\nstride=1\npad=1\nactivation=leaky\n[maxpool]\nsize=2\nstride=2\n"
            f"[convolutional]\nfilters={num * (classes + 5)}\nsize=1\nstride=1\npad=1\nactivation=linear\n"
            f"[region]\nanchors=0.77,1.02,2.3,1.9,3.9,4.4\nbias_match=1\nclasses={classes}\ncoords=4\nnum={num}\nsoftmax=1\njitter=.2\n"
            f"rescore=1\nthresh=.6\ntree={tree_path}\n")
    os.makedirs(out_dir, exist_ok=True)
    dst = os.path.join(out_dir, f"yolo9000-small_b{batch}_{size}.cfg")
    if not (os.path.exists(dst) and open(dst).read() == text):
        tmp = dst + ".%d.tmp" % os.getpid()
        with open(tmp, "w") as f:
            f.write(text)
        os.replace(tmp, dst)
    return dst


def walk_shapes(cfg_path):
    """minimal shape walk of the inference layer types -> list of dicts (type, c,h,w in, out_c,out_h,out_w, params...)"""
    secs = read_cfg(cfg_path)
    net = secs[0][1]
    h, w, c = int(net["height"]), int(net["width"]), int(net["channels"])
    inputs = h * w * c
    layers = []
    for i, (name, o) in enumerate(secs[1:]):
        t = name.strip("[]")
        L = dict(type=t, index=i, h=h, w=w, c=c, inputs=inputs, opts=o)
        if t in ("convolutional", "conv"):
            n, size, stride = int(o.get("filters", 1)), int(o.get("size", 1)), int(o.get("stride", 1))
            pad = size // 2 if int(o.get("pad", 0)) else int(o.get("padding", 0))
            oh, ow = (h + 2 * pad - size) // stride + 1, (w + 2 * pad - size) // stride + 1
            L.update(n=n, size=size, stride=stride, pad=pad, bn=int(o.get("batch_normalize", 0)), out=(n, oh, ow))
        elif t == "local":
            n, size, stride, pad = int(o["filters"]), int(o["size"]), int(o["stride"]), int(o.get("pad", 0))
            oh = ((h - 1) if pad else (h - size)) // stride + 1
            ow = ((w - 1) if pad else (w - size)) // stride + 1
            L.update(n=n, size=size, stride=stride, pad=pad, out=(n, oh, ow))
        elif t in ("maxpool", "max"):
            stride = int(o.get("stride", 1)); size = int(o.get("size", stride)); pad = int(o.get("padding", (size - 1) // 2))
            L.update(out=(c, (h + 2 * pad) // stride, (w + 2 * pad) // stride))
        elif t == "route":
            idx = [int(v) if int(v) >= 0 else i + int(v) for v in o["layers"].split(",")]
            oc = sum(layers[j]["out"][0] for j in idx)
            L.update(out=(oc, layers[idx[0]]["out"][1], layers[idx[0]]["out"][2]), src=idx)
        elif t == "upsample":
            s = int(o.get("stride", 2)); L.update(out=(c, h * s, w * s))
        elif t == "shortcut":
            L.update(out=(c, h, w))
        elif t == "reorg":
            s = int(o.get("stride", 1)); L.update(out=(c * s * s, h // s, w // s))
        elif t == "dropout":
            L.update(out=(c, h, w), outputs=inputs)
        elif t in ("connected", "conn"):
            L.update(out=(int(o["output"]), 1, 1), bn=int(o.get("batch_normalize", 0)))
        elif t in ("yolo", "region", "detection"):
            L.update(out=(c, h, w), outputs=inputs)
        elif t in ("avgpool", "avg"):
            L.update(out=(c, 1, 1))
        elif t in ("softmax", "soft", "cost"):
            L.update(out=(c, h, w), outputs=inputs)
        else:
            raise ValueError(f"layer type {t} is outside the YOLO inference path")
        c, h, w = L["out"]
        L.setdefault("outputs", c * h * w)
        inputs = L["outputs"]
        layers.append(L)
    return dict(net=net, layers=layers)


# --------------------------------------------------------------------------------------------------
# weights
# --------------------------------------------------------------------------------------------------
def _head_feeders(layers):
    """indices of the conv / connected layers whose output is consumed by a detection head or, directly or through
    [avgpool], by a classifier's [softmax]"""
    feed = {}
    for L in layers:
        if L["type"] in ("yolo", "region", "detection", "softmax", "soft"):
            j = L["index"] - 1
            while layers[j]["type"] in ("dropout", "avgpool", "avg"):
                j -= 1
            feed[j] = L
    return feed


# std of each head-feeding layer's output with the UNDAMPED seed-0 file, measured by running the reference CPU
# build on one seed-(1000+config) image (tests/golden/make_golden.py --calibrate prints these).  Damping divides
# the feeder's weights by this number and multiplies by HEAD_TARGET_STD.
HEAD_RAW_STD = {
    "yolov3-tiny": [4.300, 3.730],
    "yolov3": [410826.0, 431648.0, 582677.0],
    "yolov2": [4.011],
    "yolov1": [11.266],
    # classifiers: std of the [softmax] input (the logits) with the undamped file, computed on the CPU with the numpy port
    # (seed-1000 image at the cfg's size; `python tests/np_classifier.py --calibrate darknet53` prints them; the reference
    # build is not part of this repository, and the port is pinned to it on the detection models)
    "darknet19": [3.126],
    "darknet53": [213053.0],
}
HEAD_TARGET_STD = 1.5      # logits ~ N(0, 1.5^2)
CLASSIFIER_TARGET_STD = 2.0   # classifier logits ~ N(0, 2^2): a top-1 probability well inside (0, 1), not one-hot
# objectness-channel bias per model, tuned (with the reference CPU build, seed-0 weights) so that a realistic
# 10^1-10^2 anchors per image pass objectness 0.5: yolov3-416 ~230 of 10647, yolov3-tiny ~90 of 2535, yolov2 ~70 of 845
HEAD_OBJ_BIAS = {"yolov3-tiny": -1.2, "yolov3": -3.0, "yolov2": -0.5}
REGION_CLASS_GAIN = 4.0    # region head: softmax over 80 classes needs peaky logits for any class to clear 0.5
V1_TARGET_STD = 0.15


def model_of(cfg_path):
    name = os.path.basename(cfg_path)
    for m in sorted(HEAD_RAW_STD, key=len, reverse=True):
        if name.startswith(m):
            return m
    return None


def write_weights(cfg_path, out_path, seed=0, damp_heads=True, head_gain=None):
    """writes a `.weights` file (header 0,2,0,uint64 seen=0; parser.c:1241-1345 order). Returns #floats."""
    info = walk_shapes(cfg_path)
    layers = info["layers"]
    rng = np.random.default_rng(seed)
    feeders = _head_feeders(layers) if damp_heads else {}
    raw_std = HEAD_RAW_STD.get(model_of(cfg_path))
    feeder_rank = {j: r for r, j in enumerate(sorted(feeders))}
    total = 0
    with open(out_path, "wb") as f:
        f.write(struct.pack("<iiiQ", 0, 2, 0, 0))

        def put(a):
            nonlocal total
            a = np.ascontiguousarray(a, dtype=np.float32)
            f.write(a.tobytes()); total += a.size

        for L in layers:
            t = L["type"]
            if t in ("convolutional", "conv"):
                n, k = L["n"], L["size"] * L["size"] * L["c"]
                bias = rng.normal(0, 0.1, n)
                wts = rng.normal(0, np.sqrt(2.0 / k), (n, k))
                if L["index"] in feeders and feeders[L["index"]]["type"] in ("softmax", "soft"):
                    if head_gain is not None:
                        wts *= head_gain
                    elif raw_std:
                        wts *= CLASSIFIER_TARGET_STD / raw_std[feeder_rank[L["index"]]]
                elif L["index"] in feeders:
                    head = feeders[L["index"]]
                    if head_gain is not None:
                        wts *= head_gain
                    elif raw_std:
                        wts *= HEAD_TARGET_STD / raw_std[feeder_rank[L["index"]]]
                    else:
                        wts *= _damp_factor(layers, L["index"])
                    entries = int(head["opts"].get("classes", 20)) + int(head["opts"].get("coords", 4)) + 1
                    bias[4::entries] = HEAD_OBJ_BIAS.get(model_of(cfg_path), -3.0)
                    if head["type"] == "region":
                        rows = np.arange(n)
                        wts[(rows % entries) >= 5] *= REGION_CLASS_GAIN
                put(bias)
                if L["bn"]:
                    put(rng.uniform(0.5, 1.5, n)); put(rng.normal(0, 0.1, n)); put(rng.uniform(0.5, 1.5, n))
                put(wts)
            elif t in ("connected", "conn"):
                o, k = L["out"][0], L["inputs"]
                bias = rng.normal(0, 0.1, o)
                wts = rng.normal(0, np.sqrt(2.0 / k), (o, k))
                if L["index"] in feeders:
                    wts *= (V1_TARGET_STD / raw_std[feeder_rank[L["index"]]]) if raw_std else 0.02
                    bias = rng.uniform(0.1, 0.6, o)
                put(bias); put(wts)
                if L.get("bn"):
                    put(rng.uniform(0.5, 1.5, o)); put(rng.normal(0, 0.1, o)); put(rng.uniform(0.5, 1.5, o))
            elif t == "local":
                n, oh, ow = L["out"]
                k = L["size"] * L["size"] * L["c"]
                put(rng.normal(0, 0.1, n * oh * ow))
                # generated location by location to bound memory (115.6 M floats for YOLOv1)
                for _ in range(oh * ow):
                    put(rng.normal(0, np.sqrt(2.0 / k), (n, k)).astype(np.float32))
    return total


def _damp_factor(layers, idx):
    """analytic estimate of 1/std of the activations entering conv `idx`, so that the head logits are O(1)."""
    # variance multiplier accumulated along the main path: each shortcut adds two equal-variance tensors
    doublings = sum(1 for L in layers[:idx] if L["type"] == "shortcut")
    return float(2.0 ** (-0.5 * doublings)) * 0.5


def make_images(batch, c, h, w, seed):
    """fp32 NCHW U[0,1) (SURVEY §8d: seed = 1000 + config index)"""
    return np.random.default_rng(seed).random((batch, c, h, w), dtype=np.float32)

