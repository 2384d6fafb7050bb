#!/usr/bin/env python3
"""Derive darknet .cfg files from the reference's own parse_network_cfg printouts.

The reference ships no cfg/ directory (git-ignored upstream); the only statements of the three
topologies are the stderr layer tables YOLO_V{1,2,3}/*/yolov{1,2,3}.txt, kept here verbatim as
structural goldens under tests/golden/layer_tables/.  The rules below are SURVEY.md §8(c): a cfg
is right iff the parser reprints those tables byte-for-byte (tests/test_parser.py checks both the
reference parser, when oracle/_ref is built, and ours).

Head parameters (anchors/masks/classes) come from the reference's TF converters:
  YOLO_V3_convert_darkenet_to_Tensorflow.py:28, YOLO_V3_Tiny_convert...py:29,420-464,
  YOLO_V2_convert_darkenet_to_Tensorflow.py:24-28.
"""
import os, re, sys

HERE = os.path.dirname(os.path.abspath(__file__))
TABLES = os.path.join(HERE, "..", "tests", "golden", "layer_tables")

V3_ANCHORS = "10,13,16,30,33,23,30,61,62,45,59,119,116,90,156,198,373,326"
V3_TINY_ANCHORS = "10,14,23,27,37,58,81,82,135,169,344,319"
V2_ANCHORS = "0.57273,0.677385,1.87446,2.06253,3.33843,5.47434,7.88282,3.52778,9.77052,9.16828"


def net_section(w, h, batch=1):
    return (f"[net]\nbatch={batch}\nsubdivisions=1\nwidth={w}\nheight={h}\nchannels=3\n"
            "momentum=0.9\ndecay=0.0005\nlearning_rate=0.001\nmax_batches=500200\npolicy=constant\n")


def conv(f, k, s, bn=1, act="leaky"):
    t = "[convolutional]\n"
    if bn:
        t += "batch_normalize=1\n"
    return t + f"filters={f}\nsize={k}\nstride={s}\npad=1\nactivation={act}\n"


def from_table(path, head_filters, head_block, yolo_masks=None, rows=None):
    rows = open(path).read().splitlines()[1:][:rows]
    out, nyolo = [], 0
    for i, row in enumerate(rows):
        tok = row.split()
        assert int(tok[0]) == i, row
        kind = tok[1]
        if kind == "conv":
            f, k, s = int(tok[2]), int(tok[3]), int(tok[7])
            if f in head_filters:
                out.append(conv(f, k, s, bn=0, act="linear"))
            else:
                out.append(conv(f, k, s))
        elif kind == "max":
            out.append(f"[maxpool]\nsize={tok[2]}\nstride={tok[6]}\n")
        elif kind == "res":
            out.append(f"[shortcut]\nfrom={int(tok[2]) - i}\nactivation=linear\n")
        elif kind == "route":
            out.append("[route]\nlayers=" + ",".join(tok[2:]) + "\n")
        elif kind == "upsample":
            out.append(f"[upsample]\nstride={tok[2].rstrip('x')}\n")
        elif kind == "reorg":
            out.append(f"[reorg]\nstride={tok[3]}\n")
        elif kind == "yolo":
            out.append(f"[yolo]\nmask={yolo_masks[nyolo]}\nanchors={V3_ANCHORS}\nclasses=80\nnum=9\n"
                       "jitter=.3\nignore_thresh=.7\ntruth_thresh=1\nrandom=1\n")
            nyolo += 1
        elif kind == "detection":          # region layer prints "detection" (region_layer.c:50)
            out.append(head_block)
        elif kind == "Local":
            f = int(re.search(r"(\d+) filters", row).group(1))
            out.append(f"[local]\nsize=3\nstride=1\npad=1\nfilters={f}\nactivation=leaky\n")
        elif kind == "dropout":
            out.append("[dropout]\nprobability=.5\n")
        elif kind == "connected":
            out.append(f"[connected]\noutput={tok[-1]}\nactivation=linear\n")
        elif kind == "Detection":          # detection layer prints "Detection Layer"
            out.append(head_block)
        else:
            raise ValueError(row)
    return out


def yolov3(w=416, h=416, batch=1):
    body = from_table(os.path.join(TABLES, "yolov3.txt"), {255}, None, ["6,7,8", "3,4,5", "0,1,2"])
    return net_section(w, h, batch) + "\n" + "\n".join(body)


def yolov2(w=416, h=416, batch=1):
    head = (f"[region]\nanchors={V2_ANCHORS}\nbias_match=1\nclasses=80\ncoords=4\nnum=5\nsoftmax=1\n"
            "jitter=.3\nrescore=1\nobject_scale=5\nnoobject_scale=1\nclass_scale=1\ncoord_scale=1\n"
            "mask_scale=1\nabsolute=1\nthresh=.6\nrandom=1\n")
    body = from_table(os.path.join(TABLES, "yolov2.txt"), {425}, head)
    return net_section(w, h, batch) + "\n" + "\n".join(body)


def yolov1(w=448, h=448, batch=1):
    # whether the v1 convs carry BN is not recoverable from the table; we use BN (as yolov1.cfg of the
    # darknet era did) and the same file feeds both the reference and this engine.
    head = ("[detection]\nclasses=20\ncoords=4\nrescore=1\nside=7\nnum=3\nsoftmax=0\nsqrt=1\njitter=.2\n"
            "forced=0\nobject_scale=1\nnoobject_scale=.5\nclass_scale=1\ncoord_scale=5\n")
    body = from_table(os.path.join(TABLES, "yolov1.txt"), set(), head)
    return net_section(w, h, batch) + "\n" + "\n".join(body)


def yolov3_tiny(w=416, h=416, batch=1):
    L = []
    for f in (16, 32, 64, 128, 256):
        L += [conv(f, 3, 1), "[maxpool]\nsize=2\nstride=2\n"]
    L += [conv(512, 3, 1), "[maxpool]\nsize=2\nstride=1\n", conv(1024, 3, 1), conv(256, 1, 1), conv(512, 3, 1),
          conv(255, 1, 1, bn=0, act="linear"),
          f"[yolo]\nmask=3,4,5\nanchors={V3_TINY_ANCHORS}\nclasses=80\nnum=6\njitter=.3\nignore_thresh=.7\n"
          "truth_thresh=1\nrandom=1\n",
          "[route]\nlayers=-4\n", conv(128, 1, 1), "[upsample]\nstride=2\n", "[route]\nlayers=-1,8\n",
          conv(256, 3, 1), conv(255, 1, 1, bn=0, act="linear"),
          f"[yolo]\nmask=0,1,2\nanchors={V3_TINY_ANCHORS}\nclasses=80\nnum=6\njitter=.3\nignore_thresh=.7\n"
          "truth_thresh=1\nrandom=1\n"]
    return net_section(w, h, batch) + "\n" + "\n".join(L)


# ImageNet classifiers: the detectors' own backbones with darknet's classification tail (1000-way linear 1x1 conv, global
# average pool, softmax, and the [cost] layer training needs and inference skips).  Darknet-53 pools before the 1x1,
# Darknet-19 after it.
CLASSIFIER_TAIL = "[softmax]\ngroups=1\n", "[cost]\ntype=sse\n"


def darknet53(w=256, h=256, batch=1):
    body = from_table(os.path.join(TABLES, "yolov3.txt"), set(), None, rows=75)
    tail = ["[avgpool]\n", conv(1000, 1, 1, bn=0, act="linear"), *CLASSIFIER_TAIL]
    return net_section(w, h, batch) + "\n" + "\n".join(body + tail)


def darknet19(w=224, h=224, batch=1):
    body = from_table(os.path.join(TABLES, "yolov2.txt"), set(), None, rows=23)
    tail = [conv(1000, 1, 1, bn=0, act="linear"), "[avgpool]\n", *CLASSIFIER_TAIL]
    return net_section(w, h, batch) + "\n" + "\n".join(body + tail)


MODELS = {"yolov3": yolov3, "yolov2": yolov2, "yolov1": yolov1, "yolov3-tiny": yolov3_tiny, "darknet19": darknet19,
          "darknet53": darknet53}

if __name__ == "__main__":
    for name, fn in MODELS.items():
        with open(os.path.join(HERE, name + ".cfg"), "w") as f:
            f.write(fn())
        print("wrote", name + ".cfg")
