#!/usr/bin/env python3
"""Throughput of the batched validate_detector driver (b200_validate_images: device letterbox -> forward -> decode/NMS ->
result file) on YOLOv3-416, batch 64, over decoded 640x480 images held in host memory.
Usage: python scripts/validate_probe.py [images]"""
import os, sys, tempfile, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from yolo_tensorflow_b200 import synth, darknet as dn

m = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
work = "/tmp/b200_validate_probe"
cfg = synth.make_cfg("yolov3", work, batch=64, width=416, height=416)
wpath = os.path.join(work, "yolov3.weights")
if not os.path.exists(wpath):
    synth.write_weights(cfg, wpath, seed=0, damp_heads=True)
net = dn.Network(cfg, wpath, precision=dn.PREC_BF16)
rng = np.random.default_rng(0)
distinct = [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8) for _ in range(64)]
images = [distinct[i % 64] for i in range(m)]
paths = ["val2014/COCO_val2014_%012d.jpg" % i for i in range(m)]
out = tempfile.mkdtemp()
net.validate_images(images[:128], paths[:128], "coco", out, thresh=.5)       # warm-up
t = time.perf_counter()
n = net.validate_images(images, paths, "coco", out, thresh=.5)
dt = time.perf_counter() - t
print("validate_images: %d images, %d records, %.1f ms, %.0f images/s" % (m, n, dt * 1e3, m / dt))
net.close()
