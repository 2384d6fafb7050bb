#!/usr/bin/env python3
"""classifier_bench.py — Darknet-53 (256x256) and Darknet-19 (224x224) at batch 64 through the classification entry points.

  python scripts/classifier_bench.py --out DIR [--steps 50]

One process, one GPU, writes one JSON line to DIR/classifier_bench.json (and prints it).  Per model:
  resident_images_s : b200_classify_submitted with B200_INPUT_RESIDENT (the batch already in HBM), host clock around `steps`
                      calls; every call waits for its top-k results, so the window ends on a device synchronise
  e2e_images_s      : 64 decoded uint8 640x480 pictures (pinned host memory) -> b200_letterbox_batch_u8 -> classify, the
                      letterbox of batch k+1 overlapping the forward of batch k (the serving loop of bench.py's e2e key)
  forward_ms        : b200_profile_forward (whole pass, back to back, CUDA events) and its first layer
  conv_tflops       : darknet's FLOP formula of every convolution but the first, over the pass minus the first layer and minus
                      the classifier tail; as a share of MEASURED_PEAKS.json's bf16 burst and sustained rates
  tail_us           : device time of the avgpool / softmax / top-k kernels (torch.profiler, CUDA activities, a run of its own)
  layer_ms          : b200_profile_layers (events between layers) of the same three layers' neighbourhood
  batch1_ms         : batch-1 latency of network_predict + top_k (the reference API, predict_classifier's path), median
  top1_mean         : mean top-1 probability over the timed batch: the softmax is not saturated (synthetic weights damped so
                      that the logits have std ~2, yolo_tensorflow_b200/synth.py)
plus the card's name, power limit and SM clocks from nvidia-smi (query only), read in the same call.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from bench import peaks  # noqa: E402
from yolo_tensorflow_b200 import synth  # noqa: E402

MODELS = [("darknet53", 256), ("darknet19", 224)]
BATCH, TOP, SRC_W, SRC_H = 64, 5, 640, 480


def conv_flops(cfg):
    """darknet's formula per convolution: 2 * filters * size^2 * channels * out_h * out_w"""
    return [2 * L["n"] * L["size"] ** 2 * L["c"] * L["out"][1] * L["out"][2]
            for L in synth.walk_shapes(cfg)["layers"] if L["type"] == "convolutional"]


def gpu_info():
    q = "name,power.limit,power.max_limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except (OSError, subprocess.TimeoutExpired) as e:
        return {"error": str(e)}


def open_net(dn, model, batch, size, work):
    cfg = synth.make_cfg(model, work, batch=batch, width=size, height=size)
    w = os.path.join(work, model + ".weights")
    if not os.path.exists(w):
        synth.write_weights(cfg, w, seed=0)
    fd = os.dup(2); devnull = os.open(os.devnull, os.O_WRONLY); os.dup2(devnull, 2)
    try:
        return dn.Network(cfg, w, precision=dn.PREC_BF16), cfg
    finally:
        os.dup2(fd, 2); os.close(fd); os.close(devnull)


def measure(dn, torch, model, size, steps, work):
    net, cfg = open_net(dn, model, BATCH, size, work)
    lib, RES = dn.lib, ctypes.c_void_p(1)
    cls = np.zeros((BATCH, TOP), np.int32); prob = np.zeros((BATCH, TOP), np.float32)
    cp, pp = cls.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), prob.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    x = synth.make_images(BATCH, 3, size, size, 1000)
    net.classify_batch(x, TOP)                                           # the batch is now in the device input buffer

    def resident(n):
        lib.b200_submit_batch(net.ptr, RES)
        for k in range(n):
            assert lib.b200_classify_submitted(net.ptr, RES if k < n - 1 else None, TOP, cp, pp) == BATCH

    resident(5)
    t0 = time.perf_counter(); resident(steps); t_res = time.perf_counter() - t0
    top1_mean = float(prob[:, 0].mean())

    rng = np.random.default_rng(7)
    pics = []
    for _ in range(2):                                                   # two batches of pinned source pictures, alternating
        batch = []
        for _ in range(BATCH):
            t = torch.empty((SRC_H, SRC_W, 3), dtype=torch.uint8, pin_memory=True)
            t.numpy()[:] = (rng.random((SRC_H, SRC_W, 3)) * 255).astype(np.uint8)
            batch.append(t)
        pics.append(batch)
    ptrs = [(ctypes.c_void_p * BATCH)(*[t.data_ptr() for t in b]) for b in pics]
    ws, hs = (ctypes.c_int * BATCH)(*[SRC_W] * BATCH), (ctypes.c_int * BATCH)(*[SRC_H] * BATCH)

    def e2e(n):
        assert lib.b200_letterbox_batch_u8(net.ptr, ptrs[0], ws, hs, BATCH) == 0
        lib.b200_submit_batch(net.ptr, RES)
        for k in range(n):
            if k < n - 1:
                assert lib.b200_letterbox_batch_u8(net.ptr, ptrs[(k + 1) % 2], ws, hs, BATCH) == 0
            assert lib.b200_classify_submitted(net.ptr, RES if k < n - 1 else None, TOP, cp, pp) == BATCH

    e2e(5)
    t0 = time.perf_counter(); e2e(steps); t_e2e = time.perf_counter() - t0

    fwd, first = net.profile_forward(steps)
    layer_ms = net.profile_layers(10)
    kinds = [L["type_name"] for L in net.layers]
    tail_layers = [i for i, k in enumerate(kinds) if k in ("AVGPOOL", "SOFTMAX")]
    tail_layer_ms = float(sum(layer_ms[i] for i in tail_layers))

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            net.classify_batch(None, TOP)
        torch.cuda.synchronize()
    tail_us = {}
    for ev in prof.key_averages():
        for name in ("avgpool_kernel", "softmax_kernel", "topk_kernel"):
            if name in ev.key:
                tail_us[name.replace("_kernel", "")] = round(ev.device_time_total / max(ev.count, 1), 2)

    flops = conv_flops(cfg)
    pk = peaks()
    conv_ms = fwd - first - tail_layer_ms
    tflops = (sum(flops) - flops[0]) * BATCH / (conv_ms * 1e-3) / 1e12
    kernels = sorted({net.kernel(i) for i in range(net.n)})
    net.close()

    one, _ = open_net(dn, model, 1, size, work)
    x1 = np.ascontiguousarray(x[:1])
    idx = (ctypes.c_int * TOP)()
    lat = []
    for it in range(60):
        t0 = time.perf_counter()
        out = dn.predict(one.ptr, x1.ctypes.data_as(ctypes.POINTER(ctypes.c_float)))
        lib.top_k(out, 1000, TOP, idx)
        if it >= 10:
            lat.append((time.perf_counter() - t0) * 1e3)
    one.close()
    return dict(model=f"{model}-{size}", batch=BATCH, top=TOP, flop_per_image=sum(flops),
                resident_images_s=round(BATCH * steps / t_res, 1), e2e_images_s=round(BATCH * steps / t_e2e, 1),
                forward_ms=round(fwd, 4), first_layer_ms=round(first, 4), tail_layers_ms=round(tail_layer_ms, 4),
                conv_tflops=round(tflops, 1), conv_frac_burst=round(tflops / pk["burst"], 3) if pk["burst"] else None,
                conv_frac_sustained=round(tflops / pk["sustained"], 3) if pk["sustained"] else None, tail_us=tail_us,
                batch1_ms_median=round(float(np.median(lat)), 4), top1_mean=round(top1_mean, 4), kernels=kernels)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory for classifier_bench.json")
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("classifier_bench.py measures the GPU: no CUDA device here")
    from yolo_tensorflow_b200 import darknet as dn
    work = os.environ.get("B200_WORKDIR", "/tmp/b200_classifier_bench")
    os.makedirs(work, exist_ok=True)
    os.makedirs(args.out, exist_ok=True)
    rec = dict(gpu_before=gpu_info(), peaks=peaks(), steps=args.steps,
               models=[measure(dn, torch, m, s, args.steps, work) for m, s in MODELS])
    rec["gpu_after"] = gpu_info()
    line = json.dumps(rec)
    with open(os.path.join(args.out, "classifier_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
