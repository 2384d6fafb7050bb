#!/usr/bin/env python3
"""bench.py — YOLOv3-416 images/s through the darknet C API of this engine (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            this engine (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU implementation (oracle/_ref)
  python bench.py ... --dump-outputs DIR                    also writes the headline's last timed step as DIR/<name>.npy
                                                            (inputs are seeded: two builds can be compared output for output)

A "step" = one pass of the hot path over one batch: network forward (conv stack) + device decode +
class-wise NMS for all images of the batch.  Headline workload = configs[2] of BASELINE.json: YOLOv3 416x416,
batch 64 per GPU, bf16 (weak scaling: the per-GPU batch is fixed).
  value   : images/s with the batch already resident in HBM (b200_detect_submitted with B200_INPUT_RESIDENT), CUDA-event
            timed on the engine's stream, max over ranks.
  e2e     : the same metric through the C-ABI serving loop with HOST buffers: every timed step uploads 64 decoded uint8 RGB
            images (640x480, pinned), letterboxes them on the device (b200_letterbox_batch_u8 = load_image's conversion +
            letterbox_image), runs forward + decode + NMS and reads the kept records back (b200_detect_submitted).
            `e2e_fp32_nchw` is the same loop fed with ready-made fp32 NCHW batches (what network_predict takes: 133 MB per step).
  roofline: tensor-pipe roofline of the dominant kernel family (the tcgen05 convolutions): darknet's own BFLOPs formula
            over the device time of those launches as the step runs them (b200_profile_forward: events around the whole
            pass minus the first layer, no per-layer brackets), against MEASURED_PEAKS.json (burst and sustained).
  c4      : BASELINE configs[3]: YOLOv3 608x608, 256 images per step SPLIT over the N GPUs (strong scaling), every rank's
            records gathered to rank 0 over NCCL inside the step (b200_comm_set_gather).
  other_configs (N=1): configs[0], [1], [4] and 608x608 at batch 32 — ms/step, images/s, TFLOP/s, clocks.
  dropin (N=1): batch-1 latency through the REFERENCE API: network_predict + get_network_boxes + do_nms_sort + free_detections.
  cpu_baseline : the unmodified reference CPU build (oracle/_ref, GPU=0 OPENMP=1) timed on this box's host
                 cores on a bounded sample of the same workload (rank 0, N=1 only).
PyTorch is used for torch.distributed (rendezvous, barriers, max over ranks), pinned host memory and CUDA events on the
engine's stream; the weight broadcast and the detection gather are the library's own NCCL calls; every kernel in the timed
region is this repo's own.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORK = os.environ.get("B200_WORKDIR", "/tmp/b200_bench")
# FLOP per image = the reference's own `darknet ops` on the derived cfgs (BASELINE.md / SURVEY §8d); yolov1 + its [local] layer
CONFIGS = {
    "C3": dict(name="YOLOv3 416x416 batch 64 (BASELINE configs[2], headline)", model="yolov3", size=416, batch=64, thresh=.5, nms=.45, flop=65_864_075_264),
    "C1": dict(name="YOLOv3-tiny 416x416 batch 1 (configs[0])", model="yolov3-tiny", size=416, batch=1, thresh=.5, nms=.45, flop=5_564_961_792),
    "C2": dict(name="YOLOv2 416x416 batch 64 (configs[1])", model="yolov2", size=416, batch=64, thresh=.5, nms=.45, flop=29_464_168_448),
    "C5": dict(name="YOLOv1 448x448 batch 64 (configs[4])", model="yolov1", size=448, batch=64, thresh=.2, nms=.4, flop=40_190_248_448 + 231_211_008),
    "608x32": dict(name="YOLOv3 608x608 batch 32 (the per-GPU shard of configs[3] at 8 GPUs)", model="yolov3", size=608, batch=32, thresh=.5, nms=.45, flop=140_691_900_416),
    "C4": dict(name="YOLOv3 608x608, 256 images per step split over the GPUs (configs[3])", model="yolov3", size=608, batch=256, thresh=.5, nms=.45, flop=140_691_900_416),
}
HEAD = CONFIGS["C3"]
MODEL, SIZE, BATCH, THRESH, NMS = HEAD["model"], HEAD["size"], HEAD["batch"], HEAD["thresh"], HEAD["nms"]
FLOP_PER_IMAGE = HEAD["flop"]
SRC_W, SRC_H = 640, 480                       # decoded source pictures of the e2e loop (COCO-sized)
E2E_INPUT = os.environ.get("B200_E2E_INPUT", "u8")      # which serving loop the `e2e` key reports: "u8" or "fp32"


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(burst=p.get("bf16_tflops"), sustained=p.get("bf16_tflops_sustained", p.get("bf16_tflops")), hbm=p.get("hbm_gbs"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(burst=1650.0, sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons, streamed for the whole run (a line every 20 ms); summary(t0, t1) reports a window"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,clocks_event_reasons.active,power.draw,power.limit")
        try:
            proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        try:
            for line in proc.stdout:
                line = line.strip()
                if line:
                    self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
                if self.stop_flag:
                    break
        finally:
            proc.terminate()
            try:
                proc.wait(timeout=2)
            except Exception:
                proc.kill()

    def stop(self):
        self.stop_flag = True

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.02]
        if not rows:                              # a window shorter than the sampling period: take the nearest sample
            near = sorted(self.rows, key=lambda tr: abs(tr[0] - (t0 + t1) / 2))[:1]
            rows = [r for _, r in near]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 2 + j and r[2 + j].lower().startswith("active") for r in rows)]
        # every other bit of the event-reason mask seen under load (nvml: 0x1 idle, 0x2 application clocks, 0x10 sync boost,
        # 0x80 power brake, 0x100 display clocks), so that clocks below max never come without their reason
        other = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x10: "sync_boost", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        mask = 0
        for r in rows:
            try:
                mask |= int(r[6], 16) if len(r) > 6 else 0
            except ValueError:
                pass
        reasons += [n for bit, n in other.items() if mask & bit]

        def med(col):
            v = []
            for r in rows:
                try:
                    v.append(float(r[col]))
                except (ValueError, IndexError):
                    pass
            return sorted(v)[len(v) // 2] if v else None
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(rows[0][1]) if rows[0][1].isdigit() else None,
                "sm_min_mhz": sm[0] if sm else None, "reasons": reasons, "samples": len(rows),
                "power_w": med(7), "power_limit_w": med(8)}


def prepare_files(model, size, batch):
    from yolo_tensorflow_b200 import synth
    os.makedirs(WORK, exist_ok=True)
    cfg = synth.make_cfg(model, WORK, batch=batch, width=size, height=size)
    wpath = os.path.join(WORK, f"{model}_seed0_damped.weights")
    if not os.path.exists(wpath):
        tmp = wpath + f".{os.getpid()}.tmp"
        synth.write_weights(cfg, tmp, seed=0, damp_heads=True)
        os.replace(tmp, wpath)
    return cfg, wpath


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (oracle/_ref), host cores only.
# Nothing here imports yolo_tensorflow_b200.darknet: the product library is never mapped into this process.
# ---------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, images_per_step=1):
    """times network_predict + get_network_boxes + do_nms_sort (detector.c:596-603 idiom) per image"""
    from yolo_tensorflow_b200 import synth
    from oracle import ref_darknet as R
    cfg, wpath = prepare_files(MODEL, SIZE, 1)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host thread it can
    os.environ["OMP_NUM_THREADS"] = os.environ.get("B200_REF_THREADS", str(cores))
    kind = "reference"
    if R.available():
        net = R.RefNet(cfg, wpath)

        def one(img):
            net.predict(img)
            dets, n = net.boxes(0, SIZE, SIZE, THRESH)
            net.nms_sort(dets, n, NMS)
            net.free_dets(dets, n)
    else:                                   # the reference .so did not travel: fall back to the numpy restatement
        from oracle import np_darknet as P
        kind = "port"
        net = P.Net(cfg, wpath)

        def one(img):
            outs = net.forward(img)
            b, o, p, _ = P.get_network_boxes(net, outs, 0, SIZE, SIZE, THRESH)
            P.do_nms_sort(b, o, p, NMS)
    imgs = synth.make_images(max(1, images_per_step), 3, SIZE, SIZE, 1002)
    for _ in range(warmup):
        one(imgs[:1])
    t0 = time.perf_counter()
    for _ in range(steps):
        for j in range(images_per_step):
            one(imgs[j:j + 1])
    dt = time.perf_counter() - t0
    return dict(value=steps * images_per_step / dt, seconds=dt, kind=kind, cores=cores,
                sample=f"{steps * images_per_step} image(s) of YOLOv3-416 (predict + get_network_boxes + do_nms_sort), batch 1 as the reference runs it")


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 8))
    r = cpu_reference_run(steps, min(args.warmup, 1))
    assert "yolo_tensorflow_b200.darknet" not in sys.modules          # the reference arm never maps the product library
    line = {"impl": "reference", "metric": "YOLOv3-416 images/s (conv+decode+NMS)", "value": r["value"], "unit": "images/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": 1000.0 * r["seconds"] / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"YOLOv3 {SIZE}x{SIZE} batch {BATCH} (reference CPU arm: 1 image per step, batch 1)",
                       "thresh": THRESH, "nms": NMS},
            "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# this engine
# ---------------------------------------------------------------------------------------------------
class _DevPtr:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


RESIDENT = ctypes.c_void_p(1)


def comm_root(rank):
    return rank == 0


class Runner:
    """one network + the three serving loops over it (resident, fp32 NCHW host batches, uint8 host pictures)"""

    def __init__(self, dn, torch, conf, batch, rank, world, local, load_weights=True, comm=False):
        self.dn, self.torch, self.conf, self.batch, self.rank, self.world, self.local = dn, torch, conf, batch, rank, world, local
        self.size, self.thresh, self.nms = conf["size"], conf["thresh"], conf["nms"]
        self.wh = (1, 1) if conf["model"] == "yolov1" else (self.size, self.size)
        cfg, wpath = prepare_files(conf["model"], self.size, batch) if load_weights else (self._cfg_only(conf, batch), None)
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(2); os.dup2(devnull, 2)                 # the layer table goes to stderr like the reference's
        try:
            self.net = dn.Network(cfg, wpath, precision=dn.PREC_BF16)
        finally:
            os.dup2(saved, 2); os.close(saved); os.close(devnull)
        self.net.set_head_sync(0)
        self.stream = torch.cuda.ExternalStream(self.net.stream_ptr(), device=torch.device("cuda", local))
        # kept (box, class) records per image with the synthetic heads: ~1300 at 416x416, ~6400 at 608x608 (measured); the gather
        # slot of a rank and the result buffer are sized from these with head-room
        self.slot_per_image = 2048 if self.size <= 416 else 10240
        self.max_out = max(1 << 20, self.slot_per_image * batch * (world if comm_root(rank) else 1))
        # page-locked result buffer: the records of a step (up to 59 MB at 608x608 x 256 images) come back by DMA, not through a staging copy
        self.out_pinned = torch.empty(self.max_out * ctypes.sizeof(dn.B200_DET), dtype=torch.uint8).pin_memory()
        self.out = ctypes.cast(self.out_pinned.data_ptr(), ctypes.POINTER(dn.B200_DET))
        self.counts = (dn.c_int * batch)()
        self.primed = False
        self.comm = False

    @staticmethod
    def _cfg_only(conf, batch):
        from yolo_tensorflow_b200 import synth
        return synth.make_cfg(conf["model"], WORK, batch=batch, width=conf["size"], height=conf["size"])

    # ---- multi-GPU (library-owned NCCL) -------------------------------------------------------------
    def join(self, dist, image_base, gather=True):
        """communicator over all ranks, ONE broadcast of rank 0's parameter arena, records gathered to rank 0 from now on"""
        dn = self.dn
        ident = (ctypes.c_ubyte * 128)()
        if self.rank == 0:
            dn.lib.b200_comm_unique_id(ident, 128)
        box = [bytes(ident)]
        dist.broadcast_object_list(box, src=0)
        ident = (ctypes.c_ubyte * 128).from_buffer_copy(box[0])
        dn.lib.b200_comm_init(self.net.ptr, ident, self.rank, self.world)
        dn.lib.b200_comm_broadcast_weights(self.net.ptr, 0)
        if gather:
            dn.lib.b200_comm_set_gather(self.net.ptr, 0, image_base, self.slot_per_image * self.batch)
        self.comm = True

    # ---- inputs -----------------------------------------------------------------------------------
    def load_resident(self, seed):
        from yolo_tensorflow_b200 import synth
        torch = self.torch
        x = torch.from_numpy(synth.make_images(self.batch, 3, self.size, self.size, seed)).pin_memory()
        nbytes = x.numel() * 4
        d_in = torch.as_tensor(_DevPtr(self.net.input_device_ptr(), nbytes), device=torch.device("cuda", self.local))
        d_in.copy_(x.view(torch.uint8).reshape(-1))
        torch.cuda.synchronize()
        return x

    # ---- the loops ----------------------------------------------------------------------------------
    def step_resident(self):
        lib, n = self.dn.lib, self.net
        if not self.primed:
            lib.b200_submit_batch(n.ptr, RESIDENT)
            self.primed = True
        return lib.b200_detect_submitted(n.ptr, RESIDENT, self.wh[0], self.wh[1], self.thresh, self.nms, 1, self.out, self.max_out, self.counts)

    def drain(self):
        if self.primed:
            self.dn.lib.b200_detect_submitted(self.net.ptr, None, self.wh[0], self.wh[1], self.thresh, self.nms, 1, self.out, self.max_out, self.counts)
            self.primed = False

    def barrier(self, dist):
        if self.world > 1:
            dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, dist, fn, steps):
        torch = self.torch
        self.barrier(dist)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(self.stream)
        n = 0
        for _ in range(steps):
            n = fn()
        e1.record(self.stream)
        self.barrier(dist)
        t1 = time.time()
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device="cuda" if dist.get_backend() == "nccl" else "cpu")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, n, (t0, t1)

    def close(self):
        if self.comm:
            self.dn.lib.b200_comm_destroy(self.net.ptr)
        self.net.close()


def conv_family(net, batch):
    is_tc = [net.kernel(i).startswith("conv_tc") for i in range(net.n)]
    flops = sum(2.0 * L["n"] * L["size"] ** 2 * L["c"] * L["out_h"] * L["out_w"] * batch for i, L in enumerate(net.layers) if is_tc[i])
    bytes_ = sum((L["c"] * L["h"] * L["w"] + L["out_c"] * L["out_h"] * L["out_w"]) * 2.0 * batch + L["nweights"] * 2.0
                 for i, L in enumerate(net.layers) if is_tc[i])
    return sum(is_tc), flops, bytes_


def secondary(dn, torch, dist, key, sampler, steps, warmup, rank, world, local):
    """one of the non-headline configurations at N = 1: ms/step, images/s, TFLOP/s, clocks"""
    conf = CONFIGS[key]
    r = Runner(dn, torch, conf, conf["batch"], rank, world, local)
    r.load_resident(1000 + list(CONFIGS).index(key))
    for _ in range(max(warmup, 3)):
        r.step_resident()
    ms, nrec, win = r.timed(dist, r.step_resident, steps)
    cand = float(np.mean(list(r.counts)))
    r.drain()
    fwd_ms, first_ms = r.net.profile_forward(10)
    r.close()
    per = ms / steps
    return {"workload": conf["name"], "batch": conf["batch"], "ms_per_step": per, "images_per_s": conf["batch"] / per * 1e3,
            "tflops": conf["flop"] * conf["batch"] / per * 1e-9, "forward_ms": fwd_ms, "mean_candidates_per_image": cand,
            "kept_records_per_step": int(nrec), "steps": steps, "clocks": sampler.summary(*win) if sampler else None}


def dropin_latency(dn, sampler, iters=30):
    """the path a `darknet detect` user takes, batch 1, through the REFERENCE API only (python/darknet.py:125-143 /
    detector.c:596-603): network_predict (pageable host fp32 in, head l.output back on the host) + get_network_boxes +
    do_nms_sort + free_detections"""
    from yolo_tensorflow_b200 import synth
    cfg, wpath = prepare_files(MODEL, SIZE, 1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(2); os.dup2(devnull, 2)
    try:
        net = dn.Network(cfg, wpath, precision=dn.PREC_BF16)
    finally:
        os.dup2(saved, 2); os.close(saved); os.close(devnull)
    x = np.ascontiguousarray(synth.make_images(1, 3, SIZE, SIZE, 1002))
    xp = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    num = ctypes.c_int(0)
    t = {"predict": [], "boxes": [], "nms": [], "total": []}
    t_begin = time.time()
    for it in range(iters + 3):
        a = time.perf_counter()
        dn.network_predict(net.ptr, xp)
        b = time.perf_counter()
        dets = dn.get_network_boxes(net.ptr, SIZE, SIZE, THRESH, .5, None, 1, ctypes.byref(num))
        c = time.perf_counter()
        dn.do_nms_sort(dets, num.value, 80, NMS)
        d = time.perf_counter()
        dn.free_detections(dets, num.value)
        e = time.perf_counter()
        if it >= 3:
            t["predict"].append(b - a); t["boxes"].append(c - b); t["nms"].append(d - c); t["total"].append(e - a)
    t_end = time.time()
    net.close()
    med = {k: 1e3 * sorted(v)[len(v) // 2] for k, v in t.items()}
    return {"workload": "YOLOv3 416x416 batch 1 through network_predict + get_network_boxes + do_nms_sort + free_detections (reference API, host in / host out)",
            "ms_per_image": med["total"], "images_per_s": 1e3 / med["total"], "predict_ms": med["predict"], "get_network_boxes_ms": med["boxes"],
            "do_nms_sort_ms": med["nms"], "candidates": int(num.value), "iters": iters, "clocks": sampler.summary(t_begin, t_end) if sampler else None}


def dump_outputs(out_dir, rec, counts):
    """the last timed step's result as .npy files, so that two builds can be compared output for output: the kept
    (box, class) records of every image, ordered by (image, box id, class) because the device may emit them in any order,
    and the per-image candidate counts before NMS.  Integer fields are stored as float64, which holds them exactly.
    Under torchrun, rank 0 writes the gathered records of every rank (global image numbers) but only its own images'
    counts: counts.npy covers images 0..BATCH-1."""
    os.makedirs(out_dir, exist_ok=True)
    rec = rec[np.lexsort((rec["cls"], rec["box_id"], rec["image"]))]
    arrays = {"counts": np.asarray(counts, np.float64), "image": rec["image"].astype(np.float64),
              "box_id": rec["box_id"].astype(np.float64), "cls": rec["cls"].astype(np.float64),
              "prob": rec["prob"].astype(np.float32), "objectness": rec["objectness"].astype(np.float32),
              "bbox": np.stack([rec["bbox"][k] for k in "xywh"], axis=1).astype(np.float32)}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_T0 = time.time()


def note(rank, msg):
    """progress line on stderr (rank 0): if a run is cut off, the log says in which phase"""
    if rank == 0:
        print("[bench %6.1f s] %s" % (time.time() - _T0, msg), file=sys.stderr, flush=True)


def main_engine(args):
    import torch
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    note(rank, "torch imported, world %d" % world)
    torch.cuda.set_device(local)
    if world > 1:
        # torch.distributed is the control plane only (rendezvous, barriers, max over ranks, the 128-byte NCCL id); the data-path
        # collectives are the library's own NCCL calls.  B200_BENCH_CONTROL=gloo keeps torch off NCCL altogether.
        if os.environ.get("B200_BENCH_CONTROL", "nccl") == "gloo":
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    note(rank, "process group up")
    from yolo_tensorflow_b200 import synth, darknet as dn
    dn.set_gpu(local)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                               # nvidia-smi needs a moment to come up: start it before anything else

    # ---- headline: C3, batch 64 per GPU -----------------------------------------------------------------
    if rank == 0:
        prepare_files(MODEL, SIZE, BATCH)
    if world > 1:
        dist.barrier()
    # weights: rank 0 reads the .weights file, folds / repacks / uploads; the other ranks only parse the cfg and receive the
    # finished parameter arena with ONE NCCL broadcast issued by the library (b200_comm_broadcast_weights, SURVEY §8e)
    run = Runner(dn, torch, HEAD, BATCH, rank, world, local, load_weights=(rank == 0))
    if world > 1:
        run.join(dist, image_base=rank * BATCH, gather=True)
    note(rank, "headline network planned, weights on every rank")
    x_host = run.load_resident(1002 + rank)           # per-rank image shard: a different seeded batch on every rank
    in_bytes = BATCH * 3 * SIZE * SIZE * 4
    net = run.net

    for _ in range(max(args.warmup, 3)):
        run.step_resident()
    launches0 = dn.lib.b200_launch_count()
    ms, nrec, win = run.timed(dist, run.step_resident, args.steps)
    launches = dn.lib.b200_launch_count() - launches0
    cand = float(np.mean(list(run.counts)))
    value = world * BATCH * args.steps / (ms / 1000.0)
    if args.dump_outputs and rank == 0:               # before drain(): it overwrites the records and counts of the last step
        dump_outputs(args.dump_outputs, np.ctypeslib.as_array(run.out, shape=(run.max_out,))[:nrec], list(run.counts))
    run.drain()                                       # the forward pass pre-enqueued for a step that will not come
    total_records = int(nrec)                         # on rank 0 with the gather on: the records of ALL ranks for the last step

    note(rank, "headline timed (%.3f ms per step)" % (ms / args.steps))
    # ---- e2e (a): fp32 NCHW host batches, as network_predict takes them ---------------------------------
    x_host2 = torch.from_numpy(synth.make_images(BATCH, 3, SIZE, SIZE, 2002 + rank)).pin_memory()
    host_batches = [x_host, x_host2]
    state = {"k": 0}

    def step_fp32():
        k = state["k"]; state["k"] = k + 1
        # results of batch k; the H2D of batch k+1 is started inside the call, right after batch k became current
        return dn.lib.b200_detect_submitted(net.ptr, host_batches[(k + 1) % 2].data_ptr(), SIZE, SIZE, THRESH, NMS, 1, run.out, run.max_out, run.counts)

    dn.lib.b200_submit_batch(net.ptr, host_batches[0].data_ptr())      # prime the pipeline: every timed step still copies one batch
    for _ in range(2):
        step_fp32()
    ms_fp32, nrec_fp32, _ = run.timed(dist, step_fp32, args.steps)
    dn.lib.b200_detect_submitted(net.ptr, None, SIZE, SIZE, THRESH, NMS, 1, run.out, run.max_out, run.counts)     # drain
    e2e_fp32 = world * BATCH * args.steps / (ms_fp32 / 1000.0)

    # ---- e2e (b): decoded uint8 pictures in, device letterbox, records out ---------------------------------
    rng = np.random.default_rng(3000 + rank)
    pics = torch.from_numpy(rng.integers(0, 256, (2, BATCH, SRC_H, SRC_W, 3), dtype=np.uint8)).pin_memory()
    ptrs = [(ctypes.c_void_p * BATCH)(*[pics[s, i].data_ptr() for i in range(BATCH)]) for s in range(2)]
    ws, hs = (ctypes.c_int * BATCH)(*([SRC_W] * BATCH)), (ctypes.c_int * BATCH)(*([SRC_H] * BATCH))
    u8_bytes = BATCH * SRC_H * SRC_W * 3
    state8 = {"k": 0}

    def step_u8():
        k = state8["k"]; state8["k"] = k + 1
        # upload + letterbox batch k+1 (stream-ordered behind batch k's forward pass), then collect batch k's records while
        # batch k+1's forward pass is already enqueued; boxes are mapped back with each picture's own size (w = h = 0)
        dn.lib.b200_letterbox_batch_u8(net.ptr, ptrs[(k + 1) % 2], ws, hs, BATCH)
        return dn.lib.b200_detect_submitted(net.ptr, RESIDENT, 0, 0, THRESH, NMS, 1, run.out, run.max_out, run.counts)

    dn.lib.b200_letterbox_batch_u8(net.ptr, ptrs[0], ws, hs, BATCH)
    dn.lib.b200_submit_batch(net.ptr, RESIDENT)
    for _ in range(2):
        step_u8()
    ms_u8, nrec_u8, _ = run.timed(dist, step_u8, args.steps)
    dn.lib.b200_detect_submitted(net.ptr, None, 0, 0, THRESH, NMS, 1, run.out, run.max_out, run.counts)           # drain
    e2e_u8 = world * BATCH * args.steps / (ms_u8 / 1000.0)

    note(rank, "e2e loops timed")
    # ---- roofline of the dominant kernel family (rank 0) -------------------------------------------------
    roofline = None
    if rank == 0:
        pk = peaks()
        fwd_ms, first_ms = net.profile_forward(20)
        n_conv, conv_flops, conv_bytes = conv_family(net, BATCH)
        conv_ms = fwd_ms - first_ms                  # every launch of the pass but the first layer is a conv_tc kernel (asserted below)
        others = [net.kernel(i) for i in range(1, net.n) if not net.kernel(i).startswith("conv_tc")
                  and net.kernel(i) not in ("fused", "alias", "concat_in_place", "yolo_forward")]
        achieved = conv_flops / (conv_ms / 1000.0) / 1e12 if conv_ms > 0 else 0.0
        traffic = None                      # DRAM bytes moved by the conv_tc family per step, from the committed ncu capture
        for name in ("r2_conv_tc_dram_traffic.json", "r1_conv_tc_dram_traffic.json"):
            tpath = os.path.join(REPO, "profiles", name)
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get("dram_bytes_total")
                traffic_src = name
                break
        roofline = {"bound": "tensor", "kernel": "conv_tc family (tcgen05 implicit-GEMM convolutions, %d launches/step)" % n_conv,
                    "achieved": achieved, "peak": pk["burst"], "unit": "TFLOP/s", "frac": achieved / pk["burst"],
                    "frac_burst": achieved / pk["burst"], "frac_sustained": achieved / pk["sustained"],
                    "peak_burst": pk["burst"], "peak_sustained": pk["sustained"], "peak_source": pk["source"],
                    "peak_note": "the timed region lasts ~0.1 s at full clocks, so the burst figure is the denominator of `frac`",
                    "traffic": traffic,
                    "traffic_note": "dram__bytes_read+write summed over the conv_tc launches of one step (profiles/%s); algorithmic "
                                    "activation+weight bytes of those layers at bf16: %.2f GB" % (traffic_src if traffic else "-", conv_bytes / 1e9),
                    "conv_ms_per_step": conv_ms, "forward_ms": fwd_ms, "first_layer_ms": first_ms,
                    "timing": "b200_profile_forward: CUDA events around the whole pass as the step enqueues it (no per-layer brackets), minus the first layer",
                    "non_conv_launches_in_pass": others,
                    "why_not_higher": "DESIGN.md section 5: (1) every launch pays a batch-independent 10-25 us (profiles/r2_launch_anatomy.txt); (2) the "
                                      "cross-layer persistent kernel that removes the boundaries (B200_FLOW=1, bit-identical) reaches 82 % tensor-issue "
                                      "occupancy and is 1-3 % slower: the chip clocks down under sustained tensor load (profiles/r2_flow_*.txt); (3) the "
                                      "tensor pipe alone runs a 3x3 layer at 1709 TFLOP/s, operand delivery holds the mainloop at 0.47 us per k-block "
                                      "instead of 0.375 (profiles/r2_operand_traffic_probe.txt, r2_ncu_operand_path.txt)",
                    "conv_tflop_per_step": conv_flops / 1e12,
                    "whole_step_tflops_per_gpu": FLOP_PER_IMAGE * BATCH / (ms / args.steps) * 1e-9,
                    "whole_step_frac_burst": FLOP_PER_IMAGE * BATCH / (ms / args.steps) * 1e-9 / pk["burst"]}
    head_clocks = sampler.summary(*win) if sampler else None
    run.close()

    note(rank, "roofline record done")
    # ---- C4: 608x608, 256 images per step split over the ranks (strong scaling), records gathered to rank 0 ----------
    c4 = None
    if not args.headline_only:
        conf = CONFIGS["C4"]
        lo, hi = (rank * conf["batch"]) // world, ((rank + 1) * conf["batch"]) // world
        r4 = Runner(dn, torch, conf, hi - lo, rank, world, local, load_weights=(rank == 0))
        if world > 1:
            r4.join(dist, image_base=lo, gather=True)
        r4.load_resident(4000 + rank)
        steps4 = max(3, min(args.steps, 10))
        for _ in range(3):
            r4.step_resident()
        ms4, nrec4, win4 = r4.timed(dist, r4.step_resident, steps4)
        cand4 = float(np.mean(list(r4.counts)))
        r4.drain()
        r4.close()
        if rank == 0:
            per = ms4 / steps4
            c4 = {"metric": "YOLOv3-608 images/s, 256 images per step split over the GPUs", "workload": conf["name"], "value": conf["batch"] / per * 1e3,
                  "unit": "images/s", "scaling": "strong", "n_gpus": world, "images_per_gpu": hi - lo, "ms_per_step": per, "steps": steps4,
                  "tflops_aggregate": conf["flop"] * conf["batch"] / per * 1e-9, "mean_candidates_per_image": cand4,
                  "records_gathered_on_rank0_per_step": int(nrec4), "gather": "ncclSend/ncclRecv of fixed record slots inside the step (b200_comm_set_gather)" if world > 1 else "single GPU",
                  "clocks": sampler.summary(*win4) if sampler else None}

    note(rank, "C4 done")
    # ---- the other configurations and the drop-in latency (one GPU only) -----------------------------------------
    other, dropin = None, None
    if world == 1 and not args.headline_only:
        other = {}
        for key in ("C1", "C2", "C5", "608x32"):
            other[key] = secondary(dn, torch, dist, key, sampler, max(5, min(args.steps, 10)), args.warmup, rank, world, local)
        dropin = dropin_latency(dn, sampler)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_reference_run(4, 1)
            cpu = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        rec_bytes = 36
        e2e_records = {"u8": (e2e_u8, ms_u8, u8_bytes, nrec_u8), "fp32": (e2e_fp32, ms_fp32, in_bytes, nrec_fp32)}
        ev, ems, ebytes, erec = e2e_records["u8" if E2E_INPUT == "u8" else "fp32"]
        line = {"metric": "YOLOv3-416 images/s (conv+decode+NMS)", "value": value, "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": f"YOLOv3 {SIZE}x{SIZE} batch {BATCH} per GPU, bf16 activations, fp32 accumulate; step = forward + decode + NMS",
                           "thresh": THRESH, "nms": NMS, "mean_candidates_per_image": cand, "kept_records_last_step": total_records,
                           "l2": "working set per step (133 MB input + >5 GB activations) exceeds the 126 MB L2; no explicit flush",
                           "pipelining": "value and e2e both use b200_detect_submitted: step k+1's forward is enqueued before step k's records are awaited",
                           "weights": "seed-0 synthetic, damped heads (yolo_tensorflow_b200/synth.py); undamped / thresh .005 stress settings: tests/test_gpu_parity.py::test_nms_stress_configuration",
                           "multi_gpu": "image-sharded, weights broadcast once and records gathered to rank 0 by the library's own NCCL calls, no per-layer collective"},
                "e2e": {"value": ev, "unit": "images/s", "h2d_bytes_per_step": int(ebytes), "d2h_bytes_per_step": int(erec) * rec_bytes + 4 * BATCH + 4,
                        "ms_per_step": ems / args.steps,
                        "input": ("64 decoded uint8 RGB pictures of %dx%d (pinned) -> b200_letterbox_batch_u8 -> b200_detect_submitted" % (SRC_W, SRC_H))
                        if E2E_INPUT == "u8" else "pinned fp32 NCHW batch -> b200_detect_submitted"},
                "e2e_u8": {"value": e2e_u8, "unit": "images/s", "h2d_bytes_per_step": int(u8_bytes), "ms_per_step": ms_u8 / args.steps},
                "e2e_fp32_nchw": {"value": e2e_fp32, "unit": "images/s", "h2d_bytes_per_step": int(in_bytes), "ms_per_step": ms_fp32 / args.steps},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": head_clocks,
                "c4": c4, "other_configs": other, "dropin": dropin}
        print(json.dumps(line))
    if sampler:
        sampler.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    if os.environ.get("B200_BENCH_WATCHDOG"):            # debugging aid: dump every thread's Python stack and exit after N seconds
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["B200_BENCH_WATCHDOG"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline and of the two e2e loops, exactly; the bounded sections clamp it and report the "
                         "count they ran: c4 to 3..10, other_configs to 5..10, --impl reference to 1..8 (cpu_baseline always times 4)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip C4, the other configurations and the drop-in latency")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records and counts of the headline's last timed step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs covers this engine's records only, not those of --impl reference")
    if a.impl == "reference":
        main_reference(a)
    else:
        main_engine(a)
