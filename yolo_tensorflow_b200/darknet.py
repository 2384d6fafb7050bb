"""ctypes binding of libdarknet.so — same names, argument meaning and struct layouts as the reference
wrapper (Darknet2Tensorflow/darknet-master/python/darknet.py:20-143), so code written against it keeps
working, plus the additive batched entry points of include/b200_engine.h.

Importing this module fails loudly when the native library has not been built: there is no Python or
CPU fallback for any compute call.
"""
import os
from ctypes import (CDLL, POINTER, RTLD_GLOBAL, Structure, c_char_p, c_float, c_int, c_size_t, c_ubyte,
                    c_ulonglong, c_void_p, byref, pointer)

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200_DARKNET_LIB", os.path.join(_HERE, "lib", "libdarknet.so"))
if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "or `make -C yolo_tensorflow_b200/csrc` (no CPU fallback exists)")


class BOX(Structure):
    _fields_ = [("x", c_float), ("y", c_float), ("w", c_float), ("h", c_float)]


class DETECTION(Structure):
    _fields_ = [("bbox", BOX), ("classes", c_int), ("prob", POINTER(c_float)), ("mask", POINTER(c_float)),
                ("objectness", c_float), ("sort_class", c_int)]


class IMAGE(Structure):
    _fields_ = [("w", c_int), ("h", c_int), ("c", c_int), ("data", POINTER(c_float))]


class METADATA(Structure):
    _fields_ = [("classes", c_int), ("names", POINTER(c_char_p))]


class B200_DET(Structure):
    """include/b200_engine.h b200_det: one surviving (box, class) pair of the fused device path."""
    _fields_ = [("image", c_int), ("cls", c_int), ("box_id", c_int), ("prob", c_float), ("objectness", c_float),
                ("bbox", BOX)]


lib = CDLL(LIB_PATH, RTLD_GLOBAL)

# ---- reference surface (python/darknet.py:48-115) --------------------------------------------------
lib.network_width.argtypes = [c_void_p]; lib.network_width.restype = c_int
lib.network_height.argtypes = [c_void_p]; lib.network_height.restype = c_int
predict = lib.network_predict
predict.argtypes = [c_void_p, POINTER(c_float)]; predict.restype = POINTER(c_float)
network_predict = predict
set_gpu = lib.cuda_set_device; set_gpu.argtypes = [c_int]
make_image = lib.make_image; make_image.argtypes = [c_int, c_int, c_int]; make_image.restype = IMAGE
get_network_boxes = lib.get_network_boxes
get_network_boxes.argtypes = [c_void_p, c_int, c_int, c_float, c_float, POINTER(c_int), c_int, POINTER(c_int)]
get_network_boxes.restype = POINTER(DETECTION)
make_network_boxes = lib.make_network_boxes
make_network_boxes.argtypes = [c_void_p, c_float, POINTER(c_int)]; make_network_boxes.restype = POINTER(DETECTION)
free_detections = lib.free_detections; free_detections.argtypes = [POINTER(DETECTION), c_int]
free_ptrs = lib.free_ptrs; free_ptrs.argtypes = [POINTER(c_void_p), c_int]
reset_rnn = lib.reset_rnn; reset_rnn.argtypes = [c_void_p]
load_net = lib.load_network; load_net.argtypes = [c_char_p, c_char_p, c_int]; load_net.restype = c_void_p
parse_network_cfg = lib.parse_network_cfg; parse_network_cfg.argtypes = [c_char_p]; parse_network_cfg.restype = c_void_p
load_weights = lib.load_weights; load_weights.argtypes = [c_void_p, c_char_p]
free_network = lib.free_network; free_network.argtypes = [c_void_p]
set_batch_network = lib.set_batch_network; set_batch_network.argtypes = [c_void_p, c_int]
do_nms_obj = lib.do_nms_obj; do_nms_obj.argtypes = [POINTER(DETECTION), c_int, c_int, c_float]
do_nms_sort = lib.do_nms_sort; do_nms_sort.argtypes = [POINTER(DETECTION), c_int, c_int, c_float]
free_image = lib.free_image; free_image.argtypes = [IMAGE]
letterbox_image = lib.letterbox_image; letterbox_image.argtypes = [IMAGE, c_int, c_int]; letterbox_image.restype = IMAGE
resize_image = lib.resize_image; resize_image.argtypes = [IMAGE, c_int, c_int]; resize_image.restype = IMAGE
load_meta = lib.get_metadata; lib.get_metadata.argtypes = [c_char_p]; lib.get_metadata.restype = METADATA
load_image = lib.load_image_color; load_image.argtypes = [c_char_p, c_int, c_int]; load_image.restype = IMAGE
rgbgr_image = lib.rgbgr_image; rgbgr_image.argtypes = [IMAGE]
predict_image = lib.network_predict_image; predict_image.argtypes = [c_void_p, IMAGE]; predict_image.restype = POINTER(c_float)

# ---- additive surface (include/b200_engine.h) --------------------------------------------------------
PREC_BF16, PREC_FP32 = 0, 1
lib.b200_set_default_precision.argtypes = [c_int]
lib.b200_set_default_fusion.argtypes = [c_int]
lib.b200_get_precision.argtypes = [c_void_p]; lib.b200_get_precision.restype = c_int
lib.b200_set_conv_backend.argtypes = [c_void_p, c_int]
lib.b200_set_head_sync.argtypes = [c_void_p, c_int]
lib.b200_set_flow.argtypes = [c_void_p, c_int]
lib.b200_flow_stats.argtypes = [c_void_p, POINTER(c_ulonglong)]
lib.b200_flow_trace.argtypes = [c_void_p, c_int, c_void_p, c_int, POINTER(c_int), c_int]; lib.b200_flow_trace.restype = c_int
lib.b200_flow_count.argtypes = [c_void_p]; lib.b200_flow_count.restype = c_int
lib.b200_flow_desc.argtypes = [c_void_p, c_int, POINTER(c_int), POINTER(c_int)]; lib.b200_flow_desc.restype = c_char_p
lib.b200_fetch_layer_output.argtypes = [c_void_p, c_int, POINTER(c_float)]
lib.b200_set_layer_output.argtypes = [c_void_p, c_int, POINTER(c_float)]
lib.b200_run_layers.argtypes = [c_void_p, c_int, c_int]
lib.b200_layer_kernel.argtypes = [c_void_p, c_int]; lib.b200_layer_kernel.restype = c_char_p
lib.b200_launch_count.restype = c_ulonglong
lib.b200_layer_plan.argtypes = [c_void_p, c_int]; lib.b200_layer_plan.restype = c_char_p
lib.b200_network_layers.argtypes = [c_void_p]; lib.b200_network_layers.restype = c_int
lib.b200_letterbox_batch_u8.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_int), POINTER(c_int), c_int]; lib.b200_letterbox_batch_u8.restype = c_int
lib.b200_letterbox_batch.argtypes = [c_void_p, POINTER(IMAGE), c_int]; lib.b200_letterbox_batch.restype = c_int
lib.b200_fetch_input.argtypes = [c_void_p, c_void_p, c_int]; lib.b200_fetch_input.restype = None
lib.b200_coco_image_id.argtypes = [c_char_p]; lib.b200_coco_image_id.restype = c_int
lib.b200_append_coco.argtypes = [c_char_p, POINTER(B200_DET), c_int, POINTER(c_char_p), POINTER(c_int), POINTER(c_int)]; lib.b200_append_coco.restype = c_int
lib.b200_append_voc.argtypes = [c_char_p, POINTER(c_char_p), c_int, POINTER(B200_DET), c_int, POINTER(c_char_p), POINTER(c_int), POINTER(c_int)]; lib.b200_append_voc.restype = c_int
lib.b200_validate_images.argtypes = [c_void_p, POINTER(c_void_p), POINTER(c_int), POINTER(c_int), POINTER(c_char_p), c_int, c_char_p, c_char_p, c_char_p,
                                     POINTER(c_char_p), c_float, c_float]
lib.b200_validate_images.restype = c_int
lib.b200_append_imagenet.argtypes = [c_char_p, POINTER(B200_DET), c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]; lib.b200_append_imagenet.restype = c_int
lib.resize_network.argtypes = [c_void_p, c_int, c_int]; lib.resize_network.restype = c_int
lib.b200_layer_info.argtypes = [c_void_p, c_int, POINTER(c_int)]; lib.b200_layer_info.restype = c_int
lib.b200_layer_output_host.argtypes = [c_void_p, c_int]; lib.b200_layer_output_host.restype = POINTER(c_float)
lib.b200_weights_arena.argtypes = [c_void_p, POINTER(c_size_t)]; lib.b200_weights_arena.restype = c_void_p
lib.b200_engine_of.argtypes = [c_void_p]; lib.b200_engine_of.restype = c_void_p
lib.b200_engine_forward_resident.argtypes = [c_void_p, c_void_p]
lib.b200_engine_input_device.argtypes = [c_void_p]; lib.b200_engine_input_device.restype = c_void_p
lib.b200_engine_sync.argtypes = [c_void_p]
lib.b200_engine_stream.argtypes = [c_void_p]; lib.b200_engine_stream.restype = c_void_p
lib.b200_profile_layers.argtypes = [c_void_p, c_int, POINTER(c_float)]
lib.b200_profile_forward.argtypes = [c_void_p, c_int, POINTER(c_float)]
lib.b200_profile_tail.argtypes = [c_void_p, c_int, c_int, c_float, c_float, c_int, POINTER(c_float)]
lib.get_network_boxes_batch.argtypes = [c_void_p, c_int, c_int, c_int, c_float, c_float, POINTER(c_int), c_int, POINTER(c_int)]
lib.get_network_boxes_batch.restype = POINTER(DETECTION)
lib.b200_detect_batch.argtypes = [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_int, POINTER(B200_DET), c_int, POINTER(c_int)]
lib.b200_detect_batch.restype = c_int
lib.b200_submit_batch.argtypes = [c_void_p, c_void_p]
lib.b200_detect_submitted.argtypes = [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_int, POINTER(B200_DET), c_int, POINTER(c_int)]
lib.b200_detect_submitted.restype = c_int
lib.b200_comm_unique_id.argtypes = [c_void_p, c_int]; lib.b200_comm_unique_id.restype = c_int
lib.b200_comm_init.argtypes = [c_void_p, c_void_p, c_int, c_int]; lib.b200_comm_init.restype = c_int
lib.b200_comm_broadcast_weights.argtypes = [c_void_p, c_int]; lib.b200_comm_broadcast_weights.restype = c_int
lib.b200_comm_set_gather.argtypes = [c_void_p, c_int, c_int, c_int]; lib.b200_comm_set_gather.restype = c_int
lib.b200_comm_destroy.argtypes = [c_void_p]
lib.b200_classify_batch.argtypes = [c_void_p, c_void_p, c_int, POINTER(c_int), POINTER(c_float)]; lib.b200_classify_batch.restype = c_int
lib.b200_classify_submitted.argtypes = [c_void_p, c_void_p, c_int, POINTER(c_int), POINTER(c_float)]
lib.b200_classify_submitted.restype = c_int
lib.b200_top_k_arrays.argtypes = [POINTER(c_float), c_int, c_int, c_int, POINTER(c_int)]
lib.top_k.argtypes = [POINTER(c_float), c_int, c_int, POINTER(c_int)]
lib.b200_nms_sort_arrays.argtypes = [POINTER(c_float), POINTER(c_float), c_int, c_int, c_float]
lib.b200_nms_obj_arrays.argtypes = [POINTER(c_float), POINTER(c_float), c_int, c_float, POINTER(c_ubyte)]

LAYER_INFO_FIELDS = ("type", "batch", "inputs", "outputs", "h", "w", "c", "out_h", "out_w", "out_c", "n", "size",
                     "stride", "pad", "classes", "coords", "batch_normalize", "activation", "nweights", "index")
LAYER_TYPES = ("CONVOLUTIONAL DECONVOLUTIONAL CONNECTED MAXPOOL SOFTMAX DETECTION DROPOUT CROP ROUTE COST NORMALIZATION "
               "AVGPOOL LOCAL SHORTCUT ACTIVE RNN GRU LSTM CRNN BATCHNORM NETWORK XNOR REGION YOLO REORG UPSAMPLE "
               "LOGXENT L2NORM BLANK").split()


def _fptr(a):
    return a.ctypes.data_as(POINTER(c_float))


class Network:
    """Convenience owner of a `network*` (what the reference wrapper passes around as c_void_p)."""

    def __init__(self, cfg, weights=None, precision=None, fuse=None):
        if precision is not None:
            lib.b200_set_default_precision(int(precision))
        if fuse is not None:
            lib.b200_set_default_fusion(int(bool(fuse)))
        self.ptr = parse_network_cfg(str(cfg).encode())
        if precision is not None:
            lib.b200_set_default_precision(-1)
        if fuse is not None:
            lib.b200_set_default_fusion(-1)
        if weights:
            load_weights(self.ptr, str(weights).encode())
        self.n = lib.b200_network_layers(self.ptr)
        self.w, self.h = lib.network_width(self.ptr), lib.network_height(self.ptr)
        self.layers = [self.layer_info(i) for i in range(self.n)]
        self.batch = self.layers[0]["batch"]

    def resize(self, w, h):
        """resize_network (network.c:358): new input size, same parameters; returns 0, or -1 for unresizable layers."""
        rc = lib.resize_network(self.ptr, int(w), int(h))
        self.w, self.h = lib.network_width(self.ptr), lib.network_height(self.ptr)
        self.layers = [self.layer_info(i) for i in range(self.n)]
        return rc

    def close(self):
        if self.ptr:
            free_network(self.ptr)
            self.ptr = None

    def layer_info(self, i):
        buf = (c_int * 20)()
        lib.b200_layer_info(self.ptr, i, buf)
        d = dict(zip(LAYER_INFO_FIELDS, list(buf)))
        d["type_name"] = LAYER_TYPES[d["type"]]
        return d

    def kernel(self, i):
        return lib.b200_layer_kernel(self.ptr, i).decode()

    def predict(self, x):
        """network_predict: x is float32 [batch, c, h, w] (C-contiguous); returns the last layer's host output."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        out = predict(self.ptr, _fptr(x))
        last = self.layers[-1]
        return np.ctypeslib.as_array(out, shape=(self.batch * last["outputs"],)).copy()

    def layer_output(self, i):
        """device -> host fp32 in darknet layout, shape [batch, outputs]"""
        li = self.layers[i]
        out = np.empty((self.batch, li["outputs"]), dtype=np.float32)
        lib.b200_fetch_layer_output(self.ptr, i, _fptr(out))
        return out

    def set_layer_output(self, i, a):
        a = np.ascontiguousarray(a, dtype=np.float32)
        lib.b200_set_layer_output(self.ptr, i, _fptr(a))

    def run_layers(self, start, end):
        lib.b200_run_layers(self.ptr, start, end)

    def profile_layers(self, iters=3):
        ms = np.zeros(self.n, dtype=np.float32)
        lib.b200_profile_layers(self.ptr, iters, _fptr(ms))
        return ms

    def profile_forward(self, iters=5):
        """(whole forward pass ms, first layer ms) as the serving loop runs it"""
        ms = np.zeros(2, dtype=np.float32)
        lib.b200_profile_forward(self.ptr, iters, _fptr(ms))
        return float(ms[0]), float(ms[1])

    def profile_tail(self, w, h, thresh, nms, iters=3):
        ms = np.zeros(3, dtype=np.float32)
        lib.b200_profile_tail(self.ptr, w, h, thresh, nms, iters, _fptr(ms))
        return ms

    def stream_ptr(self):
        return lib.b200_engine_stream(self.ptr)

    def input_device_ptr(self):
        return lib.b200_engine_input_device(lib.b200_engine_of(self.ptr))

    def weights_arena(self):
        n = c_size_t(0)
        p = lib.b200_weights_arena(self.ptr, byref(n))
        return p, n.value

    def set_head_sync(self, on):
        lib.b200_set_head_sync(self.ptr, int(on))

    def set_flow(self, on):
        """1 (default): flow-capable runs of convolutions execute as one persistent kernel; 0: one launch per layer"""
        lib.b200_set_flow(self.ptr, int(on))

    def flow_stats(self):
        """(ns producers blocked on dependencies, ns residual loaders blocked, blocking waits) since the last call"""
        v = (c_ulonglong * 5)()
        lib.b200_flow_stats(self.ptr, v)
        return int(v[0]), int(v[1]), int(v[2]), int(v[3]), int(v[4])

    def flow_trace(self, k, max_items=1 << 20):
        """(stamps [items][5] uint64: 4 x ns + pair | position << 16, item0 [layers + 1]) of flow k's last launch; needs B200_FLOW_TRACE=1 when the net was parsed"""
        buf = np.zeros((max_items, 5), dtype=np.uint64)
        item0 = (c_int * 64)()
        n = lib.b200_flow_trace(self.ptr, k, buf.ctypes.data, max_items, item0, 64)
        return buf[:n], list(item0)

    def flows(self):
        """[(first layer, last layer, plan text)] of the planned flows"""
        out = []
        for k in range(lib.b200_flow_count(self.ptr)):
            a, b = c_int(0), c_int(0)
            d = lib.b200_flow_desc(self.ptr, k, byref(a), byref(b)).decode()
            out.append((a.value, b.value, d))
        return out

    def boxes(self, b, w, h, thresh, relative=1):
        """get_network_boxes_batch -> (dets pointer, count); caller frees with free_detections"""
        num = c_int(0)
        dets = lib.get_network_boxes_batch(self.ptr, b, w, h, thresh, .5, None, relative, byref(num))
        return dets, num.value

    def letterbox_batch_u8(self, images):
        """device-side letterbox of decoded RGB images (list of HxWx3 uint8 arrays) into the network input; follow with
        detect_batch(None, 0, 0, ...) so every image's boxes are corrected with its own size"""
        imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        n = len(imgs)
        ptrs = (c_void_p * n)(*[im.ctypes.data for im in imgs])
        ws = (c_int * n)(*[im.shape[1] for im in imgs]); hs = (c_int * n)(*[im.shape[0] for im in imgs])
        return lib.b200_letterbox_batch_u8(self.ptr, ptrs, ws, hs, n)

    def letterbox_batch(self, images):
        """the same for darknet images (list of 3xHxW float32 arrays)"""
        arrs = [np.ascontiguousarray(im, dtype=np.float32) for im in images]
        ims = (IMAGE * len(arrs))(*[IMAGE(a.shape[2], a.shape[1], 3, a.ctypes.data_as(POINTER(c_float))) for a in arrs])
        return lib.b200_letterbox_batch(self.ptr, ims, len(arrs))

    def validate_images(self, images, paths, eval_type, prefix, outfile=None, names=None, thresh=.005, nms=.45):
        """validate_detector (examples/detector.c:364-487) over decoded HxWx3 uint8 images, batched; returns the record count"""
        imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        m = len(imgs)
        ptrs = (c_void_p * m)(*[im.ctypes.data for im in imgs])
        ws = (c_int * m)(*[im.shape[1] for im in imgs]); hs = (c_int * m)(*[im.shape[0] for im in imgs])
        cpaths = (c_char_p * m)(*[p.encode() for p in paths])
        cnames = (c_char_p * len(names))(*[n.encode() for n in names]) if names else None
        return lib.b200_validate_images(self.ptr, ptrs, ws, hs, cpaths, m, eval_type.encode() if eval_type else None, prefix.encode(),
                                        outfile.encode() if outfile else None, cnames, thresh, nms)

    def fetch_input(self, n):
        out = np.empty((n, 3, self.h, self.w), np.float32)
        lib.b200_fetch_input(self.ptr, out.ctypes.data_as(c_void_p), n)
        return out

    def detect_batch(self, x, w, h, thresh, nms, relative=1, max_out=1 << 20):
        """fused device path; x host float32 array or None (resident input). Returns (structured array, counts)."""
        out = (B200_DET * max_out)()
        counts = (c_int * self.batch)()
        xp = None
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32)
            xp = x.ctypes.data_as(c_void_p)
        n = lib.b200_detect_batch(self.ptr, xp, w, h, thresh, nms, relative, out, max_out, counts)
        rec = np.ctypeslib.as_array(out)[:n].copy() if n else np.zeros(0, dtype=np.dtype(B200_DET))
        return rec, np.array(list(counts))


    def classify_batch(self, x, top=5):
        """b200_classify_batch: x host float32 [batch, c, h, w], or None for the resident device input.  Returns
        (classes [batch, top] int32, probs [batch, top] float32): top_k of each image's probabilities, on the device."""
        classes = np.zeros((self.batch, top), np.int32)
        probs = np.zeros((self.batch, top), np.float32)
        xp = None
        if x is not None:
            x = np.ascontiguousarray(x, dtype=np.float32)
            xp = x.ctypes.data_as(c_void_p)
        n = lib.b200_classify_batch(self.ptr, xp, top, classes.ctypes.data_as(POINTER(c_int)), _fptr(probs))
        if n < 0:
            raise ValueError("b200_classify_batch refused the network or top=%d (see stderr)" % top)
        return classes, probs


def top_k_arrays(probs, top):
    """b200_top_k_arrays: the device top-k of every row of probs [rows, n] (top_k of utils.c per row) -> [rows, top] int32"""
    probs = np.ascontiguousarray(probs, np.float32)
    out = np.zeros((probs.shape[0], top), np.int32)
    lib.b200_top_k_arrays(_fptr(probs), probs.shape[0], probs.shape[1], top, out.ctypes.data_as(POINTER(c_int)))
    return out


def dets_to_arrays(dets, n, classes):
    """DETECTION* -> (boxes [n,4], objectness [n], probs [n,classes]) numpy copies"""
    boxes = np.zeros((n, 4), np.float32); obj = np.zeros(n, np.float32); probs = np.zeros((n, classes), np.float32)
    for i in range(n):
        d = dets[i]
        boxes[i] = (d.bbox.x, d.bbox.y, d.bbox.w, d.bbox.h)
        obj[i] = d.objectness
        probs[i] = np.ctypeslib.as_array(d.prob, shape=(classes,))
    return boxes, obj, probs


def nms_sort_arrays(boxes, probs, thresh):
    boxes = np.ascontiguousarray(boxes, np.float32); probs = np.array(probs, np.float32, copy=True, order="C")
    lib.b200_nms_sort_arrays(_fptr(boxes), _fptr(probs), boxes.shape[0], probs.shape[1], thresh)
    return probs


def detect(net, meta, image, thresh=.5, hier_thresh=.5, nms=.45):
    """python/darknet.py:125-143, unchanged semantics (do_nms_obj, relative=0)."""
    im = load_image(image, 0, 0)
    num = c_int(0)
    pnum = pointer(num)
    predict_image(net, im)
    dets = get_network_boxes(net, im.w, im.h, thresh, hier_thresh, None, 0, pnum)
    num = pnum[0]
    if nms:
        do_nms_obj(dets, num, meta.classes, nms)
    res = []
    for j in range(num):
        for i in range(meta.classes):
            if dets[j].prob[i] > 0:
                b = dets[j].bbox
                res.append((meta.names[i], dets[j].prob[i], (b.x, b.y, b.w, b.h)))
    res = sorted(res, key=lambda x: -x[1])
    free_image(im)
    free_detections(dets, num)
    return res


def classify(net, meta, im):
    """python/darknet.py classify, unchanged semantics: network_predict_image, then every class with its probability,
    most probable first."""
    out = predict_image(net, im)
    res = []
    for i in range(meta.classes):
        res.append((meta.names[i], out[i]))
    res = sorted(res, key=lambda x: -x[1])
    return res
