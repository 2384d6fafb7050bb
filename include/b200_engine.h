/*
 * b200_engine.h — the thin C-ABI layer between the darknet-compatible host code (plain C) and the
 * hand-written sm_100a CUDA kernels, plus the ADDITIVE batched entry points (SURVEY.md §8b "Batch
 * semantics").  Plain pointers and sizes only; no torch / C++ types cross this boundary.
 *
 * Everything here is exported from libdarknet.so next to the reference-compatible symbols declared
 * in darknet.h.  Functions that touch the device fail loudly (message on stderr + abort()) when no
 * CUDA device / driver is available: there is NO CPU fallback anywhere in the product path.
 */
#ifndef B200_ENGINE_H
#define B200_ENGINE_H
#include "darknet.h"
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- precision of the activation path ---------------------------------------------------------- */
#define B200_PREC_BF16 0   /* NHWC bf16 activations, tcgen05 implicit-GEMM convs, fp32 accumulate (default) */
#define B200_PREC_FP32 1   /* NHWC fp32 activations, CUDA-core fp32 convs: the rtol 1e-4 parity mode        */
void b200_set_default_precision(int prec);     /* applies to networks parsed afterwards (env B200_PRECISION=fp32|bf16 too) */
int  b200_get_precision(const network *net);

/* Layer fusion (default on; env B200_FUSE=0 turns it off): a [convolutional] -> [shortcut] pair runs as ONE kernel, the
 * residual add riding in the convolution epilogue; the convolution's own output is then never materialised and
 * b200_fetch_layer_output() on it aborts.  Applies to networks parsed afterwards; -1 restores the default. */
void b200_set_default_fusion(int on);
int  b200_get_default_fusion(void);

/* conv kernel selection for the bf16 path: 0 = auto (tcgen05 wherever the shape allows), 1 = force CUDA-core kernel */
void b200_set_conv_backend(network *net, int backend);

/* When 0, network_predict() leaves head-layer outputs on the device (no D2H of l.output / net->output);
 * the batched detection entry points below never need the host copy.  Default 1 = reference behaviour
 * (network.c:505, yolo_layer.c:359-362: heads are valid host fp32 NCHW after every predict). */
void b200_set_head_sync(network *net, int on);

/* Flows (planned only when env B200_FLOW=1 is set while the network is parsed): runs of tcgen05 convolution layers executed by
 * ONE persistent kernel in which a tile of layer n+1 starts as soon as the tiles of layer n it reads are stored, instead of at
 * a kernel boundary (csrc/dev/conv_tc_flow.cu).  Results are bit-identical to one launch per layer; on a power-managed B200 it
 * measured 1-3 % slower (DESIGN.md section 5), which is why it is opt-in.  b200_set_flow(net, 0) runs a planned flow's layers
 * one launch each.  b200_flow_desc: plan text of flow k and the first / last layer index it covers. */
void b200_set_flow(network *net, int on);
int  b200_flow_count(network *net);
const char *b200_flow_desc(network *net, int k, int *first, int *last);
/* profiling, 5 values: {ns the flows' TMA producers waited on dependencies, ns their residual loaders did, number of waits that
 * blocked} summed over all launches since the previous call; under B200_FLOW_TRACE=1 also {SM clock cycles, ns} of the first
 * flow's last launch (their ratio = the SM clock while it ran) */
void b200_flow_stats(network *net, unsigned long long *out5);
/* profiling (flows planned under B200_FLOW_TRACE=1 only, else returns 0): 5 values per item of flow k's last launch — device-clock
 * stamps (ns) inputs complete, first operands landed, last MMA issued, tile stored, then pair | position in its list << 16 — and the first item number of each member layer */
int  b200_flow_trace(network *net, int k, unsigned long long *out, int max_items, int *item0, int max_layers);
/* host-only self-test of the flow scheduler (no device needed): a chain of n layers over a batch x hw x hw map,
 * spec[4k..4k+3] = {filter size 1|3, stride, input channels, filters}, is scheduled on `pairs` CTA pairs and the item lists are
 * replayed without the cost model; returns -1 when every item runs exactly once (no deadlock), else the first stuck item */
int  b200_flow_schedule_selftest(int n, const int *spec, int batch, int hw, int pairs, double *makespan_us, double *work_us);
/* host-only: the completion counters a consuming tile waits on (flow_dep_range) cover every input pixel its taps read;
 * -1 = yes for every tile, else the first offending tile */
int  b200_flow_dep_selftest(int batch, int in_h, int in_w, int size, int stride);

/* ---- opaque engine, one per network -------------------------------------------------------------- */
typedef struct b200_engine b200_engine;
b200_engine *b200_engine_of(const network *net);

/* host code → device, called by parse_network_cfg / load_weights / free_network */
b200_engine *b200_engine_create(network *net, int precision);   /* plans buffers from the layer array      */
void b200_engine_destroy(b200_engine *e);
void b200_engine_upload_weights(b200_engine *e, network *net);    /* BN folding + repack (+ bf16 cast) + H2D */
b200_engine *b200_engine_recreate(b200_engine *old, network *net); /* resize_network: re-plan, keep settings, re-upload */
void b200_engine_unpin_host(b200_engine *e);                      /* before host code frees / re-allocates l.output buffers */

/* forward_network replacement (network.c:188-211).  `input` is HOST fp32 NCHW, batch*inputs floats. */
void b200_engine_forward(b200_engine *e, network *net, const float *input);
/* same, but the input is ALREADY resident on the device (fp32 NCHW): the timed region of bench.py's `value` */
void b200_engine_forward_resident(b200_engine *e, network *net);
float *b200_engine_input_device(b200_engine *e);                  /* device fp32 NCHW staging buffer          */
void b200_engine_sync(b200_engine *e);

/* weights arena: one contiguous device allocation holding every folded/repacked parameter, so that
 * multi-GPU replicas are initialised with ONE NCCL broadcast (SURVEY.md §8e). */
void *b200_weights_arena(network *net, size_t *bytes);

/* ---- test / inspection hooks (teacher-forced per-layer parity) ----------------------------------- */
/* copies layer i's device output into host fp32 NCHW (darknet layout); `out` needs batch*outputs floats */
void b200_fetch_layer_output(network *net, int i, float *out);
/* overwrites layer i's device output from host fp32 NCHW */
void b200_set_layer_output(network *net, int i, const float *in);
/* runs layers [start, end) on the device using whatever currently sits in their input buffers */
void b200_run_layers(network *net, int start, int end);
/* name of the kernel family that executes layer i ("conv_tc", "conv_simt", "conv_stem", "maxpool", ...) */
const char *b200_layer_kernel(network *net, int i);
/* human-readable tiling plan of a tcgen05 convolution layer ("" for other layers) */
const char *b200_layer_plan(network *net, int i);
/* number of kernels launched by this library since process start (bench.py's gpu_launches) */
unsigned long long b200_launch_count(void);

/* the CUDA stream (cudaStream_t) every kernel of this network is launched on: time it with events recorded there */
void *b200_engine_stream(network *net);
/* average device milliseconds per layer over `iters` forwards (CUDA events between layers); ms has net->n entries */
void b200_profile_layers(network *net, int iters, float *ms);

/* device milliseconds of the forward pass exactly as the serving loop enqueues it (no per-layer brackets): ms[0] = whole pass,
 * ms[1] = the first layer alone; averaged over `iters` after one warm-up */
void b200_profile_forward(network *net, int iters, float *ms);

/* device milliseconds of the post-network tail on the current head outputs: ms[0] decode+compaction, ms[1] NMS, ms[2] collect */
void b200_profile_tail(network *net, int w, int h, float thresh, float nms_thresh, int iters, float *ms);

/* accessors for FFI callers: 20 ints = type, batch, inputs, outputs, h, w, c, out_h, out_w, out_c, n, size, stride, pad,
 * classes, coords, batch_normalize, activation, nweights, index */
int b200_network_layers(const network *net);
int b200_layer_info(const network *net, int i, int *out);
float *b200_layer_output_host(const network *net, int i);

/* ---- additive batched box extraction + NMS ------------------------------------------------------- */
/* get_network_boxes for batch item b (the reference only ever reads item 0: yolo_layer.c:281,326). */
detection *get_network_boxes_batch(network *net, int b, int w, int h, float thresh, float hier,
                                   int *map, int relative, int *num);

/* compact record produced by the fused device path: one per surviving (box, class) pair */
typedef struct {
    int   image;        /* batch index                      */
    int   cls;          /* class id                         */
    int   box_id;       /* global anchor index inside the image: concatenated heads, cell-major anchor-minor like get_*_detections */
    float prob;         /* objectness * class prob (post NMS, > thresh) */
    float objectness;
    box   bbox;         /* corrected exactly like correct_yolo_boxes / correct_region_boxes */
} b200_det;

/* network_predict + get_network_boxes + do_nms_sort for EVERY image of the batch, entirely on the device:
 * decode with warp-ballot compaction, class-wise bitmask NMS, and only the kept records cross PCIe.
 * `input` host fp32 NCHW (NULL = use the resident device input).  Returns the number of records written
 * to `out` (at most max_out); counts[b] (may be NULL) receives the per-image candidate count before NMS. */
/* Result writers (the step after the path, SURVEY 8f-2): the formats of examples/detector.c's print_cocos (:165-188),
 * print_detector_detections (:190-209) and print_imagenet_detections (:211-232), fed from b200_detect_batch records taken
 * with relative = 0 (pixel coordinates).  widths/heights/ids/paths are indexed by the record's image number. */
int  b200_coco_image_id(const char *filename);                       /* get_coco_image_id, detector.c:157 */
void b200_sort_records(b200_det *rec, int n);                         /* by (image, box, class): deterministic files */
int  b200_write_coco(FILE *fp, const b200_det *rec, int n, const char *const *image_paths, const int *widths, const int *heights);
int  b200_write_voc(FILE **fps, const b200_det *rec, int n, const char *const *ids, const int *widths, const int *heights);
int  b200_write_imagenet(FILE *fp, const b200_det *rec, int n, const int *image_ids, const int *widths, const int *heights);
int  b200_append_coco(const char *path, b200_det *rec, int n, const char *const *image_paths, const int *widths, const int *heights);
int  b200_append_voc(const char *prefix, const char *const *names, int classes, b200_det *rec, int n, const char *const *ids,
                     const int *widths, const int *heights);
int  b200_append_imagenet(const char *path, b200_det *rec, int n, const int *image_ids, const int *widths, const int *heights);

/* validate_detector (examples/detector.c:364-487) as a batched driver over m decoded images (RGB, HWC, 8 bit; paths[i] names
 * image i): device letterbox, forward, boxes corrected with each image's own size (pixels), NMS, result files — net->batch
 * images at a time through the pipelined serving loop.  eval "coco" -> <prefix>/<outfile|coco_results>.json, "imagenet" ->
 * <prefix>/<outfile|imagenet-detection>.txt, anything else (or NULL) -> <prefix>/<outfile|comp4_det_test_><names[class]>.txt;
 * the reference runs it with thresh .005 and nms .45 (:418-419).  Returns the number of records written, -1 on error. */
int  b200_validate_images(network *net, const unsigned char *const *rgb_hwc, const int *widths, const int *heights,
                          const char *const *paths, int m, const char *eval, const char *prefix, const char *outfile,
                          const char *const *names, float thresh, float nms);

/* Device-side preprocessing (the step before the path: letterbox_image + resize_image, image.c:960-979,1347-1390, and for
 * uint8 sources load_image_stb's HWC/255 conversion, image.c:1442-1464), bit-identical to the host functions.  n <= batch
 * images of individual sizes become the letterboxed network input in device memory; then call
 * b200_detect_batch(net, NULL, 0, 0, ...): w = h = 0 corrects each image's boxes with its own original size. */
int b200_letterbox_batch_u8(network *net, const unsigned char *const *images, const int *widths, const int *heights, int n);  /* RGB, HWC */
int b200_letterbox_batch(network *net, const image *images, int n);                                                            /* darknet images (fp32 CHW) */
void b200_fetch_input(network *net, float *dst, int images);      /* the device input buffer as host fp32 NCHW (inspection) */

/* network_predict + get_network_boxes + do_nms_sort for every image of the batch.  input: host fp32 NCHW, or NULL /
 * B200_INPUT_RESIDENT for what the device input buffer holds (e.g. after b200_letterbox_batch_u8). */
int b200_detect_batch(network *net, const float *input, int w, int h, float thresh, float nms_thresh,
                      int relative, b200_det *out, int max_out, int *counts);

/* Double-buffered serving loop (the e2e number of bench.py): b200_submit_batch starts the asynchronous H2D of a batch
 * (host fp32 NCHW, ideally pinned) into a spare device buffer and returns at once; b200_detect_submitted makes that batch
 * current, starts the H2D of `next_input` (may be NULL) into the buffer that just became free, and runs forward + decode +
 * NMS exactly like b200_detect_batch.  Pattern:
 *     submit(b[0]); for k: n = detect_submitted(b[k+1], ...)      -> results of b[k]
 * so the PCIe copy of batch k+1 hides under the compute of batch k.  A host buffer must stay valid until the call that
 * returns ITS results has returned. */
/* B200_INPUT_RESIDENT as `input` / `next_input`: nothing is copied from the host — the batch is what the engine's device
 * input buffer holds when the call is made (b200_letterbox_batch* writes there), and its forward pass is enqueued by that
 * call.  The loop
 *   b200_letterbox_batch_u8(batch 0); b200_submit_batch(net, B200_INPUT_RESIDENT);
 *   for k: b200_letterbox_batch_u8(batch k+1); b200_detect_submitted(net, B200_INPUT_RESIDENT, ...)   -> records of batch k
 * keeps the GPU busy across the result read-back exactly like the host-input loop; with w = h = 0 every batch's boxes are
 * corrected with the image sizes of ITS letterbox call. */
#define B200_INPUT_RESIDENT ((const float *)1)
void b200_submit_batch(network *net, const float *input);
int  b200_detect_submitted(network *net, const float *next_input, int w, int h, float thresh, float nms_thresh, int relative,
                           b200_det *out, int max_out, int *counts);

/* ---- classifiers (Darknet-19, Darknet-53: networks ending in [softmax]) ------------------------------------------------ */
/* network_predict + top_k for EVERY image on the device; the network must end in [softmax] (groups = 1), 1 <= top <= 64.
 * classes[b*top + j], probs[b*top + j]: the j-th entry of top_k over image b's probabilities.  input: host fp32 NCHW, or
 * B200_INPUT_RESIDENT (the device input buffer, e.g. after b200_letterbox_batch_u8).  Returns the number of images, -1 on a
 * network that does not end in [softmax] or a `top` out of range.  (b200_detect_batch / b200_detect_submitted return -1 on
 * such a network.) */
int  b200_classify_batch(network *net, const float *input, int top, int *classes, float *probs);
/* the double-buffered loop of b200_detect_submitted, same contract, for classifiers (after b200_submit_batch) */
int  b200_classify_submitted(network *net, const float *next_input, int top, int *classes, float *probs);
/* the device top-k on caller rows (rows x n, host), exposed for parity tests like b200_nms_sort_arrays */
void b200_top_k_arrays(const float *probs, int rows, int n, int top, int *classes);

/* ---- multi-GPU: image-sharded replicas, one process per GPU (SURVEY.md §8e) --------------------------------------------
 * Every process parses the same cfg; rank `root` alone loads the .weights file.  NCCL is resolved at run time (dlopen of
 * libnccl.so.2).  The 128-byte id made by b200_comm_unique_id on one rank reaches the others by any out-of-band channel
 * (bench.py: torch.distributed's store).  No collective ever runs between layers:
 *   b200_comm_broadcast_weights   one ncclBroadcast of the folded / repacked parameter arena (b200_weights_arena);
 *   b200_comm_set_gather          from then on records carry GLOBAL image numbers (image_base of the producing rank + its local
 *                                 index) and b200_detect_batch / b200_detect_submitted on `root` return the records of ALL
 *                                 ranks, in rank order — moved by ncclSend/ncclRecv on the result stream beside the next batch's
 *                                 forward pass; the other ranks keep getting their own.  slot_records = most records one rank
 *                                 may contribute per batch. */
int  b200_comm_unique_id(unsigned char *id, int bytes);           /* bytes >= 128; returns the id length */
int  b200_comm_init(network *net, const unsigned char *id, int rank, int world);
int  b200_comm_rank(network *net);
int  b200_comm_world(network *net);
int  b200_comm_broadcast_weights(network *net, int root);
int  b200_comm_set_gather(network *net, int root, int image_base, int slot_records);      /* root = -1: off */
void b200_comm_destroy(network *net);

/* device NMS on caller-provided host boxes (the kernel behind do_nms_sort); exposed for parity tests:
 * boxes[n*4] (x,y,w,h), probs[n*classes] row-major, modified in place exactly like box.c:58-89 zeroes prob[k]. */
void b200_nms_sort_arrays(const float *boxes, float *probs, int n, int classes, float thresh);
void b200_nms_obj_arrays(const float *boxes, float *objectness, int n, float thresh, unsigned char *suppressed);

#ifdef __cplusplus
}
#endif
#endif
