// kernels.h — launchers of the hand-written sm_100a kernels (internal C++ interface of dev/*.cu).
#pragma once
#include "common.cuh"

#define DT_BF16 0
#define DT_F32 1

// NHWC activation view: element (n,y,x,ch) lives at p[((n*h + y)*w + x)*ld + ch]; ld >= c lets a layer
// write straight into a channel slice of a concat buffer (route fusion).
struct TView {
    void *p;
    int n, h, w, c;
    int ld;
    int dtype;
};
static inline size_t dt_size(int dt) { return dt == DT_F32 ? 4 : 2; }

// ---- layout transforms (engine.cu I/O, tests) ----------------------------------------------------
void launch_nchw_f32_to_view(const float *src, TView dst, cudaStream_t s);   // host layout -> device layout
void launch_view_to_nchw_f32(TView src, float *dst, cudaStream_t s);         // device layout -> host layout

// ---- bandwidth-bound layers (layers.cu) ------------------------------------------------------------
void launch_maxpool(TView in, TView out, int size, int stride, int pad, cudaStream_t s);
void launch_upsample(TView in, TView out, int stride, float scale, cudaStream_t s);
void launch_shortcut(TView in, TView add, TView out, float alpha, float beta, int act, cudaStream_t s);
void launch_copy_channels(TView in, TView out, cudaStream_t s);               // out view already offset to its slice
void launch_reorg(TView in, TView out, int stride, cudaStream_t s, const int *table_dev = nullptr);   // table_dev: reorg_build_table's pairs on the device (optional)
void reorg_build_table(int h, int w, int c, int oh, int ow, int oc, int ldo, int s, int *table_xy);   // host: 2 ints per output element

// ---- convolution family ------------------------------------------------------------------------------
struct ConvParams {
    int size, stride, pad, act;
    const void *w;          // repacked weights [Cout_pad][size*size*Cin] (K order ky,kx,c), same dtype as activations
    const float *scale;     // per-output-channel multiplier (folded batch-norm), fp32
    const float *shift;     // per-output-channel addend (folded batch-norm / bias), fp32
    int cout_pad;           // rows in w (multiple of 16 for the tcgen05 path)
};
// first-layer kernel: reads the fp32 NCHW network input directly (fuses the layout/precision conversion)
void launch_conv_stem(const float *in_nchw, int n, int h, int w, int c, TView out, ConvParams p, cudaStream_t s, const TView *pool_out = nullptr);
// device-side letterbox_image + resize_image (+ uint8 HWC -> fp32 CHW): image.c:960-979, 1347-1390, 1442-1464
struct LetterboxItem {
    size_t src_off;              // byte offset of the image in the raw buffer
    int sw, sh;                  // source size
    int nw, nh, ox, oy;          // resized size and its position inside the network input
    float w_scale, h_scale;      // (sw-1)/(nw-1), (sh-1)/(nh-1) as the reference computes them (float division)
};
void launch_letterbox(const unsigned char *raw, int src_is_u8_hwc, const LetterboxItem *items_dev, int n, float *dst_nchw, int w, int h, cudaStream_t s);
bool launch_conv_stem_tc(const float *in_nchw, int n, int h, int w, int c, TView out, ConvParams p, cudaStream_t s,
                         const TView *pool_out = nullptr);   // false: shape not covered; pool_out: fused [maxpool] 2/2 output
bool conv_stem_tc_pool_supported(int h, int w, int c, TView out, ConvParams p);
void conv_stem_invalidate_bank();      // call after the stem's weights changed in place (load_weights)
// CUDA-core implicit-GEMM (fp32 accumulate); the fp32-exact path and the fallback for odd shapes
void launch_conv_simt(TView in, TView out, ConvParams p, cudaStream_t s);
// tcgen05/TMEM/TMA implicit-GEMM (bf16 in, fp32 accumulate).  Plans live in conv_tc.cu.
struct ConvTcPlan;
// nullptr if unsupported.  up_out: the convolution's result is written 2x nearest-upsampled into this view instead of `out`
ConvTcPlan *conv_tc_plan_create(TView in, TView out, ConvParams p, const TView *residual, float res_alpha, float res_beta,
                                const TView *up_out = nullptr, int local = 0);
// local = 1: unshared ("local") convolution: p.w = [location][filters][K], p.shift = bias [location][filters], p.scale = ones[filters]
void conv_tc_plan_destroy(ConvTcPlan *plan);
ConvTcPlan *conv_tc_block_plan_create(TView x, TView out, ConvParams p1, ConvParams p2, float res_alpha, float res_beta);   // fused residual block
bool conv_tc_shape_supported(int cin, int stride, int act);
void launch_conv_tc(ConvTcPlan *plan, cudaStream_t s);
const char *conv_tc_plan_desc(ConvTcPlan *plan);
// A FLOW: a run of tcgen05 convolution layers executed by ONE persistent CTA-pair kernel.  Tiles of layer n+1 start as soon as the
// tiles of layer n they read are stored (per-256-pixel completion counters in HBM) instead of at a kernel boundary, so the
// tensor pipe does not drain between layers.  members[k].dep / res_dep: index (inside the flow) of the layer producing member
// k's input / fused-shortcut operand, or -1 when that tensor is complete before the flow is launched.
struct ConvTcFlow;
struct ConvTcFlowMember { ConvTcPlan *plan; int dep, res_dep; };
bool conv_tc_plan_flow_ok(const ConvTcPlan *plan);
ConvTcFlow *conv_tc_flow_create(const ConvTcFlowMember *members, int n);      // nullptr: not worth it / does not fit
void conv_tc_flow_destroy(ConvTcFlow *flow);
void launch_conv_tc_flow(ConvTcFlow *flow, cudaStream_t s);
const char *conv_tc_flow_desc(ConvTcFlow *flow);
int conv_tc_flow_trace(ConvTcFlow *flow, unsigned long long *out, int max_items, int *item0, int max_layers);
void conv_tc_flow_read_stats(ConvTcFlow *flow, unsigned long long *out3);     // reads and clears (call with the stream idle)
// cuTensorMapEncodeTiled through the runtime's driver entry point (dtype 0 = bf16, 1 = fp32; swizzle_bytes 0/32/64/128)
void tc_encode_tiled(void *map, int dtype, int rank, void *base, const unsigned long long *dims, const unsigned long long *strides_bytes,
                     const unsigned *box, int swizzle_bytes);

// YOLOv1 dense layers (dense.cu)
void launch_local(TView in, TView out, const void *w, const float *bias, int size, int stride, int pad, int act, cudaStream_t s);
void launch_unpad_rows_f32(const float *src, int ld, float *dst, int cols, int rows, cudaStream_t s);
void launch_connected(const void *in, int in_dtype, int batch, int inputs, int outputs, const void *w, int w_dtype,
                      const float *scale, const float *shift, int act, float *out, cudaStream_t s);

// ---- heads (heads.cu): NHWC logits -> darknet-layout fp32 l.output with the layer's activations ------
void launch_yolo_forward(TView in, float *out, int anchors, int classes, cudaStream_t s);
void launch_region_forward(TView in, float *out, int anchors, int classes, int coords, int softmax, cudaStream_t s);
// [region] with tree=: logistic on x, y, objectness and one softmax per sibling group of the WordTree (temperature 1)
void launch_region_tree_forward(TView in, float *out, int anchors, int classes, int coords, const int *gsize, const int *goff, int groups, cudaStream_t s);
// hierarchy_predictions (tree.c:37-51) over every box of one batch item, in place: class j <- product of the conditional
// probabilities on its path to the root.  tmp: anchors*classes*hw floats of scratch.
void launch_region_hierarchy(float *item_out, float *tmp, int hw, int anchors, int classes, int coords, const int *parent, cudaStream_t s);
void launch_detection_forward(const float *in, float *out, int batch, int outputs, int side, int classes, int softmax, cudaStream_t s);
// l.batch == 2: item 0 <- mean(item 0, horizontally flipped item 1), in place (yolo_layer.c:290-314, region_layer.c:368-390)
void launch_avg_flipped(float *head_out, int w, int h, int anchors, int entries, int outputs, cudaStream_t s);

// ---- classifier tail (classify.cu) ---------------------------------------------------------------------
// [avgpool]: in NHWC (any h, w, ld >= c), out (n, 1, 1, c) of either dtype: the mean over the pixels, fp32 sum
void launch_avgpool(TView in, TView out, cudaStream_t s);
// [softmax] over `groups` equal slices of in's c channels (in must be a 1 x 1 map); out fp32 [batch][c]
void launch_softmax(TView in, float *out, int batch, int groups, float temp, cudaStream_t s);
// top_k of utils.c on each of `rows` rows of n values (row pitch ld): classes[r*k + j] and (if not NULL) probs[r*k + j]
void launch_topk(const float *a, int rows, int n, int ld, int k, int *classes, float *probs, cudaStream_t s);

// ---- decode + NMS (decode.cu, nms.cu) --------------------------------------------------------------
struct HeadDesc {            // one per YOLO/REGION/DETECTION layer, device-resident copy lives in the engine
    int type;                // LAYER_TYPE value
    int w, h, n, classes, coords, outputs, side, sqrt_;
    const float *out;        // darknet-layout fp32 activations [batch][outputs]
    const float *raw;        // YOLO heads: the feeding convolution's raw fp32 NHWC logits (or NULL); lets the fused
    int raw_ld;              //   detection path decode without materialising l.output (logistic applied on the fly)
    float anchors[2 * 16];   // (w,h) pairs already selected through mask[]
    int box_base;            // first global box id of this head inside an image
    // REGION head with a WordTree (YOLO9000, `tree=`): device copies of tree.parent / child / group_size / group_offset, or NULL
    const int *tree_parent, *tree_child, *tree_gsize, *tree_goff;
    int tree_groups;
};
struct CandBuffers {
    float *box;        // [batch][cap][4]
    float *obj;        // [batch][cap]
    float *prob;       // [batch][cap][classes]
    int   *id;         // [batch][cap] global box id
    int   *count;      // [batch]
    unsigned *flags;   // [batch][ceil(cap/32)] keep bitmap (decode scratch)
    int   *offsets;    // [batch][ceil(cap/32)+1] exclusive prefix of the bitmap popcounts (decode scratch)
    int   *cls_count;  // [batch][classes] live detections with a non-zero score per class (NMS scheduling)
    int cap, classes;
};
// mode 0 = reference get_network_boxes semantics (yolo: obj>thresh only; region/detection: every box)
// mode 1 = compact: additionally drops boxes whose objectness is 0 (what do_nms_sort's partition discards)
// tree_thresh / map_dev: the `hier` and `map` arguments of get_network_boxes, used by REGION heads with a WordTree
// (region_layer.c:412-424): map_dev = 200 class indices on the device, or NULL
void launch_decode(const HeadDesc *heads_dev, int nheads, int first_image, int nimages, int netw, int neth,
                   int imw, int imh, float thresh, int relative, int mode, int use_raw, CandBuffers cb, cudaStream_t s, const int *im_dims = nullptr,
                   float tree_thresh = .5f, const int *map_dev = nullptr);
void launch_count_yolo(const HeadDesc *heads_dev, int nheads, int image, float thresh, int *count_dev, cudaStream_t s);

struct NmsScratch { unsigned *mask; size_t words_per_cta; int ctas; };
void launch_nms_sort(const float *box, float *prob, const float *obj, const int *count, int images, int cap,
                     int classes, float thresh, int max_count, NmsScratch *scratch, int *cls_count, cudaStream_t s);
void launch_nms_obj(const float *box, float *obj, float *prob, const int *count, int images, int cap, int classes,
                    float thresh, int max_count, NmsScratch *scratch, cudaStream_t s);
// gathers surviving (box,class) pairs into compact records; returns via counter
struct DetRecord { int image, cls, box_id; float prob, objectness, x, y, w, h; };
void launch_collect(const float *box, const float *prob, const float *obj, const int *id, const int *count, int images,
                    int cap, int classes, DetRecord *out, int max_out, int *out_count, cudaStream_t s, int image_base = 0);   // image_base: added to every record's image number (multi-GPU shards)
