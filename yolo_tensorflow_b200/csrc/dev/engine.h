// engine.h — the engine object shared by the translation units of the device side (engine.cu: planning, forward, boxes;
// comm.cu: NCCL weight broadcast and detection gather).  Internal; the public surface is include/b200_engine.h.
#pragma once
#include "kernels.h"
#include "b200_engine.h"
#include <vector>
#include <string>

struct B200Comm;               // comm.cu

struct DevLayer {
    LAYER_TYPE type{};
    TView out{};               // NHWC output view (n = planned batch capacity)
    bool owns_out = false;
    float *head_out = nullptr; // YOLO / REGION / DETECTION / CONNECTED: fp32 [batch][outputs]
    float *fc_tmp = nullptr;   // CONNECTED on tcgen05: fp32 [batch][cout_pad] (row-padded GEMM output, compacted into head_out)
    // parameters (inside the arena)
    void *w = nullptr;
    float *scale = nullptr, *shift = nullptr, *lbias = nullptr;
    size_t w_off = 0, scale_off = 0, shift_off = 0, lbias_off = 0, w_bytes = 0;
    int cout_pad = 0;
    ConvTcPlan *tc = nullptr;
    bool stem = false;
    int fused_into = -1;       // conv whose epilogue also performs shortcut layer `fused_into` (its own output is not materialised); -1: none
    bool fused_away = false;   // shortcut executed inside the previous conv's epilogue
    bool up_fused = false;     // conv that writes its result 2x upsampled straight into the following [upsample]'s buffer
    bool up_away = false;      // [upsample] performed by the previous conv's store warp
    bool pool_fused = false;   // stem conv whose store warp also performs the following [maxpool] 2/2 (its own output is not written)
    bool pool_away = false;    // [maxpool] performed inside the stem kernel
    bool block_head = false;   // 1x1 conv computed inside the following 3x3's kernel (fused residual block): launches nothing
    int *reorg_table = nullptr;   // [reorg]: the per-image permutation as (source, destination) offset pairs on the device
    bool cls_logits = false;   // conv feeding a classifier's [softmax] (directly or through [avgpool]): fp32, rows padded to 64 filters
    std::string kernel;
};

struct b200_engine {
    int precision = 0, act_dtype = 0;
    int n = 0, cap = 0;        // layers, batch capacity
    int device = -1;           // -1: no CUDA device when the network was parsed (layer table only, nothing computes)
    int conv_backend = 0, fusion = 0;
    int head_sync = 1;         // network_predict copies the heads' outputs to their host l.output, as the reference API expects
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of the input batch, chunked so the first layer starts while later images are still in flight
    cudaEvent_t copy_done[8] = {};
    std::vector<DevLayer> L;
    float *d_input = nullptr;  // fp32 NCHW network input [cap][inputs]
    float *d_input_next = nullptr;   // spare input buffer: b200_submit_batch copies batch k+1 here while batch k computes
    cudaEvent_t submit_done = nullptr;
    int submitted = 0;
    cudaStream_t d2h_stream = nullptr;   // serving loop: results of batch k are read back here while batch k+1 already computes
    cudaEvent_t tail_done = nullptr;     // decode + NMS + collect of the current batch finished (d2h_stream waits on it)
    cudaStream_t tail_stream = nullptr;  // serving loop: decode + NMS + collect of batch k run here, beside the first layers of batch k+1
    cudaEvent_t fwd_done = nullptr;      // the forward pass of the current batch is complete (tail_stream waits on it)
    // flows (conv_tc_flow.cu): runs of convolution layers executed by one persistent kernel; flow_at[i] = index of the flow
    // whose first member is layer i, or -1.  flow_on = 0 runs the members one launch per layer (b200_set_flow).
    struct FlowRun { int first, last; ConvTcFlow *flow; };
    std::vector<FlowRun> flows;
    std::vector<int> flow_at;
    int flow_on = 0;
    int tail_guard_layer = 0;  // first layer that overwrites something the tail reads (head logits / l.output): it waits for tail_done
    cudaEvent_t lb_uploaded = nullptr, lb_done = nullptr;   // b200_letterbox_batch*: raw images are on the device / the resize kernel has consumed them
    int fwd_enqueued = 0;      // the submitted batch's forward pass is already in the compute stream (b200_detect_submitted)
    TView in_view{};           // NHWC copy of the input (only when layer 0 is not a stem conv)
    unsigned char *arena = nullptr;   // parameters
    size_t arena_bytes = 0;
    float *xfer = nullptr;     // fp32 scratch for fetch/set (max layer size)
    size_t xfer_floats = 0;
    // decode / nms
    std::vector<HeadDesc> heads;
    HeadDesc *d_heads = nullptr;
    int boxes_per_image = 0, classes = 0;
    bool raw_decode_ok = false;   // every head is a [yolo] layer fed by an fp32-logit convolution: the fused path may skip yolo_forward
    CandBuffers cand{};        // device
    int cand_slots = 0;
    NmsScratch nms_scratch{};
    DetRecord *d_records = nullptr; int records_cap = 0; int *d_record_count = nullptr;   // d_record_count = first of 4 ints {records, image base, 0, 0}: the header comm.cu sends
    B200Comm *comm = nullptr;  // NCCL communicator of this process (comm.cu), or null
    std::vector<int *> tree_arrays; bool has_tree = false; int *d_map = nullptr;     // YOLO9000: device copies of the WordTree of [region] heads, the `map` argument
    std::vector<void *> pinned_host;   // head-layer l.output buffers page-locked for the life of this plan (faster D2H / H2D on the reference API path)
    unsigned char *d_raw = nullptr; size_t raw_cap = 0;              // b200_letterbox_batch*: source images on the device
    LetterboxItem *d_lb_items = nullptr; int *d_im_dims[2] = {};     // per-image resize geometry / original sizes (box correction):
    int dims_cur = 0, dims_pending = 0;                              // [dims_cur] belongs to the batch whose forward pass was enqueued last, the other slot to the next letterbox call
    // classifiers: the device top-k results of b200_classify_*, and the [softmax] the network ends in
    int cls_layer = -1;        // -1: not a classifier
    int *d_top_cls = nullptr; float *d_top_prob = nullptr;
    // host staging for one image's candidates
    float *h_box = nullptr, *h_obj = nullptr, *h_prob = nullptr; int *h_id = nullptr; int h_cap = 0;
};

// comm.cu — hooks used by the detection tail (engine.cu)
bool b200_comm_gathers(const b200_engine *e);                       // a gather root is set
// enqueue the gather of every rank's record header + records to the root on stream s (all ranks call it in the same order)
void b200_comm_enqueue_gather(b200_engine *e, cudaStream_t s);
// root, after the stream has been synchronised: copy every rank's records to `out` (global image numbers); returns the count
int  b200_comm_collect_gathered(b200_engine *e, b200_det *out, int max_out, int own_count, cudaStream_t s);
bool b200_comm_is_root(const b200_engine *e);
int  b200_comm_image_base(const b200_engine *e);                    // global number of this rank's image 0 while a gather is set, else 0
void b200_comm_release(b200_engine *e);
