// engine.cu — the device engine behind the darknet C API: planning, memory, weight repacking, the forward
// loop (forward_network, network.c:188-211, re-expressed as a stream of sm_100a kernels), layer inspection hooks,
// and the device side of get_network_boxes / do_nms_sort.
//
// Data layout in HBM (DESIGN.md §3):
//   * activations  NHWC, bf16 (default) or fp32 (B200_PREC_FP32); a TView carries (n,h,w,c,ld) so a producer can
//                  write into a channel slice of a consumer's concat buffer;
//   * head outputs darknet layout, fp32: per image [anchor][entry][h*w] (what drivers read through l.output);
//   * parameters   one contiguous arena: per conv [Cout_pad][ky][kx][Cin] in the activation dtype + fp32
//                  scale/shift (inference batch-norm folded to one multiply-add per output);
//   * candidates   SoA per image: box[cap][4], objectness[cap], prob[cap][classes], id[cap], count.
#include "engine.h"
#include <cmath>
#include <cstring>
#include <functional>

static void *dev_alloc(size_t bytes)
{
    void *p = nullptr;
    B200_CHECK(cudaMalloc(&p, bytes ? bytes : 16));
    return p;
}

static void require_device(int device)
{
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0) {
        fprintf(stderr, "b200-darknet: no CUDA device available (%s). This engine has no CPU fallback.\n",
                err == cudaSuccess ? "device count is 0" : cudaGetErrorString(err));
        abort();
    }
    B200_CHECK(cudaSetDevice(device < count ? device : 0));
}

static bool g_cuda_ready = false;
static bool cuda_usable()
{
    int count = 0;
    return cudaGetDeviceCount(&count) == cudaSuccess && count > 0;
}

extern "C" void cuda_set_device(int n)
{
    gpu_index = n;
    if (cuda_usable()) B200_CHECK(cudaSetDevice(n));
}

extern "C" unsigned long long b200_launch_count(void) { return g_b200_launches; }

static TView view_of(const DevLayer &d, int batch)
{
    TView v = d.out;
    v.n = batch;
    return v;
}

static int act_id(ACTIVATION a)
{
    switch (a) {
    case LEAKY: return ACT_LEAKY;
    case LINEAR: return ACT_LINEAR;
    case LOGISTIC: return ACT_LOGISTIC;
    case RELU: return ACT_RELU;
    default:
        fprintf(stderr, "b200-darknet: activation %d is outside the YOLO inference path\n", (int)a);
        abort();
    }
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ----------------------------------------------------------------------------------------------------
// planning
// ----------------------------------------------------------------------------------------------------
static std::vector<std::vector<int>> consumers_of(const network *net)
{
    std::vector<std::vector<int>> c(net->n);
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if (l.type == ROUTE) {
            for (int j = 0; j < l.n; ++j) c[l.input_layers[j]].push_back(i);
        } else {
            if (i > 0) c[i - 1].push_back(i);
            if (l.type == SHORTCUT) c[l.index].push_back(i);
        }
    }
    return c;
}

// does layer j enqueue a kernel of its own (fused-away layers, aliases and in-place concatenations do not)
static bool layer_launches(const b200_engine *e, const network *net, int j)
{
    const layer &l = net->layers[j];
    const DevLayer &d = e->L[j];
    switch (l.type) {
    case CONVOLUTIONAL: return !d.block_head;
    case SHORTCUT: return !d.fused_away;
    case UPSAMPLE: return !d.up_away;
    case MAXPOOL: return !d.pool_away;
    case ROUTE: return d.kernel == "route_copy";
    case DROPOUT: case COST: return false;
    default: return true;
    }
}

// the layers whose kernels write the buffer that consumers of layer j read (through aliases and fused producers)
static void writers_of(const b200_engine *e, const network *net, int j, std::vector<int> &out)
{
    const layer &l = net->layers[j];
    const DevLayer &d = e->L[j];
    switch (l.type) {
    case SHORTCUT: if (d.fused_away) { out.push_back(j - 1); return; } break;
    case UPSAMPLE: if (d.up_away) { out.push_back(j - 1); return; } break;
    case MAXPOOL: if (d.pool_away) { out.push_back(j - 1); return; } break;
    case DROPOUT: case COST: if (j > 0) { writers_of(e, net, j - 1, out); return; } break;
    case ROUTE:
        for (int k = 0; k < l.n; ++k) writers_of(e, net, l.input_layers[k], out);
        if (d.kernel == "route_copy") out.push_back(j);
        return;
    default: break;
    }
    out.push_back(j);
}

static bool is_detection_head(LAYER_TYPE t) { return t == YOLO || t == REGION || t == DETECTION; }

// the layer whose output network_predict returns: the last one that is not a [cost]
static int output_layer(const network *net)
{
    int last = net->n - 1;
    while (last > 0 && net->layers[last].type == COST) --last;
    return last;
}

// streams and events of the serving loop and the input buffer
static void create_device_resources(b200_engine *e, const network *net)
{
    require_device(net->gpu_index);
    B200_CHECK(cudaGetDevice(&e->device));
    B200_CHECK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    B200_CHECK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    for (auto &ev : e->copy_done) B200_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    e->d_input = (float *)dev_alloc((size_t)e->cap * net->inputs * sizeof(float));
    // d_input_next is allocated on the first b200_submit_batch
    B200_CHECK(cudaEventCreateWithFlags(&e->submit_done, cudaEventDisableTiming));
    B200_CHECK(cudaStreamCreateWithFlags(&e->d2h_stream, cudaStreamNonBlocking));
    B200_CHECK(cudaEventCreateWithFlags(&e->tail_done, cudaEventDisableTiming));
    B200_CHECK(cudaStreamCreateWithFlags(&e->tail_stream, cudaStreamNonBlocking));
    B200_CHECK(cudaEventCreateWithFlags(&e->fwd_done, cudaEventDisableTiming));
    B200_CHECK(cudaEventCreateWithFlags(&e->lb_uploaded, cudaEventDisableTiming));
    B200_CHECK(cudaEventCreateWithFlags(&e->lb_done, cudaEventDisableTiming));
}

// fused_into / fused_away, block_head, up_fused / up_away: the layers whose work rides in a neighbouring kernel
static void plan_fusions(b200_engine *e, const network *net, const std::vector<std::vector<int>> &cons)
{
    // shortcut fusion: conv -> shortcut pairs whose add can ride in the conv epilogue
    for (int i = 1; i + 1 < net->n; ++i) {
        const layer &c = net->layers[i], &sc = net->layers[i + 1];
        if (!e->fusion || e->precision != B200_PREC_BF16) break;
        if (c.type != CONVOLUTIONAL || sc.type != SHORTCUT) continue;
        if (cons[i].size() != 1 || cons[i][0] != i + 1 || sc.index == i) continue;
        if (sc.activation != LINEAR || sc.w != sc.out_w || sc.h != sc.out_h || sc.c != sc.out_c) continue;
        if (c.activation != LEAKY && c.activation != LINEAR) continue;
        if (c.size == 1 && (c.stride != 1 || c.pad != 0)) continue;
        if (!conv_tc_shape_supported(c.c, c.stride, act_id(c.activation)) || c.out_c % 16 != 0) continue;
        LAYER_TYPE src = net->layers[sc.index].type;
        if (is_detection_head(src) || src == CONNECTED) continue;
        e->L[i].fused_into = i + 1;
        e->L[i + 1].fused_away = true;
    }

    // fused residual blocks: 1x1 (64 -> 32) -> 3x3 (32 -> 64) -> shortcut from the block input, in ONE kernel
    for (int i = 1; i + 2 < net->n; ++i) {
        const layer &c1 = net->layers[i], &c2 = net->layers[i + 1], &sc = net->layers[i + 2];
        if (c1.type != CONVOLUTIONAL || c2.type != CONVOLUTIONAL || sc.type != SHORTCUT) continue;
        if (e->L[i + 1].fused_into != i + 2 || sc.index != i - 1 || e->L[i].fused_into >= 0) continue;
        if (cons[i].size() != 1 || cons[i][0] != i + 1) continue;
        if (c1.size != 1 || c1.c != 64 || c1.n != 32 || c2.size != 3 || c2.stride != 1 || c2.pad != 1 || c2.n != 64) continue;
        if ((c1.activation != LEAKY && c1.activation != LINEAR) || (c2.activation != LEAKY && c2.activation != LINEAR)) continue;
        if (net->layers[i - 1].out_c != 64) continue;
        e->L[i].block_head = true;
    }

    // conv -> [upsample] (stride 2, scale 1): the conv's store warp writes the four copies itself
    for (int i = 1; i + 1 < net->n && e->fusion && e->precision == B200_PREC_BF16 && !getenv("B200_NO_UPSAMPLE_FUSION"); ++i) {
        const layer &c = net->layers[i], &u = net->layers[i + 1];
        if (c.type != CONVOLUTIONAL || u.type != UPSAMPLE || u.stride != 2 || u.reverse || u.scale != 1.f) continue;
        if (cons[i].size() != 1 || cons[i][0] != i + 1 || e->L[i].fused_into >= 0 || e->L[i].block_head) continue;
        if (c.out_c % 64 != 0 || (c.activation != LEAKY && c.activation != LINEAR)) continue;
        if (!conv_tc_shape_supported(c.c, c.stride, act_id(c.activation))) continue;
        e->L[i].up_fused = true;
        e->L[i + 1].up_away = true;
    }
}

// zero-copy concatenation: a route's inputs are produced straight into channel slices of the route's buffer
// (route_layer.c:80-95 copies every input; here only inputs that cannot be placed are copied).  An input is placed
// when its producer writes through a TView (row pitch = the route's channel count) and nothing needs it dense.
// place_route[j] = the route layer j's output is placed in (or -1), place_off[j] = its first channel there.
static void plan_route_placement(const b200_engine *e, const network *net, const std::vector<std::vector<int>> &cons,
                                 std::vector<int> &place_route, std::vector<int> &place_off)
{
    const int esize = (int)dt_size(e->act_dtype);
    place_route.assign(net->n, -1);
    place_off.assign(net->n, 0);
    for (int r = 0; r < net->n && !getenv("B200_NO_ZERO_COPY_ROUTE"); ++r) {
        const layer &rl = net->layers[r];
        if (rl.type != ROUTE || rl.n < 2 || rl.out_c == 0) continue;
        const int align = 16 / esize;                                   // slice starts stay 16-byte aligned
        if (rl.out_c % align != 0) continue;
        int coff = 0;
        for (int j = 0; j < rl.n; ++j) {
            const int sidx = rl.input_layers[j];
            const layer &sl = net->layers[sidx];
            bool ok = place_route[sidx] < 0 && coff % align == 0 && sl.out_c % 16 == 0 &&
                      (sl.type == CONVOLUTIONAL || sl.type == UPSAMPLE || sl.type == SHORTCUT || sl.type == MAXPOOL || sl.type == REORG);
            if (sl.type == CONVOLUTIONAL && e->L[sidx].fused_into >= 0) ok = false;
            for (int c : cons[sidx]) {
                LAYER_TYPE ct = net->layers[c].type;
                if (ct == CONNECTED || is_detection_head(ct)) ok = false;     // these read dense buffers
            }
            if (ok) { place_route[sidx] = r; place_off[sidx] = coff; }
            coff += sl.out_c;
        }
    }
}

// the classifier tail (cls_layer, cls_logits), every layer's output view and the fp32 transfer scratch, and the first
// layer's input (stem, in_view)
static void plan_outputs(b200_engine *e, const network *net, const std::vector<std::vector<int>> &cons,
                         const std::vector<int> &place_route, const std::vector<int> &place_off)
{
    auto concat_slice = [&](int sidx, const layer &sl, int dtype) -> TView {
        const int r = place_route[sidx];
        DevLayer &rd = e->L[r];
        const layer &rl = net->layers[r];
        if (!rd.out.p) {
            rd.out = TView{dev_alloc((size_t)e->cap * rl.outputs * dt_size(dtype)), e->cap, rl.out_h, rl.out_w, rl.out_c, rl.out_c, dtype};
            rd.owns_out = true;
        }
        return TView{(unsigned char *)rd.out.p + (size_t)place_off[sidx] * dt_size(dtype), e->cap, sl.out_h, sl.out_w, sl.out_c, rl.out_c, dtype};
    };

    // classifier tail: the [softmax] the network ends in, and the convolution feeding it (directly or through [avgpool])
    auto only_consumer_is = [&](int j, LAYER_TYPE t) { return j + 1 < net->n && cons[j].size() == 1 && cons[j][0] == j + 1 && net->layers[j + 1].type == t; };
    if (net->layers[output_layer(net)].type == SOFTMAX) e->cls_layer = output_layer(net);
    for (int i = 0; i < net->n; ++i)
        e->L[i].cls_logits = net->layers[i].type == CONVOLUTIONAL &&
                             (only_consumer_is(i, SOFTMAX) || (only_consumer_is(i, AVGPOOL) && only_consumer_is(i + 1, SOFTMAX)));

    // does a [connected] read layer j's buffer, directly or through the aliases [dropout] and a one-input [route]?  It reads
    // dense rows (launch_connected, connected_tc), so such a convolution keeps its row pitch at its filter count
    std::function<bool(int)> read_by_connected = [&](int j) {
        for (int c : cons[j]) {
            const layer &cl = net->layers[c];
            if (cl.type == CONNECTED || ((cl.type == DROPOUT || (cl.type == ROUTE && cl.n == 1)) && read_by_connected(c))) return true;
        }
        return false;
    };

    // output views
    size_t max_floats = (size_t)e->cap * net->inputs;
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        DevLayer &d = e->L[i];
        d.type = l.type;
        size_t floats = (size_t)e->cap * l.outputs;
        if (floats > max_floats) max_floats = floats;
        int dtype = e->act_dtype;
        if (l.type == CONVOLUTIONAL && e->precision == B200_PREC_BF16 && i + 1 < net->n && cons[i].size() == 1 &&
            (net->layers[i + 1].type == YOLO || net->layers[i + 1].type == REGION))
            dtype = DT_F32;                        // head logits stay fp32: no quantisation before the decode
        if (d.cls_logits || (l.type == AVGPOOL && only_consumer_is(i, SOFTMAX)))
            dtype = DT_F32;                        // so do a classifier's logits, up to its [softmax]
        switch (l.type) {
        case CONVOLUTIONAL: {
            // row pitch padded to 16 filters (255 -> 256): keeps every pixel row 16-byte aligned for vector stores; a classifier's
            // logits to 64 (1000 -> 1024), whole 64-filter tiles of the tcgen05 GEMM like the connected layer's; dense when a
            // [connected] reads it (conv_tc_plan_create refuses a pitch below the padded filter count: conv_simt runs then)
            int ld = read_by_connected(i) ? l.out_c : (int)align_up(l.out_c, d.cls_logits ? 64 : 16);
            if (d.fused_into >= 0) {            // written straight into the shortcut's buffer, never materialised
                d.out = TView{nullptr, e->cap, l.out_h, l.out_w, l.out_c, ld, dtype};
                d.owns_out = false;
                break;
            }
            if (place_route[i] >= 0 && dtype == e->act_dtype) { d.out = concat_slice(i, l, dtype); d.owns_out = false; break; }
            d.out = TView{dev_alloc((size_t)e->cap * l.out_h * l.out_w * ld * dt_size(dtype)), e->cap, l.out_h, l.out_w, l.out_c, ld, dtype};
            d.owns_out = true;
            break;
        }
        case MAXPOOL: case UPSAMPLE: case SHORTCUT: case REORG: case LOCAL:
            if (place_route[i] >= 0 && l.type != LOCAL) { d.out = concat_slice(i, l, dtype); d.owns_out = false; break; }
            d.out = TView{dev_alloc(floats * dt_size(dtype)), e->cap, l.out_h, l.out_w, l.out_c, l.out_c, dtype};
            d.owns_out = true;
            break;
        case ROUTE:
            if (l.out_c == 0) { fprintf(stderr, "b200-darknet: route %d joins layers of different spatial size\n", i); abort(); }
            if (l.n == 1) { d.out = e->L[l.input_layers[0]].out; d.owns_out = false; }
            else if (d.out.p) { /* allocated when its first placed input was planned */ }
            else {
                int dt0 = e->L[l.input_layers[0]].out.dtype;
                d.out = TView{dev_alloc(floats * dt_size(dt0)), e->cap, l.out_h, l.out_w, l.out_c, l.out_c, dt0};
                d.owns_out = true;
            }
            break;
        case DROPOUT: case COST:                   // identities at inference (cost: network_predict clears net->truth)
            d.out = e->L[i - 1].out; d.owns_out = false;
            d.head_out = e->L[i - 1].head_out;
            break;
        case AVGPOOL:
            d.out = TView{dev_alloc((size_t)e->cap * l.out_c * dt_size(dtype)), e->cap, 1, 1, l.out_c, l.out_c, dtype};
            d.owns_out = true;
            break;
        case SOFTMAX:
            if (i == 0 || net->layers[i - 1].out_h != 1 || net->layers[i - 1].out_w != 1 || net->layers[i - 1].out_c != l.inputs) {
                fprintf(stderr, "b200-darknet: [softmax] (layer %d) needs a 1 x 1 map as its input, e.g. after [avgpool]; "
                                "layer %d outputs %d x %d x %d\n", i, i - 1, i ? net->layers[i - 1].out_w : 0,
                        i ? net->layers[i - 1].out_h : 0, i ? net->layers[i - 1].out_c : 0);
                abort();
            }
            // fall through: an fp32 [batch][outputs] head like the detection layers'
        case CONNECTED: case YOLO: case REGION: case DETECTION:
            d.head_out = (float *)dev_alloc(floats * sizeof(float));
            d.out = TView{d.head_out, e->cap, 1, 1, l.outputs, l.outputs, DT_F32};
            d.owns_out = false;
            break;
        default:
            fprintf(stderr, "b200-darknet: layer %d has a type outside the inference path\n", i);
            abort();
        }
    }
    e->xfer_floats = max_floats;
    e->xfer = (float *)dev_alloc(max_floats * sizeof(float));

    // first layer input
    const layer &l0 = net->layers[0];
    e->L[0].stem = (l0.type == CONVOLUTIONAL && l0.c <= 4);
    if (!e->L[0].stem) {
        if (!(net->h && net->w && net->c)) { fprintf(stderr, "b200-darknet: network input must be an image\n"); abort(); }
        e->in_view = TView{dev_alloc((size_t)e->cap * net->inputs * dt_size(e->act_dtype)), e->cap, net->h, net->w, net->c, net->c, e->act_dtype};
    }
}

// the parameter arena: every layer's weight / scale / shift / bias offsets, then the arena itself (zeroed)
static void plan_arena(b200_engine *e, const network *net)
{
    const int esize = (int)dt_size(e->act_dtype);
    size_t off = 0;
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        DevLayer &d = e->L[i];
        if (l.type == CONVOLUTIONAL) {
            d.cout_pad = (int)align_up(l.n, d.cls_logits ? 64 : 16);
            d.w_bytes = (size_t)d.cout_pad * l.size * l.size * l.c * esize;
            d.w_off = off; off = align_up(off + d.w_bytes, 256);
            d.scale_off = off; off = align_up(off + d.cout_pad * sizeof(float), 256);
            d.shift_off = off; off = align_up(off + d.cout_pad * sizeof(float), 256);
        } else if (l.type == LOCAL) {
            d.w_bytes = (size_t)l.nweights * esize;
            d.w_off = off; off = align_up(off + d.w_bytes, 256);
            d.lbias_off = off; off = align_up(off + (size_t)l.outputs * sizeof(float), 256);
            d.scale_off = off; off = align_up(off + (size_t)l.n * sizeof(float), 256);      // ones: the tcgen05 epilogue multiplies by it
        } else if (l.type == CONNECTED) {
            d.cout_pad = (int)align_up(l.outputs, 64);                  // zero rows pad the GEMM's N to whole 64-filter tiles
            d.w_bytes = (size_t)l.inputs * d.cout_pad * esize;
            d.w_off = off; off = align_up(off + d.w_bytes, 256);
            d.scale_off = off; off = align_up(off + (size_t)d.cout_pad * sizeof(float), 256);
            d.shift_off = off; off = align_up(off + (size_t)d.cout_pad * sizeof(float), 256);
        }
    }
    e->arena_bytes = off;
    e->arena = (unsigned char *)dev_alloc(off);
    B200_CHECK(cudaMemset(e->arena, 0, off ? off : 16));
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        DevLayer &d = e->L[i];
        if (l.type == CONVOLUTIONAL || l.type == LOCAL || l.type == CONNECTED) d.w = e->arena + d.w_off;
        if (l.type == CONVOLUTIONAL || l.type == CONNECTED) { d.scale = (float *)(e->arena + d.scale_off); d.shift = (float *)(e->arena + d.shift_off); }
        if (l.type == LOCAL) { d.lbias = (float *)(e->arena + d.lbias_off); d.scale = (float *)(e->arena + d.scale_off); }
    }
}

// every layer's kernel and tcgen05 plan; a fusion whose shapes the plan does not take is undone here
static void select_kernels(b200_engine *e, const network *net, const std::vector<std::vector<int>> &cons, const std::vector<int> &place_route)
{
    // what layer i reads: the previous layer's output, or for the first layer the converted image (run_layer's `in`)
    auto input_of = [&](int i) { return i > 0 ? e->L[i - 1].out : e->in_view; };
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        DevLayer &d = e->L[i];
        switch (l.type) {
        case CONVOLUTIONAL: {
            if (l.size == 1 && (l.stride != 1 || l.pad != 0)) {
                // reference quirk (convolutional_layer.c:468-469): 1x1 convs skip im2col and ignore stride/pad
                fprintf(stderr, "b200-darknet: 1x1 convolution with stride/pad is not supported (layer %d)\n", i);
                abort();
            }
            d.kernel = d.stem ? "conv_stem" : "conv_simt";
            if (!d.stem && e->precision == B200_PREC_BF16) {
                ConvParams p{l.size, l.stride, l.pad, act_id(l.activation), d.w, d.scale, d.shift, d.cout_pad};
                if (d.block_head) { d.kernel = "conv_tc(block)"; break; }          // computed by the next layer's kernel
                if (d.fused_into >= 0 && i > 0 && e->L[i - 1].block_head) {
                    const layer &c1 = net->layers[i - 1], &sc = net->layers[d.fused_into];
                    DevLayer &d1 = e->L[i - 1];
                    ConvParams p1{c1.size, c1.stride, c1.pad, act_id(c1.activation), d1.w, d1.scale, d1.shift, d1.cout_pad};
                    d.tc = conv_tc_block_plan_create(e->L[sc.index].out, e->L[d.fused_into].out, p1, p, sc.alpha, sc.beta);
                    if (d.tc) { d.kernel = "conv_tc+shortcut"; break; }
                    // shapes the block kernel does not take: the 1x1 runs on its own after all
                    d1.block_head = false;
                    d1.tc = conv_tc_plan_create(e->L[i - 2].out, d1.out, p1, nullptr, 1.f, 1.f);
                    d1.kernel = d1.tc ? "conv_tc" : "conv_simt";
                }
                if (d.fused_into >= 0) {
                    const layer &sc = net->layers[d.fused_into];
                    d.tc = conv_tc_plan_create(input_of(i), e->L[d.fused_into].out, p, &e->L[sc.index].out, sc.alpha, sc.beta);
                    if (!d.tc) { fprintf(stderr, "b200-darknet: internal error: fused conv %d has no tcgen05 plan\n", i); abort(); }
                    d.kernel = "conv_tc+shortcut";
                } else {
                    if (d.up_fused) {
                        d.tc = conv_tc_plan_create(input_of(i), d.out, p, nullptr, 1.f, 1.f, &e->L[i + 1].out);
                        if (d.tc) { d.kernel = "conv_tc+upsample"; break; }
                        d.up_fused = false; e->L[i + 1].up_away = false;           // shape not covered: the two layers run separately
                    }
                    d.tc = conv_tc_plan_create(input_of(i), d.out, p, nullptr, 1.f, 1.f);
                    if (d.tc) d.kernel = "conv_tc";
                }
            }
            break;
        }
        case MAXPOOL: {
            d.kernel = "maxpool";
            // stem -> [maxpool] size 2 stride 2 (YOLOv2, YOLOv3-tiny): pooled by the stem kernel's store warp
            if (i == 1 && e->fusion && e->precision == B200_PREC_BF16 && e->L[0].stem && cons[0].size() == 1 &&
                l.size == 2 && l.stride == 2 && l.out_w * 2 == l.w && l.out_h * 2 == l.h && d.out.ld == d.out.c) {
                const layer &c0 = net->layers[0];
                ConvParams p0{c0.size, c0.stride, c0.pad, act_id(c0.activation), e->L[0].w, e->L[0].scale, e->L[0].shift, e->L[0].cout_pad};
                if (conv_stem_tc_pool_supported(c0.h, c0.w, c0.c, e->L[0].out, p0)) {
                    e->L[0].pool_fused = true; d.pool_away = true;
                    e->L[0].kernel = "conv_stem+maxpool"; d.kernel = "fused";
                }
            }
            break;
        }
        case UPSAMPLE: d.kernel = d.up_away ? "fused" : "upsample"; break;
        case SHORTCUT: d.kernel = d.fused_away ? "fused" : "shortcut"; break;
        case REORG: {
            d.kernel = "reorg";
            const DevLayer &pd = e->L[i - 1];
            if (!l.reverse && (size_t)l.h * l.w * l.c * dt_size(pd.out.dtype) <= 200 * 1024) {
                std::vector<int> table(2 * (size_t)l.out_h * l.out_w * l.out_c);
                reorg_build_table(l.h, l.w, l.c, l.out_h, l.out_w, l.out_c, d.out.ld, l.stride, table.data());
                d.reorg_table = (int *)dev_alloc(table.size() * sizeof(int));
                B200_CHECK(cudaMemcpy(d.reorg_table, table.data(), table.size() * sizeof(int), cudaMemcpyHostToDevice));
            }
            break;
        }
        case ROUTE: {
            bool all_placed = l.n > 1;
            for (int j = 0; j < l.n && l.n > 1; ++j) if (place_route[l.input_layers[j]] != i) all_placed = false;
            d.kernel = l.n == 1 ? "alias" : (all_placed ? "concat_in_place" : "route_copy");
            break;
        }
        case DROPOUT: d.kernel = "alias"; break;
        case LOCAL:
            d.kernel = "local";
            if (e->precision == B200_PREC_BF16) {
                // 49 independent GEMMs [images x 9C] x [9C x filters]: the conv kernel with one pixel per tile and the weight
                // box taken from that pixel's own slab
                ConvParams p{l.size, l.stride, l.pad, act_id(l.activation), d.w, d.scale, d.lbias, l.n};
                d.tc = conv_tc_plan_create(input_of(i), d.out, p, nullptr, 1.f, 1.f, nullptr, 1);
                if (d.tc) d.kernel = "local_tc";
            }
            break;
        case CONNECTED: {
            d.kernel = "connected";
            const DevLayer &pd = e->L[i - 1];
            if (e->precision == B200_PREC_BF16 && pd.out.dtype == DT_BF16 && pd.out.ld == pd.out.c && l.inputs % 64 == 0) {
                // out[b][o] = sum_i in[b][i] W[o][i] is a 1x1 convolution over a 1 x 1 "image" with `inputs` channels
                d.fc_tmp = (float *)dev_alloc((size_t)e->cap * d.cout_pad * sizeof(float));
                TView fin{pd.out.p, e->cap, 1, 1, l.inputs, l.inputs, DT_BF16};
                TView fout{d.fc_tmp, e->cap, 1, 1, l.outputs, d.cout_pad, DT_F32};
                ConvParams p{1, 1, 0, act_id(l.activation), d.w, d.scale, d.shift, d.cout_pad};
                d.tc = (l.activation == LEAKY || l.activation == LINEAR) ? conv_tc_plan_create(fin, fout, p, nullptr, 1.f, 1.f) : nullptr;
                if (d.tc) d.kernel = "connected_tc";
                else { cudaFree(d.fc_tmp); d.fc_tmp = nullptr; }
            }
            break;
        }
        case YOLO: d.kernel = "yolo_forward"; break;
        case AVGPOOL: d.kernel = "avgpool"; break;
        case SOFTMAX: d.kernel = "softmax"; break;
        case COST: d.kernel = "alias"; break;
        case REGION: d.kernel = "region_forward"; break;
        case DETECTION: d.kernel = "detection_forward"; break;
        default: break;
        }
    }
}

// flows: maximal runs of flow-capable convolutions (nothing else launching in between) become ONE persistent kernel
static void plan_flows(b200_engine *e, const network *net)
{
    e->flow_at.assign(net->n, -1);
    e->flow_on = 1;
    for (int i = 1; i < net->n && e->precision == B200_PREC_BF16;) {
        std::vector<ConvTcFlowMember> mem;
        std::vector<int> mem_layer;
        auto member_of = [&](int layer_idx) { for (size_t k = 0; k < mem_layer.size(); ++k) if (mem_layer[k] == layer_idx) return (int)k; return -1; };
        // producer inside the candidate run -> member index; all producers before the run -> -1; anything else -> -2
        auto resolve = [&](int src) {
            std::vector<int> w;
            writers_of(e, net, src, w);
            int inside = 0;
            for (int x : w) if (x >= i) ++inside;
            if (!inside) return -1;
            if (w.size() != 1) return -2;
            const int k = member_of(w[0]);
            return k >= 0 ? k : -2;
        };
        int j = i;
        bool restart_here = false;
        for (; j < net->n; ++j) {
            const layer &l = net->layers[j];
            DevLayer &d = e->L[j];
            if (!layer_launches(e, net, j)) continue;
            if (l.type != CONVOLUTIONAL || !d.tc || !conv_tc_plan_flow_ok(d.tc)) break;
            const int dep = resolve(j - 1);
            const int res_dep = d.fused_into >= 0 ? resolve(net->layers[d.fused_into].index) : -1;
            if (dep == -2 || res_dep == -2) { restart_here = !mem.empty(); break; }
            mem.push_back(ConvTcFlowMember{d.tc, dep, res_dep});
            mem_layer.push_back(j);
        }
        if (mem.size() >= 2) {
            ConvTcFlow *f = conv_tc_flow_create(mem.data(), (int)mem.size());
            if (f) {
                e->flow_at[mem_layer.front()] = (int)e->flows.size();
                e->flows.push_back(b200_engine::FlowRun{mem_layer.front(), mem_layer.back(), f});
            }
        }
        i = restart_here ? j : j + 1;
    }
}

// the decode's head descriptors (host and device copies), tail_guard_layer, and the page-locked host outputs
static void plan_heads(b200_engine *e, const network *net)
{
    int base = 0;
    e->raw_decode_ok = true;
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if (!is_detection_head(l.type)) continue;
        HeadDesc h;
        memset(&h, 0, sizeof h);
        h.type = l.type; h.w = l.w; h.h = l.h; h.n = l.n; h.classes = l.classes; h.coords = l.coords;
        h.outputs = l.outputs; h.side = l.side; h.sqrt_ = l.sqrt;
        h.out = e->L[i].head_out;
        if (l.type == YOLO && i > 0 && net->layers[i - 1].type == CONVOLUTIONAL && e->L[i - 1].out.dtype == DT_F32 && e->L[i - 1].out.p) {
            h.raw = (const float *)e->L[i - 1].out.p;
            h.raw_ld = e->L[i - 1].out.ld;
        } else e->raw_decode_ok = false;
        if (l.n > 16) { fprintf(stderr, "b200-darknet: more than 16 anchors per head\n"); abort(); }
        for (int a = 0; a < l.n && l.type != DETECTION; ++a) {
            int src = l.type == YOLO ? l.mask[a] : a;
            h.anchors[2 * a] = l.biases[2 * src];
            h.anchors[2 * a + 1] = l.biases[2 * src + 1];
        }
        if (l.type == REGION && l.softmax_tree) {
            const tree *t = l.softmax_tree;
            for (int j = 0; j < t->n; ++j) {                 // the device walk keeps a path in registers
                int depth = 0;
                for (int c = j; c >= 0; c = t->parent[c]) if (++depth > 64) { fprintf(stderr, "b200-darknet: class tree deeper than 64 levels\n"); abort(); }
            }
            auto put = [&](const int *src, int count) {
                int *d = (int *)dev_alloc((size_t)count * sizeof(int));
                B200_CHECK(cudaMemcpy(d, src, (size_t)count * sizeof(int), cudaMemcpyHostToDevice));
                e->tree_arrays.push_back(d);
                return (const int *)d;
            };
            h.tree_parent = put(t->parent, t->n); h.tree_child = put(t->child, t->n);
            h.tree_gsize = put(t->group_size, t->groups); h.tree_goff = put(t->group_offset, t->groups);
            h.tree_groups = t->groups;
            e->has_tree = true;
        }
        h.box_base = base;
        base += l.w * l.h * l.n;
        e->heads.push_back(h);
        if (e->classes && e->classes != l.classes) {
            // make_network_boxes sizes every prob[] from the LAST layer's classes (network.c:528-534) and each get_*_detections
            // writes its own l.classes of them: heads that disagree overrun the rows in the reference; rejected here
            fprintf(stderr, "b200-darknet: detection heads with different class counts (%d and %d) are not supported\n", e->classes, l.classes);
            abort();
        }
        e->classes = l.classes;                  // network.c:528 takes classes from the LAST layer
    }
    e->boxes_per_image = base;
    // the detection tail of batch k may still run (on its own stream) while batch k+1's forward pass starts: the first layer
    // that overwrites a buffer the tail reads — a head's l.output or the logits of the convolution feeding it — waits for it
    e->tail_guard_layer = net->n;
    for (int i = 0; i < net->n; ++i) {
        if (!is_detection_head(net->layers[i].type)) continue;
        int feeder = i > 0 ? i - 1 : 0;                      // the layer whose output the head (and the raw-logit decode) reads
        while (feeder > 0 && net->layers[feeder].type == DROPOUT) --feeder;
        if (feeder < e->tail_guard_layer) e->tail_guard_layer = feeder;
    }
    // the reference API moves the heads' l.output between host and device on every call (network.c:505, yolo_layer.c:359-362
    // on the way out; get_network_boxes reads them on the way in): page-lock those host buffers while this plan lives
    const int last = output_layer(net);
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if ((!is_detection_head(l.type) && i != last) || !l.output || l.type == DROPOUT) continue;
        if (cudaHostRegister(l.output, (size_t)e->cap * l.outputs * sizeof(float), cudaHostRegisterDefault) == cudaSuccess) e->pinned_host.push_back(l.output);
        else cudaGetLastError();                       // not fatal: the copies just stay pageable
    }
    if (!e->heads.empty()) {
        e->d_heads = (HeadDesc *)dev_alloc(e->heads.size() * sizeof(HeadDesc));
        B200_CHECK(cudaMemcpy(e->d_heads, e->heads.data(), e->heads.size() * sizeof(HeadDesc), cudaMemcpyHostToDevice));
    }
}

// the plan: each pass reads the decisions of the passes before it
static void build_engine_device_state(b200_engine *e, network *net)
{
    create_device_resources(e, net);
    const auto cons = consumers_of(net);
    plan_fusions(e, net, cons);
    std::vector<int> place_route, place_off;
    plan_route_placement(e, net, cons, place_route, place_off);
    plan_outputs(e, net, cons, place_route, place_off);
    plan_arena(e, net);
    select_kernels(e, net, cons, place_route);
    plan_flows(e, net);
    plan_heads(e, net);
    g_cuda_ready = true;
}

static b200_engine *engine_create(network *net, int precision, int fusion)
{
    b200_engine *e = new b200_engine();
    e->precision = precision;
    e->act_dtype = precision == B200_PREC_FP32 ? DT_F32 : DT_BF16;
    e->n = net->n;
    e->cap = net->batch;
    e->fusion = fusion;
    e->L.resize(net->n);
    // Parsing a cfg (layer table, shapes) works on a machine without a GPU; anything that computes does not.
    if (cuda_usable()) build_engine_device_state(e, net);
    return e;
}

extern "C" b200_engine *b200_engine_create(network *net, int precision)
{
    return engine_create(net, precision, b200_get_default_fusion());
}

static void need_device(const b200_engine *e, const char *what)
{
    if (e->device < 0) {
        fprintf(stderr, "b200-darknet: %s needs a CUDA device; none was available when the network was parsed. "
                        "There is no CPU fallback.\n", what);
        abort();
    }
    B200_CHECK(cudaSetDevice(e->device));
}

// host code calls this before it frees or re-allocates layer outputs (resize_network, free_network)
extern "C" void b200_engine_unpin_host(b200_engine *e)
{
    if (!e || e->device < 0) return;
    for (void *p : e->pinned_host) if (cudaHostUnregister(p) != cudaSuccess) cudaGetLastError();
    e->pinned_host.clear();
}

extern "C" void b200_engine_destroy(b200_engine *e)
{
    if (!e) return;
    if (e->device >= 0) {
        cudaSetDevice(e->device);
        cudaStreamSynchronize(e->stream);
        if (e->comm) b200_comm_release(e);
        b200_engine_unpin_host(e);
        for (auto &f : e->flows) conv_tc_flow_destroy(f.flow);
        for (auto &d : e->L) {
            if (d.tc) conv_tc_plan_destroy(d.tc);
            if (d.owns_out) cudaFree(d.out.p);
            cudaFree(d.fc_tmp); cudaFree(d.reorg_table);
            if (d.head_out && d.type != DROPOUT && d.type != COST) cudaFree(d.head_out);
        }
        cudaFree(e->d_input); cudaFree(e->d_input_next); cudaEventDestroy(e->submit_done); cudaFree(e->in_view.p); cudaFree(e->arena); cudaFree(e->xfer); cudaFree(e->d_heads);
        cudaFree(e->cand.box); cudaFree(e->cand.obj); cudaFree(e->cand.prob); cudaFree(e->cand.id); cudaFree(e->cand.count);
        cudaFree(e->cand.flags); cudaFree(e->cand.offsets); cudaFree(e->cand.cls_count);
        cudaFree(e->nms_scratch.mask); cudaFree(e->d_records); cudaFree(e->d_record_count);
        for (int *p : e->tree_arrays) cudaFree(p);
        cudaFree(e->d_map);
        cudaFree(e->d_top_cls); cudaFree(e->d_top_prob);
        cudaFree(e->d_raw); cudaFree(e->d_lb_items); cudaFree(e->d_im_dims[0]); cudaFree(e->d_im_dims[1]);
        cudaFreeHost(e->h_box); cudaFreeHost(e->h_obj); cudaFreeHost(e->h_prob); cudaFreeHost(e->h_id);
        for (auto &ev : e->copy_done) cudaEventDestroy(ev);
        cudaStreamDestroy(e->copy_stream); cudaStreamDestroy(e->d2h_stream); cudaStreamDestroy(e->tail_stream); cudaEventDestroy(e->fwd_done); cudaEventDestroy(e->tail_done); cudaEventDestroy(e->lb_uploaded); cudaEventDestroy(e->lb_done);
        cudaStreamDestroy(e->stream);
    }
    delete e;
}

// ----------------------------------------------------------------------------------------------------
// weights: fold the inference batch-norm, repack OIHW -> O(ky,kx,I), cast, upload
// ----------------------------------------------------------------------------------------------------
static void put_elem(unsigned char *dst, size_t idx, float v, int dtype)
{
    if (dtype == DT_F32) ((float *)dst)[idx] = v;
    else ((bf16 *)dst)[idx] = __float2bfloat16_rn(v);
}

static void fold_bn(const layer &l, int count, float *scale, float *shift)
{
    for (int f = 0; f < count; ++f) {
        if (l.batch_normalize) {
            // (x - mean)/(sqrt(var) + .000001f) * gamma + beta      (blas.c:154, batchnorm_layer.c:150-154)
            double s = (double)l.scales[f] / (sqrt((double)l.rolling_variance[f]) + (double).000001f);
            scale[f] = (float)s;
            shift[f] = (float)((double)l.biases[f] - (double)l.rolling_mean[f] * s);
        } else {
            scale[f] = 1.f;
            shift[f] = l.biases[f];
        }
    }
}

extern "C" void b200_engine_upload_weights(b200_engine *e, network *net)
{
    need_device(e, "load_weights");
    std::vector<unsigned char> host(e->arena_bytes, 0);
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        DevLayer &d = e->L[i];
        if (l.type == CONVOLUTIONAL) {
            const int K = l.size * l.size * l.c;
            unsigned char *w = host.data() + d.w_off;
            for (int o = 0; o < l.n; ++o)
                for (int c = 0; c < l.c; ++c)
                    for (int ky = 0; ky < l.size; ++ky)
                        for (int kx = 0; kx < l.size; ++kx) {
                            float v = l.weights[(((size_t)o * l.c + c) * l.size + ky) * l.size + kx];
                            put_elem(w, (size_t)o * K + (size_t)(ky * l.size + kx) * l.c + c, v, e->act_dtype);
                        }
            fold_bn(l, l.n, (float *)(host.data() + d.scale_off), (float *)(host.data() + d.shift_off));
        } else if (l.type == LOCAL) {
            const int locations = l.out_h * l.out_w, K = l.size * l.size * l.c;
            unsigned char *w = host.data() + d.w_off;
            for (int loc = 0; loc < locations; ++loc)
                for (int o = 0; o < l.n; ++o)
                    for (int c = 0; c < l.c; ++c)
                        for (int t = 0; t < l.size * l.size; ++t) {
                            float v = l.weights[((size_t)loc * l.n + o) * K + (size_t)c * l.size * l.size + t];
                            put_elem(w, ((size_t)loc * l.n + o) * K + (size_t)t * l.c + c, v, e->act_dtype);
                        }
            float *lb = (float *)(host.data() + d.lbias_off), *ones = (float *)(host.data() + d.scale_off);
            for (int o = 0; o < l.n; ++o) {                      // reference layout [o][loc] -> [loc][o]: one contiguous row per location
                ones[o] = 1.f;
                for (int loc = 0; loc < locations; ++loc) lb[(size_t)loc * l.n + o] = l.biases[(size_t)o * locations + loc];
            }
        } else if (l.type == CONNECTED) {
            // the producer's CHW flattening becomes HWC on the device: permute the weight columns accordingly
            const layer &prev = net->layers[i - 1];
            int pc = prev.out_c, ph = prev.out_h, pw = prev.out_w;
            bool image_in = pc > 0 && ph * pw > 1 && pc * ph * pw == l.inputs;
            unsigned char *w = host.data() + d.w_off;
            for (int o = 0; o < l.outputs; ++o)
                for (int k = 0; k < l.inputs; ++k) {
                    size_t dst = k;
                    if (image_in) { int c = k / (ph * pw), hw = k % (ph * pw); dst = (size_t)hw * pc + c; }
                    put_elem(w, (size_t)o * l.inputs + dst, l.weights[(size_t)o * l.inputs + k], e->act_dtype);
                }
            fold_bn(l, l.outputs, (float *)(host.data() + d.scale_off), (float *)(host.data() + d.shift_off));
        }
    }
    conv_stem_invalidate_bank();
    B200_CHECK(cudaMemcpyAsync(e->arena, host.data(), e->arena_bytes, cudaMemcpyHostToDevice, e->stream));
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

// resize_network: drop the plan built for the old geometry and build one for the layer table as it stands now, keeping
// the engine's settings; the parameters come from the host fp32 copies load_weights filled.
extern "C" b200_engine *b200_engine_recreate(b200_engine *old, network *net)
{
    const int precision = old->precision, fusion = old->fusion, head_sync = old->head_sync;
    B200Comm *comm = old->comm;                 // the communicator belongs to the process, not to the plan
    old->comm = nullptr;
    b200_engine_destroy(old);
    b200_engine *e = engine_create(net, precision, fusion);
    e->head_sync = head_sync;
    e->comm = comm;
    if (e->device >= 0) b200_engine_upload_weights(e, net);
    return e;
}

extern "C" void *b200_weights_arena(network *net, size_t *bytes)
{
    b200_engine *e = b200_engine_of(net);
    if (bytes) *bytes = e->arena_bytes;
    return e->arena;
}

// ----------------------------------------------------------------------------------------------------
// forward
// ----------------------------------------------------------------------------------------------------
static void run_layer(b200_engine *e, network *net, int i, int batch)
{
    const layer &l = net->layers[i];
    DevLayer &d = e->L[i];
    cudaStream_t s = e->stream;
    TView in = i > 0 ? view_of(e->L[i - 1], batch) : (d.stem ? TView{nullptr, 0, 0, 0, 0, 0, 0} : [&] { TView v = e->in_view; v.n = batch; return v; }());
    TView out = view_of(d, batch);
    switch (l.type) {
    case CONVOLUTIONAL: {
        ConvParams p{l.size, l.stride, l.pad, act_id(l.activation), d.w, d.scale, d.shift, d.cout_pad};
        if (d.block_head) break;                                   // computed inside the next layer's fused block kernel
        if (d.stem) {
            TView pool = d.pool_fused ? view_of(e->L[1], batch) : TView{nullptr, 0, 0, 0, 0, 0, 0};
            launch_conv_stem(e->d_input, batch, l.h, l.w, l.c, out, p, s, d.pool_fused && e->conv_backend == 0 ? &pool : nullptr);
        }
        else if (d.tc && e->conv_backend == 0) launch_conv_tc(d.tc, s);
        else launch_conv_simt(in, out, p, s);
        break;
    }
    case MAXPOOL:
        if (!d.pool_away || e->conv_backend != 0) launch_maxpool(in, out, l.size, l.stride, l.pad, s);
        break;
    case UPSAMPLE:
        if (!d.up_away || e->conv_backend != 0) launch_upsample(in, out, l.stride, l.scale, s);
        break;
    case SHORTCUT:
        if (!d.fused_away || e->conv_backend != 0) launch_shortcut(in, view_of(e->L[l.index], batch), out, l.alpha, l.beta, act_id(l.activation), s);
        break;
    case REORG:
        if (l.reverse) { fprintf(stderr, "b200-darknet: reorg reverse=1 is outside the YOLO inference path\n"); abort(); }
        launch_reorg(in, out, l.stride, s, d.reorg_table);
        break;
    case ROUTE:
        if (l.n > 1) {
            int coff = 0;
            for (int j = 0; j < l.n; ++j) {
                TView src = view_of(e->L[l.input_layers[j]], batch);
                TView dst = out;
                dst.p = (unsigned char *)out.p + (size_t)coff * dt_size(out.dtype);
                dst.c = src.c;
                if (src.p != dst.p) launch_copy_channels(src, dst, s);      // placed inputs were produced in this slice
                coff += src.c;
            }
        }
        break;
    case DROPOUT: case COST: break;
    case AVGPOOL: launch_avgpool(in, out, s); break;
    case SOFTMAX: launch_softmax(in, d.head_out, batch, l.groups, l.temperature, s); break;
    case LOCAL:
        if (d.tc && e->conv_backend == 0) launch_conv_tc(d.tc, s);
        else launch_local(in, out, d.w, d.lbias, l.size, l.stride, l.pad, act_id(l.activation), s);
        break;
    case CONNECTED: {
        const DevLayer &pd = e->L[i - 1];
        if (pd.out.ld != pd.out.c) { fprintf(stderr, "b200-darknet: connected input must be dense\n"); abort(); }
        if (d.tc && e->conv_backend == 0) {
            launch_conv_tc(d.tc, s);
            launch_unpad_rows_f32(d.fc_tmp, d.cout_pad, d.head_out, l.outputs, batch, s);
            break;
        }
        launch_connected(pd.out.p, pd.out.dtype, batch, l.inputs, l.outputs, d.w, e->act_dtype, d.scale, d.shift,
                         act_id(l.activation), d.head_out, s);
        break;
    }
    case YOLO: launch_yolo_forward(in, d.head_out, l.n, l.classes, s); break;
    case REGION:
        if (l.softmax_tree) {
            for (const HeadDesc &h : e->heads)
                if (h.out == d.head_out) launch_region_tree_forward(in, d.head_out, l.n, l.classes, l.coords, h.tree_gsize, h.tree_goff, h.tree_groups, s);
        } else launch_region_forward(in, d.head_out, l.n, l.classes, l.coords, l.softmax, s);
        break;
    case DETECTION: launch_detection_forward(e->L[i - 1].head_out, d.head_out, batch, l.outputs, l.side, l.classes, l.softmax, s); break;
    default: break;
    }
}

// runs layer i — or, when i opens a flow that ends before `end`, the whole flow in one launch; returns the last layer done
static int run_layer_or_flow(b200_engine *e, network *net, int i, int end, int batch)
{
    const int fi = e->flow_at[i];
    if (fi >= 0 && e->flow_on && e->conv_backend == 0 && e->flows[fi].last < end) {
        const b200_engine::FlowRun &f = e->flows[fi];
        if (e->tail_guard_layer > i && e->tail_guard_layer <= f.last) B200_CHECK(cudaStreamWaitEvent(e->stream, e->tail_done, 0));
        launch_conv_tc_flow(f.flow, e->stream);
        return f.last;
    }
    run_layer(e, net, i, batch);
    return i;
}

static int logical_batch(const b200_engine *e, const network *net)
{
    if (net->batch > e->cap) {
        fprintf(stderr, "b200-darknet: batch %d exceeds the cfg batch %d the buffers were planned for\n", net->batch, e->cap);
        abort();
    }
    return net->batch;
}

static void forward_layers(b200_engine *e, network *net, int start, int end, bool skip_yolo_forward = false)
{
    int batch = logical_batch(e, net);
    if (start == 0 && !e->L[0].stem) {
        TView v = e->in_view; v.n = batch;
        launch_nchw_f32_to_view(e->d_input, v, e->stream);
    }
    for (int i = start; i < end; ++i) {
        if (skip_yolo_forward && net->layers[i].type == YOLO) continue;   // the fused detection path decodes from the raw logits
        if (i == e->tail_guard_layer) B200_CHECK(cudaStreamWaitEvent(e->stream, e->tail_done, 0));   // no-op unless a tail is in flight
        i = run_layer_or_flow(e, net, i, end, batch);
    }
}

// H2D of a host batch.  When the first layer is the stem convolution (it reads the fp32 NCHW input directly and has no
// cross-image dependency) the copy is issued in chunks on a second stream and the stem runs chunk by chunk behind it, so
// its time hides under the PCIe transfer.  Returns the index of the first layer that still has to run.
static int stage_input(b200_engine *e, network *net, const float *input)
{
    const int batch = logical_batch(e, net);
    const layer &l0 = net->layers[0];
    DevLayer &d0 = e->L[0];
    int chunks = 1;
    if (d0.stem && !getenv("B200_NO_COPY_OVERLAP")) {
        if (batch % 8 == 0 && batch >= 16) chunks = 8;
        else if (batch % 4 == 0 && batch >= 8) chunks = 4;
        else if (batch % 2 == 0 && batch >= 4) chunks = 2;
    }
    if (chunks == 1) {
        B200_CHECK(cudaMemcpyAsync(e->d_input, input, (size_t)batch * net->inputs * sizeof(float), cudaMemcpyHostToDevice, e->stream));
        return 0;
    }
    const int per = batch / chunks;
    const size_t in_stride = (size_t)per * net->inputs;
    B200_CHECK(cudaStreamWaitEvent(e->copy_stream, e->lb_done, 0));      // a letterbox kernel may still be writing the input buffer
    for (int k = 0; k < chunks; ++k) {
        B200_CHECK(cudaMemcpyAsync(e->d_input + k * in_stride, input + k * in_stride, in_stride * sizeof(float), cudaMemcpyHostToDevice, e->copy_stream));
        B200_CHECK(cudaEventRecord(e->copy_done[k], e->copy_stream));
    }
    ConvParams p{l0.size, l0.stride, l0.pad, act_id(l0.activation), d0.w, d0.scale, d0.shift, d0.cout_pad};
    const size_t out_stride = (size_t)per * l0.out_h * l0.out_w * d0.out.ld * dt_size(d0.out.dtype);
    for (int k = 0; k < chunks; ++k) {
        B200_CHECK(cudaStreamWaitEvent(e->stream, e->copy_done[k], 0));
        TView out = d0.out;
        out.n = per;
        out.p = (unsigned char *)d0.out.p + k * out_stride;
        TView pool = e->L[d0.pool_fused ? 1 : 0].out;
        pool.n = per;
        pool.p = (unsigned char *)pool.p + (size_t)k * per * pool.h * pool.w * pool.ld * dt_size(pool.dtype);
        launch_conv_stem(e->d_input + k * in_stride, per, l0.h, l0.w, l0.c, out, p, e->stream, d0.pool_fused ? &pool : nullptr);
    }
    return 1;
}

// enqueue the copy of layer i's output (the first `batch` images, fp32 NCHW) to host memory at dst on the compute stream
static void copy_layer_to_host(b200_engine *e, const network *net, int i, int batch, float *dst)
{
    const size_t bytes = (size_t)batch * net->layers[i].outputs * sizeof(float);
    if (e->L[i].head_out) {
        B200_CHECK(cudaMemcpyAsync(dst, e->L[i].head_out, bytes, cudaMemcpyDeviceToHost, e->stream));
    } else {
        launch_view_to_nchw_f32(view_of(e->L[i], batch), e->xfer, e->stream);
        B200_CHECK(cudaMemcpyAsync(dst, e->xfer, bytes, cudaMemcpyDeviceToHost, e->stream));
    }
}

static void sync_heads_to_host(b200_engine *e, network *net)
{
    const int batch = logical_batch(e, net);
    const int last = output_layer(net);
    for (int i = 0; i < net->n; ++i)
        if (is_detection_head(net->layers[i].type) || i == last) copy_layer_to_host(e, net, i, batch, net->layers[i].output);
}

extern "C" void b200_engine_forward(b200_engine *e, network *net, const float *input)
{
    need_device(e, "network_predict");
    int first = stage_input(e, net, input);
    forward_layers(e, net, first, net->n);
    if (e->head_sync) sync_heads_to_host(e, net);
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

extern "C" void b200_engine_forward_resident(b200_engine *e, network *net)
{
    need_device(e, "network_predict");
    forward_layers(e, net, 0, net->n);
}

// with head sync off nobody reads l.output of the heads: the batched detection path skips forward_yolo_layer and decodes from
// the head convolutions' fp32 logits (identical arithmetic: the logistic is evaluated on the fly for the objectness test and for
// survivors).  Never for a classifier, which has no heads.
static bool use_raw_decode(const b200_engine *e) { return !e->head_sync && e->raw_decode_ok && !e->heads.empty(); }

// the sizes recorded by the last b200_letterbox_batch* call belong to the batch whose forward pass is enqueued next
static void adopt_letterbox_dims(b200_engine *e)
{
    if (e->dims_pending) { e->dims_cur ^= 1; e->dims_pending = 0; }
}

// enqueue the current batch's forward pass from layer `first`: 0, 1 after the chunked stage_input, or net->n when it is
// already in the stream
static void enqueue_forward(b200_engine *e, network *net, int first)
{
    if (first >= net->n) return;
    adopt_letterbox_dims(e);
    forward_layers(e, net, first, net->n, use_raw_decode(e));
}

// `input` of the batch entry points: NULL or B200_INPUT_RESIDENT is the device input buffer as it stands, anything else a
// host batch to stage.  Returns the first layer still to run.
static int stage_batch_input(b200_engine *e, network *net, const float *input)
{
    return (input && input != B200_INPUT_RESIDENT) ? stage_input(e, net, input) : 0;
}

extern "C" float *b200_engine_input_device(b200_engine *e) { return e->d_input; }
extern "C" void b200_engine_sync(b200_engine *e) { need_device(e, "sync"); B200_CHECK(cudaStreamSynchronize(e->stream)); }

extern "C" int b200_get_precision(const network *net) { return b200_engine_of(net)->precision; }
extern "C" void b200_set_conv_backend(network *net, int backend)
{
    b200_engine *e = b200_engine_of(net);
    for (auto &d : e->L)
        if (backend != 0 && (d.fused_into >= 0 || d.block_head || d.up_fused || d.pool_fused)) {
            fprintf(stderr, "b200-darknet: the CUDA-core conv backend needs an unfused plan (parse with B200_FUSE=0 B200_STEM_SIMT=1)\n");
            abort();
        }
    e->conv_backend = backend;
}
extern "C" void b200_set_head_sync(network *net, int on) { b200_engine_of(net)->head_sync = on; }
extern "C" void b200_set_flow(network *net, int on) { b200_engine_of(net)->flow_on = on; }
// profiling: nanoseconds the flow kernels' TMA producers / residual loaders spent blocked on a dependency and the number of
// blocking waits, summed over all launches since the last call (reads and clears the device counters of every flow)
extern "C" void b200_flow_stats(network *net, unsigned long long *out3)
{
    b200_engine *e = b200_engine_of(net);
    for (int i = 0; i < 5; ++i) out3[i] = 0;
    B200_CHECK(cudaStreamSynchronize(e->stream));
    for (auto &f : e->flows) {
        unsigned long long v[5];
        conv_tc_flow_read_stats(f.flow, v);
        for (int i = 0; i < 3; ++i) out3[i] += v[i];
        if (f.flow == e->flows[0].flow) { out3[3] = v[3]; out3[4] = v[4]; }
    }
}
extern "C" int b200_flow_trace(network *net, int k, unsigned long long *out, int max_items, int *item0, int max_layers)
{
    b200_engine *e = b200_engine_of(net);
    if (k < 0 || k >= (int)e->flows.size()) return 0;
    B200_CHECK(cudaStreamSynchronize(e->stream));
    return conv_tc_flow_trace(e->flows[k].flow, out, max_items, item0, max_layers);
}
extern "C" int b200_flow_count(network *net) { return (int)b200_engine_of(net)->flows.size(); }
extern "C" const char *b200_flow_desc(network *net, int k, int *first, int *last)
{
    b200_engine *e = b200_engine_of(net);
    if (k < 0 || k >= (int)e->flows.size()) return "";
    if (first) *first = e->flows[k].first;
    if (last) *last = e->flows[k].last;
    return conv_tc_flow_desc(e->flows[k].flow);
}

// ----------------------------------------------------------------------------------------------------
// inspection hooks
// ----------------------------------------------------------------------------------------------------
static void need_materialised(const b200_engine *e, int i)
{
    const DevLayer &d = e->L[i];
    const char *why = d.block_head   ? "it is computed inside the fused residual block kernel of the next layer"
                    : d.pool_fused   ? "the stem kernel stores it max-pooled into the next layer's buffer"
                    : d.up_fused     ? "it is written upsampled into the next layer's buffer"
                    : d.fused_into >= 0 ? "its shortcut is fused into the conv epilogue"
                    : nullptr;
    if (!why) return;
    fprintf(stderr, "b200-darknet: layer %d's output is not materialised: %s. "
                    "Parse with B200_FUSE=0 (or b200_set_default_fusion(0)) to inspect it.\n", i, why);
    abort();
}

extern "C" void b200_fetch_layer_output(network *net, int i, float *out)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_fetch_layer_output");
    need_materialised(e, i);
    copy_layer_to_host(e, net, i, logical_batch(e, net), out);
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

extern "C" void b200_set_layer_output(network *net, int i, const float *in)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_set_layer_output");
    need_materialised(e, i);
    int batch = logical_batch(e, net);
    size_t bytes = (size_t)batch * net->layers[i].outputs * sizeof(float);
    if (e->L[i].head_out) {
        B200_CHECK(cudaMemcpyAsync(e->L[i].head_out, in, bytes, cudaMemcpyHostToDevice, e->stream));
        const layer &l = net->layers[i];                  // the host copy get_network_boxes trusts follows (b200_engine_push_heads)
        if (is_detection_head(l.type) && l.output && l.output != in) memcpy(l.output, in, bytes);
    } else {
        B200_CHECK(cudaMemcpyAsync(e->xfer, in, bytes, cudaMemcpyHostToDevice, e->stream));
        launch_nchw_f32_to_view(e->xfer, view_of(e->L[i], batch), e->stream);
    }
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

extern "C" void b200_run_layers(network *net, int start, int end)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_run_layers");
    if (start < 0) start = 0;
    if (end > net->n) end = net->n;
    if (start == 0) {   // the caller placed the image in net->input (host) — stage it like network_predict does
        int batch = logical_batch(e, net);
        B200_CHECK(cudaMemcpyAsync(e->d_input, net->input, (size_t)batch * net->inputs * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    }
    forward_layers(e, net, start, end);
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

static void ensure_candidates(b200_engine *e, int slots);

// device time (ms) of the post-network tail: [0] decode+compaction, [1] class-wise NMS, [2] record collection
extern "C" void b200_profile_tail(network *net, int w, int h, float thresh, float nms_thresh, int iters, float *ms)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_profile_tail");
    int batch = logical_batch(e, net);
    ms[0] = ms[1] = ms[2] = 0.f;
    if (e->heads.empty()) return;
    ensure_candidates(e, e->cap);
    int max_out = 1 << 20;
    if (e->records_cap < max_out) { cudaFree(e->d_records); e->d_records = (DetRecord *)dev_alloc((size_t)max_out * sizeof(DetRecord)); e->records_cap = max_out; }
    if (!e->d_record_count) { e->d_record_count = (int *)dev_alloc(4 * sizeof(int)); B200_CHECK(cudaMemset(e->d_record_count, 0, 4 * sizeof(int))); }
    cudaEvent_t ev[4];
    for (auto &x : ev) B200_CHECK(cudaEventCreate(&x));
    for (int it = -1; it < iters; ++it) {                 // iteration -1 is an untimed warm-up (scratch allocation)
        B200_CHECK(cudaEventRecord(ev[0], e->stream));
        launch_decode(e->d_heads, (int)e->heads.size(), 0, batch, net->w, net->h, w, h, thresh, 1, 1, 0, e->cand, e->stream);
        B200_CHECK(cudaEventRecord(ev[1], e->stream));
        launch_nms_sort(e->cand.box, e->cand.prob, e->cand.obj, e->cand.count, batch, e->cand.cap, e->classes, nms_thresh,
                        e->boxes_per_image, &e->nms_scratch, e->cand.cls_count, e->stream);
        B200_CHECK(cudaEventRecord(ev[2], e->stream));
        B200_CHECK(cudaMemsetAsync(e->d_record_count, 0, sizeof(int), e->stream));
        launch_collect(e->cand.box, e->cand.prob, e->cand.obj, e->cand.id, e->cand.count, batch, e->cand.cap, e->classes,
                       e->d_records, max_out, e->d_record_count, e->stream);
        B200_CHECK(cudaEventRecord(ev[3], e->stream));
        B200_CHECK(cudaStreamSynchronize(e->stream));
        if (it < 0) continue;
        for (int k = 0; k < 3; ++k) { float t; B200_CHECK(cudaEventElapsedTime(&t, ev[k], ev[k + 1])); ms[k] += t / iters; }
    }
    for (auto &x : ev) cudaEventDestroy(x);
}

extern "C" const char *b200_layer_plan(network *net, int i)
{
    b200_engine *e = b200_engine_of(net);
    return e->L[i].tc ? conv_tc_plan_desc(e->L[i].tc) : "";
}

extern "C" void *b200_engine_stream(network *net) { return (void *)b200_engine_of(net)->stream; }

// per-layer device time (ms, averaged over `iters` forwards) measured with CUDA events on the engine stream;
// ms[net->n] receives the decode+NMS+collect tail when thresh >= 0.  Used by bench.py's roofline section.
extern "C" void b200_profile_layers(network *net, int iters, float *ms)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_profile_layers");
    int batch = logical_batch(e, net);
    std::vector<cudaEvent_t> ev(net->n + 1);
    for (auto &x : ev) B200_CHECK(cudaEventCreate(&x));
    for (int i = 0; i < net->n; ++i) ms[i] = 0.f;
    for (int it = 0; it < iters; ++it) {
        if (!e->L[0].stem) { TView v = e->in_view; v.n = batch; launch_nchw_f32_to_view(e->d_input, v, e->stream); }
        B200_CHECK(cudaEventRecord(ev[0], e->stream));
        for (int i = 0; i < net->n; ++i) {
            run_layer(e, net, i, batch);
            B200_CHECK(cudaEventRecord(ev[i + 1], e->stream));
        }
        B200_CHECK(cudaStreamSynchronize(e->stream));
        for (int i = 0; i < net->n; ++i) {
            float t = 0.f;
            B200_CHECK(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
            ms[i] += t / iters;
        }
    }
    for (auto &x : ev) cudaEventDestroy(x);
}

// device time of the forward pass as the serving loop runs it — `iters` passes enqueued back to back (no host
// synchronisation between them, programmatic dependent launch and all, the raw-logit decode plan when head sync is off):
// ms[0] = (last event - first event) / iters = one whole pass, ms[1] = the first layer alone, from one event pair around it
// inside every pass (the stem is not part of the tcgen05 convolution family whose roofline bench.py reports).
extern "C" void b200_profile_forward(network *net, int iters, float *ms)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_profile_forward");
    const int batch = logical_batch(e, net);
    const bool skip_yolo = use_raw_decode(e);
    if (iters < 1) iters = 1;
    std::vector<cudaEvent_t> ev(2 * (size_t)iters + 1);
    for (auto &x : ev) B200_CHECK(cudaEventCreate(&x));
    auto one_pass = [&](int it) {
        if (!e->L[0].stem) { TView v = e->in_view; v.n = batch; launch_nchw_f32_to_view(e->d_input, v, e->stream); }
        if (it >= 0) B200_CHECK(cudaEventRecord(ev[2 * it], e->stream));
        run_layer(e, net, 0, batch);
        if (it >= 0) B200_CHECK(cudaEventRecord(ev[2 * it + 1], e->stream));
        for (int i = 1; i < net->n; ++i) {
            if (skip_yolo && net->layers[i].type == YOLO) continue;
            i = run_layer_or_flow(e, net, i, net->n, batch);
        }
    };
    one_pass(-1);                                             // warm-up, then the timed passes without a gap
    for (int it = 0; it < iters; ++it) one_pass(it);
    B200_CHECK(cudaEventRecord(ev[2 * iters], e->stream));
    B200_CHECK(cudaStreamSynchronize(e->stream));
    float total = 0.f, first = 0.f;
    B200_CHECK(cudaEventElapsedTime(&total, ev[0], ev[2 * iters]));
    for (int it = 0; it < iters; ++it) { float t = 0.f; B200_CHECK(cudaEventElapsedTime(&t, ev[2 * it], ev[2 * it + 1])); first += t; }
    ms[0] = total / iters; ms[1] = first / iters;
    for (auto &x : ev) cudaEventDestroy(x);
}

extern "C" const char *b200_layer_kernel(network *net, int i)
{
    b200_engine *e = b200_engine_of(net);
    if (e->L[i].tc && e->conv_backend != 0) return "conv_simt";
    return e->L[i].kernel.c_str();
}

// ----------------------------------------------------------------------------------------------------
// boxes + NMS
// ----------------------------------------------------------------------------------------------------
static void ensure_candidates(b200_engine *e, int slots)
{
    if (e->cand_slots >= slots) return;
    cudaFree(e->cand.box); cudaFree(e->cand.obj); cudaFree(e->cand.prob); cudaFree(e->cand.id); cudaFree(e->cand.count);
    cudaFree(e->cand.flags); cudaFree(e->cand.offsets); cudaFree(e->cand.cls_count);
    int cap = e->boxes_per_image, cls = e->classes;
    e->cand.cap = cap; e->cand.classes = cls;
    e->cand.box = (float *)dev_alloc((size_t)slots * cap * 4 * sizeof(float));
    e->cand.obj = (float *)dev_alloc((size_t)slots * cap * sizeof(float));
    e->cand.prob = (float *)dev_alloc((size_t)slots * cap * cls * sizeof(float));
    e->cand.id = (int *)dev_alloc((size_t)slots * cap * sizeof(int));
    e->cand.count = (int *)dev_alloc((size_t)slots * sizeof(int));
    e->cand.flags = (unsigned *)dev_alloc((size_t)slots * ((cap + 31) / 32) * sizeof(unsigned));
    e->cand.offsets = (int *)dev_alloc((size_t)slots * ((cap + 31) / 32) * sizeof(int));
    e->cand.cls_count = (int *)dev_alloc(((size_t)slots * cls + 1) * sizeof(int));
    e->cand_slots = slots;
    if (e->h_cap < cap) {
        cudaFreeHost(e->h_box); cudaFreeHost(e->h_obj); cudaFreeHost(e->h_prob); cudaFreeHost(e->h_id);
        B200_CHECK(cudaMallocHost((void **)&e->h_box, (size_t)cap * 4 * sizeof(float)));
        B200_CHECK(cudaMallocHost((void **)&e->h_obj, (size_t)cap * sizeof(float)));
        B200_CHECK(cudaMallocHost((void **)&e->h_prob, (size_t)cap * cls * sizeof(float)));
        B200_CHECK(cudaMallocHost((void **)&e->h_id, (size_t)cap * sizeof(int)));
        e->h_cap = cap;
    }
}

// internal C ABI used by host/boxes.c ------------------------------------------------------------------------
extern "C" int b200_engine_count_boxes(b200_engine *e, network *net, int image, float thresh)
{
    need_device(e, "num_detections");
    if (e->heads.empty()) return 0;
    ensure_candidates(e, 1);
    launch_count_yolo(e->d_heads, (int)e->heads.size(), image, thresh, e->cand.count, e->stream);
    int n = 0;
    B200_CHECK(cudaMemcpyAsync(&n, e->cand.count, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    B200_CHECK(cudaStreamSynchronize(e->stream));
    return n;
}

// hierarchy_predictions over batch item `image` of every [region] head with a WordTree (region_layer.c:412-414), in place
// like the reference (device buffer and, with head sync, the host copy): call once per get_network_boxes
extern "C" void b200_engine_hierarchy(b200_engine *e, network *net, int image)
{
    need_device(e, "get_network_boxes");
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if (l.type != REGION || !l.softmax_tree) continue;
        for (const HeadDesc &h : e->heads) {
            if (h.out != e->L[i].head_out) continue;
            float *item = e->L[i].head_out + (size_t)image * l.outputs;
            launch_region_hierarchy(item, e->xfer, l.w * l.h, l.n, l.classes, l.coords, h.tree_parent, e->stream);
            if (e->head_sync && l.output)
                B200_CHECK(cudaMemcpyAsync(l.output + (size_t)image * l.outputs, item, (size_t)l.outputs * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        }
    }
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

extern "C" int b200_engine_has_tree(b200_engine *e) { return e->has_tree ? 1 : 0; }

extern "C" int b200_engine_decode_image(b200_engine *e, network *net, int image, int w, int h, float thresh, int relative,
                                        const float **box, const float **obj, const float **prob, const int **id, float hier, const int *map)
{
    need_device(e, "get_network_boxes");
    if (e->heads.empty()) return 0;
    ensure_candidates(e, 1);
    const int *d_map = nullptr;
    if (map && e->has_tree) {                          // the 200 class indices of coco9k.map / inet9k.map (detector.c:392, region_layer.c:415)
        if (!e->d_map) e->d_map = (int *)dev_alloc(200 * sizeof(int));
        B200_CHECK(cudaMemcpyAsync(e->d_map, map, 200 * sizeof(int), cudaMemcpyHostToDevice, e->stream));
        d_map = e->d_map;
    }
    launch_decode(e->d_heads, (int)e->heads.size(), image, 1, net->w, net->h, w, h, thresh, relative, 0, 0, e->cand, e->stream, nullptr, hier, d_map);
    int n = 0;
    B200_CHECK(cudaMemcpyAsync(&n, e->cand.count, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    B200_CHECK(cudaStreamSynchronize(e->stream));
    if (n > 0) {
        B200_CHECK(cudaMemcpyAsync(e->h_box, e->cand.box, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        B200_CHECK(cudaMemcpyAsync(e->h_obj, e->cand.obj, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        B200_CHECK(cudaMemcpyAsync(e->h_prob, e->cand.prob, (size_t)n * e->classes * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
        B200_CHECK(cudaMemcpyAsync(e->h_id, e->cand.id, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, e->stream));
        B200_CHECK(cudaStreamSynchronize(e->stream));
    }
    *box = e->h_box; *obj = e->h_obj; *prob = e->h_prob; *id = e->h_id;
    return n;
}

extern "C" int b200_engine_classes(b200_engine *e) { return e->classes; }

// get_network_boxes reads the heads' HOST l.output in the reference, and callers may have rewritten it since the last
// predict (demo.c:54-83 averages the last frames into it): with head sync on, the host buffers of the first `items` batch
// items are the truth and go back to the device before the decode.
extern "C" void b200_engine_push_heads(b200_engine *e, network *net, int items)
{
    need_device(e, "get_network_boxes");
    if (!e->head_sync) return;
    if (items > logical_batch(e, net)) items = logical_batch(e, net);
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if (!is_detection_head(l.type) || !e->L[i].head_out || !l.output) continue;
        B200_CHECK(cudaMemcpyAsync(e->L[i].head_out, l.output, (size_t)items * l.outputs * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    }
}

// `if (l.batch == 2) avg_flipped_yolo(l)` of get_yolo_detections (yolo_layer.c:320) and the same branch of
// get_region_detections (region_layer.c:368-390): in place, device and (with head sync) host copy alike.
extern "C" void b200_engine_avg_flipped(b200_engine *e, network *net)
{
    need_device(e, "get_network_boxes");
    for (int i = 0; i < net->n; ++i) {
        const layer &l = net->layers[i];
        if ((l.type != YOLO && l.type != REGION) || l.batch != 2 || e->cap < 2) continue;
        const int entries = l.type == YOLO ? l.classes + 4 + 1 : l.classes + l.coords + 1;
        launch_avg_flipped(e->L[i].head_out, l.w, l.h, l.n, entries, l.outputs, e->stream);
        if (e->head_sync && l.output)
            B200_CHECK(cudaMemcpyAsync(l.output, e->L[i].head_out, (size_t)2 * l.outputs * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    }
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

// forward (from layer `first`; first = net->n: the forward pass is already in the stream) + decode + NMS + collect, all
// enqueued on the compute stream; `after_tail` (optional) runs once they are enqueued and before the host waits, so that the
// caller can put the NEXT batch's work behind them; the results then come back on their own stream while that work runs.
template <typename F>
static int detect_core(b200_engine *e, network *net, int first, int w, int h, float thresh, float nms_thresh, int relative,
                       b200_det *out, int max_out, int *counts, F after_tail)
{
    int batch = logical_batch(e, net);
    if (e->has_tree) {
        fprintf(stderr, "b200-darknet: networks with a class tree (YOLO9000) go through get_network_boxes + do_nms_sort; the fused batched path does not take them\n");
        abort();
    }
    enqueue_forward(e, net, first);
    if (e->heads.empty()) { after_tail(); B200_CHECK(cudaStreamSynchronize(e->stream)); return 0; }
    ensure_candidates(e, e->cap);
    if (e->records_cap < max_out) {
        cudaFree(e->d_records);
        e->d_records = (DetRecord *)dev_alloc((size_t)max_out * sizeof(DetRecord));
        e->records_cap = max_out;
    }
    if (!e->d_record_count) { e->d_record_count = (int *)dev_alloc(4 * sizeof(int)); B200_CHECK(cudaMemset(e->d_record_count, 0, 4 * sizeof(int))); }
    // w == h == 0: every image is corrected with its own original size, recorded by b200_letterbox_batch*
    const int *im_dims = (w == 0 && h == 0) ? e->d_im_dims[e->dims_cur] : nullptr;
    if (w == 0 && h == 0 && !im_dims) { fprintf(stderr, "b200-darknet: w = h = 0 needs a preceding b200_letterbox_batch call\n"); abort(); }
    // decode + NMS + collect go to their own stream behind the forward pass: in the serving loop the next batch's forward pass
    // is enqueued right after (after_tail), and these small latency-bound kernels then run beside its first, bandwidth-bound
    // layers instead of in front of them
    cudaStream_t ts = e->tail_stream;
    B200_CHECK(cudaEventRecord(e->fwd_done, e->stream));
    B200_CHECK(cudaStreamWaitEvent(ts, e->fwd_done, 0));
    launch_decode(e->d_heads, (int)e->heads.size(), 0, batch, net->w, net->h, w, h, thresh, relative, 1, use_raw_decode(e) ? 1 : 0,
                  e->cand, ts, im_dims);
    launch_nms_sort(e->cand.box, e->cand.prob, e->cand.obj, e->cand.count, batch, e->cand.cap, e->classes, nms_thresh,
                    e->boxes_per_image, &e->nms_scratch, e->cand.cls_count, ts);
    B200_CHECK(cudaMemsetAsync(e->d_record_count, 0, sizeof(int), ts));
    launch_collect(e->cand.box, e->cand.prob, e->cand.obj, e->cand.id, e->cand.count, batch, e->cand.cap, e->classes,
                   e->d_records, max_out, e->d_record_count, ts, b200_comm_image_base(e));
    B200_CHECK(cudaEventRecord(e->tail_done, ts));
    B200_CHECK(cudaStreamWaitEvent(e->d2h_stream, e->tail_done, 0));
    // multi-GPU: every rank's records travel to the gather root over NCCL (send/recv on the result stream, so the transfer
    // runs beside the next batch's forward pass like the read-back does); the root then returns all of them.  Enqueued BEFORE
    // the next batch's kernels are submitted, so that the copy kernels are not queued behind a whole forward pass.
    const bool gather = b200_comm_gathers(e);
    if (gather) b200_comm_enqueue_gather(e, e->d2h_stream);
    after_tail();
    int n = 0;
    B200_CHECK(cudaMemcpyAsync(&n, e->d_record_count, sizeof(int), cudaMemcpyDeviceToHost, e->d2h_stream));
    if (counts) B200_CHECK(cudaMemcpyAsync(counts, e->cand.count, (size_t)batch * sizeof(int), cudaMemcpyDeviceToHost, e->d2h_stream));
    B200_CHECK(cudaStreamSynchronize(e->d2h_stream));
    if (n > max_out) n = max_out;
    static_assert(sizeof(DetRecord) == sizeof(b200_det), "record layouts must match");
    if (gather && b200_comm_is_root(e)) return b200_comm_collect_gathered(e, out, max_out, n, e->d2h_stream);
    if (n > 0) {
        B200_CHECK(cudaMemcpyAsync(out, e->d_records, (size_t)n * sizeof(DetRecord), cudaMemcpyDeviceToHost, e->d2h_stream));
        B200_CHECK(cudaStreamSynchronize(e->d2h_stream));
    }
    return n;
}

static int detect_core(b200_engine *e, network *net, int first, int w, int h, float thresh, float nms_thresh, int relative,
                       b200_det *out, int max_out, int *counts)
{
    int n = detect_core(e, net, first, w, h, thresh, nms_thresh, relative, out, max_out, counts, [] {});
    B200_CHECK(cudaStreamSynchronize(e->stream));       // synchronous callers expect the engine idle on return
    return n;
}

// a classifier (a network ending in [softmax]) has no detection head: the batched detection entry points refuse it
static bool refuse_classifier(const b200_engine *e, const char *what)
{
    if (e->cls_layer < 0) return false;
    fprintf(stderr, "b200-darknet: %s: the network ends in [softmax] and has no detection head; use b200_classify_batch\n", what);
    return true;
}

extern "C" int b200_detect_batch(network *net, const float *input, int w, int h, float thresh, float nms_thresh,
                                 int relative, b200_det *out, int max_out, int *counts)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_detect_batch");
    if (refuse_classifier(e, "b200_detect_batch")) return -1;
    const int first = stage_batch_input(e, net, input);
    return detect_core(e, net, first, w, h, thresh, nms_thresh, relative, out, max_out, counts);
}

// ----------------------------------------------------------------------------------------------------
// device-side preprocessing (SURVEY 8f-1): n decoded images of individual sizes -> the letterboxed fp32 NCHW network
// input, written straight into the engine's input buffer.  Follow with b200_detect_batch(net, NULL, 0, 0, ...): w = h = 0
// corrects every image's boxes with its own size (what test_detector does per image: get_network_boxes(net, im.w, im.h, ..)).
// ----------------------------------------------------------------------------------------------------
static int letterbox_batch(network *net, const void *const *images, const int *widths, const int *heights, int n, int u8)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_letterbox_batch");
    if (n < 1 || n > e->cap || net->c != 3) { fprintf(stderr, "b200-darknet: b200_letterbox_batch: 1..batch 3-channel images\n"); return -1; }
    const size_t esz = u8 ? 1 : sizeof(float);
    std::vector<LetterboxItem> items(n);
    std::vector<int> dims(2 * (size_t)e->cap);
    for (int i = 0; i < e->cap; ++i) { dims[2 * i] = net->w; dims[2 * i + 1] = net->h; }      // slots without an image: identity
    size_t total = 0;
    for (int i = 0; i < n; ++i) {
        const int sw = widths[i], sh = heights[i];
        if (sw < 1 || sh < 1 || !images[i]) return -1;
        LetterboxItem &it = items[i];
        it.src_off = total; it.sw = sw; it.sh = sh;
        if (((float)net->w / sw) < ((float)net->h / sh)) { it.nw = net->w; it.nh = (sh * net->w) / sw; }      // image.c:964-970
        else { it.nh = net->h; it.nw = (sw * net->h) / sh; }
        if (it.nw < 1) it.nw = 1;
        if (it.nh < 1) it.nh = 1;
        it.ox = (net->w - it.nw) / 2; it.oy = (net->h - it.nh) / 2;
        it.w_scale = (float)(sw - 1) / (it.nw - 1);                                                            // image.c:1352-1353
        it.h_scale = (float)(sh - 1) / (it.nh - 1);
        total += (((size_t)sw * sh * 3 * esz) + 255) / 256 * 256;
        dims[2 * i] = sw; dims[2 * i + 1] = sh;
    }
    if (total > e->raw_cap) {
        cudaFree(e->d_raw);
        e->d_raw = (unsigned char *)dev_alloc(total);
        e->raw_cap = total;
    }
    if (!e->d_lb_items) e->d_lb_items = (LetterboxItem *)dev_alloc((size_t)e->cap * sizeof(LetterboxItem));
    for (int k = 0; k < 2; ++k)
        if (!e->d_im_dims[k]) e->d_im_dims[k] = (int *)dev_alloc(2 * (size_t)e->cap * sizeof(int));
    // The uploads run on the copy stream, so that a serving loop can stage batch k+1 while batch k's forward pass still runs
    // (d_raw / d_lb_items were last read by the previous letterbox kernel, which has finished: this function waited for the
    // previous upload and the kernel was enqueued before the forward pass whose results the caller has meanwhile collected or
    // is about to; the dims slot written is the one of the batch before the one in flight).  Only the letterbox kernel itself
    // joins the compute stream, behind whatever is already there.
    cudaStream_t up = e->copy_stream;
    B200_CHECK(cudaStreamWaitEvent(up, e->lb_done, 0));                           // the previous letterbox kernel must be done with d_raw
    for (int i = 0; i < n; ++i)
        B200_CHECK(cudaMemcpyAsync(e->d_raw + items[i].src_off, images[i], (size_t)widths[i] * heights[i] * 3 * esz, cudaMemcpyHostToDevice, up));
    B200_CHECK(cudaMemcpyAsync(e->d_lb_items, items.data(), (size_t)n * sizeof(LetterboxItem), cudaMemcpyHostToDevice, up));
    B200_CHECK(cudaMemcpyAsync(e->d_im_dims[e->dims_cur ^ 1], dims.data(), dims.size() * sizeof(int), cudaMemcpyHostToDevice, up));
    B200_CHECK(cudaEventRecord(e->lb_uploaded, up));
    B200_CHECK(cudaStreamWaitEvent(e->stream, e->lb_uploaded, 0));
    launch_letterbox(e->d_raw, u8, e->d_lb_items, n, e->d_input, net->w, net->h, e->stream);
    B200_CHECK(cudaEventRecord(e->lb_done, e->stream));
    B200_CHECK(cudaStreamSynchronize(up));                  // items / dims live on this stack frame
    e->dims_pending = 1;
    return 0;
}

extern "C" int b200_letterbox_batch_u8(network *net, const unsigned char *const *images, const int *widths, const int *heights, int n)
{
    return letterbox_batch(net, (const void *const *)images, widths, heights, n, 1);
}

extern "C" int b200_letterbox_batch(network *net, const image *images, int n)
{
    std::vector<const void *> ptr(n > 0 ? n : 0); std::vector<int> w(ptr.size()), h(ptr.size());
    for (int i = 0; i < n; ++i) {
        if (images[i].c != 3) { fprintf(stderr, "b200-darknet: b200_letterbox_batch: 3-channel images only\n"); return -1; }
        ptr[i] = images[i].data; w[i] = images[i].w; h[i] = images[i].h;
    }
    return letterbox_batch(net, ptr.data(), w.data(), h.data(), n, 0);
}

// device copy of the current network input as host fp32 NCHW (inspection / tests)
extern "C" void b200_fetch_input(network *net, float *dst, int images)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_fetch_input");
    B200_CHECK(cudaMemcpyAsync(dst, e->d_input, (size_t)images * net->inputs * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    B200_CHECK(cudaStreamSynchronize(e->stream));
}

// double-buffered serving loop: submit(k+1) ; detect_submitted(k) ; submit(k+2) ; ...  The H2D of the next batch runs on
// the copy stream into the spare input buffer while the current batch computes.
extern "C" void b200_submit_batch(network *net, const float *input)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_submit_batch");
    if (e->submitted) { fprintf(stderr, "b200-darknet: b200_submit_batch called twice without b200_detect_submitted\n"); abort(); }
    if (input == B200_INPUT_RESIDENT) {          // the batch is whatever the input buffer holds now: its forward pass starts here
        enqueue_forward(e, net, 0);
        e->submitted = 1; e->fwd_enqueued = 1;
        return;
    }
    int batch = logical_batch(e, net);
    if (!e->d_input_next) e->d_input_next = (float *)dev_alloc((size_t)e->cap * net->inputs * sizeof(float));
    B200_CHECK(cudaMemcpyAsync(e->d_input_next, input, (size_t)batch * net->inputs * sizeof(float), cudaMemcpyHostToDevice, e->copy_stream));
    B200_CHECK(cudaEventRecord(e->submit_done, e->copy_stream));
    e->submitted = 1;
}

// the batch b200_submit_batch handed over becomes current: unless its forward pass is already enqueued, the spare buffer
// its copy went to becomes the input and the compute stream waits for that copy.  Returns the first layer still to
// enqueue: 0, or net->n
static int make_submitted_current(b200_engine *e, const network *net, const char *what)
{
    if (!e->submitted) { fprintf(stderr, "b200-darknet: %s without a submitted batch\n", what); abort(); }
    int first = net->n;
    if (!e->fwd_enqueued) {
        float *t = e->d_input; e->d_input = e->d_input_next; e->d_input_next = t;
        B200_CHECK(cudaStreamWaitEvent(e->stream, e->submit_done, 0));
        first = 0;
    }
    e->submitted = 0; e->fwd_enqueued = 0;
    return first;
}

// the serving loops' step after the current batch's tail is enqueued: submit `next_input` (may be NULL) and enqueue its forward
// pass, so that the next call finds that batch submitted with its forward pass in the stream
static void enqueue_next_batch(b200_engine *e, network *net, const float *next_input)
{
    if (!next_input) return;
    b200_submit_batch(net, next_input);
    enqueue_forward(e, net, make_submitted_current(e, net, "b200_submit_batch"));
    e->submitted = 1; e->fwd_enqueued = 1;
}

extern "C" int b200_detect_submitted(network *net, const float *next_input, int w, int h, float thresh, float nms_thresh,
                                     int relative, b200_det *out, int max_out, int *counts)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_detect_submitted");
    if (refuse_classifier(e, "b200_detect_submitted")) return -1;
    const int first = make_submitted_current(e, net, "b200_detect_submitted");
    // Once this batch's decode / NMS / collect are in the stream, the NEXT batch's copy is submitted and its whole forward pass
    // is enqueued behind them; the results of this batch are then read back on a separate stream while that forward runs.
    // (Waiting for the results first left the GPU idle for the two D2H round trips: ~0.25 ms of every 5 ms step.)
    return detect_core(e, net, first, w, h, thresh, nms_thresh, relative, out, max_out, counts, [&] { enqueue_next_batch(e, net, next_input); });
}

// ----------------------------------------------------------------------------------------------------
// classifiers: network_predict + top_k (predict_classifier, examples/classifier.c) for every image of the batch, the ranking
// on the device; only `top` (class, probability) pairs per image cross PCIe.
// ----------------------------------------------------------------------------------------------------
static bool classify_args_ok(const b200_engine *e, const network *net, int top, const char *what)
{
    if (e->cls_layer < 0) {
        fprintf(stderr, "b200-darknet: %s: the network does not end in [softmax]\n", what);
        return false;
    }
    const layer &l = net->layers[e->cls_layer];
    if (l.groups != 1) {
        fprintf(stderr, "b200-darknet: %s: the final [softmax] has groups = %d; ranking needs groups = 1\n", what, l.groups);
        return false;
    }
    if (top < 1 || top > 64 || top > l.outputs) {
        fprintf(stderr, "b200-darknet: %s: top = %d is outside 1..%d\n", what, top, l.outputs < 64 ? l.outputs : 64);
        return false;
    }
    return true;
}

// forward from layer `first` (net->n: already in the stream) + top-k on the compute stream; `after_tail` enqueues the next
// batch behind them before the results are read back on their own stream (the pattern of detect_core)
template <typename F>
static int classify_core(b200_engine *e, network *net, int first, int top, int *classes, float *probs, F after_tail)
{
    const int batch = logical_batch(e, net);
    const layer &l = net->layers[e->cls_layer];
    if (!e->d_top_cls) {
        e->d_top_cls = (int *)dev_alloc((size_t)e->cap * 64 * sizeof(int));
        e->d_top_prob = (float *)dev_alloc((size_t)e->cap * 64 * sizeof(float));
    }
    enqueue_forward(e, net, first);
    launch_topk(e->L[e->cls_layer].head_out, batch, l.outputs, l.outputs, top, e->d_top_cls, e->d_top_prob, e->stream);
    B200_CHECK(cudaEventRecord(e->tail_done, e->stream));
    B200_CHECK(cudaStreamWaitEvent(e->d2h_stream, e->tail_done, 0));
    after_tail();
    B200_CHECK(cudaMemcpyAsync(classes, e->d_top_cls, (size_t)batch * top * sizeof(int), cudaMemcpyDeviceToHost, e->d2h_stream));
    B200_CHECK(cudaMemcpyAsync(probs, e->d_top_prob, (size_t)batch * top * sizeof(float), cudaMemcpyDeviceToHost, e->d2h_stream));
    B200_CHECK(cudaStreamSynchronize(e->d2h_stream));
    return batch;
}

extern "C" int b200_classify_batch(network *net, const float *input, int top, int *classes, float *probs)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_classify_batch");
    if (!classify_args_ok(e, net, top, "b200_classify_batch")) return -1;
    const int first = stage_batch_input(e, net, input);
    const int n = classify_core(e, net, first, top, classes, probs, [] {});
    B200_CHECK(cudaStreamSynchronize(e->stream));
    return n;
}

extern "C" int b200_classify_submitted(network *net, const float *next_input, int top, int *classes, float *probs)
{
    b200_engine *e = b200_engine_of(net);
    need_device(e, "b200_classify_submitted");
    if (!classify_args_ok(e, net, top, "b200_classify_submitted")) return -1;
    const int first = make_submitted_current(e, net, "b200_classify_submitted");
    return classify_core(e, net, first, top, classes, probs, [&] { enqueue_next_batch(e, net, next_input); });
}

// device NMS on caller-provided host arrays (the kernel behind do_nms_sort / do_nms_obj).  Stream, scratch slab and staging
// buffers are kept per DEVICE and only ever grow: a `darknet detect`-style caller pays no cudaMalloc / cudaFree per call.
struct NmsHostPath {
    cudaStream_t stream;
    NmsScratch scratch;
    float *d_box, *d_val; int *d_cls;
    size_t box_floats, val_floats, cls_ints;
};
static NmsHostPath g_nms_path[64];

static NmsHostPath &nms_prepare(size_t box_floats, size_t val_floats, size_t cls_ints)
{
    if (!cuda_usable()) {
        fprintf(stderr, "b200-darknet: do_nms_sort/do_nms_obj need a CUDA device. There is no CPU fallback.\n");
        abort();
    }
    int dev = 0;
    B200_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) { fprintf(stderr, "b200-darknet: device ordinal %d out of range\n", dev); abort(); }
    NmsHostPath &p = g_nms_path[dev];
    if (!p.stream) B200_CHECK(cudaStreamCreateWithFlags(&p.stream, cudaStreamNonBlocking));
    if (p.box_floats < box_floats) { cudaFree(p.d_box); p.d_box = (float *)dev_alloc(box_floats * sizeof(float)); p.box_floats = box_floats; }
    if (p.val_floats < val_floats) { cudaFree(p.d_val); p.d_val = (float *)dev_alloc(val_floats * sizeof(float)); p.val_floats = val_floats; }
    if (p.cls_ints < cls_ints) { cudaFree(p.d_cls); p.d_cls = (int *)dev_alloc(cls_ints * sizeof(int)); p.cls_ints = cls_ints; }
    return p;
}

extern "C" void b200_nms_sort_arrays(const float *boxes, float *probs, int n, int classes, float thresh)
{
    if (n <= 0 || classes <= 0) return;
    NmsHostPath &p = nms_prepare((size_t)n * 4, (size_t)n * classes, (size_t)classes + 1);
    B200_CHECK(cudaMemcpyAsync(p.d_box, boxes, (size_t)n * 4 * sizeof(float), cudaMemcpyHostToDevice, p.stream));
    B200_CHECK(cudaMemcpyAsync(p.d_val, probs, (size_t)n * classes * sizeof(float), cudaMemcpyHostToDevice, p.stream));
    launch_nms_sort(p.d_box, p.d_val, nullptr, nullptr, 1, n, classes, thresh, n, &p.scratch, p.d_cls, p.stream);
    B200_CHECK(cudaMemcpyAsync(probs, p.d_val, (size_t)n * classes * sizeof(float), cudaMemcpyDeviceToHost, p.stream));
    B200_CHECK(cudaStreamSynchronize(p.stream));
}

extern "C" void b200_nms_obj_arrays(const float *boxes, float *objectness, int n, float thresh, unsigned char *suppressed)
{
    if (n <= 0) return;
    NmsHostPath &p = nms_prepare((size_t)n * 4, (size_t)n, 2);
    std::vector<float> before(objectness, objectness + n);
    B200_CHECK(cudaMemcpyAsync(p.d_box, boxes, (size_t)n * 4 * sizeof(float), cudaMemcpyHostToDevice, p.stream));
    B200_CHECK(cudaMemcpyAsync(p.d_val, objectness, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, p.stream));
    launch_nms_obj(p.d_box, p.d_val, nullptr, nullptr, 1, n, 1, thresh, n, &p.scratch, p.stream);
    B200_CHECK(cudaMemcpyAsync(objectness, p.d_val, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, p.stream));
    B200_CHECK(cudaStreamSynchronize(p.stream));
    if (suppressed) for (int i = 0; i < n; ++i) suppressed[i] = (before[i] != 0.f && objectness[i] == 0.f) ? 1 : 0;
}

extern "C" void b200_top_k_arrays(const float *probs, int rows, int n, int top, int *classes)
{
    if (rows <= 0 || n <= 0 || top < 1 || top > 64 || top > n) {
        fprintf(stderr, "b200-darknet: b200_top_k_arrays: needs rows >= 1 and 1 <= top <= min(n, 64)\n");
        abort();
    }
    NmsHostPath &p = nms_prepare(0, (size_t)rows * n, (size_t)rows * top);
    B200_CHECK(cudaMemcpyAsync(p.d_val, probs, (size_t)rows * n * sizeof(float), cudaMemcpyHostToDevice, p.stream));
    launch_topk(p.d_val, rows, n, n, top, p.d_cls, nullptr, p.stream);
    B200_CHECK(cudaMemcpyAsync(classes, p.d_cls, (size_t)rows * top * sizeof(int), cudaMemcpyDeviceToHost, p.stream));
    B200_CHECK(cudaStreamSynchronize(p.stream));
}
