/*
 * layers.c — one constructor per layer type of the YOLOv1/v2/v3 inference path.
 *
 * Each constructor reproduces, for its type, what the reference's parse_X + make_X_layer pair
 * establishes: the public geometry fields drivers read (w,h,c,out_*,n,size,stride,pad,classes,…),
 * the fp32 host parameter arrays that load_weights fills, the host `output` buffer, and the stderr
 * row of the layer table (the structural golden, tests/golden/layer_tables).  No arithmetic lives
 * here: the forward pass is planned and executed by the device engine (dev/engine.cu).
 */
#include "layers.h"
#include <math.h>
#include <assert.h>

static void fatal(const char *msg)
{
    fprintf(stderr, "b200-darknet: %s\n", msg);
    exit(-1);
}

static void forward_on_engine_only(layer l, network net)
{
    (void)l; (void)net;
    fatal("layer.forward() is not a CPU entry point in this engine; call network_predict()");
}

ACTIVATION activation_from_name(const char *s)
{
    /* activations.c:44-60 get_activation */
    static const struct { const char *name; ACTIVATION a; } table[] = {
        {"logistic", LOGISTIC}, {"loggy", LOGGY}, {"relu", RELU}, {"elu", ELU}, {"relie", RELIE},
        {"plse", PLSE}, {"hardtan", HARDTAN}, {"lhtan", LHTAN}, {"linear", LINEAR}, {"ramp", RAMP},
        {"leaky", LEAKY}, {"tanh", TANH}, {"stair", STAIR},
    };
    for (size_t i = 0; i < sizeof table / sizeof table[0]; ++i)
        if (strcmp(s, table[i].name) == 0) return table[i].a;
    fprintf(stderr, "Couldn't find activation function %s, going with ReLU\n", s);
    return RELU;
}

static float *host_floats(size_t n) { return calloc(n ? n : 1, sizeof(float)); }

static void need_image(shape_cursor cur, const char *who)
{
    if (!(cur.h && cur.w && cur.c)) {
        fprintf(stderr, "Layer before %s layer must output image.\n", who);
        exit(-1);
    }
}

/* parse a comma separated list; returns count */
static int split_ints(const char *s, int **out)
{
    int n = 1;
    for (const char *p = s; *p; ++p) if (*p == ',') ++n;
    int *v = calloc(n, sizeof(int));
    for (int i = 0; i < n; ++i) {
        v[i] = atoi(s);
        const char *comma = strchr(s, ',');
        s = comma ? comma + 1 : s + strlen(s);
    }
    *out = v;
    return n;
}

static void read_anchor_list(cfg_section *opt, float *dst, int room)
{
    const char *a = cfg_str(opt, "anchors", 0);
    if (!a) return;
    for (int i = 0; ; ++i) {
        if (i >= room) fatal("more anchor values than 2*num in the cfg");      /* the reference overruns l.biases here (parser.c:328-337) */
        dst[i] = (float)atof(a);
        const char *comma = strchr(a, ',');
        if (!comma) break;
        a = comma + 1;
    }
}

/* [convolutional]: parser.c:177-205 + convolutional_layer.c:176-328 */
static layer conv_layer(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = CONVOLUTIONAL;
    l.n       = cfg_int(opt, "filters", 1);
    l.size    = cfg_int(opt, "size", 1);
    l.stride  = cfg_int(opt, "stride", 1);
    int pad   = cfg_int_quiet(opt, "pad", 0);
    l.pad     = cfg_int_quiet(opt, "padding", 0);
    l.groups  = cfg_int_quiet(opt, "groups", 1);
    if (pad) l.pad = l.size / 2;
    l.activation = activation_from_name(cfg_str(opt, "activation", "logistic"));
    need_image(cur, "convolutional");
    l.batch_normalize = cfg_int_quiet(opt, "batch_normalize", 0);
    l.binary = cfg_int_quiet(opt, "binary", 0);
    l.xnor   = cfg_int_quiet(opt, "xnor", 0);
    if (l.binary || l.xnor) fatal("binary/xnor convolutions are outside the YOLO inference path");
    if (l.groups != 1)      fatal("grouped convolutions are outside the YOLO inference path");
    l.h = cur.h; l.w = cur.w; l.c = cur.c; l.batch = cur.batch;
    l.out_h = (l.h + 2 * l.pad - l.size) / l.stride + 1;
    l.out_w = (l.w + 2 * l.pad - l.size) / l.stride + 1;
    l.out_c = l.n;
    l.outputs  = l.out_h * l.out_w * l.out_c;
    l.inputs   = l.h * l.w * l.c;
    l.nweights = l.c / l.groups * l.n * l.size * l.size;
    l.nbiases  = l.n;
    l.weights  = host_floats(l.nweights);
    l.biases   = host_floats(l.n);
    if (l.batch_normalize) {
        l.scales = host_floats(l.n);
        for (int i = 0; i < l.n; ++i) l.scales[i] = 1;
        l.rolling_mean = host_floats(l.n);
        l.rolling_variance = host_floats(l.n);
    }
    l.output = host_floats((size_t)l.batch * l.outputs);
    l.workspace_size = (size_t)l.out_h * l.out_w * l.size * l.size * l.c / l.groups * sizeof(float);
    l.flipped = cfg_int_quiet(opt, "flipped", 0);
    l.dot = cfg_float_quiet(opt, "dot", 0);
    fprintf(stderr, "conv  %5d %2d x%2d /%2d  %4d x%4d x%4d   ->  %4d x%4d x%4d  %5.3f BFLOPs\n",
            l.n, l.size, l.size, l.stride, l.w, l.h, l.c, l.out_w, l.out_h, l.out_c,
            (2.0 * l.n * l.size * l.size * l.c / l.groups * l.out_h * l.out_w) / 1000000000.);
    return l;
}

/* [local]: parser.c:130-149 + local_layer.c:10-89 (unshared convolution of YOLOv1) */
static layer local_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = LOCAL;
    l.n      = cfg_int(opt, "filters", 1);
    l.size   = cfg_int(opt, "size", 1);
    l.stride = cfg_int(opt, "stride", 1);
    l.pad    = cfg_int(opt, "pad", 0);
    l.activation = activation_from_name(cfg_str(opt, "activation", "logistic"));
    need_image(cur, "local");
    l.h = cur.h; l.w = cur.w; l.c = cur.c; l.batch = cur.batch;
    l.out_h = (l.pad ? l.h - 1 : l.h - l.size) / l.stride + 1;
    l.out_w = (l.pad ? l.w - 1 : l.w - l.size) / l.stride + 1;
    l.out_c = l.n;
    int locations = l.out_h * l.out_w;
    l.outputs = locations * l.out_c;
    l.inputs  = l.w * l.h * l.c;
    l.nweights = l.c * l.n * l.size * l.size * locations;   /* the reference leaves nweights 0; we record it */
    l.weights = host_floats((size_t)l.nweights);
    l.biases  = host_floats(l.outputs);
    l.output  = host_floats((size_t)l.batch * l.outputs);
    l.workspace_size = (size_t)locations * l.size * l.size * l.c * sizeof(float);
    fprintf(stderr, "Local Layer: %d x %d x %d image, %d filters -> %d x %d x %d image\n",
            l.h, l.w, l.c, l.n, l.out_h, l.out_w, l.n);
    return l;
}

/* [connected]: parser.c:257-266 + connected_layer.c:14-131 */
static layer connected_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = CONNECTED;
    l.outputs = cfg_int(opt, "output", 1);
    l.activation = activation_from_name(cfg_str(opt, "activation", "logistic"));
    l.batch_normalize = cfg_int_quiet(opt, "batch_normalize", 0);
    l.inputs = cur.inputs; l.batch = cur.batch;
    l.h = 1; l.w = 1; l.c = l.inputs;
    l.out_h = 1; l.out_w = 1; l.out_c = l.outputs;
    l.nweights = l.inputs * l.outputs;
    l.nbiases = l.outputs;
    l.weights = host_floats((size_t)l.nweights);
    l.biases  = host_floats(l.outputs);
    if (l.batch_normalize) {
        l.scales = host_floats(l.outputs);
        for (int i = 0; i < l.outputs; ++i) l.scales[i] = 1;
        l.rolling_mean = host_floats(l.outputs);
        l.rolling_variance = host_floats(l.outputs);
    }
    l.output = host_floats((size_t)l.batch * l.outputs);
    fprintf(stderr, "connected                            %4d  ->  %4d\n", l.inputs, l.outputs);
    return l;
}

/* [maxpool]: parser.c:471-486 + maxpool_layer.c:21-52.  `indexes` (argmax) is training-only and not kept. */
static layer maxpool_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = MAXPOOL;
    l.stride = cfg_int(opt, "stride", 1);
    l.size   = cfg_int(opt, "size", l.stride);
    l.pad    = cfg_int_quiet(opt, "padding", (l.size - 1) / 2);
    need_image(cur, "maxpool");
    l.h = cur.h; l.w = cur.w; l.c = cur.c; l.batch = cur.batch;
    l.out_w = (l.w + 2 * l.pad) / l.stride;
    l.out_h = (l.h + 2 * l.pad) / l.stride;
    l.out_c = l.c;
    l.outputs = l.out_h * l.out_w * l.out_c;
    l.inputs  = l.h * l.w * l.c;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    fprintf(stderr, "max          %d x %d / %d  %4d x%4d x%4d   ->  %4d x%4d x%4d\n",
            l.size, l.size, l.stride, l.w, l.h, l.c, l.out_w, l.out_h, l.out_c);
    return l;
}

/* [route]: parser.c:589-628 + route_layer.c:7-39 */
static layer route_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = ROUTE;
    const char *spec = cfg_find(opt, "layers");
    if (!spec) fatal("Route Layer must specify input layers");
    l.n = split_ints(spec, &l.input_layers);
    l.input_sizes = calloc(l.n, sizeof(int));
    l.batch = cur.batch;
    fprintf(stderr, "route ");
    for (int i = 0; i < l.n; ++i) {
        if (l.input_layers[i] < 0) l.input_layers[i] += cur.index;
        if (l.input_layers[i] < 0 || l.input_layers[i] >= cur.index) fatal("route: input layer index out of range");
        l.input_sizes[i] = cur.net->layers[l.input_layers[i]].outputs;
        l.outputs += l.input_sizes[i];
        fprintf(stderr, " %d", l.input_layers[i]);
    }
    fprintf(stderr, "\n");
    l.inputs = l.outputs;
    const layer *first = &cur.net->layers[l.input_layers[0]];
    l.out_w = first->out_w; l.out_h = first->out_h; l.out_c = first->out_c;
    for (int i = 1; i < l.n; ++i) {
        const layer *next = &cur.net->layers[l.input_layers[i]];
        if (next->out_w == first->out_w && next->out_h == first->out_h) l.out_c += next->out_c;
        else l.out_h = l.out_w = l.out_c = 0;
    }
    l.w = l.out_w; l.h = l.out_h; l.c = l.out_c;
    l.output = host_floats((size_t)l.batch * l.outputs);
    return l;
}

/* [upsample]: parser.c:580-587 + upsample_layer.c:7-42 */
static layer upsample_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = UPSAMPLE;
    l.stride = cfg_int(opt, "stride", 2);
    l.batch = cur.batch; l.w = cur.w; l.h = cur.h; l.c = cur.c;
    if (l.stride < 0) fatal("downsample (negative upsample stride) is outside the YOLO inference path");
    l.out_w = l.w * l.stride; l.out_h = l.h * l.stride; l.out_c = l.c;
    l.outputs = l.out_w * l.out_h * l.out_c;
    l.inputs  = l.w * l.h * l.c;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    fprintf(stderr, "upsample           %2dx  %4d x%4d x%4d   ->  %4d x%4d x%4d\n",
            l.stride, l.w, l.h, l.c, l.out_w, l.out_h, l.out_c);
    l.scale = cfg_float_quiet(opt, "scale", 1);
    return l;
}

/* [shortcut]: parser.c:527-544 + shortcut_layer.c:9-37 */
static layer shortcut_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = SHORTCUT;
    const char *from = cfg_find(opt, "from");
    if (!from) fatal("shortcut: missing from=");
    l.index = atoi(from);
    if (l.index < 0) l.index += cur.index;
    if (l.index < 0 || l.index >= cur.index) fatal("shortcut: from= out of range");
    const layer *src = &cur.net->layers[l.index];
    l.batch = cur.batch;
    /* w,h,c describe the ADDED tensor (layer `index`); out_* the tensor flowing through (shortcut_layer.c:15-21) */
    l.w = src->out_w; l.h = src->out_h; l.c = src->out_c;
    l.out_w = cur.w; l.out_h = cur.h; l.out_c = cur.c;
    l.outputs = cur.w * cur.h * cur.c;
    l.inputs  = l.outputs;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    fprintf(stderr, "res  %3d                %4d x%4d x%4d   ->  %4d x%4d x%4d\n",
            l.index, l.w, l.h, l.c, l.out_w, l.out_h, l.out_c);
    l.activation = activation_from_name(cfg_str(opt, "activation", "linear"));
    l.alpha = cfg_float_quiet(opt, "alpha", 1);
    l.beta  = cfg_float_quiet(opt, "beta", 1);
    return l;
}

/* [reorg]: parser.c:453-469 + reorg_layer.c:10-58 */
static layer reorg_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = REORG;
    l.stride  = cfg_int(opt, "stride", 1);
    l.reverse = cfg_int_quiet(opt, "reverse", 0);
    l.flatten = cfg_int_quiet(opt, "flatten", 0);
    l.extra   = cfg_int_quiet(opt, "extra", 0);
    need_image(cur, "reorg");
    if (l.flatten || l.extra) fatal("reorg flatten/extra are outside the YOLO inference path");
    l.batch = cur.batch; l.h = cur.h; l.w = cur.w; l.c = cur.c;
    if (l.reverse) { l.out_w = l.w * l.stride; l.out_h = l.h * l.stride; l.out_c = l.c / (l.stride * l.stride); }
    else           { l.out_w = l.w / l.stride; l.out_h = l.h / l.stride; l.out_c = l.c * (l.stride * l.stride); }
    l.outputs = l.out_h * l.out_w * l.out_c;
    l.inputs  = l.h * l.w * l.c;
    fprintf(stderr, "reorg              /%2d  %4d x%4d x%4d   ->  %4d x%4d x%4d\n",
            l.stride, l.w, l.h, l.c, l.out_w, l.out_h, l.out_c);
    l.output = host_floats((size_t)l.batch * l.outputs);
    return l;
}

/* [dropout]: parser.c:501-509 + dropout_layer.c:7-26; identity at inference, output aliased by the caller */
static layer dropout_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = DROPOUT;
    l.probability = cfg_float(opt, "probability", .5);
    l.inputs = l.outputs = cur.inputs;
    l.batch = cur.batch;
    l.scale = 1.f / (1.f - l.probability);
    l.out_w = cur.w; l.out_h = cur.h; l.out_c = cur.c;
    l.w = cur.w; l.h = cur.h; l.c = cur.c;
    fprintf(stderr, "dropout       p = %.2f               %4d  ->  %4d\n", l.probability, l.inputs, l.inputs);
    return l;
}

/* [avgpool]: parser.c parse_avgpool + avgpool_layer.c make_avgpool_layer (global average pool of the classifiers) */
static layer avgpool_layer_(cfg_section *opt, shape_cursor cur)
{
    (void)opt;
    layer l = {0};
    l.type = AVGPOOL;
    need_image(cur, "avgpool");
    l.batch = cur.batch; l.w = cur.w; l.h = cur.h; l.c = cur.c;
    fprintf(stderr, "avg                     %4d x%4d x%4d   ->  %4d\n", l.w, l.h, l.c, l.c);
    l.out_w = 1; l.out_h = 1; l.out_c = l.c;
    l.outputs = l.out_c;
    l.inputs  = l.h * l.w * l.c;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    return l;
}

/* [softmax]: parser.c parse_softmax + softmax_layer.c make_softmax_layer */
static layer softmax_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = SOFTMAX;
    l.groups = cfg_int_quiet(opt, "groups", 1);
    if (l.groups < 1 || cur.inputs % l.groups != 0) fatal("softmax groups must divide the layer's inputs");
    fprintf(stderr, "softmax                                        %4d\n", cur.inputs);
    l.batch = cur.batch;
    l.inputs = l.outputs = cur.inputs;
    l.output = host_floats((size_t)l.batch * l.outputs);
    l.cost = host_floats(1);
    l.temperature = cfg_float_quiet(opt, "temperature", 1);
    if (cfg_str(opt, "tree", 0)) fatal("softmax tree= (WordTree classifiers) is outside the inference path");
    l.w = cur.w; l.h = cur.h; l.c = cur.c;
    l.spatial = (int)cfg_float_quiet(opt, "spatial", 0);
    if (l.spatial) fatal("softmax spatial= is outside the inference path");
    (void)cfg_int_quiet(opt, "noloss", 0);                  /* training only */
    return l;
}

/* [cost]: parser.c parse_cost + cost_layer.c make_cost_layer.  Identity at inference: network_predict clears net->truth, so
 * forward_cost_layer returns at once; the device engine aliases it to its input. */
static layer cost_layer_(cfg_section *opt, shape_cursor cur)
{
    static const struct { const char *name; COST_TYPE t; } types[] = {
        {"sse", SSE}, {"masked", MASKED}, {"smooth", SMOOTH}, {"L1", L1}, {"seg", SEG}, {"wgan", WGAN},
    };
    layer l = {0};
    l.type = COST;
    const char *type = cfg_str(opt, "type", "sse");
    l.cost_type = SSE;
    size_t k = 0;
    while (k < sizeof types / sizeof types[0] && strcmp(type, types[k].name) != 0) ++k;
    if (k < sizeof types / sizeof types[0]) l.cost_type = types[k].t;
    else fprintf(stderr, "Couldn't find cost type %s, going with SSE\n", type);          /* cost_layer.c get_cost_type */
    l.scale = cfg_float_quiet(opt, "scale", 1);
    fprintf(stderr, "cost                                           %4d\n", cur.inputs);
    l.batch = cur.batch;
    l.inputs = l.outputs = cur.inputs;
    l.output = host_floats((size_t)l.batch * l.outputs);
    l.cost = host_floats(1);
    l.ratio = cfg_float_quiet(opt, "ratio", 0);
    l.noobject_scale = cfg_float_quiet(opt, "noobj", 1);
    l.thresh = cfg_float_quiet(opt, "thresh", 0);
    return l;
}

/* [yolo]: parser.c:303-339 + yolo_layer.c:13-61 */
static layer yolo_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = YOLO;
    l.classes = cfg_int(opt, "classes", 20);
    l.total   = cfg_int(opt, "num", 1);
    l.n = l.total;
    const char *m = cfg_str(opt, "mask", 0);
    if (m) l.n = split_ints(m, &l.mask);
    else { l.mask = calloc(l.n, sizeof(int)); for (int i = 0; i < l.n; ++i) l.mask[i] = i; }
    l.batch = cur.batch; l.h = cur.h; l.w = cur.w;
    l.c = l.n * (l.classes + 4 + 1);
    l.out_w = l.w; l.out_h = l.h; l.out_c = l.c;
    l.outputs = l.h * l.w * l.c;
    l.inputs  = l.outputs;
    l.truths  = 90 * (4 + 1);
    l.biases  = host_floats(l.total * 2);
    for (int i = 0; i < l.total * 2; ++i) l.biases[i] = .5f;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    l.cost    = host_floats(1);
    fprintf(stderr, "yolo\n");
    srand(0);                                    /* yolo_layer.c:58 — kept: drivers may rely on the RNG reset */
    assert(l.outputs == cur.inputs);
    l.max_boxes     = cfg_int_quiet(opt, "max", 90);
    l.jitter        = cfg_float(opt, "jitter", .2);
    l.ignore_thresh = cfg_float(opt, "ignore_thresh", .5);
    l.truth_thresh  = cfg_float(opt, "truth_thresh", 1);
    l.random        = cfg_int_quiet(opt, "random", 0);
    if (cfg_str(opt, "map", 0)) fatal("yolo map= files are outside the YOLO inference path");
    read_anchor_list(opt, l.biases, l.total * 2);
    return l;
}

/* [region]: parser.c:341-391 + region_layer.c:13-54 */
static layer region_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = REGION;
    l.coords  = cfg_int(opt, "coords", 4);
    l.classes = cfg_int(opt, "classes", 20);
    l.n       = cfg_int(opt, "num", 1);
    l.batch = cur.batch; l.h = cur.h; l.w = cur.w;
    l.c = l.n * (l.classes + l.coords + 1);
    l.out_w = l.w; l.out_h = l.h; l.out_c = l.c;
    l.outputs = l.h * l.w * l.c;
    l.inputs  = l.outputs;
    l.truths  = 30 * (l.coords + 1);
    l.biases  = host_floats(l.n * 2);
    for (int i = 0; i < l.n * 2; ++i) l.biases[i] = .5f;
    l.output  = host_floats((size_t)l.batch * l.outputs);
    l.cost    = host_floats(1);
    fprintf(stderr, "detection\n");
    srand(0);
    assert(l.outputs == cur.inputs);
    l.log        = cfg_int_quiet(opt, "log", 0);
    l.sqrt       = cfg_int_quiet(opt, "sqrt", 0);
    l.softmax    = cfg_int(opt, "softmax", 0);
    l.background = cfg_int_quiet(opt, "background", 0);
    l.max_boxes  = cfg_int_quiet(opt, "max", 30);
    l.jitter     = cfg_float(opt, "jitter", .2);
    l.rescore    = cfg_int_quiet(opt, "rescore", 0);
    l.thresh     = cfg_float(opt, "thresh", .5);
    l.classfix   = cfg_int_quiet(opt, "classfix", 0);
    l.absolute   = cfg_int_quiet(opt, "absolute", 0);
    l.random     = cfg_int_quiet(opt, "random", 0);
    l.coord_scale    = cfg_float(opt, "coord_scale", 1);
    l.object_scale   = cfg_float(opt, "object_scale", 1);
    l.noobject_scale = cfg_float(opt, "noobject_scale", 1);
    l.mask_scale     = cfg_float(opt, "mask_scale", 1);
    l.class_scale    = cfg_float(opt, "class_scale", 1);
    l.bias_match     = cfg_int_quiet(opt, "bias_match", 0);
    {   /* YOLO9000 (parser.c:372-375): the class WordTree and the training-time class map */
        const char *tree_file = cfg_str(opt, "tree", 0);
        if (tree_file) {
            l.softmax_tree = read_tree((char *)tree_file);
            if (l.softmax_tree->n != l.classes) fatal("region tree= file does not list `classes` entries");
        }
        const char *map_file = cfg_str(opt, "map", 0);
        if (map_file) l.map = read_map((char *)map_file);
    }
    if (l.background || l.coords != 4) fatal("region background/coords!=4 are outside the YOLO inference path");
    read_anchor_list(opt, l.biases, l.n * 2);
    return l;
}

/* [detection]: parser.c:393-415 + detection_layer.c:14-48 (YOLOv1 head) */
static layer detection_layer_(cfg_section *opt, shape_cursor cur)
{
    layer l = {0};
    l.type = DETECTION;
    l.coords  = cfg_int(opt, "coords", 1);
    l.classes = cfg_int(opt, "classes", 1);
    l.rescore = cfg_int(opt, "rescore", 0);
    l.n       = cfg_int(opt, "num", 1);
    l.side    = cfg_int(opt, "side", 7);
    l.batch = cur.batch; l.inputs = cur.inputs;
    l.w = l.side; l.h = l.side;
    assert(l.side * l.side * ((1 + l.coords) * l.n + l.classes) == l.inputs);
    l.outputs = l.inputs;
    l.truths  = l.side * l.side * (1 + l.coords + l.classes);
    l.output  = host_floats((size_t)l.batch * l.outputs);
    l.cost    = host_floats(1);
    fprintf(stderr, "Detection Layer\n");
    srand(0);
    l.softmax   = cfg_int(opt, "softmax", 0);
    l.sqrt      = cfg_int(opt, "sqrt", 0);
    l.max_boxes = cfg_int_quiet(opt, "max", 90);
    l.coord_scale    = cfg_float(opt, "coord_scale", 1);
    l.forced         = cfg_int(opt, "forced", 0);
    l.object_scale   = cfg_float(opt, "object_scale", 1);
    l.noobject_scale = cfg_float(opt, "noobject_scale", 1);
    l.class_scale    = cfg_float(opt, "class_scale", 1);
    l.jitter         = cfg_float(opt, "jitter", .2);
    l.random         = cfg_int_quiet(opt, "random", 0);
    l.reorg          = cfg_int_quiet(opt, "reorg", 0);
    return l;
}

int build_layer(const char *type, cfg_section *opt, shape_cursor cur, layer *out)
{
    static const struct { const char *a, *b; layer (*make)(cfg_section *, shape_cursor); } ctor[] = {
        {"[convolutional]", "[conv]", conv_layer},   {"[local]", 0, local_layer_},
        {"[connected]", "[conn]", connected_layer_}, {"[maxpool]", "[max]", maxpool_layer_},
        {"[route]", 0, route_layer_},                {"[upsample]", 0, upsample_layer_},
        {"[shortcut]", 0, shortcut_layer_},          {"[reorg]", 0, reorg_layer_},
        {"[dropout]", 0, dropout_layer_},            {"[yolo]", 0, yolo_layer_},
        {"[region]", 0, region_layer_},              {"[detection]", 0, detection_layer_},
        {"[avgpool]", "[avg]", avgpool_layer_},      {"[softmax]", "[soft]", softmax_layer_},
        {"[cost]", 0, cost_layer_},
    };
    for (size_t i = 0; i < sizeof ctor / sizeof ctor[0]; ++i) {
        if (strcmp(type, ctor[i].a) == 0 || (ctor[i].b && strcmp(type, ctor[i].b) == 0)) {
            *out = ctor[i].make(opt, cur);
            out->forward = forward_on_engine_only;
            return 1;
        }
    }
    return 0;
}

void release_layer_host(layer l)
{
    /* layer.c:6-97 frees every non-NULL host pointer; DROPOUT aliases its neighbour's output (layer.c:8-13) */
    if (l.type == DROPOUT) return;
    free(l.mask); free(l.input_layers); free(l.input_sizes); free(l.cost);
    free(l.biases); free(l.scales); free(l.weights); free(l.output);
    free(l.rolling_mean); free(l.rolling_variance);
}
