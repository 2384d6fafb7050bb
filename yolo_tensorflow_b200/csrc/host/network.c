/*
 * network.c — darknet-compatible network lifetime + forward entry points (host C).
 *
 * Replaces, for the inference path, the reference's parser.c:730-874 (parse_network_cfg),
 * network.c:53-61,188-211,339-356,497-508,579-589,699-730.  The layer array it builds is the
 * public data model drivers read; the arithmetic is delegated to the device engine through the
 * C ABI in include/b200_engine.h.
 */
#include "darknet.h"
#include "b200_engine.h"
#include "cfg.h"
#include "layers.h"
#include <sys/time.h>
#include <assert.h>

int gpu_index = 0;

static int g_default_precision = -1;

void b200_set_default_precision(int prec) { g_default_precision = prec; }

static int g_default_fusion = -1;
void b200_set_default_fusion(int on) { g_default_fusion = on; }
int b200_get_default_fusion(void)
{
    if (g_default_fusion >= 0) return g_default_fusion;
    const char *env = getenv("B200_FUSE");
    return !(env && env[0] == '0');
}

static int resolve_precision(void)
{
    if (g_default_precision >= 0) return g_default_precision;
    const char *env = getenv("B200_PRECISION");
    if (env && (strcmp(env, "fp32") == 0 || strcmp(env, "FP32") == 0)) return B200_PREC_FP32;
    return B200_PREC_BF16;
}

/* The engine pointer rides in the allocation, right behind the public struct, so that by-value copies
 * `network orig = *net; ...; *net = orig;` made by callers (network.c:499-507 idiom) cannot lose it. */
typedef struct { network pub; b200_engine *engine; } network_box;

b200_engine *b200_engine_of(const network *net) { return ((const network_box *)net)->engine; }

double what_time_is_it_now(void)
{
    struct timeval t;
    if (gettimeofday(&t, NULL)) return 0;
    return (double)t.tv_sec + (double)t.tv_usec * .000001;
}

static learning_rate_policy policy_from_name(const char *s)
{
    static const struct { const char *n; learning_rate_policy p; } tab[] = {
        {"random", RANDOM}, {"poly", POLY}, {"constant", CONSTANT}, {"step", STEP},
        {"exp", EXP}, {"sigmoid", SIG}, {"steps", STEPS},
    };
    for (size_t i = 0; i < sizeof tab / sizeof tab[0]; ++i) if (strcmp(s, tab[i].n) == 0) return tab[i].p;
    fprintf(stderr, "Couldn't find policy %s, going with constant\n", s);
    return CONSTANT;
}

/* [net] section (parser.c:643-722).  Training hyper-parameters are parsed (so that no spurious
 * "Unused field" lines appear) and stored, but nothing on the inference path reads them. */
static void read_net_section(cfg_section *o, network *net)
{
    net->batch         = cfg_int(o, "batch", 1);
    net->learning_rate = cfg_float(o, "learning_rate", .001);
    net->momentum      = cfg_float(o, "momentum", .9);
    net->decay         = cfg_float(o, "decay", .0001);
    int subdivs        = cfg_int(o, "subdivisions", 1);
    net->time_steps    = cfg_int_quiet(o, "time_steps", 1);
    net->notruth       = cfg_int_quiet(o, "notruth", 0);
    net->batch /= subdivs;
    net->batch *= net->time_steps;
    net->subdivisions  = subdivs;
    net->random        = cfg_int_quiet(o, "random", 0);
    net->adam          = cfg_int_quiet(o, "adam", 0);
    if (net->adam) {
        net->B1  = cfg_float(o, "B1", .9);
        net->B2  = cfg_float(o, "B2", .999);
        net->eps = cfg_float(o, "eps", .0000001);
    }
    net->h = cfg_int_quiet(o, "height", 0);
    net->w = cfg_int_quiet(o, "width", 0);
    net->c = cfg_int_quiet(o, "channels", 0);
    net->inputs    = cfg_int_quiet(o, "inputs", net->h * net->w * net->c);
    net->max_crop  = cfg_int_quiet(o, "max_crop", net->w * 2);
    net->min_crop  = cfg_int_quiet(o, "min_crop", net->w);
    net->max_ratio = cfg_float_quiet(o, "max_ratio", (float)net->max_crop / net->w);
    net->min_ratio = cfg_float_quiet(o, "min_ratio", (float)net->min_crop / net->w);
    net->center    = cfg_int_quiet(o, "center", 0);
    net->clip      = cfg_float_quiet(o, "clip", 0);
    net->angle      = cfg_float_quiet(o, "angle", 0);
    net->aspect     = cfg_float_quiet(o, "aspect", 1);
    net->saturation = cfg_float_quiet(o, "saturation", 1);
    net->exposure   = cfg_float_quiet(o, "exposure", 1);
    net->hue        = cfg_float_quiet(o, "hue", 0);
    if (!net->inputs && !(net->h && net->w && net->c)) {
        fprintf(stderr, "No input parameters supplied\n");
        exit(-1);
    }
    net->policy  = policy_from_name(cfg_str(o, "policy", "constant"));
    net->burn_in = cfg_int_quiet(o, "burn_in", 0);
    net->power   = cfg_float_quiet(o, "power", 4);
    if (net->policy == STEP) {
        net->step  = cfg_int(o, "step", 1);
        net->scale = cfg_float(o, "scale", 1);
    } else if (net->policy == STEPS) {
        const char *l = cfg_find(o, "steps"), *p = cfg_find(o, "scales");
        if (!l || !p) { fprintf(stderr, "STEPS policy must have steps and scales in cfg file\n"); exit(-1); }
        int n = 1;
        for (const char *q = l; *q; ++q) if (*q == ',') ++n;
        net->steps = calloc(n, sizeof(int));
        net->scales = calloc(n, sizeof(float));
        for (int i = 0; i < n; ++i) {
            net->steps[i] = atoi(l);
            net->scales[i] = (float)atof(p);
            const char *cl = strchr(l, ','), *cp = strchr(p, ',');
            l = cl ? cl + 1 : l; p = cp ? cp + 1 : p;
        }
        net->num_steps = n;
    } else if (net->policy == EXP) {
        net->gamma = cfg_float(o, "gamma", 1);
    } else if (net->policy == SIG) {
        net->gamma = cfg_float(o, "gamma", 1);
        net->step  = cfg_int(o, "step", 1);
    }
    net->max_batches = cfg_int(o, "max_batches", 0);
}

layer get_network_output_layer(network *net)
{
    int i;
    for (i = net->n - 1; i >= 0; --i) if (net->layers[i].type != COST) break;
    return net->layers[i];
}

network *parse_network_cfg(char *filename)
{
    cfg_file *cfg = cfg_read(filename);
    if (cfg->n == 0) { fprintf(stderr, "Config file has no sections\n"); exit(-1); }
    if (strcmp(cfg->sec[0].type, "[net]") != 0 && strcmp(cfg->sec[0].type, "[network]") != 0) {
        fprintf(stderr, "First section must be [net] or [network]\n");
        exit(-1);
    }
    network_box *nb = calloc(1, sizeof *nb);
    network *net = &nb->pub;
    net->n      = cfg->n - 1;
    net->layers = calloc(net->n ? net->n : 1, sizeof(layer));
    net->seen   = calloc(1, sizeof(size_t));
    net->t      = calloc(1, sizeof(int));
    net->cost   = calloc(1, sizeof(float));
    net->gpu_index = gpu_index;
    read_net_section(&cfg->sec[0], net);

    shape_cursor cur = { net->batch, net->inputs, net->h, net->w, net->c, 0, net };
    size_t workspace = 0;
    fprintf(stderr, "layer     filters    size              input                output\n");
    for (int i = 0; i < net->n; ++i) {
        cfg_section *o = &cfg->sec[i + 1];
        cur.index = i;
        fprintf(stderr, "%5d ", i);
        layer l = {0};
        if (!build_layer(o->type, o, cur, &l)) {
            fprintf(stderr, "Type not recognized: %s\n", o->type);
            fprintf(stderr, "b200-darknet: only the YOLOv1/v2/v3 inference layers are implemented (SURVEY.md §8a)\n");
            exit(-1);
        }
        if (l.type == DROPOUT) {                  /* parser.c:815-817: dropout shares its input's buffer */
            if (i == 0) { fprintf(stderr, "dropout cannot be the first layer\n"); exit(-1); }
            l.output = net->layers[i - 1].output;
        }
        l.clip          = net->clip;
        l.truth         = cfg_int_quiet(o, "truth", 0);
        l.onlyforward   = cfg_int_quiet(o, "onlyforward", 0);
        l.stopbackward  = cfg_int_quiet(o, "stopbackward", 0);
        l.dontsave      = cfg_int_quiet(o, "dontsave", 0);
        l.dontload      = cfg_int_quiet(o, "dontload", 0);
        l.dontloadscales = cfg_int_quiet(o, "dontloadscales", 0);
        l.learning_rate_scale = cfg_float_quiet(o, "learning_rate", 1);
        l.smooth        = cfg_float_quiet(o, "smooth", 0);
        cfg_report_unused(o);
        net->layers[i] = l;
        if (l.workspace_size > workspace) workspace = l.workspace_size;
        cur.h = l.out_h; cur.w = l.out_w; cur.c = l.out_c; cur.inputs = l.outputs;
    }
    cfg_free(cfg);
    layer out = get_network_output_layer(net);
    net->outputs = out.outputs;
    net->truths  = out.outputs;
    if (net->layers[net->n - 1].truths) net->truths = net->layers[net->n - 1].truths;
    net->output  = out.output;
    net->input   = calloc((size_t)net->inputs * net->batch, sizeof(float));
    net->truth   = calloc((size_t)net->truths * net->batch, sizeof(float));
    /* net->workspace (host im2col scratch, parser.c:861-871) has no role here: im2col is never materialised */
    nb->engine = b200_engine_create(net, resolve_precision());
    return net;
}

network *load_network(char *cfg, char *weights, int clear)
{
    network *net = parse_network_cfg(cfg);
    if (weights && weights[0] != 0) load_weights(net, weights);
    if (clear) *net->seen = 0;
    return net;
}

void set_batch_network(network *net, int b)
{
    /* network.c:339-356: only lowers the logical batch; buffers keep their cfg-batch size */
    net->batch = b;
    for (int i = 0; i < net->n; ++i) net->layers[i].batch = b;
}

float *network_predict(network *net, float *input)
{
    b200_engine_forward(b200_engine_of(net), net, input);
    return net->output;
}

int network_width(network *net)  { return net->w; }
int network_height(network *net) { return net->h; }

float *network_predict_image(network *net, image im)
{
    image boxed = letterbox_image(im, net->w, net->h);
    set_batch_network(net, 1);
    float *p = network_predict(net, boxed.data);
    free_image(boxed);
    return p;
}

/* resize_network (network.c:358-438): re-derive every layer's geometry for a new input size, re-allocate the host
 * outputs, and re-plan the device engine (buffers, TMA descriptors, tiling) around the parameters already loaded. */
static float *regrow(float *p, size_t n)
{
    free(p);
    return calloc(n ? n : 1, sizeof(float));
}

int resize_network(network *net, int w, int h)
{
    network_box *nb = (network_box *)net;
    int cw = w, ch = h, cc = net->c;
    /* the reference dies in error() at the first layer it cannot resize (network.c:428), after it has already resized the
     * ones before it; here nothing is touched unless every layer can follow */
    for (int i = 0; i < net->n; ++i) {
        LAYER_TYPE t = net->layers[i].type;
        if (t != CONVOLUTIONAL && t != MAXPOOL && t != UPSAMPLE && t != REORG && t != SHORTCUT && t != ROUTE && t != YOLO &&
            t != REGION && t != DROPOUT && t != AVGPOOL && t != COST) {        /* [softmax]: no branch in the reference either */
            fprintf(stderr, "Cannot resize this type of layer\n");
            return -1;
        }
    }
    b200_engine_unpin_host(nb->engine);            /* the head outputs are page-locked while a plan lives: release before realloc */
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        switch (l->type) {
        case CONVOLUTIONAL:
            l->w = cw; l->h = ch;
            l->out_w = (l->w + 2 * l->pad - l->size) / l->stride + 1;
            l->out_h = (l->h + 2 * l->pad - l->size) / l->stride + 1;
            break;
        case MAXPOOL:
            l->w = cw; l->h = ch;
            l->out_w = (l->w + 2 * l->pad) / l->stride;
            l->out_h = (l->h + 2 * l->pad) / l->stride;
            break;
        case UPSAMPLE:
            l->w = cw; l->h = ch;
            l->out_w = cw * l->stride; l->out_h = ch * l->stride;
            break;
        case REORG:
            l->w = cw; l->h = ch;
            l->out_w = cw / l->stride; l->out_h = ch / l->stride;
            break;
        case SHORTCUT: {
            const layer *src = &net->layers[l->index];
            l->w = src->out_w; l->h = src->out_h;
            l->out_w = cw; l->out_h = ch;
            break;
        }
        case ROUTE: {
            const layer *first = &net->layers[l->input_layers[0]];
            l->out_w = first->out_w; l->out_h = first->out_h; l->out_c = first->out_c;
            l->outputs = 0;
            for (int j = 0; j < l->n; ++j) {
                const layer *in = &net->layers[l->input_layers[j]];
                l->input_sizes[j] = in->outputs;
                l->outputs += in->outputs;
                if (j > 0) {
                    if (in->out_w == first->out_w && in->out_h == first->out_h) l->out_c += in->out_c;
                    else l->out_w = l->out_h = l->out_c = 0;
                }
            }
            l->w = l->out_w; l->h = l->out_h; l->c = l->out_c;
            l->inputs = l->outputs;
            break;
        }
        case YOLO: case REGION:
            l->w = l->out_w = cw; l->h = l->out_h = ch;
            break;
        case DROPOUT:
            l->w = l->out_w = cw; l->h = l->out_h = ch;
            break;
        case AVGPOOL:                                       /* resize_avgpool_layer */
            l->w = cw; l->h = ch;
            break;
        case COST:                                          /* resize_cost_layer */
            l->inputs = l->outputs = net->layers[i - 1].outputs;
            break;
        default:
            fprintf(stderr, "Cannot resize this type of layer\n");      /* network.c:428 (local/connected/detection) */
            return -1;
        }
        if (l->type != ROUTE && l->type != COST) {
            l->inputs = l->w * l->h * l->c;
            l->outputs = l->out_w * l->out_h * l->out_c;
            if (l->type == SHORTCUT) l->inputs = l->outputs;
            if (l->type == DROPOUT) l->inputs = l->outputs = cw * ch * cc;
        }
        if (l->type == DROPOUT) l->output = net->layers[i - 1].output;
        else l->output = regrow(l->output, (size_t)l->batch * l->outputs);
        cw = l->out_w; ch = l->out_h; cc = l->out_c;
    }
    net->w = w; net->h = h;
    net->inputs = w * h * net->c;
    layer out = get_network_output_layer(net);
    net->outputs = out.outputs;
    net->output = out.output;
    net->truths = net->layers[net->n - 1].truths ? net->layers[net->n - 1].truths : out.outputs;      /* network.c:404-406 */
    net->input = regrow(net->input, (size_t)net->inputs * net->batch);
    net->truth = regrow(net->truth, (size_t)net->truths * net->batch);
    nb->engine = b200_engine_recreate(nb->engine, net);
    return 0;
}

void free_layer(layer l) { release_layer_host(l); }

void free_network(network *net)
{
    if (!net) return;
    b200_engine_destroy(b200_engine_of(net));
    for (int i = 0; i < net->n; ++i) release_layer_host(net->layers[i]);
    free(net->layers);
    free(net->input); free(net->truth);
    free(net->seen); free(net->t); free(net->cost);
    free(net->steps); free(net->scales);
    free(net);
}

/* ---- small accessors for foreign-function callers that do not want to mirror the 1160-byte layer struct ---- */
int b200_network_layers(const network *net) { return net->n; }

int b200_layer_info(const network *net, int i, int *out)
{
    if (i < 0 || i >= net->n) return -1;
    const layer *l = &net->layers[i];
    int v[20] = { (int)l->type, l->batch, l->inputs, l->outputs, l->h, l->w, l->c, l->out_h, l->out_w, l->out_c,
                  l->n, l->size, l->stride, l->pad, l->classes, l->coords, l->batch_normalize, (int)l->activation,
                  l->nweights, l->index };
    memcpy(out, v, sizeof v);
    return 20;
}

float *b200_layer_output_host(const network *net, int i) { return (i < 0 || i >= net->n) ? NULL : net->layers[i].output; }
