/*
 * darknet.h — public C ABI of the B200-native YOLO inference engine.
 *
 * This header is the DROP-IN BOUNDARY (SURVEY.md §8b).  It freezes the data model that darknet
 * drivers and the ctypes wrapper see when the reference is built with GPU undefined
 * (reference: Darknet2Tensorflow/darknet-master/include/darknet.h — `layer` :118-421, `network` :429-495,
 * `image` :507-512, `box` :514-516, `detection` :518-525, enums :56-94), so that existing
 * .cfg/.weights drivers compile and link against this library unchanged.  Field ORDER and TYPES are
 * the ABI and therefore identical to the reference (sizeof(layer)=1160, sizeof(network)=272 on
 * x86-64; checked by tests/test_abi_layout.py); everything behind the structs is new.
 *
 * Only the inference path is implemented (SURVEY.md §8a).  Training-only fields exist for layout
 * compatibility and are left zero.  All device state lives in an opaque engine object owned by the
 * `network` (see include/b200_engine.h), never inside `layer`.
 */
#ifndef DARKNET_API
#define DARKNET_API
#include <stdlib.h>
#include <stdio.h>
#include <string.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SECRET_NUM -1234
extern int gpu_index;                       /* reference darknet.h:9 — device ordinal used by new networks */

/* ---- small public records ------------------------------------------------------------------ */
typedef struct { int classes; char **names; } metadata;                    /* ref :35-38 */

typedef struct {                                                             /* ref :42-53 (YOLO9000 WordTree: read_tree, [region] tree=) */
    int *leaf; int n; int *parent; int *child; int *group; char **name;
    int groups; int *group_size; int *group_offset;
} tree;

typedef enum { LOGISTIC, RELU, RELIE, LINEAR, RAMP, TANH, PLSE, LEAKY, ELU, LOGGY, STAIR, HARDTAN, LHTAN } ACTIVATION;
typedef enum { MULT, ADD, SUB, DIV } BINARY_ACTIVATION;
typedef enum {
    CONVOLUTIONAL, DECONVOLUTIONAL, CONNECTED, MAXPOOL, SOFTMAX, DETECTION, DROPOUT, CROP, ROUTE, COST,
    NORMALIZATION, AVGPOOL, LOCAL, SHORTCUT, ACTIVE, RNN, GRU, LSTM, CRNN, BATCHNORM, NETWORK, XNOR,
    REGION, YOLO, REORG, UPSAMPLE, LOGXENT, L2NORM, BLANK
} LAYER_TYPE;
typedef enum { SSE, MASKED, L1, SEG, SMOOTH, WGAN } COST_TYPE;

typedef struct {
    int batch; float learning_rate, momentum, decay; int adam; float B1, B2, eps; int t;
} update_args;

struct network; typedef struct network network;
struct layer;   typedef struct layer layer;

/* ---- layer: one record per cfg section (ABI-frozen order) ------------------------------------ */
struct layer {
    LAYER_TYPE type; ACTIVATION activation; COST_TYPE cost_type;
    void (*forward)(struct layer, struct network);          /* set to a stub: layers run on the device engine */
    void (*backward)(struct layer, struct network);
    void (*update)(struct layer, update_args);
    void (*forward_gpu)(struct layer, struct network);
    void (*backward_gpu)(struct layer, struct network);
    void (*update_gpu)(struct layer, update_args);
    /* geometry + flags */
    int batch_normalize, shortcut, batch, forced, flipped, inputs, outputs, nweights, nbiases, extra, truths;
    int h, w, c, out_h, out_w, out_c, n, max_boxes, groups, size, side, stride, reverse, flatten, spatial, pad;
    int sqrt, flip, index, binary, xnor, steps, hidden, truth;
    float smooth, dot, angle, jitter, saturation, exposure, shift, ratio, learning_rate_scale, clip;
    int softmax, classes, coords, background, rescore, objectness, joint, noadjust, reorg, log, tanh;
    int *mask; int total;
    float alpha, beta, kappa;
    float coord_scale, object_scale, noobject_scale, mask_scale, class_scale;
    int bias_match, random; float ignore_thresh, truth_thresh, thresh, focus; int classfix, absolute;
    int onlyforward, stopbackward, dontload, dontsave, dontloadscales;
    float temperature, probability, scale;
    /* host buffers (fp32, NCHW, batch-major) */
    char *cweights; int *indexes, *input_layers, *input_sizes, *map;
    float *rand, *cost, *state, *prev_state, *forgot_state, *forgot_delta, *state_delta, *combine_cpu, *combine_delta_cpu;
    float *concat, *concat_delta;
    float *binary_weights;
    float *biases, *bias_updates;
    float *scales, *scale_updates;
    float *weights, *weight_updates;
    float *delta, *output, *loss, *squared, *norms;
    float *spatial_mean, *mean, *variance;
    float *mean_delta, *variance_delta;
    float *rolling_mean, *rolling_variance;
    float *x, *x_norm;
    float *m, *v;
    float *bias_m, *bias_v, *scale_m, *scale_v;
    float *z_cpu, *r_cpu, *h_cpu, *prev_state_cpu;
    float *temp_cpu, *temp2_cpu, *temp3_cpu;
    float *dh_cpu, *hh_cpu, *prev_cell_cpu, *cell_cpu, *f_cpu, *i_cpu, *g_cpu, *o_cpu, *c_cpu, *dc_cpu;
    float *binary_input;
    /* recurrent sub-layers (never instantiated by YOLO cfgs) */
    struct layer *input_layer, *self_layer, *output_layer;
    struct layer *reset_layer, *update_layer, *state_layer;
    struct layer *input_gate_layer, *state_gate_layer, *input_save_layer, *state_save_layer, *input_state_layer, *state_state_layer;
    struct layer *input_z_layer, *state_z_layer;
    struct layer *input_r_layer, *state_r_layer;
    struct layer *input_h_layer, *state_h_layer;
    struct layer *wz, *uz, *wr, *ur, *wh, *uh, *uo, *wo, *uf, *wf, *ui, *wi, *ug, *wg;
    tree *softmax_tree;
    size_t workspace_size;
};

typedef enum { CONSTANT, STEP, EXP, POLY, STEPS, SIG, RANDOM } learning_rate_policy;

/* ---- network (ABI-frozen order) ---------------------------------------------------------------- */
struct network {
    int n, batch; size_t *seen; int *t; float epoch; int subdivisions;
    layer *layers; float *output; learning_rate_policy policy;
    float learning_rate, momentum, decay, gamma, scale, power;
    int time_steps, step, max_batches; float *scales; int *steps; int num_steps, burn_in;
    int adam; float B1, B2, eps;
    int inputs, outputs, truths, notruth, h, w, c, max_crop, min_crop;
    float max_ratio, min_ratio; int center; float angle, aspect, exposure, saturation, hue; int random;
    int gpu_index; tree *hierarchy;
    float *input, *truth, *delta, *workspace; int train, index; float *cost; float clip;
};

typedef struct { int w, h, c; float *data; } image;                        /* ref :507-512, fp32 CHW in [0,1] */
typedef struct { float x, y, w, h; } box;                                   /* ref :514-516, centre + size     */
typedef struct detection {                                                   /* ref :518-525, 48 bytes          */
    box bbox; int classes; float *prob; float *mask; float objectness; int sort_class;
} detection;

/* ---- hot path (BASELINE north star) -------------------------------------------------------------- */
network   *parse_network_cfg(char *filename);                               /* ref darknet.h:680  parser.c:730   */
void       load_weights(network *net, char *filename);                      /* ref :682           parser.c:1347  */
void       load_weights_upto(network *net, char *filename, int start, int cutoff); /* ref :684    parser.c:1241  */
network   *load_network(char *cfg, char *weights, int clear);               /* ref :586           network.c:53   */
float     *network_predict(network *net, float *input);                     /* ref :739           network.c:497  */
detection *get_network_boxes(network *net, int w, int h, float thresh, float hier, int *map, int relative, int *num); /* ref :745 network.c:562 */
detection *make_network_boxes(network *net, float thresh, int *num);        /* network.c:526 */
void       fill_network_boxes(network *net, int w, int h, float thresh, float hier, int *map, int relative, detection *dets); /* network.c:542 */
int        num_detections(network *net, float thresh);                      /* network.c:510 */
void       do_nms_sort(detection *dets, int total, int classes, float thresh); /* ref :752        box.c:58       */
void       do_nms_obj(detection *dets, int total, int classes, float thresh);  /* ref :751        box.c:21       */
void       free_detections(detection *dets, int n);                         /* ref :746           network.c:569  */

/* ---- lifetime + accessors the drivers use -------------------------------------------------------- */
void   set_batch_network(network *net, int b);                              /* ref :690  network.c:339 */
void   free_network(network *net);                                          /* ref :689  network.c:716 */
void   free_layer(layer l);                                                 /* layer.c:6 */
int    network_width(network *net);                                         /* ref :741 */
int    network_height(network *net);                                        /* ref :742 */
layer  get_network_output_layer(network *net);                              /* ref :717  network.c:699 */
float *network_predict_image(network *net, image im);                       /* ref :743  network.c:579 */
int    resize_network(network *net, int w, int h);                          /* ref :704  network.c:358 (re-plans the device engine) */
void   cuda_set_device(int n);                                              /* ref :631  cuda.c:13,176 */
double what_time_is_it_now(void);                                           /* utils.c:27 */

/* ---- host image helpers used immediately before the path (plain C re-statements; SURVEY §8f-1) --- */
image  make_image(int w, int h, int c);
void   free_image(image m);
image  resize_image(image im, int w, int h);                                /* image.c:1347 */
image  letterbox_image(image im, int w, int h);                             /* image.c:960  */
float  box_iou(box a, box b);                                               /* box.c:179    */
image  load_image_color(char *filename, int w, int h);                      /* image.c:1482 (binary PPM/PGM only here) */
void   rgbgr_image(image im);
metadata get_metadata(char *file);                                          /* option_list.c:35 */
void   free_ptrs(void **ptrs, int n);
void   reset_rnn(network *net);

/* ---- what examples/detector.c, yolo.c and darknet.c call around the path (host C, csrc/host/drivers.c) ------------ */
typedef struct node { void *val; struct node *next; struct node *prev; } node;     /* ref :591-595 */
typedef struct list { int size; node *front; node *back; } list;                   /* ref :597-601 */
list  *make_list(void);                                                     /* list.c:5    */
void   list_insert(list *l, void *val);                                     /* list.c:42   */
void   free_list(list *l);                                                  /* ref :778    */
void **list_to_array(list *l);                                              /* ref :772    */
list  *read_data_cfg(char *filename);                                       /* ref :604  option_list.c:7   */
char  *option_find(list *l, char *key);                                     /* option_list.c:91            */
char  *option_find_str(list *l, char *key, char *def);                      /* ref :676  option_list.c:105 */
int    option_find_int(list *l, char *key, int def);                        /* ref :677  option_list.c:113 */
int    option_find_int_quiet(list *l, char *key, int def);                  /* ref :678  option_list.c:121 */
float  option_find_float(list *l, char *key, float def);                    /* option_list.c:135           */
float  option_find_float_quiet(list *l, char *key, float def);              /* option_list.c:128           */
void   option_unused(list *l);                                              /* option_list.c:79            */
list  *get_paths(char *filename);                                           /* ref :762  data.c:12         */
char **get_labels(char *filename);                                          /* ref :750  data.c:618        */
int   *read_map(char *filename);                                            /* ref :774  utils.c:62        */
tree  *read_tree(char *filename);                                           /* tree.c:83  (YOLO9000 WordTree, `tree=` of [region]) */
void   hierarchy_predictions(float *predictions, int n, tree *hier, int only_leaves, int stride);   /* ref :763  tree.c:37 */
int    hierarchy_top_prediction(float *predictions, tree *hier, float thresh, int stride);          /* tree.c:53 */
int    find_arg(int argc, char *argv[], char *arg);                         /* ref :768  utils.c:120       */
int    find_int_arg(int argc, char **argv, char *arg, int def);             /* ref :766  utils.c:133       */
float  find_float_arg(int argc, char **argv, char *arg, float def);         /* ref :767  utils.c:148       */
char  *find_char_arg(int argc, char **argv, char *arg, char *def);          /* ref :769  utils.c:163       */
void   top_k(float *a, int n, int k, int *index);                          /* utils.c top_k               */
char  *basecfg(char *cfgfile);                                              /* ref :770  utils.c:179       */
char  *fgetl(FILE *fp);                                                     /* ref :773  utils.c:335       */
void   strip(char *s);                                                      /* ref :774  utils.c:302       */
image  copy_image(image p);                                                 /* ref :712  */
image **load_alphabet(void);                                                /* ref :737  image.c:223 (data/labels/<char>_<size>.png holding PNM data) */
image  get_label(image **characters, char *string, int size);               /* ref :638  image.c:132 */
void   draw_label(image a, int r, int c, image label, const float *rgb);    /* ref :639  image.c:149 */
void   draw_box(image a, int x1, int y1, int x2, int y2, float r, float g, float b);             /* image.c:166 */
void   draw_box_width(image a, int x1, int y1, int x2, int y2, int w, float r, float g, float b); /* ref :713  image.c:202 */
float  get_color(int c, int x, int max);                                    /* image.c:17  */
void   draw_detections(image im, detection *dets, int num, float thresh, char **names, image **alphabet, int classes); /* ref :734 image.c:239 */
void   save_image(image im, const char *name);                              /* ref :707  image.c:713 (CPU build: <name>.png) */
void   save_image_png(image im, const char *name);                          /* ref :640  image.c:696 */

#ifdef __cplusplus
}
#endif
#endif
