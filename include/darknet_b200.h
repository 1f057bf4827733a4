/*
 * darknet_b200.h — the reference's C API for the YOLOv2 detection forward pass,
 * re-implemented on hand-written sm_100a kernels (libyolo2_b200.so).
 *
 * Source-level drop-in for the callers of SURVEY.md section 8b: a caller written against the
 * reference headers (network.h, parser.h, region_layer.h, box.h, cuda.h, option_list.h,
 * tree.h, utils.h under /root/reference/src_yolo2) recompiles against this single header.
 * Names, argument meaning, by-value struct passing, ownership and error behaviour follow the
 * reference; each declaration cites the interface it replaces.  Struct layouts are NOT
 * binary-compatible with a reference build (training-only fields are dropped, device state
 * lives behind `network.b200`).
 *
 * There is no CPU execution path: with gpu_index < 0 parse_network_cfg only builds the host
 * description (shapes, weights), and network_predict aborts through error().
 */
#ifndef DARKNET_B200_H
#define DARKNET_B200_H

#include <stddef.h>
#include <stdio.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- activations.h:6-8 ------------------------------------------------------------ */
typedef enum {
    LOGISTIC, RELU, RELIE, LINEAR, RAMP, TANH, PLSE, LEAKY, ELU, LOGGY, STAIR, HARDTAN, LHTAN
} ACTIVATION;
ACTIVATION get_activation(char *s);          /* activations.c:45-62 */
char *get_activation_string(ACTIVATION a);   /* activations.c:9-43 */

/* ---- layer.h:13-42 ---------------------------------------------------------------- */
typedef enum {
    CONVOLUTIONAL, DECONVOLUTIONAL, CONNECTED, MAXPOOL, SOFTMAX, DETECTION, DROPOUT, CROP,
    ROUTE, COST, NORMALIZATION, AVGPOOL, LOCAL, SHORTCUT, ACTIVE, RNN, GRU, CRNN, BATCHNORM,
    NETWORK, XNOR, REGION, REORG, BLANK
} LAYER_TYPE;
typedef enum { SSE, MASKED, SMOOTH } COST_TYPE;

/* ---- tree.h:4-14 ------------------------------------------------------------------- */
typedef struct {
    int *leaf;
    int n;
    int *parent;
    int *group;
    char **name;
    int groups;
    int *group_size;
    int *group_offset;
} tree;
tree *read_tree(char *filename);                                                   /* tree.c:53-103 */
void hierarchy_predictions(float *predictions, int n, tree *hier, int only_leaves); /* tree.c:37-51 */
float get_hierarchy_probability(float *x, tree *hier, int c);                      /* tree.c:26-35 */

/* ---- box.h:4-6 ---------------------------------------------------------------------- */
typedef struct { float x, y, w, h; } box;

struct network_state;
struct layer;
typedef struct layer layer;

/* ---- layer.h:44-264 (inference subset; same field names) ---------------------------- */
struct layer {
    LAYER_TYPE type;
    ACTIVATION activation;
    COST_TYPE cost_type;
    void (*forward)(struct layer, struct network_state);      /* aborts: no CPU path */
    void (*forward_gpu)(struct layer, struct network_state);
    int batch_normalize;
    int batch;
    int flipped;
    int inputs, outputs;
    int h, w, c;
    int out_h, out_w, out_c;
    int n;            /* filters (conv) / anchors (region) / inputs (route) */
    int groups;
    int size, stride, pad, reverse;
    int index;        /* shortcut source */
    int binary, xnor;
    int softmax, classes, coords;
    int max_boxes, log, sqrt, rescore, bias_match, random, absolute, classfix;
    float jitter, thresh;
    float coord_scale, object_scale, noobject_scale, class_scale;
    float temperature, dot;
    int dontload, dontloadscales;
    int adam;         /* [net] adam=1: the .weights file carries m and v behind every filter bank */
    tree *softmax_tree;
    int *map;
    float *cost;
    /* host parameter arrays, exactly as load_weights fills them (parser.c:963-1006) */
    float *biases;
    float *scales;
    float *weights;
    float *rolling_mean;
    float *rolling_variance;
    float *m, *v;     /* adam moments, only stored and re-saved (parser.c:788-791, 992-995) */
    int *input_layers;
    int *input_sizes;
    /* host activations, fp32 NCHW (REGION: flattened [hw][n][5+classes]).  Always present for
     * the network's output layer; for other layers it is filled on demand by
     * get_network_output_layer(). */
    float *output;
    size_t workspace_size;
    /* device side (opaque layouts, see yolo2_b200_kernels.h) */
    float *output_gpu;
    float *weights_gpu;
    float *biases_gpu;
    float *scales_gpu;
    void *b200;       /* per-layer plan */
};
void free_layer(layer);                                                            /* layer.c:5-96 */

/* ---- network.h:19-77 ---------------------------------------------------------------- */
typedef enum { CONSTANT, STEP, EXP, POLY, STEPS, SIG, RANDOM } learning_rate_policy;

typedef struct network {
    float *workspace;
    int n;
    int batch;
    int *seen;
    float epoch;
    int subdivisions;
    float momentum, decay;
    layer *layers;
    int outputs;
    float *output;
    learning_rate_policy policy;
    float learning_rate, gamma, scale, power;
    int time_steps, step, max_batches;
    float *scales;
    int *steps;
    int num_steps, burn_in;
    int adam;
    float B1, B2, eps;
    int inputs;
    int h, w, c;
    int max_crop, min_crop;
    float angle, aspect, exposure, saturation, hue;
    int gpu_index;
    tree *hierarchy;
    float **input_gpu;
    float **truth_gpu;
    void *b200;       /* device arena, stream, layer schedule, CUDA graph */
} network;

typedef struct network_state {
    float *truth;
    float *input;
    float *delta;
    float *workspace;
    int train;
    int index;
    network net;
} network_state;

/* ---- cuda.h:8,22-32 / cuda.c:1-158 --------------------------------------------------- */
extern int gpu_index;
#define BLOCK 512
void cuda_set_device(int n);
int cuda_get_device(void);
void check_error_code(int status, const char *what); /* y2 status codes: print, abort */
void check_error(int cuda_status);                   /* cuda.c:27-49; the argument is a cudaError_t */
/* layout-identical to CUDA's dim3 (three unsigned ints, returned by value) so this header needs no
 * CUDA include; cuda.c:51-62 */
typedef struct { unsigned int x, y, z; } y2_dim3;
y2_dim3 cuda_gridsize(size_t n);
float *cuda_make_array(float *x, size_t n);
int *cuda_make_int_array(size_t n);
void cuda_push_array(float *x_gpu, float *x, size_t n);
void cuda_pull_array(float *x_gpu, float *x, size_t n);
void cuda_free(float *x_gpu);

/* ---- parser.h:5-11 -------------------------------------------------------------------- */
network parse_network_cfg(char *filename);                         /* parser.c:585-700 */
void load_weights(network *net, char *filename);                   /* parser.c:1084-1087 */
void load_weights_upto(network *net, char *filename, int cutoff);  /* parser.c:1009-1082 */
void save_weights(network net, char *filename);                    /* parser.c:879-882 */
void save_weights_upto(network net, char *filename, int cutoff);   /* parser.c:822-878 */

/* ---- network.h:79-131 ------------------------------------------------------------------ */
network make_network(int n);                                       /* network.c:132-143 */
void free_network(network net);                                    /* network.c:592-609 */
float *network_predict(network net, float *input);                 /* network.c:458-474 */
float *network_predict_gpu(network net, float *input);             /* network_kernels.cu:392-407 */
void forward_network(network net, network_state state);            /* network.c:145-158: aborts */
void forward_network_gpu(network net, network_state state);        /* network_kernels.cu:43-56 */
float *get_network_output(network net);                            /* network.c:173-181 */
float *get_network_output_gpu(network net);                        /* network_kernels.cu:378-390 */
float *get_network_output_layer(network net, int i);               /* network.c:466 */
float *get_network_output_gpu_layer(network net, int i);          /* the name network.h:84 declares ... */
float *get_network_output_layer_gpu(network net, int i);          /* ... and the one network_kernels.cu:378 defines */
int get_network_output_size(network net);                          /* network.c:167-171 */
int get_network_output_size_layer(network net, int i);
int get_network_input_size(network net);
void set_batch_network(network *net, int b);                       /* network.c:308-320 */
int resize_network(network *net, int w, int h);                    /* network.c:322-388 */
char *get_layer_string(LAYER_TYPE a);                              /* network.c:77-130 */

/* ---- per-layer API (convolutional_layer.h:13-37, maxpool_layer.h:12-20, reorg_layer.h:9-17,
 * route_layer.h:8-16, region_layer.h:9-18, shortcut_layer.h, avgpool_layer.h, softmax_layer.h,
 * cost_layer.h).  make_* build the host-side layer (extents, host weight arrays, forward_gpu pointer);
 * the device side is planned per network by parse_network_cfg / resize_network / set_batch_network.
 * forward_*_layer_gpu are the l.forward_gpu targets.  The CPU forwards (forward_*_layer) are not
 * exported: this library has no CPU execution path (l.forward aborts with a message). -------------- */
typedef layer convolutional_layer;
typedef layer maxpool_layer;
typedef layer route_layer;
typedef layer region_layer;
typedef layer avgpool_layer;
typedef layer softmax_layer;
typedef layer cost_layer;
layer make_convolutional_layer(int batch, int h, int w, int c, int n, int size, int stride, int padding,
                               ACTIVATION activation, int batch_normalize, int binary, int xnor,
                               int adam);                          /* convolutional_layer.c:166-287 */
layer make_maxpool_layer(int batch, int h, int w, int c, int size, int stride, int padding); /* maxpool_layer.c:20-57 */
layer make_reorg_layer(int batch, int w, int h, int c, int stride, int reverse);   /* reorg_layer.c:7-49 */
layer make_route_layer(int batch, int n, int *input_layers, int *input_sizes);     /* route_layer.c:6-37 */
layer make_region_layer(int batch, int w, int h, int n, int classes, int coords);  /* region_layer.c:14-53 */
layer make_shortcut_layer(int batch, int index, int w, int h, int c, int w2, int h2, int c2); /* shortcut_layer.c:7-37 */
layer make_avgpool_layer(int batch, int w, int h, int c);                          /* avgpool_layer.c:5-30 */
layer make_softmax_layer(int batch, int inputs, int groups);                       /* softmax_layer.c:11-33 */
layer make_cost_layer(int batch, int inputs, COST_TYPE type, float scale);         /* cost_layer.c:36-60 */
layer make_connected_layer(int batch, int inputs, int outputs, ACTIVATION activation,
                           int batch_normalize);                                   /* connected_layer.c:13-100 */
layer make_dropout_layer(int batch, int inputs, float probability);                /* dropout_layer.c:7-26 */
void forward_connected_layer_gpu(layer l, network_state state);      /* connected_layer.c:271-293 */
void forward_dropout_layer_gpu(layer l, network_state state);        /* dropout_layer_kernels.cu: identity at inference */
void forward_convolutional_layer_gpu(layer l, network_state state);  /* convolutional_kernels.cu:77-131 */
void forward_maxpool_layer_gpu(layer l, network_state state);        /* maxpool_layer_kernels.cu:86-100 */
void forward_reorg_layer_gpu(layer l, network_state state);          /* reorg_layer.c:97-104 */
void forward_route_layer_gpu(layer l, network_state state);          /* route_layer.c:104-117 */
void forward_shortcut_layer_gpu(layer l, network_state state);       /* shortcut_layer.c:54-59 */
void forward_avgpool_layer_gpu(layer l, network_state state);        /* avgpool_layer_kernels.cu:46-54 */
void forward_softmax_layer_gpu(layer l, network_state state);        /* softmax_layer.c:77-96 */
void forward_cost_layer_gpu(layer l, network_state state);           /* cost_layer.c:118-140 */
void resize_convolutional_layer(convolutional_layer *l, int w, int h); /* convolutional_layer.c:343-399 */
void resize_maxpool_layer(maxpool_layer *l, int w, int h);           /* maxpool_layer.c:59-77 */
void resize_reorg_layer(layer *l, int w, int h);                     /* reorg_layer.c:51-76 */
void resize_route_layer(route_layer *l, network *net);               /* route_layer.c:39-71 */
void resize_region_layer(layer *l, int w, int h);                    /* region_layer.c:55-71 */
void resize_avgpool_layer(avgpool_layer *l, int w, int h);           /* avgpool_layer.c:32-37 */

/* ---- blas.h:16-19,43-53, activations.h:16-18: vector helpers on host arrays and on
 * cuda_make_array buffers (fp32).  gemm_ongpu / gemm_gpu / im2col_ongpu are plain fp32 device kernels for callers of
 * the helper surface; gemm, gemm_cpu, im2col_cpu and blas_handle are NOT provided: the convolution
 * is an implicit GEMM inside the tcgen05 kernels (INTEGRATION.md). ----------------------------------- */
void fill_cpu(int N, float ALPHA, float *X, int INCX);
void copy_cpu(int N, float *X, int INCX, float *Y, int INCY);
void axpy_cpu(int N, float ALPHA, float *X, int INCX, float *Y, int INCY);
void scal_cpu(int N, float ALPHA, float *X, int INCX);
void fill_ongpu(int N, float ALPHA, float *X, int INCX);
void copy_ongpu(int N, float *X, int INCX, float *Y, int INCY);
void copy_ongpu_offset(int N, float *X, int OFFX, int INCX, float *Y, int OFFY, int INCY);
void axpy_ongpu(int N, float ALPHA, float *X, int INCX, float *Y, int INCY);
void axpy_ongpu_offset(int N, float ALPHA, float *X, int OFFX, int INCX, float *Y, int OFFY, int INCY);
void scal_ongpu(int N, float ALPHA, float *X, int INCX);
float activate(float x, ACTIVATION a);                              /* activations.c:64-93 */
void activate_array(float *x, const int n, const ACTIVATION a);     /* activations.c:95-101 */
void activate_array_ongpu(float *x, int n, ACTIVATION a);           /* activation_kernels.cu:143-159 */
void gemm_ongpu(int TA, int TB, int M, int N, int K, float ALPHA, float *A_gpu, int lda, float *B_gpu, int ldb,
                float BETA, float *C_gpu, int ldc);                 /* gemm.c:173-183 */
void gemm_gpu(int TA, int TB, int M, int N, int K, float ALPHA, float *A, int lda, float *B, int ldb, float BETA,
              float *C, int ldc);                                   /* gemm.c:185-213 */
void im2col_ongpu(float *im, int channels, int height, int width, int ksize, int stride, int pad,
                  float *data_col);                                 /* im2col_kernels.cu:48-61 */

/* ---- region_layer.h:9-18, box.h:12-20 -------------------------------------------------- */
void forward_region_layer_gpu(const layer l, network_state state); /* region_layer.c:383-422 */
void get_region_boxes(layer l, int w, int h, float thresh, float **probs, box *boxes,
                      int only_objectness, int *map);              /* region_layer.c:328-379 */
void do_nms_sort(box *boxes, float **probs, int total, int classes, float thresh); /* box.c:249-277 */
void do_nms(box *boxes, float **probs, int total, int classes, float thresh);      /* box.c:279-297 */
float box_iou(box a, box b);                                       /* box.c:94-97 */
float box_intersection(box a, box b);
float box_union(box a, box b);

/* ---- detector.c:202-369: validation result writers (VOC per-class files, COCO json, ImageNet-detection) --- */
void validate_detector(char *datacfg, char *cfgfile, char *weightfile);            /* detector.c:244-369 */
void validate_detector_recall(char *datacfg, char *cfgfile, char *weightfile);     /* detector.c:371-450 */
typedef struct {                                                                   /* data.h:69-73 */
    int id;
    float x, y, w, h;
    float left, right, top, bottom;
} box_label;
box_label *read_boxes(char *filename, int *n);                                     /* data.c:135-159 */
void find_replace(char *str, char *orig, char *rep, char *output);                 /* utils.c:158-172 */
void print_detector_detections(FILE **fps, char *id, box *boxes, float **probs, int total, int classes, int w,
                               int h);                                             /* detector.c:202-221 */
void print_imagenet_detections(FILE *fp, int id, box *boxes, float **probs, int total, int classes, int w,
                               int h);                                             /* detector.c:223-242 */

/* ---- demo.c:57-230: the fetch / detect video pipeline, fed and drained by callbacks (the reference is wired to an
 * OpenCV capture and window).  source fills one uint8 interleaved RGB frame at the network's size and returns 0 at the
 * end of the stream; sink receives, per frame and in stream order, what detect_in_thread hands to the drawing code:
 * boxes[total], probs[total][classes] after the 3-frame mean, get_region_boxes and do_nms(.4). ---------------------- */
typedef int (*y2_frame_source)(void *ctx, unsigned char *rgb_hwc, int w, int h);
typedef void (*y2_detection_sink)(void *ctx, int frame, box *boxes, float **probs, int total, int classes);
int demo_frames(char *cfgfile, char *weightfile, float thresh, y2_frame_source source, void *source_ctx,
                y2_detection_sink sink, void *sink_ctx);

/* ---- option_list.h:12-21, list.h, utils.h --------------------------------------------- */
typedef struct node { void *val; struct node *next; struct node *prev; } node;
typedef struct list { int size; node *front; node *back; } list;
list *make_list(void);
void list_insert(list *, void *);
void free_list(list *l);
void free_list_contents(list *l);
void **list_to_array(list *l);

list *get_paths(char *filename);                                   /* data.c:12-23 */
list *read_data_cfg(char *filename);                               /* option_list.c:7-33 */
int read_option(char *s, list *options);                           /* option_list.c:35-51 */
void option_insert(list *l, char *key, char *val);
char *option_find(list *l, char *key);
char *option_find_str(list *l, char *key, char *def);
int option_find_int(list *l, char *key, int def);
int option_find_int_quiet(list *l, char *key, int def);
float option_find_float(list *l, char *key, float def);
float option_find_float_quiet(list *l, char *key, float def);
void option_unused(list *l);

void error(const char *s);                                         /* utils.c:195-200 */
void file_error(char *s);                                          /* utils.c:208-213 */
char *fgetl(FILE *fp);                                             /* utils.c:263-293 */
void strip(char *s);                                               /* utils.c:230-241 */
int *read_map(char *filename);                                     /* utils.c:17-33 */
int max_index(float *a, int n);                                    /* utils.c:533-545 */
void mean_arrays(float **a, int n, int els, float *avg);           /* utils.c:420-433 */
char *basecfg(char *cfgfile);                                      /* utils.c:136-153 */
char **get_labels(char *filename);                                 /* data.c:474-480 */
int find_arg(int argc, char *argv[], char *arg);
int find_int_arg(int argc, char **argv, char *arg, int def);
float find_float_arg(int argc, char **argv, char *arg, float def);
char *find_char_arg(int argc, char **argv, char *arg, char *def);

/* ---- image.h (the two calls Detector::detect needs) ------------------------------------ */
typedef struct { int h, w, c; float *data; } image;
image make_image(int w, int h, int c);                             /* image.c:1436-1441 */
void free_image(image m);
image resize_image(image im, int w, int h);                        /* image.c:1950-1993 */
/* binary PPM / PGM reader in place of the reference's stb_image decoder: `c` planes of byte / 255., then the
 * optional resize (image.c:2069-2095) */
image load_image(char *filename, int w, int h, int c);
image load_image_color(char *filename, int w, int h);
/* classifier front end (classifier.c:676-730 predict_classifier) */
void fill_image(image m, float s);                                 /* image.c:1601-1605 */
void embed_image(image source, image dest, int dx, int dy);        /* image.c:1087-1098 */
image letterbox_image(image im, int w, int h);                     /* image.c:1624-1644 */
void top_k(float *a, int n, int k, int *index);                    /* utils.c:179-193 */
/* classifier.c:676-730: classify an image file (letterbox, forward, WordTree products, top-k) */
void predict_classifier(char *datacfg, char *cfgfile, char *weightfile, char *filename, int top);
void predict_classifier_image(network net, image im, char **names, int top, FILE *out); /* the lines for one image */

/* =========================================================================================
 * B200 extensions (not in the reference): batched, device-resident detection and classification.
 * ========================================================================================= */

typedef struct y2_detection {
    float x, y, w, h;   /* centre/size in relative units, as `box` */
    float prob;
    int obj_id;
    int box_index;      /* cell-major, anchor-minor index, as probs[] rows */
} y2_detection;

/* Upload `batch` images (fp32 planar CHW, [0,1]) into the network's device input buffer. */
void network_upload_input(network net, const float *input);
/* Pinned host staging buffer ([batch][c][h][w] fp32) that network_upload_input copies from;
 * fill it directly and pass it (or NULL) to network_upload_input to skip the extra host copy. */
float *network_input_staging(network net);
/* Device address of that input buffer (fp32 [batch][c][h][w]), e.g. for a caller that decodes on the GPU. */
float *network_input_device(network net);
/* Forward pass on the already-uploaded input; nothing is copied back. */
void network_forward_device(network net);
/* Region decode + NMS + final pick on the device for every image of the batch; copies only
 * the compact per-image detection lists back.  dets: [batch][max_det], counts: [batch]. */
void network_detect_device(network net, float thresh, float nms, y2_detection *dets, int *counts,
                           int max_det);
/* upload + forward + detect, one synchronisation */
void network_detect_batch(network net, const float *input, float thresh, float nms,
                          y2_detection *dets, int *counts, int max_det);
/* Two-deep pipeline over the same work: network_detect_submit queues the H2D copy of a batch on a
 * copy stream and its forward + decode + NMS + D2H behind it on the network's stream, then returns;
 * network_detect_wait blocks for the OLDEST submitted batch and hands out its detections.  With two
 * batches in flight the upload of batch i+1 overlaps the forward pass of batch i.  Both return the
 * slot (0/1) the batch used.  network_pipeline_staging(net, slot) is the slot's pinned input buffer
 * (slots alternate 0,1,0,... starting at the oldest free one); passing any other pointer costs a
 * host-side copy into it.  Not to be mixed with the synchronous calls while batches are in flight. */
float *network_pipeline_staging(network net, int slot);
int network_pipeline_next_slot(network net); /* slot the next network_detect_submit will use */
int network_detect_submit(network net, const float *input, float thresh, float nms, int max_det);
int network_detect_wait(network net, y2_detection *dets, int *counts, int max_det);
/* the same with the batch already resident in the slot's DEVICE input (fp32 planar, written there by the caller -
 * another kernel, a peer copy, one upload for many passes): no host -> device copy at all */
float *network_pipeline_input_device(network net, int slot);
int network_detect_submit_resident(network net, float thresh, float nms, int max_det);
/* The same calls fed with raw decoded images: uint8 interleaved RGB [batch][h][w][3] at the network's
 * resolution.  Each byte becomes (float)(byte / 255.) on the device exactly as the reference's loaders
 * do on the host (yolo_v2_class.cpp:129-149 load_image_stb; yolo_v2_class.hpp mat_to_image), so the
 * detections are identical to the float calls on the converted image, at a quarter of the upload.
 * Needs a network whose first layer is the fused first-layer kernel (all north-star detector cfgs) and
 * a width that is a multiple of 16. */
unsigned char *network_pipeline_staging_u8(network net, int slot);
int network_detect_submit_u8(network net, const unsigned char *input_hwc, float thresh, float nms, int max_det);
void network_detect_batch_u8(network net, const unsigned char *input_hwc, float thresh, float nms,
                             y2_detection *dets, int *counts, int max_det);
/* Decoded frames of ANY size, uint8 interleaved RGB [batch][frame_h][frame_w][3]: the bytes are
 * uploaded as they are and both load_image_stb's byte/255. (yolo_v2_class.cpp:129-149) and resize_image
 * (image.c:1950-1993) run on the device, bit-identical to the host path of Detector::detect(filename)
 * (yolo_v2_class.cpp:173-206).  Works with every supported cfg (3 input channels). */
unsigned char *network_pipeline_staging_frames(network net, int slot, int frame_w, int frame_h);
int network_detect_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h,
                                 float thresh, float nms, int max_det);
void network_detect_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h,
                                 float thresh, float nms, y2_detection *dets, int *counts, int max_det);
/* A list of n decoded frames (1 <= n <= batch), each uint8 interleaved RGB [frame_h[i]][frame_w[i]][3] with its own
 * size: byte/255. and resize_image run on the device for every frame in one launch, bit-identical per frame to the
 * host chain of network_detect_batch_frames.  dets: [n][max_det], counts: [n]; the wait of such a batch fills only
 * the first n images.  network_pipeline_staging_frame_list grows the slot's pinned buffer for this list, returns its
 * base and fills offsets[n]: a frame already written at base + offsets[i] is not copied again on the host (every
 * other frame is); the buffer moves when a later call needs it larger. */
unsigned char *network_pipeline_staging_frame_list(network net, int slot, int n, const int *frame_w,
                                                   const int *frame_h, size_t *offsets);
int network_detect_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, int max_det);
void network_detect_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, y2_detection *dets, int *counts,
                                     int max_det);
/* ---- frames as decoders deliver them: interleaved RGB or BGR, or NV12, with a row pitch, in host memory or in memory
 * of the network's GPU (a hardware decoder's surface, a torch or cupy tensor).  Host and device frames and the formats
 * may be mixed in one list.  Per frame, the result is bit-identical to the frame-list entry fed with the frame
 * converted to tight RGB bytes: BGR with its channels swapped, NV12 with OpenCV's COLOR_YUV2RGB_NV12 (BT.601 limited
 * range, fixed point).  The conversion runs on the device, inside the resize or letterbox launch.
 * Host frames are staged and uploaded as frame-list frames (NV12 at half the bytes of RGB) and are free when the
 * submit returns.  Device frames are read in place: only the table of records crosses PCIe.  They must stay unchanged
 * until the wait that returns their batch.
 * ready: a cudaEvent_t of the network's device (or NULL); the network's stream waits for it before it reads any
 * device frame, so a decoder or another stream can hand over frames without a host synchronise.
 * Refused through error(), before anything is staged: what the frame-list entries refuse, a NULL descs, an unknown
 * format, an odd NV12 size, a row of more than INT_MAX bytes, a pitch or uv_pitch smaller than the row, a device frame
 * that is not device or managed memory of the network's GPU over all its rows inside one allocation (one cudaMalloc,
 * or one mapped chunk of a virtual-memory allocator), and a host frame in device memory. */
#ifndef Y2_FRAME_DESC_DEFINED
#define Y2_FRAME_DESC_DEFINED
enum { Y2_FRAME_RGB24 = 0, Y2_FRAME_BGR24 = 1, Y2_FRAME_NV12 = 2 };
typedef struct y2_frame_desc {
    const void *data;  /* RGB24/BGR24: first row of interleaved pixels; NV12: first row of the Y plane */
    const void *uv;    /* NV12: first row of the interleaved U,V plane (NULL: data + h * pitch); else unused */
    int w, h;          /* pixels; NV12 needs both even */
    int pitch;         /* bytes from one row to the next; 0 = tight (3w, or w for NV12) */
    int uv_pitch;      /* NV12: bytes between UV rows; 0 = pitch */
    int format;        /* Y2_FRAME_* */
    int on_device;     /* 0: host memory, staged and uploaded like a frame-list frame; 1: memory of the network's GPU,
                        * read in place */
} y2_frame_desc;
#endif
/* The slot's pinned buffer laid out for this list (only w, h, format and on_device are read): its base, and in
 * offsets[n] each host frame's place in it ((size_t)-1 for a device frame).  A host frame whose data (and NV12 uv)
 * already points at its place, tight, is not copied again on the host.  The buffer moves when a later call needs it
 * larger. */
unsigned char *network_pipeline_staging_frame_descs(network net, int slot, int n, const y2_frame_desc *descs,
                                                    size_t *offsets);
int network_detect_submit_frame_descs(network net, int n, const y2_frame_desc *descs, void *ready, float thresh,
                                      float nms, int max_det);
void network_detect_batch_frame_descs(network net, int n, const y2_frame_desc *descs, void *ready, float thresh,
                                      float nms, y2_detection *dets, int *counts, int max_det);
/* ---- tiled detection of large frames ("sliced inference"): each frame of W x H pixels goes through the network as
 * overlapping tiles, and the tiles' detections are merged per frame by do_nms_sort over their union.
 * Tiles, per frame: the whole frame first when full = 1, then a cols x rows grid, row-major, of tw x th windows with
 *   tw = min(W, ceil((W + (cols-1)*overlap) / cols)) (NV12: rounded up to even),
 *   x0_i = cols == 1 ? 0 : floor(i*(W - tw) / (cols-1)) (NV12: bit 0 cleared), the same for rows, H, th and y0_j:
 * the first tile starts at 0, the last ends at W, and neighbours share at least overlap columns (NV12: overlap - 1).
 * Each tile is converted, resized and run as a frame of network_detect_submit_frame_descs; its boxes (get_region_boxes
 * relative to the tile) go to frame coordinates as x = ((float)x0 + x*(float)tw) / (float)W, w = (w*(float)tw) /
 * (float)W (fp32, round-to-nearest, no FMA; an axis the tile spans whole passes unchanged), likewise y and h.  The
 * tiles' boxes and probability rows, in tile order (union index t * l.w*l.h*l.n + i), then take do_nms_sort (nms <= 0
 * skips it) and the final pick of Detector::detect, in union-index order.  dets [n][max_det] are relative to the frame
 * with box_index the union index; counts hold the full number.  A 1 x 1 tiling without full is exactly
 * network_detect_submit_frame_descs.
 * A frame's tiles are network images of one batch, so the list may hold at most net.batch tiles.  A host frame is
 * staged and uploaded once, however many tiles read it; device frames are read in place.  ready and the lifetimes are
 * those of the descriptor entries.  Collected by network_detect_wait (n frames).
 * Refused through error(), before anything is staged: what the descriptor entries refuse, a NULL tiling, cols or rows
 * outside 1 .. Y2_TILE_MAX, overlap < 0, full not 0 or 1, more tiles than net.batch, and a softmax-tree region. */
#ifndef Y2_TILING_DEFINED
#define Y2_TILING_DEFINED
#define Y2_TILE_MAX 16
typedef struct y2_tiling {
    int cols, rows; /* 1 .. Y2_TILE_MAX */
    int overlap;    /* columns (rows) neighbours share at least; NV12: at least overlap - 1 */
    int full;       /* 1: the whole frame is the frame's first tile */
} y2_tiling;
#endif
int network_detect_submit_tiled_descs(network net, int n, const y2_frame_desc *descs, const y2_tiling *tiling,
                                      void *ready, float thresh, float nms, int max_det);
void network_detect_batch_tiled_descs(network net, int n, const y2_frame_desc *descs, const y2_tiling *tiling,
                                      void *ready, float thresh, float nms, y2_detection *dets, int *counts,
                                      int max_det);
/* ---- many video streams in one batch, each frame detected on the 3-frame mean of its stream: per stream the
 * result is bit-identical to Detector::detect(img, thresh, use_mean = true) (yolo_v2_class.cpp:206-216) on that
 * stream's frames in order.  A stream is a ring of the last 3 region outputs, all zero at the start, and a
 * frame_index: a frame writes slot frame_index, is decoded on (((0 + slot0) + slot1) + slot2) / 3 in float, then
 * frame_index = (frame_index + 1) % 3.  The mean and the ring update run on the device; only the detections come
 * back.  Needs a flat-softmax region head (no softmax tree).
 * Streams live in the network's runtime and are freed by free_network.  open (re)allocates and starts every stream
 * over; ids are 0 .. max_streams-1.  set_batch_network keeps the streams; after resize_network open them again. */
void network_streams_open(network net, int max_streams);
/* The stream starts over (zero ring, frame_index 0).  Ordered after batches already submitted. */
void network_stream_reset(network net, int stream);
/* A frame list (as network_detect_submit_frame_list, same staging call) whose image i belongs to stream
 * stream_ids[i].  A stream may appear several times in one list; its frames are taken in list order.  Collected by
 * network_detect_wait (n images).  Streams batches share the two pipeline slots with every other kind. */
int network_detect_submit_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms, int max_det);
/* The same with the batch already in the slot's device input (fp32 planar at the network's size); images n..batch-1
 * of it are run through the network but neither decoded nor entered into any stream. */
int network_detect_submit_streams_resident(network net, int n, const int *stream_ids, float thresh, float nms,
                                           int max_det);
void network_detect_batch_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms,
                                  y2_detection *dets, int *counts, int max_det);
/* ---- tracked streams: per stream the result is bit-identical to Detector::detect(img, thresh, use_mean) followed by
 * Detector::tracking(result, frames_story) (yolo_v2_class.cpp:173-304) on that stream's frames in order: boxes in the
 * frame's pixels, each with a track id that stays the same across frames (ids start at 1 per class and stream). */
#ifndef Y2_BBOX_DEFINED
#define Y2_BBOX_DEFINED
typedef struct y2_bbox { /* bbox_t (yolo_v2_class.hpp:27-33) */
    unsigned int x, y, w, h;
    float prob;
    unsigned int obj_id, track_id;
} y2_bbox;
#endif
#ifndef Y2_TRACK_MAX_STORY
#define Y2_TRACK_MAX_STORY 32
#endif
#ifndef Y2_TRACK_MAX_TOTAL
#define Y2_TRACK_MAX_TOTAL 7168
#endif
/* Turns tracking on for the opened streams (1 <= frames_story <= Y2_TRACK_MAX_STORY; the Detector's default is 6) and
 * starts every track over; refused for a region of more than Y2_TRACK_MAX_TOTAL boxes per image (l.w * l.h * l.n).
 * The history and ids live on the device.  network_streams_open drops them (call this
 * again after it); set_batch_network keeps them; network_stream_reset also starts that stream's tracks over.
 * frames_story is fixed until the next call: a Detector whose story shrinks between calls drops one frame per call,
 * which is not reproduced. */
void network_streams_track(network net, int frames_story);
/* As network_detect_submit_streams, frame i of frame_w[i] x frame_h[i] pixels.  use_mean 1 decodes on the stream's
 * 3-frame mean and advances its ring; use_mean 0 decodes the plain region output and leaves the ring alone.  Either
 * way the tracks advance.  Tracking sees every detection; max_det caps only what is copied out, counts hold the full
 * number.  Collected by network_detect_wait_tracked (n images, boxes [n][max_det]). */
int network_detect_submit_streams_tracked(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                          const int *frame_w, const int *frame_h, float thresh, float nms,
                                          int use_mean, int max_det);
/* The same with the batch already in the slot's device input; frame_w / frame_h are the pixel sizes the boxes are
 * scaled to. */
int network_detect_submit_streams_tracked_resident(network net, int n, const int *stream_ids, const int *frame_w,
                                                   const int *frame_h, float thresh, float nms, int use_mean,
                                                   int max_det);
void network_detect_batch_streams_tracked(network net, int n, const int *stream_ids,
                                          const unsigned char *const *frames, const int *frame_w, const int *frame_h,
                                          float thresh, float nms, int use_mean, y2_bbox *boxes, int *counts,
                                          int max_det);
int network_detect_wait_tracked(network net, y2_bbox *boxes, int *counts, int max_det);
/* The streams and tracked-streams entries fed with frame descriptors (see network_detect_submit_frame_descs); tracked
 * boxes are scaled to each descriptor's w x h. */
int network_detect_submit_streams_descs(network net, int n, const int *stream_ids, const y2_frame_desc *descs,
                                        void *ready, float thresh, float nms, int max_det);
void network_detect_batch_streams_descs(network net, int n, const int *stream_ids, const y2_frame_desc *descs,
                                        void *ready, float thresh, float nms, y2_detection *dets, int *counts,
                                        int max_det);
int network_detect_submit_streams_tracked_descs(network net, int n, const int *stream_ids, const y2_frame_desc *descs,
                                                void *ready, float thresh, float nms, int use_mean, int max_det);
void network_detect_batch_streams_tracked_descs(network net, int n, const int *stream_ids,
                                                const y2_frame_desc *descs, void *ready, float thresh, float nms,
                                                int use_mean, y2_bbox *boxes, int *counts, int max_det);
/* ---- batched, device-resident classification: letterbox, forward pass, WordTree products and top-k run on the
 * device and only `top` (index, probability) pairs per image come back, equal to what predict_classifier_image
 * computes on the host (classifier.c:676-730: letterbox_image, network_predict, hierarchy_predictions for a WordTree
 * classifier, top_k).  The network's output layer must be a class vector (softmax, avgpool, connected or dropout;
 * a region network uses network_detect_*), 1 <= top <= min(outputs, Y2_CLASSIFY_MAX_TOP = 128), and a WordTree must list
 * every parent before its children and be at most 64 levels deep.  hits: [batch][top], best first, in top_k's order (which also decides which of
 * several equal probabilities are kept).  A NaN in the output ranks below every number. */
#ifndef Y2_CLASS_HIT_DEFINED
#define Y2_CLASS_HIT_DEFINED
typedef struct y2_class_hit {
    int index;
    float prob;
} y2_class_hit;
#endif
/* top-k (and the WordTree products) of the last forward pass (network_forward_device) */
void network_classify_device(network net, int top, y2_class_hit *hits);
/* upload + forward + classify of `batch` prepared images (fp32 planar CHW, already letterboxed), one synchronisation */
void network_classify_batch(network net, const float *input, int top, y2_class_hit *hits);
/* Decoded frames of any size, uint8 interleaved RGB [batch][frame_h][frame_w][3]: byte/255. and letterbox_image
 * (image.c:1624-1644) run on the device, bit-identical to the host chain.  Frames at the network's size take the
 * uint8 first-layer path when the network has one (letterbox is the identity there). */
void network_classify_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top,
                                   y2_class_hit *hits);
/* The submit/wait pipeline of network_detect_submit* for classification: the same two slots, staging buffers
 * (network_pipeline_staging, _u8, _frames) and device inputs (network_pipeline_input_device).  Detection and
 * classification batches may be interleaved; each wait must match the kind of the OLDEST batch in flight, and
 * network_classify_wait's top must be the one that batch was submitted with. */
int network_classify_submit(network net, const float *input, int top);
int network_classify_submit_u8(network net, const unsigned char *input_hwc, int top);
int network_classify_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top);
int network_classify_submit_resident(network net, int top);
int network_classify_wait(network net, y2_class_hit *hits, int top);
/* A list of n frames of any sizes (as network_detect_submit_frame_list, same staging call), each letterboxed on the
 * device: hits [n][top].  A letterbox window 1 pixel high has no defined result, as for the uniform entry. */
int network_classify_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top);
void network_classify_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top, y2_class_hit *hits);
/* A list of n frame descriptors (see network_detect_submit_frame_descs), each letterboxed on the device:
 * hits [n][top]. */
int network_classify_submit_frame_descs(network net, int n, const y2_frame_desc *descs, void *ready, int top);
void network_classify_batch_frame_descs(network net, int n, const y2_frame_desc *descs, void *ready, int top,
                                        y2_class_hit *hits);
/* ---- the same over several GPUs of one box from ONE caller (one replica and one host thread per GPU; idiom of
 * train_networks, network_kernels.cu:346-376).  Replica i owns the next nets[i].batch images of the global batch;
 * detections land in the caller's arrays in image order - nothing else crosses GPUs. ------------------------- */
network *parse_network_cfg_multi(char *cfgfile, char *weightfile, int *gpus, int ngpus, int batch);
void free_network_multi(network *nets, int n);
int network_multi_batch(network *nets, int n); /* images per call = sum of the replicas' batches */
void network_detect_batch_multi(network *nets, int n, const float *images, float thresh, float nms,
                                y2_detection *dets, int *counts, int max_det);
void network_detect_batch_u8_multi(network *nets, int n, const unsigned char *images_hwc, float thresh, float nms,
                                   y2_detection *dets, int *counts, int max_det);
void network_detect_submit_multi(network *nets, int n, const float *images, float thresh, float nms, int max_det);
void network_detect_submit_u8_multi(network *nets, int n, const unsigned char *images_hwc, float thresh, float nms,
                                    int max_det);
void network_detect_wait_multi(network *nets, int n, y2_detection *dets, int *counts, int max_det);
/* Block until the network's stream is idle. */
void network_sync(network net);
/* Device stream the network runs on (cudaStream_t) — for timing with CUDA events. */
void *network_stream(network net);
/* Algorithmic conv FLOPs per image: sum 2*n*k*k*c*out_h*out_w (darknet.c:115-131 `operations`). */
double network_conv_flops(network net);
/* Kernel that runs convolutional layer i: 0 per-tap implicit GEMM, 1 halo-slab, 2 CTA-pair
 * (cta_group::2), 3 conv + maxpool, 4 fused first layer (conv + maxpool from the fp32 image);
 * -1 if layer i is not a convolution. */
int network_conv_kernel(network net, int i);
/* Number of kernel launches one forward issues (diagnostics / bench `gpu_launches`). */
int network_launch_count(network net);
/* Per-layer device time of the last profiled forward, in ms (NULL if never profiled). */
int network_profile_layers(network net, float *ms_per_layer, int n);
/* 1 -> run layers eagerly instead of replaying the captured CUDA graph */
void network_set_eager(network net, int eager);
/* sizeof(layer|network|network_state|y2_detection|box|y2_class_hit|y2_bbox|y2_frame_desc|y2_tiling) for what = 0..8:
 * lets a
 * binding that passes these structs by value check its mirror against the library it loaded. */
size_t y2_abi_sizeof(int what);

#ifdef __cplusplus
}
#endif
#endif
