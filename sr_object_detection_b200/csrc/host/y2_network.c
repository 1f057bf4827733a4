/*
 * Network runtime of the drop-in API: layer constructors, the device planner (buffer arena,
 * in-place route aliasing, tensor-map plans), the single-stream graph-captured layer schedule,
 * network_predict and the batched detection extension.
 *
 * Reference interfaces replaced (behavioural spec only): network.c:132-181,308-388,458-474,
 * 592-609; network_kernels.cu:43-56,378-407; convolutional_layer.c:75-83,182-319;
 * maxpool_layer.c:20-51; reorg_layer.c:7-45; route_layer.c:6-37,104-117; region_layer.c:14-51;
 * shortcut_layer.c, avgpool_layer.c, softmax_layer.c, cost_layer.c; cuda.c:12-158.
 *
 * Design differences from the reference (see DESIGN.md):
 *  - one persistent device arena per network instead of cudaMalloc/cudaFree per predict;
 *  - activations live on the device as padded-NHWC bf16, the reference's NCHW fp32 view of a
 *    layer is produced on demand (get_network_output_layer);
 *  - route layers cost nothing: producers write straight into the concat buffer;
 *  - the per-layer host loop is captured once into a CUDA graph and replayed.
 */
#include "y2_host.h"

#include <assert.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

int gpu_index = 0;

/* ---- cuda.c equivalents --------------------------------------------------------------------- */
void cuda_set_device(int n)
{
    gpu_index = n;
    Y2_CHECK(y2_set_device(n));
}

int cuda_get_device(void)
{
    return gpu_index;
}

void check_error_code(int status, const char *what)
{
    if (status != Y2_OK) y2_fatal(what, status);
}

float *cuda_make_array(float *x, size_t n)
{
    void *d = 0;
    Y2_CHECK(y2_malloc(&d, n * sizeof(float)));
    if (x) {
        Y2_CHECK(y2_memcpy_h2d(d, x, n * sizeof(float), 0));
        Y2_CHECK(y2_stream_sync(0));
    } else {
        Y2_CHECK(y2_memset(d, 0, n * sizeof(float), 0));
        Y2_CHECK(y2_stream_sync(0));
    }
    return (float *)d;
}

int *cuda_make_int_array(size_t n)
{
    void *d = 0;
    Y2_CHECK(y2_malloc(&d, n * sizeof(int)));
    return (int *)d;
}

void cuda_push_array(float *x_gpu, float *x, size_t n)
{
    Y2_CHECK(y2_memcpy_h2d(x_gpu, x, n * sizeof(float), 0));
    Y2_CHECK(y2_stream_sync(0));
}

void cuda_pull_array(float *x_gpu, float *x, size_t n)
{
    Y2_CHECK(y2_memcpy_d2h(x, x_gpu, n * sizeof(float), 0));
    Y2_CHECK(y2_stream_sync(0));
}

void cuda_free(float *x_gpu)
{
    Y2_CHECK(y2_free(x_gpu));
}

static void *dev_upload(const void *host, size_t bytes)
{
    void *d = 0;
    Y2_CHECK(y2_malloc(&d, bytes));
    Y2_CHECK(y2_memcpy_h2d(d, host, bytes, 0));
    Y2_CHECK(y2_stream_sync(0));
    return d;
}

/* round-to-nearest-even fp32 -> bf16, NaN kept quiet */
uint16_t y2_f32_to_bf16(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x0040u);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

static int round_up(int v, int m) { return (v + m - 1) / m * m; }

/* channels as stored on the device: multiples of 32 below 64, multiples of 64 above */
static int storage_channels(int c) { return c < 64 ? round_up(c, 32) : round_up(c, 64); }

char *get_layer_string(LAYER_TYPE a)
{
    switch (a) {
    case CONVOLUTIONAL: return "convolutional";
    case MAXPOOL: return "maxpool";
    case REGION: return "region";
    case REORG: return "reorg";
    case ROUTE: return "route";
    case SHORTCUT: return "shortcut";
    case AVGPOOL: return "avgpool";
    case SOFTMAX: return "softmax";
    case COST: return "cost";
    case CONNECTED: return "connected";
    case DETECTION: return "detection";
    case DROPOUT: return "dropout";
    case CROP: return "crop";
    case NORMALIZATION: return "normalization";
    case BATCHNORM: return "batchnorm";
    case LOCAL: return "local";
    case ACTIVE: return "activation";
    case RNN: return "rnn";
    case GRU: return "gru";
    case CRNN: return "crnn";
    case DECONVOLUTIONAL: return "deconvolutional";
    default: return "none";
    }
}

void forward_no_cpu_path(layer l, network_state state)
{
    (void)l;
    (void)state;
    error("yolo2-b200 has no CPU execution path (gpu_index must be >= 0)");
}

/* ---- layer constructors (host description only; device buffers come from the planner) ------- */
static float rand_uniform_pm1(uint32_t *st)
{
    *st = *st * 1664525u + 1013904223u;
    return ((*st >> 8) * (1.0f / 8388608.0f)) - 1.0f;
}

layer make_convolutional_layer(int batch, int h, int w, int c, int n, int size, int stride, int padding,
                               ACTIVATION activation, int batch_normalize, int binary, int xnor, int adam)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = CONVOLUTIONAL;
    l.h = h;
    l.w = w;
    l.c = c;
    l.n = n;
    l.binary = binary;
    l.xnor = xnor;
    l.batch = batch;
    l.stride = stride;
    l.size = size;
    l.pad = padding;
    l.batch_normalize = batch_normalize;
    l.activation = activation;
    size_t nw = (size_t)c * n * size * size;
    l.weights = (float *)calloc(nw, sizeof(float));
    l.biases = (float *)calloc(n, sizeof(float));
    if (adam) { /* convolutional_layer.c:226-231: moments travel with the checkpoint */
        l.adam = 1;
        l.m = (float *)calloc(nw, sizeof(float));
        l.v = (float *)calloc(nw, sizeof(float));
    }
    /* same init scale as convolutional_layer.c:207-208 (values differ: own generator) */
    float scale = sqrtf(2.f / (size * size * c));
    uint32_t st = 0x9E3779B9u ^ (uint32_t)(n * 131 + c * 31 + size);
    for (size_t i = 0; i < nw; ++i) l.weights[i] = scale * rand_uniform_pm1(&st);
    /* convolutional_layer.c:75-83 */
    l.out_h = (h + 2 * padding - size) / stride + 1;
    l.out_w = (w + 2 * padding - size) / stride + 1;
    l.out_c = n;
    l.outputs = l.out_h * l.out_w * l.out_c;
    l.inputs = l.w * l.h * l.c;
    if (batch_normalize) {
        l.scales = (float *)calloc(n, sizeof(float));
        for (int i = 0; i < n; ++i) l.scales[i] = 1;
        l.rolling_mean = (float *)calloc(n, sizeof(float));
        l.rolling_variance = (float *)calloc(n, sizeof(float));
    }
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_convolutional_layer_gpu;
    l.workspace_size = 0; /* implicit GEMM: no im2col workspace */
    fprintf(stderr, "conv  %5d %2d x%2d /%2d  %4d x%4d x%4d   ->  %4d x%4d x%4d\n", n, size, size, stride, w,
            h, c, l.out_w, l.out_h, l.out_c);
    return l;
}

layer make_maxpool_layer(int batch, int h, int w, int c, int size, int stride, int padding)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = MAXPOOL;
    l.batch = batch;
    l.h = h;
    l.w = w;
    l.c = c;
    l.pad = padding;
    l.out_w = (w + 2 * padding) / stride; /* maxpool_layer.c:30-31 */
    l.out_h = (h + 2 * padding) / stride;
    l.out_c = c;
    l.outputs = l.out_h * l.out_w * l.out_c;
    l.inputs = h * w * c;
    l.size = size;
    l.stride = stride;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_maxpool_layer_gpu;
    fprintf(stderr, "max          %d x %d / %d  %4d x%4d x%4d   ->  %4d x%4d x%4d\n", size, size, stride, w, h, c,
            l.out_w, l.out_h, l.out_c);
    return l;
}

layer make_reorg_layer(int batch, int w, int h, int c, int stride, int reverse)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = REORG;
    l.batch = batch;
    l.stride = stride;
    l.h = h;
    l.w = w;
    l.c = c;
    if (reverse) {
        l.out_w = w * stride;
        l.out_h = h * stride;
        l.out_c = c / (stride * stride);
    } else {
        l.out_w = w / stride;
        l.out_h = h / stride;
        l.out_c = c * (stride * stride);
    }
    l.reverse = reverse;
    fprintf(stderr, "reorg              /%2d  %4d x%4d x%4d   ->  %4d x%4d x%4d\n", stride, w, h, c, l.out_w,
            l.out_h, l.out_c);
    l.outputs = l.out_h * l.out_w * l.out_c;
    l.inputs = h * w * c;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_reorg_layer_gpu;
    return l;
}

layer make_route_layer(int batch, int n, int *input_layers, int *input_sizes)
{
    fprintf(stderr, "route ");
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = ROUTE;
    l.batch = batch;
    l.n = n;
    l.input_layers = input_layers;
    l.input_sizes = input_sizes;
    int outputs = 0;
    for (int i = 0; i < n; ++i) {
        fprintf(stderr, " %d", input_layers[i]);
        outputs += input_sizes[i];
    }
    fprintf(stderr, "\n");
    l.outputs = outputs;
    l.inputs = outputs;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_route_layer_gpu;
    return l;
}

layer make_region_layer(int batch, int w, int h, int n, int classes, int coords)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = REGION;
    l.n = n;
    l.batch = batch;
    l.h = h;
    l.w = w; /* out_h / out_w stay 0, as region_layer.c:14-51 leaves them */
    l.classes = classes;
    l.coords = coords;
    l.cost = (float *)calloc(1, sizeof(float));
    l.biases = (float *)calloc((size_t)n * 2, sizeof(float));
    l.outputs = h * w * n * (classes + coords + 1);
    l.inputs = l.outputs;
    for (int i = 0; i < n * 2; ++i) l.biases[i] = .5;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_region_layer_gpu;
    fprintf(stderr, "detection\n");
    return l;
}

layer make_shortcut_layer(int batch, int index, int w, int h, int c, int w2, int h2, int c2)
{
    fprintf(stderr, "Shortcut Layer: %d\n", index);
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = SHORTCUT;
    l.batch = batch;
    /* shortcut_layer.c: (w,h,c) describe the `from` tensor, out_* the running tensor */
    l.w = w2;
    l.h = h2;
    l.c = c2;
    l.out_w = w;
    l.out_h = h;
    l.out_c = c;
    l.outputs = w * h * c;
    l.inputs = l.outputs;
    l.index = index;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_shortcut_layer_gpu;
    return l;
}

layer make_avgpool_layer(int batch, int w, int h, int c)
{
    fprintf(stderr, "avg                     %4d x%4d x%4d   ->  %4d\n", w, h, c, c);
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = AVGPOOL;
    l.batch = batch;
    l.h = h;
    l.w = w;
    l.c = c;
    l.out_w = 1;
    l.out_h = 1;
    l.out_c = c;
    l.outputs = l.out_c;
    l.inputs = h * w * c;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_avgpool_layer_gpu;
    return l;
}

layer make_softmax_layer(int batch, int inputs, int groups)
{
    assert(inputs % groups == 0);
    fprintf(stderr, "softmax                                        %4d\n", inputs);
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = SOFTMAX;
    l.batch = batch;
    l.groups = groups;
    l.inputs = inputs;
    l.outputs = inputs;
    l.temperature = 1;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_softmax_layer_gpu;
    return l;
}

layer make_cost_layer(int batch, int inputs, COST_TYPE type, float scale)
{
    (void)scale;
    fprintf(stderr, "cost                                           %4d\n", inputs);
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = COST;
    l.batch = batch;
    l.inputs = inputs;
    l.outputs = inputs;
    l.cost_type = type;
    l.cost = (float *)calloc(1, sizeof(float));
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_cost_layer_gpu; /* no-op at inference (cost_layer.c:75) */
    return l;
}

/* connected_layer.c:13-100 (host description; the device side is a 1x1 convolution plan over the flattened input) */
layer make_connected_layer(int batch, int inputs, int outputs, ACTIVATION activation, int batch_normalize)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = CONNECTED;
    l.inputs = inputs;
    l.outputs = outputs;
    l.batch = batch;
    l.batch_normalize = batch_normalize;
    l.h = 1;
    l.w = 1;
    l.c = inputs;
    l.out_h = 1;
    l.out_w = 1;
    l.out_c = outputs;
    l.n = outputs;
    l.size = 1;
    l.stride = 1;
    l.activation = activation;
    l.weights = (float *)calloc((size_t)outputs * inputs, sizeof(float));
    l.biases = (float *)calloc(outputs, sizeof(float));
    float scale = sqrtf(2.f / inputs);
    uint32_t st = 0x85EBCA6Bu ^ (uint32_t)(outputs * 131 + inputs);
    for (size_t i = 0; i < (size_t)outputs * inputs; ++i) l.weights[i] = scale * rand_uniform_pm1(&st);
    if (batch_normalize) {
        l.scales = (float *)calloc(outputs, sizeof(float));
        for (int i = 0; i < outputs; ++i) l.scales[i] = 1;
        l.rolling_mean = (float *)calloc(outputs, sizeof(float));
        l.rolling_variance = (float *)calloc(outputs, sizeof(float));
    }
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_connected_layer_gpu;
    fprintf(stderr, "connected                            %4d  ->  %4d\n", inputs, outputs);
    return l;
}

/* dropout_layer.c:7-26: identity at inference (forward_dropout_layer returns at once when !state.train) */
layer make_dropout_layer(int batch, int inputs, float probability)
{
    layer l;
    memset(&l, 0, sizeof(l));
    l.type = DROPOUT;
    l.inputs = inputs;
    l.outputs = inputs;
    l.batch = batch;
    l.forward = forward_no_cpu_path;
    l.forward_gpu = forward_dropout_layer_gpu;
    fprintf(stderr, "dropout       p = %.2f               %4d  ->  %4d\n", probability, inputs, inputs);
    return l;
}

/* ---- network queries ----------------------------------------------------------------------- */
int y2_output_layer_index(network net)
{
    int i;
    for (i = net.n - 1; i > 0; --i)
        if (net.layers[i].type != COST) break;
    return i;
}

int get_network_output_size(network net)
{
    return net.layers[y2_output_layer_index(net)].outputs;
}

int get_network_output_size_layer(network net, int i)
{
    return net.layers[i].outputs;
}

int get_network_input_size(network net)
{
    return net.layers[0].inputs;
}

double network_conv_flops(network net)
{
    double ops = 0;
    for (int i = 0; i < net.n; ++i) {
        layer l = net.layers[i];
        if (l.type == CONVOLUTIONAL) ops += 2.0 * l.n * l.size * l.size * l.c * l.out_h * l.out_w;
        else if (l.type == CONNECTED) ops += 2.0 * l.inputs * l.outputs; /* darknet.c:126-128 */
    }
    return ops;
}

/* ---- planner ---------------------------------------------------------------------------------- */
static size_t padded_bytes(int batch, int h, int w, int cs)
{
    return (size_t)batch * (h + 1) * (w + 1) * cs * 2;
}

static void *dev_alloc_zero(size_t bytes)
{
    void *d = 0;
    Y2_CHECK(y2_malloc(&d, bytes));
    Y2_CHECK(y2_memset(d, 0, bytes, 0));
    /* the network's own stream is non-blocking: nothing orders it behind the legacy stream's memset */
    Y2_CHECK(y2_stream_sync(0));
    return d;
}

/* which layer feeds layer i through state.input (the previous one) */
static int prev_layer(int i) { return i - 1; }

static int consumer_wants_f32(network *net, int i)
{
    /* a conv writes fp32 flat when the next layer is a region / avgpool head and nobody routes
     * from it */
    if (i + 1 >= net->n) return 1;
    LAYER_TYPE nt = net->layers[i + 1].type;
    if (nt != REGION && nt != AVGPOOL) return 0;
    for (int j = i + 2; j < net->n; ++j) {
        layer *lj = &net->layers[j];
        if (lj->type == ROUTE)
            for (int k = 0; k < lj->n; ++k)
                if (lj->input_layers[k] == i) return 0;
        if (lj->type == SHORTCUT && lj->index == i) return 0;
    }
    return 1;
}

static void free_layer_rt(layer *l)
{
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (!r) return;
    if (r->plan) y2_conv_plan_destroy(r->plan);
    y2_free(r->own_buf);
    y2_free(r->wt_dev);
    y2_free(r->alpha_dev);
    y2_free(r->beta_dev);
    y2_free(r->patches);
    y2_free(r->fc_in);
    y2_free(r->packed_in);
    y2_free(r->reorg_table);
    y2_free(r->stream_f32);
    y2_free(r->boxes_dev);
    y2_free(r->probs_dev);
    y2_free(r->biases_dev);
    y2_free(r->nms_cnt_dev);
    y2_free(r->collect_ws);
    y2_free(r->tile_ws);
    y2_free(r->child_ptr_dev);
    y2_free(r->child_grp_dev);
    y2_free(r->tree_rec_dev);
    y2_free(r->tree_parent_dev);
    y2_free(r->group_size_dev);
    y2_free(r->group_offset_dev);
    y2_free(r->map_dev);
    if (r->ev0) y2_event_destroy(r->ev0);
    if (r->ev1) y2_event_destroy(r->ev1);
    free(r);
    l->b200 = 0;
    l->output_gpu = 0;
    l->weights_gpu = 0;
}

void y2_unplan_network(network *net)
{
    y2_net_rt *rt = (y2_net_rt *)net->b200;
    if (!rt) return;
    Y2_CHECK(y2_set_device(rt->device));
    y2_stream_sync(rt->stream);
    for (int i = 0; i < net->n; ++i) free_layer_rt(&net->layers[i]);
    y2_host_free(rt->out_pinned);
    y2_results_free(&rt->res);
    y2_free(rt->export_dev);
    y2_pipe_free(rt);
    y2_streams_free(rt);
    y2_stream_destroy(rt->stream);
    free(rt);
    net->b200 = 0;
}

static void unsupported(int i, const char *what)
{
    fprintf(stderr, "layer %d: %s is not supported by the B200 hot path\n", i, what);
    error("unsupported layer configuration");
}

/* Pack fp32 [n][c][k][k] weights into bf16 [npad][ktot] with the K order the kernel walks, fold
 * batchnorm into (alpha, beta), upload.  Replaces push_convolutional_layer. */
void y2_push_convolutional_layer(layer *l)
{
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (!r) return;
    const int kk = l->size * l->size;
    const size_t elems = (size_t)r->npad * r->ktot;
    uint16_t *w = (uint16_t *)calloc(elems, sizeof(uint16_t));
    if (l->type == CONNECTED) {
        /* reference flat index ch*h*w + pos (NCHW) -> position-major (pos*c + ch) of y2_fc_pack_tensor */
        const int hw = r->fc_h > 0 ? r->fc_h * r->fc_w : 1, c = r->fc_c;
        for (int f = 0; f < l->outputs; ++f)
            for (int ch = 0; ch < c; ++ch)
                for (int pos = 0; pos < hw; ++pos)
                    w[(size_t)f * r->ktot + (size_t)pos * c + ch] =
                        y2_f32_to_bf16(l->weights[(size_t)f * l->inputs + (size_t)ch * hw + pos]);
    } else if (r->use_patches == 3) {
        /* K index = (c*k + r)*8 + s (y2_gather_rows_f32) */
        for (int f = 0; f < l->n; ++f)
            for (int c = 0; c < l->c; ++c)
                for (int rr = 0; rr < l->size; ++rr)
                    for (int ss = 0; ss < l->size; ++ss)
                        w[(size_t)f * r->ktot + (size_t)(c * l->size + rr) * 8 + ss] =
                            y2_f32_to_bf16(l->weights[(((size_t)f * l->c + c) * l->size + rr) * l->size + ss]);
    } else if (r->use_patches == 1) {
        /* K index = c*kk + r*k + s : the reference's own [c][kh][kw] order (im2col.c:26-28) */
        for (int f = 0; f < l->n; ++f)
            for (int k = 0; k < l->c * kk; ++k)
                w[(size_t)f * r->ktot + k] = y2_f32_to_bf16(l->weights[(size_t)f * l->c * kk + k]);
    } else {
        /* K index = tap*cin_pad + c */
        for (int f = 0; f < l->n; ++f)
            for (int c = 0; c < l->c; ++c)
                for (int t = 0; t < kk; ++t)
                    w[(size_t)f * r->ktot + (size_t)t * r->cin_pad + c] =
                        y2_f32_to_bf16(l->weights[((size_t)f * l->c + c) * kk + t]);
    }
    float *alpha = (float *)calloc(r->npad, sizeof(float));
    float *beta = (float *)calloc(r->npad, sizeof(float));
    for (int f = 0; f < l->n; ++f) {
        if (l->batch_normalize) {
            /* (x - mean)/(sqrt(var) + 1e-6) * scale + bias   (blas.c:115-126, conv_layer.c:401-423) */
            float a = (float)(l->scales[f] / (sqrt((double)l->rolling_variance[f]) + .000001f));
            alpha[f] = a;
            beta[f] = l->biases[f] - l->rolling_mean[f] * a;
        } else {
            alpha[f] = 1.f;
            beta[f] = l->biases[f];
        }
    }
    if (r->stem_fused || r->pool_fused) {
        /* the fused conv+maxpool kernels take the max before the affine map, which needs alpha >= 0:
         * negate the filter and its alpha together (alpha*acc is unchanged bit for bit) */
        for (int f = 0; f < l->n; ++f)
            if (alpha[f] < 0) {
                alpha[f] = -alpha[f];
                for (int k = 0; k < r->ktot; ++k) w[(size_t)f * r->ktot + k] ^= 0x8000u;
            }
    }
    Y2_CHECK(y2_memcpy_h2d(r->wt_dev, w, elems * 2, 0));
    Y2_CHECK(y2_memcpy_h2d(r->alpha_dev, alpha, (size_t)r->npad * 4, 0));
    Y2_CHECK(y2_memcpy_h2d(r->beta_dev, beta, (size_t)r->npad * 4, 0));
    Y2_CHECK(y2_stream_sync(0));
    free(w);
    free(alpha);
    free(beta);
    r->wt_dirty = 0;
}

static int pick_block_n(int cout)
{
    if (cout <= 32) return 32;
    if (cout <= 64) return 64;
    if (cout <= 128) return 128;
    return 256;
}

/* conv i is a 3x3/1 'same' leaky/linear layer whose output feeds ONLY the 2x2/2 unpadded maxpool
 * right behind it (no route / shortcut reads the full-resolution tensor) */
static int feeds_only_pool2x2(network *net, int i)
{
    if (i + 1 >= net->n) return 0;
    layer *l = &net->layers[i], *m = &net->layers[i + 1];
    if (l->size != 3 || l->stride != 1 || l->pad != 1) return 0;
    if (l->activation != LEAKY && l->activation != LINEAR) return 0;
    if (m->type != MAXPOOL || m->size != 2 || m->stride != 2 || m->pad != 0) return 0;
    if (l->out_h < 2 || l->out_w < 2) return 0;
    for (int j = i + 2; j < net->n; ++j) {
        layer *lj = &net->layers[j];
        if (lj->type == ROUTE)
            for (int k = 0; k < lj->n; ++k)
                if (lj->input_layers[k] == i) return 0;
        if (lj->type == SHORTCUT && lj->index == i) return 0;
    }
    return 1;
}

/* layer 0 over <= 3 channels with <= 32 filters: conv + pool run as the fused first-layer kernel */
static int stem_fusable(network *net, int i)
{
    if (i != 0) return 0;
    layer *l = &net->layers[0];
    if (l->c > 3 || l->n > 32) return 0;
    return feeds_only_pool2x2(net, 0);
}

/* a later conv with one channel block (<= 64 stored input channels) and exactly 64 or 128 filters: the
 * maxpool runs in the convolution's epilogue (conv_pool.cu) */
static int pool_fusable(network *net, int i, int cin_pad)
{
    if (i == 0) return 0;
    layer *l = &net->layers[i];
    if (cin_pad != 32 && cin_pad != 64) return 0;
    if (l->n != 64 && l->n != 128) return 0;
    return feeds_only_pool2x2(net, i);
}

/* view of the tensor a layer reads through state.input */
typedef struct {
    void *ptr;
    int cs, cpad, kind;
} y2_view;

static y2_view input_view(network *net, int i)
{
    y2_view v;
    memset(&v, 0, sizeof(v));
    int p = prev_layer(i);
    if (p < 0) {
        v.kind = Y2_KIND_NONE;
        return v;
    }
    y2_layer_rt *r = (y2_layer_rt *)net->layers[p].b200;
    v.ptr = r->out;
    v.cs = r->out_cs;
    v.cpad = r->cpad;
    v.kind = r->out_kind;
    return v;
}

/* the epilogue's activation code; anything else runs LINEAR and gets a separate activation pass (post_act) */
static int epilogue_act(ACTIVATION a)
{
    return a == LEAKY ? Y2_ACT_LEAKY : a == LOGISTIC ? Y2_ACT_LOGISTIC : Y2_ACT_LINEAR;
}

static void build_conv_plan(network *net, int i, int batch)
{
    layer *l = &net->layers[i];
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (r->plan) {
        y2_conv_plan_destroy(r->plan);
        r->plan = 0;
    }
    y2_conv_desc d;
    memset(&d, 0, sizeof(d));
    if (r->use_patches) {
        d.in = r->patches;
        d.in_cs = r->kpad;
        d.cin = r->kpad;
        d.ksize = 1;
    } else {
        y2_view v;
        if (i == 0) {
            v.ptr = r->packed_in;
            v.cs = r->cin_pad;
        } else {
            v = input_view(net, i);
        }
        d.in = v.ptr;
        d.in_cs = v.cs;
        d.cin = r->cin_pad;
        d.ksize = l->size;
        /* order in which the producer's kernel wrote this tensor (a fused maxpool was written by its conv) */
        int src = i - 1;
        if (src >= 1 && net->layers[src].type == MAXPOOL && ((y2_layer_rt *)net->layers[src].b200)->fused_into_prev)
            --src;
        if (src >= 0 && net->layers[src].type == CONVOLUTIONAL)
            d.in_order = ((y2_layer_rt *)net->layers[src].b200)->write_order;
    }
    d.batch = batch;
    d.h = l->out_h;
    d.w = l->out_w;
    d.wt = r->wt_dev;
    d.npad = r->npad;
    d.block_n = r->block_n;
    d.block_k = r->block_k;
    d.alpha = r->alpha_dev;
    d.beta = r->beta_dev;
    d.act = r->post_act >= 0 ? Y2_ACT_LINEAR : epilogue_act(l->activation);
    d.out = r->out;
    d.out_cs = r->out_cs;
    if (r->pool_fused) {
        y2_layer_rt *mr = (y2_layer_rt *)net->layers[i + 1].b200;
        d.out = mr->out;
        d.out_cs = mr->out_cs;
        d.out_mode = Y2_OUT_BF16_POOLED;
        d.cout = r->cpad;
    } else if (r->out_kind == Y2_KIND_F32_FLAT) {
        d.out_mode = Y2_OUT_F32_FLAT;
        d.cout = l->n;
    } else {
        d.out_mode = Y2_OUT_BF16_PADDED;
        d.cout = r->cpad;
    }
    Y2_CHECK(y2_conv_plan_create(&d, &r->plan));
    r->write_order = y2_conv_plan_order(r->plan);
}

static void build_fc_plan(network *net, int i, int batch)
{
    layer *l = &net->layers[i];
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (r->plan) {
        y2_conv_plan_destroy(r->plan);
        r->plan = 0;
    }
    y2_conv_desc d;
    memset(&d, 0, sizeof(d));
    d.in = r->fc_in;
    d.in_cs = r->kpad;
    d.cin = r->kpad;
    d.batch = batch;
    d.h = 1;
    d.w = 1;
    d.ksize = 1;
    d.wt = r->wt_dev;
    d.cout = l->outputs;
    d.npad = r->npad;
    d.block_n = r->block_n;
    d.block_k = r->block_k;
    d.alpha = r->alpha_dev;
    d.beta = r->beta_dev;
    d.act = r->post_act >= 0 ? Y2_ACT_LINEAR : epilogue_act(l->activation);
    d.out = r->out;
    d.out_cs = r->out_cs;
    d.out_mode = Y2_OUT_F32_FLAT;
    Y2_CHECK(y2_conv_plan_create(&d, &r->plan));
}

static void build_plans(network *net, int batch)
{
    y2_net_rt *rt = (y2_net_rt *)net->b200;
    for (int i = 0; i < net->n; ++i) {
        if (net->layers[i].type == CONVOLUTIONAL && !((y2_layer_rt *)net->layers[i].b200)->stem_fused)
            build_conv_plan(net, i, batch);
        else if (net->layers[i].type == CONNECTED) build_fc_plan(net, i, batch);
    }
    rt->plan_batch = batch;
    y2_pipe_release(rt);
}

void y2_plan_network(network *net)
{
    /* the video streams outlive the re-plan (set_batch_network, resize_network) when the device stays the same */
    y2_streams *streams = NULL;
    y2_net_rt *old = (y2_net_rt *)net->b200;
    if (old && old->device == net->gpu_index) {
        streams = old->streams;
        old->streams = NULL;
    }
    if (net->b200) y2_unplan_network(net);
    Y2_CHECK(y2_set_device(net->gpu_index));
    y2_net_rt *rt = (y2_net_rt *)calloc(1, sizeof(y2_net_rt));
    net->b200 = rt;
    rt->device = net->gpu_index;
    rt->streams = streams;
    Y2_CHECK(y2_stream_create(&rt->stream));
    const int B = net->batch;
    rt->cap_batch = B;
    rt->plan_w = net->w;
    rt->plan_h = net->h;
    rt->in_bytes = (size_t)B * net->inputs * sizeof(float);
    Y2_CHECK(y2_malloc((void **)&rt->pipe[0].in_dev, rt->in_bytes)); /* also the synchronous path's input */
    Y2_CHECK(y2_host_alloc((void **)&rt->pipe[0].in_pinned, rt->in_bytes));

    /* pass 1: per-layer storage decisions */
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        y2_layer_rt *r = (y2_layer_rt *)calloc(1, sizeof(y2_layer_rt));
        l->b200 = r;
        r->placed_in = -1;
        r->post_act = -1;
        switch (l->type) {
        case CONVOLUTIONAL: {
            /* 1x1 and 3x3 stride-1 'same' layers run on the shifted-descriptor kernels; every other
             * size / stride / padding goes through a patch gather + 1x1 GEMM (use_patches) */
            const int native = l->stride == 1 && (l->size == 1 || l->size == 3) && l->pad == l->size / 2;
            if (l->stride < 1 || l->size < 1 || l->out_h < 1 || l->out_w < 1) unsupported(i, "degenerate convolution");
            r->post_act = (l->activation != LEAKY && l->activation != LINEAR && l->activation != LOGISTIC)
                              ? (int)l->activation : -1;
            if (l->binary || l->xnor) unsupported(i, "binary/xnor convolution");
            r->out_kind = consumer_wants_f32(net, i) ? Y2_KIND_F32_FLAT : Y2_KIND_BF16_PADDED;
            r->cpad = (r->out_kind == Y2_KIND_F32_FLAT) ? l->n : storage_channels(l->n);
            /* a reorg permutes flat NCHW indices, so its input must be stored without channel
             * padding; 8-channel granularity keeps the 16-byte stores */
            if (i + 1 < net->n && net->layers[i + 1].type == REORG && l->n % 8 == 0) r->cpad = l->n;
            r->block_n = pick_block_n(l->n);
            r->npad = round_up(l->n, r->block_n);
            if (r->cpad > r->npad) r->npad = round_up(r->cpad, r->block_n);
            const int kk = l->size * l->size;
            if (!native) {
                if (i == 0 && l->size >= 5 && l->size <= 8) {
                    r->use_patches = 3; /* K = (c*k + r)*8 + s: one aligned 16-byte group per kernel row */
                    r->kpad = round_up(l->c * l->size * 8, 64);
                    r->cin_pad = r->kpad;
                } else if (i == 0) {
                    r->use_patches = 1; /* K = c*k*k + r*k + s, zero-padded to a K block */
                    r->kpad = (l->c * kk <= 32) ? 32 : round_up(l->c * kk, 64);
                    r->cin_pad = r->kpad;
                } else {
                    y2_layer_rt *pr = (y2_layer_rt *)net->layers[i - 1].b200;
                    if (pr->out_kind != Y2_KIND_BF16_PADDED) unsupported(i, "convolution after a flat layer");
                    r->use_patches = 2; /* K = tap*cin_pad + c, the order the weights are packed in anyway */
                    r->cin_pad = pr->cpad;
                    r->kpad = kk * pr->cpad;
                }
                r->ktot = r->kpad;
                r->block_k = (r->kpad % 64 == 0) ? 64 : 32;
            } else if (i == 0 && l->c * kk <= 64 && l->size == 3) {
                r->use_patches = 1;
                r->kpad = (l->c * kk <= 32) ? 32 : 64;
                r->ktot = r->kpad;
                r->block_k = r->kpad == 32 ? 32 : 64;
                r->cin_pad = r->kpad;
                r->stem_fused = stem_fusable(net, i);
            } else {
                int cin_pad;
                if (i == 0) cin_pad = storage_channels(l->c);
                else {
                    y2_layer_rt *pr = (y2_layer_rt *)net->layers[i - 1].b200;
                    if (pr->out_kind != Y2_KIND_BF16_PADDED) unsupported(i, "convolution after a flat layer");
                    cin_pad = pr->cpad;
                }
                r->cin_pad = cin_pad;
                r->block_k = (cin_pad % 64 == 0) ? 64 : 32;
                r->ktot = kk * cin_pad;
                r->pool_fused = r->out_kind == Y2_KIND_BF16_PADDED && r->cpad == l->n && pool_fusable(net, i, cin_pad);
            }
            /* 32-channel K blocks (a first layer, or a layer behind a 32-channel tensor) have no 256-filter tile in
             * the GEMM kernels that take 1x1 / gathered operands: use two 128-filter tiles */
            if (r->block_k == 32 && r->block_n == 256 && (l->size == 1 || r->use_patches)) {
                r->block_n = 128;
                r->npad = round_up(l->n > r->cpad ? l->n : r->cpad, 128);
            }
            break;
        }
        case MAXPOOL:
        case REORG: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            if (!pr || pr->out_kind != Y2_KIND_BF16_PADDED) unsupported(i, "maxpool/reorg without a tensor input");
            if (l->type == REORG && l->reverse && (l->out_c % 8 || l->c % (l->stride * l->stride)))
                unsupported(i, "reverse reorg to a channel count that is not a multiple of 8");
            r->out_kind = Y2_KIND_BF16_PADDED;
            if (l->type == MAXPOOL && (pr->stem_fused || pr->pool_fused)) r->fused_into_prev = 1;
            if (l->type == MAXPOOL) r->cpad = pr->cpad;
            else {
                if (pr->cpad != l->c) unsupported(i, "reorg of a channel-padded tensor");
                /* depth-to-space shrinks the channel count: store it like any tensor (padding channels stay zero) */
                r->cpad = l->reverse ? storage_channels(l->out_c) : l->out_c;
            }
            break;
        }
        case SHORTCUT: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            y2_layer_rt *fr = (y2_layer_rt *)net->layers[l->index].b200;
            if (!pr || pr->out_kind != Y2_KIND_BF16_PADDED || !fr || fr->out_kind != Y2_KIND_BF16_PADDED)
                unsupported(i, "shortcut between non-tensor layers");
            if (l->activation != LEAKY && l->activation != LINEAR && l->activation != LOGISTIC)
                unsupported(i, "activation other than leaky/linear/logistic");
            r->out_kind = Y2_KIND_BF16_PADDED;
            r->cpad = pr->cpad;
            break;
        }
        case ROUTE: {
            r->out_kind = Y2_KIND_BF16_PADDED;
            int total = 0, total_real = 0, padded = 0;
            for (int k = 0; k < l->n; ++k) {
                y2_layer_rt *ir = (y2_layer_rt *)net->layers[l->input_layers[k]].b200;
                const int real_c = net->layers[l->input_layers[k]].out_c;
                if (ir->out_kind != Y2_KIND_BF16_PADDED) unsupported(i, "route from a flat layer");
                if (l->n > 1 && ir->cpad != real_c) padded = 1;
                total += ir->cpad;
                total_real += real_c;
            }
            if (!l->out_w || !l->out_h) unsupported(i, "route over mismatched extents");
            r->cpad = total;
            if (padded) {
                /* an input stores more channels than it has (48 -> 64): the reference's concat has no holes
                 * (route_layer.c:73-86), so the real channels are packed next to each other by copies instead of
                 * being written in place; the tail of the buffer up to the storage granularity stays zero */
                for (int k = 0; k < l->n; ++k)
                    if (net->layers[l->input_layers[k]].out_c % 8)
                        unsupported(i, "concat of tensors whose channel count is not a multiple of 8");
                r->cpad = storage_channels(total_real);
                r->packed_concat = 1;
                r->copy_needed = (1 << l->n) - 1;
            } else if (l->n > 1) {
                /* claim the producers: they will write into this layer's concat buffer */
                for (int k = 0; k < l->n; ++k) {
                    int src = l->input_layers[k];
                    y2_layer_rt *ir = (y2_layer_rt *)net->layers[src].b200;
                    LAYER_TYPE st = net->layers[src].type;
                    int claimable = (st == CONVOLUTIONAL || st == MAXPOOL || st == REORG) && ir->placed_in < 0;
                    for (int q = 0; q < k; ++q)
                        if (l->input_layers[q] == src) claimable = 0;
                    if (claimable) ir->placed_in = i;
                    else r->copy_needed |= (1 << k);
                }
            }
            break;
        }
        case REGION: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            if (!pr || pr->out_kind != Y2_KIND_F32_FLAT) unsupported(i, "region layer without a conv head");
            if (l->coords != 4) unsupported(i, "region layer with coords != 4");
            r->out_kind = Y2_KIND_F32_FLAT;
            r->cpad = l->n * (l->classes + 5);
            break;
        }
        case AVGPOOL: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            if (!pr || pr->out_kind != Y2_KIND_F32_FLAT) unsupported(i, "avgpool without a conv head");
            r->out_kind = Y2_KIND_F32_VEC;
            r->cpad = l->c;
            break;
        }
        case SOFTMAX: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            if (!pr || pr->out_kind != Y2_KIND_F32_VEC) unsupported(i, "softmax without a vector input");
            if (l->softmax_tree && l->softmax_tree->n != l->inputs / l->groups)
                unsupported(i, "softmax tree whose size differs from the layer's inputs");
            r->out_kind = Y2_KIND_F32_VEC;
            r->cpad = l->inputs;
            break;
        }
        case CONNECTED: {
            /* the tensor (or vector) this layer flattens: the previous layer, looking through dropout layers */
            int src = i - 1;
            while (src >= 0 && net->layers[src].type == DROPOUT) --src;
            if (src < 0) unsupported(i, "connected layer without an input layer");
            y2_layer_rt *sr = (y2_layer_rt *)net->layers[src].b200;
            layer *sl = &net->layers[src];
            r->fc_src = src;
            if (sr->out_kind == Y2_KIND_BF16_PADDED) {
                r->fc_h = sl->out_h;
                r->fc_w = sl->out_w;
                r->fc_c = sl->out_c;
                if (l->inputs != sl->out_h * sl->out_w * sl->out_c) unsupported(i, "connected layer input size");
            } else if (sr->out_kind == Y2_KIND_F32_VEC) {
                r->fc_c = l->inputs;
                if (l->inputs != sr->cpad) unsupported(i, "connected layer input size");
            } else {
                unsupported(i, "connected layer behind a flat head");
            }
            r->post_act = (l->activation != LEAKY && l->activation != LINEAR && l->activation != LOGISTIC)
                              ? (int)l->activation : -1;
            r->out_kind = Y2_KIND_F32_VEC;
            r->cpad = l->outputs;
            r->block_n = pick_block_n(l->outputs);
            r->npad = round_up(l->outputs, r->block_n);
            r->kpad = round_up(l->inputs, 64);
            r->cin_pad = r->kpad;
            r->ktot = r->kpad;
            r->block_k = 64;
            break;
        }
        case DROPOUT: {
            y2_layer_rt *pr = i ? (y2_layer_rt *)net->layers[i - 1].b200 : 0;
            if (!pr) unsupported(i, "dropout without an input layer");
            r->out_kind = pr->out_kind; /* identity at inference: aliases its input (resolved in pass 3) */
            r->cpad = pr->cpad;
            break;
        }
        case COST:
            r->out_kind = Y2_KIND_NONE;
            break;
        default:
            unsupported(i, get_layer_string(l->type));
        }
    }

    /* pass 2: allocate outputs (placed producers get a slice of their route's buffer) */
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        y2_layer_rt *r = (y2_layer_rt *)l->b200;
        if (l->type == ROUTE) {
            if (l->n == 1) {
                y2_layer_rt *ir = (y2_layer_rt *)net->layers[l->input_layers[0]].b200;
                r->out = 0; /* resolved in pass 3 (the producer may itself be placed later) */
                (void)ir;
            } else {
                r->own_bytes = padded_bytes(B, l->out_h, l->out_w, r->cpad);
                r->own_buf = dev_alloc_zero(r->own_bytes);
                r->out = r->own_buf;
                r->out_cs = r->cpad;
            }
        }
    }
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        y2_layer_rt *r = (y2_layer_rt *)l->b200;
        if (l->type == ROUTE || l->type == DROPOUT || r->out_kind == Y2_KIND_NONE) continue;
        if (r->stem_fused || r->pool_fused) { /* the full-resolution activation is never materialised */
            r->out = 0;
            r->out_cs = r->cpad;
            continue;
        }
        if (r->placed_in >= 0) {
            layer *rl = &net->layers[r->placed_in];
            y2_layer_rt *rr = (y2_layer_rt *)rl->b200;
            int off = 0;
            for (int k = 0; k < rl->n && rl->input_layers[k] != i; ++k)
                off += ((y2_layer_rt *)net->layers[rl->input_layers[k]].b200)->cpad;
            r->out = (char *)rr->own_buf + (size_t)off * 2;
            r->out_cs = rr->cpad;
            continue;
        }
        if (r->out_kind == Y2_KIND_BF16_PADDED) {
            r->own_bytes = padded_bytes(B, l->out_h, l->out_w, r->cpad);
            r->out_cs = r->cpad;
        } else if (r->out_kind == Y2_KIND_F32_FLAT) {
            const int oh = l->type == REGION ? l->h : l->out_h, ow = l->type == REGION ? l->w : l->out_w;
            /* conv heads: rows padded to 16 bytes so that the epilogue can store them with 16-byte accesses */
            r->out_cs = (l->type == CONVOLUTIONAL) ? round_up(r->cpad, 4) : r->cpad;
            r->own_bytes = (size_t)B * oh * ow * r->out_cs * sizeof(float);
        } else {
            r->own_bytes = (size_t)B * r->cpad * sizeof(float);
            r->out_cs = r->cpad;
        }
        r->own_buf = dev_alloc_zero(r->own_bytes);
        r->out = r->own_buf;
    }
    /* pass 3: single-input routes alias their producer */
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        y2_layer_rt *r = (y2_layer_rt *)l->b200;
        if (l->type == ROUTE && l->n == 1) {
            y2_layer_rt *ir = (y2_layer_rt *)net->layers[l->input_layers[0]].b200;
            r->out = ir->out;
            r->out_cs = ir->out_cs;
        }
        if (l->type == DROPOUT) { /* layers are visited in order: the input's view is final */
            y2_layer_rt *pr = (y2_layer_rt *)net->layers[i - 1].b200;
            r->out = pr->out;
            r->out_cs = pr->out_cs;
        }
        l->output_gpu = (float *)r->out;
    }

    /* pass 4: layer-specific device state */
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        y2_layer_rt *r = (y2_layer_rt *)l->b200;
        if (l->type == CONVOLUTIONAL) {
            Y2_CHECK(y2_malloc(&r->wt_dev, (size_t)r->npad * r->ktot * 2));
            Y2_CHECK(y2_malloc((void **)&r->alpha_dev, (size_t)r->npad * 4));
            Y2_CHECK(y2_malloc((void **)&r->beta_dev, (size_t)r->npad * 4));
            l->weights_gpu = (float *)r->wt_dev;
            l->biases_gpu = r->beta_dev;
            l->scales_gpu = r->alpha_dev;
            if (r->stem_fused) Y2_CHECK(y2_stem_prepare());
            else if (r->use_patches) r->patches = dev_alloc_zero(padded_bytes(B, l->out_h, l->out_w, r->kpad));
            else if (i == 0) r->packed_in = dev_alloc_zero(padded_bytes(B, l->h, l->w, r->cin_pad));
            y2_push_convolutional_layer(l);
        } else if (l->type == CONNECTED) {
            Y2_CHECK(y2_malloc(&r->wt_dev, (size_t)r->npad * r->ktot * 2));
            Y2_CHECK(y2_malloc((void **)&r->alpha_dev, (size_t)r->npad * 4));
            Y2_CHECK(y2_malloc((void **)&r->beta_dev, (size_t)r->npad * 4));
            l->weights_gpu = (float *)r->wt_dev;
            l->biases_gpu = r->beta_dev;
            l->scales_gpu = r->alpha_dev;
            r->fc_in = dev_alloc_zero(padded_bytes(B, 1, 1, r->kpad));
            y2_push_convolutional_layer(l);
        } else if (l->type == SHORTCUT) {
            /* a later shortcut that adds this one's output reads it in fp32, so the residual stream is
             * not rounded to bf16 once per block (it would random-walk away over resnet50's 16 blocks) */
            for (int j = i + 1; j < net->n; ++j)
                if (net->layers[j].type == SHORTCUT && net->layers[j].index == i && !r->stream_f32)
                    r->stream_f32 = (float *)dev_alloc_zero((size_t)B * (l->out_h + 1) * (l->out_w + 1) * r->cpad * 4);
        } else if (l->type == REORG) {
            y2_layer_rt *pr = (y2_layer_rt *)net->layers[i - 1].b200;
            if (l->out_c % 8 == 0 && r->out_cs % 8 == 0) {
                Y2_CHECK(y2_malloc((void **)&r->reorg_table, (size_t)l->out_h * l->out_w * l->out_c * sizeof(int)));
                if (l->reverse) Y2_CHECK(y2_reorg_table_reverse(r->reorg_table, pr->out_cs, l->c, l->h, l->w, l->stride, 0));
                else Y2_CHECK(y2_reorg_table(r->reorg_table, pr->out_cs, l->c, l->h, l->w, l->stride, 0));
            } else if (l->reverse) {
                unsupported(i, "reverse reorg into an unaligned channel slice");
            }
        } else if (l->type == SOFTMAX && l->softmax_tree) {
            tree *t = l->softmax_tree;
            r->group_size_dev = (int *)dev_upload(t->group_size, (size_t)t->groups * sizeof(int));
            r->group_offset_dev = (int *)dev_upload(t->group_offset, (size_t)t->groups * sizeof(int));
            /* hierarchy_predictions of the classify entries walks parents before children and at most
             * Y2_CLASSIFY_MAX_TREE_DEPTH levels; the host path takes any tree, so another tree only leaves the
             * classify entries unavailable */
            int usable = 1;
            int *depth = (int *)calloc((size_t)t->n, sizeof(int));
            for (int j = 0; j < t->n && usable; ++j) {
                const int p = t->parent[j];
                if (p >= j) usable = 0;
                else depth[j] = p < 0 ? 1 : depth[p] + 1;
                if (depth[j] > Y2_CLASSIFY_MAX_TREE_DEPTH) usable = 0;
            }
            free(depth);
            if (usable) r->tree_parent_dev = (int *)dev_upload(t->parent, (size_t)t->n * sizeof(int));
        } else if (l->type == REGION) {
            const size_t total = (size_t)l->w * l->h * l->n;
            r->probs_classes = l->map ? 200 : l->classes;
            Y2_CHECK(y2_malloc((void **)&r->boxes_dev, (size_t)B * total * 4 * sizeof(float)));
            Y2_CHECK(y2_malloc((void **)&r->probs_dev, (size_t)B * total * l->classes * sizeof(float)));
            r->biases_dev = (float *)dev_upload(l->biases, (size_t)l->n * 2 * sizeof(float));
            r->nms_cnt_dev = (int *)dev_alloc_zero((size_t)B * l->classes * sizeof(int));
            if (y2_collect_ws_bytes(B, (int)total, l->classes))
                Y2_CHECK(y2_malloc(&r->collect_ws, y2_collect_ws_bytes(B, (int)total, l->classes)));
            if (l->softmax_tree) {
                tree *t = l->softmax_tree;
                if (t->n != l->classes) unsupported(i, "softmax tree whose size differs from classes");
                for (int j = 0; j < t->n; ++j)
                    if (t->parent[j] >= j) unsupported(i, "softmax tree with a parent after its child");
                r->tree_parent_dev = (int *)dev_upload(t->parent, (size_t)t->n * sizeof(int));
                r->group_size_dev = (int *)dev_upload(t->group_size, (size_t)t->groups * sizeof(int));
                r->group_offset_dev = (int *)dev_upload(t->group_offset, (size_t)t->groups * sizeof(int));
                /* groups below every node (a group = a run of consecutive nodes with one parent, tree.c:72-82) */
                int *cptr = (int *)calloc((size_t)t->n + 2, sizeof(int));
                int *cgrp = (int *)calloc((size_t)t->groups > 0 ? t->groups : 1, sizeof(int));
                for (int g = 0; g < t->groups; ++g) {
                    int par = t->parent[t->group_offset[g]];
                    ++cptr[(par < 0 ? t->n : par) + 1];
                }
                for (int j = 0; j <= t->n; ++j) cptr[j + 1] += cptr[j];
                int *fill = (int *)calloc((size_t)t->n + 1, sizeof(int));
                for (int g = 0; g < t->groups; ++g) {
                    int par = t->parent[t->group_offset[g]];
                    if (par < 0) par = t->n;
                    cgrp[cptr[par] + fill[par]++] = g;
                }
                r->child_ptr_dev = (int *)dev_upload(cptr, ((size_t)t->n + 2) * sizeof(int));
                r->child_grp_dev = (int *)dev_upload(cgrp, (size_t)(t->groups > 0 ? t->groups : 1) * sizeof(int));
                free(cptr);
                free(cgrp);
                free(fill);
                Y2_CHECK(y2_malloc(&r->tree_rec_dev, (size_t)B * total * y2_tree_rec_bytes()));
                rt->defer_region = 1;
            }
            if (l->map) r->map_dev = (int *)dev_upload(l->map, 200 * sizeof(int));
        }
    }
    /* host output of the network's output layer */
    int oi = y2_output_layer_index(*net);
    layer *ol = &net->layers[oi];
    if (!ol->output) ol->output = (float *)calloc((size_t)B * ol->outputs, sizeof(float));
    rt->out_bytes = (size_t)B * ol->outputs * sizeof(float);
    Y2_CHECK(y2_host_alloc((void **)&rt->out_pinned, rt->out_bytes));
    build_plans(net, B);
    Y2_CHECK(y2_device_sync());
}

/* ---- layer forwards (function-pointer targets, as layer.h:48-53) -------------------------------- */
static y2_stream_t net_stream(network net)
{
    y2_net_rt *rt = y2_rt(net);
    return rt ? rt->stream : 0;
}

static void count_launch(network net, int n)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt) rt->launches += n;
}

void forward_convolutional_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_stream_t s = net_stream(state.net);
    if (r->stem_fused) {
        y2_layer_rt *mr = y2_lrt(state.net.layers[state.index + 1]);
        const int act = (l.activation == LEAKY) ? Y2_ACT_LEAKY : Y2_ACT_LINEAR;
        if (y2_rt(state.net)->input_u8)
            Y2_CHECK(y2_stem_conv_pool_u8((const unsigned char *)state.input, l.batch, l.h, l.w, r->wt_dev, r->npad,
                                          r->alpha_dev, r->beta_dev, act, mr->out, mr->out_cs, s));
        else
            Y2_CHECK(y2_stem_conv_pool(state.input, l.batch, l.c, l.h, l.w, r->wt_dev, r->npad, r->alpha_dev,
                                       r->beta_dev, act, mr->out, mr->out_cs, s));
        count_launch(state.net, 1);
        return;
    }
    if (r->use_patches == 2) {
        y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
        Y2_CHECK(y2_gather_patches_bf16(pr->out, pr->out_cs, r->cin_pad, l.h, l.w, r->patches, l.batch, l.size,
                                        l.stride, l.pad, l.out_h, l.out_w, s));
        count_launch(state.net, 1);
    } else if (r->use_patches == 3) {
        Y2_CHECK(y2_gather_rows_f32(state.input, r->patches, l.batch, l.c, l.h, l.w, l.size, l.stride, l.pad, l.out_h,
                                    l.out_w, r->kpad, s));
        count_launch(state.net, 1);
    } else if (r->use_patches) {
        Y2_CHECK(y2_gather_patches_f32(state.input, r->patches, l.batch, l.c, l.h, l.w, l.size, l.stride, l.pad,
                                       l.out_h, l.out_w, r->kpad, s));
        count_launch(state.net, 1);
    } else if (r->packed_in) {
        Y2_CHECK(y2_pack_nchw_f32(state.input, r->packed_in, l.batch, l.c, l.h, l.w, r->cin_pad, r->cin_pad, s));
        count_launch(state.net, 1);
    }
    Y2_CHECK(y2_conv_plan_launch(r->plan, s));
    count_launch(state.net, 1);
    if (r->post_act >= 0) { /* an activation the epilogue does not implement: the plan ran LINEAR */
        if (r->out_kind == Y2_KIND_F32_FLAT)
            Y2_CHECK(y2_vec_activate((float *)r->out, (long long)l.batch * l.out_h * l.out_w * r->out_cs, r->post_act, s));
        else
            Y2_CHECK(y2_activate_bf16(r->out, r->out_cs, l.out_c, l.batch, l.out_h, l.out_w, r->post_act, s));
        count_launch(state.net, 1);
    }
}

/* connected_layer.c:271-293 as a 1x1 convolution: flatten the input into one position per image, run the plan */
void forward_connected_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_stream_t s = net_stream(state.net);
    y2_layer_rt *sr = y2_lrt(state.net.layers[r->fc_src]);
    if (r->fc_h > 0)
        Y2_CHECK(y2_fc_pack_tensor(sr->out, sr->out_cs, r->fc_c, r->fc_h, r->fc_w, r->fc_in, r->kpad, l.batch, s));
    else
        Y2_CHECK(y2_fc_pack_vec((const float *)sr->out, sr->out_cs, r->fc_c, r->fc_in, r->kpad, l.batch, s));
    Y2_CHECK(y2_conv_plan_launch(r->plan, s));
    count_launch(state.net, 2);
    if (r->post_act >= 0) {
        Y2_CHECK(y2_vec_activate((float *)r->out, (long long)l.batch * r->out_cs, r->post_act, s));
        count_launch(state.net, 1);
    }
}

void forward_dropout_layer_gpu(layer l, network_state state)
{
    (void)l;
    (void)state; /* dropout_layer.c:40: if (!state.train) return; */
}

void forward_maxpool_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    if (r->fused_into_prev) return; /* the convolution before it already wrote this layer's output */
    Y2_CHECK(y2_maxpool(pr->out, pr->out_cs, r->out, r->out_cs, l.batch, r->cpad, l.h, l.w, l.out_h, l.out_w,
                        l.size, l.stride, l.pad, net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_reorg_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    if (r->reorg_table && l.reverse)
        Y2_CHECK(y2_reorg_gather_reverse(pr->out, pr->out_cs, r->out, r->out_cs, r->reorg_table, l.batch, l.c, l.h, l.w,
                                         l.stride, net_stream(state.net)));
    else if (r->reorg_table)
        Y2_CHECK(y2_reorg_gather(pr->out, pr->out_cs, r->out, r->out_cs, r->reorg_table, l.batch, l.c, l.h, l.w,
                                 l.stride, net_stream(state.net)));
    else
        Y2_CHECK(y2_reorg(pr->out, pr->out_cs, r->out, r->out_cs, l.batch, l.c, l.h, l.w, l.stride,
                          net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_route_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    if (l.n == 1 || !r->copy_needed) return; /* producers already wrote in place */
    int off = 0;
    for (int k = 0; k < l.n; ++k) {
        layer src = state.net.layers[l.input_layers[k]];
        y2_layer_rt *ir = y2_lrt(src);
        const int nch = r->packed_concat ? src.out_c : ir->cpad;  /* packed: real channels only */
        if (r->copy_needed & (1 << k)) {
            Y2_CHECK(y2_copy_channels(ir->out, ir->out_cs, (char *)r->out + (size_t)off * 2, r->out_cs, l.batch,
                                      nch, l.out_h, l.out_w, net_stream(state.net)));
            count_launch(state.net, 1);
        }
        off += nch;
    }
}

void forward_region_layer_gpu(const layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    y2_net_rt *rt = y2_rt(state.net);
    if (rt && rt->defer_region && !rt->profile) {
        /* 9418-way softmax tree: the detection entries read the head output directly (y2_region_tree_detect);
         * the dense softmax runs when the layer's output is asked for (export_layer) */
        rt->region_stale = 1;
        return;
    }
    int groups = 0;
    if (l.softmax_tree) groups = l.softmax_tree->groups;
    Y2_CHECK(y2_region_forward_strided((const float *)pr->out, pr->out_cs, (float *)r->out, l.batch, l.w * l.h, l.n,
                                       l.classes, l.softmax || l.softmax_tree, groups, r->group_size_dev,
                                       r->group_offset_dev, net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_avgpool_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    Y2_CHECK(y2_avgpool_flat((const float *)pr->out, (float *)r->out, l.batch, l.h * l.w, l.c, pr->out_cs,
                             net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_softmax_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    const int n = l.inputs / l.groups;
    if (l.softmax_tree)
        Y2_CHECK(y2_softmax_tree_rows((const float *)pr->out, (float *)r->out, l.batch * l.groups, n, l.temperature,
                                      l.softmax_tree->groups, r->group_size_dev, r->group_offset_dev,
                                      net_stream(state.net)));
    else
        Y2_CHECK(y2_softmax_rows((const float *)pr->out, (float *)r->out, l.batch * l.groups, n, l.temperature,
                                 net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_shortcut_layer_gpu(layer l, network_state state)
{
    y2_layer_rt *r = y2_lrt(l);
    y2_layer_rt *pr = y2_lrt(state.net.layers[state.index - 1]);
    y2_layer_rt *fr = y2_lrt(state.net.layers[l.index]);
    const int act = (l.activation == LEAKY) ? Y2_ACT_LEAKY : (l.activation == LOGISTIC) ? Y2_ACT_LOGISTIC : Y2_ACT_LINEAR;
    /* (l.w, l.h, l.c) describe the `from` tensor, out_* the running one (shortcut_layer.c:7-34) */
    Y2_CHECK(y2_shortcut(pr->out, pr->out_cs, fr->out, fr->out_cs, l.c, l.h, l.w, r->out, r->out_cs, l.out_c,
                         r->cpad, l.out_h, l.out_w, l.batch, act, fr->stream_f32, fr->cpad, r->stream_f32,
                         net_stream(state.net)));
    count_launch(state.net, 1);
}

void forward_cost_layer_gpu(layer l, network_state state)
{
    (void)l;
    (void)state; /* cost_layer.c:75: if(!state.truth) return; */
}

/* ---- schedule ------------------------------------------------------------------------------------ */
void forward_network(network net, network_state state)
{
    (void)net;
    (void)state;
    error("yolo2-b200 has no CPU execution path (gpu_index must be >= 0)");
}

/* network_kernels.cu:43-56 without the per-layer fill_ongpu(delta) */
void forward_network_gpu(network net, network_state state)
{
    y2_net_rt *rt = y2_rt(net);
    state.workspace = net.workspace;
    for (int i = 0; i < net.n; ++i) {
        state.index = i;
        layer l = net.layers[i];
        y2_layer_rt *r = y2_lrt(l);
        if (rt->profile && r) {
            if (!r->ev0) {
                Y2_CHECK(y2_event_create(&r->ev0));
                Y2_CHECK(y2_event_create(&r->ev1));
            }
            Y2_CHECK(y2_event_record(r->ev0, rt->stream));
        }
        l.forward_gpu(l, state);
        if (rt->profile && r) Y2_CHECK(y2_event_record(r->ev1, rt->stream));
        if (l.output_gpu) state.input = l.output_gpu;
    }
}

static void ensure_ready(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network has no device plan (gpu_index < 0 at parse time?)");
    Y2_CHECK(y2_set_device(rt->device));
    if (net.batch > rt->cap_batch) error("network batch exceeds the planned capacity; call set_batch_network");
    if (net.batch != rt->plan_batch) error("network batch changed without set_batch_network");
}

/* forward pass reading the fp32 NCHW batch at in_dev; the layer list is captured once per input
 * buffer into *graph and replayed afterwards */
void y2_run_forward_from(network net, float *in_dev, y2_graph_t *graph, int *graph_valid)
{
    y2_net_rt *rt = y2_rt(net);
    network_state state;
    memset(&state, 0, sizeof(state));
    state.net = net;
    state.input = in_dev;
    if (rt->eager || rt->profile) {
        rt->launches = 0;
        forward_network_gpu(net, state);
        return;
    }
    if (!*graph_valid) {
        rt->launches = 0;
        Y2_CHECK(y2_graph_begin(rt->stream));
        forward_network_gpu(net, state);
        Y2_CHECK(y2_graph_end(rt->stream, graph));
        *graph_valid = 1;
    }
    Y2_CHECK(y2_graph_launch(*graph, rt->stream));
    if (rt->defer_region) rt->region_stale = 1;
}

static void run_forward(network net)
{
    y2_net_rt *rt = y2_rt(net);
    y2_run_forward_from(net, rt->pipe[0].in_dev, &rt->pipe[0].graph, &rt->pipe[0].graph_valid);
}

void network_set_eager(network net, int eager)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt) rt->eager = eager;
}

int network_launch_count(network net)
{
    y2_net_rt *rt = y2_rt(net);
    return rt ? rt->launches : 0;
}

/* kernel behind layer i: 0 per-tap, 1 halo slab, 2 CTA pair, 3 conv + maxpool, 4 fused first layer,
 * -1 not a convolution */
int network_conv_kernel(network net, int i)
{
    if (i < 0 || i >= net.n || net.layers[i].type != CONVOLUTIONAL) return -1;
    y2_layer_rt *r = y2_lrt(net.layers[i]);
    if (!r) return -1;
    if (r->stem_fused) return 4;
    return r->plan ? y2_conv_plan_variant(r->plan) : -1;
}

void *network_stream(network net)
{
    return net_stream(net);
}

void network_sync(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt) Y2_CHECK(y2_stream_sync(rt->stream));
}

float *network_input_staging(network net)
{
    y2_net_rt *rt = y2_rt(net);
    return rt ? rt->pipe[0].in_pinned : 0;
}

float *network_input_device(network net)
{
    y2_net_rt *rt = y2_rt(net);
    return rt ? rt->pipe[0].in_dev : 0;
}

void network_upload_input(network net, const float *input)
{
    ensure_ready(net);
    y2_net_rt *rt = y2_rt(net);
    const size_t bytes = (size_t)net.batch * net.inputs * sizeof(float);
    /* caller memory is pageable in the reference API: stage through the pinned buffer, unless the
     * caller already filled the staging buffer itself (network_input_staging) */
    if (input && input != rt->pipe[0].in_pinned) {
        Y2_CHECK(y2_stream_sync(rt->stream));
        memcpy(rt->pipe[0].in_pinned, input, bytes);
    }
    Y2_CHECK(y2_memcpy_h2d(rt->pipe[0].in_dev, rt->pipe[0].in_pinned, bytes, rt->stream));
}

/* struct sizes for language bindings that pass network/layer by value (ctypes, cgo ...) */
size_t y2_abi_sizeof(int what)
{
    switch (what) {
    case 0: return sizeof(layer);
    case 1: return sizeof(network);
    case 2: return sizeof(network_state);
    case 3: return sizeof(y2_detection);
    case 4: return sizeof(box);
    case 5: return sizeof(y2_class_hit);
    case 6: return sizeof(y2_bbox);
    case 7: return sizeof(y2_frame_desc);
    case 8: return sizeof(y2_tiling);
    default: return 0;
    }
}

void network_forward_device(network net)
{
    ensure_ready(net);
    run_forward(net);
}

int network_profile_layers(network net, float *ms_per_layer, int n)
{
    ensure_ready(net);
    y2_net_rt *rt = y2_rt(net);
    rt->profile = 1;
    run_forward(net);
    Y2_CHECK(y2_stream_sync(rt->stream));
    rt->profile = 0;
    int m = n < net.n ? n : net.n;
    for (int i = 0; i < m; ++i) {
        y2_layer_rt *r = y2_lrt(net.layers[i]);
        ms_per_layer[i] = 0.f;
        if (r && r->ev0) Y2_CHECK(y2_event_elapsed_ms(r->ev0, r->ev1, &ms_per_layer[i]));
    }
    return m;
}

/* device tensor of layer i -> reference layout on the host (fp32 NCHW, or as-is for flat kinds) */
static float *export_layer(network net, int i)
{
    y2_net_rt *rt = y2_rt(net);
    layer *l = &net.layers[i];
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (!r || r->out_kind == Y2_KIND_NONE) return l->output;
    const size_t n = (size_t)net.batch * l->outputs;
    if (!l->output) l->output = (float *)calloc((size_t)rt->cap_batch * l->outputs, sizeof(float));
    if (rt->export_bytes < n * sizeof(float)) {
        y2_free(rt->export_dev);
        rt->export_bytes = n * sizeof(float);
        Y2_CHECK(y2_malloc((void **)&rt->export_dev, rt->export_bytes));
    }
    const float *src = rt->export_dev;
    if (l->type == REGION && rt->defer_region && rt->region_stale) {
        y2_layer_rt *pr = (y2_layer_rt *)net.layers[i - 1].b200;
        Y2_CHECK(y2_region_forward_strided((const float *)pr->out, pr->out_cs, (float *)r->out, net.batch, l->w * l->h,
                                           l->n, l->classes, l->softmax || l->softmax_tree,
                                           l->softmax_tree ? l->softmax_tree->groups : 0, r->group_size_dev,
                                           r->group_offset_dev, rt->stream));
        rt->region_stale = 0;
    }
    if (r->stem_fused) {
        /* inspection path: the fused kernel never stores this activation, so recompute it with the
         * generic patch-gather + convolution kernels into scratch buffers */
        void *patches = dev_alloc_zero(padded_bytes(net.batch, l->h, l->w, r->kpad));
        void *full = dev_alloc_zero(padded_bytes(net.batch, l->out_h, l->out_w, r->cpad));
        y2_conv_desc d;
        memset(&d, 0, sizeof(d));
        d.in = patches; d.in_cs = r->kpad; d.cin = r->kpad; d.ksize = 1;
        d.batch = net.batch; d.h = l->out_h; d.w = l->out_w;
        d.wt = r->wt_dev; d.cout = r->cpad; d.npad = r->npad; d.block_n = r->block_n; d.block_k = r->block_k;
        d.alpha = r->alpha_dev; d.beta = r->beta_dev;
        d.act = (l->activation == LEAKY) ? Y2_ACT_LEAKY : Y2_ACT_LINEAR;
        d.out = full; d.out_cs = r->cpad; d.out_mode = Y2_OUT_BF16_PADDED;
        y2_conv_plan *plan = 0;
        Y2_CHECK(y2_conv_plan_create(&d, &plan));
        Y2_CHECK(y2_pack_patches_f32(rt->pipe[0].in_dev, patches, net.batch, l->c, l->h, l->w, l->size, r->kpad,
                                     rt->stream));
        Y2_CHECK(y2_conv_plan_launch(plan, rt->stream));
        Y2_CHECK(y2_unpack_to_nchw_f32(full, rt->export_dev, net.batch, l->out_c, l->out_h, l->out_w, r->cpad,
                                       rt->stream));
        Y2_CHECK(y2_stream_sync(rt->stream));
        y2_conv_plan_destroy(plan);
        y2_free(patches);
        y2_free(full);
    } else if (r->pool_fused) {
        /* inspection path: the conv+pool kernel never stores the full-resolution activation, recompute it
         * from the (still resident) input with the plain convolution kernel into a scratch buffer */
        void *full = dev_alloc_zero(padded_bytes(net.batch, l->out_h, l->out_w, r->cpad));
        y2_view v = input_view(&net, i);
        y2_conv_desc d;
        memset(&d, 0, sizeof(d));
        d.in = v.ptr; d.in_cs = v.cs; d.cin = r->cin_pad; d.ksize = l->size;
        d.batch = net.batch; d.h = l->out_h; d.w = l->out_w;
        d.wt = r->wt_dev; d.cout = r->cpad; d.npad = r->npad; d.block_n = r->block_n; d.block_k = r->block_k;
        d.alpha = r->alpha_dev; d.beta = r->beta_dev;
        d.act = (l->activation == LEAKY) ? Y2_ACT_LEAKY : Y2_ACT_LINEAR;
        d.out = full; d.out_cs = r->cpad; d.out_mode = Y2_OUT_BF16_PADDED;
        y2_conv_plan *plan = 0;
        Y2_CHECK(y2_conv_plan_create(&d, &plan));
        Y2_CHECK(y2_conv_plan_launch(plan, rt->stream));
        Y2_CHECK(y2_unpack_to_nchw_f32(full, rt->export_dev, net.batch, l->out_c, l->out_h, l->out_w, r->cpad,
                                       rt->stream));
        Y2_CHECK(y2_stream_sync(rt->stream));
        y2_conv_plan_destroy(plan);
        y2_free(full);
    } else if (r->out_kind == Y2_KIND_BF16_PADDED) {
        Y2_CHECK(y2_unpack_to_nchw_f32(r->out, rt->export_dev, net.batch, l->out_c, l->out_h, l->out_w, r->out_cs,
                                       rt->stream));
    } else if (r->out_kind == Y2_KIND_F32_FLAT && l->type == CONVOLUTIONAL) {
        Y2_CHECK(y2_flat_to_nchw_f32((const float *)r->out, rt->export_dev, net.batch, l->out_c,
                                     l->out_h * l->out_w, r->out_cs, rt->stream));
    } else {
        src = (const float *)r->out; /* region / avgpool / softmax outputs already match */
    }
    Y2_CHECK(y2_memcpy_d2h(l->output, src, n * sizeof(float), rt->stream));
    Y2_CHECK(y2_stream_sync(rt->stream));
    return l->output;
}

float *get_network_output_gpu_layer(network net, int i)
{
    return export_layer(net, i);
}

/* the reference's header and definition disagree on the name (network.h:84 vs network_kernels.cu:378): both exist */
float *get_network_output_layer_gpu(network net, int i)
{
    return export_layer(net, i);
}

float *get_network_output_layer(network net, int i)
{
    if (net.b200) return export_layer(net, i);
    return net.layers[i].output;
}

float *get_network_output_gpu(network net)
{
    return export_layer(net, y2_output_layer_index(net));
}

float *get_network_output(network net)
{
    int i = y2_output_layer_index(net);
    return net.layers[i].output;
}

float *network_predict_gpu(network net, float *input)
{
    network_upload_input(net, input);
    run_forward(net);
    return get_network_output_gpu(net);
}

float *network_predict(network net, float *input)
{
    if (gpu_index < 0 || !net.b200) error("yolo2-b200 has no CPU execution path (gpu_index must be >= 0)");
    return network_predict_gpu(net, input);
}

/* network.c:308-320 rewrites the batch fields only; here the plans follow, and growing past the
 * planned capacity re-plans instead of overflowing. */
void set_batch_network(network *net, int b)
{
    y2_net_rt *rt = (y2_net_rt *)net->b200;
    net->batch = b;
    for (int i = 0; i < net->n; ++i) net->layers[i].batch = b;
    if (!rt) return;
    Y2_CHECK(y2_set_device(rt->device));
    Y2_CHECK(y2_stream_sync(rt->stream));
    if (b > rt->cap_batch) {
        int oi = y2_output_layer_index(*net);
        free(net->layers[oi].output);
        net->layers[oi].output = 0;
        for (int i = 0; i < net->n; ++i)
            if (i != oi && net->layers[i].output) {
                free(net->layers[i].output);
                net->layers[i].output = 0;
            }
        y2_plan_network(net);
        net->output = get_network_output(*net);
    } else if (b != rt->plan_batch) {
        build_plans(net, b);
    }
}

/* network.c:322-388: recompute every layer's extent for a new input size and re-plan */
int resize_network(network *net, int w, int h)
{
    net->w = w;
    net->h = h;
    net->inputs = w * h * net->c;
    int c = net->c;
    for (int i = 0; i < net->n; ++i) {
        layer *l = &net->layers[i];
        switch (l->type) {
        case CONVOLUTIONAL: resize_convolutional_layer(l, w, h); break;
        case MAXPOOL: resize_maxpool_layer(l, w, h); break;
        case REGION: resize_region_layer(l, w, h); break;
        case ROUTE: resize_route_layer(l, net); break;
        case REORG: resize_reorg_layer(l, w, h); break;
        case AVGPOOL: resize_avgpool_layer(l, w, h); break;
        case COST:
        case SOFTMAX:
            break;
        default:
            fprintf(stderr, "Resizing type %d \n", (int)l->type);
            error("Cannot resize this type of layer");
        }
        if (l->output) {
            free(l->output);
            l->output = 0;
        }
        w = l->out_w;
        h = l->out_h;
        c = l->out_c;
        if (l->type == AVGPOOL) break;
    }
    (void)c;
    net->outputs = get_network_output_size(*net);
    if (net->gpu_index >= 0) y2_plan_network(net);
    else {
        int oi = y2_output_layer_index(*net);
        net->layers[oi].output = (float *)calloc((size_t)net->batch * net->layers[oi].outputs, sizeof(float));
    }
    net->output = get_network_output(*net);
    return 0;
}

void free_layer(layer l)
{
    free_layer_rt(&l);
    free(l.cost);
    free(l.biases);
    free(l.scales);
    free(l.weights);
    free(l.rolling_mean);
    free(l.rolling_variance);
    free(l.m);
    free(l.v);
    free(l.input_layers);
    free(l.input_sizes);
    free(l.output);
    free(l.map);
    if (l.softmax_tree) {
        tree *t = l.softmax_tree;
        for (int i = 0; i < t->n; ++i) free(t->name[i]);
        free(t->name);
        free(t->leaf);
        free(t->parent);
        free(t->group);
        free(t->group_size);
        free(t->group_offset);
        free(t);
    }
}

void free_network(network net)
{
    y2_unplan_network(&net); /* the network-level device state first, the layers below */
    for (int i = 0; i < net.n; ++i) free_layer(net.layers[i]);
    free(net.layers);
    free(net.seen);
    free(net.scales);
    free(net.steps);
    free(net.input_gpu);
    free(net.truth_gpu);
}
