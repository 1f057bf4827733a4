/*
 * Post-processing entry points of the drop-in API and the batched device-resident detection and
 * classification extensions.  The arithmetic runs in the region / NMS kernels; these functions only move the
 * caller-owned host arrays (boxes[total], probs[total][classes]) across, as the reference's
 * callers expect (detector.c:486-495, yolo_v2_class.cpp:71-73,215-216).
 *
 * Reference interfaces replaced: get_region_boxes (region_layer.c:328-379), do_nms_sort
 * (box.c:249-277), box_iou & friends (box.c:67-97); for classification, the tail of predict_classifier
 * (classifier.c:676-730: letterbox_image, hierarchy_predictions, top_k).
 */
#include "y2_host.h"

#include <stdlib.h>
#include <string.h>

_Static_assert(sizeof(y2_detection) == sizeof(y2_det), "y2_detection must mirror y2_det");

/* ---- box helpers (box.c:67-97), plain float arithmetic for API users ------------------------- */
static float overlap(float x1, float w1, float x2, float w2)
{
    float l1 = x1 - w1 / 2;
    float l2 = x2 - w2 / 2;
    float left = l1 > l2 ? l1 : l2;
    float r1 = x1 + w1 / 2;
    float r2 = x2 + w2 / 2;
    float right = r1 < r2 ? r1 : r2;
    return right - left;
}

float box_intersection(box a, box b)
{
    float w = overlap(a.x, a.w, b.x, b.w);
    float h = overlap(a.y, a.h, b.y, b.h);
    if (w < 0 || h < 0) return 0;
    return w * h;
}

float box_union(box a, box b)
{
    float i = box_intersection(a, b);
    return a.w * a.h + b.w * b.h - i;
}

float box_iou(box a, box b)
{
    return box_intersection(a, b) / box_union(a, b);
}

/* ---- scratch -------------------------------------------------------------------------------- */
typedef struct {
    void *dev;
    size_t dev_bytes;
    void *host;
    size_t host_bytes;
} scratch_t;

static void scratch_reserve(scratch_t *s, size_t bytes)
{
    if (s->dev_bytes < bytes) {
        y2_free(s->dev);
        Y2_CHECK(y2_malloc(&s->dev, bytes));
        s->dev_bytes = bytes;
    }
    if (s->host_bytes < bytes) {
        y2_host_free(s->host);
        Y2_CHECK(y2_host_alloc(&s->host, bytes));
        s->host_bytes = bytes;
    }
}

/* per host thread AND per device: a thread that drives several GPUs (Detector objects on different
 * gpu_ids) must not hand one device's scratch to another */
#define Y2_MAX_DEV 16
static __thread scratch_t g_pred_d[Y2_MAX_DEV], g_boxes_d[Y2_MAX_DEV], g_probs_d[Y2_MAX_DEV];
static int cur_dev(void)
{
    int dev = 0;
    Y2_CHECK(y2_get_device(&dev));
    if (dev < 0 || dev >= Y2_MAX_DEV) error("device index beyond the scratch table");
    return dev;
}
#define g_pred g_pred_d[cur_dev()]
#define g_boxes g_boxes_d[cur_dev()]
#define g_probs g_probs_d[cur_dev()]

/* region_layer.c:328-379.  Reads l.output on the HOST (callers may have replaced it, e.g. the
 * 3-frame mean of yolo_v2_class.cpp:208-213), decodes on the device, writes the caller's arrays.
 * In the tree case l.output is mutated exactly like the reference does. */
void get_region_boxes(layer l, int w, int h, float thresh, float **probs, box *boxes, int only_objectness,
                      int *map)
{
    y2_layer_rt *r = y2_lrt(l);
    if (!r || l.type != REGION) error("get_region_boxes: not a planned region layer");
    const int total = l.w * l.h * l.n;
    /* the 200-entry map is only read inside the softmax-tree branch (region_layer.c:349-356) */
    const int use_map = map && l.softmax_tree;
    const int out_classes = use_map ? 200 : l.classes;
    const size_t pred_bytes = (size_t)l.outputs * sizeof(float);
    scratch_reserve(&g_pred, pred_bytes);
    scratch_reserve(&g_boxes, (size_t)total * 4 * sizeof(float));
    scratch_reserve(&g_probs, (size_t)total * l.classes * sizeof(float));
    memcpy(g_pred.host, l.output, pred_bytes);
    Y2_CHECK(y2_memcpy_h2d(g_pred.dev, g_pred.host, pred_bytes, 0));
    int *map_dev = 0;
    if (use_map) {
        if (map == l.map && r->map_dev) map_dev = r->map_dev;
        else {
            Y2_CHECK(y2_malloc((void **)&map_dev, 200 * sizeof(int)));
            Y2_CHECK(y2_memcpy_h2d(map_dev, map, 200 * sizeof(int), 0));
        }
    }
    Y2_CHECK(y2_region_boxes((float *)g_pred.dev, r->biases_dev, (float *)g_boxes.dev, (float *)g_probs.dev, 1,
                             l.w, l.h, l.n, l.classes, (float)w, (float)h, thresh, only_objectness, l.classfix,
                             l.softmax_tree ? l.softmax_tree->n : 0, r->tree_parent_dev, map_dev, use_map ? 200 : 0,
                             0));
    Y2_CHECK(y2_memcpy_d2h(g_boxes.host, g_boxes.dev, (size_t)total * 4 * sizeof(float), 0));
    Y2_CHECK(y2_memcpy_d2h(g_probs.host, g_probs.dev, (size_t)total * out_classes * sizeof(float), 0));
    if (l.softmax_tree) Y2_CHECK(y2_memcpy_d2h(g_pred.host, g_pred.dev, pred_bytes, 0));
    Y2_CHECK(y2_stream_sync(0));
    if (map_dev && map_dev != r->map_dev) y2_free(map_dev);
    memcpy(boxes, g_boxes.host, (size_t)total * sizeof(box));
    for (int j = 0; j < total; ++j)
        memcpy(probs[j], (float *)g_probs.host + (size_t)j * out_classes, (size_t)out_classes * sizeof(float));
    if (l.softmax_tree) memcpy(l.output, g_pred.host, pred_bytes);
}

/* box.c:249-277 */
void do_nms_sort(box *boxes, float **probs, int total, int classes, float thresh)
{
    if (total <= 0 || classes <= 0) return;
    scratch_reserve(&g_boxes, (size_t)total * 4 * sizeof(float));
    scratch_reserve(&g_probs, (size_t)total * classes * sizeof(float));
    memcpy(g_boxes.host, boxes, (size_t)total * sizeof(box));
    for (int j = 0; j < total; ++j)
        memcpy((float *)g_probs.host + (size_t)j * classes, probs[j], (size_t)classes * sizeof(float));
    Y2_CHECK(y2_memcpy_h2d(g_boxes.dev, g_boxes.host, (size_t)total * 4 * sizeof(float), 0));
    Y2_CHECK(y2_memcpy_h2d(g_probs.dev, g_probs.host, (size_t)total * classes * sizeof(float), 0));
    Y2_CHECK(y2_nms_sort((const float *)g_boxes.dev, (float *)g_probs.dev, 1, total, classes, thresh, 0));
    Y2_CHECK(y2_memcpy_d2h(g_probs.host, g_probs.dev, (size_t)total * classes * sizeof(float), 0));
    Y2_CHECK(y2_stream_sync(0));
    for (int j = 0; j < total; ++j)
        memcpy(probs[j], (float *)g_probs.host + (size_t)j * classes, (size_t)classes * sizeof(float));
}

/* box.c:279-297, the unsorted variant demo.c and validate_detector_recall call */
void do_nms(box *boxes, float **probs, int total, int classes, float thresh)
{
    if (total <= 0 || classes <= 0) return;
    scratch_reserve(&g_boxes, (size_t)total * 4 * sizeof(float));
    scratch_reserve(&g_probs, (size_t)total * classes * sizeof(float));
    memcpy(g_boxes.host, boxes, (size_t)total * sizeof(box));
    for (int j = 0; j < total; ++j)
        memcpy((float *)g_probs.host + (size_t)j * classes, probs[j], (size_t)classes * sizeof(float));
    Y2_CHECK(y2_memcpy_h2d(g_boxes.dev, g_boxes.host, (size_t)total * 4 * sizeof(float), 0));
    Y2_CHECK(y2_memcpy_h2d(g_probs.dev, g_probs.host, (size_t)total * classes * sizeof(float), 0));
    Y2_CHECK(y2_nms_unsorted((const float *)g_boxes.dev, (float *)g_probs.dev, total, classes, thresh, 0));
    Y2_CHECK(y2_memcpy_d2h(g_probs.host, g_probs.dev, (size_t)total * classes * sizeof(float), 0));
    Y2_CHECK(y2_stream_sync(0));
    for (int j = 0; j < total; ++j)
        memcpy(probs[j], (float *)g_probs.host + (size_t)j * classes, (size_t)classes * sizeof(float));
}

/* ---- batched, device-resident detection (extension) -------------------------------------------- */
static layer *region_of(network net)
{
    layer *l = &net.layers[net.n - 1];
    if (l->type != REGION || !l->b200) error("network_detect: last layer is not a planned region layer");
    return l;
}

/* get_region_boxes + do_nms_sort + the final pick for the first B images of pred ([B][outputs], the region output or
 * the 3-frame means of a streams batch) on the network's stream: the decode counts the NMS candidates while it writes
 * the probabilities, the suppression pass marks losers negative and the pick reads negative as zero (3 launches; the
 * counters and scratch are the network's own) */
static void detect_tail(y2_net_rt *rt, layer *l, void *head_rt, float *pred, int B, float thresh, float nms,
                        y2_det *det_dev, int *cnt_dev, int det_cap)
{
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    const int total = l->w * l->h * l->n;
    if (l->softmax_tree && rt->defer_region) {
        /* softmax tree: only the groups on the path of classes above .5 are evaluated, straight from the head's
         * raw output; NMS and the pick work on one (class, value) record per box (2 launches) */
        y2_layer_rt *hr = (y2_layer_rt *)head_rt;
        Y2_CHECK(y2_region_tree_detect((const float *)hr->out, hr->out_cs, r->biases_dev, B, l->w, l->h, l->n,
                                       l->classes, thresh, l->classfix, r->group_size_dev, r->group_offset_dev,
                                       r->child_ptr_dev, r->child_grp_dev, r->tree_rec_dev, rt->stream));
        Y2_CHECK(y2_tree_nms_collect(r->tree_rec_dev, B, total, thresh, nms, det_dev, cnt_dev, det_cap, rt->stream));
        return;
    }
    Y2_CHECK(y2_region_boxes_counted(pred, r->biases_dev, r->boxes_dev, r->probs_dev, B, l->w, l->h, l->n,
                                     l->classes, 1.f, 1.f, thresh, 0, l->classfix,
                                     l->softmax_tree ? l->softmax_tree->n : 0, r->tree_parent_dev, 0, 0,
                                     r->nms_cnt_dev, rt->stream));
    if (nms > 0)
        Y2_CHECK(y2_nms_mark(r->boxes_dev, r->probs_dev, r->nms_cnt_dev, B, total, l->classes, nms, rt->stream));
    Y2_CHECK(y2_collect_ws(r->boxes_dev, r->probs_dev, B, total, l->classes, thresh, det_dev, cnt_dev, det_cap,
                           r->collect_ws, r->nms_cnt_dev, rt->stream));
}

void network_detect_device(network net, float thresh, float nms, y2_detection *dets, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_detect: network has no device plan");
    Y2_CHECK(y2_set_device(rt->device));
    layer *l = region_of(net);
    const int B = net.batch;
    if (rt->det_cap < max_det || rt->det_batch < B) {
        y2_free(rt->det_dev);
        y2_host_free(rt->det_pinned);
        y2_free(rt->cnt_dev);
        y2_host_free(rt->cnt_pinned);
        rt->det_cap = max_det;
        rt->det_batch = B > rt->cap_batch ? B : rt->cap_batch;
        const size_t nd = (size_t)rt->det_batch * rt->det_cap;
        Y2_CHECK(y2_malloc((void **)&rt->det_dev, nd * sizeof(y2_det)));
        Y2_CHECK(y2_host_alloc((void **)&rt->det_pinned, nd * sizeof(y2_det)));
        Y2_CHECK(y2_malloc((void **)&rt->cnt_dev, (size_t)rt->det_batch * sizeof(int)));
        Y2_CHECK(y2_host_alloc((void **)&rt->cnt_pinned, (size_t)rt->det_batch * sizeof(int)));
    }
    detect_tail(rt, l, net.layers[net.n - 2].b200, (float *)((y2_layer_rt *)l->b200)->out, B, thresh, nms, rt->det_dev,
                rt->cnt_dev, rt->det_cap);
    Y2_CHECK(y2_memcpy_d2h(rt->cnt_pinned, rt->cnt_dev, (size_t)B * sizeof(int), rt->stream));
    Y2_CHECK(y2_memcpy_d2h(rt->det_pinned, rt->det_dev, (size_t)B * rt->det_cap * sizeof(y2_det), rt->stream));
    Y2_CHECK(y2_stream_sync(rt->stream));
    for (int b = 0; b < B; ++b) {
        int c = rt->cnt_pinned[b];
        counts[b] = c;
        if (c > max_det) c = max_det;
        memcpy(dets + (size_t)b * max_det, rt->det_pinned + (size_t)b * rt->det_cap, (size_t)c * sizeof(y2_det));
    }
}

void network_detect_batch(network net, const float *input, float thresh, float nms, y2_detection *dets,
                          int *counts, int max_det)
{
    network_upload_input(net, input);
    network_forward_device(net);
    network_detect_device(net, thresh, nms, dets, counts, max_det);
}

/* ---- two-deep pipeline: the H2D copy of batch i+1 overlaps the forward pass of batch i ---------- */
static void pipe_init(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt->pipe_ready) return;
    Y2_CHECK(y2_set_device(rt->device));
    Y2_CHECK(y2_stream_create(&rt->copy_stream));
    Y2_CHECK(y2_stream_create(&rt->d2h_stream));
    rt->pipe[0].in_dev = rt->in_dev;
    rt->pipe[0].in_pinned = rt->in_pinned;
    Y2_CHECK(y2_malloc((void **)&rt->pipe[1].in_dev, rt->in_bytes));
    Y2_CHECK(y2_host_alloc((void **)&rt->pipe[1].in_pinned, rt->in_bytes));
    for (int s = 0; s < 2; ++s) {
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_h2d));
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_tail));
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_done));
        rt->pipe[s].busy = 0;
    }
    rt->pipe_head = 0;
    rt->pipe_inflight = 0;
    rt->pipe_ready = 1;
}

static void pipe_reserve_dets(y2_net_rt *rt, int s, int batch, int max_det)
{
    struct y2_pipe_slot *ps = &rt->pipe[s];
    if (ps->det_cap >= max_det && ps->det_dev) return;
    y2_free(ps->det_dev);
    y2_host_free(ps->det_pinned);
    y2_free(ps->cnt_dev);
    y2_host_free(ps->cnt_pinned);
    const int cap_b = batch > rt->cap_batch ? batch : rt->cap_batch;
    const size_t nd = (size_t)cap_b * max_det;
    Y2_CHECK(y2_malloc((void **)&ps->det_dev, nd * sizeof(y2_det)));
    Y2_CHECK(y2_host_alloc((void **)&ps->det_pinned, nd * sizeof(y2_det)));
    Y2_CHECK(y2_malloc((void **)&ps->cnt_dev, (size_t)cap_b * sizeof(int)));
    Y2_CHECK(y2_host_alloc((void **)&ps->cnt_pinned, (size_t)cap_b * sizeof(int)));
    ps->det_cap = max_det;
}

float *network_pipeline_staging(network net, int slot)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || slot < 0 || slot > 1) error("network_pipeline_staging: bad slot or unplanned network");
    pipe_init(net);
    return rt->pipe[slot].in_pinned;
}

int network_pipeline_next_slot(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_pipeline_next_slot: network has no device plan");
    pipe_init(net);
    return (rt->pipe_head + rt->pipe_inflight) & 1;
}

static void pipe_init_u8(network net)
{
    y2_net_rt *rt = y2_rt(net);
    pipe_init(net);
    if (rt->pipe[0].in_u8_dev) return;
    layer *l0 = &net.layers[0];
    y2_layer_rt *r0 = (y2_layer_rt *)l0->b200;
    if (!r0 || !r0->stem_fused || l0->c != 3 || !y2_stem_u8_supported(net.h, net.w))
        error("uint8 input needs a network whose first layer runs the fused first-layer kernel (3x3 conv over 3 "
              "channels followed by a 2x2/2 maxpool) and a width that is a multiple of 16; use the frames entry");
    const size_t bytes = (size_t)rt->cap_batch * net.h * net.w * 3;
    for (int s = 0; s < 2; ++s) {
        Y2_CHECK(y2_malloc((void **)&rt->pipe[s].in_u8_dev, bytes));
        Y2_CHECK(y2_host_alloc((void **)&rt->pipe[s].in_u8_pinned, bytes));
    }
}

unsigned char *network_pipeline_staging_u8(network net, int slot)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || slot < 0 || slot > 1) error("network_pipeline_staging_u8: bad slot or unplanned network");
    pipe_init_u8(net);
    return rt->pipe[slot].in_u8_pinned;
}

/* grows slot s's frame buffers to `bytes`; with old_pinned, the old pinned buffer is handed to the caller (to copy
 * frames out of it before freeing it) instead of being freed here */
static void pipe_reserve_frames(y2_net_rt *rt, int s, size_t bytes, unsigned char **old_pinned)
{
    struct y2_pipe_slot *ps = &rt->pipe[s];
    if (ps->frames_cap >= bytes) return;
    y2_free(ps->frames_dev);
    if (old_pinned) *old_pinned = ps->frames_pinned;
    else y2_host_free(ps->frames_pinned);
    Y2_CHECK(y2_malloc((void **)&ps->frames_dev, bytes));
    Y2_CHECK(y2_host_alloc((void **)&ps->frames_pinned, bytes));
    ps->frames_cap = bytes;
}

/* n frames of their own sizes (the *_frame_list entries) */
typedef struct {
    int n;
    const unsigned char *const *frames;
    const int *w, *h;
} frame_list;

/* the refusals of every frame-list entry, before anything is staged */
static void check_frame_list(network net, const frame_list *fl)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network frame list: network has no device plan");
    if (net.c != 3) error("network frame list: needs a network with 3 input channels");
    if (fl->n < 1 || fl->n > net.batch) error("network frame list: the list must hold 1 .. batch frames");
    if (!fl->frames || !fl->w || !fl->h) error("network frame list: NULL frame, width or height array");
    for (int i = 0; i < fl->n; ++i) {
        if (!fl->frames[i]) error("network frame list: NULL frame pointer");
        if (fl->w[i] <= 0 || fl->h[i] <= 0) error("network frame list: a frame size of 0 or less");
    }
}

unsigned char *network_pipeline_staging_frame_list(network net, int slot, int n, const int *frame_w,
                                                   const int *frame_h, size_t *offsets)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_pipeline_staging_frame_list: network has no device plan");
    if (slot < 0 || slot > 1 || n < 1 || n > net.batch || !offsets)
        error("network_pipeline_staging_frame_list: bad slot or offsets, or a list not of 1 .. batch frames");
    const size_t bytes = y2_frame_list_layout(n, frame_w, frame_h, net.w, net.h, 0, NULL, NULL);
    if (!bytes) error("network_pipeline_staging_frame_list: a frame size of 0 or less");
    pipe_init(net);
    Y2_CHECK(y2_set_device(rt->device));
    pipe_reserve_frames(rt, slot, bytes, NULL);
    y2_frame_window *win = (y2_frame_window *)calloc((size_t)n, sizeof(y2_frame_window));
    if (!win) error("network_pipeline_staging_frame_list: out of host memory");
    y2_frame_list_layout(n, frame_w, frame_h, net.w, net.h, 0, win, NULL);
    for (int i = 0; i < n; ++i) offsets[i] = (size_t)win[i].offset;
    free(win);
    return rt->pipe[slot].frames_pinned;
}

/* A frame list into slot s: the frames and the record table behind them in the slot's pinned buffer (frames already
 * at their place there are not copied), then one H2D copy of the whole region on the copy stream.  Returns the
 * table's offset in the region. */
static size_t stage_frame_list(network net, int s, const frame_list *fl, int letterbox)
{
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    size_t table_off = 0;
    const size_t bytes = y2_frame_list_layout(fl->n, fl->w, fl->h, net.w, net.h, letterbox, NULL, &table_off);
    unsigned char *old = NULL;
    pipe_reserve_frames(rt, s, bytes, &old);
    y2_frame_window *win = (y2_frame_window *)(ps->frames_pinned + table_off);
    y2_frame_list_layout(fl->n, fl->w, fl->h, net.w, net.h, letterbox, win, NULL);
    for (int i = 0; i < fl->n; ++i) {
        unsigned char *dst = ps->frames_pinned + win[i].offset;
        if (fl->frames[i] != dst) memcpy(dst, fl->frames[i], (size_t)fl->w[i] * fl->h[i] * 3);
    }
    Y2_CHECK(y2_host_free(old));
    Y2_CHECK(y2_memcpy_h2d(ps->frames_dev, ps->frames_pinned, bytes, rt->copy_stream));
    return table_off;
}

/* The input half of a submission, into slot s: the staging copy, the H2D copy on the copy stream, resize (or
 * letterbox) and the forward pass on the network's stream.  input: fp32 planar [B][c][h][w] (u8 == 0), uint8
 * interleaved RGB [B][h][w][3] at the network's resolution (u8 == 1), uint8 interleaved RGB frames [B][fh][fw][3]
 * of any size (u8 == 2), nothing: the slot's device input already holds the batch (u8 == 3, *_submit_resident), or
 * a frame_list (u8 == 4) */
static void submit_input(network net, int s, const void *input, int u8, int fw, int fh, int letterbox)
{
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    const int B = net.batch;
    size_t table_off = 0;
    /* pageable caller memory is staged through the slot's pinned buffer (a host copy; fill the slot's
     * staging buffer directly to avoid it) */
    if (u8 == 4) {
        table_off = stage_frame_list(net, s, (const frame_list *)input, letterbox);
    } else if (u8 == 2) {
        const size_t bytes = (size_t)B * fh * fw * 3;
        pipe_reserve_frames(rt, s, bytes, NULL);
        if (input && input != ps->frames_pinned) memcpy(ps->frames_pinned, input, bytes);
        Y2_CHECK(y2_memcpy_h2d(ps->frames_dev, ps->frames_pinned, bytes, rt->copy_stream));
    } else if (u8 == 1) {
        const size_t bytes = (size_t)B * net.h * net.w * 3;
        if (input && input != ps->in_u8_pinned) memcpy(ps->in_u8_pinned, input, bytes);
        Y2_CHECK(y2_memcpy_h2d(ps->in_u8_dev, ps->in_u8_pinned, bytes, rt->copy_stream));
    } else if (u8 == 0) {
        const size_t bytes = (size_t)B * net.inputs * sizeof(float);
        if (input && input != ps->in_pinned) memcpy(ps->in_pinned, input, bytes);
        Y2_CHECK(y2_memcpy_h2d(ps->in_dev, ps->in_pinned, bytes, rt->copy_stream));
    }
    if (u8 != 3) {
        Y2_CHECK(y2_event_record(ps->ev_h2d, rt->copy_stream));
        Y2_CHECK(y2_stream_wait_event(rt->stream, ps->ev_h2d));
    }
    if (u8 == 4) /* byte/255. + resize_image or letterbox_image per frame, one launch, .5f behind the list */
        Y2_CHECK(y2_frames_u8_to_f32(ps->frames_dev, (const y2_frame_window *)(ps->frames_dev + table_off),
                                     ((const frame_list *)input)->n, ps->in_dev, B, net.w, net.h, rt->stream));
    else if (u8 == 2 && letterbox) /* byte/255. + letterbox_image on the device, into the slot's fp32 input */
        Y2_CHECK(y2_letterbox_u8_to_f32(ps->frames_dev, ps->in_dev, B, fw, fh, net.w, net.h, rt->stream));
    else if (u8 == 2) /* byte/255. + resize_image on the device, into the slot's fp32 input */
        Y2_CHECK(y2_resize_u8_to_f32(ps->frames_dev, ps->in_dev, B, fw, fh, net.w, net.h, rt->stream));
    if (u8 == 1) {
        rt->input_u8 = 1; /* read while the layer list is captured */
        y2_run_forward_from(net, (float *)ps->in_u8_dev, &ps->graph_u8, &ps->graph_u8_valid);
        rt->input_u8 = 0;
    } else if (s == 0) {
        y2_run_forward_from(net, ps->in_dev, &rt->graph, &rt->graph_valid);
    } else {
        y2_run_forward_from(net, ps->in_dev, &ps->graph, &ps->graph_valid);
    }
}

/* checks shared by both kinds of submission; returns the slot the batch goes to */
static int submit_slot(network net, int u8, int fw, int fh)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network submit: network has no device plan");
    if (net.batch != rt->plan_batch) error("network batch changed without set_batch_network");
    if (u8 == 1) pipe_init_u8(net);
    else pipe_init(net);
    if (u8 == 2 && (net.c != 3 || fw <= 0 || fh <= 0)) error("network submit of frames: needs 3-channel input and a frame size");
    if (rt->pipe_inflight >= 2)
        error("network submit: two batches already in flight, wait for one first");
    Y2_CHECK(y2_set_device(rt->device));
    return (rt->pipe_head + rt->pipe_inflight) & 1;
}

/* the tail half's results travel on their own stream: the next batch's forward pass (same compute stream) does not
 * wait behind the device -> host copies of this one */
static void submit_results(y2_net_rt *rt, int s)
{
    struct y2_pipe_slot *ps = &rt->pipe[s];
    Y2_CHECK(y2_event_record(ps->ev_tail, rt->stream));
    Y2_CHECK(y2_stream_wait_event(rt->d2h_stream, ps->ev_tail));
}

static void submit_done(y2_net_rt *rt, int s, int kind, int n_images)
{
    struct y2_pipe_slot *ps = &rt->pipe[s];
    Y2_CHECK(y2_event_record(ps->ev_done, rt->d2h_stream));
    ps->kind = kind;
    ps->n_images = n_images;
    ps->busy = 1;
    rt->pipe_inflight++;
}

/* ---- video streams: each image is decoded on the 3-frame mean of its stream (yolo_v2_class.cpp:206-216) ------- */
static layer *streams_region(network net)
{
    layer *l = region_of(net);
    if (l->softmax_tree || y2_rt(net)->defer_region)
        error("network streams: needs a flat-softmax region head (a softmax tree defers the region forward, so there "
              "is no dense region output to average)");
    return l;
}

/* the refusals of every streams submission, before anything is staged */
static void check_streams(network net, int n, const int *stream_ids)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network streams: network has no device plan");
    const layer *l = streams_region(net);
    const y2_streams *st = rt->streams;
    if (!st) error("network streams: streams not opened, call network_streams_open");
    if (l->outputs != st->outputs)
        error("network streams: the region output size differs from the one the streams were opened with (after "
              "resize_network, open them again)");
    if (n < 1 || n > net.batch) error("network streams: the list must hold 1 .. batch images");
    if (!stream_ids) error("network streams: NULL stream id array");
    for (int i = 0; i < n; ++i)
        if (stream_ids[i] < 0 || stream_ids[i] >= st->max_streams)
            error("network streams: a stream id outside 0 .. max_streams-1");
}

void y2_streams_free(y2_net_rt *rt)
{
    y2_streams *st = rt->streams;
    if (!st) return;
    y2_free(st->ring_dev);
    y2_free(st->mean_dev);
    for (int s = 0; s < 2; ++s) {
        y2_free(st->table_dev[s]);
        y2_host_free(st->table_pinned[s]);
    }
    free(st->frame_index);
    free(st->frames_seen);
    free(st);
    rt->streams = NULL;
}

void network_streams_open(network net, int max_streams)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_streams_open: network has no device plan");
    if (max_streams < 1) error("network_streams_open: max_streams must be 1 or more");
    const layer *l = streams_region(net);
    Y2_CHECK(y2_set_device(rt->device));
    Y2_CHECK(y2_stream_sync(rt->stream)); /* batches in flight read and write the old ring */
    y2_streams_free(rt);
    y2_streams *st = (y2_streams *)calloc(1, sizeof(y2_streams));
    if (!st) error("network_streams_open: out of host memory");
    st->max_streams = max_streams;
    st->outputs = l->outputs;
    st->frame_index = (int *)calloc((size_t)max_streams, sizeof(int));
    st->frames_seen = (int *)calloc((size_t)max_streams, sizeof(int));
    if (!st->frame_index || !st->frames_seen) error("network_streams_open: out of host memory");
    /* not cleared: a ring row is read only after it was written (y2_stream_plan reads unwritten slots as zero) */
    Y2_CHECK(y2_malloc((void **)&st->ring_dev, (size_t)max_streams * 3 * l->outputs * sizeof(float)));
    rt->streams = st;
}

void network_stream_reset(network net, int stream)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_stream_reset: network has no device plan");
    y2_streams *st = rt->streams;
    if (!st) error("network_stream_reset: streams not opened, call network_streams_open");
    if (stream < 0 || stream >= st->max_streams) error("network_stream_reset: a stream id outside 0 .. max_streams-1");
    /* host only: batches already submitted keep the table they were given */
    st->frame_index[stream] = 0;
    st->frames_seen[stream] = 0;
}

/* A streams batch into slot s: its ring plan in the slot's table, copied on the copy stream (ahead of the slot's
 * input copies, so the slot's ev_h2d covers it) */
static void streams_stage(y2_net_rt *rt, int s, int n, const int *stream_ids, int batch)
{
    y2_streams *st = rt->streams;
    const int cap_b = batch > rt->cap_batch ? batch : rt->cap_batch;
    if (st->mean_cap < batch) {
        Y2_CHECK(y2_stream_sync(rt->stream)); /* the other slot's decode may still read the means */
        y2_free(st->mean_dev);
        Y2_CHECK(y2_malloc((void **)&st->mean_dev, (size_t)cap_b * st->outputs * sizeof(float)));
        st->mean_cap = cap_b;
    }
    if (st->table_cap[s] < batch) {
        y2_free(st->table_dev[s]);
        y2_host_free(st->table_pinned[s]);
        Y2_CHECK(y2_malloc((void **)&st->table_dev[s], (size_t)cap_b * sizeof(y2_stream_src)));
        Y2_CHECK(y2_host_alloc((void **)&st->table_pinned[s], (size_t)cap_b * sizeof(y2_stream_src)));
        st->table_cap[s] = cap_b;
    }
    Y2_CHECK(y2_stream_plan(n, stream_ids, st->max_streams, st->frame_index, st->frames_seen, st->table_pinned[s]));
    Y2_CHECK(y2_memcpy_h2d(st->table_dev[s], st->table_pinned[s], (size_t)n * sizeof(y2_stream_src), rt->copy_stream));
}

/* n images come back.  stream_ids (n of them): a streams batch, decoded on the 3-frame means; else the tail runs on
 * the region output of all B images. */
static int submit_common(network net, const void *input, int u8, int fw, int fh, int n, const int *stream_ids,
                         float thresh, float nms, int max_det)
{
    const int s = submit_slot(net, u8, fw, fh);
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    layer *l = region_of(net);
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    void *head_rt = net.layers[net.n - 2].b200;
    const int B = net.batch;
    pipe_reserve_dets(rt, s, B, max_det);
    if (stream_ids) streams_stage(rt, s, n, stream_ids, B);
    submit_input(net, s, input, u8, fw, fh, 0);
    if (stream_ids) {
        y2_streams *st = rt->streams;
        if (u8 == 3) { /* no input copy: the compute stream waits for the table alone */
            Y2_CHECK(y2_event_record(ps->ev_h2d, rt->copy_stream));
            Y2_CHECK(y2_stream_wait_event(rt->stream, ps->ev_h2d));
        }
        Y2_CHECK(y2_stream_mean((const float *)r->out, st->ring_dev, st->table_dev[s], n, st->outputs, st->mean_dev,
                                rt->stream));
        Y2_CHECK(y2_stream_commit((const float *)r->out, st->ring_dev, st->table_dev[s], n, st->outputs, rt->stream));
        detect_tail(rt, l, head_rt, st->mean_dev, n, thresh, nms, ps->det_dev, ps->cnt_dev, ps->det_cap);
    } else {
        detect_tail(rt, l, head_rt, (float *)r->out, B, thresh, nms, ps->det_dev, ps->cnt_dev, ps->det_cap);
    }
    submit_results(rt, s);
    Y2_CHECK(y2_memcpy_d2h(ps->cnt_pinned, ps->cnt_dev, (size_t)n * sizeof(int), rt->d2h_stream));
    Y2_CHECK(y2_memcpy_d2h(ps->det_pinned, ps->det_dev, (size_t)n * ps->det_cap * sizeof(y2_det), rt->d2h_stream));
    submit_done(rt, s, Y2_PIPE_DETECT, n);
    return s;
}

int network_detect_submit(network net, const float *input, float thresh, float nms, int max_det)
{
    return submit_common(net, input, 0, 0, 0, net.batch, NULL, thresh, nms, max_det);
}

int network_detect_submit_u8(network net, const unsigned char *input_hwc, float thresh, float nms, int max_det)
{
    return submit_common(net, input_hwc, 1, 0, 0, net.batch, NULL, thresh, nms, max_det);
}

/* The batch is already in the slot's device input (network_pipeline_input_device(net, slot), e.g. written by another
 * kernel or uploaded once): forward + decode + NMS + pick without any host -> device copy, pipelined like the others. */
int network_detect_submit_resident(network net, float thresh, float nms, int max_det)
{
    return submit_common(net, 0, 3, 0, 0, net.batch, NULL, thresh, nms, max_det);
}

float *network_pipeline_input_device(network net, int slot)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || slot < 0 || slot > 1) error("network_pipeline_input_device: bad slot or unplanned network");
    pipe_init(net);
    return rt->pipe[slot].in_dev;
}

int network_detect_wait(network net, y2_detection *dets, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || !rt->pipe_ready || rt->pipe_inflight <= 0) error("network_detect_wait: nothing in flight");
    const int s = rt->pipe_head;
    struct y2_pipe_slot *ps = &rt->pipe[s];
    if (ps->kind != Y2_PIPE_DETECT)
        error("network_detect_wait: the oldest batch in flight is a classify batch, call network_classify_wait");
    Y2_CHECK(y2_event_sync(ps->ev_done));
    for (int b = 0; b < ps->n_images; ++b) {
        int c = ps->cnt_pinned[b];
        counts[b] = c;
        if (c > max_det) c = max_det;
        if (c > ps->det_cap) c = ps->det_cap;
        memcpy(dets + (size_t)b * max_det, ps->det_pinned + (size_t)b * ps->det_cap, (size_t)c * sizeof(y2_det));
    }
    ps->busy = 0;
    rt->pipe_head ^= 1;
    rt->pipe_inflight--;
    return s;
}

void network_detect_batch_u8(network net, const unsigned char *input_hwc, float thresh, float nms, y2_detection *dets,
                             int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight) error("network_detect_batch_u8: batches of the submit/wait pipeline are in flight");
    submit_common(net, input_hwc, 1, 0, 0, net.batch, NULL, thresh, nms, max_det);
    network_detect_wait(net, dets, counts, max_det);
}

/* frames at the network's resolution go to the uint8 first-layer kernel when the network has one */
static int frames_take_u8(network net, int frame_w, int frame_h)
{
    y2_layer_rt *r0 = (y2_layer_rt *)net.layers[0].b200;
    return frame_w == net.w && frame_h == net.h && r0 && r0->stem_fused && net.c == 3 &&
           y2_stem_u8_supported(net.h, net.w);
}

/* Decoded frames of any size: upload the raw bytes, then byte/255. (load_image_stb) and resize_image
 * (image.c:1950-1993) run on the device, bit-identical to Detector::detect(filename)'s host path
 * (yolo_v2_class.cpp:173-206).  Frames already at the network's resolution take the uint8 first-layer
 * path when the network has one. */
int network_detect_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, float thresh,
                                 float nms, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_detect_submit_frames: network has no device plan");
    if (frames_take_u8(net, frame_w, frame_h))
        return submit_common(net, frames_hwc, 1, 0, 0, net.batch, NULL, thresh, nms, max_det);
    return submit_common(net, frames_hwc, 2, frame_w, frame_h, net.batch, NULL, thresh, nms, max_det);
}

int network_detect_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, int max_det)
{
    const frame_list fl = {n, frames, frame_w, frame_h};
    check_frame_list(net, &fl);
    return submit_common(net, &fl, 4, 0, 0, n, NULL, thresh, nms, max_det);
}

void network_detect_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, y2_detection *dets, int *counts,
                                     int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight)
        error("network_detect_batch_frame_list: batches of the submit/wait pipeline are in flight");
    network_detect_submit_frame_list(net, n, frames, frame_w, frame_h, thresh, nms, max_det);
    network_detect_wait(net, dets, counts, max_det);
}

int network_detect_submit_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms, int max_det)
{
    const frame_list fl = {n, frames, frame_w, frame_h};
    check_frame_list(net, &fl);
    check_streams(net, n, stream_ids);
    return submit_common(net, &fl, 4, 0, 0, n, stream_ids, thresh, nms, max_det);
}

int network_detect_submit_streams_resident(network net, int n, const int *stream_ids, float thresh, float nms,
                                           int max_det)
{
    check_streams(net, n, stream_ids);
    return submit_common(net, 0, 3, 0, 0, n, stream_ids, thresh, nms, max_det);
}

void network_detect_batch_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms,
                                  y2_detection *dets, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight)
        error("network_detect_batch_streams: batches of the submit/wait pipeline are in flight");
    network_detect_submit_streams(net, n, stream_ids, frames, frame_w, frame_h, thresh, nms, max_det);
    network_detect_wait(net, dets, counts, max_det);
}

unsigned char *network_pipeline_staging_frames(network net, int slot, int frame_w, int frame_h)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || slot < 0 || slot > 1 || frame_w <= 0 || frame_h <= 0)
        error("network_pipeline_staging_frames: bad slot, frame size or unplanned network");
    if (frames_take_u8(net, frame_w, frame_h)) return network_pipeline_staging_u8(net, slot);
    pipe_init(net);
    Y2_CHECK(y2_set_device(rt->device));
    pipe_reserve_frames(rt, slot, (size_t)rt->cap_batch * frame_h * frame_w * 3, NULL);
    return rt->pipe[slot].frames_pinned;
}

void network_detect_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, float thresh,
                                 float nms, y2_detection *dets, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight) error("network_detect_batch_frames: batches of the submit/wait pipeline are in flight");
    network_detect_submit_frames(net, frames_hwc, frame_w, frame_h, thresh, nms, max_det);
    network_detect_wait(net, dets, counts, max_det);
}

/* ---- batched, device-resident classification (extension) --------------------------------------- */
/* the output layer the classify entries read, after the checks every entry makes */
static layer *classify_layer(network net, int top)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_classify: network has no device plan");
    if (net.batch != rt->plan_batch) error("network batch changed without set_batch_network");
    layer *l = &net.layers[y2_output_layer_index(net)];
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    if (l->type == REGION) error("network_classify: the network ends in a region layer, use network_detect_*");
    if (!r || r->out_kind != Y2_KIND_F32_VEC)
        error("network_classify: the output layer is not a class vector (softmax, avgpool, connected or dropout)");
    if (l->outputs > Y2_CLASSIFY_MAX_N) error("network_classify: more outputs than Y2_CLASSIFY_MAX_N");
    if (top < 1 || top > l->outputs || top > Y2_CLASSIFY_MAX_TOP)
        error("network_classify: top must be in 1 .. min(outputs, Y2_CLASSIFY_MAX_TOP)");
    if (net.hierarchy && (l->softmax_tree != net.hierarchy || net.hierarchy->n != l->outputs || !r->tree_parent_dev))
        error("network_classify: the WordTree must belong to the output softmax layer, list every parent before "
              "its children and be at most 64 levels deep");
    return l;
}

/* hierarchy_predictions (net.hierarchy) + top_k for every image of the batch, on the network's stream. The output
 * layer's rows are read in place (fp32 [B][out_cs]). */
static void classify_tail(y2_net_rt *rt, network net, layer *l, int top, y2_class_hit *hits_dev)
{
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    Y2_CHECK(y2_classify_topk((const float *)r->out, r->out_cs, net.batch, l->outputs, top,
                              net.hierarchy ? r->tree_parent_dev : 0, hits_dev, rt->stream));
}

/* grows a [cap_batch][*cap] hit buffer pair to hold `top` hits per image */
static void reserve_hits(y2_net_rt *rt, y2_class_hit **dev, y2_class_hit **pinned, int *cap, int top)
{
    if (*cap >= top && *dev) return;
    y2_free(*dev);
    y2_host_free(*pinned);
    const size_t n = (size_t)rt->cap_batch * top;
    Y2_CHECK(y2_malloc((void **)dev, n * sizeof(y2_class_hit)));
    Y2_CHECK(y2_host_alloc((void **)pinned, n * sizeof(y2_class_hit)));
    *cap = top;
}

void network_classify_device(network net, int top, y2_class_hit *hits)
{
    layer *l = classify_layer(net, top);
    y2_net_rt *rt = y2_rt(net);
    Y2_CHECK(y2_set_device(rt->device));
    reserve_hits(rt, &rt->hits_dev, &rt->hits_pinned, &rt->hits_cap, top);
    classify_tail(rt, net, l, top, rt->hits_dev);
    const size_t bytes = (size_t)net.batch * top * sizeof(y2_class_hit);
    Y2_CHECK(y2_memcpy_d2h(rt->hits_pinned, rt->hits_dev, bytes, rt->stream));
    Y2_CHECK(y2_stream_sync(rt->stream));
    memcpy(hits, rt->hits_pinned, bytes);
}

void network_classify_batch(network net, const float *input, int top, y2_class_hit *hits)
{
    classify_layer(net, top);
    network_upload_input(net, input);
    network_forward_device(net);
    network_classify_device(net, top, hits);
}

static int classify_submit_common(network net, const void *input, int u8, int fw, int fh, int top)
{
    layer *l = classify_layer(net, top);
    const int s = submit_slot(net, u8, fw, fh);
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    const int n = u8 == 4 ? ((const frame_list *)input)->n : net.batch;
    reserve_hits(rt, &ps->hits_dev, &ps->hits_pinned, &ps->hits_cap, top);
    submit_input(net, s, input, u8, fw, fh, 1);
    classify_tail(rt, net, l, top, ps->hits_dev);
    submit_results(rt, s);
    Y2_CHECK(y2_memcpy_d2h(ps->hits_pinned, ps->hits_dev, (size_t)n * top * sizeof(y2_class_hit), rt->d2h_stream));
    ps->hits_top = top;
    submit_done(rt, s, Y2_PIPE_CLASSIFY, n);
    return s;
}

int network_classify_submit(network net, const float *input, int top)
{
    return classify_submit_common(net, input, 0, 0, 0, top);
}

int network_classify_submit_u8(network net, const unsigned char *input_hwc, int top)
{
    return classify_submit_common(net, input_hwc, 1, 0, 0, top);
}

/* frames of any size: byte/255. and letterbox_image (image.c:1624-1644) on the device */
int network_classify_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top)
{
    if (!y2_rt(net)) error("network_classify_submit_frames: network has no device plan");
    if (frames_take_u8(net, frame_w, frame_h)) return classify_submit_common(net, frames_hwc, 1, 0, 0, top);
    return classify_submit_common(net, frames_hwc, 2, frame_w, frame_h, top);
}

int network_classify_submit_resident(network net, int top)
{
    return classify_submit_common(net, 0, 3, 0, 0, top);
}

int network_classify_wait(network net, y2_class_hit *hits, int top)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || !rt->pipe_ready || rt->pipe_inflight <= 0) error("network_classify_wait: nothing in flight");
    const int s = rt->pipe_head;
    struct y2_pipe_slot *ps = &rt->pipe[s];
    if (ps->kind != Y2_PIPE_CLASSIFY)
        error("network_classify_wait: the oldest batch in flight is a detection batch, call network_detect_wait");
    if (top != ps->hits_top) error("network_classify_wait: top differs from the one the batch was submitted with");
    Y2_CHECK(y2_event_sync(ps->ev_done));
    memcpy(hits, ps->hits_pinned, (size_t)ps->n_images * top * sizeof(y2_class_hit));
    ps->busy = 0;
    rt->pipe_head ^= 1;
    rt->pipe_inflight--;
    return s;
}

void network_classify_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top,
                                   y2_class_hit *hits)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight) error("network_classify_batch_frames: batches of the submit/wait pipeline are in flight");
    network_classify_submit_frames(net, frames_hwc, frame_w, frame_h, top);
    network_classify_wait(net, hits, top);
}

int network_classify_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top)
{
    const frame_list fl = {n, frames, frame_w, frame_h};
    check_frame_list(net, &fl);
    return classify_submit_common(net, &fl, 4, 0, 0, top);
}

void network_classify_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top, y2_class_hit *hits)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight)
        error("network_classify_batch_frame_list: batches of the submit/wait pipeline are in flight");
    network_classify_submit_frame_list(net, n, frames, frame_w, frame_h, top);
    network_classify_wait(net, hits, top);
}
