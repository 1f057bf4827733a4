/*
 * Post-processing entry points of the drop-in API and the batched device-resident detection and
 * classification extensions.  The arithmetic runs in the region / NMS kernels; these functions only move the
 * caller-owned host arrays (boxes[total], probs[total][classes]) across, as the reference's
 * callers expect (detector.c:486-495, yolo_v2_class.cpp:71-73,215-216).  The batched entries describe their input
 * (y2_input) and hand it to the submit/wait pipeline of y2_pipeline.c; what is left here is their tails: decode, NMS
 * and pick (also on the 3-frame means of video streams), or WordTree and top-k.
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
 * the 3-frame means of a streams batch) on the network's stream, into res's detection lists: the decode counts the NMS
 * candidates while it writes the probabilities, the suppression pass marks losers negative and the pick reads
 * negative as zero (3 launches; the counters and scratch are the network's own) */
static void detect_tail(y2_net_rt *rt, layer *l, void *head_rt, float *pred, int B, float thresh, float nms,
                        const y2_results *res)
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
        Y2_CHECK(y2_tree_nms_collect(r->tree_rec_dev, B, total, thresh, nms, res->det_dev, res->cnt_dev, res->det_cap,
                                     rt->stream));
        return;
    }
    Y2_CHECK(y2_region_boxes_counted(pred, r->biases_dev, r->boxes_dev, r->probs_dev, B, l->w, l->h, l->n,
                                     l->classes, 1.f, 1.f, thresh, 0, l->classfix,
                                     l->softmax_tree ? l->softmax_tree->n : 0, r->tree_parent_dev, 0, 0,
                                     r->nms_cnt_dev, rt->stream));
    if (nms > 0)
        Y2_CHECK(y2_nms_mark(r->boxes_dev, r->probs_dev, r->nms_cnt_dev, B, total, l->classes, nms, rt->stream));
    Y2_CHECK(y2_collect_ws(r->boxes_dev, r->probs_dev, B, total, l->classes, thresh, res->det_dev, res->cnt_dev,
                           res->det_cap, r->collect_ws, r->nms_cnt_dev, rt->stream));
}

void network_detect_device(network net, float thresh, float nms, y2_detection *dets, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_detect: network has no device plan");
    Y2_CHECK(y2_set_device(rt->device));
    layer *l = region_of(net);
    const int B = net.batch;
    y2_results *res = &rt->res;
    y2_results_reserve_dets(rt, res, B, max_det);
    detect_tail(rt, l, net.layers[net.n - 2].b200, (float *)((y2_layer_rt *)l->b200)->out, B, thresh, nms, res);
    y2_results_to_host(res, Y2_PIPE_DETECT, B, 0, rt->stream);
    Y2_CHECK(y2_stream_sync(rt->stream));
    y2_results_copy_dets(res, B, dets, counts, max_det);
}

void network_detect_batch(network net, const float *input, float thresh, float nms, y2_detection *dets,
                          int *counts, int max_det)
{
    network_upload_input(net, input);
    network_forward_device(net);
    network_detect_device(net, thresh, nms, dets, counts, max_det);
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

/* the stream ids of a streams batch, one per image; a tracked batch also has the frame sizes in pixels */
typedef struct {
    int n;
    const int *ids;
    int tracked;
    int use_mean;     /* decoded on the 3-frame means (always, untracked) */
    const int *w, *h; /* tracked */
} stream_list;

/* the refusals of every streams submission, after the pipeline's and the frame list's, before anything is staged */
static void check_streams(network net, const stream_list *sl)
{
    y2_net_rt *rt = y2_rt(net);
    const layer *l = streams_region(net);
    const y2_streams *st = rt->streams;
    if (!st) error("network streams: streams not opened, call network_streams_open");
    if (l->outputs != st->outputs)
        error("network streams: the region output size differs from the one the streams were opened with (after "
              "resize_network, open them again)");
    if (sl->n < 1 || sl->n > net.batch) error("network streams: the list must hold 1 .. batch images");
    if (!sl->ids) error("network streams: NULL stream id array");
    for (int i = 0; i < sl->n; ++i)
        if (sl->ids[i] < 0 || sl->ids[i] >= st->max_streams)
            error("network streams: a stream id outside 0 .. max_streams-1");
    if (!sl->tracked) return;
    if (!st->story) error("network streams tracked: tracking not enabled, call network_streams_track");
    if (sl->use_mean != 0 && sl->use_mean != 1) error("network streams tracked: use_mean must be 0 or 1");
    if (!sl->w || !sl->h) error("network streams tracked: NULL frame width or height array");
    for (int i = 0; i < sl->n; ++i)
        if (sl->w[i] <= 0 || sl->h[i] <= 0) error("network streams tracked: a frame size of 0 or less");
}

static void track_free(y2_streams *st)
{
    y2_free(st->hist_dev);
    y2_free(st->hist_cnt_dev);
    y2_free(st->next_id_dev);
    free(st->track_head);
    free(st->track_len);
    free(st->track_restart);
    st->hist_dev = NULL;
    st->hist_cnt_dev = NULL;
    st->next_id_dev = NULL;
    st->track_head = st->track_len = st->track_restart = NULL;
    st->story = 0;
}

void y2_streams_free(y2_net_rt *rt)
{
    y2_streams *st = rt->streams;
    if (!st) return;
    track_free(st);
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
    if (st->story) { /* an empty history; the stream's next tracked image restarts its ids on the device */
        st->track_head[stream] = 0;
        st->track_len[stream] = 0;
        st->track_restart[stream] = 1;
    }
}

void network_streams_track(network net, int frames_story)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_streams_track: network has no device plan");
    y2_streams *st = rt->streams;
    if (!st) error("network_streams_track: streams not opened, call network_streams_open");
    if (frames_story < 1 || frames_story > Y2_TRACK_MAX_STORY)
        error("network_streams_track: frames_story must be in 1 .. Y2_TRACK_MAX_STORY");
    const layer *l = streams_region(net);
    if (l->w * l->h * l->n > Y2_TRACK_MAX_TOTAL)
        error("network_streams_track: more region boxes per image than Y2_TRACK_MAX_TOTAL (the tracking kernel holds a "
              "frame's boxes in shared memory)");
    Y2_CHECK(y2_set_device(rt->device));
    Y2_CHECK(y2_stream_sync(rt->stream)); /* batches in flight read and write the old history */
    track_free(st);
    const int S = st->max_streams, total = l->w * l->h * l->n;
    st->track_head = (int *)calloc((size_t)S, sizeof(int));
    st->track_len = (int *)calloc((size_t)S, sizeof(int));
    st->track_restart = (int *)malloc((size_t)S * sizeof(int));
    if (!st->track_head || !st->track_len || !st->track_restart) error("network_streams_track: out of host memory");
    for (int s = 0; s < S; ++s) st->track_restart[s] = 1;
    /* not cleared: a history slot is read only below its fill, ids only after the restart that sets them */
    Y2_CHECK(y2_malloc((void **)&st->hist_dev, (size_t)S * frames_story * total * sizeof(y2_bbox)));
    Y2_CHECK(y2_malloc((void **)&st->hist_cnt_dev, (size_t)S * frames_story * sizeof(int)));
    Y2_CHECK(y2_malloc((void **)&st->next_id_dev, (size_t)S * l->classes * sizeof(unsigned int)));
    st->story = frames_story;
    st->total = total;
    st->classes = l->classes;
}

/* where the parts of a slot's stream table sit for a batch of n images */
static size_t track_recs_at(int n) { return (size_t)n * sizeof(y2_stream_src); }
static size_t track_offsets_at(int n) { return track_recs_at(n) + (size_t)n * sizeof(y2_track_img); }
static size_t table_bytes(int n) { return track_offsets_at(n) + (size_t)(n + 1) * sizeof(int); }

/* A streams batch into slot s: its ring plan (decoded on the means) and its tracking plan (tracked) in the slot's
 * table, copied in one piece on the copy stream (ahead of the slot's input copies, so the slot's ev_h2d covers it).
 * Returns the number of distinct streams of a tracked batch. */
static int streams_stage(y2_net_rt *rt, int s, const stream_list *sl, int batch)
{
    y2_streams *st = rt->streams;
    const int n = sl->n;
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
        Y2_CHECK(y2_malloc((void **)&st->table_dev[s], table_bytes(cap_b)));
        Y2_CHECK(y2_host_alloc((void **)&st->table_pinned[s], table_bytes(cap_b)));
        st->table_cap[s] = cap_b;
    }
    unsigned char *tab = st->table_pinned[s];
    if (sl->use_mean)
        Y2_CHECK(y2_stream_plan(n, sl->ids, st->max_streams, st->frame_index, st->frames_seen, (y2_stream_src *)tab));
    int n_streams = 0;
    if (sl->tracked) {
        n_streams = y2_track_plan(n, sl->ids, sl->w, sl->h, st->max_streams, st->story, st->track_head, st->track_len,
                                  st->track_restart, (y2_track_img *)(tab + track_recs_at(n)),
                                  (int *)(tab + track_offsets_at(n)));
        Y2_CHECK(n_streams < 1 ? Y2_EINVAL : Y2_OK);
    }
    const size_t from = sl->use_mean ? 0 : track_recs_at(n), to = sl->tracked ? table_bytes(n) : track_recs_at(n);
    Y2_CHECK(y2_memcpy_h2d(st->table_dev[s] + from, tab + from, to - from, rt->copy_stream));
    return n_streams;
}

/* A detection batch into the pipeline.  With streams it is a streams batch: decoded on the 3-frame means (or, tracked
 * without use_mean, on the region output), streams->n images come back, tracked as pixel boxes with track ids;
 * otherwise (NULL) the tail runs on the region output of all B images and in.n come back. */
static int detect_submit(network net, y2_input in, const stream_list *streams, float thresh, float nms, int max_det)
{
    const int s = y2_pipe_claim(net, &in);
    if (streams) check_streams(net, streams);
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    layer *l = region_of(net);
    y2_layer_rt *r = (y2_layer_rt *)l->b200;
    void *head_rt = net.layers[net.n - 2].b200;
    const int B = net.batch;
    const int n = streams ? streams->n : in.n;
    const int tracked = streams && streams->tracked;
    const int total = l->w * l->h * l->n;
    /* tracking sees every detection of a frame: the lists hold all `total` boxes, max_det cuts only the copy out */
    y2_results_reserve_dets(rt, &ps->res, B, tracked ? total : max_det);
    if (tracked) {
        y2_results_reserve_boxes(rt, &ps->res, B, total);
        ps->res.box_stride = max_det < total ? max_det : total; /* rows of the copy back */
    }
    const int n_streams = streams ? streams_stage(rt, s, streams, B) : 0;
    y2_pipe_submit_input(net, s, &in, 0);
    if (streams) {
        y2_streams *st = rt->streams;
        if (in.kind == Y2_IN_RESIDENT) { /* no input copy: the compute stream waits for the table alone */
            Y2_CHECK(y2_event_record(ps->ev_h2d, rt->copy_stream));
            Y2_CHECK(y2_stream_wait_event(rt->stream, ps->ev_h2d));
        }
        const y2_stream_src *ring_plan = (const y2_stream_src *)st->table_dev[s];
        if (streams->use_mean) {
            Y2_CHECK(y2_stream_mean((const float *)r->out, st->ring_dev, ring_plan, n, st->outputs, st->mean_dev,
                                    rt->stream));
            Y2_CHECK(y2_stream_commit((const float *)r->out, st->ring_dev, ring_plan, n, st->outputs, rt->stream));
        }
        detect_tail(rt, l, head_rt, streams->use_mean ? st->mean_dev : (float *)r->out, n, thresh, nms, &ps->res);
        if (tracked)
            Y2_CHECK(y2_stream_track((const y2_det *)ps->res.det_dev, ps->res.det_cap, ps->res.cnt_dev,
                                     (const y2_track_img *)(st->table_dev[s] + track_recs_at(n)),
                                     (const int *)(st->table_dev[s] + track_offsets_at(n)), n_streams, total,
                                     st->classes, st->story, st->hist_dev, st->hist_cnt_dev, st->next_id_dev,
                                     ps->res.box_dev, ps->res.box_stride, rt->stream));
    } else {
        detect_tail(rt, l, head_rt, (float *)r->out, B, thresh, nms, &ps->res);
    }
    y2_pipe_queue(rt, s, tracked ? Y2_PIPE_TRACK : Y2_PIPE_DETECT, n, 0);
    return s;
}

int network_detect_wait(network net, y2_detection *dets, int *counts, int max_det)
{
    const int s = y2_pipe_retire(net, Y2_PIPE_DETECT, 0);
    const struct y2_pipe_slot *ps = &y2_rt(net)->pipe[s];
    y2_results_copy_dets(&ps->res, ps->n_images, dets, counts, max_det);
    return s;
}

int network_detect_wait_tracked(network net, y2_bbox *boxes, int *counts, int max_det)
{
    const int s = y2_pipe_retire(net, Y2_PIPE_TRACK, 0);
    const struct y2_pipe_slot *ps = &y2_rt(net)->pipe[s];
    y2_results_copy_boxes(&ps->res, ps->n_images, boxes, counts, max_det);
    return s;
}

/* the detection *_batch_* entries: one submission and its wait, refused while batches of the pipeline are in flight.
 * A tracked batch hands out boxes, every other one dets. */
static void detect_batch(network net, const char *in_flight, y2_input in, const stream_list *streams, float thresh,
                         float nms, y2_detection *dets, y2_bbox *boxes, int *counts, int max_det)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight) error(in_flight);
    detect_submit(net, in, streams, thresh, nms, max_det);
    if (streams && streams->tracked) network_detect_wait_tracked(net, boxes, counts, max_det);
    else network_detect_wait(net, dets, counts, max_det);
}

int network_detect_submit(network net, const float *input, float thresh, float nms, int max_det)
{
    return detect_submit(net, (y2_input){.kind = Y2_IN_F32, .data = input}, NULL, thresh, nms, max_det);
}

int network_detect_submit_u8(network net, const unsigned char *input_hwc, float thresh, float nms, int max_det)
{
    return detect_submit(net, (y2_input){.kind = Y2_IN_U8, .data = input_hwc}, NULL, thresh, nms, max_det);
}

void network_detect_batch_u8(network net, const unsigned char *input_hwc, float thresh, float nms, y2_detection *dets,
                             int *counts, int max_det)
{
    detect_batch(net, "network_detect_batch_u8: batches of the submit/wait pipeline are in flight",
                 (y2_input){.kind = Y2_IN_U8, .data = input_hwc}, NULL, thresh, nms, dets, NULL, counts, max_det);
}

/* The batch is already in the slot's device input (network_pipeline_input_device(net, slot), e.g. written by another
 * kernel or uploaded once): forward + decode + NMS + pick without any host -> device copy, pipelined like the others. */
int network_detect_submit_resident(network net, float thresh, float nms, int max_det)
{
    return detect_submit(net, (y2_input){.kind = Y2_IN_RESIDENT}, NULL, thresh, nms, max_det);
}

/* Decoded frames of any size: upload the raw bytes, then byte/255. (load_image_stb) and resize_image
 * (image.c:1950-1993) run on the device, bit-identical to Detector::detect(filename)'s host path
 * (yolo_v2_class.cpp:173-206).  Frames already at the network's resolution take the uint8 first-layer
 * path when the network has one. */
int network_detect_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, float thresh,
                                 float nms, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAMES, .data = frames_hwc, .fw = frame_w, .fh = frame_h};
    return detect_submit(net, in, NULL, thresh, nms, max_det);
}

void network_detect_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, float thresh,
                                 float nms, y2_detection *dets, int *counts, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAMES, .data = frames_hwc, .fw = frame_w, .fh = frame_h};
    detect_batch(net, "network_detect_batch_frames: batches of the submit/wait pipeline are in flight", in, NULL,
                 thresh, nms, dets, NULL, counts, max_det);
}

int network_detect_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    return detect_submit(net, in, NULL, thresh, nms, max_det);
}

void network_detect_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                     const int *frame_h, float thresh, float nms, y2_detection *dets, int *counts,
                                     int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    detect_batch(net, "network_detect_batch_frame_list: batches of the submit/wait pipeline are in flight", in,
                 NULL, thresh, nms, dets, NULL, counts, max_det);
}

int network_detect_submit_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    return detect_submit(net, in, &(stream_list){n, stream_ids, 0, 1}, thresh, nms, max_det);
}

int network_detect_submit_streams_resident(network net, int n, const int *stream_ids, float thresh, float nms,
                                           int max_det)
{
    return detect_submit(net, (y2_input){.kind = Y2_IN_RESIDENT}, &(stream_list){n, stream_ids, 0, 1}, thresh, nms,
                         max_det);
}

void network_detect_batch_streams(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                  const int *frame_w, const int *frame_h, float thresh, float nms,
                                  y2_detection *dets, int *counts, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    detect_batch(net, "network_detect_batch_streams: batches of the submit/wait pipeline are in flight", in,
                 &(stream_list){n, stream_ids, 0, 1}, thresh, nms, dets, NULL, counts, max_det);
}

int network_detect_submit_streams_tracked(network net, int n, const int *stream_ids, const unsigned char *const *frames,
                                          const int *frame_w, const int *frame_h, float thresh, float nms,
                                          int use_mean, int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    return detect_submit(net, in, &(stream_list){n, stream_ids, 1, use_mean, frame_w, frame_h}, thresh, nms, max_det);
}

int network_detect_submit_streams_tracked_resident(network net, int n, const int *stream_ids, const int *frame_w,
                                                   const int *frame_h, float thresh, float nms, int use_mean,
                                                   int max_det)
{
    return detect_submit(net, (y2_input){.kind = Y2_IN_RESIDENT},
                         &(stream_list){n, stream_ids, 1, use_mean, frame_w, frame_h}, thresh, nms, max_det);
}

void network_detect_batch_streams_tracked(network net, int n, const int *stream_ids,
                                          const unsigned char *const *frames, const int *frame_w, const int *frame_h,
                                          float thresh, float nms, int use_mean, y2_bbox *boxes, int *counts,
                                          int max_det)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    detect_batch(net, "network_detect_batch_streams_tracked: batches of the submit/wait pipeline are in flight", in,
                 &(stream_list){n, stream_ids, 1, use_mean, frame_w, frame_h}, thresh, nms, NULL, boxes, counts,
                 max_det);
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

void network_classify_device(network net, int top, y2_class_hit *hits)
{
    layer *l = classify_layer(net, top);
    y2_net_rt *rt = y2_rt(net);
    Y2_CHECK(y2_set_device(rt->device));
    y2_results_reserve_hits(rt, &rt->res, top);
    classify_tail(rt, net, l, top, rt->res.hits_dev);
    y2_results_to_host(&rt->res, Y2_PIPE_CLASSIFY, net.batch, top, rt->stream);
    Y2_CHECK(y2_stream_sync(rt->stream));
    memcpy(hits, rt->res.hits_pinned, (size_t)net.batch * top * sizeof(y2_class_hit));
}

void network_classify_batch(network net, const float *input, int top, y2_class_hit *hits)
{
    classify_layer(net, top);
    network_upload_input(net, input);
    network_forward_device(net);
    network_classify_device(net, top, hits);
}

/* a classify batch into the pipeline: frames are letterboxed (letterbox_image, image.c:1624-1644) on the device */
static int classify_submit(network net, y2_input in, int top)
{
    layer *l = classify_layer(net, top);
    const int s = y2_pipe_claim(net, &in);
    y2_net_rt *rt = y2_rt(net);
    y2_results *res = &rt->pipe[s].res;
    y2_results_reserve_hits(rt, res, top);
    y2_pipe_submit_input(net, s, &in, 1);
    classify_tail(rt, net, l, top, res->hits_dev);
    y2_pipe_queue(rt, s, Y2_PIPE_CLASSIFY, in.n, top);
    return s;
}

int network_classify_wait(network net, y2_class_hit *hits, int top)
{
    const int s = y2_pipe_retire(net, Y2_PIPE_CLASSIFY, top);
    const struct y2_pipe_slot *ps = &y2_rt(net)->pipe[s];
    memcpy(hits, ps->res.hits_pinned, (size_t)ps->n_images * top * sizeof(y2_class_hit));
    return s;
}

/* the classify *_batch_* entries: one submission and its wait, refused while batches of the pipeline are in flight */
static void classify_batch(network net, const char *in_flight, y2_input in, int top, y2_class_hit *hits)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt && rt->pipe_inflight) error(in_flight);
    classify_submit(net, in, top);
    network_classify_wait(net, hits, top);
}

int network_classify_submit(network net, const float *input, int top)
{
    return classify_submit(net, (y2_input){.kind = Y2_IN_F32, .data = input}, top);
}

int network_classify_submit_u8(network net, const unsigned char *input_hwc, int top)
{
    return classify_submit(net, (y2_input){.kind = Y2_IN_U8, .data = input_hwc}, top);
}

int network_classify_submit_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top)
{
    return classify_submit(net, (y2_input){.kind = Y2_IN_FRAMES, .data = frames_hwc, .fw = frame_w, .fh = frame_h},
                           top);
}

int network_classify_submit_resident(network net, int top)
{
    return classify_submit(net, (y2_input){.kind = Y2_IN_RESIDENT}, top);
}

void network_classify_batch_frames(network net, const unsigned char *frames_hwc, int frame_w, int frame_h, int top,
                                   y2_class_hit *hits)
{
    classify_batch(net, "network_classify_batch_frames: batches of the submit/wait pipeline are in flight",
                   (y2_input){.kind = Y2_IN_FRAMES, .data = frames_hwc, .fw = frame_w, .fh = frame_h}, top, hits);
}

int network_classify_submit_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    return classify_submit(net, in, top);
}

void network_classify_batch_frame_list(network net, int n, const unsigned char *const *frames, const int *frame_w,
                                       const int *frame_h, int top, y2_class_hit *hits)
{
    const y2_input in = {.kind = Y2_IN_FRAME_LIST, .list = {n, frames, frame_w, frame_h}};
    classify_batch(net, "network_classify_batch_frame_list: batches of the submit/wait pipeline are in flight", in,
                   top, hits);
}
