/*
 * The two-deep submit/wait pipeline: the H2D copy of batch i+1 overlaps the forward pass of batch i, and the results
 * of batch i return under the forward pass of batch i+1.  This file owns the slots (creating them, growing their
 * buffers, releasing them on a re-plan, freeing them), the staging getters, the input half of a submission, and
 * claiming and retiring a slot.  The detection and classify tails and their entry points are in y2_detect.c.
 */
#include "y2_host.h"

#include <stdlib.h>
#include <string.h>

/* ---- results buffers ----------------------------------------------------------------------------- */
/* grows the detection lists to max_det per image for at least `batch` (and cap_batch) images */
void y2_results_reserve_dets(y2_net_rt *rt, y2_results *res, int batch, int max_det)
{
    if (res->det_cap >= max_det && res->det_images >= batch) return;
    y2_free(res->det_dev);
    y2_host_free(res->det_pinned);
    y2_free(res->cnt_dev);
    y2_host_free(res->cnt_pinned);
    res->det_cap = max_det;
    res->det_images = batch > rt->cap_batch ? batch : rt->cap_batch;
    const size_t nd = (size_t)res->det_images * max_det;
    Y2_CHECK(y2_malloc((void **)&res->det_dev, nd * sizeof(y2_det)));
    Y2_CHECK(y2_host_alloc((void **)&res->det_pinned, nd * sizeof(y2_det)));
    Y2_CHECK(y2_malloc((void **)&res->cnt_dev, (size_t)res->det_images * sizeof(int)));
    Y2_CHECK(y2_host_alloc((void **)&res->cnt_pinned, (size_t)res->det_images * sizeof(int)));
}

/* grows the class hits to `top` per image */
void y2_results_reserve_hits(y2_net_rt *rt, y2_results *res, int top)
{
    if (res->hits_cap >= top && res->hits_dev) return;
    y2_free(res->hits_dev);
    y2_host_free(res->hits_pinned);
    const size_t n = (size_t)rt->cap_batch * top;
    Y2_CHECK(y2_malloc((void **)&res->hits_dev, n * sizeof(y2_class_hit)));
    Y2_CHECK(y2_host_alloc((void **)&res->hits_pinned, n * sizeof(y2_class_hit)));
    res->hits_cap = top;
}

/* grows the tracked boxes to `total` per image for at least `batch` (and cap_batch) images */
void y2_results_reserve_boxes(y2_net_rt *rt, y2_results *res, int batch, int total)
{
    if (res->box_cap >= total && res->box_images >= batch) return;
    y2_free(res->box_dev);
    y2_host_free(res->box_pinned);
    res->box_cap = total;
    res->box_images = batch > rt->cap_batch ? batch : rt->cap_batch;
    const size_t nb = (size_t)res->box_images * total;
    Y2_CHECK(y2_malloc((void **)&res->box_dev, nb * sizeof(y2_bbox)));
    Y2_CHECK(y2_host_alloc((void **)&res->box_pinned, nb * sizeof(y2_bbox)));
}

/* queues the device -> host copies of n images' results of a Y2_PIPE_* kind on `stream`: top class hits each, the
 * detection counts and lists, or the counts and tracked boxes */
void y2_results_to_host(const y2_results *res, int kind, int n, int top, y2_stream_t stream)
{
    if (kind == Y2_PIPE_CLASSIFY) {
        Y2_CHECK(y2_memcpy_d2h(res->hits_pinned, res->hits_dev, (size_t)n * top * sizeof(y2_class_hit), stream));
        return;
    }
    Y2_CHECK(y2_memcpy_d2h(res->cnt_pinned, res->cnt_dev, (size_t)n * sizeof(int), stream));
    if (kind == Y2_PIPE_TRACK)
        Y2_CHECK(y2_memcpy_d2h(res->box_pinned, res->box_dev, (size_t)n * res->box_stride * sizeof(y2_bbox), stream));
    else
        Y2_CHECK(y2_memcpy_d2h(res->det_pinned, res->det_dev, (size_t)n * res->det_cap * sizeof(y2_det), stream));
}

/* the first n images' detection lists out of the pinned mirror, each cut to max_det; counts keep the full number */
void y2_results_copy_dets(const y2_results *res, int n, y2_detection *dets, int *counts, int max_det)
{
    for (int b = 0; b < n; ++b) {
        int c = res->cnt_pinned[b];
        counts[b] = c;
        if (c > max_det) c = max_det;
        if (c > res->det_cap) c = res->det_cap;
        memcpy(dets + (size_t)b * max_det, res->det_pinned + (size_t)b * res->det_cap, (size_t)c * sizeof(y2_det));
    }
}

/* the same for the tracked boxes */
void y2_results_copy_boxes(const y2_results *res, int n, y2_bbox *boxes, int *counts, int max_det)
{
    for (int b = 0; b < n; ++b) {
        int c = res->cnt_pinned[b];
        counts[b] = c;
        if (c > max_det) c = max_det;
        if (c > res->box_stride) c = res->box_stride;
        memcpy(boxes + (size_t)b * max_det, res->box_pinned + (size_t)b * res->box_stride, (size_t)c * sizeof(y2_bbox));
    }
}

void y2_results_free(y2_results *res)
{
    y2_free(res->det_dev);
    y2_host_free(res->det_pinned);
    y2_free(res->cnt_dev);
    y2_host_free(res->cnt_pinned);
    y2_free(res->hits_dev);
    y2_host_free(res->hits_pinned);
    y2_free(res->box_dev);
    y2_host_free(res->box_pinned);
}

/* ---- slot lifecycle ------------------------------------------------------------------------------ */
static void pipe_init(y2_net_rt *rt)
{
    if (rt->pipe_ready) return;
    Y2_CHECK(y2_set_device(rt->device));
    Y2_CHECK(y2_stream_create(&rt->copy_stream));
    Y2_CHECK(y2_stream_create(&rt->d2h_stream));
    Y2_CHECK(y2_malloc((void **)&rt->pipe[1].in_dev, rt->in_bytes)); /* slot 0's exists from plan time on */
    Y2_CHECK(y2_host_alloc((void **)&rt->pipe[1].in_pinned, rt->in_bytes));
    for (int s = 0; s < 2; ++s) {
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_h2d));
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_tail));
        Y2_CHECK(y2_event_create(&rt->pipe[s].ev_done));
    }
    rt->pipe_ready = 1;
}

/* the network's first layer runs the fused first-layer kernel, which also reads uint8 input */
static int takes_u8(network net)
{
    y2_layer_rt *r0 = (y2_layer_rt *)net.layers[0].b200;
    return r0 && r0->stem_fused && net.c == 3 && y2_stem_u8_supported(net.h, net.w);
}

/* the uint8 inputs of both slots, once the pipeline is set up */
static void pipe_init_u8(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (rt->pipe[0].in_u8_dev) return;
    if (!takes_u8(net))
        error("uint8 input needs a network whose first layer runs the fused first-layer kernel (3x3 conv over 3 "
              "channels followed by a 2x2/2 maxpool) and a width that is a multiple of 16; use the frames entry");
    const size_t bytes = (size_t)rt->cap_batch * net.h * net.w * 3;
    for (int s = 0; s < 2; ++s) {
        Y2_CHECK(y2_malloc((void **)&rt->pipe[s].in_u8_dev, bytes));
        Y2_CHECK(y2_host_alloc((void **)&rt->pipe[s].in_u8_pinned, bytes));
    }
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

/* the graphs were captured for the old plans and do not survive a re-plan or batch change */
void y2_pipe_release(y2_net_rt *rt)
{
    for (int s = 0; s < 2; ++s) {
        struct y2_pipe_slot *ps = &rt->pipe[s];
        if (ps->graph) y2_graph_destroy(ps->graph);
        if (ps->graph_u8) y2_graph_destroy(ps->graph_u8);
        ps->graph = ps->graph_u8 = 0;
        ps->graph_valid = ps->graph_u8_valid = 0;
    }
}

void y2_pipe_free(y2_net_rt *rt)
{
    y2_pipe_release(rt);
    for (int s = 0; s < 2; ++s) {
        struct y2_pipe_slot *ps = &rt->pipe[s];
        y2_free(ps->in_dev);
        y2_host_free(ps->in_pinned);
        y2_free(ps->in_u8_dev);
        y2_host_free(ps->in_u8_pinned);
        y2_free(ps->frames_dev);
        y2_host_free(ps->frames_pinned);
        y2_results_free(&ps->res);
        if (ps->ev_h2d) y2_event_destroy(ps->ev_h2d);
        if (ps->ev_done) y2_event_destroy(ps->ev_done);
        if (ps->ev_tail) y2_event_destroy(ps->ev_tail);
    }
    if (rt->copy_stream) y2_stream_destroy(rt->copy_stream);
    if (rt->d2h_stream) y2_stream_destroy(rt->d2h_stream);
}

/* ---- staging ------------------------------------------------------------------------------------- */
/* the refusals of every frame-list entry, before anything is staged */
static void check_frame_list(network net, const struct y2_frame_list *fl)
{
    if (!y2_rt(net)) error("network frame list: network has no device plan");
    if (net.c != 3) error("network frame list: needs a network with 3 input channels");
    if (fl->n < 1 || fl->n > net.batch) error("network frame list: the list must hold 1 .. batch frames");
    if (!fl->frames || !fl->w || !fl->h) error("network frame list: NULL frame, width or height array");
    for (int i = 0; i < fl->n; ++i) {
        if (!fl->frames[i]) error("network frame list: NULL frame pointer");
        if (fl->w[i] <= 0 || fl->h[i] <= 0) error("network frame list: a frame size of 0 or less");
    }
}

/* The one place an input is decided: frames at the network's resolution become uint8 input when the network has the
 * first-layer kernel for it; each kind's refusals and lazy set-up; in.n. */
static y2_input pipe_input(network net, y2_input in)
{
    if (in.kind == Y2_IN_FRAME_LIST) check_frame_list(net, &in.list);
    if (!y2_rt(net)) error("network submit: network has no device plan");
    if (in.kind == Y2_IN_FRAMES && in.fw == net.w && in.fh == net.h && takes_u8(net)) in.kind = Y2_IN_U8;
    pipe_init(y2_rt(net));
    if (in.kind == Y2_IN_U8) pipe_init_u8(net);
    if (in.kind == Y2_IN_FRAMES && (net.c != 3 || in.fw <= 0 || in.fh <= 0))
        error("network submit of frames: needs 3-channel input and a frame size");
    in.n = in.kind == Y2_IN_FRAME_LIST ? in.list.n : net.batch;
    return in;
}

/* the checks every staging getter makes (ok: its own argument checks), with the pipeline set up */
static y2_net_rt *staging_rt(network net, int slot, int ok, const char *refusal)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt || slot < 0 || slot > 1 || !ok) error(refusal);
    pipe_init(rt);
    return rt;
}

float *network_pipeline_staging(network net, int slot)
{
    return staging_rt(net, slot, 1, "network_pipeline_staging: bad slot or unplanned network")->pipe[slot].in_pinned;
}

float *network_pipeline_input_device(network net, int slot)
{
    return staging_rt(net, slot, 1, "network_pipeline_input_device: bad slot or unplanned network")->pipe[slot].in_dev;
}

unsigned char *network_pipeline_staging_u8(network net, int slot)
{
    y2_net_rt *rt = staging_rt(net, slot, 1, "network_pipeline_staging_u8: bad slot or unplanned network");
    pipe_init_u8(net);
    return rt->pipe[slot].in_u8_pinned;
}

unsigned char *network_pipeline_staging_frames(network net, int slot, int frame_w, int frame_h)
{
    y2_net_rt *rt = staging_rt(net, slot, frame_w > 0 && frame_h > 0,
                               "network_pipeline_staging_frames: bad slot, frame size or unplanned network");
    if (pipe_input(net, (y2_input){.kind = Y2_IN_FRAMES, .fw = frame_w, .fh = frame_h}).kind == Y2_IN_U8)
        return rt->pipe[slot].in_u8_pinned;
    Y2_CHECK(y2_set_device(rt->device));
    pipe_reserve_frames(rt, slot, (size_t)rt->cap_batch * frame_h * frame_w * 3, NULL);
    return rt->pipe[slot].frames_pinned;
}

unsigned char *network_pipeline_staging_frame_list(network net, int slot, int n, const int *frame_w,
                                                   const int *frame_h, size_t *offsets)
{
    if (!y2_rt(net)) error("network_pipeline_staging_frame_list: network has no device plan");
    y2_net_rt *rt = staging_rt(net, slot, n >= 1 && n <= net.batch && offsets,
                               "network_pipeline_staging_frame_list: bad slot or offsets, or a list not of 1 .. batch "
                               "frames");
    const size_t bytes = y2_frame_list_layout(n, frame_w, frame_h, net.w, net.h, 0, NULL, NULL);
    if (!bytes) error("network_pipeline_staging_frame_list: a frame size of 0 or less");
    Y2_CHECK(y2_set_device(rt->device));
    pipe_reserve_frames(rt, slot, bytes, NULL);
    y2_frame_window *win = (y2_frame_window *)calloc((size_t)n, sizeof(y2_frame_window));
    if (!win) error("network_pipeline_staging_frame_list: out of host memory");
    y2_frame_list_layout(n, frame_w, frame_h, net.w, net.h, 0, win, NULL);
    for (int i = 0; i < n; ++i) offsets[i] = (size_t)win[i].offset;
    free(win);
    return rt->pipe[slot].frames_pinned;
}

int network_pipeline_next_slot(network net)
{
    y2_net_rt *rt = y2_rt(net);
    if (!rt) error("network_pipeline_next_slot: network has no device plan");
    pipe_init(rt);
    return (rt->pipe_head + rt->pipe_inflight) & 1;
}

/* A frame list into slot s: the frames and the record table behind them in the slot's pinned buffer (frames already
 * at their place there are not copied), then one H2D copy of the whole region on the copy stream.  Returns the
 * table's offset in the region. */
static size_t stage_frame_list(network net, int s, const struct y2_frame_list *fl, int letterbox)
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

/* pageable caller memory is staged through the slot's pinned buffer (a host copy; fill the slot's staging buffer
 * directly to avoid it), then copied to the device on the copy stream */
static void stage(void *dev, void *pinned, const void *src, size_t bytes, y2_stream_t copy_stream)
{
    if (src && src != pinned) memcpy(pinned, src, bytes);
    Y2_CHECK(y2_memcpy_h2d(dev, pinned, bytes, copy_stream));
}

/* ---- submission ---------------------------------------------------------------------------------- */
/* Claims the slot the next batch goes to, after the input's checks and the pipeline's own; completes *in. */
int y2_pipe_claim(network net, y2_input *in)
{
    *in = pipe_input(net, *in);
    y2_net_rt *rt = y2_rt(net);
    if (net.batch != rt->plan_batch) error("network batch changed without set_batch_network");
    if (rt->pipe_inflight >= 2) error("network submit: two batches already in flight, wait for one first");
    Y2_CHECK(y2_set_device(rt->device));
    return (rt->pipe_head + rt->pipe_inflight) & 1;
}

/* The input half of a submission, into slot s: the staging copy, the H2D copy on the copy stream, resize (letterbox:
 * letterbox_image) and the forward pass on the network's stream. */
void y2_pipe_submit_input(network net, int s, const y2_input *in, int letterbox)
{
    y2_net_rt *rt = y2_rt(net);
    struct y2_pipe_slot *ps = &rt->pipe[s];
    const int B = net.batch;
    size_t table_off = 0;
    if (in->kind == Y2_IN_FRAME_LIST) {
        table_off = stage_frame_list(net, s, &in->list, letterbox);
    } else if (in->kind == Y2_IN_FRAMES) {
        const size_t bytes = (size_t)B * in->fh * in->fw * 3;
        pipe_reserve_frames(rt, s, bytes, NULL);
        stage(ps->frames_dev, ps->frames_pinned, in->data, bytes, rt->copy_stream);
    } else if (in->kind == Y2_IN_U8) {
        stage(ps->in_u8_dev, ps->in_u8_pinned, in->data, (size_t)B * net.h * net.w * 3, rt->copy_stream);
    } else if (in->kind == Y2_IN_F32) {
        stage(ps->in_dev, ps->in_pinned, in->data, (size_t)B * net.inputs * sizeof(float), rt->copy_stream);
    }
    if (in->kind != Y2_IN_RESIDENT) {
        Y2_CHECK(y2_event_record(ps->ev_h2d, rt->copy_stream));
        Y2_CHECK(y2_stream_wait_event(rt->stream, ps->ev_h2d));
    }
    if (in->kind == Y2_IN_FRAME_LIST) /* byte/255. + resize_image or letterbox_image per frame, .5f behind the list */
        Y2_CHECK(y2_frames_u8_to_f32(ps->frames_dev, (const y2_frame_window *)(ps->frames_dev + table_off), in->n,
                                     ps->in_dev, B, net.w, net.h, rt->stream));
    else if (in->kind == Y2_IN_FRAMES && letterbox) /* byte/255. + letterbox_image, into the slot's fp32 input */
        Y2_CHECK(y2_letterbox_u8_to_f32(ps->frames_dev, ps->in_dev, B, in->fw, in->fh, net.w, net.h, rt->stream));
    else if (in->kind == Y2_IN_FRAMES) /* byte/255. + resize_image, into the slot's fp32 input */
        Y2_CHECK(y2_resize_u8_to_f32(ps->frames_dev, ps->in_dev, B, in->fw, in->fh, net.w, net.h, rt->stream));
    if (in->kind == Y2_IN_U8) {
        rt->input_u8 = 1; /* read while the layer list is captured */
        y2_run_forward_from(net, (float *)ps->in_u8_dev, &ps->graph_u8, &ps->graph_u8_valid);
        rt->input_u8 = 0;
    } else {
        y2_run_forward_from(net, ps->in_dev, &ps->graph, &ps->graph_valid);
    }
}

/* Puts the batch in slot s in flight behind its tail: the results travel on their own stream, so the next batch's
 * forward pass (same compute stream) does not wait behind the device -> host copies of this one. */
void y2_pipe_queue(y2_net_rt *rt, int s, int kind, int n_images, int top)
{
    struct y2_pipe_slot *ps = &rt->pipe[s];
    Y2_CHECK(y2_event_record(ps->ev_tail, rt->stream));
    Y2_CHECK(y2_stream_wait_event(rt->d2h_stream, ps->ev_tail));
    y2_results_to_host(&ps->res, kind, n_images, top, rt->d2h_stream);
    Y2_CHECK(y2_event_record(ps->ev_done, rt->d2h_stream));
    ps->kind = kind;
    ps->n_images = n_images;
    ps->top = top;
    rt->pipe_inflight++;
}

/* Retires the oldest batch in flight once its results are on the host, after checking that it is a batch the caller's
 * wait collects (kind, and top for a classify batch); the caller then copies the results out of the returned slot. */
int y2_pipe_retire(network net, int kind, int top)
{
    static const char *const nothing[] = {"network_detect_wait: nothing in flight",
                                          "network_classify_wait: nothing in flight",
                                          "network_detect_wait_tracked: nothing in flight"};
    /* [wait's kind][kind of the oldest batch] */
    static const char *const other[3][3] = {
        {NULL, "network_detect_wait: the oldest batch in flight is a classify batch, call network_classify_wait",
         "network_detect_wait: the oldest batch in flight is a tracked batch, call network_detect_wait_tracked"},
        {"network_classify_wait: the oldest batch in flight is a detection batch, call network_detect_wait", NULL,
         "network_classify_wait: the oldest batch in flight is a tracked batch, call network_detect_wait_tracked"},
        {"network_detect_wait_tracked: the oldest batch in flight is an untracked detection batch, call "
         "network_detect_wait",
         "network_detect_wait_tracked: the oldest batch in flight is a classify batch, call network_classify_wait",
         NULL}};
    y2_net_rt *rt = y2_rt(net);
    if (!rt || !rt->pipe_ready || rt->pipe_inflight <= 0) error(nothing[kind]);
    const int s = rt->pipe_head;
    struct y2_pipe_slot *ps = &rt->pipe[s];
    if (ps->kind != kind) error(other[kind][ps->kind]);
    if (top != ps->top) error("network_classify_wait: top differs from the one the batch was submitted with");
    Y2_CHECK(y2_event_sync(ps->ev_done));
    rt->pipe_head ^= 1;
    rt->pipe_inflight--;
    return s;
}
