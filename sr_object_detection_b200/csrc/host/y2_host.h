/* Internal header of the C host runtime (not installed). */
#ifndef Y2_HOST_H
#define Y2_HOST_H

#include "darknet_b200.h"
#include "yolo2_b200_kernels.h"

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* abort through the reference's fatal-exit convention when a kernel-ABI call fails */
void y2_fatal(const char *where, int rc);
#define Y2_CHECK(call)                                  \
    do {                                                \
        int _rc = (call);                               \
        if (_rc != Y2_OK) y2_fatal(#call, _rc);         \
    } while (0)

enum { Y2_KIND_BF16_PADDED = 0, Y2_KIND_F32_FLAT = 1, Y2_KIND_F32_VEC = 2, Y2_KIND_NONE = 3 };
enum { Y2_PIPE_DETECT = 0, Y2_PIPE_CLASSIFY = 1, Y2_PIPE_TRACK = 2 }; /* what a pipeline slot's batch computes */

/* per-layer device plan, owned by net.layers[i].b200 */
typedef struct y2_layer_rt {
    /* output view */
    void *out;          /* first channel of this layer's output */
    int out_cs;         /* channel stride (elements) */
    int out_kind;       /* Y2_KIND_* */
    int cpad;           /* channels stored (>= out_c) */
    void *own_buf;      /* allocation owned by this layer, NULL when aliased / placed */
    size_t own_bytes;
    int placed_in;      /* route layer index whose concat buffer holds this output, or -1 */
    int copy_needed;    /* route: bitmask of inputs that need an explicit copy */
    int packed_concat;  /* route: inputs carry padding channels, their real channels are packed by copies */
    /* convolution */
    y2_conv_plan *plan;
    void *wt_dev;       /* bf16 [npad][ktot] */
    float *alpha_dev, *beta_dev;
    int npad, block_n, block_k, cin_pad, ktot;
    int use_patches, kpad;
    int stem_fused;     /* layer 0: conv + the following 2x2/2 maxpool run as one kernel that writes
                           the maxpool layer's buffer; this layer has no device output of its own */
    int pool_fused;     /* a later 3x3 conv whose 2x2/2 maxpool runs in its epilogue (Y2_OUT_BF16_POOLED): same
                           convention, the conv writes the maxpool layer's buffer */
    int fused_into_prev; /* the maxpool of such a pair: its forward is a no-op */
    void *patches;      /* bf16 [B][H+1][W+1][kpad] */
    int wt_dirty;
    int post_act;       /* ACTIVATION applied by a separate pass behind a LINEAR epilogue (the tensor-core epilogue
                           implements leaky / linear / logistic only), -1: none */
    /* connected layer: runs as a 1x1 convolution over one position per image */
    void *fc_in;        /* bf16 [B][2][2][kpad] */
    int fc_src;         /* layer whose output is flattened into fc_in */
    int fc_h, fc_w, fc_c; /* extent of that tensor (h = w = 0: an fp32 vector of fc_c values) */
    /* input packing for a non-patch first layer */
    void *packed_in;
    /* reorg */
    int *reorg_table;   /* gather table of the layer (y2_reorg_table) */
    int write_order;    /* 1: this layer's kernel wrote its output last position first (y2_conv_plan_order) */
    float *stream_f32;  /* shortcut layers: fp32 copy of the output [B][H+1][W+1][cpad] (residual stream) */
    /* region; softmax with tree= (tree_parent_dev only: set when every parent precedes its child) */
    float *boxes_dev, *probs_dev;
    float *biases_dev;
    int *tree_parent_dev, *group_size_dev, *group_offset_dev, *map_dev;
    int probs_classes;
    int *nms_cnt_dev;   /* [B][classes] NMS candidate counters, zero between batches (owned per network: two
                           networks in flight on one GPU must not share them) */
    void *collect_ws;   /* per-box maxima scratch of the final pick (wide class rows) */
    void *tile_ws;      /* spill scratch of the tiled merge's NMS (y2_tile_nms_ws_bytes), grown on demand */
    size_t tile_ws_bytes;
    /* softmax tree: CSR of the groups below every node (node `classes` = virtual root) and the per-box records
     * of the sparse detection path; the dense region forward then runs on demand only (region_stale) */
    int *child_ptr_dev, *child_grp_dev;
    void *tree_rec_dev;
    /* profiling */
    y2_event_t ev0, ev1;
} y2_layer_rt;

/* video streams of network_detect_submit_streams (network_streams_open).  They outlive a re-plan
 * (set_batch_network, resize_network) and are freed with the network. */
typedef struct y2_streams {
    int max_streams;
    int outputs;           /* region outputs per image when opened */
    float *ring_dev;       /* [max_streams][3][outputs], rows defined once written (y2_stream_plan never reads others) */
    int *frame_index;      /* [max_streams] ring slot of the stream's next frame */
    int *frames_seen;      /* [max_streams] frames since open / reset, saturating at 3 */
    float *mean_dev;       /* [mean_cap][outputs] the means the decode reads */
    int mean_cap;
    /* per pipeline slot, for table_cap[slot] images: the ring plan (y2_stream_src[n]), then the tracking plan
     * (y2_track_img[n], int offsets[n + 1]); one host -> device copy a batch */
    unsigned char *table_pinned[2], *table_dev[2];
    int table_cap[2];
    /* tracking (network_streams_track), story 0 when off.  The device holds the boxes and ids, the host the ring
     * position, fill and start-over flag of each stream (y2_track_plan). */
    int story, total, classes;
    y2_bbox *hist_dev;          /* [max_streams][story][total] */
    int *hist_cnt_dev;          /* [max_streams][story] */
    unsigned int *next_id_dev;  /* [max_streams][classes] */
    int *track_head, *track_len, *track_restart; /* [max_streams] */
} y2_streams;

/* what a batch hands back, each a device buffer with a pinned mirror (y2_pipeline.c) */
typedef struct y2_results {
    y2_det *det_dev, *det_pinned;         /* [det_images][det_cap] detection lists */
    int *cnt_dev, *cnt_pinned;            /* [det_images] detections per image */
    int det_cap, det_images;
    y2_class_hit *hits_dev, *hits_pinned; /* [cap_batch][hits_cap] class hits */
    int hits_cap;
    y2_bbox *box_dev, *box_pinned;        /* [box_images][box_cap] tracked boxes; a batch uses rows of box_stride */
    int box_cap, box_images, box_stride;
} y2_results;

/* what a submission feeds the network; y2_pipe_claim completes it */
typedef enum {
    Y2_IN_F32,        /* fp32 planar [B][c][h][w] */
    Y2_IN_U8,         /* uint8 interleaved RGB [B][h][w][3] at the network's resolution */
    Y2_IN_FRAMES,     /* uint8 interleaved RGB frames [B][fh][fw][3] of any size */
    Y2_IN_FRAME_LIST, /* 1 .. B frames of their own sizes */
    Y2_IN_FRAME_DESCS, /* 1 .. B frame descriptors: RGB, BGR or NV12 with a pitch, in host or device memory */
    Y2_IN_TILED,      /* frame descriptors cut into tiles (descs + tiling), 1 .. B tiles in all */
    Y2_IN_RESIDENT,   /* nothing: the slot's device input already holds the batch */
} y2_input_kind;

typedef struct {
    y2_input_kind kind;
    const void *data;          /* NULL: already in the slot's pinned staging buffer */
    int fw, fh;                /* Y2_IN_FRAMES */
    struct y2_frame_list {     /* Y2_IN_FRAME_LIST: n frames of their own sizes */
        int n;
        const unsigned char *const *frames;
        const int *w, *h;
    } list;
    struct y2_frame_descs {    /* Y2_IN_FRAME_DESCS */
        int n;
        const y2_frame_desc *d;
        void *ready;           /* cudaEvent_t the compute stream waits for before it reads device frames, or NULL */
    } descs;
    const y2_tiling *tiling;   /* Y2_IN_TILED */
    y2_tile_layout tiles;      /* Y2_IN_TILED: the staged plan, y2_pipe_claim fills it */
    int n;                     /* images the batch hands back: the list's length (frames), else the batch */
} y2_input;

typedef struct y2_net_rt {
    int device;
    y2_streams *streams; /* NULL until network_streams_open */
    y2_stream_t stream;
    int cap_batch;       /* batch the buffers were sized for */
    int plan_batch;      /* batch the plans/tensor maps were built for */
    int plan_w, plan_h;
    size_t in_bytes;     /* of a slot's fp32 input */
    float *out_pinned;   /* staging of the network output */
    size_t out_bytes;
    int eager;
    int launches;
    int profile;
    y2_results res;      /* of network_detect_device / network_classify_device */
    float *export_dev;   /* fp32 scratch for layer export */
    size_t export_bytes;
    /* two-deep submit/wait pipeline (y2_pipeline.c).  Slot 0's fp32 input and graph are also the synchronous
     * path's (network_upload_input, network_forward_device) and exist from plan time on; everything else in a slot
     * is allocated at first use.  The graphs go when the plans are rebuilt (set_batch_network), the rest with the
     * network's device plan. */
    struct y2_pipe_slot {
        float *in_dev, *in_pinned; /* fp32 NCHW input */
        y2_graph_t graph;
        int graph_valid;
        /* raw uint8 HWC input of the same slot (Y2_IN_U8) */
        unsigned char *in_u8_dev, *in_u8_pinned;
        y2_graph_t graph_u8;
        int graph_u8_valid;
        /* decoded frames of any size or a frame list: resized or letterboxed on the device into in_dev */
        unsigned char *frames_dev, *frames_pinned;
        size_t frames_cap;
        y2_results res;
        y2_event_t ev_h2d, ev_tail, ev_done;
        int kind;           /* Y2_PIPE_* of the batch in the slot */
        int n_images;       /* images the wait hands back */
        int top;            /* hits per image of a classify batch, 0 for a detection batch */
    } pipe[2];
    y2_stream_t copy_stream; /* host -> device uploads of the pipeline */
    y2_stream_t d2h_stream;  /* detection lists back to the host, under the next batch's forward pass */
    int pipe_ready, pipe_head, pipe_inflight;
    int input_u8;        /* the forward pass being issued reads uint8 HWC images (first-layer kernel only) */
    int defer_region;    /* softmax-tree region layer: its dense forward is not part of the schedule, it runs when
                            somebody asks for the layer's output (the detection entries never do) */
    int region_stale;    /* a forward pass ran since the region output was last computed */
} y2_net_rt;

static inline y2_net_rt *y2_rt(network net) { return (y2_net_rt *)net.b200; }
static inline y2_layer_rt *y2_lrt(layer l) { return (y2_layer_rt *)l.b200; }

/* y2_network.c */
void y2_plan_network(network *net);
void y2_unplan_network(network *net);
void y2_push_convolutional_layer(layer *l);
int y2_output_layer_index(network net);
void y2_run_forward_from(network net, float *in_dev, y2_graph_t *graph, int *graph_valid);

/* y2_pipeline.c */
void y2_pipe_release(y2_net_rt *rt);
void y2_pipe_free(y2_net_rt *rt);
int y2_pipe_claim(network net, y2_input *in);
void y2_pipe_submit_input(network net, int s, const y2_input *in, int letterbox);
void y2_pipe_queue(y2_net_rt *rt, int s, int kind, int n_images, int top);
int y2_pipe_retire(network net, int kind, int top);
void y2_results_reserve_dets(y2_net_rt *rt, y2_results *res, int batch, int max_det);
void y2_results_reserve_hits(y2_net_rt *rt, y2_results *res, int top);
void y2_results_reserve_boxes(y2_net_rt *rt, y2_results *res, int batch, int total);
void y2_results_to_host(const y2_results *res, int kind, int n, int top, y2_stream_t stream);
void y2_results_copy_dets(const y2_results *res, int n, y2_detection *dets, int *counts, int max_det);
void y2_results_copy_boxes(const y2_results *res, int n, y2_bbox *boxes, int *counts, int max_det);
void y2_results_free(y2_results *res);

/* y2_detect.c */
void y2_streams_free(y2_net_rt *rt);

/* layer constructors, per-layer forwards and resizes: declared in include/darknet_b200.h */
void forward_no_cpu_path(layer l, network_state state);

uint16_t y2_f32_to_bf16(float f);

#ifdef __cplusplus
}
#endif
#endif
