/*
 * yolo2_b200_kernels.h — thin C-ABI over the sm_100a CUDA kernels of the
 * YOLOv2 detection forward pass.  Plain pointers and sizes only; no C++ or
 * torch types.  The C host runtime (darknet_b200.h) is written against this
 * header exactly the way the reference's layer code is written against its
 * own `*_ongpu` launchers.
 *
 * Each entry point names the reference interface it replaces
 * (paths relative to /root/reference/src_yolo2).
 *
 * Device tensor layout ("padded NHWC"): an activation tensor with valid
 * extent H x W and C channels is stored as bf16 [B][H+1][W+1][CS] where CS is
 * the channel stride of the buffer it lives in (CS >= C; CS > C when the
 * tensor is a channel slice of a route/concat buffer).  Row H and column W of
 * every image are zero.  With that single zero row/column, the 3x3 "same"
 * convolution becomes a sum of nine GEMMs over *flat* positions
 * p = (b*(H+1) + y)*(W+1) + x, tap (r,s) reading position
 * p + (r-1)*(W+1) + (s-1); every halo read lands on a zero.
 *
 * All functions return 0 on success, a negative Y2_E* code otherwise, and
 * never fall back to a CPU path.
 */
#ifndef YOLO2_B200_KERNELS_H
#define YOLO2_B200_KERNELS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Y2_OK 0
#define Y2_EINVAL (-1)
#define Y2_ECUDA (-2)
#define Y2_ENOMEM (-3)

/* Opaque CUDA stream handle (cudaStream_t).  NULL = legacy default stream. */
typedef void *y2_stream_t;

const char *y2_last_error(void);

/* ---- device runtime (replaces cuda.c:12-158 cuda_set_device / cuda_make_array /
 *      cuda_push_array / cuda_pull_array / cuda_free) -------------------------------- */
int y2_device_count(int *count);
int y2_set_device(int dev);
int y2_get_device(int *dev);
/* keep the calling host thread on the CPUs next to GPU `dev` (PCI local_cpulist); returns the size of the new
 * CPU mask, 0 when the topology is not visible and nothing changed.  y2_host_alloc does the same temporarily so
 * that pinned staging buffers live in the GPU's own NUMA node. */
int y2_bind_thread_to_device(int dev);
int y2_malloc(void **dptr, size_t bytes);
int y2_free(void *dptr);
int y2_memset(void *dptr, int value, size_t bytes, y2_stream_t s);
int y2_host_alloc(void **hptr, size_t bytes);           /* pinned */
int y2_host_free(void *hptr);
int y2_memcpy_h2d(void *dst, const void *src, size_t bytes, y2_stream_t s);
int y2_memcpy_d2h(void *dst, const void *src, size_t bytes, y2_stream_t s);
int y2_stream_create(y2_stream_t *s);
int y2_stream_destroy(y2_stream_t s);
int y2_stream_sync(y2_stream_t s);
int y2_device_sync(void);

/* CUDA-graph capture of a layer schedule (replaces the host loop of
 * network_kernels.cu:43-56 forward_network_gpu). */
typedef void *y2_graph_t;
int y2_graph_begin(y2_stream_t s);
int y2_graph_end(y2_stream_t s, y2_graph_t *g);
int y2_graph_launch(y2_graph_t g, y2_stream_t s);
int y2_graph_destroy(y2_graph_t g);

/* Events for device-side timing. */
typedef void *y2_event_t;
int y2_event_create(y2_event_t *e);
int y2_event_record(y2_event_t e, y2_stream_t s);
int y2_event_elapsed_ms(y2_event_t a, y2_event_t b, float *ms);
int y2_event_sync(y2_event_t e);                       /* host blocks until the event has fired */
int y2_stream_wait_event(y2_stream_t s, y2_event_t e);  /* later work of s waits for e on the device */
int y2_event_destroy(y2_event_t e);

/* ---- convolution (replaces convolutional_kernels.cu:77-131
 *      forward_convolutional_layer_gpu = fill + im2col_ongpu + gemm_ongpu +
 *      normalize_gpu + scale_bias_gpu + add_bias_gpu + activate_array_ongpu) ---------- */

#define Y2_ACT_LINEAR 0
#define Y2_ACT_LEAKY 1
#define Y2_ACT_LOGISTIC 2

#define Y2_OUT_BF16_PADDED 0 /* bf16 [B][H+1][W+1][out_cs], pads written as 0 */
#define Y2_OUT_F32_FLAT 1    /* fp32 [B][H*W][out_cs] (the reference's "flatten"ed NHWC) */
#define Y2_OUT_BF16_POOLED 2 /* the convolution AND the 2x2/2 maxpool behind it (maxpool_layer_kernels.cu:10-48):
                              * bf16 [B][H/2+1][W/2+1][out_cs], pads left untouched (zero at plan time).  3x3 layers
                              * with cin == block_k and cout == npad in {64, 128}, leaky / linear, alpha >= 0 (a
                              * filter with negative alpha has weights and alpha negated by the caller) */

typedef struct y2_conv_desc {
    const void *in;   /* bf16 padded NHWC, already offset to the first input channel */
    int in_cs;        /* channel stride of `in` (elements) */
    int cin;          /* channels read per tap; multiple of block_k */
    int batch, h, w;  /* valid extent (stride-1 'same' conv: output extent is identical) */
    int ksize;        /* 1 or 3 */
    const void *wt;   /* bf16 [npad][ksize*ksize*cin], K index = (r*ksize+s)*cin + c */
    int cout;         /* real filters */
    int npad;         /* rows in wt, multiple of block_n */
    int block_n;      /* 32, 64, 128 or 256 */
    int block_k;      /* 64 (128-byte swizzle) or 32 (64-byte swizzle) */
    const float *alpha; /* [npad]  scale_f / (sqrt(var_f) + 1e-6)  (1 when no batchnorm) */
    const float *beta;  /* [npad]  bias_f - mean_f * alpha_f */
    int act;          /* Y2_ACT_* */
    void *out;        /* already offset to the first output channel */
    int out_cs;       /* channel stride of `out` (elements) */
    int out_mode;     /* Y2_OUT_* */
    int in_order;     /* how the producer of `in` walked it: 0 = first position to last (or unknown), 1 = last to
                       * first.  A plan over a tensor near / above the L2 capacity walks it the other way round so
                       * that it starts with the part that is still L2-resident (y2_conv_plan_order tells which). */
} y2_conv_desc;

typedef struct y2_conv_plan y2_conv_plan; /* tensor maps + launch geometry */

int y2_conv_plan_create(const y2_conv_desc *d, y2_conv_plan **plan);
/* 0: the plan visits (and writes) positions first to last, 1: last to first */
int y2_conv_plan_order(const y2_conv_plan *plan);
int y2_conv_plan_launch(const y2_conv_plan *plan, y2_stream_t s);
void y2_conv_plan_destroy(y2_conv_plan *plan);
/* algorithmic flops of one launch: 2*cout*ksize^2*cin_real*B*H*W is the caller's
 * business; this returns the number of MMA tiles for diagnostics. */
int y2_conv_plan_tiles(const y2_conv_plan *plan);
/* which kernel the plan launches: 0 per-tap (conv_tcgen05_kernel), 1 halo slab (conv_slab_kernel),
 * 2 CTA pair (conv_pair_kernel, tcgen05.mma.cta_group::2), 3 conv + maxpool (conv_pool_kernel) */
int y2_conv_plan_variant(const y2_conv_plan *plan);
/* Host logic of the CTA-pair kernel, exported for the CPU tests: the work lists it hands to `pairs` CTA pairs for
 * `rows` position tiles of `units` 64-filter units each (units % 4 == 0).  balanced = 0: whole 256-filter tiles
 * round-robin; 1: contiguous unit ranges of minimal largest cost, split into pieces of 64..256 filters.
 * out: 4 ints per entry (position tile, first filter, filters, 0), *stride entries per pair, filters == 0 ends a
 * pair's list.  Returns the number of entries written (pairs * *stride) or Y2_EINVAL when cap is too small. */
int y2_pair_schedule(int rows, int units, int pairs, int balanced, int *out, int cap_entries, int *stride);

/* ---- first layer (replaces, for a 3x3/1 'same' convolution over <= 3 input channels followed by a
 *      2x2/2 maxpool: cuda_make_array of the input (network_kernels.cu:399) +
 *      forward_convolutional_layer_gpu (convolutional_kernels.cu:77-131) +
 *      forward_maxpool_layer_gpu (maxpool_layer_kernels.cu:87-97)) ------------------------------ */
/* in: fp32 NCHW [B][c][h][w];  wt: bf16 [32][32] with K index c*9 + r*3 + s (im2col.c:16-39 order),
 * rows >= filters zero;  alpha >= 0 (fold the sign into wt);  out: bf16 padded NHWC of the POOLED
 * extent [B][h/2+1][w/2+1][out_cs], channels 0..31 written, pads left untouched (zero at plan time). */
int y2_stem_prepare(void);
int y2_stem_conv_pool(const float *in, int batch, int c, int h, int w, const void *wt, int npad,
                      const float *alpha, const float *beta, int act, void *out, int out_cs,
                      y2_stream_t s);
/* Same layer fed with the raw decoded image: uint8 interleaved RGB [B][h][w][3]; every byte becomes
 * (float)(byte / 255.) exactly as the reference's loaders do on the host (yolo_v2_class.cpp:129-149
 * load_image_stb, yolo_v2_class.hpp:95-115 mat_to_image), so the result is bit-identical to
 * y2_stem_conv_pool on the converted planar image at a quarter of the upload.  w % 16 == 0. */
int y2_stem_u8_supported(int h, int w); /* 1 when y2_stem_conv_pool_u8 accepts this image size */
int y2_stem_conv_pool_u8(const unsigned char *in_hwc, int batch, int h, int w, const void *wt, int npad,
                         const float *alpha, const float *beta, int act, void *out, int out_cs,
                         y2_stream_t s);

/* ---- layout / packing kernels ------------------------------------------------------ */

/* fp32 NCHW [B][C][H][W] -> bf16 padded NHWC [B][H+1][W+1][cs] (channels >= C zeroed up
 * to cpad).  Replaces the cuda_make_array upload of network_kernels.cu:399. */
int y2_pack_nchw_f32(const float *src, void *dst, int batch, int c, int h, int w,
                     int cpad, int cs, y2_stream_t s);

/* First-layer patch gather: fp32 NCHW [B][C][H][W] -> bf16 [B][H+1][W+1][kpad] where
 * channel k = c*ksize*ksize + r*ksize + s holds in[c][y+r-pad][x+s-pad] (0 outside),
 * the K ordering of im2col.c:16-39.  k >= C*ksize*ksize zeroed. */
int y2_pack_patches_f32(const float *src, void *dst, int batch, int c, int h, int w,
                        int ksize, int kpad, y2_stream_t s);

/* General patch gather for convolutions of any size / stride / padding (the 7x7/2 first layer and
 * the 3x3/2 layers of cfg/resnet50.cfg): the rows of the reference's im2col_cpu (im2col.c:16-39),
 * written as bf16 [B][oh+1][ow+1][kpad] so the convolution becomes a 1x1 GEMM over them.
 *   _f32 : first layer, fp32 NCHW input, K index = c*k*k + r*k + s (the reference's own order);
 *   _bf16: later layers, bf16 padded NHWC input, K index = (r*k + s)*cin_pad + c, kpad = k*k*cin_pad. */
int y2_gather_patches_f32(const float *src, void *dst, int batch, int c, int h, int w, int ksize,
                          int stride, int pad, int oh, int ow, int kpad, y2_stream_t s);
int y2_gather_patches_bf16(const void *in, int in_cs, int cin_pad, int h, int w, void *dst, int batch,
                           int ksize, int stride, int pad, int oh, int ow, y2_stream_t s);
/* _rows_f32: first layer with a 5..8-wide kernel (resnet50's 7x7/2): K index = (c*ksize + r)*8 + s, one
 * aligned 16-byte group per kernel row (s >= ksize zero), kpad >= c*ksize*8. */
int y2_gather_rows_f32(const float *src, void *dst, int batch, int c, int h, int w, int ksize, int stride,
                       int pad, int oh, int ow, int kpad, y2_stream_t s);

/* Decoded frames -> network input on the device: uint8 interleaved RGB [B][src_h][src_w][3] ->
 * fp32 planar [B][3][h][w], = load_image_stb's byte/255. (yolo_v2_class.cpp:129-149) followed by
 * resize_image (image.c:1950-1993), bit-identical to that host path. */
int y2_resize_u8_to_f32(const unsigned char *src, float *dst, int batch, int src_w, int src_h, int w,
                        int h, y2_stream_t s);

/* letterbox_image's geometry (image.c:1624-1644): the src_w x src_h image scaled to fit inside w x h keeping
 * its aspect ratio - the side that limits (compared as (float)w / src_w < (float)h / src_h) gets the target
 * extent, the other src_h*w/src_w resp. src_w*h/src_h in integer arithmetic - placed at
 * ((w - new_w) / 2, (h - new_h) / 2).  new_w or new_h can be 0 (a very thin image): nothing is placed. */
void y2_letterbox_geometry(int src_w, int src_h, int w, int h, int *new_w, int *new_h, int *dx, int *dy);
/* Decoded frames -> letterboxed network input: uint8 interleaved RGB [B][src_h][src_w][3] -> fp32 planar
 * [B][3][h][w], bit-identical to letterbox_image(im, w, h) (image.c:1624-1644) of the (float)(byte / 255.) image:
 * resize_image into the window of y2_letterbox_geometry, .5f everywhere else.  A window 1 pixel wide takes
 * resize_image's edge column.  A window 1 pixel high has no defined result: resize_image's vertical scale
 * divides by zero there and the host code reads outside its image. */
int y2_letterbox_u8_to_f32(const unsigned char *src, float *dst, int batch, int src_w, int src_h, int w, int h,
                           y2_stream_t s);

/* A list of decoded frames, each with its own size, packed into one buffer: frame i (uint8 interleaved RGB
 * [src_h][src_w][3]) starts at byte `offset`, and its resized image fills the window [dx, dx+new_w) x
 * [dy, dy+new_h) of the network canvas, with resize_image's scales (image.c:1954-1955) computed on the host. */
typedef struct y2_frame_window {
    unsigned long long offset;
    int src_w, src_h;
    int dx, dy, new_w, new_h;
    float w_scale, h_scale;
} y2_frame_window;
/* The layout of such a list for a w x h network: frames in list order, each at a 16-byte-aligned offset, then the
 * table of n records (at *table_offset, also 16-byte aligned).  letterbox = 0: every window is the whole canvas
 * (resize_image); 1: the window of y2_letterbox_geometry (letterbox_image).  win (may be NULL) receives the n
 * records.  Returns the packed size in bytes, frames and table, or 0 when n < 1 or a size is <= 0. */
size_t y2_frame_list_layout(int n, const int *frame_w, const int *frame_h, int w, int h, int letterbox,
                            y2_frame_window *win, size_t *table_offset);
/* Packed frames -> fp32 planar [batch][3][h][w] in one launch: image i < n is byte/255. + resize_image into the
 * window of table[i] (a device pointer, normally inside the packed buffer) on a .5f canvas, bit-identical to the
 * host chain; images n..batch-1 are all .5f.  A window 1 pixel high has no defined result (see above). */
int y2_frames_u8_to_f32(const unsigned char *packed, const y2_frame_window *table, int n, float *dst, int batch,
                        int w, int h, y2_stream_t s);

/* bf16 padded NHWC slice -> fp32 NCHW [B][C][H][W] (host-visible l.output layout). */
int y2_unpack_to_nchw_f32(const void *src, float *dst, int batch, int c, int h, int w,
                          int cs, y2_stream_t s);

/* fp32 flat NHWC [B][H*W][cs] -> fp32 NCHW [B][C][H][W]. */
int y2_flat_to_nchw_f32(const float *src, float *dst, int batch, int c, int hw, int cs,
                        y2_stream_t s);

/* fp32 NCHW -> fp32 flat NHWC (blas_kernels.cu:550-572 flatten_kernel, forward=1). */
int y2_nchw_to_flat_f32(const float *src, float *dst, int batch, int c, int hw,
                        y2_stream_t s);

/* ---- maxpool (replaces maxpool_layer_kernels.cu:10-48,87-97) ------------------------ */
int y2_maxpool(const void *in, int in_cs, void *out, int out_cs, int batch, int c,
               int h, int w, int out_h, int out_w, int size, int stride, int pad,
               y2_stream_t s);

/* ---- reorg (replaces blas_kernels.cu:332-362 reorg_kernel, forward=0 as called by
 *      reorg_layer.c:97-104) --------------------------------------------------------- */
int y2_reorg(const void *in, int in_cs, void *out, int out_cs, int batch, int c, int h,
             int w, int stride, y2_stream_t s);

/* The same permutation through a lookup table built once per layer (the index map costs ~15 integer
 * divisions per element): y2_reorg_table fills table[(h/s)*(w/s)*(c*s*s)] with the element offset of
 * every output element's source inside one padded input image; y2_reorg_gather applies it. */
int y2_reorg_table(int *table, int in_cs, int c, int h, int w, int stride, y2_stream_t s);
int y2_reorg_gather(const void *in, int in_cs, void *out, int out_cs, const int *table, int batch,
                    int c, int h, int w, int stride, y2_stream_t s);

/* reverse = 1 layers (reorg_layer.c:80-81, reorg_cpu with forward = 1): in (c, h, w) -> out (c/s^2, h*s, w*s) */
int y2_reorg_table_reverse(int *table, int in_cs, int c, int h, int w, int stride, y2_stream_t s);
int y2_reorg_gather_reverse(const void *in, int in_cs, void *out, int out_cs, const int *table, int batch,
                            int c, int h, int w, int stride, y2_stream_t s);

/* ---- route fallback copy (replaces route_layer.c:104-117 copy_ongpu loop); the
 *      planner normally aliases producers into the concat buffer instead ------------- */
int y2_copy_channels(const void *in, int in_cs, void *out, int out_cs, int batch, int c,
                     int h, int w, y2_stream_t s);

/* ---- region layer forward (replaces region_layer.c:383-422 + 144-177:
 *      flatten + softmax + D2H + CPU logistic) ---------------------------------------- */
/* in: fp32 flat [B][hw][n*(5+classes)] raw conv output; out: same shape, tx..th raw,
 * objectness logistic'd, classes softmax'd (flat or per tree group). */
int y2_region_forward(const float *in, float *out, int batch, int hw, int n, int classes,
                      int softmax, int n_groups, const int *d_group_size,
                      const int *d_group_offset, y2_stream_t s);

/* the same with a row stride on the input: position p's n*(5+classes) values start at in + p*in_cs (wide fp32 heads
 * are stored with rows padded to 16 bytes) */
int y2_region_forward_strided(const float *in, int in_cs, float *out, int batch, int hw, int n, int classes,
                              int softmax, int n_groups, const int *d_group_size,
                              const int *d_group_offset, y2_stream_t s);

/* ---- get_region_boxes (replaces region_layer.c:328-379, flat softmax and
 *      tree-without-map / tree-with-map variants) ------------------------------------- */
/* pred: [B][hw*n][5+classes] (mutated in the tree case, like the reference);
 * boxes: [B][hw*n][4]; probs: [B][hw*n][classes_out]. */
int y2_region_boxes(float *pred, const float *d_biases, float *boxes, float *probs,
                    int batch, int lw, int lh, int n, int classes, float img_w,
                    float img_h, float thresh, int only_objectness, int classfix,
                    int tree_n, const int *d_tree_parent, const int *d_map, int map_n,
                    y2_stream_t s);

/* Same decode that also counts the non-zero probabilities per (image, class) into nz_count[B][classes_out]
 * (atomic increments: the caller zeroes the counters once, y2_collect_ws hands them back zeroed): the
 * candidate counts y2_nms_mark needs, without a separate pass over the probabilities. */
int y2_region_boxes_counted(float *pred, const float *d_biases, float *boxes, float *probs,
                            int batch, int lw, int lh, int n, int classes, float img_w,
                            float img_h, float thresh, int only_objectness, int classfix,
                            int tree_n, const int *d_tree_parent, const int *d_map, int map_n,
                            int *nz_count, y2_stream_t s);

/* ---- 3-frame mean of video streams (replaces, for many streams in one batch, the ring + mean_arrays of
 *      yolo_v2_class.cpp:206-213 and utils.c:420-433) ---------------------------------------------------------- */
/* Stream s owns ring rows 3s .. 3s+2 (slots 0..2) of a ring [max_streams][3][outputs].  For image i of a batch:
 *   src[j]  >= 0: slot j is row src[j] of this batch's region output (an image at or before i wrote it);
 *          == -1: slot j has not been written since open / reset and reads as +0.0f;
 *          <= -2: slot j is ring row -2 - src[j] as it stood before the batch;
 *   commit >= 0: the ring row image i's region output is copied to after the means; -1 when a later image of the
 *          same stream in this batch writes that row. */
typedef struct y2_stream_src {
    int src[3];
    int commit;
} y2_stream_src;
/* The Detector's ring rule (write slot frame_index, mean over the three slots, frame_index = (frame_index + 1) % 3)
 * for a list of n images, image i from stream stream_ids[i], a stream's images in list order.  frame_index and
 * frames_seen ([max_streams]; frames since open / reset, saturating at 3; both 0 for a fresh stream) are read and
 * advanced; plan[n] receives the records.  Host only; Y2_EINVAL (nothing changed) for an id outside 0..max_streams-1. */
int y2_stream_plan(int n, const int *stream_ids, int max_streams, int *frame_index, int *frames_seen,
                   y2_stream_src *plan);
/* mean[i][e] = ((0 + slot0) + slot1) + slot2) / 3 in float with round-to-nearest for the n images of table (a device
 * copy of y2_stream_plan's records); out: the batch's region output [>= n][outputs], ring as above, mean [n][outputs]. */
int y2_stream_mean(const float *out, const float *ring, const y2_stream_src *table, int n, int outputs, float *mean,
                   y2_stream_t s);
/* ring[table[i].commit] = out[i] for every committing image; launch after y2_stream_mean of the same table. */
int y2_stream_commit(const float *out, float *ring, const y2_stream_src *table, int n, int outputs, y2_stream_t s);

/* ---- tracking of video streams (replaces, for many streams in one batch, the pixel conversion of
 *      yolo_v2_class.cpp:228-236 and Detector::tracking, yolo_v2_class.cpp:251-304) ----------------------------------- */
#ifndef Y2_BBOX_DEFINED
#define Y2_BBOX_DEFINED
typedef struct y2_bbox { /* bbox_t (yolo_v2_class.hpp:27-33): pixels, class, track id */
    unsigned int x, y, w, h;
    float prob;
    unsigned int obj_id, track_id;
} y2_bbox;
#endif
#define Y2_TRACK_MAX_STORY 32
/* boxes per frame y2_stream_track holds in shared memory (32 bytes each, within the 227 KB of a block) */
#define Y2_TRACK_MAX_TOTAL 7168
/* One image of a tracked batch.  Stream s keeps a history ring of `story` frames (slot k holds up to `total` boxes and
 * their count) and one next-id counter per class.  The host owns the ring position and fill; the device owns the
 * boxes and the ids. */
typedef struct y2_track_img {
    int image;   /* row of the batch's detection lists */
    int stream;
    int w, h;    /* frame size in pixels, the boxes are scaled to it */
    int head;    /* history slot this frame is pushed to; the newest earlier frame is in slot head-1 (mod story) */
    int len;     /* frames in the history before this one, 0 .. story */
    int restart; /* 1: the stream's ids restart at 1 before this frame (open, reset) */
} y2_track_img;
/* For a list of n images (image i from stream stream_ids[i], frame_w[i] x frame_h[i] pixels): the distinct streams in
 * order of first appearance, each with its images in list order (records recs[offsets[k] .. offsets[k+1]) for stream k,
 * offsets[n_streams] = n).  head, len and restart ([max_streams]; 0, 0, 1 for a stream that starts over) are read and
 * advanced.  Returns n_streams; Y2_EINVAL (nothing changed) for an id outside 0..max_streams-1, a frame size of 0 or
 * less or a story outside 1..Y2_TRACK_MAX_STORY.  Host only. */
int y2_track_plan(int n, const int *stream_ids, const int *frame_w, const int *frame_h, int max_streams, int story,
                  int *head, int *len, int *restart, y2_track_img *recs, int *offsets);
/* Detector::tracking(to_bbox(detections), story) for every image of the plan, one block per stream walking its images
 * in order.  det [images][det_stride] / count [images]: the detection lists (count <= min(total, det_stride));
 * hist [max_streams][story][total], hist_count [max_streams][story], next_id [max_streams][classes] (every
 * obj_id < classes): the device state, read and advanced; out [images][out_stride] receives the first out_stride
 * tracked boxes of each image (tracking itself sees all count[image]).  1 <= total <= Y2_TRACK_MAX_TOTAL. */
struct y2_det; /* below, with the final pick */
int y2_stream_track(const struct y2_det *det, int det_stride, const int *count, const y2_track_img *recs,
                    const int *offsets, int n_streams, int total, int classes, int story, y2_bbox *hist, int *hist_count,
                    unsigned int *next_id, y2_bbox *out, int out_stride, y2_stream_t s);

/* ---- do_nms_sort (replaces box.c:249-277) ------------------------------------------- */
/* boxes [B][total][4], probs [B][total][classes] updated in place. */
int y2_nms_sort(const float *boxes, float *probs, int batch, int total, int classes,
                float thresh, y2_stream_t s);
/* The suppression pass alone, on caller-owned candidate counters nz_count[B][classes]: suppressed entries
 * are left NEGATIVE (-|p|) instead of zero; y2_collect / y2_collect_ws read a negative entry as 0. */
int y2_nms_mark(const float *boxes, float *probs, const int *nz_count, int batch, int total, int classes,
                float thresh, y2_stream_t s);
/* do_nms (box.c:279-297, the unsorted variant used by demo.c / validate_detector_recall): for every pair
 * i < j with box_iou > thresh, per class the smaller of the two probabilities is zeroed, pairs visited in
 * the reference's order.  boxes [total][4], probs [total][classes] updated in place. */
int y2_nms_unsorted(const float *boxes, float *probs, int total, int classes, float thresh, y2_stream_t s);

/* ---- final pick (replaces yolo_v2_class.cpp:221-239): per box max_index over classes,
 *      keep prob > thresh; compacts to det[B][max_det] + count[B] --------------------- */
typedef struct y2_det {
    float x, y, w, h; /* box centre / size, relative units (as box.h:4-6) */
    float prob;
    int obj_id;
    int box_index;
} y2_det;
int y2_collect(const float *boxes, const float *probs, int batch, int total, int classes,
               float thresh, y2_det *det, int *count, int max_det, y2_stream_t s);
/* The same with caller-owned scratch `ws` of y2_collect_ws_bytes() bytes (may be NULL when that is 0) and,
 * optionally, the NMS candidate counters nz_count[B][classes] to be zeroed for the next batch. */
size_t y2_collect_ws_bytes(int batch, int total, int classes);
int y2_collect_ws(const float *boxes, const float *probs, int batch, int total, int classes,
                  float thresh, y2_det *det, int *count, int max_det, void *ws, int *nz_count,
                  y2_stream_t s);

/* ---- softmax-tree detection without the dense pass (yolo9000).  Replaces, for the detection entry points,
 *      softmax_tree (softmax_layer.c:35-47) + hierarchy_predictions (tree.c:37-51) + the tree branch of
 *      get_region_boxes (region_layer.c:349-366) + do_nms_sort + the final pick: only the groups on the path of
 *      classes above .5 are evaluated (see region.cu), results bit-identical to the dense kernels above.
 *  head: the RAW conv output, fp32 [B][lw*lh][head_cs] (box a of a cell at a*(5+classes));
 *  d_child_ptr [classes+2] / d_child_grp: CSR of the groups below every node, node `classes` = the virtual root;
 *  rec: [B][lw*lh*n] records of y2_tree_rec_bytes() bytes each. */
size_t y2_tree_rec_bytes(void);
int y2_region_tree_detect(const float *head, int head_cs, const float *d_biases, int batch, int lw, int lh,
                          int n, int classes, float thresh, int classfix, const int *d_group_size,
                          const int *d_group_offset, const int *d_child_ptr, const int *d_child_grp,
                          void *rec, y2_stream_t s);
int y2_tree_nms_collect(const void *rec, int batch, int total, float thresh, float nms, y2_det *det,
                        int *count, int max_det, y2_stream_t s);

/* ---- classifier tail (config 5) ----------------------------------------------------- */
int y2_avgpool_flat(const float *in, float *out, int batch, int hw, int c, int cs,
                    y2_stream_t s);
int y2_softmax_rows(const float *in, float *out, int rows, int n, float temp,
                    y2_stream_t s);
/* softmax_tree of a [softmax] layer with tree= (softmax_layer.c:35-47): per row, one softmax per WordTree group */
int y2_softmax_tree_rows(const float *in, float *out, int rows, int n, float temp, int n_groups,
                         const int *d_group_size, const int *d_group_offset, y2_stream_t s);
/* hierarchy_predictions (tree.c:37-51, only_leaves = 0) + top_k (utils.c:179-193) per row of a classifier's
 * output: row b is out[b * row_stride .. + n).  With d_tree_parent (parent[n], every parent before its child, at
 * most Y2_CLASSIFY_MAX_TREE_DEPTH levels from a root to a leaf; -1 for a root) the WordTree products are formed first, in scratch: `out` is not modified.  hits[b][top] gets the
 * `top` largest entries in descending order, exactly top_k's result on a NaN-free row, including which of several
 * equal values it keeps and in which order (+0 and -0 are equal).  A NaN ranks below every number, so a row with
 * NaNs still gives `top` distinct valid indices, the numbers first.
 * 1 <= top <= min(n, Y2_CLASSIFY_MAX_TOP), n <= Y2_CLASSIFY_MAX_N. */
#define Y2_CLASSIFY_MAX_TOP 128
#define Y2_CLASSIFY_MAX_N 32768
#define Y2_CLASSIFY_MAX_TREE_DEPTH 64
#ifndef Y2_CLASS_HIT_DEFINED
#define Y2_CLASS_HIT_DEFINED
typedef struct y2_class_hit {
    int index;
    float prob;
} y2_class_hit;
#endif
int y2_classify_topk(const float *out, int row_stride, int batch, int n, int top, const int *d_tree_parent,
                     y2_class_hit *hits, y2_stream_t s);
/* shortcut (replaces shortcut_layer.c:54-59 copy_ongpu + shortcut_gpu (blas_kernels.cu:618-651)
 * + activate_array_ongpu): out = act(in + add sampled per blas.c:57-81).  in/out: bf16 padded
 * NHWC of extent out_h x out_w, out_cpad stored channels (out_c real); add: the `from` layer. */
int y2_shortcut(const void *in, int in_cs, const void *add, int add_cs, int add_c, int add_h,
                int add_w, void *out, int out_cs, int out_c, int out_cpad, int out_h, int out_w,
                int batch, int act, const float *add_f32, int add_f32_cs, float *out_f32, y2_stream_t s);
/* add_f32 / out_f32 (either may be NULL): fp32 copies of the residual stream, padded NHWC with
 * add_f32_cs / out_cpad floats per position.  A chain of shortcuts then accumulates in fp32 (as the
 * reference does) while the convolutions keep reading the bf16 tensors. */

/* ---- connected layer (replaces connected_layer.c:271-293: fill + gemm_ongpu + batchnorm + axpy bias + activate):
 *      the input (a bf16 padded-NHWC tensor, or an fp32 vector with row stride in_stride) becomes one padded-NHWC
 *      position per image, bf16 [B][2][2][kpad] (zero-initialised by the caller), and the layer runs as a 1x1
 *      convolution plan over it.  Tensor sources are packed position-major: k = (y*w + x)*c + ch. */
int y2_fc_pack_tensor(const void *in, int in_cs, int c, int h, int w, void *dst, int kpad, int batch, y2_stream_t s);
int y2_fc_pack_vec(const float *in, int in_stride, int n, void *dst, int kpad, int batch, y2_stream_t s);
/* any activation of activations.h:6-8 in place on a bf16 padded-NHWC tensor (valid positions, real channels) */
int y2_activate_bf16(void *x, int cs, int c, int batch, int h, int w, int activation, y2_stream_t s);

/* ---- fp32 vector helpers behind fill/copy/axpy/scal_ongpu and activate_array_ongpu
 * (blas_kernels.cu:402-470,560-616; activation_kernels.cu:143-159).  inc* in elements.  Not on the
 * detection hot path. */
int y2_vec_fill(long long n, float alpha, float *x, long long incx, y2_stream_t s);
int y2_vec_copy(long long n, const float *x, long long incx, float *y, long long incy, y2_stream_t s);
int y2_vec_axpy(long long n, float alpha, const float *x, long long incx, float *y, long long incy,
                y2_stream_t s);
int y2_vec_scal(long long n, float alpha, float *x, long long incx, y2_stream_t s);
/* activation = the ACTIVATION enum value of activations.h:6-8 (0 LOGISTIC ... 12 LHTAN) */
int y2_vec_activate(float *x, long long n, int activation, y2_stream_t s);
/* fp32 helpers behind gemm_ongpu (gemm.c:173-183: C = ALPHA op(A) op(B) + BETA C, row-major) and im2col_ongpu
 * (im2col_kernels.cu:48-61).  CUDA-core kernels for callers of the helper surface; the network's convolutions are
 * implicit GEMMs on the tensor cores and never use them. */
int y2_sgemm(int TA, int TB, int M, int N, int K, float alpha, const float *A, int lda, const float *B, int ldb,
             float beta, float *C, int ldc, y2_stream_t s);
int y2_im2col_f32(const float *im, int channels, int height, int width, int ksize, int stride, int pad,
                  float *col, y2_stream_t s);
/* for check_error(cudaError_t) (cuda.c:27-49) */
const char *y2_cuda_error_string(int cuda_status);
int y2_cuda_last_status(void);

/* library identity, for the loader tests */
const char *y2_version(void);

#ifdef __cplusplus
}
#endif
#endif
