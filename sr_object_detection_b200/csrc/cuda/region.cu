// Region layer forward, box decoding and final pick on the GPU.
// Compiled with -fmad=false -prec-div=true: every float expression below mirrors the
// C expression types of the reference so that thresholds, ties and the keep set come out
// bit-identical (SURVEY.md section 8 "numerical contract").
//
// Replaces: forward_region_layer_gpu / forward_region_layer (region_layer.c:383-422,
// 144-177), softmax (blas.c:205-221), softmax_tree (softmax_layer.c:35-47),
// get_region_boxes / get_region_box (region_layer.c:328-379, 73-85),
// hierarchy_predictions (tree.c:37-51), max_index pick (yolo_v2_class.cpp:221-239).
#include "y2_common.cuh"

#include <float.h>
#include <stdlib.h>

namespace y2 {

// activations.h:35  static inline float logistic_activate(float x){return 1./(1. + exp(-x));}
__device__ __forceinline__ float logistic_ref(float x)
{
    return (float)(1. / (1. + exp((double)(-x))));
}

// ---------------------------------------------------------------------------------
// region forward, WordTree softmax (softmax_tree, softmax_layer.c:35-47): one LANE per (box, group).
// The groups of a WordTree are small (9k.tree: 1723 groups, median 3, 99th percentile 28 classes), so a
// warp per group wastes 29 of 32 lanes on 26 million warp tasks at yolo9000 batch 16 (8 ms; that
// warp-per-group kernel was removed later and is in the history).  Here every lane runs the
// reference's three serial loops over its own group; the few groups wider than a warp are then
// finished by the whole warp, lanes over classes, the float sum still accumulated in class order.
// ---------------------------------------------------------------------------------
__global__ void region_forward_tree_kernel(const float *__restrict__ in, int in_cs, int anchors, float *__restrict__ out, long long boxes,
                                           int classes, int softmax, int n_groups,
                                           const int *__restrict__ group_size, const int *__restrict__ group_offset)
{
    const int lane = threadIdx.x & 31;
    const long long t0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const int size = classes + 5;
    const long long work = boxes * n_groups;
    for (long long wb = t0 - lane; wb < work; wb += nthreads) {  // warp-uniform trip count
        const long long t = wb + lane;
        const bool active = t < work;
        const long long box = active ? t / n_groups : 0;
        const int g = active ? (int)(t - box * n_groups) : 0;
        const int off = group_offset[g];
        const int n = active ? group_size[g] : 0;
        const float *x = in + (box / anchors) * in_cs + (box % anchors) * size;
        float *o = out + box * size;
        if (active && g == 0) {
            o[0] = x[0];
            o[1] = x[1];
            o[2] = x[2];
            o[3] = x[3];
            o[4] = logistic_ref(x[4]);
        }
        const float *xi = x + 5 + off;
        float *oi = o + 5 + off;
        const bool wide = n > 32;
        if (!wide) {
            if (!softmax) {
                for (int i = 0; i < n; ++i) oi[i] = xi[i];
            } else {
                float largest = -FLT_MAX;
                for (int i = 0; i < n; ++i) {
                    const float v = xi[i];
                    if (v > largest) largest = v;
                }
                float sum = 0.f;
                for (int i = 0; i < n; ++i) {
                    const float arg = xi[i] / 1.f - largest / 1.f;  // temperature 1, float expression
                    const float e = (float)exp((double)arg);
                    sum = sum + e;
                    oi[i] = e;
                }
                for (int i = 0; i < n; ++i) oi[i] = oi[i] / sum;
            }
        }
        // groups wider than a warp: all lanes, one such group at a time
        unsigned todo = __ballot_sync(0xffffffffu, wide);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const long long wbox = __shfl_sync(0xffffffffu, box, src);
            const int woff = __shfl_sync(0xffffffffu, off, src);
            const int wn = __shfl_sync(0xffffffffu, n, src);
            const float *wx = in + (wbox / anchors) * in_cs + (wbox % anchors) * size + 5 + woff;
            float *wo = out + wbox * size + 5 + woff;
            if (!softmax) {
                for (int i = lane; i < wn; i += 32) wo[i] = wx[i];
                continue;
            }
            float largest = -FLT_MAX;
            for (int i = lane; i < wn; i += 32) {
                const float v = wx[i];
                if (v > largest) largest = v;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const float other = __shfl_xor_sync(0xffffffffu, largest, d);
                if (other > largest) largest = other;
            }
            float sum = 0.f;
            for (int base = 0; base < wn; base += 32) {
                const int i = base + lane;
                float e = 0.f;
                if (i < wn) {
                    const float arg = wx[i] / 1.f - largest / 1.f;
                    e = (float)exp((double)arg);
                    wo[i] = e;
                }
                const int cnt = (wn - base) < 32 ? (wn - base) : 32;
                for (int j = 0; j < cnt; ++j) sum = sum + __shfl_sync(0xffffffffu, e, j);
            }
            for (int i = lane; i < wn; i += 32) wo[i] = wo[i] / sum;
        }
    }
}

// ---------------------------------------------------------------------------------
// region forward, flat softmax (no tree): FOUR lanes per box, eight boxes per warp.
// A warp per box spends a whole warp on 20 classes plus a serial logistic in one
// lane and is issue-bound (54 080 boxes x ~250 warp instructions at yolo-voc b64).  Here lane q of
// a box evaluates the double-precision exps of classes q, q+4, ... and one of the pass-through /
// objectness values; the float sum still runs in class order: round k hands the four terms of
// classes 4k..4k+3 through quad shuffles and every lane adds them in that order, so the sequence of
// roundings is the reference's serial loop (blas.c:205-221).
// ---------------------------------------------------------------------------------
__global__ void region_forward_flat_kernel(const float *__restrict__ in, int in_cs, int anchors, float *__restrict__ out, long long boxes,
                                           int classes, int softmax)
{
    const int lane = threadIdx.x & 31;
    const int q = lane & 3;
    const int qbase = lane & ~3;
    const long long quad0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 2;
    const long long nquads = ((long long)gridDim.x * blockDim.x) >> 2;
    const int size = classes + 5;
    const int rounds = (classes + 3) >> 2;
    // warp-uniform trip count: the first quad of the warp decides
    for (long long wb = quad0 - (lane >> 2); wb < boxes; wb += nquads) {
        const long long box = wb + (lane >> 2);
        const bool active = box < boxes;
        const long long bx = active ? box : 0;
        const float *x = in + (bx / anchors) * in_cs + (bx % anchors) * size;
        float *o = out + bx * size;
        if (active) {
            if (q == 0) {
                o[0] = x[0];
                o[1] = x[1];
            } else if (q == 1) {
                o[2] = x[2];
                o[3] = x[3];
            } else if (q == 2) {
                o[4] = logistic_ref(x[4]);
            }
        }
        const float *xi = x + 5;
        float *oi = o + 5;
        if (!softmax) {
            if (active)
                for (int i = q; i < classes; i += 4) oi[i] = xi[i];
            continue;
        }
        float largest = -FLT_MAX;
        for (int i = q; i < classes; i += 4) {
            const float v = xi[i];
            if (v > largest) largest = v;
        }
#pragma unroll
        for (int d = 1; d <= 2; d <<= 1) {
            const float other = __shfl_xor_sync(0xffffffffu, largest, d);
            if (other > largest) largest = other;
        }
        float sum = 0.f;
        for (int k = 0; k < rounds; ++k) {
            const int i = 4 * k + q;
            float e = 0.f;
            if (i < classes) {
                const float arg = xi[i] / 1.f - largest / 1.f;  // temperature 1, float expression
                e = (float)exp((double)arg);
                if (active) oi[i] = e;
            }
            const int cnt = (classes - 4 * k) < 4 ? (classes - 4 * k) : 4;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float t = __shfl_sync(0xffffffffu, e, qbase + j);
                if (j < cnt) sum = sum + t;
            }
        }
        if (active)
            for (int i = q; i < classes; i += 4) oi[i] = oi[i] / sum;
    }
}

// ---------------------------------------------------------------------------------
// get_region_boxes, flat-softmax variant (region_layer.c:328-347, 367-377).
// Two grid-stride passes in one launch: (1) one thread per box COMPONENT (x, y, w, h), so the four
// double-precision transcendentals of a box run in four adjacent lanes and the float4 box comes out
// of coalesced stores; (2) one thread per (box, class) probability.  (One thread per box doing all
// four, as a side job of the class-0 thread, left 19 of 20 lanes idle through ~300 instructions.)
// ---------------------------------------------------------------------------------
__global__ void region_boxes_flat_kernel(const float *__restrict__ pred, const float *__restrict__ biases,
                                         float *__restrict__ boxes, float *__restrict__ probs, int batch,
                                         int lw, int lh, int n, int classes, float img_w, float img_h,
                                         float thresh, int only_objectness, int classfix, int *__restrict__ nz_count)
{
    const int per_img = lw * lh * n;
    const int size = classes + 5;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    // get_region_box, DOABS branch (region_layer.c:76-83)
    const long long ncomp = (long long)batch * per_img * 4;
    for (long long t = tid; t < ncomp; t += nthreads) {
        const int comp = (int)(t & 3);
        const long long bi = t >> 2;
        const int index = (int)(bi % per_img);
        const float *x = pred + bi * size;
        const int an = index % n;
        const int cell = index / n;
        float v;
        if (comp == 0) {
            v = ((cell % lw) + logistic_ref(x[0])) / lw;
            v *= img_w;
        } else if (comp == 1) {
            v = ((cell / lw) + logistic_ref(x[1])) / lh;
            v *= img_h;
        } else if (comp == 2) {
            v = (float)(exp((double)x[2]) * (double)biases[2 * an] / (double)lw);
            v *= img_w;
        } else {
            v = (float)(exp((double)x[3]) * (double)biases[2 * an + 1] / (double)lh);
            v *= img_h;
        }
        boxes[t] = v;
    }
    const long long total = (long long)batch * per_img * classes;
    for (long long t = tid; t < total; t += nthreads) {
        const int j = (int)(t % classes);
        const long long bi = t / classes; // b*per_img + index
        const float *x = pred + bi * size;
        float scale = x[4];
        if (classfix == -1 && scale < .5) scale = 0;
        const float prob = scale * x[5 + j];
        float pv = (prob > thresh) ? prob : 0;
        if (j == 0 && only_objectness) pv = scale;
        probs[t] = pv;
        // candidate counters of the NMS behind it (nms_count_kernel's job, folded in): non-zero entries per
        // (image, class)
        if (nz_count && pv != 0.f) atomicAdd(&nz_count[(bi / per_img) * classes + j], 1);
    }
}

// ---------------------------------------------------------------------------------
// hierarchy_predictions (tree.c:37-51, only_leaves = 0) by one block: hv[j] = x[j] * hv[parent[j]], parents
// precede children.  Walked in chunks of blockDim classes: a node climbs only to its first ancestor BELOW the
// chunk, whose value is final, and multiplies back down in the reference's association (a WordTree is nearly
// breadth-first, so that is one or two steps instead of the whole path to the root).  Every thread of the block
// calls it; it ends with a __syncthreads, so hv is complete on return.  A node climbs at most 64 steps: trees
// deeper than 64 levels are not supported (the classify entries refuse them at plan time).
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void hierarchy_walk(const float *x, float *hv, const int *__restrict__ parent, int classes)
{
    for (int base = 0; base < classes; base += blockDim.x) {
        const int j = base + threadIdx.x;
        if (j < classes) {
            int path[64];
            int depth = 0;
            int c = j;
            while (c >= base && depth < 64) {
                path[depth++] = c;
                c = parent[c];
            }
            float v = (c >= 0) ? hv[c] : 1.f;  // x * 1.f is exact: a root keeps its own value
            for (int d = depth - 1; d >= 0; --d) v = x[path[d]] * v;
            hv[j] = v;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
// get_region_boxes, softmax-tree variants (region_layer.c:349-366).  One block per box:
// the class scores are staged in shared memory, hierarchy_predictions is evaluated per
// node by walking to the root and multiplying back down (float multiply commutes, so
// v(j) = x[j] * v(parent) is reproduced exactly), then either the coco9k map lookup or
// the "highest index above .5" selection runs.  pred is mutated like the reference.
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) region_boxes_tree_kernel(float *__restrict__ pred, const float *__restrict__ biases,
                                         float *__restrict__ boxes, float *__restrict__ probs, int batch,
                                         int lw, int lh, int n, int classes, float img_w, float img_h,
                                         float thresh, int only_objectness, int classfix,
                                         const int *__restrict__ parent, const int *__restrict__ map, int map_n,
                                         int *__restrict__ nz_count)
{
    extern __shared__ float sh[]; // [classes] raw, [classes] hierarchical
    float *sx = sh;
    float *hv = sh + classes;
    __shared__ int s_found;
    const int per_img = lw * lh * n;
    const long long nboxes = (long long)batch * per_img;
    const int size = classes + 5;
    const int out_classes = map ? map_n : classes;
    for (long long bi = blockIdx.x; bi < nboxes; bi += gridDim.x) {
        float *x = pred + bi * size;
        const int index = (int)(bi % per_img);
        for (int j = threadIdx.x; j < classes; j += blockDim.x) sx[j] = x[5 + j];
        if (threadIdx.x == 0) s_found = -1;
        __syncthreads();
        float scale = x[4];
        if (classfix == -1 && scale < .5) scale = 0;
        hierarchy_walk(sx, hv, parent, classes);
        float *pr = probs + bi * out_classes;
        if (map) {
            for (int j = threadIdx.x; j < classes; j += blockDim.x) x[5 + j] = hv[j];
            for (int j = threadIdx.x; j < map_n; j += blockDim.x) {
                const float prob = scale * hv[map[j]];
                const float pv = (prob > thresh) ? prob : 0;
                pr[j] = pv;
                if (nz_count && pv != 0.f && !(only_objectness && j == 0))
                    atomicAdd(&nz_count[(bi / per_img) * out_classes + j], 1);
            }
        } else {
            int best = -1;
            for (int j = threadIdx.x; j < classes; j += blockDim.x)
                if (hv[j] > .5 && j > best) best = j;
            if (best >= 0) atomicMax(&s_found, best);
            __syncthreads();
            const int found = s_found;
            for (int j = threadIdx.x; j < classes; j += blockDim.x) {
                const float v = (j == found) ? hv[j] : 0.f;
                x[5 + j] = v;
                const float pv = (scale > thresh) ? v : 0;
                pr[j] = pv;
                if (nz_count && pv != 0.f && !(only_objectness && j == 0))
                    atomicAdd(&nz_count[(bi / per_img) * out_classes + j], 1);
            }
        }
        if (threadIdx.x == 0) {
            if (only_objectness) {
                pr[0] = scale;
                if (nz_count && scale != 0.f) atomicAdd(&nz_count[(bi / per_img) * out_classes], 1);
            }
            const int an = index % n;
            const int cell = index / n;
            const int row = cell / lw;
            const int col = cell % lw;
            float bx = (col + logistic_ref(x[0])) / lw;
            float by = (row + logistic_ref(x[1])) / lh;
            float bw = (float)(exp((double)x[2]) * (double)biases[2 * an] / (double)lw);
            float bh = (float)(exp((double)x[3]) * (double)biases[2 * an + 1] / (double)lh);
            bx *= img_w;
            by *= img_h;
            bw *= img_w;
            bh *= img_h;
            *reinterpret_cast<float4 *>(boxes + bi * 4) = make_float4(bx, by, bw, bh);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
// final pick (yolo_v2_class.cpp:221-239 / utils.c:533-545 max_index): per box the first
// maximum over classes; keep when prob > thresh; emit in box-index order.
// One block per image, one warp per box, ordered compaction by a block scan.
// ---------------------------------------------------------------------------------
// Wide class rows (yolo9000: 9418 classes): the first-maximum scan of one box is spread over a warp and the
// boxes of ALL images over the grid; collect_kernel then only compacts.  Lane l scans classes l, l+32, ...
// in increasing order with strict > (its first maximum), the warp keeps the largest value and, among equal
// values, the smallest index - the result of the reference's serial scan.
__global__ void box_argmax_kernel(const float *__restrict__ probs, long long nboxes, int classes,
                                  float *__restrict__ best_out, int *__restrict__ arg_out)
{
    const int lane = threadIdx.x & 31;
    const long long w0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long i = w0; i < nboxes; i += nw) {
        const float *p = probs + i * classes;
        float best = -FLT_MAX;
        int arg = 0x7fffffff;
        for (int j = lane; j < classes; j += 32) {
            const float v = fmaxf(__ldg(p + j), 0.f);  // negative = suppressed by nms_mark_kernel = 0
            if (arg == 0x7fffffff || v > best) { best = v; arg = j; }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, d);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, d);
            if (oa != 0x7fffffff && (arg == 0x7fffffff || ob > best || (ob == best && oa < arg))) { best = ob; arg = oa; }
        }
        if (lane == 0) {
            best_out[i] = best;
            arg_out[i] = arg;
        }
    }
}

__global__ void collect_kernel(const float *__restrict__ boxes, const float *__restrict__ probs, int total,
                               int classes, float thresh, y2_det *__restrict__ det, int *__restrict__ count,
                               int max_det, const float *__restrict__ pre_best, const int *__restrict__ pre_arg,
                               int *__restrict__ nz_count)
{
    extern __shared__ int s_flag[]; // [total] obj id or -1, then prefix
    float *s_prob = reinterpret_cast<float *>(s_flag + total);
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const float *pb = probs + (size_t)b * total * classes;
    // one thread per box: max_index (utils.c:533-545) is a sequential scan with strict >, the first
    // maximum wins; a box's class row is contiguous, so the scan runs on 16-byte loads where it can
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        if (pre_best) {  // box_argmax_kernel did the scan
            const float bv = pre_best[(size_t)b * total + i];
            s_flag[i] = (bv > thresh) ? pre_arg[(size_t)b * total + i] : -1;
            s_prob[i] = bv;
            continue;
        }
        const float *p = pb + (size_t)i * classes;
        // probabilities are >= 0; a negative entry is one nms_mark_kernel suppressed (the reference has
        // written 0 there, box.c:271): the fmaxf below is nms_clear_kernel folded into this scan
        float best = fmaxf(p[0], 0.f);
        int arg = 0;
        int j = 1;
        if ((classes & 3) == 0 && ((uintptr_t)p & 15) == 0) {
            const float4 *p4 = reinterpret_cast<const float4 *>(p);
            for (int q = 0; q < classes / 4; ++q) {
                float4 v = __ldg(p4 + q);
                v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                if (q > 0 && v.x > best) { best = v.x; arg = 4 * q; }
                if (v.y > best) { best = v.y; arg = 4 * q + 1; }
                if (v.z > best) { best = v.z; arg = 4 * q + 2; }
                if (v.w > best) { best = v.w; arg = 4 * q + 3; }
            }
            j = classes;
        }
        for (; j < classes; ++j) {
            const float v = fmaxf(__ldg(p + j), 0.f);
            if (v > best) { best = v; arg = j; }
        }
        s_flag[i] = (best > thresh) ? arg : -1;
        s_prob[i] = best;
    }
    __syncthreads();
    // ordered compaction (box-index order, like the reference's loop): ballot + warp-total scan per
    // chunk of blockDim boxes, running offset carried from chunk to chunk
    __shared__ int s_warp_total[32];
    __shared__ int s_running;
    if (threadIdx.x == 0) s_running = 0;
    __syncthreads();
    y2_det *d = det + (size_t)b * max_det;
    const float4 *bx = reinterpret_cast<const float4 *>(boxes) + (size_t)b * total;
    for (int base = 0; base < total; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int obj = (i < total) ? s_flag[i] : -1;
        const unsigned ballot = __ballot_sync(0xffffffffu, obj >= 0);
        if (lane == 0) s_warp_total[warp] = __popc(ballot);
        __syncthreads();
        int before = s_running;
        for (int wv = 0; wv < warp; ++wv) before += s_warp_total[wv];
        const int pos = before + __popc(ballot & ((1u << lane) - 1u));
        if (obj >= 0 && pos < max_det) {
            const float4 q = bx[i];
            y2_det o;
            o.x = q.x; o.y = q.y; o.w = q.z; o.h = q.w;
            o.prob = s_prob[i];
            o.obj_id = obj;
            o.box_index = i;
            d[pos] = o;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = s_running;
            for (int wv = 0; wv < nw; ++wv) t += s_warp_total[wv];
            s_running = t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) count[b] = s_running;
    // hand the NMS candidate counters of this image back zeroed for the next batch (they are only ever
    // incremented by the box decode, which runs before this kernel on the same stream)
    if (nz_count)
        for (int j = threadIdx.x; j < classes; j += blockDim.x) nz_count[(size_t)b * classes + j] = 0;
}

// ---------------------------------------------------------------------------------
// Softmax-tree detection without the dense pass (yolo9000: 9418 classes x 867 boxes x batch).
//
// What the reference computes per box (region_layer.c:349-366 on top of softmax_tree, softmax_layer.c:35-47, and
// hierarchy_predictions, tree.c:37-51): the softmax of EVERY group, the product along every root path, then it
// keeps the highest-index class whose product exceeds .5 and zeroes the rest.  Which class that is, and its value,
// depend on a handful of groups only:
//   * p = e / sum <= 1 in float arithmetic and a product RN(p * h) never exceeds h, so a class above .5 has all
//     its ancestors above .5 and its own softmax value above .5;
//   * inside one group at most one member is above .5 (the float sum of the group is >= twice the smaller of any
//     two members - rounding is monotone and 2e is representable);
//   * children follow their parents in the file (checked at plan time), so the highest index is the deepest one.
// So the kernel walks down from the root group(s): softmax of the group exactly as the dense kernel does it (double
// exp rounded to float, float sum in index order), take the member above .5, multiply, descend into its child
// group(s).  ~30 of the 9418 logits of a box are read; the values are bit-identical to the dense path (tests:
// golden tree fixtures + yolo9000 against the reference end to end).  A warp per box.
// ---------------------------------------------------------------------------------
struct TreeRec {      // one per box
    float x, y, w, h; // get_region_box
    float val;        // probs[box][cls] as get_region_boxes leaves it (0: no class above .5, or objectness <= thresh)
    int cls;          // -1 when val == 0
    int pad0, pad1;
};

// softmax value of member `lane + 32 i` of one group, all lanes of the warp cooperating (blas.c:205-221);
// returns through `visit` every member whose hierarchy value exceeds .5
template <typename F>
__device__ __forceinline__ void tree_group_softmax(const float *__restrict__ xi, int n, float hpar, bool is_root, int lane,
                                                   F visit)
{
    float largest = -FLT_MAX;
    for (int i = lane; i < n; i += 32) {
        const float v = xi[i];
        if (v > largest) largest = v;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const float other = __shfl_xor_sync(0xffffffffu, largest, d);
        if (other > largest) largest = other;
    }
    float sum = 0.f;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        float e = 0.f;
        if (i < n) {
            const float arg = xi[i] / 1.f - largest / 1.f;  // temperature 1, float expression
            e = (float)exp((double)arg);
        }
        const int cnt = (n - base) < 32 ? (n - base) : 32;
        for (int j = 0; j < cnt; ++j) sum = sum + __shfl_sync(0xffffffffu, e, j);
    }
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        float hv = 0.f;
        if (i < n) {
            const float arg = xi[i] / 1.f - largest / 1.f;
            const float pj = (float)exp((double)arg) / sum;
            hv = is_root ? pj : pj * hpar;  // tree.c:44-45: predictions[j] *= predictions[parent]
        }
        unsigned hot = __ballot_sync(0xffffffffu, hv > .5);
        while (hot) {
            const int src = __ffs(hot) - 1;
            hot &= hot - 1;
            visit(base + src, __shfl_sync(0xffffffffu, hv, src));
        }
    }
}

__global__ void region_tree_detect_kernel(const float *__restrict__ head, int head_cs, const float *__restrict__ biases,
                                          long long nboxes, int lw, int lh, int n, int classes, float thresh, int classfix,
                                          const int *__restrict__ group_size, const int *__restrict__ group_offset,
                                          const int *__restrict__ child_ptr, const int *__restrict__ child_grp,
                                          TreeRec *__restrict__ rec)
{
    const int lane = threadIdx.x & 31;
    const long long w0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    const int size = classes + 5;
    const int per_img = lw * lh * n;
    for (long long bi = w0; bi < nboxes; bi += nw) {
        const int index = (int)(bi % per_img);
        const long long pos = bi / n;  // b * hw + cell
        const int an = index % n;
        const float *x = head + pos * head_cs + (long long)an * size;
        // pending groups: (group, hierarchy value of its parent); the walk is warp-uniform
        int stk_g[24];
        float stk_h[24];
        int sp = 0;
        for (int q = child_ptr[classes]; q < child_ptr[classes + 1] && sp < 24; ++q) {
            stk_g[sp] = child_grp[q];
            stk_h[sp] = -1.f;  // marks a root group
            ++sp;
        }
        int best = -1;
        float best_val = 0.f;
        while (sp > 0) {
            --sp;
            const int g = stk_g[sp];
            const float hpar = stk_h[sp];
            const int off = group_offset[g];
            tree_group_softmax(x + 5 + off, group_size[g], hpar, hpar < 0.f, lane, [&](int member, float hv) {
                const int j = off + member;
                if (j > best) {
                    best = j;
                    best_val = hv;
                }
                for (int q = child_ptr[j]; q < child_ptr[j + 1] && sp < 24; ++q) {
                    stk_g[sp] = child_grp[q];
                    stk_h[sp] = hv;
                    ++sp;
                }
            });
        }
        if (lane == 0) {
            float scale = logistic_ref(x[4]);  // forward_region_layer (region_layer.c:160)
            if (classfix == -1 && scale < .5) scale = 0;
            const float val = (best >= 0 && scale > thresh) ? best_val : 0.f;
            const int cell = index / n;
            const int row = cell / lw;
            const int col = cell % lw;
            TreeRec r;
            r.x = (col + logistic_ref(x[0])) / lw;
            r.y = (row + logistic_ref(x[1])) / lh;
            r.w = (float)(exp((double)x[2]) * (double)biases[2 * an] / (double)lw);
            r.h = (float)(exp((double)x[3]) * (double)biases[2 * an + 1] / (double)lh);
            r.val = val;
            r.cls = val != 0.f ? best : -1;
            r.pad0 = r.pad1 = 0;
            rec[bi] = r;
        }
    }
}

// do_nms_sort + the final pick on the sparse records of one image (a box carries at most one non-zero class): class
// k's candidates in the order (value descending, index ascending) - the reference's carried sort order reduces to
// that when every other column of the two rows is zero (see nms.cu) -, greedy suppression inside the class, then the
// survivors above thresh in box-index order.
__device__ __forceinline__ float tree_overlap(float x1, float w1, float x2, float w2)
{
    const float l1 = x1 - w1 / 2;
    const float l2 = x2 - w2 / 2;
    const float left = l1 > l2 ? l1 : l2;
    const float r1 = x1 + w1 / 2;
    const float r2 = x2 + w2 / 2;
    const float right = r1 < r2 ? r1 : r2;
    return right - left;
}

__device__ __forceinline__ float tree_iou(const TreeRec &a, const TreeRec &b)
{
    const float w = tree_overlap(a.x, a.w, b.x, b.w);
    const float h = tree_overlap(a.y, a.h, b.y, b.h);
    float inter;
    if (w < 0 || h < 0) inter = 0;
    else inter = w * h;
    const float uni = a.w * a.h + b.w * b.h - inter;
    return inter / uni;
}

__global__ void tree_nms_collect_kernel(const TreeRec *__restrict__ rec, int total, float thresh, float nms,
                                        y2_det *__restrict__ det, int *__restrict__ count, int max_det)
{
    extern __shared__ int tsm[];
    int *s_idx = tsm;              // candidates in index order
    int *s_sorted = tsm + total;   // positions in s_idx, sorted
    int *s_alive = tsm + 2 * total;
    __shared__ int s_warp_tot[32];
    __shared__ int s_base;
    const int b = blockIdx.x;
    const TreeRec *r = rec + (size_t)b * total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int start = 0; start < total; start += blockDim.x) {
        const int i = start + threadIdx.x;
        const bool is = i < total && r[i].cls >= 0;
        const unsigned m = __ballot_sync(0xffffffffu, is);
        if (lane == 0) s_warp_tot[warp] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp_tot[w];
        if (is) s_idx[off + __popc(m & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < nw; ++w) t += s_warp_tot[w];
            s_base += t;
        }
        __syncthreads();
    }
    const int m = s_base;
    for (int a = threadIdx.x; a < m; a += blockDim.x) {
        const int ia = s_idx[a];
        const int ca = r[ia].cls;
        const float va = r[ia].val;
        int rank = 0;
        for (int o = 0; o < m; ++o) {
            const int io = s_idx[o];
            const int co = r[io].cls;
            const float vo = r[io].val;
            const bool before = co != ca ? co < ca : (vo != va ? vo > va : io < ia);
            if (o != a && before) ++rank;
        }
        s_sorted[rank] = ia;
        s_alive[rank] = 1;
    }
    __syncthreads();
    if (nms > 0) {
        for (int i = 0; i < m - 1; ++i) {
            if (!s_alive[i]) continue;  // uniform
            const TreeRec a = r[s_sorted[i]];
            for (int j = i + 1 + threadIdx.x; j < m; j += blockDim.x) {
                const TreeRec o = r[s_sorted[j]];
                if (o.cls != a.cls) break;  // sorted by class: the rest of this thread's stride is further away still
                if (s_alive[j] && tree_iou(a, o) > nms) s_alive[j] = 0;
            }
            __syncthreads();
        }
    }
    // survivors above thresh, in box-index order: mark per box, then the same ordered compaction
    int *s_keep = s_idx;  // reuse: 1 per box index
    __syncthreads();
    for (int i = threadIdx.x; i < total; i += blockDim.x) s_keep[i] = 0;
    __syncthreads();
    for (int a = threadIdx.x; a < m; a += blockDim.x)
        if (s_alive[a] && r[s_sorted[a]].val > thresh) s_keep[s_sorted[a]] = 1;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    y2_det *d = det + (size_t)b * max_det;
    for (int start = 0; start < total; start += blockDim.x) {
        const int i = start + threadIdx.x;
        const bool is = i < total && s_keep[i];
        const unsigned mk = __ballot_sync(0xffffffffu, is);
        if (lane == 0) s_warp_tot[warp] = __popc(mk);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp_tot[w];
        const int pos = off + __popc(mk & ((1u << lane) - 1));
        if (is && pos < max_det) {
            const TreeRec q = r[i];
            y2_det o;
            o.x = q.x; o.y = q.y; o.w = q.w; o.h = q.h;
            o.prob = q.val;
            o.obj_id = q.cls;
            o.box_index = i;
            d[pos] = o;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < nw; ++w) t += s_warp_tot[w];
            s_base += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) count[b] = s_base;
}

// 3-frame mean of video streams ----------------------------------------------------
// yolo_v2_class.cpp:206-213: every frame is decoded on mean_arrays (utils.c:420-433) over its stream's ring of the
// last three region outputs: avg = 0; avg += ring[0]; avg += ring[1]; avg += ring[2]; avg /= 3, in float, by ring
// slot.  The sources of the three slots come from y2_stream_plan (one y2_stream_src per image, on blockIdx.y).
// A block covers STREAM_CHUNK elements of one image row, 4 per thread (one float4 when every row is 16-byte aligned).
constexpr int STREAM_THREADS = 256;
constexpr int STREAM_CHUNK = STREAM_THREADS * 4;

// the row a source code names (y2_stream_src), NULL for a slot not written since open / reset
__device__ __forceinline__ const float *stream_row(int code, const float *out, const float *ring, int outputs)
{
    if (code >= 0) return out + (size_t)code * outputs;
    if (code == -1) return nullptr;
    return ring + (size_t)(-2 - code) * outputs;
}

__device__ __forceinline__ float stream_mean3(float a, float b, float c)
{
    return __fdiv_rn(__fadd_rn(__fadd_rn(__fadd_rn(0.f, a), b), c), 3.f);
}

template <bool VEC>
__global__ void __launch_bounds__(STREAM_THREADS) stream_mean_kernel(const float *__restrict__ out,
                                                                     const float *__restrict__ ring,
                                                                     const y2_stream_src *__restrict__ table,
                                                                     int outputs, float *__restrict__ mean)
{
    const y2_stream_src rec = table[blockIdx.y];
    const float *s0 = stream_row(rec.src[0], out, ring, outputs);
    const float *s1 = stream_row(rec.src[1], out, ring, outputs);
    const float *s2 = stream_row(rec.src[2], out, ring, outputs);
    float *dst = mean + (size_t)blockIdx.y * outputs;
    const int base = blockIdx.x * STREAM_CHUNK;
    if (VEC) {
        const int e = base + threadIdx.x * 4;
        if (e >= outputs) return;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 a = s0 ? __ldg((const float4 *)(s0 + e)) : z;
        const float4 b = s1 ? __ldg((const float4 *)(s1 + e)) : z;
        const float4 c = s2 ? __ldg((const float4 *)(s2 + e)) : z;
        *(float4 *)(dst + e) = make_float4(stream_mean3(a.x, b.x, c.x), stream_mean3(a.y, b.y, c.y),
                                           stream_mean3(a.z, b.z, c.z), stream_mean3(a.w, b.w, c.w));
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = base + q * STREAM_THREADS + threadIdx.x;
            if (e < outputs)
                dst[e] = stream_mean3(s0 ? __ldg(s0 + e) : 0.f, s1 ? __ldg(s1 + e) : 0.f, s2 ? __ldg(s2 + e) : 0.f);
        }
    }
}

// image i's region output row -> its ring row (rec.commit >= 0).  A separate launch from the mean: an earlier image
// of the same list may still read the old value of a ring row that a later one commits to.
template <bool VEC>
__global__ void __launch_bounds__(STREAM_THREADS) stream_commit_kernel(const float *__restrict__ out,
                                                                       float *__restrict__ ring,
                                                                       const y2_stream_src *__restrict__ table,
                                                                       int outputs)
{
    const int row = table[blockIdx.y].commit;
    if (row < 0) return;
    const float *src = out + (size_t)blockIdx.y * outputs;
    float *dst = ring + (size_t)row * outputs;
    const int base = blockIdx.x * STREAM_CHUNK;
    if (VEC) {
        const int e = base + threadIdx.x * 4;
        if (e < outputs) *(float4 *)(dst + e) = __ldg((const float4 *)(src + e));
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = base + q * STREAM_THREADS + threadIdx.x;
            if (e < outputs) dst[e] = __ldg(src + e);
        }
    }
}

// tracking of video streams ----------------------------------------------------------
// yolo_v2_class.cpp:228-236 (to_bbox) and 251-304 (Detector::tracking) for the images of each stream in order.  One
// block per stream.  The current frame's boxes live in shared memory next to best[]; every old box of the history
// (newest frame first, boxes in list order) is one block-wide step, because a match halves the matched box's extent
// and so moves the centre that later old boxes see.  Thread t alone reads and writes the current boxes m = t (mod
// TRACK_THREADS), so a step needs one barrier: the reduction of the match and of id_taken, after which the owner of
// the match applies it.  The match goes through one of three shared slots in turn, so that the slot a step reduces
// into was reset by thread 0 behind an earlier barrier while no thread could still read it.
constexpr int TRACK_THREADS = 128;

// float / double -> unsigned as x86-64 compilers convert (through a 64-bit integer): what the host Detector computes
__device__ __forceinline__ unsigned int track_u32(double v) { return (unsigned int)(long long)v; }

__device__ __forceinline__ y2_bbox track_to_bbox(const y2_det &d, int img_w, int img_h)
{
    const double cx = __dmul_rn(__dsub_rn((double)d.x, __ddiv_rn((double)d.w, 2.)), (double)img_w);
    const double cy = __dmul_rn(__dsub_rn((double)d.y, __ddiv_rn((double)d.h, 2.)), (double)img_h);
    y2_bbox b;
    b.x = track_u32(0. < cx ? cx : 0.); // std::max((double)0, v)
    b.y = track_u32(0. < cy ? cy : 0.);
    b.w = track_u32((double)__fmul_rn(d.w, (float)img_w));
    b.h = track_u32((double)__fmul_rn(d.h, (float)img_h));
    b.prob = d.prob;
    b.obj_id = (unsigned int)d.obj_id;
    b.track_id = 0;
    return b;
}

__global__ void __launch_bounds__(TRACK_THREADS) stream_track_kernel(const y2_det *__restrict__ det, int det_stride,
                                                                     const int *__restrict__ count,
                                                                     const y2_track_img *__restrict__ recs,
                                                                     const int *__restrict__ offsets, int total,
                                                                     int classes, int story, y2_bbox *hist,
                                                                     int *hist_count, unsigned int *next_id,
                                                                     y2_bbox *__restrict__ out, int out_stride)
{
    extern __shared__ __align__(16) unsigned char track_smem[];
    y2_bbox *cur = (y2_bbox *)track_smem;
    unsigned int *best = (unsigned int *)(cur + total);
    __shared__ int s_match[3];
    const int tid = threadIdx.x;
    const int first = offsets[blockIdx.x], last = offsets[blockIdx.x + 1];
    const int s = recs[first].stream;
    unsigned int *ids = next_id + (size_t)s * classes;
    if (tid < 3) s_match[tid] = -1;
    int q = 0; // block-wide steps so far
    for (int r = first; r < last; ++r) {
        const y2_track_img rec = recs[r];
        if (rec.restart)
            for (int c = tid; c < classes; c += TRACK_THREADS) ids[c] = 1u;
        const int n = min(max(count[rec.image], 0), min(total, det_stride));
        const y2_det *d = det + (size_t)rec.image * det_stride;
        for (int m = tid; m < n; m += TRACK_THREADS) {
            cur[m] = track_to_bbox(d[m], rec.w, rec.h);
            best[m] = 0xffffffffu;
        }
        __syncthreads();
        for (int k = 1; k <= rec.len; ++k) {
            const int slot = (rec.head - k + story) % story;
            const y2_bbox *frame = hist + ((size_t)s * story + slot) * total;
            const int on = hist_count[s * story + slot];
            y2_bbox next = frame[0]; // the next step's old box, loaded a step ahead (unused when the frame is empty)
            for (int j = 0; j < on; ++j, ++q) {
                const y2_bbox old = next;
                if (j + 1 < on) next = frame[j + 1];
                const float ox = (float)(old.x + old.w / 2), oy = (float)(old.y + old.h / 2);
                int match = -1;
                int taken = 0;
                for (int m = tid; m < n; m += TRACK_THREADS) {
                    const y2_bbox k = cur[m];
                    if (k.obj_id != old.obj_id) continue;
                    taken |= k.track_id == old.track_id;
                    const float dx = __fsub_rn(ox, (float)(k.x + k.w / 2));
                    const float dy = __fsub_rn(oy, (float)(k.y + k.h / 2));
                    const unsigned int dist = track_u32((double)__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))));
                    if (dist < 100 && (k.track_id == 0 || best[m] > dist)) {
                        best[m] = dist;
                        match = m; // the last m that qualifies wins, not the nearest
                    }
                }
                match = __reduce_max_sync(0xffffffffu, match);
                if ((tid & 31) == 0 && match >= 0) atomicMax(&s_match[q % 3], match);
                taken = __syncthreads_or(taken);
                const int m = s_match[q % 3];
                if (tid == 0) s_match[(q + 2) % 3] = -1; // read by every thread before this step's barrier
                if (m >= 0 && !taken && m % TRACK_THREADS == tid) {
                    cur[m].track_id = old.track_id;
                    cur[m].w = (cur[m].w + old.w) / 2;
                    cur[m].h = (cur[m].h + old.h) / 2;
                }
            }
        }
        __syncthreads();
        if (tid == 0)
            for (int m = 0; m < n; ++m)
                if (cur[m].track_id == 0) cur[m].track_id = ids[cur[m].obj_id]++;
        __syncthreads();
        y2_bbox *push = hist + ((size_t)s * story + rec.head) * total;
        y2_bbox *dst = out + (size_t)rec.image * out_stride;
        for (int m = tid; m < n; m += TRACK_THREADS) {
            push[m] = cur[m];
            if (m < out_stride) dst[m] = cur[m];
        }
        if (tid == 0) hist_count[s * story + rec.head] = n;
        __syncthreads();
    }
}

// classifier tail ------------------------------------------------------------------
// avgpool_layer.c:40-55: sequential float sum over h*w, then / (h*w).  One thread per
// (b, c) keeps the reference's summation order; reads are coalesced along c.
__global__ void avgpool_flat_kernel(const float *__restrict__ in, float *__restrict__ out, int batch, int hw,
                                    int c, int cs)
{
    const long long total = (long long)batch * c;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int ch = (int)(t % c);
        const int b = (int)(t / c);
        const float *p = in + (size_t)b * hw * cs + ch;
        float s = 0.f;
        int i = 0;
        // sixteen loads in flight per thread, summed in the reference's order (the additions are one dependent chain
        // either way; issued one at a time each of them waited for its own load)
        for (; i + 16 <= hw; i += 16) {
            float v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) v[q] = __ldg(p + (size_t)(i + q) * cs);
#pragma unroll
            for (int q = 0; q < 16; ++q) s += v[q];
        }
        for (; i < hw; ++i) s += __ldg(p + (size_t)i * cs);
        out[t] = s / hw;
    }
}

// softmax_layer.c:49-61 -> softmax(blas.c:205-221) per row, warp per row
__global__ void softmax_rows_kernel(const float *__restrict__ in, float *__restrict__ out, int rows, int n,
                                    float temp)
{
    const int lane = threadIdx.x & 31;
    const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp_global; r < rows; r += nwarps) {
        const float *xi = in + r * n;
        float *oi = out + r * n;
        float largest = -FLT_MAX;
        for (int i = lane; i < n; i += 32) {
            const float v = xi[i];
            if (v > largest) largest = v;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float other = __shfl_xor_sync(0xffffffffu, largest, d);
            if (other > largest) largest = other;
        }
        float sum = 0.f;
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            float e = 0.f;
            if (i < n) {
                const float arg = xi[i] / temp - largest / temp;
                e = (float)exp((double)arg);
                oi[i] = e;
            }
            const int cnt = (n - base) < 32 ? (n - base) : 32;
            for (int j = 0; j < cnt; ++j) sum = sum + __shfl_sync(0xffffffffu, e, j);
        }
        for (int i = lane; i < n; i += 32) oi[i] = oi[i] / sum;
    }
}

// The same with a BLOCK per row, for wide rows (the 1000-way classifiers): the exps - double precision, the bulk of
// the work - are spread over 256 threads and parked in shared memory, ONE thread then adds them in index order (the
// reference's serial float sum: a dependent chain of n additions either way, but 4 clk each from shared memory
// instead of a shuffle per term), everybody divides.  n <= 4096.
__global__ void softmax_rows_block_kernel(const float *__restrict__ in, float *__restrict__ out, int rows, int n,
                                          float temp)
{
    __shared__ float s_e[4096];
    __shared__ float s_red[8];
    __shared__ float s_sum;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int r = blockIdx.x; r < rows; r += gridDim.x) {
        const float *xi = in + (size_t)r * n;
        float *oi = out + (size_t)r * n;
        float largest = -FLT_MAX;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const float v = xi[i];
            if (v > largest) largest = v;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float other = __shfl_xor_sync(0xffffffffu, largest, d);
            if (other > largest) largest = other;
        }
        if (lane == 0) s_red[warp] = largest;
        __syncthreads();
        largest = s_red[0];
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
            if (s_red[w] > largest) largest = s_red[w];
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const float arg = xi[i] / temp - largest / temp;
            s_e[i] = (float)exp((double)arg);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            float sum = 0.f;
            int i = 0;
            for (; i + 8 <= n; i += 8) {
                float v[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) v[q] = s_e[i + q];
#pragma unroll
                for (int q = 0; q < 8; ++q) sum = sum + v[q];
            }
            for (; i < n; ++i) sum = sum + s_e[i];
            s_sum = sum;
        }
        __syncthreads();
        const float sum = s_sum;
        for (int i = threadIdx.x; i < n; i += blockDim.x) oi[i] = s_e[i] / sum;
        __syncthreads();  // s_e / s_red are reused by the next row
    }
}

// softmax_tree (softmax_layer.c:35-47) over plain rows: warp per (row, group), blas.c:205-221 per group
__global__ void softmax_tree_rows_kernel(const float *__restrict__ in, float *__restrict__ out, int rows, int n, float temp,
                                         int n_groups, const int *__restrict__ group_size,
                                         const int *__restrict__ group_offset)
{
    const int lane = threadIdx.x & 31;
    const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long work = (long long)rows * n_groups;
    for (long long wi = warp_global; wi < work; wi += nwarps) {
        const long long r = wi / n_groups;
        const int g = (int)(wi - r * n_groups);
        const int off = group_offset[g], m = group_size[g];
        const float *xi = in + r * n + off;
        float *oi = out + r * n + off;
        float largest = -FLT_MAX;
        for (int i = lane; i < m; i += 32) {
            const float v = xi[i];
            if (v > largest) largest = v;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float other = __shfl_xor_sync(0xffffffffu, largest, d);
            if (other > largest) largest = other;
        }
        float sum = 0.f;
        for (int base = 0; base < m; base += 32) {
            const int i = base + lane;
            float e = 0.f;
            if (i < m) {
                const float arg = xi[i] / temp - largest / temp;
                e = (float)exp((double)arg);
                oi[i] = e;
            }
            const int cnt = (m - base) < 32 ? (m - base) : 32;
            for (int j = 0; j < cnt; ++j) sum = sum + __shfl_sync(0xffffffffu, e, j);
        }
        for (int i = lane; i < m; i += 32) oi[i] = oi[i] / sum;
    }
}

// ---------------------------------------------------------------------------------
// classifier tail (classifier.c:676-730 after network_predict): hierarchy_predictions (tree.c:37-51) when a
// tree is given, then top_k (utils.c:179-193).  One block per image.
// top_k keeps a list sorted by value; an entry displaces the first list entry it is strictly greater than, and the
// displaced one moves on down the list the same way.  Among equal values the order therefore depends on the order
// of arrival (a displaced entry goes behind its equals), so the result is reproduced by running that same loop -
// but only over the few entries that can matter: the values above the top-th largest value T, and the first `top`
// entries equal to T.  An entry equal to T that comes later finds the list full of values >= T and changes
// nothing; an entry below T never changes where the entries >= T end up.
// Every entry gets the distinct 47-bit key (order(value) << 15) | (32767 - index); the m = 2*top-1 largest keys
// hold all entries above T and at least `top` entries equal to T, lowest indices first (or, when there are fewer,
// some below T, which is harmless).  A radix select over 8-bit digits finds the m-th largest key; those m entries,
// in index order, go through top_k's loop on one thread, comparing order(value): +0 and -0 are equal and a NaN
// is below every number.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ unsigned topk_order(float v)
{
    if (v != v) return 0u;                                   // NaN: below every number
    const unsigned u = __float_as_uint(v == 0.f ? 0.f : v);  // -0 ties with +0
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ unsigned long long topk_key(float v, int j)
{
    return ((unsigned long long)topk_order(v) << 15) | (unsigned)(32767 - j);
}

__global__ void __launch_bounds__(1024) classify_topk_kernel(const float *__restrict__ out, int row_stride, int batch,
                                                             int n, int top, const int *__restrict__ parent,
                                                             y2_class_hit *__restrict__ hits)
{
    extern __shared__ float val[]; // [n]: the row, after hierarchy_predictions
    __shared__ unsigned hist[256];
    __shared__ unsigned long long cand[2 * Y2_CLASSIFY_MAX_TOP - 1];
    __shared__ unsigned ck[2 * Y2_CLASSIFY_MAX_TOP - 1];  // candidates in index order: order(value), index
    __shared__ int ci[2 * Y2_CLASSIFY_MAX_TOP - 1];
    __shared__ int lst[Y2_CLASSIFY_MAX_TOP];
    __shared__ unsigned s_digit, s_remaining;
    __shared__ int s_count;
    const int lane = threadIdx.x & 31;
    const int m = (2 * top - 1 < n) ? 2 * top - 1 : n;
    for (int b = blockIdx.x; b < batch; b += gridDim.x) {
        const float *row = out + (size_t)b * row_stride;
        if (parent) {
            hierarchy_walk(row, val, parent, n);
        } else {
            for (int j = threadIdx.x; j < n; j += blockDim.x) val[j] = row[j];
            __syncthreads();
        }
        unsigned long long prefix = 0, mask = 0;
        unsigned remaining = (unsigned)m;
        for (int shift = 40; shift >= 0; shift -= 8) {
            for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
            __syncthreads();
            for (int base = 0; base < n; base += blockDim.x) {
                const int j = base + threadIdx.x;
                unsigned bin = 256; // not counted
                if (j < n) {
                    const unsigned long long k = topk_key(val[j], j);
                    if ((k & mask) == prefix) bin = (unsigned)(k >> shift) & 255u;
                }
                const unsigned peers = __match_any_sync(0xffffffffu, bin);
                if (bin < 256 && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
            }
            __syncthreads();
            if (threadIdx.x < 32) {
                // lane l owns digits 255-8l down to 248-8l; the lane in which the count from the top reaches
                // `remaining` picks the digit
                unsigned own = 0;
                for (int q = 0; q < 8; ++q) own += hist[255 - 8 * lane - q];
                unsigned incl = own;
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                unsigned cum = incl - own;
                if (cum < remaining && incl >= remaining) {
                    int d = 255 - 8 * lane;
                    while (cum + hist[d] < remaining) cum += hist[d--];
                    s_digit = (unsigned)d;
                    s_remaining = remaining - cum;
                }
            }
            __syncthreads();
            prefix |= (unsigned long long)s_digit << shift;
            mask |= 255ull << shift;
            remaining = s_remaining;
        }
        // prefix is now the m-th largest key: exactly m keys are >= prefix
        if (threadIdx.x == 0) s_count = 0;
        __syncthreads();
        for (int j = threadIdx.x; j < n; j += blockDim.x) {
            const unsigned long long k = topk_key(val[j], j);
            if (k >= prefix) cand[atomicAdd(&s_count, 1)] = k;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < m; i += blockDim.x) { // sort the candidates by index
            const int j = 32767 - (int)(cand[i] & 32767u);
            int rank = 0;
            for (int q = 0; q < m; ++q) rank += (32767 - (int)(cand[q] & 32767u)) < j;
            ck[rank] = (unsigned)(cand[i] >> 15);
            ci[rank] = j;
        }
        __syncthreads();
        if (threadIdx.x == 0) { // utils.c:179-193 over the candidates
            for (int j = 0; j < top; ++j) lst[j] = -1;
            for (int c = 0; c < m; ++c) {
                int cur = c;
                for (int j = 0; j < top && cur >= 0; ++j) {
                    if (lst[j] < 0 || ck[cur] > ck[lst[j]]) {
                        const int displaced = lst[j];
                        lst[j] = cur;
                        cur = displaced;
                    }
                }
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < top; i += blockDim.x) {
            const int j = ci[lst[i]];
            hits[(size_t)b * top + i] = y2_class_hit{j, val[j]};
        }
        __syncthreads();
    }
}

static inline int grid_cap(long long blocks, int per_sm)
{
    long long cap = (long long)sm_count() * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

} // namespace y2

using namespace y2;

extern "C" int y2_region_forward_strided(const float *in, int in_cs, float *out, int batch, int hw, int n, int classes,
                                         int softmax, int n_groups, const int *d_group_size,
                                         const int *d_group_offset, y2_stream_t s)
{
    if (!in || !out || batch <= 0 || hw <= 0 || n <= 0 || classes <= 0 || in_cs < n * (classes + 5)) return Y2_EINVAL;
    if (n_groups > 0 && (!d_group_size || !d_group_offset)) return Y2_EINVAL;
    const long long boxes = (long long)batch * hw * n;
    const int threads = 256;
    if (n_groups <= 0) {  // flat softmax (or none): four lanes per box
        const int grid = grid_cap((boxes * 4 + threads - 1) / threads, 8);
        region_forward_flat_kernel<<<grid, threads, 0, to_stream(s)>>>(in, in_cs, n, out, boxes, classes, softmax);
        Y2_LAUNCH_CHECK();
        return Y2_OK;
    }
    const long long work = boxes * n_groups;
    const int grid = grid_cap((work + threads - 1) / threads, 8);
    region_forward_tree_kernel<<<grid, threads, 0, to_stream(s)>>>(in, in_cs, n, out, boxes, classes, softmax, n_groups,
                                                                   d_group_size, d_group_offset);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_region_forward(const float *in, float *out, int batch, int hw, int n, int classes,
                                 int softmax, int n_groups, const int *d_group_size,
                                 const int *d_group_offset, y2_stream_t s)
{
    return y2_region_forward_strided(in, n * (classes + 5), out, batch, hw, n, classes, softmax, n_groups, d_group_size,
                                     d_group_offset, s);
}

extern "C" int y2_region_boxes_counted(float *pred, const float *d_biases, float *boxes, float *probs, int batch,
                                       int lw, int lh, int n, int classes, float img_w, float img_h, float thresh,
                                       int only_objectness, int classfix, int tree_n, const int *d_tree_parent,
                                       const int *d_map, int map_n, int *nz_count, y2_stream_t s)
{
    if (!pred || !d_biases || !boxes || !probs || batch <= 0) return Y2_EINVAL;
    const long long nboxes = (long long)batch * lw * lh * n;
    if (tree_n > 0) {
        if (!d_tree_parent || tree_n != classes) {
            set_error("y2_region_boxes: tree size %d != classes %d", tree_n, classes);
            return Y2_EINVAL;
        }
        const size_t smem = (size_t)classes * 2 * sizeof(float);
        // the attribute is per device: a second network on another GPU needs it raised there too.  Raised whatever
        // the size: the kernel's static shared memory counts against the 48 KB default as well
        static bool attr_done[64] = {false};
        int dev = 0;
        Y2_CUDA_CHECK(cudaGetDevice(&dev));
        if (dev < 0 || dev >= 64 || !attr_done[dev]) {
            Y2_CUDA_CHECK(cudaFuncSetAttribute(region_boxes_tree_kernel,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            if (dev >= 0 && dev < 64) attr_done[dev] = true;
        }
        if (smem > 200 * 1024) {
            set_error("y2_region_boxes: %d classes exceed the shared-memory staging", classes);
            return Y2_EINVAL;
        }
        // one block per box; wide trees get wide blocks (fewer chunk rounds of the hierarchy walk)
        const int tree_threads = classes > 2048 ? 1024 : 256;
        region_boxes_tree_kernel<<<grid_cap(nboxes, 4), tree_threads, smem, to_stream(s)>>>(
            pred, d_biases, boxes, probs, batch, lw, lh, n, classes, img_w, img_h, thresh, only_objectness,
            classfix, d_tree_parent, d_map, map_n, nz_count);
    } else {
        const long long total = nboxes * classes;
        region_boxes_flat_kernel<<<grid_cap((total + 255) / 256, 16), 256, 0, to_stream(s)>>>(
            pred, d_biases, boxes, probs, batch, lw, lh, n, classes, img_w, img_h, thresh, only_objectness,
            classfix, nz_count);
    }
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_classify_topk(const float *out, int row_stride, int batch, int n, int top,
                                const int *d_tree_parent, y2_class_hit *hits, y2_stream_t s)
{
    if (!out || !hits || batch <= 0 || n <= 0 || n > Y2_CLASSIFY_MAX_N || row_stride < n || top < 1 || top > n ||
        top > Y2_CLASSIFY_MAX_TOP) {
        set_error("y2_classify_topk: invalid arguments (n=%d row_stride=%d top=%d)", n, row_stride, top);
        return Y2_EINVAL;
    }
    const size_t smem = (size_t)n * sizeof(float);
    // raised on every device before its first launch, whatever n: the kernel's static shared memory (histogram and
    // candidates, ~5.5 KB) counts against the 48 KB default too, so comparing n * 4 alone with 48 KB is not enough
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(classify_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           Y2_CLASSIFY_MAX_N * sizeof(float)));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    classify_topk_kernel<<<grid_cap(batch, 2), 1024, smem, to_stream(s)>>>(out, row_stride, batch, n, top,
                                                                          d_tree_parent, hits);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_region_boxes(float *pred, const float *d_biases, float *boxes, float *probs, int batch,
                               int lw, int lh, int n, int classes, float img_w, float img_h, float thresh,
                               int only_objectness, int classfix, int tree_n, const int *d_tree_parent,
                               const int *d_map, int map_n, y2_stream_t s)
{
    return y2_region_boxes_counted(pred, d_biases, boxes, probs, batch, lw, lh, n, classes, img_w, img_h, thresh,
                                   only_objectness, classfix, tree_n, d_tree_parent, d_map, map_n, nullptr, s);
}

extern "C" int y2_stream_plan(int n, const int *stream_ids, int max_streams, int *frame_index, int *frames_seen,
                              y2_stream_src *plan)
{
    if (n < 1 || !stream_ids || max_streams < 1 || !frame_index || !frames_seen || !plan) return Y2_EINVAL;
    for (int i = 0; i < n; ++i)
        if (stream_ids[i] < 0 || stream_ids[i] >= max_streams) return Y2_EINVAL;
    // slot[i]: the ring slot image i writes, its stream's frame_index advanced by the stream's earlier images here
    int *slot = (int *)malloc((size_t)n * sizeof(int));
    if (!slot) return Y2_ENOMEM;
    for (int i = 0; i < n; ++i) {
        const int s = stream_ids[i];
        int before = 0;
        for (int k = 0; k < i; ++k) before += stream_ids[k] == s;
        slot[i] = (frame_index[s] + before) % 3;
    }
    for (int i = 0; i < n; ++i) {
        const int s = stream_ids[i];
        for (int j = 0; j < 3; ++j) {
            // the latest writer of slot j up to and including image i: this batch, else the ring as it stood
            int code = frames_seen[s] > j ? -2 - (s * 3 + j) : -1;
            for (int k = i; k >= 0; --k)
                if (stream_ids[k] == s && slot[k] == j) {
                    code = k;
                    break;
                }
            plan[i].src[j] = code;
        }
        plan[i].commit = s * 3 + slot[i];
        for (int k = i + 1; k < n; ++k)
            if (stream_ids[k] == s && slot[k] == slot[i]) plan[i].commit = -1;
    }
    for (int i = 0; i < n; ++i) {
        const int s = stream_ids[i];
        frame_index[s] = (frame_index[s] + 1) % 3;
        if (frames_seen[s] < 3) frames_seen[s]++;
    }
    free(slot);
    return Y2_OK;
}

extern "C" int y2_track_plan(int n, const int *stream_ids, const int *frame_w, const int *frame_h, int max_streams,
                             int story, int *head, int *len, int *restart, y2_track_img *recs, int *offsets)
{
    if (n < 1 || !stream_ids || !frame_w || !frame_h || max_streams < 1 || story < 1 || story > Y2_TRACK_MAX_STORY ||
        !head || !len || !restart || !recs || !offsets)
        return Y2_EINVAL;
    for (int i = 0; i < n; ++i)
        if (stream_ids[i] < 0 || stream_ids[i] >= max_streams || frame_w[i] <= 0 || frame_h[i] <= 0) return Y2_EINVAL;
    int n_streams = 0, k = 0;
    for (int i = 0; i < n; ++i) {
        const int s = stream_ids[i];
        bool seen = false;
        for (int q = 0; q < i && !seen; ++q) seen = stream_ids[q] == s;
        if (seen) continue;
        offsets[n_streams++] = k;
        for (int j = i; j < n; ++j) {
            if (stream_ids[j] != s) continue;
            recs[k++] = y2_track_img{j, s, frame_w[j], frame_h[j], head[s], len[s], restart[s]};
            restart[s] = 0;
            head[s] = (head[s] + 1) % story;
            if (len[s] < story) len[s]++;
        }
    }
    offsets[n_streams] = n;
    return n_streams;
}

extern "C" int y2_stream_track(const y2_det *det, int det_stride, const int *count, const y2_track_img *recs,
                               const int *offsets, int n_streams, int total, int classes, int story, y2_bbox *hist,
                               int *hist_count, unsigned int *next_id, y2_bbox *out, int out_stride, y2_stream_t s)
{
    if (!det || !count || !recs || !offsets || !hist || !hist_count || !next_id || !out || n_streams < 1 || total < 1 ||
        total > Y2_TRACK_MAX_TOTAL || det_stride < 1 || out_stride < 1 || classes < 1 || story < 1 ||
        story > Y2_TRACK_MAX_STORY) {
        set_error("y2_stream_track: invalid arguments (n_streams=%d total=%d det_stride=%d out_stride=%d classes=%d "
                  "story=%d)", n_streams, total, det_stride, out_stride, classes, story);
        return Y2_EINVAL;
    }
    const size_t smem = (size_t)total * (sizeof(y2_bbox) + sizeof(unsigned int));
    static bool attr_done[64] = {};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) { /* once per device, for the largest list the ABI takes */
        Y2_CUDA_CHECK(cudaFuncSetAttribute(stream_track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)((size_t)Y2_TRACK_MAX_TOTAL * (sizeof(y2_bbox) + sizeof(unsigned int)))));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    stream_track_kernel<<<n_streams, TRACK_THREADS, smem, to_stream(s)>>>(det, det_stride, count, recs, offsets, total,
                                                                         classes, story, hist, hist_count, next_id,
                                                                         out, out_stride);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

static bool stream_vec_ok(int outputs, const void *a, const void *b, const void *c)
{
    return outputs % 4 == 0 && (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c) & 15) == 0;
}

extern "C" int y2_stream_mean(const float *out, const float *ring, const y2_stream_src *table, int n, int outputs,
                              float *mean, y2_stream_t s)
{
    if (!out || !ring || !table || !mean || n < 1 || n > 65535 || outputs < 1) {
        set_error("y2_stream_mean: invalid arguments (n=%d outputs=%d)", n, outputs);
        return Y2_EINVAL;
    }
    const dim3 grid((outputs + STREAM_CHUNK - 1) / STREAM_CHUNK, n);
    if (stream_vec_ok(outputs, out, ring, mean))
        stream_mean_kernel<true><<<grid, STREAM_THREADS, 0, to_stream(s)>>>(out, ring, table, outputs, mean);
    else
        stream_mean_kernel<false><<<grid, STREAM_THREADS, 0, to_stream(s)>>>(out, ring, table, outputs, mean);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_stream_commit(const float *out, float *ring, const y2_stream_src *table, int n, int outputs,
                                y2_stream_t s)
{
    if (!out || !ring || !table || n < 1 || n > 65535 || outputs < 1) {
        set_error("y2_stream_commit: invalid arguments (n=%d outputs=%d)", n, outputs);
        return Y2_EINVAL;
    }
    const dim3 grid((outputs + STREAM_CHUNK - 1) / STREAM_CHUNK, n);
    if (stream_vec_ok(outputs, out, ring, ring))
        stream_commit_kernel<true><<<grid, STREAM_THREADS, 0, to_stream(s)>>>(out, ring, table, outputs);
    else
        stream_commit_kernel<false><<<grid, STREAM_THREADS, 0, to_stream(s)>>>(out, ring, table, outputs);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// ws: caller-owned scratch of y2_collect_ws_bytes(batch, total, classes) bytes (per-box maxima of wide class
// rows), nz_count: the NMS candidate counters to hand back zeroed (or NULL).
extern "C" size_t y2_collect_ws_bytes(int batch, int total, int classes)
{
    return classes >= 256 ? (size_t)batch * total * 8 : 0;
}

extern "C" int y2_collect_ws(const float *boxes, const float *probs, int batch, int total, int classes,
                             float thresh, y2_det *det, int *count, int max_det, void *ws, int *nz_count,
                             y2_stream_t s)
{
    if (!boxes || !probs || !det || !count || batch <= 0 || total <= 0) return Y2_EINVAL;
    const size_t smem = (size_t)total * 8;
    if (smem > 48 * 1024) {
        set_error("y2_collect: %d boxes per image exceed the staging buffer", total);
        return Y2_EINVAL;
    }
    const float *pre_best = nullptr;
    const int *pre_arg = nullptr;
    if (classes >= 256) {
        if (!ws) return Y2_EINVAL;
        const size_t nb = (size_t)batch * total;
        float *best = (float *)ws;
        int *arg = (int *)(best + nb);
        box_argmax_kernel<<<grid_cap((long long)(nb * 32 + 255) / 256, 8), 256, 0, to_stream(s)>>>(
            probs, (long long)nb, classes, best, arg);
        Y2_LAUNCH_CHECK();
        pre_best = best;
        pre_arg = arg;
    }
    collect_kernel<<<batch, 256, smem, to_stream(s)>>>(boxes, probs, total, classes, thresh, det, count,
                                                       max_det, pre_best, pre_arg, nz_count);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// stand-alone form: the scratch lives for the duration of the call
extern "C" int y2_collect(const float *boxes, const float *probs, int batch, int total, int classes,
                          float thresh, y2_det *det, int *count, int max_det, y2_stream_t s)
{
    void *ws = nullptr;
    const size_t bytes = y2_collect_ws_bytes(batch, total, classes);
    if (bytes) Y2_CUDA_CHECK(cudaMalloc(&ws, bytes));
    const int rc = y2_collect_ws(boxes, probs, batch, total, classes, thresh, det, count, max_det, ws, nullptr, s);
    if (ws) {
        cudaStreamSynchronize(to_stream(s));
        cudaFree(ws);
    }
    return rc;
}

extern "C" size_t y2_tree_rec_bytes(void) { return sizeof(TreeRec); }

extern "C" int y2_region_tree_detect(const float *head, int head_cs, const float *d_biases, int batch, int lw, int lh,
                                     int n, int classes, float thresh, int classfix, const int *d_group_size,
                                     const int *d_group_offset, const int *d_child_ptr, const int *d_child_grp,
                                     void *rec, y2_stream_t s)
{
    if (!head || !d_biases || !d_group_size || !d_group_offset || !d_child_ptr || !d_child_grp || !rec || batch <= 0 ||
        head_cs < n * (classes + 5))
        return Y2_EINVAL;
    const long long nboxes = (long long)batch * lw * lh * n;
    region_tree_detect_kernel<<<grid_cap((nboxes * 32 + 255) / 256, 8), 256, 0, to_stream(s)>>>(
        head, head_cs, d_biases, nboxes, lw, lh, n, classes, thresh, classfix, d_group_size, d_group_offset, d_child_ptr,
        d_child_grp, (TreeRec *)rec);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_tree_nms_collect(const void *rec, int batch, int total, float thresh, float nms, y2_det *det,
                                   int *count, int max_det, y2_stream_t s)
{
    if (!rec || !det || !count || batch <= 0 || total <= 0) return Y2_EINVAL;
    const size_t smem = (size_t)total * 3 * sizeof(int);
    if (smem > 48 * 1024) {
        set_error("y2_tree_nms_collect: %d boxes per image exceed the staging buffer", total);
        return Y2_EINVAL;
    }
    tree_nms_collect_kernel<<<batch, 256, smem, to_stream(s)>>>((const TreeRec *)rec, total, thresh, nms, det, count,
                                                                max_det);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_avgpool_flat(const float *in, float *out, int batch, int hw, int c, int cs, y2_stream_t s)
{
    if (!in || !out) return Y2_EINVAL;
    const long long total = (long long)batch * c;
    avgpool_flat_kernel<<<grid_cap((total + 127) / 128, 16), 128, 0, to_stream(s)>>>(in, out, batch, hw, c, cs);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_softmax_rows(const float *in, float *out, int rows, int n, float temp, y2_stream_t s)
{
    if (!in || !out) return Y2_EINVAL;
    if (n >= 256 && n <= 4096 && rows <= 8 * sm_count() && !getenv("Y2_SOFTMAX_WARP_ROWS")) {
        // few wide rows: a warp per row leaves the device empty (64 rows = 64 warps)
        softmax_rows_block_kernel<<<rows, 256, 0, to_stream(s)>>>(in, out, rows, n, temp);
        Y2_LAUNCH_CHECK();
        return Y2_OK;
    }
    softmax_rows_kernel<<<grid_cap(((long long)rows * 32 + 255) / 256, 8), 256, 0, to_stream(s)>>>(in, out, rows,
                                                                                                   n, temp);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_softmax_tree_rows(const float *in, float *out, int rows, int n, float temp, int n_groups,
                                    const int *d_group_size, const int *d_group_offset, y2_stream_t s)
{
    if (!in || !out || rows <= 0 || n <= 0 || n_groups <= 0 || !d_group_size || !d_group_offset) return Y2_EINVAL;
    const long long work = (long long)rows * n_groups;
    softmax_tree_rows_kernel<<<grid_cap((work * 32 + 255) / 256, 8), 256, 0, to_stream(s)>>>(
        in, out, rows, n, temp, n_groups, d_group_size, d_group_offset);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}
