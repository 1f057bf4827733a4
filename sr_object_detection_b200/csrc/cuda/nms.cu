// Per-class sorted non-maximum suppression on the GPU, bit-exact with do_nms_sort
// (reference box.c:249-277 with nms_comparator 239-247 and box_iou 67-97).
//
// What the reference does, per class k in ascending order: stable-sort (glibc qsort is a
// merge sort) ALL boxes by probs[.][k] descending, starting from the order the previous
// class left behind; then walk the sorted list, and every box whose prob is still non-zero
// zeroes the class-k prob of every later box with IoU > thresh.
//
// Two facts make this parallel over (image, class) without changing a single result:
//  * boxes with prob 0 never suppress and being suppressed changes nothing for them, so only
//    the non-zero "candidates" of a class matter;
//  * the carried-over order is a closed form: class k sees the boxes ordered by
//    (p[k-1] desc, p[k-2] desc, ..., p[0] desc, index asc) of the ORIGINAL probabilities
//    (each class is sorted before its own suppression runs), so ties in p[k] are broken by
//    walking back through the previous classes.
// Suppressed entries are first marked by flipping their sign (|p| keeps the original value
// for the tie-breaks of other classes running concurrently); a second pass writes the zeros.
//
// Compiled with -fmad=false: IoU must round exactly like the C code.
#include "y2_common.cuh"

namespace y2 {

__device__ __forceinline__ float overlap_ref(float x1, float w1, float x2, float w2)
{
    const float l1 = x1 - w1 / 2;
    const float l2 = x2 - w2 / 2;
    const float left = l1 > l2 ? l1 : l2;
    const float r1 = x1 + w1 / 2;
    const float r2 = x2 + w2 / 2;
    const float right = r1 < r2 ? r1 : r2;
    return right - left;
}

__device__ __forceinline__ float box_iou_ref(const float4 a, const float4 b)
{
    // float4 = (x, y, w, h)
    const float w = overlap_ref(a.x, a.z, b.x, b.z);
    const float h = overlap_ref(a.y, a.w, b.y, b.w);
    float inter;
    if (w < 0 || h < 0) inter = 0;
    else inter = w * h;
    const float uni = a.z * a.w + b.z * b.w - inter;
    return inter / uni;
}

// does candidate (ia, pa) sort before candidate (ib, pb) for class k?
__device__ __forceinline__ bool sorts_before(const float *__restrict__ probs_img, int classes, int k,
                                             int ia, float pa, int ib, float pb)
{
    if (pa != pb) return pa > pb;
    for (int c = k - 1; c >= 0; --c) {
        const float qa = fabsf(probs_img[(size_t)ia * classes + c]);
        const float qb = fabsf(probs_img[(size_t)ib * classes + c]);
        if (qa != qb) return qa > qb;
    }
    return ia < ib;
}

// count non-zero entries per (image, class); coalesced over the probs matrix
__global__ void nms_count_kernel(const float *__restrict__ probs, int *__restrict__ cnt, int batch, int total,
                                 int classes)
{
    const long long n = (long long)batch * total * classes;
    const long long per_img = (long long)total * classes;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n;
         t += (long long)gridDim.x * blockDim.x) {
        if (probs[t] != 0.f) {
            const int b = (int)(t / per_img);
            const int k = (int)(t % classes);
            atomicAdd(&cnt[(size_t)b * classes + k], 1);
        }
    }
}

// Persistent grid: every block walks the (image, class) counter array with a grid stride and works on the
// pairs that have at least two candidates (yolo9000: 9418 classes x batch pairs, a handful of them live).
// Dynamic smem: idx[cap] int, key[cap] float, sorted[cap] int, alive[cap] int, box[cap] float4.
__global__ void nms_mark_kernel(const float4 *__restrict__ boxes, float *probs, const int *__restrict__ cnt,
                                int batch, int total, int classes, float thresh, int cap)
{
    extern __shared__ __align__(16) unsigned char nms_smem[];
    const long long pairs = (long long)batch * classes;
  for (long long pair = blockIdx.x; pair < pairs; pair += gridDim.x) {
    if (cnt[pair] <= 1) continue; // a lone candidate only "suppresses" zeros (uniform per block)
    const int b = (int)(pair / classes), k = (int)(pair - (long long)b * classes);
    float4 *s_box = reinterpret_cast<float4 *>(nms_smem);
    int *s_idx = reinterpret_cast<int *>(s_box + cap);
    float *s_key = reinterpret_cast<float *>(s_idx + cap);
    int *s_sorted = reinterpret_cast<int *>(s_key + cap);
    int *s_alive = s_sorted + cap;
    __shared__ int s_warp_tot[32];
    __shared__ int s_base;

    float *pimg = probs + (size_t)b * total * classes;
    const float4 *bimg = boxes + (size_t)b * total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;

    // 1. ordered compaction of the candidates (index order)
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int start = 0; start < total; start += blockDim.x) {
        const int i = start + threadIdx.x;
        float p = 0.f;
        if (i < total) p = pimg[(size_t)i * classes + k];
        const bool is = (p != 0.f);
        const unsigned m = __ballot_sync(0xffffffffu, is);
        const int within = __popc(m & ((1u << lane) - 1));
        if (lane == 0) s_warp_tot[warp] = __popc(m);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp_tot[w];
        if (is) {
            const int pos = off + within;
            if (pos < cap) {
                s_idx[pos] = i;
                s_key[pos] = fabsf(p);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < nw; ++w) t += s_warp_tot[w];
            s_base += t;
        }
        __syncthreads();
    }
    const int m = s_base < cap ? s_base : cap;

    // 2. rank sort: position = number of candidates that sort before me
    for (int a = threadIdx.x; a < m; a += blockDim.x) {
        const int ia = s_idx[a];
        const float pa = s_key[a];
        int rank = 0;
        for (int o = 0; o < m; ++o) {
            if (o == a) continue;
            if (sorts_before(pimg, classes, k, s_idx[o], s_key[o], ia, pa)) ++rank;
        }
        s_sorted[rank] = ia;
    }
    __syncthreads();
    for (int a = threadIdx.x; a < m; a += blockDim.x) {
        s_box[a] = bimg[s_sorted[a]];
        s_alive[a] = 1;
    }
    __syncthreads();

    // 3. greedy suppression in sorted order; a barrier only after a live box acted
    for (int i = 0; i < m - 1; ++i) {
        if (!s_alive[i]) continue; // uniform: everyone reads the same flag
        const float4 a = s_box[i];
        for (int j = i + 1 + threadIdx.x; j < m; j += blockDim.x) {
            if (s_alive[j] && box_iou_ref(a, s_box[j]) > thresh) s_alive[j] = 0;
        }
        __syncthreads();
    }

    // 4. mark the suppressed entries (sign flip keeps |p| for concurrent tie-breaks)
    for (int a = threadIdx.x; a < m; a += blockDim.x) {
        if (!s_alive[a]) {
            float *q = pimg + (size_t)s_sorted[a] * classes + k;
            *q = -fabsf(*q);
        }
    }
    __syncthreads(); // the shared arrays are reused by this block's next pair
  }
}

// negative == suppressed -> 0
__global__ void nms_clear_kernel(float *__restrict__ probs, long long n)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n;
         t += (long long)gridDim.x * blockDim.x) {
        if (probs[t] < 0.f) probs[t] = 0.f;
    }
}

// ---- do_nms (box.c:279-297), the unsorted variant --------------------------------------------------
// bit j of mask[i][j / 32] : j > i and box_iou(boxes[i], boxes[j]) > thresh
__global__ void iou_mask_kernel(const float4 *__restrict__ boxes, int total, float thresh, unsigned *__restrict__ mask,
                                int words)
{
    const long long n = (long long)total * words;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / words), w = (int)(t - (long long)i * words);
        const float4 a = boxes[i];
        unsigned bits = 0;
        for (int bit = 0; bit < 32; ++bit) {
            const int j = w * 32 + bit;
            if (j > i && j < total && box_iou_ref(a, boxes[j]) > thresh) bits |= 1u << bit;
        }
        mask[t] = bits;
    }
}

// One block.  The reference walks rows i in order, skips a row none of whose probabilities is positive AT THAT
// MOMENT (a test that couples all classes), then for every later overlapping row j zeroes, per class, the
// smaller of the two entries.  Here a thread owns whole class columns (no two threads ever touch the same
// entry); only the row test needs the block.
__global__ void __launch_bounds__(1024) nms_unsorted_kernel(float *probs, const unsigned *__restrict__ mask, int total,
                                                            int classes, int words)
{
    for (int i = 0; i < total; ++i) {
        float *pi = probs + (size_t)i * classes;
        int mine = 0;
        for (int k = threadIdx.x; k < classes; k += blockDim.x) mine |= (pi[k] > 0);
        if (!__syncthreads_or(mine)) continue;
        for (int w = (i + 1) >> 5; w < words; ++w) {
            unsigned bits = mask[(size_t)i * words + w];
            while (bits) {
                const int j = (w << 5) + __ffs(bits) - 1;
                bits &= bits - 1;
                float *pj = probs + (size_t)j * classes;
                for (int k = threadIdx.x; k < classes; k += blockDim.x) {
                    if (pi[k] < pj[k]) pi[k] = 0;
                    else pj[k] = 0;
                }
            }
        }
    }
}

// ---- tiled detection: do_nms_sort over a frame's union of tiles --------------------------------------------------
// A frame's tiles are consecutive images of the batch, so the union of their boxes and probability rows is one
// contiguous span of count * total rows, union index u = tile * total + box.

// boxes relative to a tile -> relative to its frame (x0 == 0 && tw == W: the axis passes unchanged)
__global__ void tile_map_kernel(float4 *__restrict__ boxes, const y2_tile *__restrict__ tiles, long long nboxes,
                                int total)
{
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < nboxes;
         t += (long long)gridDim.x * blockDim.x) {
        const y2_tile g = tiles[t / total];
        float4 b = boxes[t];
        if (!(g.x0 == 0 && g.w == g.frame_w)) {
            const float tw = (float)g.w, fw = (float)g.frame_w;
            b.x = ((float)g.x0 + b.x * tw) / fw;
            b.z = (b.z * tw) / fw;
        }
        if (!(g.y0 == 0 && g.h == g.frame_h)) {
            const float th = (float)g.h, fh = (float)g.frame_h;
            b.y = ((float)g.y0 + b.y * th) / fh;
            b.w = (b.w * th) / fh;
        }
        boxes[t] = b;
    }
}

static const int TILE_NMS_THREADS = 256;
static const int TILE_NMS_SMEM_CAP = 2048; // candidates a block stages in shared memory (a power of two)
static const int TILE_NMS_PER_SM = 4;      // blocks of TILE_NMS_SMEM_CAP * 25 bytes each fit an SM

// a candidate's sort key: ascending keys are p descending, then union index ascending (p > 0, so its bits order like
// its value)
__device__ __forceinline__ unsigned long long cand_key(float p, int u)
{
    return ((unsigned long long)(0xffffffffu - __float_as_uint(p)) << 32) | (unsigned)u;
}
__device__ __forceinline__ unsigned key_hi(unsigned long long k) { return (unsigned)(k >> 32); }

// Persistent grid over (frame, class) pairs with two or more candidates, as nms_mark_kernel, but without a bound on
// the candidates: up to TILE_NMS_SMEM_CAP they are staged in shared memory, beyond that in the block's slice of ws
// (ws_stride 8-byte words: the keys, the boxes in sorted order, one alive byte per key).  The order is
// nms_mark_kernel's rank order, found by a bitonic sort on (p desc, union index asc) and then, inside each run of
// equal p, an insertion sort with sorts_before; sorts_before is a total order that agrees with the key wherever the p
// differ, so both give the same sequence.  Dynamic smem: box[cap] float4, key[cap] u64, alive[cap] u8.
__global__ void __launch_bounds__(TILE_NMS_THREADS)
    tile_nms_kernel(const float4 *__restrict__ boxes, float *probs, const int *__restrict__ cnt,
                    const y2_tile_span *__restrict__ spans, int n, int total, int classes, float thresh,
                    unsigned long long *__restrict__ ws, long long ws_stride)
{
    extern __shared__ __align__(16) unsigned char tile_smem[];
    float4 *s_box = reinterpret_cast<float4 *>(tile_smem);
    unsigned long long *s_key = reinterpret_cast<unsigned long long *>(s_box + TILE_NMS_SMEM_CAP);
    unsigned char *s_alive = reinterpret_cast<unsigned char *>(s_key + TILE_NMS_SMEM_CAP);
    __shared__ int s_m;
    const long long pairs = (long long)n * classes;
    for (long long pair = blockIdx.x; pair < pairs; pair += gridDim.x) {
        const int f = (int)(pair / classes), k = (int)(pair - (long long)f * classes);
        const y2_tile_span sp = spans[f];
        int m = 0;
        for (int t = 0; t < sp.count; ++t) m += cnt[(size_t)(sp.first + t) * classes + k];
        if (m <= 1) continue; // uniform per block
        const int span = sp.count * total;
        float *pimg = probs + (size_t)sp.first * total * classes;
        const float4 *bimg = boxes + (size_t)sp.first * total;
        int P = 1;
        while (P < m) P <<= 1;
        const bool fits = P <= TILE_NMS_SMEM_CAP;
        unsigned long long *key = fits ? s_key : ws + blockIdx.x * ws_stride;
        float4 *box = fits ? s_box : reinterpret_cast<float4 *>(key + P);
        unsigned char *alive = fits ? s_alive : reinterpret_cast<unsigned char *>(key + 3 * (long long)P);

        // 1. the candidates, in any order (the sort decides it)
        if (threadIdx.x == 0) s_m = 0;
        __syncthreads();
        for (int u = threadIdx.x; u < span; u += blockDim.x) {
            const float p = pimg[(size_t)u * classes + k];
            if (p != 0.f) {
                const int pos = atomicAdd(&s_m, 1);
                if (pos < P) key[pos] = cand_key(fabsf(p), u);
            }
        }
        __syncthreads();
        m = min(s_m, P);
        for (int a = m + threadIdx.x; a < P; a += blockDim.x) key[a] = ~0ull;
        __syncthreads();

        // 2. bitonic sort of the keys
        for (int size = 2; size <= P; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int a = threadIdx.x; a < P; a += blockDim.x) {
                    const int b = a ^ stride;
                    if (b > a) {
                        const unsigned long long ka = key[a], kb = key[b];
                        if ((ka > kb) == ((a & size) == 0)) {
                            key[a] = kb;
                            key[b] = ka;
                        }
                    }
                }
                __syncthreads();
            }

        // 3. runs of equal p, now in union-index order, take the order do_nms_sort carried over from the earlier
        //    classes: the thread at a run's start sorts it (a run only permutes keys with its own p)
        if (k > 0)
            for (int a = threadIdx.x; a < m; a += blockDim.x) {
                const unsigned hi = key_hi(key[a]);
                if ((a > 0 && key_hi(key[a - 1]) == hi) || a + 1 >= m || key_hi(key[a + 1]) != hi) continue;
                const float p = __uint_as_float(0xffffffffu - hi);
                int e = a + 1;
                while (e < m && key_hi(key[e]) == hi) ++e;
                for (int x = a + 1; x < e; ++x) {
                    const unsigned long long kx = key[x];
                    int y = x - 1;
                    while (y >= a && sorts_before(pimg, classes, k, (int)(unsigned)kx, p, (int)(unsigned)key[y], p)) {
                        key[y + 1] = key[y];
                        --y;
                    }
                    key[y + 1] = kx;
                }
            }
        __syncthreads();

        // 4. greedy suppression in that order, the boxes staged in it; a barrier only after a live box acted
        for (int a = threadIdx.x; a < m; a += blockDim.x) {
            box[a] = bimg[(unsigned)key[a]];
            alive[a] = 1;
        }
        __syncthreads();
        for (int i = 0; i < m - 1; ++i) {
            if (!alive[i]) continue; // uniform: everyone reads the same flag
            const float4 a = box[i];
            for (int j = i + 1 + threadIdx.x; j < m; j += blockDim.x)
                if (alive[j] && box_iou_ref(a, box[j]) > thresh) alive[j] = 0;
            __syncthreads();
        }

        // 5. mark the suppressed entries (the sign flip keeps |p| for the other classes' tie-breaks)
        for (int a = threadIdx.x; a < m; a += blockDim.x)
            if (!alive[a]) {
                float *q = pimg + (size_t)(unsigned)key[a] * classes + k;
                *q = -fabsf(*q);
            }
        __syncthreads(); // the staging is reused by this block's next pair
    }
}

// The final pick over each frame's union (one block per frame): per row max_index (utils.c:533-545, first maximum,
// negative = suppressed = 0), kept when > thresh, compacted in union-index order as collect_kernel does.  Hands the
// frame's tiles' candidate counters back zeroed.
static const int TILE_COLLECT_THREADS = 512;
__global__ void __launch_bounds__(TILE_COLLECT_THREADS)
    tile_collect_kernel(const float4 *__restrict__ boxes, const float *__restrict__ probs,
                        const y2_tile_span *__restrict__ spans, int total, int classes, float thresh,
                        y2_det *__restrict__ det, int *__restrict__ count, int max_det, int *__restrict__ nz_count)
{
    __shared__ int s_warp_total[32];
    __shared__ int s_running;
    const int f = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const y2_tile_span sp = spans[f];
    const int span = sp.count * total;
    const float *pimg = probs + (size_t)sp.first * total * classes;
    const float4 *bimg = boxes + (size_t)sp.first * total;
    y2_det *d = det + (size_t)f * max_det;
    if (threadIdx.x == 0) s_running = 0;
    __syncthreads();
    for (int base = 0; base < span; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int obj = -1;
        float best = 0.f;
        if (i < span) {
            const float *p = pimg + (size_t)i * classes;
            best = fmaxf(p[0], 0.f);
            int arg = 0;
            for (int j = 1; j < classes; ++j) {
                const float v = fmaxf(p[j], 0.f);
                if (v > best) {
                    best = v;
                    arg = j;
                }
            }
            if (best > thresh) obj = arg;
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, obj >= 0);
        if (lane == 0) s_warp_total[warp] = __popc(ballot);
        __syncthreads();
        int before = s_running;
        for (int wv = 0; wv < warp; ++wv) before += s_warp_total[wv];
        const int pos = before + __popc(ballot & ((1u << lane) - 1u));
        if (obj >= 0 && pos < max_det) {
            const float4 q = bimg[i];
            d[pos] = y2_det{q.x, q.y, q.z, q.w, best, obj, i};
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = s_running;
            for (int wv = 0; wv < nw; ++wv) t += s_warp_total[wv];
            s_running = t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) count[f] = s_running;
    for (int j = threadIdx.x; j < sp.count * classes; j += blockDim.x) nz_count[(size_t)sp.first * classes + j] = 0;
}

} // namespace y2

using namespace y2;

extern "C" int y2_tile_map(float *boxes, const y2_tile *tiles, int n_tiles, int total, y2_stream_t s)
{
    if (!boxes || !tiles || n_tiles < 1 || total < 1) return Y2_EINVAL;
    const long long nb = (long long)n_tiles * total;
    long long blocks = (nb + 255) / 256;
    if (blocks > (long long)sm_count() * 8) blocks = (long long)sm_count() * 8;
    tile_map_kernel<<<(int)blocks, 256, 0, to_stream(s)>>>(reinterpret_cast<float4 *>(boxes), tiles, nb, total);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

static int tile_nms_grid(int n, int classes)
{
    const long long pairs = (long long)n * classes, cap = (long long)sm_count() * TILE_NMS_PER_SM;
    return (int)(pairs < cap ? pairs : cap);
}

static long long pow2_at_least(long long v)
{
    long long p = 1;
    while (p < v) p <<= 1;
    return p;
}

extern "C" size_t y2_tile_nms_ws_bytes(int n, int classes, long long max_span)
{
    if (n < 1 || classes < 1 || max_span <= TILE_NMS_SMEM_CAP) return 0;
    const long long P = pow2_at_least(max_span);
    return (size_t)tile_nms_grid(n, classes) * (size_t)(3 * P + P / 8) * 8;
}

extern "C" int y2_tile_nms(const float *boxes, float *probs, const int *cnt, const y2_tile_span *spans, int n,
                           int total, int classes, int max_tiles, float thresh, void *ws, size_t ws_bytes,
                           y2_stream_t s)
{
    const long long max_span = (long long)max_tiles * total;
    if (!boxes || !probs || !cnt || !spans || n < 1 || total < 1 || classes < 1 || max_tiles < 1 ||
        max_span > 0x40000000LL) {
        set_error("y2_tile_nms: invalid arguments (n=%d total=%d classes=%d max_tiles=%d)", n, total, classes,
                  max_tiles);
        return Y2_EINVAL;
    }
    const size_t need = y2_tile_nms_ws_bytes(n, classes, max_span);
    if (need > ws_bytes || (need && !ws)) {
        set_error("y2_tile_nms: %zu bytes of scratch needed, %zu given", need, ws_bytes);
        return Y2_EINVAL;
    }
    const long long P = pow2_at_least(max_span);
    const size_t smem = (size_t)TILE_NMS_SMEM_CAP * (sizeof(float4) + sizeof(unsigned long long) + 1);
    static bool attr_done[64] = {false};
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !attr_done[dev]) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(tile_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (dev >= 0 && dev < 64) attr_done[dev] = true;
    }
    tile_nms_kernel<<<tile_nms_grid(n, classes), TILE_NMS_THREADS, smem, to_stream(s)>>>(
        reinterpret_cast<const float4 *>(boxes), probs, cnt, spans, n, total, classes, thresh,
        (unsigned long long *)ws, need ? 3 * P + P / 8 : 0);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_tile_collect(const float *boxes, const float *probs, const y2_tile_span *spans, int n, int total,
                               int classes, float thresh, y2_det *det, int *count, int max_det, int *nz_count,
                               y2_stream_t s)
{
    if (!boxes || !probs || !spans || !det || !count || !nz_count || n < 1 || n > 65535 || total < 1 ||
        classes < 1 || max_det < 0) {
        set_error("y2_tile_collect: invalid arguments (n=%d total=%d classes=%d max_det=%d)", n, total, classes,
                  max_det);
        return Y2_EINVAL;
    }
    tile_collect_kernel<<<n, TILE_COLLECT_THREADS, 0, to_stream(s)>>>(reinterpret_cast<const float4 *>(boxes), probs,
                                                                     spans, total, classes, thresh, det, count,
                                                                     max_det, nz_count);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_nms_unsorted(const float *boxes, float *probs, int total, int classes, float thresh, y2_stream_t s)
{
    if (!boxes || !probs || total <= 0 || classes <= 0) return Y2_EINVAL;
    cudaStream_t st = to_stream(s);
    const int words = (total + 31) / 32;
    unsigned *mask = nullptr;
    Y2_CUDA_CHECK(cudaMalloc(&mask, (size_t)total * words * sizeof(unsigned)));
    const long long n = (long long)total * words;
    long long blocks = (n + 255) / 256;
    const long long capb = (long long)sm_count() * 16;
    if (blocks > capb) blocks = capb;
    iou_mask_kernel<<<(int)blocks, 256, 0, st>>>(reinterpret_cast<const float4 *>(boxes), total, thresh, mask, words);
    int rc = cudaGetLastError() == cudaSuccess ? Y2_OK : Y2_ECUDA;
    if (rc == Y2_OK) {
        int threads = classes < 1024 ? (classes + 31) / 32 * 32 : 1024;
        nms_unsorted_kernel<<<1, threads, 0, st>>>(probs, mask, total, classes, words);
        if (cudaGetLastError() != cudaSuccess) rc = Y2_ECUDA;
    }
    cudaStreamSynchronize(st);
    cudaFree(mask);
    return rc;
}

static int nms_mark_launch(const float *boxes, float *probs, const int *cnt, int batch, int total, int classes,
                           float thresh, cudaStream_t st)
{
    const int cap = total;
    const size_t smem = (size_t)cap * (sizeof(float4) + 4 * sizeof(int));
    if (smem > 200 * 1024) {
        set_error("y2_nms_sort: %d boxes per image exceed the shared-memory staging", total);
        return Y2_EINVAL;
    }
    int dev = 0;
    Y2_CUDA_CHECK(cudaGetDevice(&dev));
    static bool attr_done[64] = {false};
    if (dev >= 0 && dev < 64 && !attr_done[dev] && smem > 48 * 1024) {
        Y2_CUDA_CHECK(cudaFuncSetAttribute(nms_mark_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           200 * 1024));
        attr_done[dev] = true;
    }
    const long long pairs = (long long)batch * classes;
    const int per_sm = smem > 100 * 1024 ? 1 : smem > 48 * 1024 ? 2 : 4;
    long long blocks = (long long)sm_count() * per_sm;
    if (blocks > pairs) blocks = pairs;
    nms_mark_kernel<<<(int)blocks, 256, smem, st>>>(reinterpret_cast<const float4 *>(boxes), probs, cnt, batch, total,
                                                    classes, thresh, cap);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// Suppression only, for callers that own the candidate counters (the network's detection path: the box
// decode counts while it writes the probabilities, the final pick reads "negative" as suppressed).
extern "C" int y2_nms_mark(const float *boxes, float *probs, const int *cnt, int batch, int total, int classes,
                           float thresh, y2_stream_t s)
{
    if (!boxes || !probs || !cnt || batch <= 0 || total <= 0 || classes <= 0) return Y2_EINVAL;
    return nms_mark_launch(boxes, probs, cnt, batch, total, classes, thresh, to_stream(s));
}

// Stand-alone do_nms_sort: owns nothing between calls (the counters live for the duration of the call), so any
// number of networks, streams and host threads may use it concurrently.
extern "C" int y2_nms_sort(const float *boxes, float *probs, int batch, int total, int classes, float thresh,
                           y2_stream_t s)
{
    if (!boxes || !probs || batch <= 0 || total <= 0 || classes <= 0) return Y2_EINVAL;
    cudaStream_t st = to_stream(s);
    const size_t need = (size_t)batch * classes;
    int *cnt = nullptr;
    Y2_CUDA_CHECK(cudaMalloc(&cnt, need * sizeof(int)));
    cudaError_t e = cudaMemsetAsync(cnt, 0, need * sizeof(int), st);
    int rc = Y2_OK;
    if (e != cudaSuccess) rc = Y2_ECUDA;
    const long long n = (long long)batch * total * classes;
    long long blocks = (n + 255) / 256;
    const long long capb = (long long)sm_count() * 16;
    if (blocks > capb) blocks = capb;
    if (rc == Y2_OK) {
        nms_count_kernel<<<(int)blocks, 256, 0, st>>>(probs, cnt, batch, total, classes);
        if (cudaGetLastError() != cudaSuccess) rc = Y2_ECUDA;
    }
    if (rc == Y2_OK) rc = nms_mark_launch(boxes, probs, cnt, batch, total, classes, thresh, st);
    if (rc == Y2_OK) {
        nms_clear_kernel<<<(int)blocks, 256, 0, st>>>(probs, n);
        if (cudaGetLastError() != cudaSuccess) rc = Y2_ECUDA;
    }
    cudaStreamSynchronize(st); // the counters are freed below
    cudaFree(cnt);
    return rc;
}
