// HBM-bound data-movement kernels on the padded-NHWC bf16 layout:
// input packing, maxpool, reorg, route copy, export to the reference's NCHW fp32.
// All are grid-stride kernels launched with a multiple of the SM count; channel-innermost
// 16-byte accesses wherever the layout allows.
#include "y2_common.cuh"

#include <float.h>
#include <limits.h>

namespace y2 {

static inline int grid_for(long long work_items, int threads)
{
    long long blocks = (work_items + threads - 1) / threads;
    long long cap = (long long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// ---------------------------------------------------------------------------------
// fp32 NCHW -> bf16 padded NHWC
// ---------------------------------------------------------------------------------
__global__ void pack_nchw_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst,
                                 int batch, int c, int h, int w, int cpad, int cs)
{
    const int hp = h + 1, wp = w + 1;
    const long long total = (long long)batch * hp * wp;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total;
         p += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(p % wp);
        const int y = (int)((p / wp) % hp);
        const int b = (int)(p / ((long long)wp * hp));
        __nv_bfloat16 *o = dst + p * cs;
        const bool valid = (x < w) && (y < h);
        const float *s = src + ((size_t)b * c * h + y) * w + x;
        for (int k = 0; k < cpad; ++k) {
            float v = (valid && k < c) ? __ldg(s + (size_t)k * h * w) : 0.f;
            o[k] = __float2bfloat16_rn(v);
        }
    }
}

// ---------------------------------------------------------------------------------
// first-layer patch gather (K ordering of the reference's im2col.c:16-39)
// ---------------------------------------------------------------------------------
template <int KPAD>
__global__ void pack_patches_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst,
                                    int batch, int c, int h, int w, int ksize)
{
    const int hp = h + 1, wp = w + 1;
    const int pad = ksize / 2;
    const int kk = ksize * ksize;
    const long long total = (long long)batch * hp * wp;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total;
         p += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(p % wp);
        const int y = (int)((p / wp) % hp);
        const int b = (int)(p / ((long long)wp * hp));
        float v[KPAD];
#pragma unroll
        for (int k = 0; k < KPAD; ++k) v[k] = 0.f;
        if (x < w && y < h) {
            const float *s = src + (size_t)b * c * h * w;
#pragma unroll
            for (int k = 0; k < KPAD; ++k) {
                if (k < c * kk) {
                    const int ci = k / kk;
                    const int r = (k % kk) / ksize;
                    const int q = k % ksize;
                    const int yy = y + r - pad, xx = x + q - pad;
                    if (yy >= 0 && yy < h && xx >= 0 && xx < w)
                        v[k] = __ldg(s + ((size_t)ci * h + yy) * w + xx);
                }
            }
        }
        uint4 *o = reinterpret_cast<uint4 *>(dst + p * KPAD);
#pragma unroll
        for (int g = 0; g < KPAD / 8; ++g) {
            uint4 t;
            t.x = pack_bf16x2(v[g * 8 + 0], v[g * 8 + 1]);
            t.y = pack_bf16x2(v[g * 8 + 2], v[g * 8 + 3]);
            t.z = pack_bf16x2(v[g * 8 + 4], v[g * 8 + 5]);
            t.w = pack_bf16x2(v[g * 8 + 6], v[g * 8 + 7]);
            o[g] = t;
        }
    }
}

// ---------------------------------------------------------------------------------
// general patch gather for the convolutions the shifted-descriptor kernels do not cover
// (any size / stride / padding: the 7x7/2 first layer and the 3x3/2 layers of resnet50.cfg).
// The convolution then runs as a 1x1 tcgen05 GEMM over the gathered rows.  One thread per
// (output position, 8 K values), one 16-byte store each.
//   first layer:  fp32 NCHW in,  K index = c*k*k + r*k + s          (im2col.c:26-28)
//   later layers: bf16 padded NHWC in, K index = (r*k + s)*cin_pad + c
// ---------------------------------------------------------------------------------
__global__ void gather_patches_f32_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst,
                                          int batch, int c, int h, int w, int ksize, int stride, int pad,
                                          int oh, int ow, int kpad)
{
    const int ohp = oh + 1, owp = ow + 1, k8 = kpad / 8, kk = ksize * ksize, kreal = c * kk;
    const long long total = (long long)batch * ohp * owp * k8;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(t % k8);
        const long long p = t / k8;
        const int ox = (int)(p % owp);
        const int oy = (int)((p / owp) % ohp);
        const int b = (int)(p / ((long long)owp * ohp));
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = 0.f;
        if (ox < ow && oy < oh) {
            const float *s = src + (size_t)b * c * h * w;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = g * 8 + q;
                if (k < kreal) {
                    const int ci = k / kk, r = (k % kk) / ksize, sx = k % ksize;
                    const int yy = oy * stride + r - pad, xx = ox * stride + sx - pad;
                    if (yy >= 0 && yy < h && xx >= 0 && xx < w) v[q] = __ldg(s + ((size_t)ci * h + yy) * w + xx);
                }
            }
        }
        uint4 o;
        o.x = pack_bf16x2(v[0], v[1]);
        o.y = pack_bf16x2(v[2], v[3]);
        o.z = pack_bf16x2(v[4], v[5]);
        o.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4 *>(dst + (size_t)p * kpad + g * 8) = o;
    }
}

// First-layer gather for 5..8-wide kernels (resnet50's 7x7/2): K index = (c*k + r)*8 + s, i.e. every kernel
// ROW owns one aligned 16-byte group (s >= k zero).  One thread per (position, c, r) reads k neighbouring
// pixels of one image row and writes one group - no per-element div/mod, no scattered scalar loads (the
// [c][kh][kw] order above took 0.8 ms for resnet50's first layer at batch 64).
__global__ void gather_rows_f32_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, int batch,
                                       int c, int h, int w, int ksize, int stride, int pad, int oh, int ow, int kpad)
{
    // a block per output row (b, oy): the per-element index math is 32-bit with small divisors (the 64-bit
    // div / mod chain of a flat index cost more than the copy itself: 0.4 of resnet50's 0.5 ms first layer)
    const int ohp = oh + 1, owp = ow + 1, k8 = kpad / 8, groups = c * ksize;
    const int rows = batch * ohp, per_row = owp * k8;
    for (int rowi = blockIdx.x; rowi < rows; rowi += gridDim.x) {
        const int b = rowi / ohp, oy = rowi - b * ohp;
        __nv_bfloat16 *drow = dst + (size_t)rowi * owp * kpad;
        for (int t = threadIdx.x; t < per_row; t += blockDim.x) {
            const int ox = t / k8, g = t - ox * k8;
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = 0.f;
            if (ox < ow && oy < oh && g < groups) {
                const int ci = g / ksize, r = g - ci * ksize;
                const int yy = oy * stride + r - pad;
                if (yy >= 0 && yy < h) {
                    const float *row = src + (((size_t)b * c + ci) * h + yy) * w;
                    const int x0 = ox * stride - pad;
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const int xx = x0 + q;
                        if (q < ksize && xx >= 0 && xx < w) v[q] = __ldg(row + xx);
                    }
                }
            }
            uint4 o;
            o.x = pack_bf16x2(v[0], v[1]);
            o.y = pack_bf16x2(v[2], v[3]);
            o.z = pack_bf16x2(v[4], v[5]);
            o.w = pack_bf16x2(v[6], v[7]);
            *reinterpret_cast<uint4 *>(drow + (size_t)t * 8) = o;
        }
    }
}

// The same gather with the c*ksize input rows an output row needs staged in shared memory: the image is read with
// coalesced loads once per output row (the direct form issues seven scalar loads per thread whose 32 lanes touch ~24
// different sectors - the L1 tag path, not the 409 MB patch write, bounded resnet50's first layer), the groups are
// assembled from shared memory and written back 16 bytes per thread, consecutive threads to consecutive addresses.
__global__ void gather_rows_f32_smem_kernel(const float *__restrict__ src, __nv_bfloat16 *__restrict__ dst, int batch,
                                            int c, int h, int w, int ksize, int stride, int pad, int oh, int ow, int kpad)
{
    extern __shared__ float srow[];  // [c*ksize][ws], ws odd: the lanes of a warp read different rows at one column
    const int ws = w | 1;
    const int ohp = oh + 1, owp = ow + 1, k8 = kpad / 8, groups = c * ksize;
    const int rows = batch * ohp, per_row = owp * k8;
    for (int rowi = blockIdx.x; rowi < rows; rowi += gridDim.x) {
        const int b = rowi / ohp, oy = rowi - b * ohp;
        __nv_bfloat16 *drow = dst + (size_t)rowi * owp * kpad;
        __syncthreads();  // the previous row's groups have been read
        if (oy < oh) {
            // (g, x) and (ci, r) advance by a constant stride: carried instead of divided (the per-element divisions
            // by w, ksize and k8 made this kernel instruction-bound at 1.7 TB/s)
            const int dg = (int)blockDim.x / w, dx = (int)blockDim.x - dg * w;
            int g = (int)threadIdx.x / w, x = (int)threadIdx.x - g * w;
            int ci = g / ksize, r = g - ci * ksize;
            while (g < groups) {
                const int yy = oy * stride + r - pad;
                srow[g * ws + x] = (yy >= 0 && yy < h) ? __ldg(src + (((size_t)b * c + ci) * h + yy) * w + x) : 0.f;
                x += dx;
                int step = dg;
                if (x >= w) { x -= w; ++step; }
                g += step;
                r += step;
                while (r >= ksize) { r -= ksize; ++ci; }
            }
        }
        __syncthreads();
        const int dox = (int)blockDim.x / k8, dgw = (int)blockDim.x - dox * k8;
        int ox = (int)threadIdx.x / k8, g = (int)threadIdx.x - ox * k8;
        for (int t = threadIdx.x; t < per_row; t += blockDim.x, ox += dox, g += dgw) {
            if (g >= k8) { g -= k8; ++ox; }
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = 0.f;
            if (ox < ow && oy < oh && g < groups) {
                const float *row = srow + g * ws;
                const int x0 = ox * stride - pad;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int xx = x0 + q;
                    if (q < ksize && xx >= 0 && xx < w) v[q] = row[xx];
                }
            }
            uint4 o;
            o.x = pack_bf16x2(v[0], v[1]);
            o.y = pack_bf16x2(v[2], v[3]);
            o.z = pack_bf16x2(v[4], v[5]);
            o.w = pack_bf16x2(v[6], v[7]);
            *reinterpret_cast<uint4 *>(drow + (size_t)t * 8) = o;
        }
    }
}

__global__ void gather_patches_bf16_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs, int cin_pad, int h,
                                           int w, __nv_bfloat16 *__restrict__ dst, int batch, int ksize,
                                           int stride, int pad, int oh, int ow)
{
    // a block per output row (b, oy), threads over (ox, tap, 8-channel group): 32-bit index math
    const int ohp = oh + 1, owp = ow + 1, c8 = cin_pad / 8, kk = ksize * ksize;
    const int hp = h + 1, wp = w + 1;
    const int rows = batch * ohp, per_pos = kk * c8, per_row = owp * per_pos;
    for (int rowi = blockIdx.x; rowi < rows; rowi += gridDim.x) {
        const int b = rowi / ohp, oy = rowi - b * ohp;
        __nv_bfloat16 *drow = dst + (size_t)rowi * owp * per_pos * 8;
        // (ox, tap, g) advance by a constant stride: carried instead of divided per 16-byte element
        const int bd = (int)blockDim.x;
        const int d_ox = bd / per_pos, d_tap = (bd - d_ox * per_pos) / c8, d_g = bd - d_ox * per_pos - d_tap * c8;
        const unsigned inv_k = (65536u + (unsigned)ksize - 1u) / (unsigned)ksize;  // tap / ksize for tap < 256
        int ox = (int)threadIdx.x / per_pos, tap = ((int)threadIdx.x - ox * per_pos) / c8,
            g = (int)threadIdx.x - ox * per_pos - tap * c8;
        for (int t = threadIdx.x; t < per_row; t += bd, g += d_g, tap += d_tap, ox += d_ox) {
            if (g >= c8) { g -= c8; ++tap; }
            if (tap >= kk) { tap -= kk; ++ox; }
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (ox < ow && oy < oh) {
                const int ty = (int)(((unsigned)tap * inv_k) >> 16);
                const int yy = oy * stride + ty - pad, xx = ox * stride + (tap - ty * ksize) - pad;
                if (yy >= 0 && yy < h && xx >= 0 && xx < w)
                    v = __ldg(reinterpret_cast<const uint4 *>(in + (((size_t)b * hp + yy) * wp + xx) * in_cs + g * 8));
            }
            *reinterpret_cast<uint4 *>(drow + (size_t)t * 8) = v;  // dst[p][tap*cin_pad + g*8]: t*8 within the row
        }
    }
}

// ---------------------------------------------------------------------------------
// decoded frame -> network input: uint8 interleaved RGB [B][sh][sw][3] -> fp32 planar [B][3][h][w],
// the composition of the reference's loaders and its resize on the host:
//   load_image_stb        im[k][y][x] = (float)byte / 255.           (yolo_v2_class.cpp:129-149)
//   resize_image          two-pass bilinear, horizontal into `part`, then vertical (image.c:1950-1993)
// Every float expression keeps the reference's operation order and roundings (explicit _rn
// intrinsics, no fma), so the result is bit-identical to the host path; the horizontal pass is
// recomputed for the two source rows a target pixel needs instead of materialising `part`.
// Quirk kept: the last target row takes only the (1-dy) term (image.c:1985 `continue`).
// ---------------------------------------------------------------------------------

// One source pixel's three bytes, R G B, already loaded (the tap of a converted format).
struct px3 {
    unsigned char v[3];
    __device__ __forceinline__ unsigned char operator[](int k) const { return v[k]; }
};

// resize_image's taps for canvas pixel (c, r) inside window f, all three planes from the same taps: out[k * hw] =
// plane k.  src.row(y) gives source row y and src.at(row, x) the tap of its pixel x, whose tap[k] is byte k (R G B);
// an interleaved tap is a pointer, so its bytes are loaded channel by channel next to the arithmetic that uses them.
// All four taps are formed, also where the edge column or the last row does not use them: every tap has
// 0 <= x <= src_w - 1 and 0 <= y <= src_h - 1 (ix is below src_w - 1 off the edge column, ix1, iy and iy1 are
// clamped), so it stays inside its frame's rows.  Shared by every frame kernel, so they agree bit for bit.
template <class Src>
__device__ __forceinline__ void resize_taps(const y2_frame_window &f, int c, int r, const float *lut, const Src &src,
                                            float *out, int hw)
{
    const int sw = f.src_w, sh = f.src_h;
    // horizontal taps of resize_part: the edge column, or ix / ix1 with weight dx
    const bool edge = c == f.new_w - 1 || sw == 1;
    int ix = sw - 1, ix1 = sw - 1;
    float dx = 0.f;
    if (!edge) {
        const float sx = __fmul_rn((float)c, f.w_scale);
        ix = (int)sx;
        dx = __fsub_rn(sx, (float)ix);
        ix1 = ix + 1;
        if (ix1 > sw - 1) ix1 = sw - 1; // the reference would assert here; unreachable for exact scales
    }
    const float sy = __fmul_rn((float)r, f.h_scale);
    int iy = (int)sy;
    if (iy > sh - 1) iy = sh - 1;
    const float fy = __fsub_rn(sy, (float)iy);
    const bool two_rows = !(r == f.new_h - 1 || sh == 1); // image.c:1985: the last row takes the (1-dy) term only
    int iy1 = iy + 1;
    if (iy1 > sh - 1) iy1 = sh - 1;
    const auto r0 = src.row(iy), r1 = src.row(iy1);
    const auto a0 = src.at(r0, ix), b0 = src.at(r0, ix1), a1 = src.at(r1, ix), b1 = src.at(r1, ix1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float part0 = lut[a0[k]];
        if (!edge) part0 = __fadd_rn(__fmul_rn(__fsub_rn(1.f, dx), part0), __fmul_rn(dx, lut[b0[k]]));
        float val = __fmul_rn(__fsub_rn(1.f, fy), part0);
        if (two_rows) {
            float part1 = lut[a1[k]];
            if (!edge) part1 = __fadd_rn(__fmul_rn(__fsub_rn(1.f, dx), part1), __fmul_rn(dx, lut[b1[k]]));
            val = __fadd_rn(val, __fmul_rn(fy, part1));
        }
        out[(size_t)k * hw] = val;
    }
}

// Interleaved 3-byte pixels, rows `pitch` bytes apart; SWAP: stored B G R.  A tap is the pixel's address.
template <bool SWAP>
struct Interleaved {
    const unsigned char *data;
    size_t pitch;
    struct Tap {
        const unsigned char *q;
        __device__ __forceinline__ unsigned char operator[](int k) const { return q[SWAP ? 2 - k : k]; }
    };
    __device__ __forceinline__ const unsigned char *row(int y) const { return data + (size_t)y * pitch; }
    __device__ __forceinline__ Tap at(const unsigned char *row, int x) const { return Tap{row + x * 3}; }
};

// A packed frame-list frame: tight RGB rows of 3 * sw bytes, each row's address computed as (size_t)y * sw * 3.
struct PackedRGB {
    const unsigned char *data;
    int sw;
    __device__ __forceinline__ const unsigned char *row(int y) const { return data + (size_t)y * sw * 3; }
    __device__ __forceinline__ Interleaved<false>::Tap at(const unsigned char *row, int x) const
    {
        return Interleaved<false>::Tap{row + x * 3};
    }
};

// The (float)(byte / 255.) table of load_image_stb, in shared memory.
__device__ __forceinline__ void fill_lut(float *lut)
{
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = (float)((double)(float)i / 255.);
    __syncthreads();
}

// The resized image fills the window [dx, dx+nw) x [dy, dy+nh) of the w x h canvas and the rest is .5f: the whole
// canvas for resize_image, the centred window of letterbox_image (image.c:1624-1644: fill_image(.5) + embed_image).
// Image b = blockIdx.y reads its record once: table[b], or for a uniform batch (table == NULL) the by-value record
// with the frame at uni.offset + b * stride.  One thread per output pixel writes all three planes from the same
// 3-byte taps.  Images b >= n are the .5f canvas.
__global__ void frames_u8_to_f32_kernel(const unsigned char *__restrict__ packed,
                                        const y2_frame_window *__restrict__ table, y2_frame_window uni,
                                        unsigned long long stride, int n, float *__restrict__ dst, int w, int h)
{
    __shared__ float lut[256];
    fill_lut(lut);
    const int b = blockIdx.y;
    const int hw = w * h;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    float *out = dst + (size_t)b * 3 * hw + p;
    const int y = p / w;
    y2_frame_window f = uni;
    if (b < n) {
        if (table) f = table[b];
        else f.offset += (unsigned long long)b * stride;
    }
    const int c = p - y * w - f.dx, r = y - f.dy;
    if (b >= n || c < 0 || c >= f.new_w || r < 0 || r >= f.new_h) {
        out[0] = .5f;
        out[hw] = .5f;
        out[2 * hw] = .5f;
        return;
    }
    resize_taps(f, c, r, lut, PackedRGB{packed + f.offset, f.src_w}, out, hw);
}

// NV12 -> RGB as OpenCV's cvtColor(COLOR_YUV2RGB_NV12): BT.601 limited range in 20-bit fixed point.  Exact in int32:
// every intermediate stays within +-6e8.
__device__ __forceinline__ px3 nv12_rgb(int Y, int U, int V)
{
    const int y = max(Y - 16, 0) * 1220542, half = 1 << 19, u = U - 128, v = V - 128;
    const int r = (y + half + 1673527 * v) >> 20;
    const int g = (y + half - 852492 * v - 409993 * u) >> 20;
    const int bl = (y + half + 2116026 * u) >> 20;
    return px3{{(unsigned char)min(max(r, 0), 255), (unsigned char)min(max(g, 0), 255),
                (unsigned char)min(max(bl, 0), 255)}};
}

// NV12: a Y plane and an interleaved U,V plane at half the rows; pixel x of row y takes the pair at (x & ~1) of UV
// row y >> 1.
struct Nv12 {
    const unsigned char *y, *uv;
    size_t pitch, uv_pitch;
    struct Row {
        const unsigned char *y, *uv;
    };
    __device__ __forceinline__ Row row(int yy) const
    {
        return Row{y + (size_t)yy * pitch, uv + (size_t)(yy >> 1) * uv_pitch};
    }
    __device__ __forceinline__ px3 at(const Row &r, int x) const
    {
        const unsigned char *q = r.uv + (x & ~1);
        return nv12_rgb(r.y[x], q[0], q[1]);
    }
};

// frames_u8_to_f32_kernel over frame sources: each record names its frame's device address, pitch and format, and
// the format is uniform per block (one image per blockIdx.y), so the switch does not diverge.  Bounds: a fetch has
// 0 <= x <= src_w - 1 and 0 <= y <= src_h - 1 (resize_taps), so an RGB/BGR fetch reads inside
// [data, data + (src_h-1)*pitch + 3*src_w) and an NV12 fetch inside [data, data + (src_h-1)*pitch + src_w) and, with
// src_w and src_h even, (y>>1) <= src_h/2 - 1 and (x&~1) + 1 <= src_w - 1, inside
// [uv, uv + (src_h/2-1)*uv_pitch + src_w).  The host checks those ranges before it launches.
__global__ void frames_src_to_f32_kernel(const y2_frame_src *__restrict__ table, int n, float *__restrict__ dst, int w,
                                         int h)
{
    __shared__ float lut[256];
    fill_lut(lut);
    const int b = blockIdx.y;
    const int hw = w * h;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= hw) return;
    float *out = dst + (size_t)b * 3 * hw + p;
    const int y = p / w;
    y2_frame_src s = {};
    if (b < n) s = table[b];
    const y2_frame_window &f = s.win;
    const int c = p - y * w - f.dx, r = y - f.dy;
    if (b >= n || c < 0 || c >= f.new_w || r < 0 || r >= f.new_h) {
        out[0] = .5f;
        out[hw] = .5f;
        out[2 * hw] = .5f;
        return;
    }
    const unsigned char *img = (const unsigned char *)f.offset;
    const size_t pitch = (size_t)s.pitch;
    if (s.format == Y2_FRAME_NV12)
        resize_taps(f, c, r, lut, Nv12{img, (const unsigned char *)s.uv, pitch, (size_t)s.uv_pitch}, out, hw);
    else if (s.format == Y2_FRAME_BGR24)
        resize_taps(f, c, r, lut, Interleaved<true>{img, pitch}, out, hw);
    else
        resize_taps(f, c, r, lut, Interleaved<false>{img, pitch}, out, hw);
}

// ---------------------------------------------------------------------------------
// bf16 padded NHWC slice -> fp32 NCHW (export of l.output).  32x32 smem transpose so
// both sides are coalesced: reads run along channels, writes along x.
// ---------------------------------------------------------------------------------
__global__ void unpack_nchw_kernel(const __nv_bfloat16 *__restrict__ src, float *__restrict__ dst,
                                   int batch, int c, int h, int w, int cs)
{
    __shared__ float tile[32][33];
    const int wp = w + 1, hp = h + 1;
    const int xt = (w + 31) / 32, ct = (c + 31) / 32;
    const long long ntiles = (long long)batch * h * xt * ct;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int cti = (int)(t % ct);
        const int xti = (int)((t / ct) % xt);
        const int y = (int)((t / ((long long)ct * xt)) % h);
        const int b = (int)(t / ((long long)ct * xt * h));
        // load: threadIdx.x -> channel, threadIdx.y -> x
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int x = xti * 32 + j, ch = cti * 32 + threadIdx.x;
            float v = 0.f;
            if (x < w && ch < c)
                v = __bfloat162float(src[(((size_t)b * hp + y) * wp + x) * cs + ch]);
            tile[j][threadIdx.x] = v;
        }
        __syncthreads();
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const int ch = cti * 32 + j, x = xti * 32 + threadIdx.x;
            if (x < w && ch < c) dst[(((size_t)b * c + ch) * h + y) * w + x] = tile[threadIdx.x][j];
        }
        __syncthreads();
    }
}

// fp32 flat NHWC [B][hw][cs] <-> fp32 NCHW [B][c][hw]
__global__ void flat_to_nchw_kernel(const float *__restrict__ src, float *__restrict__ dst, int batch,
                                    int c, int hw, int cs)
{
    const long long total = (long long)batch * c * hw;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i % hw);
        const int ch = (int)((i / hw) % c);
        const int b = (int)(i / ((long long)hw * c));
        dst[i] = src[((size_t)b * hw + s) * cs + ch];
    }
}
__global__ void nchw_to_flat_kernel(const float *__restrict__ src, float *__restrict__ dst, int batch,
                                    int c, int hw)
{
    const long long total = (long long)batch * c * hw;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int ch = (int)(i % c);
        const int s = (int)((i / c) % hw);
        const int b = (int)(i / ((long long)hw * c));
        dst[i] = src[((size_t)b * c + ch) * hw + s];
    }
}

// ---------------------------------------------------------------------------------
// maxpool: out[b,y,x,k] = max_{n,m<size} in[b, y*stride+n-pad, x*stride+m-pad, k], cells
// outside the valid extent are skipped (== -FLT_MAX in maxpool_layer.c:95-105).
// One thread per (output position, 8-channel group): 16-byte loads/stores, channel
// innermost -> fully coalesced.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ void bf16x8_max(uint4 &acc, const uint4 &v)
{
    __nv_bfloat162 *a = reinterpret_cast<__nv_bfloat162 *>(&acc);
    const __nv_bfloat162 *b = reinterpret_cast<const __nv_bfloat162 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = __hmax2(a[i], b[i]);
}

__global__ void maxpool_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs,
                               __nv_bfloat16 *__restrict__ out, int out_cs, int batch, int c8, int h,
                               int w, int oh, int ow, int size, int stride, int pad)
{
    const int ohp = oh + 1, owp = ow + 1, hp = h + 1, wp = w + 1;
    const long long total = (long long)batch * ohp * owp * c8;
    // -FLT_MAX is not representable in bf16; the most negative finite bf16 plays its role
    // (only reachable when a window has no valid cell, which the cfgs never produce).
    const uint32_t neg = 0xFF7FFF7Fu;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(i % c8);
        const long long p = i / c8;
        const int ox = (int)(p % owp);
        const int oy = (int)((p / owp) % ohp);
        const int b = (int)(p / ((long long)owp * ohp));
        uint4 acc = make_uint4(0u, 0u, 0u, 0u);
        if (ox < ow && oy < oh) {
            acc = make_uint4(neg, neg, neg, neg);
            for (int n = 0; n < size; ++n) {
                const int yy = oy * stride + n - pad;
                if (yy < 0 || yy >= h) continue;
                for (int m = 0; m < size; ++m) {
                    const int xx = ox * stride + m - pad;
                    if (xx < 0 || xx >= w) continue;
                    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(
                        in + (((size_t)b * hp + yy) * wp + xx) * in_cs + g * 8));
                    bf16x8_max(acc, v);
                }
            }
        }
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) = acc;
    }
}

// 2x2 / stride 2 / no padding, the pool of every north-star cfg: 32-bit index math, one thread per
// output position x 8 channels, the four window loads issued before the first max.  The layer is a
// pure stream: (4 + 1) * 16 bytes per thread.
__global__ void maxpool2x2_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs, __nv_bfloat16 *__restrict__ out,
                                  int out_cs, int batch, int c8, int h, int w, int oh, int ow)
{
    const int ohp = oh + 1, owp = ow + 1, hp = h + 1, wp = w + 1;
    const unsigned total = (unsigned)batch * ohp * owp * c8;
    const size_t row = (size_t)wp * in_cs;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const unsigned g = i % c8;
        const unsigned p = i / c8;
        const unsigned ox = p % owp;
        const unsigned q = p / owp;
        const unsigned oy = q % ohp;
        const unsigned b = q / ohp;
        uint4 acc = make_uint4(0u, 0u, 0u, 0u);
        if (ox < (unsigned)ow && oy < (unsigned)oh) {
            const __nv_bfloat16 *src = in + (((size_t)b * hp + 2 * oy) * wp + 2 * ox) * in_cs + g * 8;
            const uint4 v00 = __ldg(reinterpret_cast<const uint4 *>(src));
            const uint4 v01 = __ldg(reinterpret_cast<const uint4 *>(src + in_cs));
            const uint4 v10 = __ldg(reinterpret_cast<const uint4 *>(src + row));
            const uint4 v11 = __ldg(reinterpret_cast<const uint4 *>(src + row + in_cs));
            acc = v00;
            bf16x8_max(acc, v01);
            bf16x8_max(acc, v10);
            bf16x8_max(acc, v11);
        }
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) = acc;
    }
}

// ---------------------------------------------------------------------------------
// reorg, exactly the index map of reorg_cpu(..., forward=0) (blas.c:8-29) as invoked by
// reorg_layer.c:78-85 with the INPUT dims: out[in_index] = x[out_index], both flat NCHW
// indices, x re-read as [c/s^2][h*s][w*s].  Output reports (w/s, h/s, c*s^2).
// One thread per output element, channel innermost on the write side.
// ---------------------------------------------------------------------------------
__global__ void reorg_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs,
                             __nv_bfloat16 *__restrict__ out, int out_cs, int batch, int c, int h, int w,
                             int stride)
{
    const int oc = c * stride * stride, oh = h / stride, ow = w / stride;
    const int ohp = oh + 1, owp = ow + 1, hp = h + 1, wp = w + 1;
    const int out_c = c / (stride * stride);
    const long long total = (long long)batch * ohp * owp * oc;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int ch = (int)(t % oc);
        const long long p = t / oc;
        const int ox = (int)(p % owp);
        const int oy = (int)((p / owp) % ohp);
        const int b = (int)(p / ((long long)owp * ohp));
        __nv_bfloat16 v = __float2bfloat16_rn(0.f);
        if (ox < ow && oy < oh) {
            // flat NCHW index of this output element inside its image
            const int in_index = ox + ow * (oy + oh * ch);
            // decompose as (k, j, i) over the INPUT dims (c, h, w)
            const int i = in_index % w;
            const int j = (in_index / w) % h;
            const int k = in_index / (w * h);
            const int c2 = k % out_c;
            const int offset = k / out_c;
            const int w2 = i * stride + offset % stride;
            const int h2 = j * stride + offset / stride;
            const int out_index = w2 + w * stride * (h2 + h * stride * c2);
            // out_index is a flat NCHW index into the true input (c, h, w)
            const int sx = out_index % w;
            const int sy = (out_index / w) % h;
            const int sc = out_index / (w * h);
            v = in[(((size_t)b * hp + sy) * wp + sx) * in_cs + sc];
        }
        out[(size_t)p * out_cs + ch] = v;
    }
}

// The same permutation through a per-layer lookup table (built once at plan time): the index map
// costs ~15 integer divisions per element, the table makes the layer a plain gather.
// table[(oy*ow + ox)*oc + ch] = element offset of the source inside one padded input image.
__global__ void reorg_table_kernel(int *__restrict__ table, int in_cs, int c, int h, int w, int stride)
{
    const int oc = c * stride * stride, oh = h / stride, ow = w / stride;
    const int wp = w + 1;
    const int out_c = c / (stride * stride);
    const int total = oh * ow * oc;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const int ch = t % oc;
        const int pos = t / oc;
        const int ox = pos % ow, oy = pos / ow;
        const int in_index = ox + ow * (oy + oh * ch);
        const int i = in_index % w;
        const int j = (in_index / w) % h;
        const int k = in_index / (w * h);
        const int c2 = k % out_c;
        const int offset = k / out_c;
        const int w2 = i * stride + offset % stride;
        const int h2 = j * stride + offset / stride;
        const int out_index = w2 + w * stride * (h2 + h * stride * c2);
        const int sx = out_index % w;
        const int sy = (out_index / w) % h;
        const int sc = out_index / (w * h);
        table[t] = (sy * wp + sx) * in_cs + sc;
    }
}

// reverse = 1 (reorg_layer.c:80-81 -> reorg_cpu(..., forward = 1): out[out_index] = x[in_index]): a true
// depth-to-space.  Input (c, h, w), output (c/s^2, h*s, w*s); output element (c2, h2, w2) comes from input channel
// (h2 % s * s + w2 % s) * out_c + c2 at (h2 / s, w2 / s).  Same table layout as above, over the OUTPUT extent.
__global__ void reorg_table_reverse_kernel(int *__restrict__ table, int in_cs, int c, int h, int w, int stride)
{
    const int oc = c / (stride * stride), oh = h * stride, ow = w * stride;
    const int wp = w + 1;
    const int total = oh * ow * oc;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        const int c2 = t % oc;
        const int pos = t / oc;
        const int w2 = pos % ow, h2 = pos / ow;
        const int i = w2 / stride, j = h2 / stride;
        const int offset = (h2 % stride) * stride + (w2 % stride);
        const int k = offset * oc + c2;
        table[t] = (j * wp + i) * in_cs + k;
    }
}

// one thread per 8 output channels: 8 table entries, 8 two-byte gathers, one 16-byte store
__global__ void reorg_gather_kernel(const __nv_bfloat16 *__restrict__ in, size_t in_img_elems,
                                    __nv_bfloat16 *__restrict__ out, int out_cs, const int *__restrict__ table,
                                    int batch, int oc, int oh, int ow)
{
    const int ohp = oh + 1, owp = ow + 1;
    const int c8 = oc / 8;
    const long long total = (long long)batch * ohp * owp * c8;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(t % c8);
        const long long p = t / c8;
        const int ox = (int)(p % owp);
        const int oy = (int)((p / owp) % ohp);
        const int b = (int)(p / ((long long)owp * ohp));
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (ox < ow && oy < oh) {
            const int4 *tp = reinterpret_cast<const int4 *>(table + ((size_t)(oy * ow + ox) * oc + g * 8));
            const int4 t0 = __ldg(tp), t1 = __ldg(tp + 1);
            const unsigned short *src = reinterpret_cast<const unsigned short *>(in) + (size_t)b * in_img_elems;
            v.x = (uint32_t)__ldg(src + t0.x) | ((uint32_t)__ldg(src + t0.y) << 16);
            v.y = (uint32_t)__ldg(src + t0.z) | ((uint32_t)__ldg(src + t0.w) << 16);
            v.z = (uint32_t)__ldg(src + t1.x) | ((uint32_t)__ldg(src + t1.y) << 16);
            v.w = (uint32_t)__ldg(src + t1.z) | ((uint32_t)__ldg(src + t1.w) << 16);
        }
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) = v;
    }
}

// route fallback: copy a channel slice between padded buffers of equal extent
__global__ void copy_channels_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs,
                                     __nv_bfloat16 *__restrict__ out, int out_cs, long long positions,
                                     int c8)
{
    const long long total = positions * c8;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(i % c8);
        const long long p = i / c8;
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) =
            __ldg(reinterpret_cast<const uint4 *>(in + (size_t)p * in_cs + g * 8));
    }
}

// ---------------------------------------------------------------------------------
// shortcut: out = act(in + add sampled), the fused form of shortcut_layer.c:39-44
// (copy_cpu + shortcut_cpu + activate_array) with the index map of blas.c:57-81:
//   out[b, j*sample, i*sample, k] += add[b, j*stride, i*stride, k]   for k < min(c1, c2),
//   j < min(h1, h2), i < min(w1, w2), stride = w1/w2, sample = w2/w1 (each at least 1).
// One thread per (output position, 8-channel group), 16-byte accesses.
// ---------------------------------------------------------------------------------
__global__ void shortcut_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs,
                                const __nv_bfloat16 *__restrict__ add, int add_cs, int add_c, int add_h,
                                int add_w, __nv_bfloat16 *__restrict__ out, int out_cs, int c8, int out_c,
                                int out_h, int out_w, int batch, int act, const float *__restrict__ add32,
                                int add32_cs, float *__restrict__ out32)
{
    const int ohp = out_h + 1, owp = out_w + 1, ahp = add_h + 1, awp = add_w + 1;
    int stride = add_w / out_w, sample = out_w / add_w;
    if (stride < 1) stride = 1;
    if (sample < 1) sample = 1;
    const int minw = add_w < out_w ? add_w : out_w, minh = add_h < out_h ? add_h : out_h;
    const int minc = add_c < out_c ? add_c : out_c;
    const long long total = (long long)batch * ohp * owp * c8;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(t % c8);
        const long long p = t / c8;
        const int ox = (int)(p % owp);
        const int oy = (int)((p / owp) % ohp);
        const int b = (int)(p / ((long long)owp * ohp));
        uint4 res = make_uint4(0u, 0u, 0u, 0u);
        if (ox < out_w && oy < out_h) {
            const uint4 vi = __ldg(reinterpret_cast<const uint4 *>(in + (size_t)p * in_cs + g * 8));
            const __nv_bfloat16 *hi = reinterpret_cast<const __nv_bfloat16 *>(&vi);
            float f[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) f[q] = __bfloat162float(hi[q]);
            const int i = ox / sample, j = oy / sample;
            if (ox % sample == 0 && oy % sample == 0 && i < minw && j < minh && g * 8 < minc) {
                const size_t apos = ((size_t)b * ahp + (size_t)j * stride) * awp + (size_t)i * stride;
                float a[8];
                if (add32) { /* the residual stream's fp32 copy */
                    const float4 *pa = reinterpret_cast<const float4 *>(add32 + apos * add32_cs + g * 8);
                    const float4 a0 = __ldg(pa), a1 = __ldg(pa + 1);
                    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
                    a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
                } else {
                    const uint4 va = __ldg(reinterpret_cast<const uint4 *>(add + apos * add_cs + g * 8));
                    const __nv_bfloat16 *ha = reinterpret_cast<const __nv_bfloat16 *>(&va);
#pragma unroll
                    for (int q = 0; q < 8; ++q) a[q] = __bfloat162float(ha[q]);
                }
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (g * 8 + q < minc) f[q] += a[q];
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (act == Y2_ACT_LEAKY) f[q] = (f[q] > 0.f) ? f[q] : 0.1f * f[q];
                else if (act == Y2_ACT_LOGISTIC) f[q] = 1.f / (1.f + __expf(-f[q]));
                if (g * 8 + q >= out_c) f[q] = 0.f;
            }
            res.x = pack_bf16x2(f[0], f[1]);
            res.y = pack_bf16x2(f[2], f[3]);
            res.z = pack_bf16x2(f[4], f[5]);
            res.w = pack_bf16x2(f[6], f[7]);
            if (out32) {
                float4 *po = reinterpret_cast<float4 *>(out32 + (size_t)p * (c8 * 8) + g * 8);
                po[0] = make_float4(f[0], f[1], f[2], f[3]);
                po[1] = make_float4(f[4], f[5], f[6], f[7]);
            }
        }
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) = res;
    }
}

// The common case of the above (every block of resnet50 but the first of a stage): `add` has the running tensor's
// extent and at least its channels, the activation maps 0 to 0 (linear / leaky).  Pad positions of all operands
// hold zeros (the producers store them, fp32 streams are allocated zeroed and only ever written here), so
// act(0 + 0) = 0 is what belongs there and the kernel is a flat elementwise pass over 8-channel groups: no
// coordinates, no divisions (the general kernel spends four 64-bit divisions per group and reaches 4.6 TB/s).
// ---------------------------------------------------------------------------------
template <bool ADD32, bool OUT32, bool LEAKY>
__global__ void shortcut_same_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs,
                                     const __nv_bfloat16 *__restrict__ add, int add_cs, __nv_bfloat16 *__restrict__ out,
                                     int out_cs, int c8, int c8_shift, unsigned total,
                                     const float *__restrict__ add32, int add32_cs, float *__restrict__ out32)
{
    for (unsigned t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        unsigned p, g;
        if (c8_shift >= 0) {
            p = t >> c8_shift;
            g = t & (unsigned)(c8 - 1);
        } else {
            p = t / (unsigned)c8;
            g = t - p * (unsigned)c8;
        }
        const uint4 vi = __ldg(reinterpret_cast<const uint4 *>(in + (size_t)p * in_cs + g * 8));
        const __nv_bfloat16 *hi = reinterpret_cast<const __nv_bfloat16 *>(&vi);
        float f[8], a[8];
        if (ADD32) {
            const float4 *pa = reinterpret_cast<const float4 *>(add32 + (size_t)p * add32_cs + g * 8);
            const float4 a0 = __ldg(pa), a1 = __ldg(pa + 1);
            a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
            a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
        } else {
            const uint4 va = __ldg(reinterpret_cast<const uint4 *>(add + (size_t)p * add_cs + g * 8));
            const __nv_bfloat16 *ha = reinterpret_cast<const __nv_bfloat16 *>(&va);
#pragma unroll
            for (int q = 0; q < 8; ++q) a[q] = __bfloat162float(ha[q]);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            f[q] = __bfloat162float(hi[q]) + a[q];
            if (LEAKY) f[q] = (f[q] > 0.f) ? f[q] : 0.1f * f[q];
        }
        if (OUT32) {
            float4 *po = reinterpret_cast<float4 *>(out32 + (size_t)p * (c8 * 8) + g * 8);
            po[0] = make_float4(f[0], f[1], f[2], f[3]);
            po[1] = make_float4(f[4], f[5], f[6], f[7]);
        }
        *reinterpret_cast<uint4 *>(out + (size_t)p * out_cs + g * 8) =
            make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    }
}

// ---------------------------------------------------------------------------------
// connected layer input (connected_layer.c:122-155 reads state.input as a flat vector): the tensor of the layer
// before it, or a vector, as ONE padded-NHWC position per image ([B][2][2][kpad], h = w = 1), so that the layer is a
// 1x1 convolution on the tensor cores.  A tensor source is laid out position-major ((y*w + x)*c + ch); the weights
// are permuted to that order when they are uploaded (the reference's flat index is ch*h*w + y*w + x).
// ---------------------------------------------------------------------------------
__global__ void fc_pack_tensor_kernel(const __nv_bfloat16 *__restrict__ in, int in_cs, int c, int h, int w,
                                      __nv_bfloat16 *__restrict__ dst, int kpad, int batch)
{
    const long long per = (long long)h * w * c;
    const long long total = (long long)batch * per;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / per);
        const long long k = t - (long long)b * per;
        const int ch = (int)(k % c);
        const int pos = (int)(k / c);
        const int y = pos / w, x = pos - y * w;
        dst[(size_t)b * 4 * kpad + k] = in[(((size_t)b * (h + 1) + y) * (w + 1) + x) * in_cs + ch];
    }
}

__global__ void fc_pack_vec_kernel(const float *__restrict__ in, int in_stride, int n, __nv_bfloat16 *__restrict__ dst,
                                   int kpad, int batch)
{
    const long long total = (long long)batch * n;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(t / n);
        const int k = (int)(t - (long long)b * n);
        dst[(size_t)b * 4 * kpad + k] = __float2bfloat16_rn(in[(size_t)b * in_stride + k]);
    }
}

// ACTIVATION numbering of activations.h:6-8 (same table as vec_f32.cu)
__device__ __forceinline__ float activate_any(float x, int a)
{
    switch (a) {
    case 0: return 1.f / (1.f + expf(-x));
    case 1: return x > 0.f ? x : 0.f;
    case 2: return x > 0.f ? x : .01f * x;
    case 3: return x;
    case 4: return (x > 0.f ? x : 0.f) + .1f * x;
    case 5: return tanhf(x); /* = 2/(1+e^-2x) - 1, which keeps only a few bits for |x| << 1 */
    case 6: return x < -4.f ? .01f * (x + 4.f) : x > 4.f ? .01f * (x - 4.f) + 1.f : .125f * x + .5f;
    case 7: return x > 0.f ? x : .1f * x;
    case 8: return x >= 0.f ? x : expm1f(x);
    case 9: return tanhf(.5f * x); /* = 2/(1+e^-x) - 1 */
    case 10: {
        /* floor(x / 2.) of the reference, in double there: floor(floor(x) / 2), x / 2.f would underflow to -0
         * for the smallest negative denormal */
        const int n = (int)floorf(x);
        const float half = (float)(n >> 1);
        return (n % 2 == 0) ? half : (x - n) + half;
    }
    case 11: return x < -1.f ? -1.f : x > 1.f ? 1.f : x;
    case 12: return x < 0.f ? .001f * x : x > 1.f ? .001f * (x - 1.f) + 1.f : x;
    }
    return x;
}

// any of the 13 activations on a bf16 padded-NHWC tensor in place: valid positions and real channels only (pads and
// padding channels stay zero whatever f(0) is).  Used behind a convolution whose activation the tensor-core epilogue
// does not implement (it then runs LINEAR): relu, elu, tanh, ... of classifier cfgs.
__global__ void activate_bf16_kernel(__nv_bfloat16 *__restrict__ x, int cs, int c, int batch, int h, int w, int act)
{
    const long long total = (long long)batch * h * w * c;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int ch = (int)(t % c);
        const long long p = t / c;
        const int xx = (int)(p % w);
        const int yy = (int)((p / w) % h);
        const int b = (int)(p / ((long long)w * h));
        __nv_bfloat16 *q = x + (((size_t)b * (h + 1) + yy) * (w + 1) + xx) * cs + ch;
        *q = __float2bfloat16_rn(activate_any(__bfloat162float(*q), act));
    }
}

} // namespace y2

using namespace y2;

extern "C" int y2_fc_pack_tensor(const void *in, int in_cs, int c, int h, int w, void *dst, int kpad, int batch,
                                 y2_stream_t s)
{
    if (!in || !dst || batch <= 0 || (long long)h * w * c > kpad) return Y2_EINVAL;
    fc_pack_tensor_kernel<<<grid_for((long long)batch * h * w * c, 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, in_cs, c, h, w, (__nv_bfloat16 *)dst, kpad, batch);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_fc_pack_vec(const float *in, int in_stride, int n, void *dst, int kpad, int batch, y2_stream_t s)
{
    if (!in || !dst || batch <= 0 || n > kpad) return Y2_EINVAL;
    fc_pack_vec_kernel<<<grid_for((long long)batch * n, 256), 256, 0, to_stream(s)>>>(in, in_stride, n,
                                                                                    (__nv_bfloat16 *)dst, kpad, batch);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_activate_bf16(void *x, int cs, int c, int batch, int h, int w, int activation, y2_stream_t s)
{
    if (!x || activation < 0 || activation > 12) return Y2_EINVAL;
    activate_bf16_kernel<<<grid_for((long long)batch * h * w * c, 256), 256, 0, to_stream(s)>>>(
        (__nv_bfloat16 *)x, cs, c, batch, h, w, activation);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_shortcut(const void *in, int in_cs, const void *add, int add_cs, int add_c, int add_h,
                           int add_w, void *out, int out_cs, int out_c, int out_cpad, int out_h, int out_w,
                           int batch, int act, const float *add_f32, int add_f32_cs, float *out_f32, y2_stream_t s)
{
    if (!in || !add || !out || out_cpad % 8 || in_cs % 8 || add_cs % 8 || out_cs % 8 || out_c > out_cpad ||
        add_h <= 0 || add_w <= 0 || out_h <= 0 || out_w <= 0 || (add_f32 && add_f32_cs % 4)) {
        set_error("y2_shortcut: invalid arguments (out_cpad=%d in_cs=%d add_cs=%d out_cs=%d)", out_cpad, in_cs,
                  add_cs, out_cs);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (out_h + 1) * (out_w + 1) * (out_cpad / 8);
    if (add_h == out_h && add_w == out_w && add_c >= out_c && out_c == out_cpad && act != Y2_ACT_LOGISTIC &&
        total < 0x7fffffffLL && !getenv("Y2_SHORTCUT_GENERAL")) {
        const int c8 = out_cpad / 8;
        int shift = -1;
        if ((c8 & (c8 - 1)) == 0)
            for (shift = 0; (1 << shift) < c8; ++shift) {}
        const int grid = grid_for(total, 256);
        const bool leaky = act == Y2_ACT_LEAKY;
#define Y2_SC(A, O, L)                                                                                           \
    shortcut_same_kernel<A, O, L><<<grid, 256, 0, to_stream(s)>>>(                                              \
        (const __nv_bfloat16 *)in, in_cs, (const __nv_bfloat16 *)add, add_cs, (__nv_bfloat16 *)out, out_cs, c8, \
        shift, (unsigned)total, add_f32, add_f32_cs, out_f32)
        if (add_f32 && out_f32) { if (leaky) Y2_SC(true, true, true); else Y2_SC(true, true, false); }
        else if (add_f32) { if (leaky) Y2_SC(true, false, true); else Y2_SC(true, false, false); }
        else if (out_f32) { if (leaky) Y2_SC(false, true, true); else Y2_SC(false, true, false); }
        else { if (leaky) Y2_SC(false, false, true); else Y2_SC(false, false, false); }
#undef Y2_SC
        Y2_LAUNCH_CHECK();
        return Y2_OK;
    }
    shortcut_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, in_cs, (const __nv_bfloat16 *)add, add_cs, add_c, add_h, add_w,
        (__nv_bfloat16 *)out, out_cs, out_cpad / 8, out_c, out_h, out_w, batch, act, add_f32, add_f32_cs, out_f32);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_pack_nchw_f32(const float *src, void *dst, int batch, int c, int h, int w, int cpad,
                                int cs, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || c <= 0 || cpad < c || cs < cpad) return Y2_EINVAL;
    const long long total = (long long)batch * (h + 1) * (w + 1);
    pack_nchw_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(src, (__nv_bfloat16 *)dst, batch, c, h,
                                                                     w, cpad, cs);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_pack_patches_f32(const float *src, void *dst, int batch, int c, int h, int w, int ksize,
                                   int kpad, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || c * ksize * ksize > kpad) {
        set_error("y2_pack_patches_f32: c*k*k=%d does not fit kpad=%d", c * ksize * ksize, kpad);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (h + 1) * (w + 1);
    const int grid = grid_for(total, 128);
    if (kpad == 32)
        pack_patches_kernel<32><<<grid, 128, 0, to_stream(s)>>>(src, (__nv_bfloat16 *)dst, batch, c, h, w, ksize);
    else if (kpad == 64)
        pack_patches_kernel<64><<<grid, 128, 0, to_stream(s)>>>(src, (__nv_bfloat16 *)dst, batch, c, h, w, ksize);
    else {
        set_error("y2_pack_patches_f32: kpad must be 32 or 64");
        return Y2_EINVAL;
    }
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_gather_patches_f32(const float *src, void *dst, int batch, int c, int h, int w, int ksize,
                                     int stride, int pad, int oh, int ow, int kpad, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || kpad % 8 || c * ksize * ksize > kpad || stride < 1 || oh <= 0 || ow <= 0) {
        set_error("y2_gather_patches_f32: invalid arguments (c*k*k=%d kpad=%d stride=%d)", c * ksize * ksize, kpad,
                  stride);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (oh + 1) * (ow + 1) * (kpad / 8);
    gather_patches_f32_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(
        src, (__nv_bfloat16 *)dst, batch, c, h, w, ksize, stride, pad, oh, ow, kpad);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_gather_rows_f32(const float *src, void *dst, int batch, int c, int h, int w, int ksize, int stride,
                                  int pad, int oh, int ow, int kpad, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || kpad % 8 || ksize < 1 || ksize > 8 || c * ksize * 8 > kpad || stride < 1 ||
        oh <= 0 || ow <= 0) {
        set_error("y2_gather_rows_f32: invalid arguments (c=%d k=%d kpad=%d stride=%d)", c, ksize, kpad, stride);
        return Y2_EINVAL;
    }
    const int rows = batch * (oh + 1);
    const int cap = sm_count() * 8;
    const size_t smem = (size_t)c * ksize * (w | 1) * sizeof(float);
    if (smem <= 48 * 1024)
        gather_rows_f32_smem_kernel<<<rows < cap ? rows : cap, 512, smem, to_stream(s)>>>(
            src, (__nv_bfloat16 *)dst, batch, c, h, w, ksize, stride, pad, oh, ow, kpad);
    else
        gather_rows_f32_kernel<<<rows < cap ? rows : cap, 256, 0, to_stream(s)>>>(
            src, (__nv_bfloat16 *)dst, batch, c, h, w, ksize, stride, pad, oh, ow, kpad);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_gather_patches_bf16(const void *in, int in_cs, int cin_pad, int h, int w, void *dst, int batch,
                                      int ksize, int stride, int pad, int oh, int ow, y2_stream_t s)
{
    if (!in || !dst || batch <= 0 || cin_pad % 8 || in_cs % 8 || cin_pad > in_cs || stride < 1 || oh <= 0 ||
        ow <= 0 || ksize < 1) {
        set_error("y2_gather_patches_bf16: invalid arguments (cin_pad=%d in_cs=%d stride=%d)", cin_pad, in_cs, stride);
        return Y2_EINVAL;
    }
    const int rows = batch * (oh + 1);
    const int cap = sm_count() * 8;
    gather_patches_bf16_kernel<<<rows < cap ? rows : cap, 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, in_cs, cin_pad, h, w, (__nv_bfloat16 *)dst, batch, ksize, stride, pad, oh, ow);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

static const int FRAMES_THREADS = 256;

static int launch_frames(const unsigned char *packed, const y2_frame_window *table, const y2_frame_window &uni,
                         unsigned long long stride, int n, float *dst, int batch, int w, int h, y2_stream_t s)
{
    const long long hw = (long long)w * h;
    if (batch > 65535 || hw > 0x7fffffffLL - FRAMES_THREADS) {
        set_error("y2_frames_u8_to_f32: batch %d or canvas %dx%d beyond the launch limits", batch, w, h);
        return Y2_EINVAL;
    }
    const dim3 grid((unsigned)((hw + FRAMES_THREADS - 1) / FRAMES_THREADS), (unsigned)batch);
    frames_u8_to_f32_kernel<<<grid, FRAMES_THREADS, 0, to_stream(s)>>>(packed, table, uni, stride, n, dst, w, h);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// The window of one frame: the whole canvas (resize_image) or letterbox_image's, with resize_image's scales.
static y2_frame_window frame_window(int src_w, int src_h, int w, int h, int letterbox)
{
    y2_frame_window f = {};
    f.src_w = src_w;
    f.src_h = src_h;
    f.new_w = w;
    f.new_h = h;
    if (letterbox) y2_letterbox_geometry(src_w, src_h, w, h, &f.new_w, &f.new_h, &f.dx, &f.dy);
    // image.c:1954-1955: float w_scale = (float)(im.w - 1) / (w - 1)  (w == 1 divides by zero there too)
    f.w_scale = (float)(src_w - 1) / (f.new_w - 1);
    f.h_scale = (float)(src_h - 1) / (f.new_h - 1);
    return f;
}

extern "C" size_t y2_frame_list_layout(int n, const int *frame_w, const int *frame_h, int w, int h, int letterbox,
                                       y2_frame_window *win, size_t *table_offset)
{
    if (n < 1 || !frame_w || !frame_h || w <= 0 || h <= 0) return 0;
    size_t off = 0;
    for (int i = 0; i < n; ++i) {
        if (frame_w[i] <= 0 || frame_h[i] <= 0) return 0;
        if (win) {
            win[i] = frame_window(frame_w[i], frame_h[i], w, h, letterbox);
            win[i].offset = off;
        }
        off += ((size_t)frame_w[i] * frame_h[i] * 3 + 15) & ~(size_t)15;
    }
    if (table_offset) *table_offset = off;
    return off + (size_t)n * sizeof(y2_frame_window);
}

extern "C" int y2_frames_u8_to_f32(const unsigned char *packed, const y2_frame_window *table, int n, float *dst,
                                   int batch, int w, int h, y2_stream_t s)
{
    if (!packed || !table || !dst || n < 1 || n > batch || w <= 0 || h <= 0) {
        set_error("y2_frames_u8_to_f32: invalid arguments (n=%d batch=%d %dx%d)", n, batch, w, h);
        return Y2_EINVAL;
    }
    const y2_frame_window none = {};
    return launch_frames(packed, table, none, 0, n, dst, batch, w, h, s);
}

extern "C" int y2_frame_desc_rows(const y2_frame_desc *d, y2_frame_rows *rows)
{
    if (d->w <= 0 || d->h <= 0) return Y2_FRAME_BAD_SIZE;
    if (d->format != Y2_FRAME_RGB24 && d->format != Y2_FRAME_BGR24 && d->format != Y2_FRAME_NV12)
        return Y2_FRAME_BAD_FORMAT;
    const bool nv12 = d->format == Y2_FRAME_NV12;
    if (nv12 && (d->w % 2 || d->h % 2)) return Y2_FRAME_BAD_NV12_SIZE;
    const size_t row = (size_t)d->w * (nv12 ? 1 : 3);
    if (row > (size_t)INT_MAX) return Y2_FRAME_BAD_ROW; // the record and the kernel's byte offsets are int
    const size_t pitch = d->pitch ? (size_t)d->pitch : row;
    if (d->pitch < 0 || pitch < row) return Y2_FRAME_BAD_PITCH;
    const size_t uv_pitch = d->uv_pitch ? (size_t)d->uv_pitch : pitch;
    if (nv12 && (d->uv_pitch < 0 || uv_pitch < row)) return Y2_FRAME_BAD_UV_PITCH;
    rows->row = row;
    rows->pitch = pitch;
    rows->uv_pitch = nv12 ? uv_pitch : 0;
    rows->uv = !nv12 ? nullptr
                     : d->uv ? (const unsigned char *)d->uv : (const unsigned char *)d->data + (size_t)d->h * pitch;
    return Y2_FRAME_OK;
}

extern "C" size_t y2_frame_desc_layout(int n, const y2_frame_desc *descs, int w, int h, int letterbox,
                                       y2_frame_src *recs, size_t *table_offset)
{
    if (n < 1 || !descs || w <= 0 || h <= 0) return 0;
    size_t off = 0;
    for (int i = 0; i < n; ++i) {
        const y2_frame_desc &d = descs[i];
        y2_frame_rows fr;
        if (y2_frame_desc_rows(&d, &fr) != Y2_FRAME_OK) return 0;
        const bool nv12 = d.format == Y2_FRAME_NV12;
        y2_frame_src r = {};
        r.win = frame_window(d.w, d.h, w, h, letterbox);
        r.format = d.format;
        if (d.on_device) {
            r.win.offset = (unsigned long long)(uintptr_t)d.data;
            r.uv = (unsigned long long)(uintptr_t)fr.uv;
            r.pitch = (int)fr.pitch;
            r.uv_pitch = (int)fr.uv_pitch;
        } else { // staged tight: NV12 as the Y plane then the UV plane
            const size_t plane = fr.row * d.h;
            r.win.offset = off;
            r.uv = nv12 ? off + plane : 0;
            r.pitch = (int)fr.row;
            r.uv_pitch = nv12 ? (int)fr.row : 0;
            off += (plane + (nv12 ? plane / 2 : 0) + 15) & ~(size_t)15;
        }
        if (recs) recs[i] = r;
    }
    if (table_offset) *table_offset = off;
    return off + (size_t)n * sizeof(y2_frame_src);
}

// One axis of the tiling: the tile extent of a frame extent `ext`, and the origin of tile i of `k`.
static int tile_extent(int ext, int k, int overlap, bool nv12)
{
    long long t = ((long long)ext + (long long)(k - 1) * overlap + k - 1) / k;
    if (t > ext) t = ext;
    if (nv12 && (t & 1)) ++t; // ext is even, so t stays <= ext
    return (int)t;
}
static int tile_origin(int i, int k, int ext, int t, bool nv12)
{
    const int o = k == 1 ? 0 : (int)((long long)i * (ext - t) / (k - 1));
    return nv12 ? o & ~1 : o;
}

static size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

extern "C" int y2_tile_plan(int n, const y2_frame_desc *descs, const y2_tiling *tiling, int w, int h, int max_tiles,
                            unsigned char *staged, y2_tile_layout *layout)
{
    if (n < 1 || !descs || w <= 0 || h <= 0) return Y2_TILE_BAD_DESC;
    for (int i = 0; i < n; ++i) {
        y2_frame_rows fr;
        if (y2_frame_desc_rows(&descs[i], &fr) != Y2_FRAME_OK) return Y2_TILE_BAD_DESC;
    }
    if (!tiling) return Y2_TILE_NULL;
    const y2_tiling t = *tiling;
    if (t.cols < 1 || t.cols > Y2_TILE_MAX || t.rows < 1 || t.rows > Y2_TILE_MAX) return Y2_TILE_BAD_GRID;
    if (t.overlap < 0) return Y2_TILE_BAD_OVERLAP;
    if (t.full != 0 && t.full != 1) return Y2_TILE_BAD_FULL;
    const int per_frame = t.full + t.cols * t.rows;
    const long long n_tiles = (long long)n * per_frame;
    if (n_tiles > max_tiles) return Y2_TILE_TOO_MANY;
    y2_tile_layout lay = {};
    lay.n_tiles = (int)n_tiles;
    lay.max_tiles = per_frame;
    lay.recs_offset = y2_frame_desc_layout(n, descs, w, h, 0, nullptr, nullptr) - (size_t)n * sizeof(y2_frame_src);
    lay.tiles_offset = align16(lay.recs_offset + (size_t)n_tiles * sizeof(y2_frame_src));
    lay.spans_offset = align16(lay.tiles_offset + (size_t)n_tiles * sizeof(y2_tile));
    lay.bytes = lay.spans_offset + (size_t)n * sizeof(y2_tile_span);
    if (layout) *layout = lay;
    if (!staged) return Y2_TILE_OK;
    // each frame's own record (host frames at their staged offsets), written where the tile records go, then each
    // frame's tiles from the last frame back, so a frame's record is read before a tile record covers it
    y2_frame_src *recs = reinterpret_cast<y2_frame_src *>(staged + lay.recs_offset);
    y2_tile *tiles = reinterpret_cast<y2_tile *>(staged + lay.tiles_offset);
    y2_tile_span *spans = reinterpret_cast<y2_tile_span *>(staged + lay.spans_offset);
    y2_frame_desc_layout(n, descs, w, h, 0, recs, nullptr);
    for (int f = n - 1; f >= 0; --f) {
        const y2_frame_src fr = recs[f];
        const y2_frame_desc &d = descs[f];
        const bool nv12 = d.format == Y2_FRAME_NV12;
        const int tw = tile_extent(d.w, t.cols, t.overlap, nv12), th = tile_extent(d.h, t.rows, t.overlap, nv12);
        const int first = f * per_frame;
        spans[f] = y2_tile_span{first, per_frame};
        for (int k = per_frame - 1; k >= 0; --k) {
            y2_tile g = {f, 0, 0, d.w, d.h, d.w, d.h, 0};
            if (k >= t.full) {
                const int j = k - t.full;
                g.w = tw;
                g.h = th;
                g.x0 = tile_origin(j % t.cols, t.cols, d.w, tw, nv12);
                g.y0 = tile_origin(j / t.cols, t.rows, d.h, th, nv12);
            }
            y2_frame_src r = fr;
            r.win = frame_window(g.w, g.h, w, h, 0);
            r.win.offset = fr.win.offset + (unsigned long long)g.y0 * fr.pitch + (unsigned long long)g.x0 * (nv12 ? 1 : 3);
            if (nv12) r.uv = fr.uv + (unsigned long long)(g.y0 / 2) * fr.uv_pitch + g.x0;
            recs[first + k] = r;
            tiles[first + k] = g;
        }
    }
    return Y2_TILE_OK;
}

extern "C" int y2_frames_src_to_f32(const y2_frame_src *table, int n, float *dst, int batch, int w, int h,
                                    y2_stream_t s)
{
    const long long hw = (long long)w * h;
    if (!table || !dst || n < 1 || n > batch || w <= 0 || h <= 0 || batch > 65535 ||
        hw > 0x7fffffffLL - FRAMES_THREADS) {
        set_error("y2_frames_src_to_f32: invalid arguments (n=%d batch=%d %dx%d)", n, batch, w, h);
        return Y2_EINVAL;
    }
    const dim3 grid((unsigned)((hw + FRAMES_THREADS - 1) / FRAMES_THREADS), (unsigned)batch);
    frames_src_to_f32_kernel<<<grid, FRAMES_THREADS, 0, to_stream(s)>>>(table, n, dst, w, h);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// a uniform batch: one record passed by value, frame b at b * src_h * src_w * 3
static int uniform_frames(const unsigned char *src, float *dst, int batch, int src_w, int src_h, int w, int h,
                          int letterbox, y2_stream_t s)
{
    const y2_frame_window f = frame_window(src_w, src_h, w, h, letterbox);
    return launch_frames(src, nullptr, f, (unsigned long long)src_w * src_h * 3, batch, dst, batch, w, h, s);
}

extern "C" int y2_resize_u8_to_f32(const unsigned char *src, float *dst, int batch, int src_w, int src_h, int w,
                                   int h, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || src_w <= 0 || src_h <= 0 || w <= 0 || h <= 0) {
        set_error("y2_resize_u8_to_f32: invalid arguments (%dx%d -> %dx%d)", src_w, src_h, w, h);
        return Y2_EINVAL;
    }
    return uniform_frames(src, dst, batch, src_w, src_h, w, h, 0, s);
}

extern "C" void y2_letterbox_geometry(int src_w, int src_h, int w, int h, int *new_w, int *new_h, int *dx, int *dy)
{
    if (((float)w / src_w) < ((float)h / src_h)) {
        *new_w = w;
        *new_h = (src_h * w) / src_w;
    } else {
        *new_h = h;
        *new_w = (src_w * h) / src_h;
    }
    *dx = (w - *new_w) / 2;
    *dy = (h - *new_h) / 2;
}

extern "C" int y2_letterbox_u8_to_f32(const unsigned char *src, float *dst, int batch, int src_w, int src_h, int w,
                                      int h, y2_stream_t s)
{
    if (!src || !dst || batch <= 0 || src_w <= 0 || src_h <= 0 || w <= 0 || h <= 0) {
        set_error("y2_letterbox_u8_to_f32: invalid arguments (%dx%d -> %dx%d)", src_w, src_h, w, h);
        return Y2_EINVAL;
    }
    return uniform_frames(src, dst, batch, src_w, src_h, w, h, 1, s);
}

extern "C" int y2_unpack_to_nchw_f32(const void *src, float *dst, int batch, int c, int h, int w, int cs,
                                     y2_stream_t s)
{
    if (!src || !dst || batch <= 0) return Y2_EINVAL;
    const long long ntiles = (long long)batch * h * ((w + 31) / 32) * ((c + 31) / 32);
    long long grid = ntiles;
    const long long cap = (long long)sm_count() * 32;
    if (grid > cap) grid = cap;
    unpack_nchw_kernel<<<(int)grid, dim3(32, 8), 0, to_stream(s)>>>((const __nv_bfloat16 *)src, dst, batch, c, h,
                                                                    w, cs);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_flat_to_nchw_f32(const float *src, float *dst, int batch, int c, int hw, int cs,
                                   y2_stream_t s)
{
    if (!src || !dst) return Y2_EINVAL;
    const long long total = (long long)batch * c * hw;
    flat_to_nchw_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(src, dst, batch, c, hw, cs);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_nchw_to_flat_f32(const float *src, float *dst, int batch, int c, int hw, y2_stream_t s)
{
    if (!src || !dst) return Y2_EINVAL;
    const long long total = (long long)batch * c * hw;
    nchw_to_flat_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(src, dst, batch, c, hw);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_maxpool(const void *in, int in_cs, void *out, int out_cs, int batch, int c, int h, int w,
                          int out_h, int out_w, int size, int stride, int pad, y2_stream_t s)
{
    if (!in || !out || c % 8 || in_cs % 8 || out_cs % 8) {
        set_error("y2_maxpool: channel counts must be multiples of 8 (c=%d in_cs=%d out_cs=%d)", c, in_cs, out_cs);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (out_h + 1) * (out_w + 1) * (c / 8);
    if (size == 2 && stride == 2 && pad == 0 && out_h == h / 2 && out_w == w / 2 && total < 0x7fffffffLL) {
        long long blocks = (total + 255) / 256;
        const long long cap = (long long)sm_count() * 32;
        if (blocks > cap) blocks = cap;
        maxpool2x2_kernel<<<(int)blocks, 256, 0, to_stream(s)>>>((const __nv_bfloat16 *)in, in_cs, (__nv_bfloat16 *)out,
                                                                 out_cs, batch, c / 8, h, w, out_h, out_w);
        Y2_LAUNCH_CHECK();
        return Y2_OK;
    }
    maxpool_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, in_cs, (__nv_bfloat16 *)out, out_cs, batch, c / 8, h, w, out_h, out_w, size,
        stride, pad);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_reorg(const void *in, int in_cs, void *out, int out_cs, int batch, int c, int h, int w,
                        int stride, y2_stream_t s)
{
    if (!in || !out || stride <= 0 || c % (stride * stride) || h % stride || w % stride) {
        set_error("y2_reorg: c=%d h=%d w=%d not divisible by stride=%d", c, h, w, stride);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (h / stride + 1) * (w / stride + 1) * c * stride * stride;
    reorg_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>((const __nv_bfloat16 *)in, in_cs,
                                                                 (__nv_bfloat16 *)out, out_cs, batch, c, h, w,
                                                                 stride);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_reorg_table(int *table, int in_cs, int c, int h, int w, int stride, y2_stream_t s)
{
    if (!table || stride <= 0 || c % (stride * stride) || h % stride || w % stride) {
        set_error("y2_reorg_table: c=%d h=%d w=%d not divisible by stride=%d", c, h, w, stride);
        return Y2_EINVAL;
    }
    const long long total = (long long)(h / stride) * (w / stride) * c * stride * stride;
    reorg_table_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(table, in_cs, c, h, w, stride);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_reorg_gather(const void *in, int in_cs, void *out, int out_cs, const int *table, int batch, int c,
                               int h, int w, int stride, y2_stream_t s)
{
    const int oc = c * stride * stride;
    if (!in || !out || !table || stride <= 0 || c % (stride * stride) || h % stride || w % stride || oc % 8 ||
        out_cs % 8 || ((uintptr_t)out & 15) || ((uintptr_t)table & 15)) {
        set_error("y2_reorg_gather: invalid arguments (c=%d h=%d w=%d stride=%d out_cs=%d)", c, h, w, stride, out_cs);
        return Y2_EINVAL;
    }
    const int oh = h / stride, ow = w / stride;
    const long long total = (long long)batch * (oh + 1) * (ow + 1) * (oc / 8);
    reorg_gather_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, (size_t)(h + 1) * (w + 1) * in_cs, (__nv_bfloat16 *)out, out_cs, table, batch, oc,
        oh, ow);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_reorg_table_reverse(int *table, int in_cs, int c, int h, int w, int stride, y2_stream_t s)
{
    if (!table || stride <= 0 || c % (stride * stride)) {
        set_error("y2_reorg_table_reverse: c=%d not divisible by stride^2=%d", c, stride * stride);
        return Y2_EINVAL;
    }
    const long long total = (long long)h * w * c;
    reorg_table_reverse_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(table, in_cs, c, h, w, stride);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

// gather through a table built by y2_reorg_table_reverse: in (c, h, w) -> out (c/s^2, h*s, w*s)
extern "C" int y2_reorg_gather_reverse(const void *in, int in_cs, void *out, int out_cs, const int *table, int batch,
                                       int c, int h, int w, int stride, y2_stream_t s)
{
    if (!in || !out || !table || stride <= 0 || c % (stride * stride)) return Y2_EINVAL;
    const int oc = c / (stride * stride), oh = h * stride, ow = w * stride;
    if (oc % 8 || out_cs % 8 || ((uintptr_t)out & 15) || ((uintptr_t)table & 15)) {
        set_error("y2_reorg_gather_reverse: needs a multiple of 8 output channels (c=%d stride=%d out_cs=%d)", c, stride,
                  out_cs);
        return Y2_EINVAL;
    }
    const long long total = (long long)batch * (oh + 1) * (ow + 1) * (oc / 8);
    reorg_gather_kernel<<<grid_for(total, 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, (size_t)(h + 1) * (w + 1) * in_cs, (__nv_bfloat16 *)out, out_cs, table, batch, oc,
        oh, ow);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}

extern "C" int y2_copy_channels(const void *in, int in_cs, void *out, int out_cs, int batch, int c, int h,
                                int w, y2_stream_t s)
{
    if (!in || !out || c % 8 || in_cs % 8 || out_cs % 8) return Y2_EINVAL;
    const long long positions = (long long)batch * (h + 1) * (w + 1);
    copy_channels_kernel<<<grid_for(positions * (c / 8), 256), 256, 0, to_stream(s)>>>(
        (const __nv_bfloat16 *)in, in_cs, (__nv_bfloat16 *)out, out_cs, positions, c / 8);
    Y2_LAUNCH_CHECK();
    return Y2_OK;
}
